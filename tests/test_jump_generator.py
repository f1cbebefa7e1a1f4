"""The jump generator on the device (reference src/erlamsa_gen.erl:123-150, eb_decide.cuh force_jump): with eb200_opts.jump_on_device
a run whose parent draw lands on `jump` is run by the engine -- every case picks two files, cuts each into random-size blocks, picks
one block of each and mutates a random slice of the first ++ a random slice of the second.

  CPU: the parent's draw with the option against the oracle; without it the engine still refuses such a run; the option map key.
  GPU: the reference's own jump vectors; randomised runs against the oracle (big files, exact block multiples, tiny and empty
       files, three block scales, LIGHT and FULL kernels); the three host / device entry points, including a batch big enough for
       the pipelined host path; slot sizing; Philox mode; the Python mirror of fuzzer/1 over three files."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import corpus

HERE = os.path.dirname(os.path.abspath(__file__))
JUMP_PATH = os.path.join(HERE, "golden", "reference_vectors_jump.json")
JVEC = json.load(open(JUMP_PATH))["vectors"] if os.path.exists(JUMP_PATH) else []
LIGHT = {c: 1 for c in ("bd", "bei", "bed", "bf", "bi", "ber", "br", "sd", "num", "ld", "lr2", "ls", "uw", "ui", "sr", "lp")}
CAP = 1 << 22


def _first_thread_seed(a1, a2, a3):
    out = []
    for _ in range(3):                      # gen_predictable_seed/0 = 3 x erand(99999) over AS183
        a1, a2, a3 = a1 * 171 % 30269, a2 * 172 % 30307, a3 * 170 % 30323
        r = a1 / 30269 + a2 / 30307 + a3 / 30323
        out.append(int((r - int(r)) * 99999) + 1)
    return out


def _engine_parent(opts, n_blobs, n_cases=1):
    import erlamsa_b200
    from erlamsa_b200 import _native as N
    o = erlamsa_b200.make_opts(opts)
    out = (C.c_int64 * 8)()
    rc = N.lib().eb200_debug_parent_draws(C.byref(o), n_blobs, n_cases, out)
    return rc, list(out)


# ---------------------------------------------------------------- CPU
def test_parent_draws_with_jump_on_device_match_the_oracle(oracle):
    import erlamsa_b200
    r = np.random.Generator(np.random.PCG64(20261017))
    codes = [c for c, _ in erlamsa_b200.default_mutations() if c in erlamsa_b200.supported_mutations()]
    pcodes = ["od", "nd", "bu", "sk", "sz", "cs", "co", "nu"]
    files = [b"alpha 1\nbeta 22\n", b"gamma 333\ndelta\n" * 40, b"x" * 300]
    n_jump = 0
    for it in range(300):
        seed = tuple(int(x) for x in r.integers(0, 100000, size=3))
        muts = {c: int(r.integers(1, 6)) for c in r.choice(codes, size=int(r.integers(1, 12)), replace=False)}
        pats = {c: int(r.integers(1, 4)) for c in r.choice(pcodes, size=int(r.integers(1, 4)), replace=False)}
        kind = it % 3
        if kind == 0:
            gens, blobs = {"jump": 100}, files[:2]
        elif kind == 1:
            gens, blobs = {"random": 1, "jump": 100, "file": 1000}, files
        else:
            gens, blobs = {"random": int(r.integers(0, 5)), "jump": int(r.integers(1, 3000)), "file": int(r.integers(1, 2000))}, files
        rc, out = _engine_parent({"seed": seed, "mutations": muts, "patterns": pats, "generators": gens, "jump_on_device": True}, len(blobs))
        _, meta = oracle.fuzzer(blobs, mutations=muts, patterns=pats, seed=seed, generators=gens, n_cases=1, max_case_out=1 << 20)
        assert rc == 0, (it, seed, gens)
        assert out[0] == meta[0].generator, (it, seed, gens, out, meta[0].generator)
        assert _first_thread_seed(out[4], out[5], out[6]) == list(meta[0].thread_seed), (it, seed)
        assert out[2] == len(muts) and out[3] == len(pats)
        n_jump += out[0] == 4
    assert n_jump >= 100


def test_without_the_option_a_jump_draw_is_still_refused():
    rc, out = _engine_parent({"generators": {"jump": 100}, "seed": (1, 2, 3)}, 2)
    assert rc == -3 and out[0] == 4
    rc, out = _engine_parent({"generators": {"jump": 100}, "seed": (1, 2, 3), "jump_on_device": False}, 2)
    assert rc == -3 and out[0] == 4
    rc, out = _engine_parent({"generators": {"jump": 100}, "seed": (1, 2, 3), "jump_on_device": True}, 2)
    assert rc == 0 and out[0] == 4


def test_make_opts_maps_jump_on_device():
    import erlamsa_b200
    assert erlamsa_b200.make_opts({}).jump_on_device == 0
    assert erlamsa_b200.make_opts({"jump_on_device": True}).jump_on_device == 1
    assert erlamsa_b200.make_opts({"jump_on_device": False}).jump_on_device == 0


# ---------------------------------------------------------------- GPU helpers
def _digest(o):
    return [len(o), hashlib.sha256(o).hexdigest()]


def _compare(engine, oracle, blobs, gens, muts, pats, seed, n, first_case=1, blockscale=1.0, min_cmp=0.8):
    """engine vs oracle over one batch: every case both sides complete agrees in bytes and draws; a died case dies on both"""
    opts = {"seed": seed, "first_case": first_case, "max_case_out": CAP, "generators": gens, "jump_on_device": True, "blockscale": blockscale}
    if muts is not None:
        opts["mutations"] = muts
    if pats is not None:
        opts["patterns"] = pats
    got, gm = engine.fuzz_batch(blobs, opts, n_cases=n)
    ogens = dict(gens)
    if len(blobs) < 2:
        ogens.pop("jump", None)          # make_generator keeps jump only with two or more paths; the oracle does not apply that rule
    want, wm = oracle.fuzzer(blobs, mutations=muts, patterns=pats, seed=seed, generators=ogens, n_cases=n, first_case=first_case,
                             max_case_out=CAP, blockscale=blockscale)
    bad, n_cmp, n_flag = [], 0, 0
    for k in range(n):
        assert list(gm[k].thread_seed) == list(wm[k].thread_seed), k
        assert gm[k].generator == wm[k].generator, k
        if gm[k].status in (1, 3):
            n_flag += 1
            assert got[k] == b"" or gm[k].generator != 4, k       # a flagged jump case outputs nothing
            continue
        if wm[k].status == 2:
            if gm[k].status != 2:
                bad.append((k, "oracle died", gm[k].status))
            continue
        if wm[k].status != 0:
            continue
        n_cmp += 1
        if gm[k].status != 0 or got[k] != want[k] or gm[k].draws != wm[k].draws:
            bad.append((k, gm[k].status, len(got[k]), len(want[k]), gm[k].draws, wm[k].draws))
    assert not bad, "engine differs from the oracle (case, status, len, oracle len, draws, oracle draws): %r" % bad[:8]
    assert n_cmp >= min_cmp * n, (n_cmp, n_flag, n)
    return gm


def _files(seed, sizes):
    r = corpus.rng(seed)
    out = []
    for i, s in enumerate(sizes):
        if i % 2:
            out.append(corpus.numeric_text(r, s)[:s].ljust(s, b"7"))
        else:
            out.append(corpus.random_bytes(r, s))
    return out


# ---------------------------------------------------------------- GPU: the reference's vectors
@pytest.mark.gpu
@pytest.mark.parametrize("v", JVEC, ids=[v["name"] for v in JVEC])
def test_engine_matches_reference_jump_vectors(v, engine):
    blobs = [bytes.fromhex(b) for b in v["files"]]
    cases = v["cases"]
    assert cases == list(range(cases[0], cases[0] + len(cases)))
    opts = {"seed": tuple(v["seed"]), "first_case": cases[0], "max_case_out": 1 << 26, "generators": v["generators"], "jump_on_device": True}
    if v["mutations"] is not None:
        opts["mutations"] = v["mutations"]
    if v["patterns"] is not None:
        opts["patterns"] = v["patterns"]
    opts.update(v["extra"])
    outs, meta = engine.fuzz_batch(blobs, opts, n_cases=len(cases))
    flagged = {str(i): [meta[idx].status, meta[idx].pad] for idx, i in enumerate(cases) if meta[idx].status not in (0, 2)}
    bad = []
    for idx, i in enumerate(cases):
        st = v["status"][idx]
        if st == "ok" and (meta[idx].status != 0 or _digest(outs[idx]) != v["digests"][idx] or meta[idx].draws != v["draws"][idx]):
            bad.append((i, meta[idx].status, len(outs[idx]), v["digests"][idx][0], meta[idx].draws, v["draws"][idx]))
        elif st == "died" and meta[idx].status != 2:
            bad.append((i, "reference died, engine status", meta[idx].status))
    assert not bad, "engine differs from the reference at %r" % bad[:8]
    assert flagged == {}, flagged


# ---------------------------------------------------------------- GPU: randomised against the oracle
@pytest.mark.gpu
def test_big_files_cross_many_cutter_steps(engine, oracle):
    """files of 64 KiB - 2 MiB: a file is hundreds of blocks, the picked block is found by replaying the cutter far into the stream"""
    blobs = _files(0x1A3B01, [64 << 10, 2 << 20, 700 << 10, 1 << 20, 130 << 10])
    for seed in ((1, 2, 3), (77, 5, 901)):
        gm = _compare(engine, oracle, blobs, {"jump": 100}, LIGHT, {"od": 1, "nd": 1, "bu": 1}, seed, 160)
        assert all(m.generator == 4 for m in gm)


@pytest.mark.gpu
def test_exact_block_multiples_tiny_and_empty_files(engine, oracle):
    """files of exactly k x 256 and k x 4096 bytes (a block that ends on the last byte fits), 0 - 2 byte files and files of a few
    dozen bytes, where the finish/1 tail is often the picked block and an empty file can leave no block at all (the worker dies)"""
    blobs = _files(0x1A3B02, [4096, 8192, 256 * 7, 4096 * 5, 0, 1, 2, 3, 17, 40, 255, 256, 257])
    gm = _compare(engine, oracle, blobs, {"jump": 100}, LIGHT, {"od": 1, "nd": 1, "bu": 1, "nu": 1}, (5, 4, 3), 600, min_cmp=0.6)
    assert sum(m.status == 2 for m in gm) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("bs", [0.25, 1.0, 4.0])
def test_block_scales(engine, oracle, bs):
    blobs = _files(0x1A3B03, [3000, 50000, 9000, 200000, 100])
    _compare(engine, oracle, blobs, {"jump": 100}, LIGHT, {"od": 1, "nd": 1, "bu": 1}, (3, 1, 4), 300, blockscale=bs)


@pytest.mark.gpu
def test_default_table_all_patterns_full_kernel(engine, oracle):
    """the whole default mutator table and every pattern: the FULL flavour of the case kernel"""
    import erlamsa_b200
    muts = {c: p for c, p in erlamsa_b200.default_mutations() if c in erlamsa_b200.supported_mutations()}
    blobs = corpus.mixed_corpus(0x1A3B04, 6, max_len=20000) + corpus.text_corpus(0x1A3B05, 4, 6000)
    _compare(engine, oracle, blobs, {"jump": 100}, muts, None, (9, 8, 7), 300, min_cmp=0.7)


@pytest.mark.gpu
def test_jump_among_the_default_generators_and_one_blob(engine, oracle):
    blobs = _files(0x1A3B06, [5000, 12000, 700])
    gens = {"random": 1, "jump": 100, "file": 1000}
    for seed in ((5, 6, 7), (11, 12, 13), (1, 2, 3)):
        _compare(engine, oracle, blobs, gens, LIGHT, {"od": 1, "nd": 1}, seed, 100)
    _compare(engine, oracle, blobs[:1], gens, LIGHT, {"od": 1, "nd": 1}, (5, 6, 7), 100)


@pytest.mark.gpu
def test_zero_block_size_is_flagged_not_looped(engine):
    """blockscale < 1/512: rand_block_size can be 0 and the reference would loop forever; the engine flags such a case (reason 12)"""
    outs, meta = engine.fuzz_batch([b"abc" * 100, b"xyz" * 50], {"seed": (1, 2, 3), "generators": {"jump": 100}, "jump_on_device": True,
                                                                 "blockscale": 0.001, "mutations": LIGHT, "patterns": {"od": 1}}, n_cases=20)
    assert all(m.status == 1 and m.pad == 12 and o == b"" for m, o in zip(meta, outs))


# ---------------------------------------------------------------- GPU: entry points, pipeline, slots
def _host_into(engine, opts, data, off, n_blobs, n, cap):
    from erlamsa_b200 import _native as N
    out = np.zeros(cap, dtype=np.uint8)
    o_off = np.zeros(n + 1, dtype=np.uint64); o_len = np.zeros(n, dtype=np.uint64)
    meta = (N.Meta * n)(); st = N.Stats()
    rc = N.lib().eb200_fuzz_batch_into(engine._ctx, C.byref(opts), data.ctypes.data, off.ctypes.data, n_blobs, n, out.ctypes.data, out.size,
                                       o_off.ctypes.data, o_len.ctypes.data, meta, C.byref(st))
    assert rc == 0, rc
    return [out[int(o_off[k]):int(o_off[k]) + int(o_len[k])].tobytes() for k in range(n)], meta, st


def _host_plain(engine, opts, data, off, n_blobs, n):
    from erlamsa_b200 import _native as N
    out_p = C.c_void_p(); o_off = np.zeros(n + 1, dtype=np.uint64); o_len = np.zeros(n, dtype=np.uint64)
    meta = (N.Meta * n)(); st = N.Stats()
    u64p = C.POINTER(C.c_uint64)
    rc = N.lib().eb200_fuzz_batch(engine._ctx, C.byref(opts), data.ctypes.data, C.cast(off.ctypes.data, u64p), n_blobs, n, C.byref(out_p),
                                  C.cast(o_off.ctypes.data, u64p), C.cast(o_len.ctypes.data, u64p), meta, C.byref(st))
    assert rc == 0, rc
    try:
        raw = np.ctypeslib.as_array(C.cast(out_p, C.POINTER(C.c_uint8)), shape=(max(int(o_off[n]), 1),))
        outs = [raw[int(o_off[k]):int(o_off[k]) + int(o_len[k])].tobytes() for k in range(n)]
    finally:
        N.lib().eb200_free(out_p)
    return outs, meta, st, int(o_off[n])


def _device(engine, opts, data, off, n_blobs, n, cap):
    import torch
    from erlamsa_b200 import _native as N
    dev = torch.device("cuda:0")
    d_data = torch.zeros(data.size + 64, dtype=torch.uint8, device=dev)
    d_data[:data.size] = torch.from_numpy(data).to(dev)
    d_off = torch.from_numpy(off.astype(np.int64)).to(dev)
    msz = C.sizeof(N.Meta)
    d_out = torch.zeros(cap, dtype=torch.uint8, device=dev)
    d_oo = torch.zeros(n + 1, dtype=torch.int64, device=dev); d_ol = torch.zeros(n, dtype=torch.int64, device=dev)
    d_meta = torch.zeros(n * msz, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    engine.fuzz_batch_device(opts, d_data.data_ptr(), d_off.data_ptr(), n_blobs, data.size, n, d_out.data_ptr(), cap, d_oo.data_ptr(),
                             d_ol.data_ptr(), d_meta.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    o, f, l = d_out.cpu().numpy(), d_oo.cpu().numpy(), d_ol.cpu().numpy()
    mb = d_meta.cpu().numpy().tobytes()
    meta = [N.Meta.from_buffer_copy(mb[k * msz:(k + 1) * msz]) for k in range(n)]
    return [o[int(f[k]):int(f[k]) + int(l[k])].tobytes() for k in range(n)], meta


def _meta_key(m):
    return (m.pattern, m.generator, m.n_used, m.n_failed, tuple(m.used), m.draws, m.status, m.pad, tuple(m.thread_seed))


def _packed(blobs):
    data = np.frombuffer(b"".join(blobs), dtype=np.uint8).copy()
    off = np.zeros(len(blobs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(b) for b in blobs])
    return data, off


@pytest.mark.gpu
@pytest.mark.parametrize("gen", ["jump", "file"])
def test_entry_points_agree(engine, gen):
    import erlamsa_b200
    blobs = _files(0x1A3B07, [int(x) for x in corpus.rng(0x1A3B08).integers(0, 100000, size=40)])
    data, off = _packed(blobs)
    n = 3000
    cap = 3 * sum(len(blobs[k % len(blobs)]) for k in range(n)) + 512 * n + (128 << 20)   # file cases outgrow input-sized slots
    opts = erlamsa_b200.make_opts({"seed": (2, 4, 6), "generators": {gen: 100}, "jump_on_device": True, "mutations": LIGHT,
                                   "patterns": {"od": 1, "nd": 1, "bu": 1}, "max_case_out": CAP})
    a, am, _, _ = _host_plain(engine, opts, data, off, len(blobs), n)
    b, bm, _ = _host_into(engine, opts, data, off, len(blobs), n, cap)
    c, cm = _device(engine, opts, data, off, len(blobs), n, cap)
    assert all(m.generator == (4 if gen == "jump" else 2) for m in am)
    for k in range(n):
        assert a[k] == b[k] == c[k], k
        assert _meta_key(am[k]) == _meta_key(bm[k]) == _meta_key(cm[k]), k


def _oracle_cases(oracle, opts, data, off, n_blobs, first_case, n):
    out_p = C.c_void_p()
    out_off = (C.c_uint64 * (n + 1))()
    meta = (oracle.Meta * n)()
    rc = oracle.lib().eo_fuzzer(C.byref(opts), data.ctypes.data, C.cast(off.ctypes.data, C.POINTER(C.c_uint64)), n_blobs, first_case, n,
                                C.byref(out_p), out_off, meta)
    assert rc == 0
    total = out_off[n]
    raw = bytes((C.c_char * total).from_address(out_p.value)) if total else b""
    return [raw[out_off[i]:out_off[i + 1]] for i in range(n)], list(meta)


@pytest.mark.gpu
@pytest.mark.parametrize("gen", ["jump", "file"])
def test_big_into_batch_reads_every_blob(engine, oracle, gen):
    """A batch shaped for eb200_fuzz_batch_into's pipelined path (512 MiB corpus, 8192 cases over the blob range, two 256 MiB
    chunks): that path uploads each chunk's own blobs only, while a file / jump case reads any blob. Such a batch must give what
    the plain host call gives, and what the oracle gives."""
    import erlamsa_b200
    n, size = 8192, 64 << 10
    r = corpus.rng(0x1A3B09)
    data = r.integers(0, 256, size=n * size, dtype=np.uint8)
    data[::89] = 0x35
    off = np.arange(0, (n + 1) * size, size, dtype=np.uint64)
    o = {"seed": (6, 5, 4), "generators": {gen: 100}, "jump_on_device": True, "mutations": LIGHT, "patterns": {"od": 1, "nd": 1},
         "first_case": 1, "max_case_out": CAP}
    opts = erlamsa_b200.make_opts(o)
    b, bm, bst = _host_into(engine, opts, data, off, n, n, n * size * 17 // 16 + 512 * n + (128 << 20))
    a, am, ast, _ = _host_plain(engine, opts, data, off, n, n)
    assert bst.kernels_launched < 10       # one batch (4 slot kernels + the case kernel), not two pipelined chunks of 5
    for k in range(n):
        assert a[k] == b[k], k
        assert _meta_key(am[k]) == _meta_key(bm[k]), k
    oo = oracle.make_opts(seed=(6, 5, 4), mutations=LIGHT, patterns={"od": 1, "nd": 1}, generators={gen: 100}, max_case_out=CAP)
    for first in (1, n - 63):
        want, wm = _oracle_cases(oracle, oo, data, off, n, first, 64)
        for j in range(64):
            k = first - 1 + j
            if wm[j].status == 0 and bm[k].status == 0:
                assert b[k] == want[j] and bm[k].draws == wm[j].draws, k


@pytest.mark.gpu
def test_slots_are_sized_from_the_block_size(engine):
    """2000 jump cases over two 8 MiB files: input-sized slots would need 16 GB; the outputs take a few MiB"""
    import erlamsa_b200
    blobs = _files(0x1A3B0A, [8 << 20, 8 << 20])
    data, off = _packed(blobs)
    opts = erlamsa_b200.make_opts({"seed": (1, 2, 3), "generators": {"jump": 100}, "jump_on_device": True, "mutations": LIGHT,
                                   "patterns": {"od": 1, "nd": 1}, "max_case_out": CAP})
    outs, meta, _, used = _host_plain(engine, opts, data, off, 2, 2000)
    assert used < (64 << 20), used
    assert sum(m.status == 0 for m in meta) == 2000


@pytest.mark.gpu
def test_philox_jump_is_deterministic_and_distributed_like_as183(engine):
    """Philox mode: the same run twice gives the same bytes, and with the `nu` pattern (the output IS the jump block) which file
    and region each slice starts in, and how long the result is, are distributed as under AS183"""
    import collections
    # file f, byte i = 32 f + i / 8 KiB: the first output byte says which file and which 8 KiB region the first slice starts in
    blobs = [bytes((32 * f + (i >> 13)) & 255 for i in range(64 << 10)) for f in range(4)]
    base = {"seed": (1, 2, 3), "generators": {"jump": 100}, "jump_on_device": True, "mutations": LIGHT, "patterns": {"nu": 1}}
    n = 6000
    p1, _ = engine.fuzz_batch(blobs, dict(base, rng="philox"), n_cases=n)
    p2, _ = engine.fuzz_batch(blobs, dict(base, rng="philox"), n_cases=n)
    assert p1 == p2
    a, _ = engine.fuzz_batch(blobs, base, n_cases=n)
    assert p1 != a

    def hists(outs):
        start = collections.Counter(o[0] if o else -1 for o in outs)
        length = collections.Counter(min(len(o).bit_length(), 14) for o in outs)
        return start, length

    for name, x, y in zip(("slice start", "length"), hists(a), hists(p1)):
        keys = sorted(set(x) | set(y))
        chi2 = sum((x[k] - y[k]) ** 2 / max(x[k] + y[k], 1) for k in keys)
        dof = max(len(keys) - 1, 1)
        assert chi2 < 3.0 * dof + 25, "%s histograms differ: chi2 %.1f on %d dof\n%r\n%r" % (name, chi2, dof, dict(x), dict(y))


@pytest.mark.gpu
def test_mirror_runs_jump_for_several_paths(engine, oracle, tmp_path):
    """erlamsa_main.fuzzer over three files with the reference's default generators: a seed whose parent draw lands on jump (found
    on the CPU) writes, case for case, the oracle's outputs"""
    from erlamsa_b200 import erlamsa_main
    files = _files(0x1A3B0B, [6000, 15000, 900])
    paths = []
    for i, b in enumerate(files):
        p = tmp_path / ("in%d.bin" % i)
        p.write_bytes(b)
        paths.append(str(p))
    gens = {"random": 1, "jump": 100, "file": 1000}
    pats = {"od": 1, "nd": 1, "bu": 1}
    seed = None
    for s in range(1, 5000):
        rc, out = _engine_parent({"seed": (s, 2, 3), "mutations": LIGHT, "patterns": pats, "generators": gens, "jump_on_device": True}, 3)
        if rc == 0 and out[0] == 4:
            seed = (s, 2, 3)
            break
    assert seed is not None
    n = 30
    erlamsa_main.fuzzer({"paths": paths, "output": str(tmp_path / "out" / "%n"), "n": n, "seed": seed, "mutations": LIGHT, "patterns": pats})
    want, wm = oracle.fuzzer(files, mutations=LIGHT, patterns=pats, seed=seed, generators=gens, n_cases=n, max_case_out=1 << 26)
    n_cmp = 0
    for k in range(n):
        assert wm[k].generator == 4
        got = (tmp_path / "out" / str(k + 1)).read_bytes()
        if wm[k].status == 0:
            assert got == want[k], k
            n_cmp += 1
    assert n_cmp >= n * 0.9
