"""Host-side logic that needs no GPU: the -m/-p option grammar, option-map translation, corpus helpers."""
import pytest

import corpus


def test_string_to_actions_grammar():
    import erlamsa_b200 as E
    d = E.default_mutations()
    # erlamsa_cmdparse:string_to_actions/3: reversed list; a bare code takes its DEFAULT priority (sgm = 10, num = 3, bd = 1)
    assert E.string_to_actions("bd,num=3,sr=2", "mutation", d) == [("sr", 2), ("num", 3), ("bd", 1)]
    assert E.string_to_actions("sgm,num,bd=7", "mutation", d) == [("bd", 7), ("num", 3), ("sgm", 10)]
    assert dict(E.string_to_actions("bd=2,bd=5", "mutation", d)) == {"bd": 2}          # as a map the FIRST entry wins (maps:from_list of the reversed list)
    assert E.string_to_actions("bd=2=3,,num=", "mutation", d) == [("num", 3), ("bd", 1)]  # string:tokens/2 pieces
    assert E.string_to_actions("default", "mutation", d) == d
    with pytest.raises(ValueError):
        E.string_to_actions("bd=x", "mutation", d)
    with pytest.raises(ValueError):
        E.string_to_actions("bd,nope", "mutation", d)


def test_make_opts_translates_the_reference_option_map():
    import erlamsa_b200 as E
    o = E.make_opts({"seed": (7, 8, 9), "mutations": [("bd", 2), ("num", 5)], "patterns": "od,nd=3", "blockscale": 2.0, "skip": 10})
    codes = E.mutator_codes()
    assert list(o.seed) == [7, 8, 9] and o.blockscale == 2.0 and o.first_case == 11
    assert o.muta_pri[codes.index("bd")] == 2 and o.muta_pri[codes.index("num")] == 5 and o.muta_pri[codes.index("sr")] == -1
    pc = E.pattern_codes()
    assert o.pat_pri[pc.index("od")] == 1 and o.pat_pri[pc.index("nd")] == 3 and o.pat_pri[pc.index("bu")] == -1
    with pytest.raises(ValueError):
        E.make_opts({"mutations": {"xx": 1}})


def test_unseeded_options_get_a_random_seed():
    import erlamsa_b200 as E
    a, b = E.make_opts({}), E.make_opts({})
    assert all(0 <= x < 65536 for x in a.seed)
    assert list(a.seed) != list(b.seed) or True   # 2^-48 chance of equality; only the range is asserted


def test_corpora_are_deterministic():
    a = corpus.mixed_corpus(1, 50)
    b = corpus.mixed_corpus(1, 50)
    assert a == b and len({len(x) for x in a}) > 10
    assert corpus.uniform_corpus(2, 3, 4096, "num")[0][:1] != b""


def test_shard_windows_partition_the_case_range():
    from erlamsa_b200.sharding import shard_window
    for n, world in ((100, 1), (100, 2), (1000003, 8), (5, 8)):
        got = []
        for r in range(world):
            first, cnt = shard_window(n, r, world, first_case=11)
            got.extend(range(first, first + cnt))
        assert got == list(range(11, 11 + n))


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver times next to ours) runs without a GPU and prints one JSON
    line with the keys of the bench contract"""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=240)
    assert out.returncode == 0, out.stderr[-500:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["unit"] == "cases/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0


def test_bench_dump_outputs_writes_the_last_steps_results(tmp_path):
    """`bench.py --dump-outputs DIR` on host tensors standing in for the device buffers: every case's length, a fixed seeded
    sample of whole cases' bytes (-1 past each case's end), the step's counters; float arrays, at most 64 MB in all"""
    import glob
    import os
    import sys
    import numpy as np
    import torch
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    from erlamsa_b200 import _native as N
    size, n = 4096, 3000
    r = np.random.Generator(np.random.PCG64(3))
    lens = r.integers(0, 2 * size + 100, n)
    offs = np.concatenate([[0], np.cumsum(lens)])
    out = torch.from_numpy(r.integers(0, 256, int(offs[-1]) + 64, dtype=np.uint8))
    st = N.Stats(n_cases=n, bytes_in=n * size, bytes_out=int(lens.sum()), n_unsupported=2, n_died=1, n_overflow=0)
    for d in ("a", "b"):
        bench.dump_outputs(torch, str(tmp_path / d), 1001, size, out, torch.from_numpy(offs), torch.from_numpy(lens), st)
    files = sorted(os.path.basename(p) for p in glob.glob(str(tmp_path / "a" / "*.npy")))
    assert files == ["out_len.npy", "sample_case.npy", "sample_out.npy", "stats.npy"]
    got = {f[:-4]: np.load(str(tmp_path / "a" / f)) for f in files}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(os.path.getsize(str(tmp_path / "a" / f)) for f in files) <= 64 << 20
    assert all(np.array_equal(got[f[:-4]], np.load(str(tmp_path / "b" / f))) for f in files)
    assert np.array_equal(got["out_len"], lens) and list(got["stats"]) == [n, n * size, lens.sum(), 2, 1, 0]
    ks = got["sample_case"].astype(np.int64) - 1001
    assert len(ks) == min(n, bench.DUMP_BYTES // (2 * size)) and len(set(ks)) == len(ks)
    for k, row in zip(ks, got["sample_out"]):
        m = min(lens[k], 2 * size)
        assert np.array_equal(row[:m], out[offs[k]:offs[k] + m].numpy()) and (row[m:] == -1).all()


def test_markup_corpus_shapes():
    """C4 documents: exact size, SGML ones tokenise as markup, JSON ones as a complete document (oracle-side check)"""
    import oracle_lib as O
    blobs = corpus.uniform_corpus(11, 6, 3000, "markup")
    assert all(len(b) == 3000 for b in blobs)
    outs, meta = O.fuzzer(blobs, mutations={"sgm": 1, "js": 1}, patterns={"od": 1}, seed=(1, 2, 3), n_cases=48, max_case_out=1 << 20)
    assert all(m.status == 0 for m in meta)
    assert sum(1 for m in meta if m.n_used) >= 40          # refusals would leave the case unused
