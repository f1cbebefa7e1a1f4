"""The reference's multi-threaded mode (`workers` > 1 with a file output; src/erlamsa_main.erl:88-111,254-280) as the host mirror plans it
(erlamsa_b200/workers.py) and as the engine's host code seeds it (eb200_opts.case_stream_*), on the CPU:
  * threading_mode/3 == the reference's get_threading_mode/3 for every (n, workers) up to (40, 9);
  * the plan's batches, run through the oracle, give exactly the files the reference's own run writes (workers, same-seed workers, more
    workers than cases);
  * the parent state the engine's host code hands the device makes case I take the (I - A)-th seed of the worker's stream (checked
    against the oracle's thread seeds through eb200_debug_parent_draws).
The reference's side of the first two, executed from its source, is stored in tests/golden/reference_workers.json."""
import ctypes as C
import hashlib
import json
import os

import pytest

import corpus

HERE = os.path.dirname(os.path.abspath(__file__))
PLANS = [(11, 3, (1, 2, 3), False), (12, 4, (4, 5, 6), False), (10, 3, (5, 1, 2), True), (5, 8, (3, 3, 3), False)]
MUTS = {"bd": 1, "bf": 1, "num": 2, "ld": 1, "sr": 1, "fn": 1}
PATS = {"od": 1, "nd": 1, "sk": 1}
GENS = {"random": 1, "file": 1000}


def plan_files():
    return [corpus.text_lines(corpus.rng(1200), 900), corpus.numeric_text(corpus.rng(1201), 500), corpus.random_bytes(corpus.rng(3), 700)]


def plan_name(n, w, seed, same):
    return "%d_%d_%d.%d.%d_%s" % ((n, w) + tuple(seed) + ("same" if same else "own",))


def reference_answers():
    """what the reference's own source answered (tests/golden/make_reference_workers.py)"""
    with open(os.path.join(HERE, "golden", "reference_workers.json")) as f:
        return json.load(f)


def test_threading_mode_equals_the_reference_function():
    from erlamsa_b200.workers import threading_mode
    modes = reference_answers()["threading_mode"]
    assert len(modes) == 40 * 9
    for n, w, ref in modes:
        got = threading_mode("out/%n", n, w)
        if ref is None:
            assert got is None, (n, w)
            continue
        assert [[a, b, wn, r] for wn, (a, b, r) in enumerate(got)] == ref, (n, w, got, ref)
    assert threading_mode("return", 100, 4) is None and threading_mode("-", 100, 4) is None


@pytest.mark.parametrize("n,w,seed,same", PLANS)
def test_plan_through_the_oracle_writes_the_reference_files(oracle, n, w, seed, same):
    from erlamsa_b200.workers import worker_plan
    files = plan_files()
    written = reference_answers()["plans"][plan_name(n, w, seed, same)]                 # file name -> [length, sha256] of what the reference wrote
    assert sorted(written) == sorted("out/%d" % i for i in range(1, n + 1))
    seen = set()
    for wseed, first, cnt, stream_first in worker_plan(seed, "out/%n", n, w, same):
        outs, meta = oracle.fuzzer(files, mutations=MUTS, patterns=PATS, seed=seed, generators=GENS, n_cases=cnt, first_case=first, max_case_out=1 << 24,
                                   case_stream=(wseed, stream_first))
        for k in range(cnt):
            assert meta[k].status == 0 and written["out/%d" % (first + k)] == [len(outs[k]), hashlib.sha256(outs[k]).hexdigest()], (first + k)
            seen.add(first + k)
    assert seen == set(range(1, n + 1))


def _seed_of_case(state, i):
    a = list(state)
    for _ in range(3 * (i - 1)):
        a[0], a[1], a[2] = a[0] * 171 % 30269, a[1] * 172 % 30307, a[2] * 170 % 30323
    out = []
    for _ in range(3):
        a[0], a[1], a[2] = a[0] * 171 % 30269, a[1] * 172 % 30307, a[2] * 170 % 30323
        r = a[0] / 30269 + a[1] / 30307 + a[2] / 30323
        out.append(int((r - int(r)) * 99999) + 1)
    return out


def test_engine_host_code_seeds_a_worker_like_the_oracle(oracle):
    import erlamsa_b200
    from erlamsa_b200 import _native as N
    blobs = [b"alpha 1\n", b"beta 22\n", b"gamma 333\n"]
    muts = {"bd": 1, "num": 2}
    for wseed, a in (((5075, 67279, 16423), 1), ((68415, 61859, 16086), 3), ((10898, 6310, 86030), 600), ((1, 2, 3), 123457)):
        for i in (a, a + 1, a + 7):
            o = erlamsa_b200.make_opts({"seed": (1, 2, 3), "mutations": muts, "patterns": {"od": 1}, "first_case": i, "case_stream": (wseed, a)})
            out = (C.c_int64 * 8)()
            assert N.lib().eb200_debug_parent_draws(C.byref(o), len(blobs), 1, out) == 0
            _, meta = oracle.fuzzer(blobs, mutations=muts, patterns={"od": 1}, seed=(1, 2, 3), n_cases=1, first_case=i, case_stream=(wseed, a))
            # the device takes case I's seed from the state it is handed advanced by 3 (I - 1) steps
            assert _seed_of_case(out[4:7], i) == list(meta[0].thread_seed), (wseed, a, i)
    # a batch that starts before its worker's first case is refused
    o = erlamsa_b200.make_opts({"seed": (1, 2, 3), "first_case": 2, "case_stream": ((1, 2, 3), 5)})
    assert N.lib().eb200_debug_parent_draws(C.byref(o), 3, 1, (C.c_int64 * 8)()) == -2
