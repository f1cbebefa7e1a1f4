#!/usr/bin/env python
"""Regenerates tests/golden/reference_workers.json: the reference's multi-threaded mode (src/erlamsa_main.erl:88-111,254-280),
run from the reference's own source by oracle/erlref, for tests/test_workers.py:
  threading_mode  [n, workers, plan] for every (n, workers) up to (40, 9): erlamsa_main:get_threading_mode("out/%n", n, workers)
                  as [[first, last, worker, seed], ...] in worker order, or null when it answers 1 (single-threaded);
  plans           per test configuration, the files fuzzer/1 writes: name -> [length, sha256].
Same provenance and purpose as make_reference_vectors.py; needs the reference's sources (ERLAMSA_REFERENCE_SRC)."""
import hashlib
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
from test_workers import GENS, MUTS, PATS, PLANS, plan_files, plan_name  # noqa: E402


def main():
    sys.setrecursionlimit(3000000)
    from erlref.refrun import Reference
    from erlref.terms import from_py, to_py
    rt = Reference().rt
    out = from_py([ord(c) for c in "out/%n"])
    modes = []
    for n in range(1, 41):
        for w in range(1, 10):
            ref = rt.call("erlamsa_main", "get_threading_mode", out, n, w)
            modes.append([n, w, None if ref == 1 else [[t[0][0], t[0][1], t[0][2], t[1]] for t in to_py(ref)]])
    plans = {}
    for n, w, seed, same in PLANS:
        ref = Reference(budget=400_000_000)
        rt = ref.rt
        rt.vfs = {"f%d" % i: b for i, b in enumerate(plan_files())}
        opts = ref.opts_map(b"", seed, MUTS, PATS, n=n, skip=0, generators=GENS)
        del opts["input"]
        opts["paths"] = from_py([from_py([ord(c) for c in p]) for p in ["f0", "f1", "f2"]])
        opts["output"] = from_py([ord(c) for c in "out/%n"])
        opts["workers"] = w
        if same:
            opts["workers_same_seed"] = "true"
        opts["maxrunningtime"] = 600000
        rt.vfs_out = {}
        rt.steps = 0; rt.budget = ref.budget; rt.child_draws = []; rt.last_crash = None
        rt.call("erlamsa_main", "fuzzer", opts)
        plans[plan_name(n, w, seed, same)] = {k: [len(v), hashlib.sha256(v).hexdigest()] for k, v in sorted(rt.vfs_out.items())}
    with open(os.path.join(HERE, "reference_workers.json"), "w") as f:
        json.dump({"threading_mode": modes, "plans": plans}, f, separators=(",", ":"))
        f.write("\n")


if __name__ == "__main__":
    main()
