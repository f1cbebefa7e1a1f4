"""The Erlang side of the boundary (erlang/erlamsa_b200.erl), EXECUTED: there is no OTP in the build image, so the module
runs under the Erlang evaluator that also runs the reference's sources (oracle/erlref) next to the reference's own modules
it calls (erlamsa_main, erlamsa_mutations, erlamsa_patterns, erlamsa_gen).

 * without the NIF (its stub answers {error, nif_not_loaded}) every call must take the reference path with the caller's n
   and skip and the engine's case numbering;
 * with a MOCK NIF -- the C++ oracle behind the NIF's calling convention, so the arguments the shim builds are the ones
   the real NIF receives -- fuzz_batch/2 must return what the reference returns case by case, including a case the
   mock reports as {flagged, I, St, Why} (re-run alone through erlamsa_main:fuzzer/1) and empty results being dropped.

The reference's sources are not part of this repository: what its modules answered to these tests is recorded in
tests/golden/erlang_shim_calls.json and replayed (oracle/erlref/replay.py), so a call the project's Erlang makes with other
arguments than when it was recorded fails. With the reference's sources present (ERLAMSA_REFERENCE_SRC),
`ERLREF_RECORD=1 python -m pytest tests/test_erlang_shim.py` runs them there and rewrites the file. CPU only."""
import os
import sys

import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "oracle"))
from erlref import refrun, replay  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CALLS = replay.Calls(os.path.join(ROOT, "tests", "golden", "erlang_shim_calls.json"), record=bool(os.environ.get("ERLREF_RECORD")))
if CALLS.record and not refrun.available():
    raise RuntimeError("ERLREF_RECORD needs the reference's sources (ERLAMSA_REFERENCE_SRC)")

SEED = (11, 22, 33)
BLOBS = [b"hello 100 world 42\n", b"alpha beta\ngamma delta\nalpha beta\n", b"<a href=\"x\">t</a> 7 'q' 12345\n", bytes(range(64)) * 3]


def in_evaluator(fn):
    from erlref.interp import run_with_big_stack
    box = {}

    def go():
        box["v"] = fn()
    run_with_big_stack(go)
    return box["v"]


def reference(*extra_dirs):
    """an evaluator with the project's Erlang modules loaded on demand and the reference's modules answered by CALLS"""
    r = refrun.Reference()
    r.rt.src_dirs.extend([os.path.join(ROOT, "erlang")] + list(extra_dirs))
    CALLS.attach(r.rt, refrun.REF_SRC)
    return r


@pytest.fixture(scope="module", autouse=True)
def recorded_calls():
    yield CALLS
    if CALLS.record:
        CALLS.save()


@pytest.fixture(scope="module")
def ref():
    return reference()


def call(ref, mod, fun, *args):
    rt = ref.rt
    rt.steps = 0
    rt.budget = 60_000_000
    return rt.call(mod, fun, *args)


def test_tables_the_shim_sends_are_in_the_engines_order(ref):
    import oracle_lib as O
    from erlref.terms import to_py
    assert in_evaluator(lambda: list(to_py(call(ref, "erlamsa_b200", "mutator_table")))) == list(O.MUT_CODES)
    assert in_evaluator(lambda: list(to_py(call(ref, "erlamsa_b200", "pattern_table")))) == list(O.PAT_CODES)


def test_supported_routes_only_the_direct_return_path(ref):
    from erlref.terms import from_py
    base = {"paths": from_py(["direct"]), "output": "return", "input": b"x", "seed": SEED}

    def sup(**ch):
        d = dict(base); d.update(ch)
        for k in [k for k, v in d.items() if v is None]:
            del d[k]
        return in_evaluator(lambda: call(ref, "erlamsa_b200", "supported", d))
    assert sup() == "true"                                              # the DEFAULT generator list is fine: stdin / file / jump are dropped for [direct]
    assert sup(output=None) == "false"                                  # the reference's default output is stdout
    assert sup(seed=None) == "false"                                    # unseeded: urandom seed, Erlang path
    assert sup(paths=from_py([from_py([ord(c) for c in "-"])])) == "false"
    assert sup(generators=from_py([("direct", 5), ("random", 1)])) == "true"
    assert sup(generators=from_py([("genfuz", 5), ("direct", 1)])) == "true"      # no external module: genfuz is dropped by the reference too
    assert sup(generators=from_py([("genfuz", 5)]), external_generator=from_py([ord(c) for c in "m"])) == "false"
    assert sup(generators=from_py([("nosuch", 1)])) == "false"
    assert sup(external_mutations=from_py([from_py([ord(c) for c in "m"])])) == "false"


def test_without_the_nif_every_call_is_the_reference_with_the_callers_numbering(ref):
    import oracle_lib as O
    from erlref.terms import from_py, to_py
    opts = {"paths": from_py(["direct"]), "output": "return", "input": BLOBS[0], "seed": SEED, "n": 4}
    a = in_evaluator(lambda: [x for x in to_py(call(ref, "erlamsa_main", "fuzzer", dict(opts)))])
    b = in_evaluator(lambda: [x for x in to_py(call(ref, "erlamsa_b200", "fuzzer", dict(opts)))])
    assert a == b and len(a) == 4
    # corpus mode: case I (skip < I =< n) reads blob (I-1) rem length -- the engine's batch semantics, here the C++ oracle's
    got = in_evaluator(lambda: [x for x in to_py(call(ref, "erlamsa_b200", "fuzz_batch", from_py(BLOBS), {"seed": SEED, "n": 7, "skip": 2}))])
    want, meta = O.fuzzer(BLOBS, seed=SEED, n_cases=5, first_case=3)
    assert all(m.status == 0 for m in meta)
    assert got == [w for w in want if w != b""]


def test_with_a_mock_nif_the_gpu_branch_returns_what_the_reference_returns():
    import oracle_lib as O
    ref = reference()                                                   # a fresh runtime: call sites cache their targets, the stub must never have run
    from erlref.interp import Bif
    from erlref.terms import from_py, to_py
    seen = {}

    def mock_nif(blobs, n, seed, muta_pri, pat_pri, first, blockscale, ssrf, gens, device):
        blobs = [bytes(b) for b in to_py(blobs)]
        mp, pp = list(to_py(muta_pri)), list(to_py(pat_pri))
        seen.update(n=n, first=first, seed=tuple(seed), mp=mp, pp=pp, bs=blockscale, ssrf=ssrf, gens=gens, device=device)
        muts = {c: p for c, p in zip(O.MUT_CODES, mp) if p >= 0}
        pats = {c: p for c, p in zip(O.PAT_CODES, pp) if p >= 0}
        outs, meta = O.fuzzer(blobs, seed=tuple(seed), mutations=muts, patterns=pats, n_cases=n, first_case=first, blockscale=blockscale)
        res = [o for o in outs]
        res[2] = ("flagged", first + 2, 1, 0)                          # pretend the device could not do the third case of the window
        return ("ok", from_py(res), from_py([(m.pattern, m.n_used, m.draws) for m in meta]))

    def run():
        mod = ref.rt.load_module("erlamsa_b200")
        mod.funs[("fuzz_batch_nif", 10)] = Bif(mock_nif, 10, "erlamsa_b200:fuzz_batch_nif")
        return [x for x in to_py(call(ref, "erlamsa_b200", "fuzz_batch", from_py(BLOBS),
                                      {"seed": SEED, "n": 9, "skip": 1, "mutations": from_py([("bd", 1), ("num", 3), ("sr", 1), ("lr2", 1), ("ab", 1)]),
                                       "patterns": from_py([("od", 2), ("nd", 1)]), "blockscale": 1.0}))]
    got = in_evaluator(run)
    assert seen["n"] == 8 and seen["first"] == 2 and seen["seed"] == SEED and seen["device"] == 0
    assert len(seen["mp"]) == len(O.MUT_CODES) and len(seen["pp"]) == len(O.PAT_CODES)
    assert {c: p for c, p in zip(O.MUT_CODES, seen["mp"]) if p >= 0} == {"bd": 1, "num": 3, "sr": 1, "lr2": 1, "ab": 1}
    assert seen["gens"] == (500, 1)                                     # direct and random out of erlamsa_gen:default/0
    want, meta = O.fuzzer(BLOBS, seed=SEED, mutations={"bd": 1, "num": 3, "sr": 1, "lr2": 1, "ab": 1}, patterns={"od": 2, "nd": 1}, n_cases=8, first_case=2)
    assert all(m.status == 0 for m in meta)
    assert got == [w for w in want if w != b""]                         # the flagged case came back from the reference path, in place


def test_faas_batch_endpoint_answers_what_the_reference_would_case_by_case():
    """erlang/erlamsa_b200_esi.erl (SURVEY section 8 row f4) end to end: JSON in, option strings through the reference's own parsers,
    erlamsa_b200:fuzz_batch/2 underneath (here on its reference fallback), JSON out; mod_esi and the client manager are mocked"""
    import base64
    import json
    import oracle_lib as O
    from erlref.terms import from_py, to_py
    ref = reference()
    sent = []

    def flat(x, out):
        if isinstance(x, (bytes, bytearray)):
            out += x
        elif isinstance(x, int):
            out.append(x)
        else:
            for y in x:
                flat(y, out)
        return out
    ref.rt.register("mod_esi", "deliver", 2, lambda sid, data: sent.append(bytes(flat(data, bytearray()))) or "ok")
    ref.rt.register("erlamsa_cmanager", "get_client_context", 2, lambda tok, ses: ("error", "unauth") if tok == "bad" else ("ok", (from_py([ord(c) for c in "S1"]), {})))
    body = json.dumps({"data": [base64.b64encode(b).decode() for b in BLOBS], "n": 6, "skip": 1, "seed": "11,22,33",
                       "mutations": "bd,num=3,sr", "patterns": "od,nd=2", "blockscale": 1.0, "ignored": [1, 2]})
    env = from_py([("remote_addr", from_py([ord(c) for c in "127.0.0.1"]))])
    in_evaluator(lambda: call(ref, "erlamsa_b200_esi", "batch", "sid", env, from_py([ord(c) for c in body])))
    assert sent[0] == b"erlamsa-status: 0\r\nerlamsa-session: S1\r\n\r\n"
    got = [base64.b64decode(x) for x in json.loads(sent[1].decode())]
    want, meta = O.fuzzer(BLOBS, seed=SEED, mutations={"bd": 1, "num": 3, "sr": 1}, patterns={"od": 1, "nd": 2}, n_cases=5, first_case=2)
    assert all(m.status == 0 for m in meta)
    assert got == [w for w in want if w != b""]
    # a request without a seed, and an unauthenticated one
    del sent[:]
    in_evaluator(lambda: call(ref, "erlamsa_b200_esi", "batch", "sid", env, from_py([ord(c) for c in json.dumps({"data": ["QUJD"]})])))
    assert sent[0].startswith(b"erlamsa-status: 500")
    del sent[:]
    bad_env = from_py([("http_erlamsa_token", "bad")])
    in_evaluator(lambda: call(ref, "erlamsa_b200_esi", "batch", "sid", bad_env, from_py([ord(c) for c in body])))
    assert sent[0].startswith(b"erlamsa-status: 401") and sent[1] == b""


def test_otp_dump_tool_runs_and_reproduces_the_committed_vectors(tmp_path):
    """tools/dump_reference_vectors.erl is the one-command recipe for whoever has a real OTP; its Erlang had never been executed.
    Here its own text (shebang and -mode line stripped, a -module line added) runs under the evaluator with file:consult/1,
    file:open/2 and io:format/3 backed by Python, over a sample of tests/golden/reference_cases.term, and its output goes
    through the same check the OTP hook applies (tests/test_reference_vectors.py::test_otp_run_matches_committed_vectors)."""
    import hashlib
    import json
    from erlref.terms import from_py, to_py
    src = open(os.path.join(ROOT, "tools", "dump_reference_vectors.erl")).read().split("\n")
    body = [ln for ln in src if not ln.startswith("#!") and not ln.startswith("-mode(")]
    (tmp_path / "dump_reference_vectors.erl").write_text("-module(dump_reference_vectors).\n-export([main/1]).\n" + "\n".join(body))
    vec = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_vectors.json")))["vectors"]

    def plist(d):
        return "default" if d is None else "[" + ",".join("{%s,%d}" % (k, v) for k, v in d.items()) + "]"
    lines, want = [], {}
    for v in vec[::5]:                                                   # every fifth configuration, its first two cases
        extra = []
        if "generators" in v["extra"]:
            extra.append("{generators,%s}" % plist(v["extra"]["generators"]))
        if "blockscale" in v["extra"]:
            extra.append("{blockscale,%r}" % float(v["extra"]["blockscale"]))
        for k in range(min(2, v["n_cases"])):
            i = v["first_case"] + k
            lines.append('{"%s",%d,"%s",%d,{%d,%d,%d},%s,%s,[%s]}' % (v["name"], k, v["blobs"][(i - 1) % len(v["blobs"])], i, v["seed"][0], v["seed"][1], v["seed"][2],
                                                                     plist(v["mutations"]), plist(v["patterns"]), ",".join(extra)))
            want[(v["name"], k)] = (v["status"][k], v["digests"][k])
    ref = reference(str(tmp_path))
    rt = ref.rt
    out = []

    def flat(x, acc):
        if isinstance(x, (bytes, bytearray)):
            acc += x
        elif isinstance(x, int):
            acc.append(x)
        else:
            for y in x:
                flat(y, acc)
        return acc
    rt.register("code", "add_patha", 1, lambda p: "true")
    rt.register("file", "consult", 1, lambda p: ("ok", from_py([rt.eval(ln) for ln in lines])))
    rt.register("file", "open", 2, lambda p, m: ("ok", "the_fd"))
    fmt = rt.bifs[("io_lib", "format", 2)].fn
    rt.register("io", "format", 3, lambda fd, f, a: out.append(bytes(flat(fmt(f, a), bytearray())).decode("latin-1")) or "ok")

    def s(x):
        return from_py([ord(c) for c in x])
    in_evaluator(lambda: call(ref, "dump_reference_vectors", "main", from_py([s("ebin"), s("cases.term"), s("out.txt")])))
    got = {}
    for ln in "".join(out).split("\n"):
        f = ln.split()
        if len(f) >= 3:
            got[(f[0], int(f[1]))] = (f[2], bytes.fromhex(f[3]) if len(f) > 3 else b"")
    assert set(got) == set(want) and len(want) >= 20
    for key, (st, dig) in want.items():
        if st != "ok":
            continue
        assert got[key][0] == "ok", (key, got[key][0])
        assert [len(got[key][1]), hashlib.sha256(got[key][1]).hexdigest()] == list(dig), key


def test_option_string_grammar_of_the_python_mirror_is_the_references(ref):
    """erlamsa_b200.options.string_to_actions against erlamsa_cmdparse:string_to_actions/3 run by the evaluator, on random -m / -p strings
    (bare names, name=N, duplicates, empty pieces, unknown names, bad priorities): same list, or both refuse"""
    import random
    from erlref.terms import from_py, to_py
    from erlamsa_b200.options import string_to_actions
    r = random.Random(5)
    dm = [(str(c), int(p)) for c, p in to_py(in_evaluator(lambda: call(ref, "erlamsa_mutations", "default", from_py([]))))]
    dp = [(str(c), int(p)) for c, p in to_py(in_evaluator(lambda: call(ref, "erlamsa_patterns", "default")))]
    n_ok = n_bad = 0
    for it in range(300):
        table, what = (dm, "mutations") if it % 2 == 0 else (dp, "patterns")
        names = [c for c, _ in table]
        toks = []
        for _ in range(r.randrange(0, 6)):
            name = r.choice(names) if r.random() < 0.9 else r.choice(["nosuch", "", "x1"])
            k = r.random()
            toks.append(name if k < 0.4 else "%s=%d" % (name, r.randrange(0, 40)) if k < 0.85 else name + r.choice(["=", "=2=3", "=x", "=+4", "=-1", "= 5"]))
        s = ",".join(toks)
        want = in_evaluator(lambda: call(ref, "erlamsa_cmdparse", "string_to_actions", from_py([ord(c) for c in s]), from_py([ord(c) for c in what]), from_py(table)))
        try:
            got = string_to_actions(s, what, table)
        except ValueError:
            got = None
        if want[0] == "ok":
            assert got == [(str(c), int(p)) for c, p in to_py(want[1])], (s, got, want)
            n_ok += 1
        else:
            assert got is None, (s, got, want)
            n_bad += 1
    assert n_ok > 100 and n_bad > 30
