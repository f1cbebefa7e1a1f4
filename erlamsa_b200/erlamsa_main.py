"""Python mirror of the reference's driver entry, erlamsa_main:fuzzer/1 (reference src/erlamsa_main.erl:124-247), backed by the
CUDA engine, for the generators and outputs that are part of the hot path's surroundings (SURVEY.md section 8 f3):

    paths  => [direct] with input => Bin | [Bin]   direct generator (src/erlamsa_gen.erl:152-164); a LIST is a corpus: case I
                                                     mutates element (I-1) rem length -- the batched generalisation
    paths  => ["file1", "dir/file2", ...]           file generator (:104-121): every case picks one of the files (erand), which is
                                                     cut lazily into random-size blocks (rand_block_size :55-56); with two or more
                                                     files the parent's draw may land on jump (:123-150): a slice of a block of one
                                                     file ++ a slice of a block of another
    paths  => ["-"]                                 stdin generator (:92-102), n == 1 only (the reference pre-reads stdin in the
                                                     parent process for n > 1, which is not modelled)
    output => return                                -> [binary()], empty results dropped like record_result/2 (:120-122)
    output => "out/fuzz-%n.bin"                     file writer (src/erlamsa_out.erl:103-123): %n = case number; returns []
                                                     like the reference does for non-direct outputs
    workers => W, workers_same_seed => Bool         with a file output and n > 1: the reference's multi-threaded mode (:88-111,254-280) --
                                                     every worker's case range is one engine batch seeded the way that worker process is

`fuzz/1` is the spelling BASELINE.json's north star uses for the same entry.
"""
import os
import sys

from .engine import Engine
from .workers import worker_plan

_engine = None


def _get_engine():
    global _engine
    if _engine is None:
        _engine = Engine(0)
    return _engine


def _file_name(template, n):
    """build_name/3 (src/erlamsa_out.erl:103-107): every %n becomes the case number"""
    return template.replace("%n", str(n))


def fuzzer(opts):
    opts = dict(opts)
    paths = list(opts.get("paths", ["-"]))
    output = opts.get("output", "-")
    if output != "return" and not isinstance(output, str):
        raise NotImplementedError("network / exec outputs stay in Erlang (SURVEY.md section 2)")
    for k in ("sequence_muta", "external_mutations", "external_post", "external_generator"):
        if opts.get(k):      # the Erlang shim routes these option maps to the untouched reference (erlang/erlamsa_b200.erl supported/1)
            raise NotImplementedError("option `%s` has no device implementation" % k)
    o = dict(opts)
    if "seed" not in o:      # the reference falls back to gen_urandom_seed/0 (src/erlamsa_rnd.erl:50-62); fixed here so that the workers' plan sees it
        r = os.urandom(6)
        o["seed"] = opts["seed"] = tuple(int.from_bytes(r[i:i + 2], "big") for i in (0, 2, 4))
    skip = int(opts.get("skip", 0))
    if paths == ["direct"]:
        inp = opts.get("input")
        if inp is None:
            raise ValueError("direct generator needs `input`")
        blobs = [bytes(inp)] if isinstance(inp, (bytes, bytearray, memoryview)) else [bytes(b) for b in inp]
        n = int(opts.get("n", len(blobs) if len(blobs) > 1 else 1))
    elif paths == ["-"]:
        n = int(opts.get("n", 1))
        if n != 1:
            raise NotImplementedError("stdin with n > 1: the reference pre-reads stdin in the parent process (src/erlamsa_gen.erl:98-101)")
        blobs = [opts["stdin_data"] if "stdin_data" in opts else sys.stdin.buffer.read()]
        o.setdefault("generators", {"stdin": 100000, "random": 1})       # what make_generator keeps of the defaults for ["-"]
    else:
        blobs = []
        for p in paths:
            with open(p, "rb") as f:
                blobs.append(f.read())
        n = int(opts.get("n", 1))
        if "generators" not in o:
            # what make_generator keeps of erlamsa_gen:default/0 for file paths (src/erlamsa_gen.erl:204-237): jump only with two or
            # more paths. jump takes part in the parent's generator draw as in the reference (100 in 1101 runs land on it)
            o["generators"] = {"random": 1, "jump": 100, "file": 1000} if len(paths) > 1 else {"random": 1, "file": 1000}
        if len(paths) > 1:
            o.setdefault("jump_on_device", True)      # a run whose draw lands on jump runs it on the device
    plan = worker_plan(opts["seed"], output, n, int(opts.get("workers", 1)), bool(opts.get("workers_same_seed", False))) 
    for k in ("paths", "output", "input", "n", "skip", "stdin_data", "workers", "workers_same_seed"):
        o.pop(k, None)
    if plan is not None:
        # multi-threaded mode: file output only (threading_mode), so every case goes to its own file; cases <= skip are run (their seeds
        # are drawn all the same) but not written
        for wseed, first, cnt, stream_first in plan:
            ow = dict(o, first_case=first, case_stream=(wseed, stream_first))
            outs, _meta = _get_engine().fuzz_batch(blobs, ow, n_cases=cnt)
            _write_files(output, [(first + k, x) for k, x in enumerate(outs) if first + k > skip])
        return []
    o["first_case"] = skip + 1
    outs, _meta = _get_engine().fuzz_batch(blobs, o, n_cases=max(n - skip, 0))
    if output == "return":
        return [x for x in outs if x != b""] if paths == ["direct"] else []
    if output == "-":
        for x in outs:
            sys.stdout.buffer.write(x)
        return []
    # file_writer/1: one file per case, numbered from skip + 1. (The reference also OPENS -- creates, empty -- the files of the skipped
    # case numbers 1..skip before discarding the descriptor, src/erlamsa_main.erl:188-191; that side effect is not reproduced: with
    # skip used for sharding it would mean millions of empty files.)
    _write_files(output, [(skip + 1 + k, x) for k, x in enumerate(outs)])
    return []


def _write_files(template, numbered):
    for i, x in numbered:
        name = _file_name(template, i)
        d = os.path.dirname(name)
        if d:
            os.makedirs(d, exist_ok=True)
        with open(name, "wb") as f:
            f.write(x)


fuzz = fuzzer
