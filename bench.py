#!/usr/bin/env python
"""bench.py -- mutated test cases / s of the erlamsa hot path on B200 (BASELINE.json metric).

A "step" = one pass of the hot path (slot prefix sum -> eb_case_kernel: the one persistent kernel that decides every case
and moves its bytes) over one batch of synthetic seeds resident in HBM. Default workload = BASELINE config C3 (the one the 1e7 cases/s target
is quoted on): 100 000 x 65 536 B uniform-random seeds, mutators bd,bei,bed,bf,bi,ber,br,num at
priority 1, pattern od, AS183-exact RNG. Every step mutates the NEXT window of case ids (first_case
advances), so no step repeats work and the 6.5 GB corpus + 6.5 GB of outputs per step never fit L2.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3|c3num|c2|c4|c5] [--async-depth D]
                  [--dump-outputs DIR]

The default (C3) line also carries `parity_sample` (sampled case ids of the last timed step re-run through the oracle),
`extra_workloads` (short C2 and C4 runs, value net of flagged cases, all-threads CPU port beside them) and, for c5, `collective`.

Under torchrun (N > 1) every rank owns one GPU and its own shard of case ids (weak scaling: per-GPU work
fixed; cases are independent, so there is no data-path collective); timing = max over ranks.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {
    # name: (n_cases, seed_bytes, corpus kind, mutators, patterns, description)
    "c3": (100000, 65536, "bin", ["bd", "bei", "bed", "bf", "bi", "ber", "br", "num"], {"od": 1},
           "C3: 100000 x 65536 B uniform-random seeds; bd,bei,bed,bf,bi,ber,br,num; pattern od"),
    "c3num": (100000, 65536, "num", ["bd", "bei", "bed", "bf", "bi", "ber", "br", "num"], {"od": 1},
              "C3(ii): 100000 x 65536 B numeric text; bd,bei,bed,bf,bi,ber,br,num; pattern od"),
    "c4": (12500, 262144, "markup", ["ab", "ad", "tr2", "td", "ts1", "ts2", "tr", "sgm", "js"], {"od": 1},
           "C4 (one GPU's quarter): 12500 x 262144 B documents, half SGML half JSON, tiled from 64 distinct ones; ab,ad,tr2,td,ts1,ts2,tr,sgm,js; pattern od"),
    "c5": (125000, 4096, "text", ["ft", "fn", "fo"], {"od": 1},
           "C5 (one GPU's eighth of 1 000 000 seeds): 125000 x 4096 B text-like seeds; ft,fn,fo; pattern od; cross-seed donor pool "
           "(4096 windows of 2048 B per GPU, all-gathered over NCCL) for fo"),
    "c2": (10000, 4096, "bin", None, {"od": 1, "nd": 2, "bu": 1, "sk": 2, "sz": 2, "cs": 1, "ar": 1, "cp": 1, "co": 0, "nu": 0},
           "C2: 10000 x 4096 B uniform-random seeds; all 41 mutators at the reference's default priorities; default patterns"),
}


def config_of(workload, n_cases, size, rng):
    """the `config` object of the JSON line: static per workload, so that both arms (--impl ours | reference) print the same one"""
    desc = WORKLOADS[workload][5]
    gb = n_cases * size / 1e9
    l2 = ("inputs larger than L2 (%.2f GB of seeds read and about as much written per step, a new window of case ids every step; 126 MB L2)" % gb
          if n_cases * size > (126 << 20) else
          "inputs (%.3f GB per step) fit the 126 MB L2: this workload is bound by the per-case program, not by memory -- see hbm_frac" % gb)
    return {"workload": desc, "cases_per_gpu_per_step": n_cases, "seed_bytes": size, "rng": rng, "l2_policy": l2,
            "parallelism": "cases sharded by id, no collective" if workload != "c5" else "cases sharded by id; one all-gather of the donor pool per step"}


def ncu_traffic(workload, fused):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the committed ncu capture of this
    workload (profiles/<kernel>_<tag>.txt, `ncu --set full`, one launch); None when there is no capture for it."""
    tag = {"c3": TRAFFIC_PROFILE[bool(fused)]}.get(workload)
    p = os.path.join(ROOT, "profiles", tag) if tag else None
    if not p or not os.path.exists(p):
        return None
    tot = 0.0
    for ln in open(p):
        f = ln.split()
        if len(f) >= 3 and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            tot += float(f[1]) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}.get(f[2], 1.0)
    return tot or None


TRAFFIC_PROFILE = {True: "fused_r2c.txt", False: "apply_r1b.txt"}


def peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    def __init__(self, gpu_index):
        self.proc = None
        self.lines = []
        self.idx = gpu_index

    def start(self):
        # started BEFORE the warm-up steps: nvidia-smi's own start-up (NVML initialisation on the driver) must not fall
        # into the timed region (it cost the first measurements of this bench ~10 % of kernel time); once running it only
        # polls. Every line carries the wall-clock time it was taken, stop() keeps the ones inside the timed window.
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def close(self):
        """ends nvidia-smi whatever happened in between: no poller outlives the benchmark"""
        if self.proc and self.proc.poll() is None:
            self.proc.terminate()
            self.proc.wait(10)

    def stop(self, t0=None, t1=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.close()
        inside = [ln for (t, ln) in self.lines if t0 is not None and t0 <= t <= t1 + 0.03]
        window = "timed region"
        if not inside:      # a region shorter than the polling period: the samples right around it
            inside = [ln for (t, ln) in self.lines if t0 is None or t0 - 0.2 <= t <= t1 + 0.1] or [ln for (_, ln) in self.lines]
            window = "timed region +- 0.2 s"
        sm, mx, reasons = [], None, set()
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm), "window": window}


def make_corpus_device(torch, kind, n, size, dev, seed):
    """synthetic seeds of the configured shape, generated on the device (uniform bytes) or on the host (text)"""
    if kind == "bin":
        g = torch.Generator(device=dev); g.manual_seed(seed)
        data = torch.randint(0, 256, (n * size + 64,), dtype=torch.uint8, device=dev, generator=g)
    else:
        import corpus
        import numpy as np
        r = corpus.rng(seed)
        distinct = 64 if kind == "markup" else 256
        if kind == "markup":
            docs = corpus.uniform_corpus(seed, distinct, size, "markup")
        elif kind == "text":
            docs = [corpus.structured_text(r, size).ljust(size, b" ")[:size] for _ in range(distinct)]
        else:
            docs = [corpus.numeric_text(r, size) for _ in range(distinct)]
        base = np.frombuffer(b"".join(docs), dtype=np.uint8)
        t = torch.from_numpy(base.copy()).to(dev)
        reps = (n + distinct - 1) // distinct
        data = torch.cat([t.repeat(reps)[: n * size], torch.zeros(64, dtype=torch.uint8, device=dev)])
    off = torch.arange(0, (n + 1) * size, size, dtype=torch.int64, device=dev)
    return data, off


DUMP_BYTES = 12 << 20        # output bytes sampled by --dump-outputs: 48 MiB as float32, beside 8 bytes per case of lengths


def dump_outputs(torch, out_dir, first_case, size, d_out, d_out_off, d_out_len, st):
    """What the caller of the timed step received in the last step, as .npy files (float64 / float32) for comparing two builds:
      out_len      every case's output length;
      sample_case  the case ids of a fixed sample (seeded, independent of the outputs, so two builds sample the same cases);
      sample_out   their output bytes, one row per sampled case, the first 2 x seed_bytes of each, -1 past the case's end;
      stats        n_cases, bytes_in, bytes_out, n_unsupported, n_died, n_overflow of the step (eb200_stats without the timings)."""
    import numpy as np
    n = d_out_len.numel()
    width = 2 * size
    count = max(1, min(n, 4096, DUMP_BYTES // width))
    ks = np.sort(np.random.Generator(np.random.PCG64(0xD0)).choice(n, size=count, replace=False))
    kt = torch.from_numpy(ks).to(d_out.device)
    col = torch.arange(width, dtype=torch.int64, device=d_out.device)
    idx = d_out_off[kt][:, None] + col[None, :]
    inside = col[None, :] < d_out_len[kt][:, None]
    rows = torch.where(inside, d_out[idx.clamp(0, d_out.numel() - 1)].float(), torch.full_like(idx, -1, dtype=torch.float32))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "out_len.npy"), d_out_len.cpu().numpy().astype(np.float64))
    np.save(os.path.join(out_dir, "sample_case.npy"), (first_case + ks).astype(np.float64))
    np.save(os.path.join(out_dir, "sample_out.npy"), rows.cpu().numpy())
    np.save(os.path.join(out_dir, "stats.npy"), np.array([st.n_cases, st.bytes_in, st.bytes_out, st.n_unsupported, st.n_died, st.n_overflow], dtype=np.float64))


def measure(torch, dist, eng, args, workload, steps, warmup, rank, world, local, n_override=0, want_e2e=True, sampler=None, dump_dir=None):
    """W warm-up steps + K timed steps of one workload on this rank's GPU; returns the fields of the JSON line (rank 0) or None"""
    import erlamsa_b200
    from erlamsa_b200 import _native as N
    dev = torch.device("cuda", local)
    n_cases, size, kind, muts, pats, desc = WORKLOADS[workload]
    if n_override:
        n_cases = n_override
    if muts is None:
        muts = {c: p for c, p in erlamsa_b200.default_mutations() if c in erlamsa_b200.supported_mutations()}
    else:
        muts = {c: 1 for c in muts}
    data, off = make_corpus_device(torch, kind, n_cases, size, dev, 0xE21A0003 + rank)
    data_bytes = n_cases * size
    out_cap = data_bytes + data_bytes // 12 + 512 * n_cases + (256 << 20)   # output slots (input + 1/16 slack) + overflow region
    base_opts = {"mutations": muts, "patterns": pats, "seed": (1, 2, 3), "rng": args.rng, "scratch_bytes": 512 << 20}
    if workload == "c2":   # repeat mutators compounded by nd/bu rounds: cap a case at 128 KiB = 32 x its seed (flagged, not dropped)
        base_opts.update({"scratch_bytes": 8 << 30, "max_case_out": 128 << 10})
        out_cap += 4 << 30
    if workload == "c4":   # re-serialised documents and their literals live in scratch; pump / repeat may double a document
        base_opts.update({"scratch_bytes": 16 << 30, "max_case_out": 4 << 20})
        out_cap += 8 << 30
    if workload == "c5":   # fuse splices are at most twice a block
        base_opts.update({"scratch_bytes": 4 << 30, "max_case_out": 1 << 20})
        out_cap += 2 << 30
    d_out = torch.empty(out_cap, dtype=torch.uint8, device=dev)
    d_out_off = torch.empty(n_cases + 1, dtype=torch.int64, device=dev)
    d_out_len = torch.empty(n_cases, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream()
    # config C5: the one exchange step of the path -- every GPU samples donor windows from its shard, the pools are all-gathered
    donors = None
    coll_ms, coll_bytes = [], 0
    if workload == "c5":
        from erlamsa_b200.donors import DEFAULT_DONORS, DEFAULT_STRIDE, all_gather_pool
        d_pool = torch.zeros((DEFAULT_DONORS, DEFAULT_STRIDE), dtype=torch.uint8, device=dev)
        d_len = torch.zeros((DEFAULT_DONORS,), dtype=torch.int32, device=dev)
        donors = (d_pool, d_len)
        coll_bytes = (world - 1) * (d_pool.numel() + 4 * d_len.numel())     # bytes this GPU receives over NVLink per step

    def step(i, timed=False):
        o = dict(base_opts)
        o["first_case"] = 1 + (rank + world * i) * n_cases       # every rank / step gets its own window of case ids
        if donors is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            eng.sample_donors(data.data_ptr(), off.data_ptr(), n_cases, donors[0].shape[0], donors[0].shape[1], donors[0].data_ptr(), donors[1].data_ptr(), stream.cuda_stream)
            e0.record(stream)
            gp, gl = all_gather_pool(donors[0], donors[1])
            e1.record(stream)
            o["donor_pool"] = (gp.data_ptr(), gl.data_ptr(), gp.shape[0], gp.shape[1])
            st = eng.fuzz_batch_device(o, data.data_ptr(), off.data_ptr(), n_cases, data_bytes, n_cases, d_out.data_ptr(), out_cap,
                                       d_out_off.data_ptr(), d_out_len.data_ptr(), 0, stream.cuda_stream)
            if timed:
                coll_ms.append(e0.elapsed_time(e1))
            return st
        return eng.fuzz_batch_device(o, data.data_ptr(), off.data_ptr(), n_cases, data_bytes, n_cases, d_out.data_ptr(), out_cap,
                                     d_out_off.data_ptr(), d_out_len.data_ptr(), 0, stream.cuda_stream)

    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    wall0 = time.time()
    ev0.record(stream)
    apply_ms, decide_ms, scan_ms, launches, bytes_out = [], [], [], 0, 0
    flagged = {"unsupported": 0, "died": 0, "overflow": 0}
    for i in range(steps):
        st = step(warmup + i, timed=True)
        apply_ms.append(st.ms_apply); decide_ms.append(st.ms_decide); scan_ms.append(st.ms_scan)
        launches += st.kernels_launched; bytes_out += st.bytes_out
        flagged["unsupported"] += st.n_unsupported; flagged["died"] += st.n_died; flagged["overflow"] += st.n_overflow
    ev1.record(stream)
    torch.cuda.synchronize()
    wall1 = time.time()
    if os.environ.get("EB200_BENCH_VERBOSE"):
        print("per-step kernel ms:", " ".join("%.3f" % x for x in decide_ms), file=sys.stderr)
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop(wall0, wall1) if (sampler is not None and rank == 0) else None
    nflag = flagged["unsupported"] + flagged["overflow"]
    if world > 1:
        t = torch.tensor([ms, float(nflag)], device=dev, dtype=torch.float64)
        dist.all_reduce(t[:1], op=dist.ReduceOp.MAX)
        dist.all_reduce(t[1:], op=dist.ReduceOp.SUM)
        ms = float(t[0].item()); nflag = int(t[1].item())
        dist.barrier()
    out_len_sum = int(d_out_len.sum().item())
    if dump_dir and rank == 0:
        dump_outputs(torch, dump_dir, 1 + (rank + world * (warmup + steps - 1)) * n_cases, size, d_out, d_out_off, d_out_len, st)

    # ---- parity sample: case ids of the LAST timed step, re-run through the oracle on the host (checker only, after the clock)
    parity = None
    if rank == 0 and not args.no_parity and workload != "c5":
        import numpy as np
        import oracle_lib
        r = np.random.Generator(np.random.PCG64(12345))
        n_s = min(args.parity_cases, n_cases)
        ks = sorted(int(k) for k in r.choice(n_cases, size=n_s, replace=False))
        last_first = 1 + (rank + world * (warmup + steps - 1)) * n_cases
        offs = d_out_off[ks].cpu().tolist(); lens = d_out_len[ks].cpu().tolist()
        oo = oracle_lib.make_opts(seed=(1, 2, 3), mutations=muts, patterns=pats, max_case_out=base_opts.get("max_case_out", 0))
        bad, checked, skipped = 0, 0, 0
        for k, o_, l_ in zip(ks, offs, lens):
            blob = bytes(data[k * size:(k + 1) * size].cpu().numpy().tobytes())
            # case I reads blob (I-1) mod n_blobs: hand the oracle a one-blob corpus and the same case number
            want, wm = oracle_lib.fuzzer([blob], opts=oo, n_cases=1, first_case=last_first + k)
            got = bytes(d_out[o_:o_ + l_].cpu().numpy().tobytes())
            if wm[0].status != 0:
                skipped += 1
                continue
            checked += 1
            if got != want[0]:
                # a case the engine flagged comes back unchanged: not a mismatch, but not a mutated case either
                if got == blob and (flagged["unsupported"] or flagged["overflow"]):
                    skipped += 1; checked -= 1
                else:
                    bad += 1
        parity = {"checked": checked, "mismatches": bad, "skipped_flagged_or_capped": skipped, "against": "oracle (C++ restatement, pinned to the reference's own source by tests/golden/reference_vectors.json)"}

    # ---- e2e: the C-ABI call with HOST buffers (pinned), H2D + D2H inside the timed region
    e2e = None
    e2e_error = None
    if want_e2e and not args.no_e2e:
        try:
            e2e_cases = min(n_cases, args.e2e_cases) if args.e2e_cases else n_cases
            # host buffers: pinned and on the GPU's NUMA node (eb200_host_alloc), as the NIF's staging rings are. The whole config's step
            # needs ~14 GB of pinned memory per rank on C3; if the box cannot pin that much (8 ranks at once), halve the step and say so.
            p_in = p_out = None
            while True:
                in_bytes = e2e_cases * size + 64
                out_bytes = e2e_cases * size + e2e_cases * size // 12 + 512 * e2e_cases + ((3 << 30) if workload == "c2" else (128 << 20))
                p_in = N.lib().eb200_host_alloc(eng._ctx, in_bytes)
                p_out = N.lib().eb200_host_alloc(eng._ctx, out_bytes) if p_in else None
                if p_in and p_out:
                    break
                if p_in:
                    N.lib().eb200_host_free(eng._ctx, p_in)
                assert e2e_cases > 8192, "pinned host allocation failed"
                e2e_cases //= 2
            if world > 1:      # every rank runs the same e2e step size
                t = torch.tensor([e2e_cases], device=dev, dtype=torch.int64); dist.all_reduce(t, op=dist.ReduceOp.MIN); e2e_cases = int(t.item())
            hb = torch.frombuffer((C.c_uint8 * in_bytes).from_address(p_in), dtype=torch.uint8)
            hb[: e2e_cases * size].copy_(data[: e2e_cases * size])
            hoff = (C.c_uint64 * (e2e_cases + 1))(*[i * size for i in range(e2e_cases + 1)])
            ho_off = (C.c_uint64 * (e2e_cases + 1))(); ho_len = (C.c_uint64 * e2e_cases)()
            st2 = N.Stats()
            o = erlamsa_b200.make_opts(base_opts)
            times = []
            for i in range(args.e2e_steps + 1):
                o.first_case = 1 + (10_000 + rank + world * i) * n_cases
                t0 = time.perf_counter()
                rc = N.lib().eb200_fuzz_batch_into(eng._ctx, C.byref(o), p_in, C.cast(hoff, C.c_void_p), e2e_cases, e2e_cases,
                                                   p_out, out_bytes, C.cast(ho_off, C.c_void_p), C.cast(ho_len, C.c_void_p), None, C.byref(st2))
                t1 = time.perf_counter()
                assert rc == 0, rc
                if i > 0:
                    times.append(t1 - t0)
            dt = max(times)
            if world > 1:
                t = torch.tensor([dt], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); dt = float(t.item())
            h2d_b, d2h_b = e2e_cases * size + 8 * (e2e_cases + 1), int(sum(ho_len)) + 16 * e2e_cases + 8
            e2e = {"value": e2e_cases * world / dt, "unit": "cases/s", "h2d_bytes_per_step": h2d_b, "d2h_bytes_per_step": d2h_b,
                   "cases_per_step": e2e_cases * world, "pcie_gb_per_s_each_way": [h2d_b / dt / 1e9, d2h_b / dt / 1e9], "numa_node_of_gpu": N.lib().eb200_numa_node(eng._ctx),
                   "note": "eb200_fuzz_batch_into: pinned NUMA-local host corpus -> H2D (chunks, 2 uploads ahead) -> eb_case_kernel -> D2H of outputs, offsets and lengths"}
            del hb
            N.lib().eb200_host_free(eng._ctx, p_in); N.lib().eb200_host_free(eng._ctx, p_out)
        except Exception as e:      # the device-timed line above stands on its own: report, do not lose it
            e2e, e2e_error = None, repr(e)[:300]

    # ---- opt-in (--async-depth D): the same steps through eb200_submit_device / eb200_collect with D batches in flight, each with its
    # own output arena. Lanes run on their own streams, so this is timed by the host clock between two device synchronisations and
    # reported beside the device-timed synchronous number, never instead of it.
    async_line = None
    if args.async_depth > 0 and workload != "c5":
        try:
            D = args.async_depth
            arenas = [(d_out, d_out_off, d_out_len)] + [(torch.empty(out_cap, dtype=torch.uint8, device=dev), torch.empty(n_cases + 1, dtype=torch.int64, device=dev),
                                                           torch.empty(n_cases, dtype=torch.int64, device=dev)) for _ in range(D - 1)]

            def submit(i):
                o = dict(base_opts); o["first_case"] = 1 + (20_000 + rank + world * i) * n_cases
                a = arenas[i % D]
                return eng.submit_device(o, data.data_ptr(), off.data_ptr(), n_cases, data_bytes, n_cases, a[0].data_ptr(), out_cap, a[1].data_ptr(), a[2].data_ptr())
            for i in range(max(warmup, D)):
                eng.collect(submit(i))
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            q = []
            for i in range(steps):
                if len(q) == D:
                    eng.collect(q.pop(0))
                q.append(submit(100 + i))
            while q:
                eng.collect(q.pop(0))
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if world > 1:
                t = torch.tensor([dt], device=dev, dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX); dt = float(t.item())
            async_line = {"depth": D, "lanes": N.lib().eb200_async_lanes(eng._ctx), "ms_per_step": dt / steps * 1e3, "value": n_cases * world * steps / dt, "unit": "cases/s",
                          "timing": "host clock between device synchronisations, max over ranks; the synchronous call's device-timed ms_per_step is this line's own"}
            del arenas
        except Exception as e:      # an auxiliary measurement must never cost the line
            async_line = {"error": repr(e)[:200]}
    del d_out, data
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    total_cases = n_cases * world * steps
    peak, peak_src = peak_hbm()
    # algorithmic bytes of the dominant kernel per launch: len_in + len_out + 16 per case (DESIGN.md, SURVEY.md 8d)
    alg_bytes = data_bytes + out_len_sum + 16 * n_cases
    avg_apply = sum(apply_ms) / len(apply_ms)
    fused = avg_apply == 0.0          # single-pass mode: one kernel decides and moves the bytes
    dom_ms = sum(decide_ms) / len(decide_ms) if fused else avg_apply
    dom_kernel = "eb_case_kernel (single pass: decide + copy)" if fused else "eb_apply_kernel"
    achieved = alg_bytes / (dom_ms * 1e-3) / 1e9
    line = {
        "metric": "mutated testcases/sec", "value": (total_cases - nflag) / (ms * 1e-3), "unit": "cases/s",
        "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": config_of(workload, n_cases, size, args.rng),
        "bytes_per_step": {"in": data_bytes, "out": out_len_sum},
        "gb_per_s_mutated": (data_bytes + out_len_sum) * world * steps / (ms * 1e-3) / 1e9,
        "roofline": {"bound": "hbm", "kernel": dom_kernel, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": ncu_traffic(workload, fused) if not n_override else None,
                     "traffic_source": "ncu --set full capture, profiles/" + TRAFFIC_PROFILE[bool(fused)],
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes, "ms_per_launch": dom_ms},
        "kernel_ms": {"decide": sum(decide_ms) / len(decide_ms), "scan": sum(scan_ms) / len(scan_ms), "apply": avg_apply},
        "gpu_launches": launches, "clocks": clocks, "e2e": e2e if e2e_error is None else {"error": e2e_error},
        # cases the engine did not mutate (paths without a device implementation, per-case output cap: output = input, reported
        # per case in eb200_meta.status) are NOT counted in `value`; worker crashes the reference has too (died) are
        "flagged_cases": dict(flagged, of=n_cases * steps, note="rank 0; unsupported + overflow are subtracted from value"),
    }
    if parity is not None:
        line["parity_sample"] = parity
    if async_line is not None:
        line["async_pair"] = async_line
    if workload == "c5":
        cm = sum(coll_ms) / max(len(coll_ms), 1)
        line["collective"] = {"op": "all_gather (NCCL) of the donor pool + lengths", "ms_per_step": cm, "share_of_step": cm / (ms / steps),
                              "nvlink_bytes_received_per_gpu_per_step": coll_bytes, "donors_per_gpu": 4096, "window_bytes": 2048}
    return line


def run_ours(args):
    import torch
    import torch.distributed as dist
    import erlamsa_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    eng = erlamsa_b200.Engine(local)
    sampler = ClockSampler(local)
    if rank == 0 and not os.environ.get("EB200_BENCH_NO_SAMPLER"):
        sampler.start()
        time.sleep(0.5)
    try:
        line = measure(torch, dist, eng, args, args.workload, args.steps, args.warmup, rank, world, local, n_override=args.cases, sampler=sampler,
                       dump_dir=args.dump_outputs)
    finally:
        sampler.close()
    if rank == 0 and not args.no_cpu:
        n_cases, size, kind, muts, pats, desc = WORKLOADS[args.workload]
        muts = {c: 1 for c in muts} if muts is not None else {c: p for c, p in erlamsa_b200.default_mutations() if c in erlamsa_b200.supported_mutations()}
        line["cpu_baseline"] = cpu_baseline(args, size, kind, muts, pats, threads=1, budget_s=12.0)
    # the other configs, made driver-visible: short runs, value net of flagged cases, the all-threads CPU port beside each
    if args.workload == "c3" and not args.no_extra and not args.cases:
        extra = {}
        for wl, n_x in (("c2", 0), ("c4", 0)):
            try:
                x = measure(torch, dist, eng, args, wl, 2, 3, rank, world, local, n_override=n_x, want_e2e=False)
            except Exception as e:      # a short extra run must never cost the headline line
                if rank == 0:
                    extra[wl] = {"error": repr(e)[:300]}
                continue
            if rank == 0:
                n_cases, size, kind, muts, pats, desc = WORKLOADS[wl]
                muts = {c: 1 for c in muts} if muts is not None else {c: p for c, p in erlamsa_b200.default_mutations() if c in erlamsa_b200.supported_mutations()}
                cb = cpu_baseline(args, size, kind, muts, pats, threads=os.cpu_count() or 1, budget_s=6.0)
                extra[wl] = {"workload": x["config"]["workload"], "value": x["value"], "unit": "cases/s", "ms_per_step": x["ms_per_step"], "steps": 2, "warmup": 3,
                             "gb_per_s_mutated": x["gb_per_s_mutated"], "hbm_frac": x["roofline"]["frac"], "flagged_cases": x["flagged_cases"],
                             "parity_sample": x.get("parity_sample"), "cpu_all_threads": cb, "ratio_vs_cpu_all_threads": x["value"] / cb["value"]}
        if rank == 0:
            line["extra_workloads"] = extra
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def cpu_corpus(kind, n, size, seed):
    import corpus
    if kind == "text":
        r = corpus.rng(seed)
        return [corpus.structured_text(r, size).ljust(size, b" ")[:size] for _ in range(n)]
    return corpus.uniform_corpus(seed, n, size, kind)


def cpu_run(blobs, muts, pats, n_cases, first_case, threads):
    """oracle (CPU restatement of the reference path) over n_cases cases, split across host threads"""
    import oracle_lib
    opts = oracle_lib.make_opts(seed=(1, 2, 3), mutations=muts, patterns=pats)
    oracle_lib.lib()
    per = (n_cases + threads - 1) // threads
    res = [0] * threads

    def work(t):
        lo = t * per
        cnt = max(0, min(per, n_cases - lo))
        if cnt:
            res[t] = oracle_lib.fuzzer_total_bytes(blobs, opts, cnt, first_case + lo)   # the C++ work only, no copies into Python

    th = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
    t0 = time.perf_counter()
    for t in th:
        t.start()
    for t in th:
        t.join()
    return time.perf_counter() - t0, sum(res)


def cpu_baseline(args, size, kind, muts, pats, threads, budget_s):
    blobs = cpu_corpus(kind, 64, size, 0xE21A0003)
    ncal = 64 * threads if threads == 1 else 4 * threads                   # calibration
    dt, _ = cpu_run(blobs, muts, pats, ncal, 1, threads)
    rate = ncal / dt
    n = max(ncal, int(rate * budget_s))
    dt, _ = cpu_run(blobs, muts, pats, n, 1000, threads)
    return {"value": n / dt, "unit": "cases/s", "cores": threads, "kind": "port",
            "sample": "%d cases of the same workload (64 distinct %d-byte seeds reused), oracle C++ restatement, %d thread(s), %.1f s"
                      % (n, size, threads, dt)}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path. The reference is Erlang and OTP is not in
    this image (DESIGN.md), so this arm times the oracle port with all host threads on a bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    n_cases, size, kind, muts, pats, desc = WORKLOADS[args.workload]
    if muts is None:
        import erlamsa_b200
        muts = {c: p for c, p in erlamsa_b200.default_mutations() if c in erlamsa_b200.supported_mutations()}
    else:
        muts = {c: 1 for c in muts}
    threads = os.cpu_count() or 1
    blobs = cpu_corpus(kind, 64, size, 0xE21A0003)
    # calibrate in two rounds so that thread start-up does not dominate the estimate, then give every step ~3 s of wall time
    dt, _ = cpu_run(blobs, muts, pats, 32 * threads, 1, threads)
    rate = 32 * threads / dt
    dt, _ = cpu_run(blobs, muts, pats, max(32 * threads, int(rate * 1.0)), 1, threads)
    rate = max(32 * threads, int(rate * 1.0)) / dt
    per_step = max(threads, int(rate * 3.0))
    for i in range(args.warmup):
        cpu_run(blobs, muts, pats, max(threads, per_step // 8), 1 + i * per_step, threads)
    t_total = 0.0
    for i in range(args.steps):
        dt, _ = cpu_run(blobs, muts, pats, per_step, 1 + (args.warmup + i) * per_step, threads)
        t_total += dt
    v = per_step * args.steps / t_total
    sample = "%d cases/step of the same workload (64 distinct %d-byte seeds reused), %d host threads" % (per_step, size, threads)
    print(json.dumps({
        "impl": "reference", "metric": "mutated testcases/sec", "value": v, "unit": "cases/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t_total / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic", "config": config_of(args.workload, args.cases or n_cases, size, args.rng), "sample": sample,
        "cpu_baseline": {"value": v, "unit": "cases/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "cases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--cases", type=int, default=0, help="override cases per GPU per step")
    ap.add_argument("--rng", default="as183", choices=["as183", "philox"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the short C2 / C4 runs appended to the default C3 line")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--parity-cases", type=int, default=256)
    ap.add_argument("--e2e-cases", type=int, default=0, help="cases per e2e step (0 = the whole config)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--async-depth", type=int, default=0, help="also time the steps through eb200_submit_device / eb200_collect with this many batches in flight (0 = off)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (lengths, a fixed sample of output bytes, counters) as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
