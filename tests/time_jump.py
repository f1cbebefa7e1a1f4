"""Device time of the jump generator next to the file generator on the same corpus (not a test; run on the GPU box).
usage: python tests/time_jump.py [n_cases] [n_files]

Corpus: n_files (default 1024) files of 64 KiB - 1 MiB, resident on the device; n_cases (default 100 000) cases per batch, LIGHT
mutators under od / nd / bu, AS183. Each generator runs one warm-up batch and three timed ones through eb200_fuzz_batch_device;
the line gives the median kernel time (ms_decide: the case kernel, follow-up launches included), the whole call's device time,
cases/s over the latter, kernel launches per batch and the case status counts. Under `file` every case's output is about one whole
file (input-sized slots), under `jump` about one block."""
import collections
import ctypes as C
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import numpy as np  # noqa: E402

import corpus  # noqa: E402
import erlamsa_b200  # noqa: E402
from erlamsa_b200 import _native as N  # noqa: E402

LIGHT = {c: 1 for c in ("bd", "bei", "bed", "bf", "bi", "ber", "br", "sd", "num", "ld", "lr2", "ls", "uw", "ui", "sr", "lp")}


def main():
    import torch
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 100000
    n_files = int(sys.argv[2]) if len(sys.argv) > 2 else 1024
    dev = torch.device("cuda:0")
    r = corpus.rng(0x71A3)
    sizes = r.integers(64 << 10, (1 << 20) + 1, size=n_files)
    off = np.zeros(n_files + 1, dtype=np.int64)
    off[1:] = np.cumsum(sizes)
    total = int(off[-1])
    d_data = torch.randint(0, 256, (total + 64,), dtype=torch.uint8, device=dev)
    d_data[::61] = 0x34                                      # digits for num
    d_off = torch.from_numpy(off).to(dev)
    print("device %s, corpus %d files, %.1f MiB, %d cases per batch, lib %s" % (torch.cuda.get_device_name(0), n_files, total / 2**20, n, N.LIB_PATH))
    eng = erlamsa_b200.Engine(0)
    msz = C.sizeof(N.Meta)
    for gen in ("jump", "file"):
        if gen == "file":
            slot = [((int(sizes[k % n_files]) + min(max(int(sizes[k % n_files]) // 16, 256), 65536)) + 15) // 16 * 16 for k in range(n)]
            cap = sum(slot) * 5 // 4 + (256 << 20)
        else:
            cap = n * 8192 + (256 << 20)
        d_out = torch.empty(cap, dtype=torch.uint8, device=dev)
        d_oo = torch.empty(n + 1, dtype=torch.int64, device=dev)
        d_ol = torch.empty(n, dtype=torch.int64, device=dev)
        d_meta = torch.empty(n * msz, dtype=torch.uint8, device=dev)
        rows = []
        for rep in range(4):
            opts = {"seed": (1, 2, 3), "generators": {gen: 100}, "jump_on_device": True, "mutations": LIGHT,
                    "patterns": {"od": 1, "nd": 1, "bu": 1}, "first_case": 1 + rep * n, "max_case_out": 1 << 22}
            torch.cuda.synchronize()
            st = eng.fuzz_batch_device(opts, d_data.data_ptr(), d_off.data_ptr(), n_files, total, n, d_out.data_ptr(), cap, d_oo.data_ptr(),
                                       d_ol.data_ptr(), d_meta.data_ptr(), torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            if rep:
                rows.append((st.ms_decide, st.ms_total, st.kernels_launched, st.bytes_out))
        mb = d_meta.cpu().numpy().reshape(n, msz)
        so = N.Meta.status.offset
        status = collections.Counter(int(x) for x in mb[:, so:so + 4].copy().view(np.int32).ravel())
        rows.sort()
        dec, tot, kl, bo = rows[len(rows) // 2]
        print("%-4s kernel %8.2f ms  call %8.2f ms  %10.0f cases/s  %d launches  arena %.1f MiB  status %s"
              % (gen, dec, tot, n / (tot / 1e3), kl, bo / 2**20, dict(status)), flush=True)
        del d_out, d_oo, d_ol, d_meta
        torch.cuda.empty_cache()
    eng.close()


if __name__ == "__main__":
    main()
