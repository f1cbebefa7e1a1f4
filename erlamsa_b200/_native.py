"""ctypes binding of the C ABI in include/erlamsa_b200.h (liberlamsa_b200.so, built in-tree).

The library is the product; this module only loads it. There is no Python or CPU fallback:
if the shared object is missing or no CUDA device is present, calls raise.
"""
import ctypes as C
import os
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
LIB_PATH = os.environ.get("EB200_LIB") or os.path.join(PKG_DIR, "liberlamsa_b200.so")   # EB200_LIB: A/B builds of the same engine
SRC = os.path.join(PKG_DIR, "csrc", "eb_engine.cu")
SRC_WIDE = os.path.join(PKG_DIR, "csrc", "eb_wide.cu")   # the general kernel once more, for 512 threads / 128 registers
SRC_ASYNC = os.path.join(PKG_DIR, "csrc", "eb_async.cpp")   # submit / collect lanes (host code only)

N_MUTATORS = 41
N_PATTERNS = 10

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]


class Opts(C.Structure):
    _fields_ = [("seed", C.c_int64 * 3), ("blockscale", C.c_double),
                ("muta_pri", C.c_int32 * N_MUTATORS), ("pat_pri", C.c_int32 * N_PATTERNS),
                ("gen_direct_pri", C.c_int32), ("gen_random_pri", C.c_int32),
                ("ssrf_host", C.c_char * 64), ("ssrf_port", C.c_int32), ("rng_mode", C.c_int32),
                ("first_case", C.c_uint64), ("max_case_out", C.c_uint64), ("scratch_bytes", C.c_uint64),
                ("donor_pool", C.c_void_p), ("donor_len", C.c_void_p), ("n_donors", C.c_uint64), ("donor_stride", C.c_uint32), ("reserved0", C.c_uint32),
                ("gen_file_pri", C.c_int32), ("gen_stdin_pri", C.c_int32), ("gen_jump_pri", C.c_int32), ("jump_on_device", C.c_int32),
                ("case_stream_seed", C.c_int64 * 3), ("case_stream_first", C.c_uint64)]


class Meta(C.Structure):
    _fields_ = [("pattern", C.c_int32), ("generator", C.c_int32), ("n_used", C.c_int32), ("n_failed", C.c_int32),
                ("used", C.c_int32 * 16), ("draws", C.c_uint64), ("status", C.c_int32), ("pad", C.c_int32),
                ("thread_seed", C.c_int64 * 3)]


class Stats(C.Structure):
    _fields_ = [("n_cases", C.c_uint64), ("bytes_in", C.c_uint64), ("bytes_out", C.c_uint64),
                ("n_unsupported", C.c_uint64), ("n_died", C.c_uint64), ("n_overflow", C.c_uint64),
                ("ms_decide", C.c_float), ("ms_scan", C.c_float), ("ms_apply", C.c_float), ("ms_total", C.c_float),
                ("kernels_launched", C.c_uint32), ("pad", C.c_uint32)]


def build(force=False):
    """Compile the CUDA engine for sm_100a into the package directory (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(PKG_DIR, "csrc", f) for f in os.listdir(os.path.join(PKG_DIR, "csrc"))]
    srcs.append(os.path.join(ROOT, "include", "erlamsa_b200.h"))
    if not force and os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(s) for s in srcs):
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    subprocess.check_call([nvcc] + NVCC_FLAGS + [SRC, SRC_WIDE, SRC_ASYNC, "-o", LIB_PATH])
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("liberlamsa_b200.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'`); "
                           "the engine has no CPU fallback")
    L = C.CDLL(LIB_PATH)
    vp, u64p = C.c_void_p, C.POINTER(C.c_uint64)
    L.eb200_default_opts.argtypes = [C.POINTER(Opts)]
    L.eb200_init.argtypes = [C.c_int, C.POINTER(vp)]
    L.eb200_shutdown.argtypes = [vp]
    L.eb200_fuzz_batch.argtypes = [vp, C.POINTER(Opts), vp, u64p, C.c_uint64, C.c_uint64,
                                   C.POINTER(vp), u64p, u64p, C.POINTER(Meta), C.POINTER(Stats)]
    L.eb200_fuzz_batch_device.argtypes = [vp, C.POINTER(Opts), vp, vp, C.c_uint64, C.c_uint64, C.c_uint64,
                                          vp, C.c_uint64, vp, vp, vp, vp, C.POINTER(Stats)]
    L.eb200_fuzz_batch_into.argtypes = [vp, C.POINTER(Opts), vp, vp, C.c_uint64, C.c_uint64,
                                        vp, C.c_uint64, vp, vp, vp, C.POINTER(Stats)]
    L.eb200_submit_device.argtypes = [vp, C.POINTER(Opts), vp, vp, C.c_uint64, C.c_uint64, C.c_uint64,
                                      vp, C.c_uint64, vp, vp, vp, C.POINTER(vp)]
    L.eb200_collect.argtypes = [vp, vp, C.POINTER(Stats)]
    L.eb200_async_lanes.argtypes = [vp]
    L.eb200_debug_parent_draws.argtypes = [C.POINTER(Opts), C.c_uint64, C.c_uint64, C.POINTER(C.c_int64)]
    L.eb200_free.argtypes = [vp]
    L.eb200_host_alloc.argtypes = [vp, C.c_uint64]
    L.eb200_host_alloc.restype = vp
    L.eb200_host_free.argtypes = [vp, vp]
    L.eb200_numa_node.argtypes = [vp]
    L.eb200_sample_donors.argtypes = [vp, vp, vp, C.c_uint64, C.c_uint64, C.c_uint32, vp, vp, vp]
    for f in ("eb200_mutator_code", "eb200_pattern_code", "eb200_strerror", "eb200_version"):
        getattr(L, f).restype = C.c_char_p
    L.eb200_last_cuda_error.restype = C.c_char_p
    L.eb200_last_cuda_error.argtypes = [vp]
    _lib = L
    return L


EXPORTED_SYMBOLS = [
    "eb200_default_opts", "eb200_init", "eb200_shutdown", "eb200_fuzz_batch", "eb200_fuzz_batch_into", "eb200_free",
    "eb200_fuzz_batch_device", "eb200_mutator_code", "eb200_mutator_default_pri", "eb200_mutator_supported",
    "eb200_pattern_code", "eb200_pattern_default_pri", "eb200_pattern_supported",
    "eb200_strerror", "eb200_last_cuda_error", "eb200_version",
    "eb200_submit_device", "eb200_collect", "eb200_async_lanes",
    "eb200_debug_parent_draws", "eb200_sample_donors", "eb200_debug_case_times", "eb200_debug_mutator_times", "eb200_host_alloc", "eb200_host_free", "eb200_numa_node",
]
