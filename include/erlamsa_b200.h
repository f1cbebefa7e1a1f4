/*
 * erlamsa_b200.h -- C ABI of the B200 batched mutation engine.
 *
 * This is the drop-in boundary for ONE path of erlamsa: erlamsa_mutations + erlamsa_rnd
 * applied per test case over a corpus (the per-case loop of erlamsa_main:fuzzer/1).
 * The reference has no FFI today; the entry points below are what a NIF for this path binds
 * (see INTEGRATION.md and erlang/erlamsa_b200_nif.c):
 *
 *   eb200_opts          <- the option map read by erlamsa_main:fuzzer/1
 *                          (reference src/erlamsa_main.erl:127-163: seed, mutations, patterns,
 *                          generators, blockscale, skip) and the ssrf endpoint the mutators read from
 *                          ETS (src/erlamsa_mutations.erl:697-726)
 *   eb200_fuzz_batch    <- the case loop FuzzingLoopFun, src/erlamsa_main.erl:166-243, with
 *                          output => return (src/erlamsa_out.erl:66-77,676): case I of the call is
 *                          seeded with the I-th erlamsa_rnd:gen_predictable_seed() of the parent
 *                          stream (:179) and mutates corpus blob (I-1) mod n_blobs. With one blob
 *                          and n cases this IS erlamsa_main:fuzzer(#{paths=>[direct], input=>Blob,
 *                          n=>N, output=>return}); with n = 1 it is erlamsa_app:fuzz/2
 *                          (src/erlamsa_app.erl:255-263).
 *   eb200_meta          <- the per-case metadata list (-M), src/erlamsa_main.erl:58-70,195
 *
 * Conventions: plain pointers and sizes, no C++ or torch types; every function returns 0 or a
 * negative EB200_ERR_* code, never throws. Inputs are borrowed for the duration of the call.
 * A ctx is bound to one CUDA device; use one ctx per host thread / per GPU.
 */
#ifndef ERLAMSA_B200_H
#define ERLAMSA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EB200_N_MUTATORS 41   /* table order of erlamsa_mutations:mutations/1, src/erlamsa_mutations.erl:1291-1331 */
#define EB200_N_PATTERNS 10   /* table order of erlamsa_patterns:patterns/0, src/erlamsa_patterns.erl:395-404 */

/* error codes */
#define EB200_OK                 0
#define EB200_ERR_CUDA          -1   /* a CUDA runtime call failed (eb200_last_cuda_error has the text) */
#define EB200_ERR_ARG           -2   /* bad argument */
#define EB200_ERR_UNSUPPORTED   -3   /* a selected mutator/pattern has no device implementation yet */
#define EB200_ERR_NOMEM         -4
#define EB200_ERR_SCRATCH       -5   /* scratch / literal / segment arena too small: raise eb200_opts.scratch_bytes */
#define EB200_ERR_NO_DEVICE     -6   /* no CUDA device: the engine has no CPU fallback */

/* eb200_opts.rng_mode */
#define EB200_RNG_AS183   0   /* OTP `random` (AS183), draw-for-draw identical to the reference */
#define EB200_RNG_PHILOX  1   /* Philox4x32-10 keyed (seed, case id) with fixed counter slots (round, who draws, index): same
                                 decision logic, distribution-equivalent, no serial state -- per-byte draws are lane-parallel */

/* eb200_meta.status (per case) */
#define EB200_CASE_OK            0
#define EB200_CASE_UNSUPPORTED   1   /* the case walked into a path with no device implementation (e.g. sk chose
                                        the `ar` pattern as continuation); output = input unchanged */
#define EB200_CASE_DIED          2   /* the reference's worker process would have crashed; output empty */
#define EB200_CASE_OVERFLOW      3   /* out of scratch, output cap or descriptor space; output = input unchanged */
/* Under the jump generator a flagged case (UNSUPPORTED or OVERFLOW) outputs NOTHING: its slot is sized from the block size, not
 * from an input, so "the input unchanged" need not fit it. status / reason say why. Reason 12 (jump only): blockscale < 1/512
 * makes rand_block_size 0 possible, and a zero-size block never ends the file's stream (the reference loops forever). */

typedef struct eb200_ctx eb200_ctx;

typedef struct eb200_opts {
    int64_t  seed[3];                       /* option `seed` {A,B,C} */
    double   blockscale;                    /* option `blockscale` (default 1.0) */
    int32_t  muta_pri[EB200_N_MUTATORS];    /* option `mutations` [{Code,Pri}]: priority per table row, -1 = not selected */
    int32_t  pat_pri[EB200_N_PATTERNS];     /* option `patterns`  [{Code,Pri}]: -1 = not selected */
    /* option `generators`: priorities only. make_generator walks the option list as given and sort_by_priority keeps that order among
     * EQUAL priorities (src/erlamsa_gen.erl:233-236, src/erlamsa_utils.erl:114-117); here equal priorities are resolved as if the list
     * were in the order of erlamsa_gen:generators/0 (random, jump, direct, file, stdin) -- the reference's defaults have no ties. */
    int32_t  gen_direct_pri;                /* direct (500), -1 = not selected */
    int32_t  gen_random_pri;                /* option `generators`: random (1),  -1 = not selected */
    char     ssrf_host[64];                 /* cm_host / cm_host_user; default "localhost" */
    int32_t  ssrf_port;                     /* cm_port; default 51234 */
    int32_t  rng_mode;                      /* EB200_RNG_* */
    uint64_t first_case;                    /* 1-based I of the first case of this batch (option `skip` + 1, or the
                                               shard start when a corpus is split over GPUs) */
    uint64_t max_case_out;                  /* per-case output cap in bytes (0 = default 64 MiB) */
    uint64_t scratch_bytes;                 /* device scratch arena (0 = default: 4 x input bytes + 64 MiB) */
    /* Cross-seed donor pool for `fo` (BASELINE config C5; NOT a reference option). The reference's sed_fuse_old starts out
     * remembering the block it was first given (src/erlamsa_mutations.erl:404-427); with a pool the first remembered block of a
     * case is donor number (31*S1 + 17*S2 + S3) mod n_donors, {S1,S2,S3} = the case's thread seed -- no draw of the case's
     * stream is consumed. DEVICE pointers: n_donors windows of donor_stride bytes each, and their lengths. NULL / 0 = off.
     * eb200_sample_donors fills a pool from a device-resident corpus; multi-GPU callers all-gather the per-GPU pools. */
    const uint8_t*  donor_pool;
    const uint32_t* donor_len;
    uint64_t n_donors;
    uint32_t donor_stride;
    uint32_t reserved0;
    /* option `generators` for paths that are files / stdin (reference src/erlamsa_gen.erl:59-121, :232-236): `file` (1000) makes every
     * case pick its blob with erand(n_blobs) and cuts it lazily into random-size blocks (256..4095 x blockscale); `stdin` (100000) is
     * the same over blob (I-1) mod n_blobs and is only the reference's behaviour for n == 1 (with n > 1 the reference pre-reads stdin
     * in the parent process: EB200_ERR_UNSUPPORTED). -1 = not selected (default). */
    int32_t  gen_file_pri;
    int32_t  gen_stdin_pri;
    /* `jump` (100; src/erlamsa_gen.erl:123-150, kept by make_generator only when there are two or more paths): it takes part in the
     * parent's generator draw exactly as in the reference (rand over the priority sum, :194-199). A run whose draw lands on jump is
     * run on the device when jump_on_device is 1: every case picks two blobs (erand(n_blobs) twice), cuts each into random-size
     * blocks, picks one block of each and outputs the mutation of a random slice of the first ++ a random slice of the second.
     * With jump_on_device 0 (the default) such a run is refused with EB200_ERR_UNSUPPORTED, so that a caller can route it elsewhere. */
    int32_t  gen_jump_pri;
    int32_t  jump_on_device;                /* 1: run the jump generator when the draw lands on it; 0: EB200_ERR_UNSUPPORTED */
    /* Multi-threaded mode of the reference (option `workers` > 1 with a file / network output, run_fuzzing_loop/7, src/erlamsa_main.erl:
     * 254-280): every worker process is re-seeded with its own seed S (the W-th gen_predictable_seed() of the re-seeded parent, or the
     * run's seed with `workers_same_seed`) and draws the thread seed of ITS first case, number A, as the first three draws of that
     * stream, while the mutator table, generator and pattern list made by the parent are shared. One worker = one batch with
     * case_stream_seed = S, case_stream_first = A (> 0 switches it on) and first_case >= A: case I takes the (I - A)-th seed of
     * the stream. 0 = the single-threaded numbering (case I = the I-th seed of the parent stream). */
    int64_t  case_stream_seed[3];
    uint64_t case_stream_first;
} eb200_opts;

typedef struct eb200_meta {
    int32_t  pattern;        /* first pattern chosen (index into the pattern table) */
    int32_t  generator;      /* 0 direct, 1 random, 2 file, 3 stdin, 4 jump */
    int32_t  n_used;         /* successful mutator applications */
    int32_t  n_failed;       /* attempts that left hd(Ll) unchanged */
    int32_t  used[16];       /* first 16 used mutator ids (table index), -1 padded */
    uint64_t draws;          /* RNG draws consumed by the case's worker stream */
    int32_t  status;         /* EB200_CASE_* */
    int32_t  reason;         /* why a case was flagged (DESIGN.md section 6): 1 scratch, 4 block runs, 5 output cap, 8 fuse tables, 11 output arena,
                                12 jump with a zero block size, ... */
    int64_t  thread_seed[3]; /* the case's erlamsa_rnd:gen_predictable_seed() */
} eb200_meta;

typedef struct eb200_stats {
    uint64_t n_cases;
    uint64_t bytes_in;           /* sum of input blob lengths read by the cases */
    uint64_t bytes_out;          /* sum of output lengths */
    uint64_t n_unsupported, n_died, n_overflow;
    float    ms_decide;          /* device time of the decision kernel (CUDA events) */
    float    ms_scan;            /* device time of the output-offset prefix sum */
    float    ms_apply;           /* device time of the copy/apply kernel */
    float    ms_total;           /* device time of the whole batch incl. copies issued by the call */
    uint32_t kernels_launched;   /* kernels of this library launched for the batch */
    uint32_t pad;
} eb200_stats;

/* defaults of the reference (all 41 mutators / 10 patterns at their table priorities, seed {1,2,3}) */
void eb200_default_opts(eb200_opts* o);

int  eb200_init(int device, eb200_ctx** out);
void eb200_shutdown(eb200_ctx* ctx);

/*
 * Whole batch, host buffers in, host buffers out (what the NIF calls).
 *   data/off : packed corpus, blob b = data[off[b] .. off[b+1]);  n_blobs >= 1
 *   n_cases  : number of cases; case k (0-based) has I = first_case + k and reads blob (I-1) mod n_blobs
 *   out_data : *out_data receives a malloc()ed buffer with the outputs (free with eb200_free)
 *   out_off  : caller array of n_cases+1 entries: case k output = (*out_data)[out_off[k] .. out_off[k]+out_len[k]);
 *              out_off[n_cases] = bytes used in the buffer. Case regions are 16-byte aligned and do not overlap, but
 *              they are NOT back to back: in the default single-pass mode each case owns a slot sized from its input
 *              (plus slack; under jump from the block size) and larger results live behind the slots, so always go through
 *              out_off / out_len.
 *   out_len  : caller array of n_cases entries
 *   meta     : optional caller array of n_cases entries
 */
int  eb200_fuzz_batch(eb200_ctx* ctx, const eb200_opts* opts,
                      const uint8_t* data, const uint64_t* off, uint64_t n_blobs, uint64_t n_cases,
                      uint8_t** out_data, uint64_t* out_off, uint64_t* out_len,
                      eb200_meta* meta, eb200_stats* stats);
/* Sample n_donors windows (each at most `stride` bytes) from a DEVICE-resident packed corpus into d_pool [n_donors * stride]
 * and d_len [n_donors]: window d comes from blob floor(d * n_blobs / n_donors), starts at (d * 2654435761 mod 2^32) mod
 * (len - wlen + 1) with wlen = min(len, stride). Asynchronous on `stream`. */
int eb200_sample_donors(eb200_ctx* ctx, const uint8_t* d_data, const uint64_t* d_off, uint64_t n_blobs, uint64_t n_donors, uint32_t stride,
                        uint8_t* d_pool, uint32_t* d_len, void* stream);
/* Pinned host memory on the GPU's NUMA node (first-touched while the calling thread is bound to that node's CPUs): what
 * eb200_fuzz_batch_into needs to overlap its copies at full PCIe rate. The NIF keeps its staging rings here. */
void* eb200_host_alloc(eb200_ctx* ctx, uint64_t bytes);
void  eb200_host_free(eb200_ctx* ctx, void* p);
int   eb200_numa_node(eb200_ctx* ctx);    /* NUMA node of the GPU from sysfs, -1 when unknown */
void eb200_free(void* p);
/* profiling aid: with EB200_CASE_TIMES=1 in the environment at eb200_init, microseconds the general per-case program spent on
 * each case of the last launch (0 for cases decided by the front warps). Returns the number of entries copied. */
uint64_t eb200_debug_case_times(eb200_ctx* ctx, uint32_t* out, uint64_t n);
/* ... and per mutator (table order): out[2*i] = nanoseconds spent inside mutator i, out[2*i+1] = calls; then five (ns, steps) pairs for the
 * phases of the fuse search; out holds 98 entries */
int eb200_debug_mutator_times(eb200_ctx* ctx, uint64_t* out);

/* Same as eb200_fuzz_batch, but the outputs are written into a caller buffer (e.g. a resource binary or pinned
 * staging memory owned by the NIF); EB200_ERR_NOMEM when out_capacity is too small. Size it as
 * sum(input of the cases) * 17/16 + 512 * n_cases + room for the cases that outgrow their slot. */
int  eb200_fuzz_batch_into(eb200_ctx* ctx, const eb200_opts* opts,
                           const uint8_t* data, const uint64_t* off, uint64_t n_blobs, uint64_t n_cases,
                           uint8_t* out_buf, uint64_t out_capacity, uint64_t* out_off, uint64_t* out_len,
                           eb200_meta* meta, eb200_stats* stats);

/*
 * Same batch with the corpus already resident in device memory and outputs left in device memory
 * (the steady-state path: corpora stay in HBM between rounds). All d_* pointers are device pointers.
 *   d_data must be 16-byte aligned and readable up to the next 16-byte boundary past its end.
 *   d_out / out_capacity : output arena; case k's bytes start at d_out + d_out_off[k] (16-byte aligned)
 *   d_out_off (n_cases+1), d_out_len (n_cases), d_meta (n_cases, optional)
 *   stream : a cudaStream_t cast to void* (NULL = default stream). The call enqueues all work on that
 *            stream and returns after a stream synchronise (arena overflow is reported synchronously).
 */
int  eb200_fuzz_batch_device(eb200_ctx* ctx, const eb200_opts* opts,
                             const uint8_t* d_data, const uint64_t* d_off, uint64_t n_blobs, uint64_t data_bytes,
                             uint64_t n_cases,
                             uint8_t* d_out, uint64_t out_capacity, uint64_t* d_out_off, uint64_t* d_out_len,
                             eb200_meta* d_meta, void* stream, eb200_stats* stats);

/*
 * Asynchronous pair for the device path (the submit / collect shape sketched in SURVEY.md 8b). eb200_submit_device takes the
 * arguments of eb200_fuzz_batch_device (minus stream and stats), copies the options, queues the batch and returns at once with a
 * ticket; eb200_collect blocks until that batch is complete, fills `stats` and returns the batch's own result code (what the
 * synchronous call would have returned). A context runs submitted batches on EB200_ASYNC_LANES (default 2, at most 4) lanes --
 * each lane has its own arenas, its own CUDA stream and a host thread -- so while one batch's host side reads its counters back
 * the next batch's kernel is already running: the stream synchronisations of the synchronous call no longer idle the GPU.
 *   - batches in flight must not overlap in d_out / d_out_off / d_out_len / d_meta, and a batch must not read what another
 *     batch in flight writes: lanes are independent streams, there is no ordering between tickets;
 *   - every buffer of a batch stays valid until its ticket is collected; each ticket is collected exactly once
 *     (EB200_ERR_ARG for a foreign or already collected ticket); eb200_shutdown waits for batches still queued;
 *   - results are bit-identical to eb200_fuzz_batch_device (the lanes call it); submit / collect of one context may be called
 *     from any host thread.
 */
typedef struct eb200_ticket eb200_ticket;
int  eb200_submit_device(eb200_ctx* ctx, const eb200_opts* opts,
                         const uint8_t* d_data, const uint64_t* d_off, uint64_t n_blobs, uint64_t data_bytes,
                         uint64_t n_cases,
                         uint8_t* d_out, uint64_t out_capacity, uint64_t* d_out_off, uint64_t* d_out_len,
                         eb200_meta* d_meta, eb200_ticket** ticket);
int  eb200_collect(eb200_ctx* ctx, eb200_ticket* ticket, eb200_stats* stats);
int  eb200_async_lanes(eb200_ctx* ctx);        /* lanes created so far (0 before the first submit) */

/* Host-only aid (no CUDA call, works without a GPU): the parent-process part of erlamsa_main:fuzzer/1 that every batch entry point
 * restates before it launches anything (src/erlamsa_main.erl:127-163; SURVEY.md appendix A, T0..T3). out[0] = generator chosen
 * (0 direct, 1 random, 2 file, 3 stdin, 4 jump), out[1] = snand mask kind, out[2] = table rows, out[3] = patterns, out[4..6] = the
 * parent's AS183 state after its draws (the first case's thread seed is the next three erand(99999)). Returns what the batch call
 * would return for these options (EB200_ERR_UNSUPPORTED when the draw lands on jump and jump_on_device is 0). */
int eb200_debug_parent_draws(const eb200_opts* opts, uint64_t n_blobs, uint64_t n_cases, int64_t out[8]);

/* name surface of the reference (-m / -p codes, src/erlamsa_cmdparse.erl:233-257) */
const char* eb200_mutator_code(int idx);       /* "sgm", "js", "uw", ... "nil"; NULL when out of range */
int         eb200_mutator_default_pri(int idx);
int         eb200_mutator_supported(int idx);  /* 1 when the mutator has a device implementation */
const char* eb200_pattern_code(int idx);       /* "od", "nd", "bu", "sk", "sz", "cs", "ar", "cp", "co", "nu" */
int         eb200_pattern_default_pri(int idx);
int         eb200_pattern_supported(int idx);

const char* eb200_strerror(int code);
const char* eb200_last_cuda_error(eb200_ctx* ctx);
const char* eb200_version(void);

#ifdef __cplusplus
}
#endif
#endif /* ERLAMSA_B200_H */
