// erlamsa_b200 -- host side of the engine and the C ABI (include/erlamsa_b200.h).
//
// Per batch the host restates the PARENT-process part of erlamsa_main:fuzzer/1
// (reference src/erlamsa_main.erl:124-163: seed, make_mutator, make_generator, make_pattern --
// a few dozen RNG draws) and hands the result to the device as BatchParams; everything per case
// runs on the GPU: eb_decide_kernel -> prefix sum -> eb_apply_kernel.
// There is deliberately NO CPU fallback: without a CUDA device every entry point fails.
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <algorithm>
#include <cmath>
#include <chrono>
#include <sched.h>
#include <cctype>
#include "../../include/erlamsa_b200.h"
#include "eb_fast.cuh"
#include "eb_apply.cuh"
#include "eb_erlsort.hpp"

// eb_wide.cu: eb_case_kernel<FULL> compiled for 512 threads per CTA (128 registers per thread)
extern "C" int eb200_wide_init(void);
extern "C" void eb200_wide_launch(int grid, int threads, size_t smem, cudaStream_t st, const uint8_t* d_data, const uint64_t* d_off,
                                  const void* bp, const void* ar, void* cases, uint64_t* out_len, uint64_t* sz16, void* meta, const void* fa);

using namespace eb;

static const char* const kMutCodes[EB200_N_MUTATORS] = {
    "sgm", "js", "uw", "ui", "ab", "ad", "tr2", "td", "num", "ts1", "tr", "ts2",
    "bd", "bei", "bed", "bf", "bi", "ber", "br", "sp", "sr", "sd", "snand", "srnd",
    "ld", "lds", "lr2", "lri", "lr", "ls", "lp", "lis", "lrs", "ft", "fn", "fo",
    "len", "b64", "uri", "zip", "nil"};
static const int kMutPri[EB200_N_MUTATORS] = {10, 3, 1, 2, 1, 1, 1, 1, 3, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1,
                                              1, 1, 1, 1, 1, 1, 1, 1, 1, 2, 1, 2, 2, 7, 1, 1, 0};
static const char* const kPatCodes[EB200_N_PATTERNS] = {"od", "nd", "bu", "sk", "sz", "cs", "ar", "cp", "co", "nu"};
static const int kPatPri[EB200_N_PATTERNS] = {1, 2, 1, 2, 2, 1, 1, 1, 0, 0};

struct DevBuf {
    void* p = nullptr; size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct eb200_ctx {
    int device = 0;
    int num_sms = 148;
    std::string last_err;
    DevBuf cases, out_len, sz16, tile_sum, tile_case, slot_off, counters, segs, scratch, temp, data, off, out, out_off, meta;
    int fused = 1;          // single-pass mode (EB200_MODE=twopass selects decide -> scan -> apply)
    unsigned long long flag_counts[3] = {0, 0, 0};   // unsupported / died / overflow of the last batch (device counters)
    cudaEvent_t ev[6];
    bool funny_loaded = false;
    int apply_variant = 0;
    int wide = 0;                 // general kernel at 512 threads / 128 registers: -1 chosen per launch, 0 never, 1 always (EB200_WIDE)
    int threads = CASE_THREADS;   // eb_case_kernel: threads per CTA (EB200_THREADS) ...
    int deciders = 0;             // ... of which this many warps run the general per-case program (EB200_DECIDERS; 0 = chosen per batch),
    int tma_workers = 0;          // workers that copy through shared memory with cp.async.bulk (EB200_TMA_WORKERS; A/B, profiles/variants_r2.txt)
    int front_depth = 32;         // fronts post while fewer than this many jobs are waiting in the ring (EB200_FRONT_DEPTH)
    int fronts = -1;              // this many decide 32 byte-mutator cases at a time, lane per case (EB200_FRONTS; -1 = chosen per batch), the rest are copy/scan workers
    DevBuf case_status, retry_list, case_usec;
    int chunk_mb = 256, h2d_ahead = 2;      // host pipeline: bytes of input per chunk (EB200_CHUNK_MB), uploads queued ahead of the compute (EB200_H2D_AHEAD)
    int numa_node = -1;                    // of the GPU (sysfs), -1 unknown
    bool want_case_times = false; uint64_t case_times_n = 0;
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr, s_comp = nullptr;   // host-path pipeline (created on first use)
    void* async_state = nullptr;           // lanes of eb200_submit_device / eb200_collect (eb_async.cpp), created on first submit
};
// eb_async.cpp: the submit / collect pair is host code over the entry points of this file; it hangs its lanes on the context here
extern "C" void eb200_async_teardown(void* state);

// apply-kernel configurations (words per thread, loads in flight per thread, min CTAs/SM); index 0 ships,
// the others are kept for A/B measurements (env EB200_APPLY_VARIANT)
struct ApplyVariant {
    uint32_t tile; const char* name;
    void (*launch)(unsigned, cudaStream_t, const CaseOut*, const Seg*, const uint64_t*, const uint32_t*, uint64_t, uint8_t*, uint64_t);
};
template <int W, int B, int M>
static void launch_apply(unsigned ctas, cudaStream_t st, const CaseOut* c, const Seg* s, const uint64_t* oo, const uint32_t* tc, uint64_t n, uint8_t* out, uint64_t cap) {
    eb_apply_kernel<W, B, M><<<ctas, APPLY_THREADS, 0, st>>>(c, s, oo, tc, n, out, cap);
}
#define AV(W, B, M) {APPLY_THREADS * W * 16, #W "w" #B "b" #M "m", launch_apply<W, B, M>}
// measured on C3 (profiles/variants_r1.txt): 16w2b8m 2.20 ms (5969 GB/s) | 32w1b8m 2.35 | 16w1b8m 2.37 | 32w2b6m 2.42 | 16w2b6m 2.45 | 8w2b6m 2.55
static const ApplyVariant apply_variants[] = {AV(16, 2, 8), AV(16, 1, 8), AV(16, 2, 6), AV(32, 2, 8), AV(8, 2, 8), AV(32, 1, 8)};
static const int n_apply_variants = (int)(sizeof(apply_variants) / sizeof(apply_variants[0]));

// does this batch fit the LIGHT flavour?
static bool batch_is_light(const BatchParams& bp) {
    if (getenv("EB200_FORCE_FULL")) return false;
    for (int i = 0; i < bp.n_rows; i++) if (!mut_is_light(bp.row_id[i])) return false;
    for (int i = 0; i < bp.n_pats; i++) { int p = bp.pat_id[i]; if (!(p == P_OD || p == P_ND || p == P_BU || p == P_CO || p == P_NU)) return false; }
    return true;
}
// shared memory of eb_case_kernel: job queue + parent-stream power table + one WarpState per deciding warp
static size_t case_smem(int deciders, int tma_workers = 0) { return case_smem_layout(deciders, nullptr, nullptr, nullptr, nullptr, tma_workers, nullptr); }
// counters block (device, 8 x u64): [0] scratch_used [1] segs_used [2] overflow bits [3] ovf_used [4..6] flagged [7] next case
enum { CNT_SCRATCH = 0, CNT_SEGS = 1, CNT_OVERFLOW = 2, CNT_OVF_USED = 3, CNT_FLAGGED = 4, CNT_NEXT_CASE = 7 };

#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { ctx->last_err = std::string(#call) + ": " + cudaGetErrorString(e_); return EB200_ERR_CUDA; } } while (0)

static int64_t erl_round(double x) { return (int64_t)(x >= 0 ? std::floor(x + 0.5) : -std::floor(-x + 0.5)); }

// funny_unicode/0, reference src/erlamsa_mutations.erl:1052-1078: 17 hand-written byte strings, then the UTF-8
// encodings (encode_point :1036-1049) of a code-point list that a foldl builds back to front.
static void build_funny(std::vector<FunnyEntry>& out) {
    auto put = [&](std::initializer_list<int> l) { FunnyEntry e; e.len = (uint32_t)l.size(); e.bytes = 0; int i = 0; for (int b : l) e.bytes |= (uint32_t)(b & 255) << (8 * i++); out.push_back(e); };
    put({239, 191, 191}); put({240, 144, 128, 128}); put({0xef, 0xbb, 0xbf}); put({0xfe, 0xff}); put({0xff, 0xfe});
    put({0, 0, 0xff, 0xff}); put({0xff, 0xff, 0, 0}); put({43, 47, 118, 56}); put({43, 47, 118, 57}); put({43, 47, 118, 43});
    put({43, 47, 118, 47}); put({247, 100, 76}); put({221, 115, 102, 115}); put({14, 254, 255}); put({251, 238, 40});
    put({251, 238, 40, 255}); put({132, 49, 149, 51});
    struct R { int a, b; };
    const R codes[] = {{0x0009, 0x000d}, {0x008D, 0}, {0x00a0, 0}, {0x1680, 0}, {0x180e, 0}, {0x2000, 0x200a}, {0x2028, 0}, {0x2029, 0},
                       {0x202f, 0}, {0x205f, 0}, {0x3000, 0}, {0x200e, 0x200f}, {0x202a, 0x202e}, {0x200c, 0x200d}, {0x0345, 0}, {0x00b7, 0},
                       {0x02d0, 0x02d1}, {0xff70, 0}, {0x02b0, 0x02b8}, {0xfdd0, 0}, {0x034f, 0}, {0x115f, 0x1160}, {0x2065, 0x2069},
                       {0x3164, 0}, {0xffa0, 0}, {0xe0001, 0}, {0xe0020, 0xe007f}, {0x0e40, 0x0e44}, {0x1f4a9, 0}};
    std::vector<int> pts;
    for (const R& r : codes) {   // each group is prepended, ranges ascending inside the group
        std::vector<int> grp; if (r.b == 0) grp.push_back(r.a); else for (int x = r.a; x <= r.b; x++) grp.push_back(x);
        pts.insert(pts.begin(), grp.begin(), grp.end());
    }
    for (int p : pts) {
        if (p < 0x80) put({p});
        else if (p < 0x800) put({0xc0 | (0x1f & (p >> 6)), (p & 0x3f) | 0x80});
        else if (p < 0x10000) put({0xe0 | (0x0f & (p >> 12)), ((p >> 6) & 0x3f) | 0x80, (p & 0x3f) | 0x80});
        else put({0xf0 | (0x7 & (p >> 18)), ((p >> 12) & 0x3f) | 0x80, ((p >> 6) & 0x3f) | 0x80, (p & 0x3f) | 0x80});
    }
}

// choose_pri/2, reference src/erlamsa_utils.erl:155-160
static int choose_pri(const std::vector<std::pair<int, int>>& sorted, int64_t n) {
    for (auto& p : sorted) { if (n == 0 || n < p.first) return p.second; n -= p.first; }
    return -1;
}
static std::vector<std::pair<int, int>> sort_by_priority(const std::vector<std::pair<int, int>>& l) {
    ErlangListSort<std::pair<int, int>> s([](const std::pair<int, int>& a, const std::pair<int, int>& b) { return a.first > b.first; });
    return s(l);
}

// The parent process' draws: T0..T3 of SURVEY.md appendix A.
static int compute_batch_params(const eb200_opts* o, uint64_t n_blobs, uint64_t n_cases, BatchParams& bp) {
    memset(&bp, 0, sizeof(bp));
    Rng par; par.mode = 0; par.key = 0; par.ctr_hi = 0; par.draws = 0;
    par.seed(o->seed[0], o->seed[1], o->seed[2]);                       // erlamsa_main.erl:134
    bp.snand_kind = (int)par.rand_elem_idx(3);                           // mutations/1 :1313
    (void)par.rand_elem_idx(1);                                          //             :1314
    int n = 0;
    for (int i = 0; i < M_COUNT; i++) if (o->muta_pri[i] >= 0) {
        if (!mut_supported(i)) return EB200_ERR_UNSUPPORTED;
        bp.row_id[n] = (uint8_t)i; bp.row_pri[n] = o->muta_pri[i]; n++;
    }
    bp.n_rows = n;
    for (int i = n - 1; i >= 0; i--) { uint64_t s = par.rand(10); bp.row_score[i] = (int)(s < 2 ? 2 : s); }   // mutators_mutator :1390-1395
    std::vector<std::pair<int, int>> gs;                                 // make_generator :233-236, in the order of erlamsa_gen:generators/0
    if (o->gen_random_pri >= 0) gs.push_back({o->gen_random_pri, 1});
    if (o->gen_jump_pri >= 0 && n_blobs > 1) gs.push_back({o->gen_jump_pri, 4});   // `jump when length(Args) > 1` :220
    if (o->gen_direct_pri >= 0) gs.push_back({o->gen_direct_pri, 0});
    if (o->gen_file_pri >= 0) gs.push_back({o->gen_file_pri, 2});
    if (o->gen_stdin_pri >= 0) { if (n_cases != 1 || o->first_case > 1) return EB200_ERR_UNSUPPORTED; gs.push_back({o->gen_stdin_pri, 3}); }
    if (gs.empty()) return EB200_ERR_ARG;
    { auto sg = sort_by_priority(gs); int sum = 0; for (auto& g : sg) sum += g.first;
      int g = choose_pri(sg, (int64_t)par.rand((uint64_t)sum)); if (g < 0) return EB200_ERR_ARG; bp.generator = g;
      if (g == 4 && !o->jump_on_device) return EB200_ERR_UNSUPPORTED; }  // the draw is the reference's; running jump is opt-in
    std::vector<std::pair<int, int>> ps;                                 // make_pattern: foldl prepends -> reversed table
    for (int i = P_COUNT - 1; i >= 0; i--) if (o->pat_pri[i] >= 0) {
        if (o->pat_pri[i] > 0 && !pat_supported(i)) return EB200_ERR_UNSUPPORTED;
        ps.push_back({o->pat_pri[i], i});
    }
    if (ps.empty()) return EB200_ERR_ARG;
    auto sp = sort_by_priority(ps);
    bp.n_pats = (int)sp.size(); bp.pat_sum = 0;
    for (int i = 0; i < bp.n_pats; i++) { bp.pat_pri[i] = sp[i].first; bp.pat_id[i] = sp[i].second; bp.pat_sum += sp[i].first; }
    bp.parent_a1 = par.a1; bp.parent_a2 = par.a2; bp.parent_a3 = par.a3;
    if (o->case_stream_first) {
        // A worker of the multi-threaded mode (erlamsa_main.erl:254-280): case I takes the (I - A)-th seed of the stream seeded with S.
        // The device jumps to case I as x0 * a^(3(I-1)) per AS183 component, so x0 is S's seeded state REWOUND by 3(A-1) steps
        // (each component is a multiplicative group modulo a prime: the inverse multiplier is a^(p-2)).
        if (o->first_case < o->case_stream_first) return EB200_ERR_ARG;
        Rng w; w.mode = 0; w.key = 0; w.ctr_hi = 0; w.draws = 0;
        w.seed(o->case_stream_seed[0], o->case_stream_seed[1], o->case_stream_seed[2]);
        auto powmod = [](uint64_t b, uint64_t e, uint64_t p) { uint64_t r = 1; b %= p; while (e) { if (e & 1) r = r * b % p; b = b * b % p; e >>= 1; } return r; };
        auto rewind = [&](uint64_t x, uint64_t mul, uint64_t p, uint64_t steps) { return x * powmod(powmod(mul, p - 2, p), steps % (p - 1), p) % p; };
        uint64_t steps = 3 * (o->case_stream_first - 1);
        bp.parent_a1 = (int32_t)rewind((uint64_t)w.a1, 171, 30269, steps);
        bp.parent_a2 = (int32_t)rewind((uint64_t)w.a2, 172, 30307, steps);
        bp.parent_a3 = (int32_t)rewind((uint64_t)w.a3, 170, 30323, steps);
    }
    bp.rng_mode = o->rng_mode;
    bp.philox_key = ((uint64_t)(uint32_t)o->seed[0] * 0x9E3779B97F4A7C15ull) ^ ((uint64_t)(uint32_t)o->seed[1] << 32) ^ (uint64_t)(uint32_t)o->seed[2] * 0xD1B54A32D192ED03ull;
    double bs = o->blockscale > 0 ? o->blockscale : 1.0;
    bp.rbs_bound = (int)erl_round(4096.0 * bs); bp.rbs_min = (int)erl_round(256.0 * bs);
    bp.first_case = o->first_case ? o->first_case : 1;
    bp.n_blobs = n_blobs; bp.n_cases = n_cases;
    bp.max_case_out = o->max_case_out ? o->max_case_out : (64ull << 20);
    if (bp.max_case_out > 0x7fffffffull) bp.max_case_out = 0x7fffffffull;
    bp.ssrf_port = o->ssrf_port;
    memcpy(bp.ssrf_host, o->ssrf_host, 64);
    bp.donor_pool = o->donor_pool; bp.donor_len = o->donor_len; bp.n_donors = o->donor_pool && o->donor_len ? o->n_donors : 0; bp.donor_stride = o->donor_stride;
    return EB200_OK;
}

extern "C" {

void eb200_default_opts(eb200_opts* o) {
    memset(o, 0, sizeof(*o));
    o->seed[0] = 1; o->seed[1] = 2; o->seed[2] = 3;
    o->blockscale = 1.0;
    for (int i = 0; i < EB200_N_MUTATORS; i++) o->muta_pri[i] = kMutPri[i];
    for (int i = 0; i < EB200_N_PATTERNS; i++) o->pat_pri[i] = kPatPri[i];
    o->gen_direct_pri = 500; o->gen_random_pri = 1; o->gen_file_pri = -1; o->gen_stdin_pri = -1; o->gen_jump_pri = -1;
    strcpy(o->ssrf_host, "localhost"); o->ssrf_port = 51234;
    o->rng_mode = EB200_RNG_AS183; o->first_case = 1;
}

int eb200_init(int device, eb200_ctx** out) {
    if (!out) return EB200_ERR_ARG;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) return EB200_ERR_NO_DEVICE;
    if (device < 0 || device >= n) return EB200_ERR_ARG;
    eb200_ctx* ctx = new eb200_ctx(); ctx->device = device;
    if (cudaSetDevice(device) != cudaSuccess) { delete ctx; return EB200_ERR_CUDA; }
    cudaDeviceProp prop; if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->num_sms = prop.multiProcessorCount;
    for (auto& e : ctx->ev) cudaEventCreate(&e);
    if (const char* v = getenv("EB200_APPLY_VARIANT")) { int k = atoi(v); if (k >= 0 && k < n_apply_variants) ctx->apply_variant = k; }
    std::vector<FunnyEntry> f; build_funny(f);
    int fn = (int)f.size(); f.resize(192);
    if (cudaMemcpyToSymbol(c_funny, f.data(), sizeof(FunnyEntry) * 192) != cudaSuccess || cudaMemcpyToSymbol(c_funny_n, &fn, sizeof(int)) != cudaSuccess) { delete ctx; return EB200_ERR_CUDA; }
    if (const char* v = getenv("EB200_MODE")) ctx->fused = strcmp(v, "twopass") != 0;
    if (const char* v = getenv("EB200_CHUNK_MB")) { int k = atoi(v); if (k >= 4 && k <= 4096) ctx->chunk_mb = k; }
    if (const char* v = getenv("EB200_H2D_AHEAD")) { int k = atoi(v); if (k >= 1 && k <= 16) ctx->h2d_ahead = k; }
    {   // the GPU's NUMA node: /sys/bus/pci/devices/<domain:bus:dev.fn>/numa_node
        char bdf[32] = {0};
        if (cudaDeviceGetPCIBusId(bdf, sizeof(bdf), device) == cudaSuccess) {
            for (char* c = bdf; *c; c++) *c = (char)tolower(*c);
            std::string path = std::string("/sys/bus/pci/devices/") + bdf + "/numa_node";
            if (FILE* f = fopen(path.c_str(), "r")) { int nn = -1; if (fscanf(f, "%d", &nn) == 1) ctx->numa_node = nn; fclose(f); }
        }
    }
    if (const char* v = getenv("EB200_CASE_TIMES")) ctx->want_case_times = atoi(v) != 0;
    if (const char* v = getenv("EB200_THREADS")) { int k = atoi(v); if (k >= 64 && k <= CASE_THREADS && k % 32 == 0) ctx->threads = k; }
    if (const char* v = getenv("EB200_WIDE")) { int k = atoi(v); if (k >= -1 && k <= 1) ctx->wide = k; }
    if (const char* v = getenv("EB200_DECIDERS")) { int k = atoi(v); if (k >= 0 && k <= 32) ctx->deciders = k; }
    if (const char* v = getenv("EB200_TMA_WORKERS")) { int k = atoi(v); if (k >= 0 && k <= 12) ctx->tma_workers = k; }
    if (const char* v = getenv("EB200_FRONT_DEPTH")) { int k = atoi(v); if (k >= 0 && k <= 200) ctx->front_depth = k; }
    if (const char* v = getenv("EB200_FRONTS")) { int k = atoi(v); if (k >= -1 && k <= MAX_FRONTS) ctx->fronts = k; }
    if (ctx->deciders > ctx->threads / 32) ctx->deciders = ctx->threads / 32;
    if (cudaFuncSetAttribute(eb_case_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448) != cudaSuccess ||
        cudaFuncSetAttribute(eb_case_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448) != cudaSuccess || eb200_wide_init() != 0) { delete ctx; return EB200_ERR_CUDA; }
    *out = ctx; return EB200_OK;
}

void eb200_shutdown(eb200_ctx* ctx) {
    if (!ctx) return;
    if (ctx->async_state) { eb200_async_teardown(ctx->async_state); ctx->async_state = nullptr; }   // joins the lane threads first
    cudaSetDevice(ctx->device);
    for (DevBuf* b : {&ctx->cases, &ctx->out_len, &ctx->sz16, &ctx->tile_sum, &ctx->tile_case, &ctx->slot_off, &ctx->temp, &ctx->counters, &ctx->segs, &ctx->scratch, &ctx->data, &ctx->off, &ctx->out, &ctx->out_off, &ctx->meta, &ctx->case_status, &ctx->retry_list, &ctx->case_usec}) b->release();
    for (auto& e : ctx->ev) cudaEventDestroy(e);
    if (ctx->s_h2d) { cudaStreamDestroy(ctx->s_h2d); cudaStreamDestroy(ctx->s_d2h); cudaStreamDestroy(ctx->s_comp); }
    delete ctx;
}

// How the CTA's warps are split for a batch. The front warps can decide a case on their own when its pattern is `od` and
// the first scheduled mutator is a single-byte mutator or sed_num (eb_fast.cuh); `share` estimates how many cases that is
// from the priorities. Mostly-front batches (C3) want a few general deciders and many copy workers; batches the fronts
// cannot help keep the warps on the general program. Measured on C3 (profiles/variants_r2.txt): fronts 3 / deciders 2
// 2.55 ms, 2/2 2.65, 4/2 2.58, 1/2 3.10; without fronts 5.3 ms (32 deciders, inline copies) .. 9.6 ms (8 deciders).
struct Roles { int fronts, deciders; };
static Roles choose_roles(const eb200_ctx* ctx, const BatchParams& bp, bool fused, uint64_t mean_len, int threads) {
    Roles r;
    double pod = 0, psum = 0, mfast = 0, msum = 0;
    for (int i = 0; i < bp.n_pats; i++) { psum += bp.pat_pri[i]; if (bp.pat_id[i] == P_OD) pod += bp.pat_pri[i]; }
    for (int i = 0; i < bp.n_rows; i++) { double w = bp.row_pri[i] * 5.5; msum += w; if (fast_byte_mut(bp.row_id[i]) || bp.row_id[i] == M_NUM) mfast += w; }
    double share = (psum > 0 && msum > 0 && fused && bp.generator == 0) ? (pod / psum) * (mfast / msum) : 0.0;
    int warps = threads / 32;
    if (share >= 0.5) { r.fronts = 3; r.deciders = 2; }
    else if (share >= 0.02) { r.fronts = 1; r.deciders = warps >= 32 ? 20 : warps / 2; }
    else { r.fronts = 0; r.deciders = warps >= 32 ? 24 : warps == 16 ? 12 : warps / 2; }
    // (measured on C2, 4 KiB blocks copied inline by their decider: 24 deciders 1153 ms per step, 32 deciders 1303 ms -- more warps on
    //  the general program only fight over the instruction-miss path)
    (void)mean_len;
    if (ctx->fronts >= 0) r.fronts = ctx->fronts;
    if (ctx->deciders > 0) r.deciders = ctx->deciders;
    if (r.deciders > warps) r.deciders = warps;
    if (r.fronts + r.deciders >= warps) r.fronts = 0;
    return r;
}
// arenas + launch geometry shared by both modes
struct LaunchPlan { Arenas ar; int grid; Roles roles; int threads; bool wide; };
static int plan_launch(eb200_ctx* ctx, const BatchParams& bp, uint64_t data_bytes, uint64_t n_launch, bool fused, LaunchPlan& lp) {
    lp.threads = ctx->threads; lp.wide = false;
    lp.roles = choose_roles(ctx, bp, fused, bp.n_blobs ? data_bytes / bp.n_blobs : 0, lp.threads);
    // The general program with no front warps: when the launch has only a few cases per deciding warp, its time is the latency
    // of the slowest cases, not throughput -- run it at 512 threads per CTA, where the program has 128 registers per thread and
    // stops spilling to a stack that misses L1 (eb_wide.cu). Measured in profiles/variants_r2.txt section 8.
    if (!batch_is_light(bp) && lp.roles.fronts == 0 && ctx->threads == CASE_THREADS &&
        (ctx->wide == 1 || (ctx->wide < 0 && n_launch < (uint64_t)ctx->num_sms * lp.roles.deciders * 8))) {
        lp.wide = true; lp.threads = 512;
        lp.roles = choose_roles(ctx, bp, fused, bp.n_blobs ? data_bytes / bp.n_blobs : 0, lp.threads);
    }
    const int deciders = lp.roles.deciders;
    unsigned long long* cnt = (unsigned long long*)ctx->counters.p;
    Arenas& ar = lp.ar;
    ar.scratch = (uint8_t*)ctx->scratch.p; ar.scratch_cap = ctx->scratch.cap - 64;
    ar.scratch_used = cnt + CNT_SCRATCH;
    ar.segs = (Seg*)ctx->segs.p; ar.segs_cap = ctx->segs.cap / sizeof(Seg); ar.segs_used = cnt + CNT_SEGS;
    ar.overflow = (uint32_t*)(cnt + CNT_OVERFLOW);
    ar.flagged = cnt + CNT_FLAGGED;
    ar.case_status = (uint8_t*)ctx->case_status.p;
    ar.case_usec = nullptr; ar.mut_ns = nullptr;
    if (ctx->want_case_times) { CK(ctx->case_usec.ensure(bp.n_cases * 4 + 128 + 2 * (M_COUNT + 8) * 8)); ar.case_usec = (uint32_t*)ctx->case_usec.p; ar.mut_ns = (unsigned long long*)((uint8_t*)ctx->case_usec.p + ((bp.n_cases * 4 + 63) & ~63ull)); ctx->case_times_n = bp.n_cases; if (!fused || n_launch == bp.n_cases) CK(cudaMemset(ar.case_usec, 0, bp.n_cases * 4 + 128 + 2 * (M_COUNT + 8) * 8)); }
    uint64_t want_ctas = (n_launch + deciders - 1) / deciders;
    lp.grid = (int)std::min<uint64_t>(want_ctas, (uint64_t)ctx->num_sms);
    if (lp.grid < 1) lp.grid = 1;
    ar.temp = nullptr; ar.temp_per_warp = 0;
    bool needs_temp = false;
    for (int i = 0; i < bp.n_rows; i++) needs_temp |= mut_needs_temp(bp.row_id[i]);
    for (int i = 0; i < bp.n_pats; i++) needs_temp |= bp.pat_pri[i] > 0 && (bp.pat_id[i] == P_SK || bp.pat_id[i] == P_SZ || bp.pat_id[i] == P_CS);
    if (needs_temp) {   // parse tables are proportional to the block being mutated: size the per-warp region from the mean blob
        uint64_t mean = bp.n_blobs ? data_bytes / bp.n_blobs : 0;
        uint64_t per = std::min<uint64_t>(std::max<uint64_t>(64 * mean, 256u << 10), 16u << 20);
        per = (per + 255) & ~255ull;
        uint64_t nw = (uint64_t)ctx->num_sms * deciders;
        while (per > (256u << 10) && per * nw > (48ull << 30)) per >>= 1;
        CK(ctx->temp.ensure(per * nw + 256));
        ar.temp = (uint8_t*)ctx->temp.p; ar.temp_per_warp = per;
    }
    return EB200_OK;
}
static void launch_cases(eb200_ctx* ctx, const BatchParams& bp, const LaunchPlan& lp, cudaStream_t st, const uint8_t* d_data, const uint64_t* d_off,
                         uint64_t* d_out_len, eb200_meta* d_meta, const FusedArgs& fa) {
    size_t sm = case_smem(lp.roles.deciders, fa.tma_workers);
    if (lp.wide) eb200_wide_launch(lp.grid, lp.threads, sm, st, d_data, d_off, &bp, &lp.ar, ctx->cases.p, d_out_len, (uint64_t*)ctx->sz16.p, d_meta, &fa);
    else if (!batch_is_light(bp)) eb_case_kernel<true><<<lp.grid, lp.threads, sm, st>>>(d_data, d_off, bp, lp.ar, (CaseOut*)ctx->cases.p, d_out_len, (uint64_t*)ctx->sz16.p, (MetaDev*)d_meta, fa);
    else eb_case_kernel<false><<<lp.grid, lp.threads, sm, st>>>(d_data, d_off, bp, lp.ar, (CaseOut*)ctx->cases.p, d_out_len, (uint64_t*)ctx->sz16.p, (MetaDev*)d_meta, fa);
}

// Output slot of every case of a jump batch: the result is a slice of one block of each file (blocks are below rbs_bound, a finish/1
// tail below 64 KiB), mostly well under one block, so the slot is what eb_slot_sizes gives an input of rbs_bound bytes; a bigger
// result goes to the overflow region like any other.
static uint64_t jump_slot_bytes(const BatchParams& bp) {
    uint64_t len = (uint64_t)bp.rbs_bound;
    return align16(len + std::min<uint64_t>(std::max<uint64_t>(len / 16, 256), 65536));
}
// scratch a batch wants up front: four times its input for the mutators' rounds, plus (jump) every case's result block
static uint64_t scratch_bytes_for(const BatchParams& bp, const eb200_opts* opts, uint64_t data_bytes) {
    if (opts->scratch_bytes) return opts->scratch_bytes;
    uint64_t jump = bp.generator == 4 ? bp.n_cases * ((uint64_t)bp.rbs_bound + 32) : 0;
    return std::min<uint64_t>(4 * data_bytes + jump + (64ull << 20), 8ull << 30);
}

// decide + scan for a batch resident on the device (two-pass mode). On return *total_out = packed output size.
static int run_decide_scan(eb200_ctx* ctx, const BatchParams& bp, const eb200_opts* opts, const uint8_t* d_data, const uint64_t* d_off,
                           uint64_t data_bytes, uint64_t* d_out_off, uint64_t* d_out_len, eb200_meta* d_meta, cudaStream_t st, uint64_t* total_out, uint32_t* launches) {
    uint64_t n = bp.n_cases;
    CK(ctx->cases.ensure(n * sizeof(CaseOut)));
    CK(ctx->sz16.ensure(n * 8));
    CK(ctx->case_status.ensure(n + 64));
    uint64_t ntiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    CK(ctx->tile_sum.ensure((ntiles + 1) * 8));
    CK(ctx->counters.ensure(64));
    uint64_t seg_cap = ctx->segs.cap / sizeof(Seg);
    if (seg_cap < n * 6 + 1024) { CK(ctx->segs.ensure((n * 6 + 1024) * sizeof(Seg))); seg_cap = ctx->segs.cap / sizeof(Seg); }
    uint64_t scratch_want = scratch_bytes_for(bp, opts, data_bytes);
    if (ctx->scratch.cap < scratch_want) CK(ctx->scratch.ensure(scratch_want));
    // edit scripts published by this mode point into scratch, so an exhausted arena means running the batch again
    for (int attempt = 0;; attempt++) {
        CK(cudaMemsetAsync(ctx->counters.p, 0, 64, st));
        LaunchPlan lp; int rc = plan_launch(ctx, bp, data_bytes, n, false, lp); if (rc) return rc;
        CK(cudaEventRecord(ctx->ev[0], st));
        FusedArgs fa; memset(&fa, 0, sizeof(fa));
        fa.case_counter = (unsigned long long*)ctx->counters.p + CNT_NEXT_CASE; fa.deciders = lp.roles.deciders; fa.fronts = 0;
        launch_cases(ctx, bp, lp, st, d_data, d_off, d_out_len, d_meta, fa);
        CK(cudaGetLastError());
        CK(cudaEventRecord(ctx->ev[1], st));
        (*launches)++;
        uint32_t ovf = 0;
        CK(cudaMemcpyAsync(&ovf, lp.ar.overflow, 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(ctx->flag_counts, lp.ar.flagged, 24, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (!ovf) break;
        if (attempt >= 3) return EB200_ERR_SCRATCH;
        if (ovf & 1) { size_t nw = ctx->scratch.cap * 2; CK(ctx->scratch.ensure(nw)); }
        if (ovf & 2) { size_t nw = ctx->segs.cap * 2; CK(ctx->segs.ensure(nw)); }
    }
    eb_scan_tiles<<<(unsigned)ntiles, SCAN_THREADS, 0, st>>>((const uint64_t*)ctx->sz16.p, n, (uint64_t*)ctx->tile_sum.p);
    eb_scan_tile_offsets<<<1, SCAN_THREADS, 0, st>>>((uint64_t*)ctx->tile_sum.p, ntiles, (uint64_t*)ctx->tile_sum.p + ntiles);
    eb_scan_finish<<<(unsigned)ntiles, SCAN_THREADS, 0, st>>>((const uint64_t*)ctx->sz16.p, n, (const uint64_t*)ctx->tile_sum.p, (const uint64_t*)ctx->tile_sum.p + ntiles, d_out_off);
    CK(cudaGetLastError());
    CK(cudaEventRecord(ctx->ev[2], st));
    *launches += 3;
    CK(cudaMemcpyAsync(total_out, d_out_off + n, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return EB200_OK;
}

// grow a device buffer keeping its first `keep` bytes
static cudaError_t grow_preserving(DevBuf& b, size_t want, size_t keep, cudaStream_t st) {
    void* np = nullptr;
    size_t cap = want + want / 8 + 256;
    cudaError_t e = cudaMalloc(&np, cap);
    if (e != cudaSuccess) return e;
    if (keep) e = cudaMemcpyAsync(np, b.p, keep, cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { cudaFree(np); return e; }
    cudaFree(b.p); b.p = np; b.cap = cap;
    return cudaSuccess;
}

// Single-pass mode: slot offsets from INPUT sizes (+ slack) first, then one kernel decides and writes every case.
// own_out: the output arena is ctx->out (host paths) and may be grown; otherwise the caller's arena is used as is.
// A case that finds the scratch arena or the overflow region exhausted flags ITSELF (status OVERFLOW, reason 1 / 11, its
// input copied to its slot); the host then grows the arena and re-runs exactly those case numbers in a follow-up
// launch -- the batch is never run twice.
static int run_fused(eb200_ctx* ctx, const BatchParams& bp, const eb200_opts* opts, const uint8_t* d_data, const uint64_t* d_off, uint64_t data_bytes,
                     bool own_out, uint8_t* d_out, uint64_t out_capacity, uint64_t out_base, uint64_t* d_out_off, uint64_t* d_out_len, eb200_meta* d_meta,
                     cudaStream_t st, uint64_t* total_out, uint32_t* launches, uint64_t host_slots = 0) {
    uint64_t n = bp.n_cases;
    CK(ctx->sz16.ensure(n * 8));
    CK(ctx->case_status.ensure(n + 64));
    uint64_t ntiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    CK(ctx->tile_sum.ensure((ntiles + 1) * 8));
    CK(ctx->slot_off.ensure((n + 1) * 8));
    CK(ctx->counters.ensure(64));
    CK(ctx->cases.ensure(sizeof(CaseOut)));
    uint64_t scratch_want = scratch_bytes_for(bp, opts, data_bytes);
    if (ctx->scratch.cap < scratch_want) CK(ctx->scratch.ensure(scratch_want));
    CK(cudaEventRecord(ctx->ev[1], st));
    eb_slot_sizes<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_off, bp.first_case, bp.n_blobs, n, bp.generator == 4 ? jump_slot_bytes(bp) : 0,
                                                               (uint64_t*)ctx->sz16.p);
    eb_scan_tiles<<<(unsigned)ntiles, SCAN_THREADS, 0, st>>>((const uint64_t*)ctx->sz16.p, n, (uint64_t*)ctx->tile_sum.p);
    eb_scan_tile_offsets<<<1, SCAN_THREADS, 0, st>>>((uint64_t*)ctx->tile_sum.p, ntiles, (uint64_t*)ctx->tile_sum.p + ntiles);
    eb_scan_finish<<<(unsigned)ntiles, SCAN_THREADS, 0, st>>>((const uint64_t*)ctx->sz16.p, n, (const uint64_t*)ctx->tile_sum.p, (const uint64_t*)ctx->tile_sum.p + ntiles, (uint64_t*)ctx->slot_off.p);
    CK(cudaGetLastError());
    CK(cudaEventRecord(ctx->ev[2], st));
    *launches += 4;
    uint64_t slots = host_slots;      // the pipelined host path sums the slot sizes itself (it has the offsets): one sync less per chunk
    if (!slots) {
        CK(cudaMemcpyAsync(&slots, (uint64_t*)ctx->slot_off.p + n, 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    if (own_out) {
        uint64_t want = out_base + slots + std::max<uint64_t>(64ull << 20, slots / 8) + 64;
        if (ctx->out.cap < want) {
            if (out_base) return EB200_ERR_NOMEM;       // pipelined chunks cannot move the arena under in-flight downloads; the caller sized it
            CK(ctx->out.ensure(want));
        }
        d_out = (uint8_t*)ctx->out.p + out_base; out_capacity = ctx->out.cap - out_base - 64;
    }
    if (slots > out_capacity) return EB200_ERR_NOMEM;
    unsigned long long used[5] = {0, 0, 0, 0, 0};     // overflow bits, ovf_used, flagged[3]
    unsigned long long* cnt = (unsigned long long*)ctx->counters.p;
    CK(cudaMemsetAsync(ctx->counters.p, 0, 64, st));
    uint64_t n_retried = 0, n_list = 0;
    std::vector<uint8_t> status_host;
    std::vector<uint32_t> list_host;
    for (int attempt = 0;; attempt++) {
        LaunchPlan lp; int rc = plan_launch(ctx, bp, data_bytes, attempt ? n_list : n, true, lp); if (rc) return rc;
        FusedArgs fa; memset(&fa, 0, sizeof(fa));
        fa.fused = 1; fa.out = d_out; fa.out_capacity = out_capacity; fa.slot_off = (const uint64_t*)ctx->slot_off.p; fa.out_off = d_out_off;
        fa.ovf_base = slots; fa.ovf_used = cnt + CNT_OVF_USED; fa.data_bytes = data_bytes;
        fa.case_counter = cnt + CNT_NEXT_CASE; fa.deciders = lp.roles.deciders; fa.fronts = lp.roles.fronts; fa.front_depth = ctx->front_depth; fa.tma_workers = ctx->tma_workers;
        if (attempt) { fa.case_list = (const uint32_t*)ctx->retry_list.p; fa.n_list = n_list; }
        if (attempt == 0) CK(cudaEventRecord(ctx->ev[0], st));
        launch_cases(ctx, bp, lp, st, d_data, d_off, d_out_len, d_meta, fa);
        CK(cudaGetLastError());
        CK(cudaEventRecord(ctx->ev[3], st));
        (*launches)++;
        CK(cudaMemcpyAsync(used, cnt + CNT_OVERFLOW, 40, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        uint32_t ovf = (uint32_t)used[0];
        bool need_scratch = (ovf & 1) != 0, need_out = (ovf & 4) && own_out && !out_base;
        if ((!need_scratch && !need_out) || attempt >= 4 || n > 0xffffffffull) break;
        // which cases ran out of arena space?
        status_host.resize(n);
        CK(cudaMemcpyAsync(status_host.data(), ctx->case_status.p, n, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        list_host.clear();
        for (uint64_t k = 0; k < n; k++) {
            uint32_t stt = status_host[k] & 15u, reason = status_host[k] >> 4;
            if (stt == CASE_OVERFLOW && ((reason == 1 && need_scratch) || (reason == 11 && need_out))) list_host.push_back((uint32_t)k);
        }
        if (list_host.empty()) break;
        n_list = list_host.size(); n_retried += n_list;
        CK(ctx->retry_list.ensure(n_list * 4));
        CK(cudaMemcpyAsync(ctx->retry_list.p, list_host.data(), n_list * 4, cudaMemcpyHostToDevice, st));
        if (need_scratch) { CK(cudaStreamSynchronize(st)); CK(ctx->scratch.ensure(ctx->scratch.cap * 2)); }
        if (need_out) {
            uint64_t keep = slots + used[1];
            CK(grow_preserving(ctx->out, ctx->out.cap * 2, keep, st));
            d_out = (uint8_t*)ctx->out.p; out_capacity = ctx->out.cap - 64;
        }
        // the follow-up launch starts with an empty scratch arena (finished cases have their bytes in `out` already),
        // keeps the overflow region's fill level and the flag counters, and restarts the case counter
        unsigned long long zero = 0; uint32_t zero32 = 0;
        CK(cudaMemcpyAsync(cnt + CNT_SCRATCH, &zero, 8, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(cnt + CNT_OVERFLOW, &zero32, 4, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(cnt + CNT_NEXT_CASE, &zero, 8, cudaMemcpyHostToDevice, st));
        CK(cudaStreamSynchronize(st));
    }
    ctx->flag_counts[0] = used[2]; ctx->flag_counts[1] = used[3]; ctx->flag_counts[2] = used[4] >= n_retried ? used[4] - n_retried : 0;
    *total_out = slots + used[1];
    CK(cudaMemcpyAsync(d_out_off + n, total_out, 8, cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));
    return EB200_OK;
}

static int run_apply(eb200_ctx* ctx, uint64_t n, const uint64_t* d_out_off, uint8_t* d_out, uint64_t out_capacity, uint64_t total, cudaStream_t st, uint32_t* launches) {
    CK(cudaEventRecord(ctx->ev[3], st));
    if (total > 0) {
        const ApplyVariant& av = apply_variants[ctx->apply_variant];
        uint64_t ctas = (total + av.tile - 1) / av.tile;
        CK(ctx->tile_case.ensure((ctas + 1) * sizeof(uint32_t)));
        eb_tile_cases<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_out_off, n, (uint32_t*)ctx->tile_case.p, av.tile);
        av.launch((unsigned)ctas, st, (const CaseOut*)ctx->cases.p, (const Seg*)ctx->segs.p, d_out_off, (const uint32_t*)ctx->tile_case.p, n, d_out, out_capacity);
        CK(cudaGetLastError());
        (*launches) += 2;
    }
    CK(cudaEventRecord(ctx->ev[4], st));
    return EB200_OK;
}

static void fill_stats(eb200_ctx* ctx, eb200_stats* s) {
    if (!s) return;
    s->n_unsupported = ctx->flag_counts[0]; s->n_died = ctx->flag_counts[1]; s->n_overflow = ctx->flag_counts[2];
    if (ctx->fused) {   // single pass: the "decide" kernel also moved the bytes; there is no apply kernel
        cudaEventElapsedTime(&s->ms_decide, ctx->ev[0], ctx->ev[3]);
        cudaEventElapsedTime(&s->ms_scan, ctx->ev[1], ctx->ev[2]);
        s->ms_apply = 0.f;
        return;
    }
    cudaEventElapsedTime(&s->ms_decide, ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&s->ms_scan, ctx->ev[1], ctx->ev[2]);
    cudaEventElapsedTime(&s->ms_apply, ctx->ev[3], ctx->ev[4]);
}

int eb200_fuzz_batch_device(eb200_ctx* ctx, const eb200_opts* opts, const uint8_t* d_data, const uint64_t* d_off, uint64_t n_blobs, uint64_t data_bytes,
                            uint64_t n_cases, uint8_t* d_out, uint64_t out_capacity, uint64_t* d_out_off, uint64_t* d_out_len,
                            eb200_meta* d_meta, void* stream, eb200_stats* stats) {
    if (!ctx || !opts || !d_data || !d_off || !d_out || !d_out_off || !d_out_len || n_blobs == 0) return EB200_ERR_ARG;
    if (((uintptr_t)d_data & 15u) || ((uintptr_t)d_out & 15u)) return EB200_ERR_ARG;
    static_assert(sizeof(eb200_meta) == sizeof(MetaDev), "meta layout");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (stats) memset(stats, 0, sizeof(*stats));
    if (n_cases == 0) return EB200_OK;
    BatchParams bp; int rc = compute_batch_params(opts, n_blobs, n_cases, bp);
    if (rc) return rc;
    uint32_t launches = 0; uint64_t total = 0;
    CK(cudaEventRecord(ctx->ev[5], st));
    if (ctx->fused) {
        rc = run_fused(ctx, bp, opts, d_data, d_off, data_bytes, false, d_out, out_capacity, 0, d_out_off, d_out_len, d_meta, st, &total, &launches);
        if (rc) return rc;
        CK(cudaEventRecord(ctx->ev[4], st));
    } else {
        rc = run_decide_scan(ctx, bp, opts, d_data, d_off, data_bytes, d_out_off, d_out_len, d_meta, st, &total, &launches);
        if (rc) return rc;
        if (total > out_capacity) return EB200_ERR_NOMEM;
        rc = run_apply(ctx, n_cases, d_out_off, d_out, out_capacity, total, st, &launches);
        if (rc) return rc;
    }
    CK(cudaStreamSynchronize(st));
    if (stats) {
        fill_stats(ctx, stats); cudaEventElapsedTime(&stats->ms_total, ctx->ev[5], ctx->ev[4]);
        stats->n_cases = n_cases; stats->kernels_launched = launches; stats->bytes_out = total;
    }
    return EB200_OK;
}

static int fuzz_batch_host(eb200_ctx* ctx, const eb200_opts* opts, const uint8_t* data, const uint64_t* off, uint64_t n_blobs, uint64_t n_cases,
                           uint8_t** out_data, uint8_t* user_out, uint64_t user_cap, uint64_t* out_off, uint64_t* out_len, eb200_meta* meta, eb200_stats* stats);

int eb200_fuzz_batch(eb200_ctx* ctx, const eb200_opts* opts, const uint8_t* data, const uint64_t* off, uint64_t n_blobs, uint64_t n_cases,
                     uint8_t** out_data, uint64_t* out_off, uint64_t* out_len, eb200_meta* meta, eb200_stats* stats) {
    if (!out_data) return EB200_ERR_ARG;
    return fuzz_batch_host(ctx, opts, data, off, n_blobs, n_cases, out_data, nullptr, 0, out_off, out_len, meta, stats);
}
// Chunked, copy/compute-overlapped variant of the host path: the corpus is uploaded in chunks of cases on a copy
// stream (EB200_H2D_AHEAD chunks ahead of the compute) while earlier chunks are being decided on the compute stream and
// downloaded on a third stream. Compute for consecutive chunks stays on ONE stream, so the per-batch arenas (scratch,
// counters) are reused safely; only PCIe traffic overlaps. Needs pinned host buffers to overlap (eb200_host_alloc gives
// NUMA-local ones). Every exit, error or not, drains all three streams before returning: the caller's buffers are never
// the target of a DMA still in flight, and the events are always destroyed.
static int fuzz_batch_host_pipelined(eb200_ctx* ctx, const eb200_opts* opts, const uint8_t* data, const uint64_t* off, uint64_t n_blobs, uint64_t n_cases,
                                     uint8_t* user_out, uint64_t user_cap, uint64_t* out_off, uint64_t* out_len, eb200_meta* meta, eb200_stats* stats,
                                     uint64_t chunk) {
    CK(cudaSetDevice(ctx->device));
    if (stats) memset(stats, 0, sizeof(*stats));
    uint64_t data_bytes = off[n_blobs];
    uint64_t first = opts->first_case ? opts->first_case : 1;
    uint64_t b0 = (first - 1) % n_blobs;                 // blob of the first case; the caller checked that the range does not wrap
    if (!ctx->s_h2d) { CK(cudaStreamCreateWithFlags(&ctx->s_h2d, cudaStreamNonBlocking)); CK(cudaStreamCreateWithFlags(&ctx->s_d2h, cudaStreamNonBlocking));
                       CK(cudaStreamCreateWithFlags(&ctx->s_comp, cudaStreamNonBlocking)); }
    uint64_t nchunks = (n_cases + chunk - 1) / chunk;
    std::vector<cudaEvent_t> ev_up(nchunks, nullptr), ev_done(nchunks, nullptr);
    std::vector<uint64_t> bases(nchunks + 1, 0);
    uint64_t base = 0; uint32_t launches = 0; int rc = EB200_OK;
    cudaError_t ce = cudaSuccess;
    auto t0 = std::chrono::steady_clock::now();
#define PCK(call) do { ce = (call); if (ce != cudaSuccess) { ctx->last_err = std::string(#call) + ": " + cudaGetErrorString(ce); rc = EB200_ERR_CUDA; goto drain; } } while (0)
    {
        for (uint64_t j = 0; j < nchunks; j++) { PCK(cudaEventCreateWithFlags(&ev_up[j], cudaEventDisableTiming)); PCK(cudaEventCreateWithFlags(&ev_done[j], cudaEventDisableTiming)); }
        PCK(ctx->data.ensure(data_bytes + 64));
        PCK(ctx->off.ensure((n_blobs + 1) * 8));
        PCK(ctx->out_off.ensure((n_cases + nchunks + 1) * 8));
        PCK(ctx->out_len.ensure(n_cases * 8));
        PCK(ctx->meta.ensure(n_cases * sizeof(MetaDev)));
        {   // output arena: the slots of every chunk (same formula as eb_slot_sizes: input + clamp(len/16, 256, 65536), 16-byte
            // aligned) + an overflow region per chunk. Pipelined chunks cannot move the arena under downloads in flight, so it
            // is sized here once -- small blobs need several times their input (a 100-byte blob has a 368-byte slot).
            uint64_t slots = 0;
            for (uint64_t k = 0; k < n_cases; k++) { uint64_t len = off[b0 + k + 1] - off[b0 + k]; uint64_t slack = std::min<uint64_t>(std::max<uint64_t>(len / 16, 256), 65536); slots += align16(len + slack); }
            PCK(ctx->out.ensure(slots + std::max<uint64_t>(64ull << 20, slots / 8 / std::max<uint64_t>(nchunks, 1)) * (nchunks + 1) + 4096));
        }
        PCK(cudaMemcpyAsync(ctx->off.p, off, (n_blobs + 1) * 8, cudaMemcpyHostToDevice, ctx->s_h2d));
        uint64_t next_up = 0;
        auto upload_until = [&](uint64_t hi) -> cudaError_t {
            for (; next_up < std::min(hi, nchunks); next_up++) {
                uint64_t k0 = next_up * chunk, k1 = std::min(n_cases, k0 + chunk);
                uint64_t lo = off[b0 + k0], h = off[b0 + k1];
                cudaError_t e = cudaSuccess;
                if (h > lo) e = cudaMemcpyAsync((uint8_t*)ctx->data.p + lo, data + lo, h - lo, cudaMemcpyHostToDevice, ctx->s_h2d);
                if (e == cudaSuccess) e = cudaEventRecord(ev_up[next_up], ctx->s_h2d);
                if (e != cudaSuccess) return e;
            }
            return cudaSuccess;
        };
        for (uint64_t j = 0; j < nchunks; j++) {
            PCK(upload_until(j + 1 + (uint64_t)ctx->h2d_ahead));               // uploads run ahead of the compute
            uint64_t k0 = j * chunk, k1 = std::min(n_cases, k0 + chunk), nc = k1 - k0;
            PCK(cudaStreamWaitEvent(ctx->s_comp, ev_up[j], 0));
            eb200_opts o = *opts; o.first_case = first + k0;
            BatchParams bp; rc = compute_batch_params(&o, n_blobs, nc, bp);
            if (rc) goto drain;
            uint64_t* d_off_j = (uint64_t*)ctx->out_off.p + k0 + j;          // nc + 1 entries per chunk
            uint64_t total = 0;
            if (ctx->fused) {
                uint64_t cslots = 0;
                for (uint64_t k = k0; k < k1; k++) { uint64_t len = off[b0 + k + 1] - off[b0 + k]; uint64_t slack = std::min<uint64_t>(std::max<uint64_t>(len / 16, 256), 65536); cslots += align16(len + slack); }
                rc = run_fused(ctx, bp, &o, (const uint8_t*)ctx->data.p, (const uint64_t*)ctx->off.p, data_bytes, true, nullptr, 0, base, d_off_j,
                               (uint64_t*)ctx->out_len.p + k0, meta ? (eb200_meta*)ctx->meta.p + k0 : nullptr, ctx->s_comp, &total, &launches, cslots);
                if (rc) goto drain;
                if (base + total > user_cap) { rc = EB200_ERR_NOMEM; goto drain; }
            } else {
                rc = run_decide_scan(ctx, bp, &o, (const uint8_t*)ctx->data.p, (const uint64_t*)ctx->off.p, data_bytes, d_off_j,
                                     (uint64_t*)ctx->out_len.p + k0, meta ? (eb200_meta*)ctx->meta.p + k0 : nullptr, ctx->s_comp, &total, &launches);
                if (rc) goto drain;
                if (base + total > user_cap) { rc = EB200_ERR_NOMEM; goto drain; }
                if (base + total + 64 > ctx->out.cap) {                          // rare: the estimate was too small -- drain and grow
                    PCK(cudaStreamSynchronize(ctx->s_d2h)); PCK(cudaStreamSynchronize(ctx->s_comp));
                    PCK(grow_preserving(ctx->out, (base + total) * 2 + 64, base, ctx->s_comp));
                }
                rc = run_apply(ctx, nc, d_off_j, (uint8_t*)ctx->out.p + base, ctx->out.cap - base, total, ctx->s_comp, &launches);
                if (rc) goto drain;
            }
            PCK(cudaEventRecord(ev_done[j], ctx->s_comp));
            PCK(cudaStreamWaitEvent(ctx->s_d2h, ev_done[j], 0));
            if (total) PCK(cudaMemcpyAsync(user_out + base, (uint8_t*)ctx->out.p + base, total, cudaMemcpyDeviceToHost, ctx->s_d2h));
            PCK(cudaMemcpyAsync(out_off + k0, d_off_j, nc * 8, cudaMemcpyDeviceToHost, ctx->s_d2h));
            PCK(cudaMemcpyAsync(out_len + k0, (uint64_t*)ctx->out_len.p + k0, nc * 8, cudaMemcpyDeviceToHost, ctx->s_d2h));
            if (meta) PCK(cudaMemcpyAsync(meta + k0, (MetaDev*)ctx->meta.p + k0, nc * sizeof(MetaDev), cudaMemcpyDeviceToHost, ctx->s_d2h));
            bases[j] = base; base += total;
        }
    }
drain:
#undef PCK
    {   // one way out: nothing may still be writing into the caller's buffers, and nothing leaks
        cudaError_t e1 = cudaStreamSynchronize(ctx->s_h2d), e2 = cudaStreamSynchronize(ctx->s_comp), e3 = cudaStreamSynchronize(ctx->s_d2h);
        for (uint64_t j = 0; j < nchunks; j++) { if (ev_up[j]) cudaEventDestroy(ev_up[j]); if (ev_done[j]) cudaEventDestroy(ev_done[j]); }
        if (rc == EB200_OK) { cudaError_t e = e1 != cudaSuccess ? e1 : e2 != cudaSuccess ? e2 : e3; if (e != cudaSuccess) { ctx->last_err = cudaGetErrorString(e); rc = EB200_ERR_CUDA; } }
    }
    if (rc) return rc;
    for (uint64_t j = 0; j < nchunks; j++) { uint64_t k0 = j * chunk, k1 = std::min(n_cases, k0 + chunk); for (uint64_t k = k0; k < k1; k++) out_off[k] += bases[j]; }
    out_off[n_cases] = base;
    if (stats) {
        stats->ms_total = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
        stats->n_cases = n_cases; stats->kernels_launched = launches;
        for (uint64_t k = 0; k < n_cases; k++) { stats->bytes_out += out_len[k]; stats->bytes_in += off[b0 + k + 1] - off[b0 + k]; }
    }
    return EB200_OK;
}

int eb200_fuzz_batch_into(eb200_ctx* ctx, const eb200_opts* opts, const uint8_t* data, const uint64_t* off, uint64_t n_blobs, uint64_t n_cases,
                          uint8_t* out_buf, uint64_t out_capacity, uint64_t* out_off, uint64_t* out_len, eb200_meta* meta, eb200_stats* stats) {
    if (!out_buf) return EB200_ERR_ARG;
    if (ctx && opts && off && data && out_off && out_len && n_blobs) {
        // big batches whose cases read a contiguous run of blobs go through the overlapped pipeline. It uploads each chunk's
        // own blobs only, so it is for generators that read blob (I-1) mod n (direct, random, stdin): a file or jump case reads
        // any blob. The generator draw is the parent's, host-only and cheap.
        uint64_t data_bytes = off[n_blobs];
        uint64_t first = opts->first_case ? opts->first_case : 1;
        uint64_t b0 = (first - 1) % n_blobs;
        bool ok = true;
        for (uint64_t b = 0; b < n_blobs && ok; b++) ok = off[b + 1] >= off[b] && off[b + 1] - off[b] <= 0xfffffff0ull;
        if (!ok) return EB200_ERR_ARG;
        BatchParams bp;
        bool own_blob = compute_batch_params(opts, n_blobs, n_cases, bp) == EB200_OK && bp.generator != 2 && bp.generator != 4;
        if (own_blob && b0 + n_cases <= n_blobs && data_bytes >= (256ull << 20) && n_cases >= 4096) {
            uint64_t avg = std::max<uint64_t>(1, data_bytes / n_blobs);
            uint64_t chunk = std::max<uint64_t>(1024, ((uint64_t)ctx->chunk_mb << 20) / avg);
            if (chunk * 2 <= n_cases) return fuzz_batch_host_pipelined(ctx, opts, data, off, n_blobs, n_cases, out_buf, out_capacity, out_off, out_len, meta, stats, chunk);
        }
    }
    uint8_t* dummy = nullptr;
    return fuzz_batch_host(ctx, opts, data, off, n_blobs, n_cases, &dummy, out_buf, out_capacity, out_off, out_len, meta, stats);
}

static int fuzz_batch_host(eb200_ctx* ctx, const eb200_opts* opts, const uint8_t* data, const uint64_t* off, uint64_t n_blobs, uint64_t n_cases,
                           uint8_t** out_data, uint8_t* user_out, uint64_t user_cap, uint64_t* out_off, uint64_t* out_len, eb200_meta* meta, eb200_stats* stats) {
    if (!ctx || !opts || !off || !out_data || !out_off || !out_len || n_blobs == 0) return EB200_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    if (stats) memset(stats, 0, sizeof(*stats));
    *out_data = nullptr;
    if (n_cases == 0) return EB200_OK;
    uint64_t data_bytes = off[n_blobs];
    if (data_bytes && !data) return EB200_ERR_ARG;
    for (uint64_t b = 0; b < n_blobs; b++) if (off[b + 1] < off[b] || off[b + 1] - off[b] > 0xfffffff0ull) return EB200_ERR_ARG;
    BatchParams bp; int rc = compute_batch_params(opts, n_blobs, n_cases, bp);
    if (rc) return rc;
    cudaStream_t st = 0;
    CK(ctx->data.ensure(data_bytes + 64));
    CK(ctx->off.ensure((n_blobs + 1) * 8));
    CK(ctx->out_off.ensure((n_cases + 1) * 8));
    CK(ctx->out_len.ensure(n_cases * 8));
    CK(ctx->meta.ensure(n_cases * sizeof(MetaDev)));
    CK(cudaEventRecord(ctx->ev[5], st));
    if (data_bytes) CK(cudaMemcpyAsync(ctx->data.p, data, data_bytes, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->off.p, off, (n_blobs + 1) * 8, cudaMemcpyHostToDevice, st));
    uint32_t launches = 0; uint64_t total = 0;
    if (ctx->fused) {
        rc = run_fused(ctx, bp, opts, (const uint8_t*)ctx->data.p, (const uint64_t*)ctx->off.p, data_bytes, true, nullptr, 0, 0, (uint64_t*)ctx->out_off.p,
                       (uint64_t*)ctx->out_len.p, (eb200_meta*)ctx->meta.p, st, &total, &launches);
        if (rc) return rc;
        CK(cudaEventRecord(ctx->ev[4], st));
    } else {
        rc = run_decide_scan(ctx, bp, opts, (const uint8_t*)ctx->data.p, (const uint64_t*)ctx->off.p, data_bytes, (uint64_t*)ctx->out_off.p,
                             (uint64_t*)ctx->out_len.p, (eb200_meta*)ctx->meta.p, st, &total, &launches);
        if (rc) return rc;
        CK(ctx->out.ensure(total + 64));
        rc = run_apply(ctx, n_cases, (const uint64_t*)ctx->out_off.p, (uint8_t*)ctx->out.p, ctx->out.cap, total, st, &launches);
        if (rc) return rc;
    }
    uint8_t* host_out = user_out;
    if (user_out) { if (total > user_cap) return EB200_ERR_NOMEM; }
    else { host_out = (uint8_t*)malloc(total ? total : 1); if (!host_out) return EB200_ERR_NOMEM; }
    cudaError_t e = cudaSuccess;
    if (total) e = cudaMemcpyAsync(host_out, ctx->out.p, total, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out_off, ctx->out_off.p, (n_cases + 1) * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out_len, ctx->out_len.p, n_cases * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && meta) e = cudaMemcpyAsync(meta, ctx->meta.p, n_cases * sizeof(MetaDev), cudaMemcpyDeviceToHost, st);
    cudaEvent_t evEnd = ctx->ev[4];
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { if (!user_out) free(host_out); ctx->last_err = cudaGetErrorString(e); return EB200_ERR_CUDA; }
    *out_data = user_out ? nullptr : host_out;
    if (stats) {
        fill_stats(ctx, stats); cudaEventElapsedTime(&stats->ms_total, ctx->ev[5], evEnd);
        stats->n_cases = n_cases; stats->kernels_launched = launches; stats->bytes_out = 0; stats->bytes_in = 0;
        for (uint64_t k = 0; k < n_cases; k++) { stats->bytes_out += out_len[k]; uint64_t b = (bp.first_case - 1 + k) % n_blobs; stats->bytes_in += off[b + 1] - off[b]; }
        if (meta) { stats->n_unsupported = stats->n_died = stats->n_overflow = 0; }   // recount from the per-case records
        if (meta) for (uint64_t k = 0; k < n_cases; k++) { if (meta[k].status == EB200_CASE_UNSUPPORTED) stats->n_unsupported++; else if (meta[k].status == EB200_CASE_DIED) stats->n_died++; else if (meta[k].status == EB200_CASE_OVERFLOW) stats->n_overflow++; }
    }
    return EB200_OK;
}

void eb200_free(void* p) { free(p); }

// Pinned host memory on the GPU's NUMA node (staging rings of the NIF, bench.py's e2e buffers). The pages are first-touched by
// this thread while it is bound to the CPUs of that node, then the thread's affinity is restored: a DMA out of remote-node
// memory crosses the socket interconnect and showed up as 38 GB/s per direction instead of the link's ~55 (VERDICT round 1).
void* eb200_host_alloc(eb200_ctx* ctx, uint64_t bytes) {
    if (!ctx || bytes == 0) return nullptr;
    cudaSetDevice(ctx->device);
    cpu_set_t old_set, node_set; bool bound = false;
    if (ctx->numa_node >= 0 && sched_getaffinity(0, sizeof(old_set), &old_set) == 0) {
        char path[96]; snprintf(path, sizeof(path), "/sys/devices/system/node/node%d/cpulist", ctx->numa_node);
        if (FILE* f = fopen(path, "r")) {
            char buf[4096] = {0};
            if (fgets(buf, sizeof(buf), f)) {
                CPU_ZERO(&node_set); int any = 0;
                char* save = nullptr;     // strtok_r: lanes and NIF threads may allocate at the same time
                for (char* tok = strtok_r(buf, ",\n", &save); tok; tok = strtok_r(nullptr, ",\n", &save)) {
                    int a = 0, b = 0; int n = sscanf(tok, "%d-%d", &a, &b); if (n == 1) b = a; if (n < 1) continue;
                    for (int c = a; c <= b && c < CPU_SETSIZE; c++) { CPU_SET(c, &node_set); any = 1; }
                }
                if (any && sched_setaffinity(0, sizeof(node_set), &node_set) == 0) bound = true;
            }
            fclose(f);
        }
    }
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) p = nullptr;
    if (p) { volatile uint8_t* q = (volatile uint8_t*)p; for (uint64_t i = 0; i < bytes; i += 4096) q[i] = 0; }   // first touch (cudaHostAlloc usually did already)
    if (bound) sched_setaffinity(0, sizeof(old_set), &old_set);
    return p;
}
void eb200_host_free(eb200_ctx* ctx, void* p) { if (ctx) cudaSetDevice(ctx->device); if (p) cudaFreeHost(p); }
int eb200_numa_node(eb200_ctx* ctx) { return ctx ? ctx->numa_node : -1; }

// donor sampling for config C5: one warp per window
__global__ void __launch_bounds__(256) eb_sample_donors_kernel(const uint8_t* __restrict__ data, const uint64_t* __restrict__ off, uint64_t n_blobs, uint64_t n_donors, uint32_t stride,
                                                              uint8_t* __restrict__ pool, uint32_t* __restrict__ lens) {
    uint64_t d = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (d >= n_donors) return;
    uint64_t b = (unsigned __int128)d * n_blobs / n_donors;
    uint64_t len = off[b + 1] - off[b];
    uint32_t wlen = (uint32_t)(len < stride ? len : stride);
    uint64_t start = ((d * 2654435761ull) & 0xffffffffull) % (len - wlen + 1);
    const uint8_t* src = data + off[b] + start;
    uint8_t* dst = pool + d * stride;
    for (uint32_t i = threadIdx.x & 31; i < wlen; i += 32) dst[i] = src[i];
    if ((threadIdx.x & 31) == 0) lens[d] = wlen;
}
int eb200_sample_donors(eb200_ctx* ctx, const uint8_t* d_data, const uint64_t* d_off, uint64_t n_blobs, uint64_t n_donors, uint32_t stride,
                        uint8_t* d_pool, uint32_t* d_len, void* stream) {
    if (!ctx || !d_data || !d_off || !d_pool || !d_len || n_blobs == 0 || stride == 0) return EB200_ERR_ARG;
    if (n_donors == 0) return EB200_OK;
    CK(cudaSetDevice(ctx->device));
    uint64_t threads = n_donors * 32;
    eb_sample_donors_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_data, d_off, n_blobs, n_donors, stride, d_pool, d_len);
    CK(cudaGetLastError());
    return EB200_OK;
}

// profiling aid (EB200_CASE_TIMES=1): microseconds the general per-case program spent on each case of the last launch
// (0 for cases the front warps decided); returns the number of entries copied
uint64_t eb200_debug_case_times(eb200_ctx* ctx, uint32_t* out, uint64_t n) {
    if (!ctx || !ctx->want_case_times || !ctx->case_usec.p) return 0;
    if (n > ctx->case_times_n) n = ctx->case_times_n;
    cudaSetDevice(ctx->device);
    if (cudaMemcpy(out, ctx->case_usec.p, n * 4, cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
    return n;
}
// ... and per mutator: out[2 * i] = nanoseconds inside mutator i (table order), out[2 * i + 1] = calls; 41 pairs, then 8 pairs for the
// phases of the fuse search (class tables / registers / packed runs / one-suffix runs / flat levels; eb_mut_fuse.cuh): 98 entries
int eb200_debug_mutator_times(eb200_ctx* ctx, uint64_t* out) {
    if (!ctx || !ctx->want_case_times || !ctx->case_usec.p) return 0;
    cudaSetDevice(ctx->device);
    const uint8_t* src = (const uint8_t*)ctx->case_usec.p + ((ctx->case_times_n * 4 + 63) & ~63ull);
    return cudaMemcpy(out, src, 2 * (M_COUNT + 8) * 8, cudaMemcpyDeviceToHost) == cudaSuccess ? M_COUNT : 0;
}

const char* eb200_mutator_code(int i) { return (i >= 0 && i < EB200_N_MUTATORS) ? kMutCodes[i] : nullptr; }
int eb200_mutator_default_pri(int i) { return (i >= 0 && i < EB200_N_MUTATORS) ? kMutPri[i] : -1; }
int eb200_mutator_supported(int i) { return (i >= 0 && i < EB200_N_MUTATORS) ? (mut_supported(i) ? 1 : 0) : 0; }
const char* eb200_pattern_code(int i) { return (i >= 0 && i < EB200_N_PATTERNS) ? kPatCodes[i] : nullptr; }
int eb200_pattern_default_pri(int i) { return (i >= 0 && i < EB200_N_PATTERNS) ? kPatPri[i] : -1; }
int eb200_pattern_supported(int i) { return (i >= 0 && i < EB200_N_PATTERNS) ? (pat_supported(i) ? 1 : 0) : 0; }

const char* eb200_strerror(int code) {
    switch (code) {
    case EB200_OK: return "ok";
    case EB200_ERR_CUDA: return "CUDA runtime error";
    case EB200_ERR_ARG: return "bad argument";
    case EB200_ERR_UNSUPPORTED: return "selected mutator/pattern has no device implementation";
    case EB200_ERR_NOMEM: return "out of memory / output arena too small";
    case EB200_ERR_SCRATCH: return "device scratch arena exhausted";
    case EB200_ERR_NO_DEVICE: return "no CUDA device (the engine has no CPU fallback)";
    default: return "unknown error";
    }
}
const char* eb200_last_cuda_error(eb200_ctx* ctx) { return ctx ? ctx->last_err.c_str() : ""; }
int eb200_debug_parent_draws(const eb200_opts* opts, uint64_t n_blobs, uint64_t n_cases, int64_t out[8]) {
    if (!opts || !out || n_blobs == 0) return EB200_ERR_ARG;
    BatchParams bp; int rc = compute_batch_params(opts, n_blobs, n_cases, bp);
    out[0] = bp.generator; out[1] = bp.snand_kind; out[2] = bp.n_rows; out[3] = bp.n_pats;
    out[4] = bp.parent_a1; out[5] = bp.parent_a2; out[6] = bp.parent_a3; out[7] = 0;
    return rc;
}
// internal hooks for eb_async.cpp (not in the public header)
void** eb200_ctx_async_slot(eb200_ctx* ctx) { return ctx ? &ctx->async_state : nullptr; }
int eb200_ctx_device(eb200_ctx* ctx) { return ctx ? ctx->device : -1; }
void eb200_ctx_set_error(eb200_ctx* ctx, const char* msg) { if (ctx && msg) ctx->last_err = msg; }
const char* eb200_version(void) { return "erlamsa_b200 0.1 (sm_100a)"; }

}  // extern "C"
