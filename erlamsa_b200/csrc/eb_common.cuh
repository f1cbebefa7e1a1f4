// erlamsa_b200 -- shared device/host definitions for the batched mutation engine.
//
// Data layout in HBM (see DESIGN.md):
//   corpus   : packed blobs  data[u8] + off[u64, n_blobs+1]
//   segments : every case's result is an "edit script": an ordered list of Seg records whose
//              concatenation is the output. A Seg copies a byte range from the corpus / the scratch
//              arena, repeats a range, fills a byte, or carries up to 8 literal bytes inline.
//   outputs  : out[u8] packed, every case starts on a 16-byte boundary; out_off[n+1], out_len[n]
//   scratch  : bump-allocated arena for intermediate rounds and large literals
#pragma once
#include <stdint.h>

#ifndef __CUDACC__
#define __host__
#define __device__
#endif

// Device functions of the decision pipeline are kept out of line: the pipeline is a long scalar
// program (scheduler + ~25 mutators, each with several RNG call sites) and full inlining produced
// ~47k SASS instructions whose instruction-cache misses were a third of all stall samples
// (profiles/decide_r1a). Calls are cheap next to an FP64 RNG draw.
#define EB_DEV __device__ __noinline__
// The general program's scalar parts are executed by all 32 lanes, which read-modify-write the same shared words (counters of the
// block-run / segment tables): right only while the warp is converged. EB_RECONVERGE() marks the entry of every such helper. It is
// empty in the shipped kernel -- whose results are pinned by the GPU suite -- and a __syncwarp() in the 128-register build of
// eb_wide.cu (DESIGN.md section 9: the experiment that says whether a lost reconvergence explains that build's differences).
#ifdef EB_WIDE_RECONVERGE
#define EB_RECONVERGE() __syncwarp()
#else
#define EB_RECONVERGE()
#endif

namespace eb {

// ---- table indices: reference src/erlamsa_mutations.erl:1291-1331
enum MutId : int {
    M_SGM = 0, M_JS, M_UW, M_UI, M_AB, M_AD, M_TR2, M_TD, M_NUM, M_TS1, M_TR, M_TS2,
    M_BD, M_BEI, M_BED, M_BF, M_BI, M_BER, M_BR, M_SP, M_SR, M_SD, M_SNAND, M_SRND,
    M_LD, M_LDS, M_LR2, M_LRI, M_LR, M_LS, M_LP, M_LIS, M_LRS, M_FT, M_FN, M_FO,
    M_LEN, M_B64, M_URI, M_ZIP, M_NIL, M_COUNT
};
// ---- reference src/erlamsa_patterns.erl:395-404
enum PatId : int { P_OD = 0, P_ND, P_BU, P_SK, P_SZ, P_CS, P_AR, P_CP, P_CO, P_NU, P_COUNT };

// reference src/erlamsa.hrl:44-58
constexpr uint32_t INITIAL_IP = 24;
constexpr uint32_t AVG_BLOCK_SIZE = 2048;
constexpr uint32_t ABSMAXHALF_BINARY_BLOCK = 500000;
constexpr uint32_t ABSMAX_BINARY_BLOCK = 1000000;

// ---- edit-script segment (16 bytes)
enum SegKind : uint32_t {
    SEG_COPY = 0,     // len bytes from device address src
    SEG_INLINE = 1,   // len (<= 8) literal bytes stored in the src field itself (little endian)
    SEG_REPEAT = 2,   // len bytes: src[j mod unit], unit = meta >> 4
    SEG_FILL = 3      // len copies of byte (meta >> 4)
};
struct __align__(16) Seg {
    uint64_t src;     // device address, or inline literal bytes
    uint32_t len;     // bytes this segment contributes to the output
    uint32_t meta;    // low 4 bits: SegKind; high 28 bits: repeat unit / fill byte
    __host__ __device__ uint32_t kind() const { return meta & 15u; }
    __host__ __device__ uint32_t arg() const { return meta >> 4; }
};

// ---- per-case result header written by the decide kernel
struct __align__(16) CaseOut {
    uint64_t seg_begin;   // index of the first Seg in the segment arena
    uint32_t nseg;
    uint32_t status;
    uint64_t out_len;
    uint64_t pad;
};

// ---- what the host computes once per batch from the options (the parent process' part of
//      erlamsa_main:fuzzer/1: T0..T3 of SURVEY.md appendix A)
struct BatchParams {
    // parent stream state right before the first gen_predictable_seed() of case I = 1
    int32_t parent_a1, parent_a2, parent_a3;
    int32_t rng_mode;
    uint64_t philox_key;
    // scheduler table after make_mutator/mutators_mutator: selected rows in table order
    int32_t n_rows;
    int32_t snand_kind;            // 0 nand, 1 or, 2 xor
    uint8_t row_id[M_COUNT];
    int32_t row_pri[M_COUNT];
    int32_t row_score[M_COUNT];    // initial integer scores 2..9
    // patterns after sort_by_priority
    int32_t n_pats;
    int32_t pat_sum;
    int32_t pat_pri[P_COUNT];
    int32_t pat_id[P_COUNT];
    int32_t generator;             // 0 direct, 1 random, 2 file, 3 stdin, 4 jump
    int32_t rbs_bound;             // round(4096 * blockscale): bound of the unused rand_block_size draw
    int32_t rbs_min;               // round(256 * blockscale)
    uint64_t first_case;
    uint64_t n_blobs, n_cases;
    uint64_t max_case_out;
    int32_t ssrf_port;
    char ssrf_host[64];
    // cross-seed donor pool of sed_fuse_old (config C5), device pointers
    const uint8_t* donor_pool; const uint32_t* donor_len; uint64_t n_donors; uint32_t donor_stride;
};

// ---- arenas (device) -- bump allocated with atomics; `overflow` is sticky
struct Arenas {
    uint8_t* scratch; uint64_t scratch_cap; unsigned long long* scratch_used;
    Seg* segs; uint64_t segs_cap; unsigned long long* segs_used;
    uint32_t* overflow;   // bit 0 scratch, bit 1 segs
    // per-warp reusable temporaries (parse tables, stacks, sort keys): warp slot w owns
    // temp + w * temp_per_warp; reset for every mutator attempt, never referenced by a result
    uint8_t* temp; uint64_t temp_per_warp;
    unsigned long long* flagged;   // [3]: cases that ended unsupported / died / over a cap
    uint8_t* case_status;          // [n_cases]: status | reason << 4 (the host re-runs arena-overflow cases from it)
    unsigned long long* mut_ns;    // [2 * (M_COUNT + 8)] or null: nanoseconds and calls per mutator, then per fuse phase (same profiling aid)
    uint32_t* case_usec;           // [n_cases] or null: wall time of the general per-case program (EB200_CASE_TIMES=1, profiling aid)
};

struct __align__(8) MetaDev {
    int32_t pattern, generator, n_used, n_failed;
    int32_t used[16];
    uint64_t draws;
    int32_t status, pad;
    int64_t thread_seed[3];
};

constexpr uint32_t CASE_OK = 0, CASE_UNSUPPORTED = 1, CASE_DIED = 2, CASE_OVERFLOW = 3;

__host__ __device__ inline uint64_t align16(uint64_t x) { return (x + 15ull) & ~15ull; }

}  // namespace eb
