// erlamsa_b200 -- per-warp case state (shared memory) and edit-script helpers.
//
// A test case is a list of blocks ("Ll", reference src/erlamsa.hrl:110-142). On the device the
// list is a short table of RUNS (ptr, len, count): `count` equal-length blocks contiguous in
// memory (what flush_bvecs' 2048-byte re-chunking produces, reference src/erlamsa_utils.erl:169-175).
// Blocks already passed by the pattern walk are final and live in the OUTPUT edit script (oseg);
// the result of the latest mutation stays VIRTUAL (vseg: an edit script over existing memory)
// until something needs its bytes -- in the common one-mutation case it is never materialised and
// the apply kernel performs the only copy.
#pragma once
#include "eb_common.cuh"
#include "eb_warp.cuh"
#include "eb_jobs.cuh"
#include "eb_rng.cuh"

namespace eb {

constexpr int MAX_RUNS = 64;
constexpr int MAX_VSEG = 16;
constexpr int MAX_OSEG = 48;

struct MutRow { double score; int32_t pri; uint8_t name; uint8_t fn; uint16_t pad; };
struct Blk { const uint8_t* p; uint32_t len; uint32_t cnt; };
struct StSlot { const uint8_t* hp; const uint8_t* tp; uint32_t hl; uint32_t tl; };

// fuse search (eb_mut_fuse.cuh): a node = (source suffixes, target suffixes) as two ranges of the level's position arrays
struct FNode { uint32_t fo, fc, to, tc; };
// ... and the search state of the warp, kept in shared memory so that the node paths (separate functions) exchange it without
// going through the stack
struct FuseSh {
    const uint8_t* a; const uint8_t* b; uint32_t na, nb;
    uint32_t* F[2]; uint32_t* T[2]; FNode* ND[2];      // ping-pong: positions per side, nodes
    uint32_t fcap, tcap, ncap;
    uint32_t* tabs;                                    // class tables in global memory (starts, sizes; counters for very long lists)
    int cur; uint32_t ncur;                            // the level being split
    uint32_t e;                                        // its nodes not yet taken (from the top)
    uint32_t fo, to, nnext, maxsz;                     // the level being built
    unsigned long long* clk;                           // profiling aid
};

struct WarpState {
    MutRow rows[M_COUNT];
    MutRow tried[M_COUNT];
    uint32_t keys[M_COUNT];
    uint8_t order[M_COUNT];
    int nrows;
    // active block list
    Blk runs[MAX_RUNS]; int nruns;
    // virtual head (result of the last mutation): vlen bytes described by vseg; when vchunked the
    // bytes form floor(vlen/2048) blocks of 2048 plus one block of the remainder (possibly empty)
    int vhead; int vchunked; int nvseg; uint32_t vlen;
    Seg vseg[MAX_VSEG];
    // candidate result of the mutator being tried
    Seg tseg[MAX_VSEG]; int ntseg; uint32_t tlen;
    // output edit script
    Seg oseg[MAX_OSEG]; int noseg; uint64_t olen;
    // closure state: construct_st_line_muta (lis = 0, lrs = 1), remember/1 of sed_fuse_old
    StSlot st[2][10]; int st_n[2];
    // RES_RUNS results: the new head is handed back as real block runs (fo: two re-chunked regions)
    Blk rrun[4]; int rrun_n;
    // pending sizer / checksum wrappers (patterns sz, cs): everything emitted after `mark` is the enclosed
    // blob; when the case is complete the length field at `field_pos` is patched / the checksum appended
    struct Wrap { uint32_t kind; uint32_t bits; uint32_t big; uint32_t tail_n; uint64_t field_pos; uint64_t mark; const uint8_t* tail_p; } wrap[8];
    int nwrap;
    const uint8_t* fo_p; uint32_t fo_n; int fo_has;
    // file / stdin / jump generators: the block list does not exist until the pattern's first uncons (eb_decide.cuh force_stream);
    // jump keeps its second file in lz_p2 / lz_n2
    int lazy; const uint8_t* lz_p; uint32_t lz_n;
    const uint8_t* lz_p2; uint32_t lz_n2;
    uint32_t round;          // mux_fuzzers rounds so far in this case (Philox counter slots, eb_rng.cuh)
    uint64_t donor;          // this case's donor index (thread seed hash, see mut_fuse)
    uint16_t sc[SC_MAX];
    FuseSh fsh;
    uint32_t qpend;          // countdown of this warp's outstanding scan jobs (eb_jobs.cuh)
    uint32_t status; uint32_t reason;
    int n_used, n_failed; int used[16];
};

struct CaseCtx {
    WarpState* ws;
    Rng rng;
    const BatchParams* bp;
    Arenas ar;
    const uint8_t* next_p; uint32_t next_n; int has_next;   // the block after This (sed_fuse_next reads it)
    uint8_t* temp_base;      // this warp's reusable temp region
    uint64_t temp_used;
    uint64_t temp_floor;     // temp_reset() rewinds to here: a mutator that runs a nested scheduler parks its own tables below
    int snand_kind;          // mask function bound to `snand` when the current table was built (mutations/1 :1313)
    JobQ* q;                 // the CTA's job queue (nullptr: no worker warps, everything inline)
};

// profiling aid (EB200_CASE_TIMES=1): nanoseconds and steps per phase, eight (ns, count) pairs after the per-mutator table
enum { FPH_BIG = 0, FPH_MID, FPH_SMALL, FPH_TINY, FPH_COMPACT, PH_SGM_TOK, PH_SGM_PAIR, PH_JS_TOK, FPH_COUNT };
struct FuseClock {
    unsigned long long* tab; unsigned long long t0;
    __device__ __forceinline__ void start() { if (tab) asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t0)); }
    __device__ __forceinline__ void stop(int ph) {
        if (!tab) return;
        unsigned long long t1; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t1));
        if (lane_id() == 0) { atomicAdd(&tab[2 * ph], t1 - t0); atomicAdd(&tab[2 * ph + 1], 1ull); }
    }
};
__device__ __forceinline__ FuseClock phase_clock(const CaseCtx& c) { FuseClock k; k.tab = c.ar.mut_ns ? c.ar.mut_ns + 2 * M_COUNT : nullptr; k.t0 = 0; return k; }

// ------------------------------------------------------------------ arenas
EB_DEV uint8_t* scratch_alloc(CaseCtx& c, uint64_t bytes) {
    unsigned long long off = 0;
    uint64_t need = align16(bytes) + 16;   // +16: realigning loads may touch the next aligned word
    if (lane_id() == 0) off = atomicAdd(c.ar.scratch_used, (unsigned long long)need);
    off = __shfl_sync(0xffffffffu, off, 0);
    if (off + need > c.ar.scratch_cap) {
        if (lane_id() == 0) atomicOr(c.ar.overflow, 1u);
        c.ws->status = CASE_OVERFLOW; c.ws->reason = 1;
        return nullptr;
    }
    return c.ar.scratch + off;
}

// temporaries that die with the mutator attempt: bump inside the warp's private region, spilling to
// the (never freed) scratch arena only when a single attempt needs more than the region holds
EB_DEV void temp_reset(CaseCtx& c) { c.temp_used = c.temp_floor; }
EB_DEV uint8_t* temp_alloc(CaseCtx& c, uint64_t bytes) {
    uint64_t need = align16(bytes) + 16;
    if (c.temp_base && c.temp_used + need <= c.ar.temp_per_warp) { uint8_t* p = c.temp_base + c.temp_used; c.temp_used += need; return p; }
    return scratch_alloc(c, bytes);
}

// ------------------------------------------------------------------ segment constructors
__device__ __forceinline__ Seg seg_copy(const uint8_t* p, uint32_t len) { Seg s; s.src = (uint64_t)(uintptr_t)p; s.len = len; s.meta = SEG_COPY; return s; }
__device__ __forceinline__ Seg seg_inline(uint64_t bytes, uint32_t len) { Seg s; s.src = bytes; s.len = len; s.meta = SEG_INLINE; return s; }
__device__ __forceinline__ Seg seg_repeat(const uint8_t* p, uint32_t unit, uint32_t total) { Seg s; s.src = (uint64_t)(uintptr_t)p; s.len = total; s.meta = SEG_REPEAT | (unit << 4); return s; }
__device__ __forceinline__ Seg seg_fill(uint8_t b, uint32_t len) { Seg s; s.src = 0; s.len = len; s.meta = SEG_FILL | ((uint32_t)b << 4); return s; }

// candidate list (tseg) builder; zero-length segments are dropped, adjacent copies coalesce
__device__ __forceinline__ void t_reset(WarpState* ws) { ws->ntseg = 0; ws->tlen = 0; }
EB_DEV void t_push(WarpState* ws, Seg s) {
    EB_RECONVERGE();
    if (s.len == 0) return;
    int n = ws->ntseg;
    if (n > 0 && s.kind() == SEG_COPY && ws->tseg[n - 1].kind() == SEG_COPY && ws->tseg[n - 1].src + ws->tseg[n - 1].len == s.src) {
        ws->tseg[n - 1].len += s.len; ws->tlen += s.len; return;
    }
    if (n >= MAX_VSEG) { ws->status = CASE_OVERFLOW; ws->reason = 2; return; }
    ws->tseg[n] = s; ws->ntseg = n + 1; ws->tlen += s.len;
}
// byte i of the concatenation of segs (warp-uniform)
EB_DEV uint32_t segs_byte(const Seg* s, int n, uint32_t i) {
    for (int k = 0; k < n; k++) {
        if (i < s[k].len) {
            switch (s[k].kind()) {
            case SEG_COPY: return ((const uint8_t*)(uintptr_t)s[k].src)[i];
            case SEG_INLINE: return (uint32_t)((s[k].src >> (8 * i)) & 0xff);
            case SEG_REPEAT: return ((const uint8_t*)(uintptr_t)s[k].src)[i % s[k].arg()];
            default: return s[k].arg() & 0xff;
            }
        }
        i -= s[k].len;
    }
    return 0;
}
// erlamsa_utils:binarish/1 (reference src/erlamsa_utils.erl:238-247) over an edit script
EB_DEV bool segs_binarish(const Seg* s, int n, uint32_t len) {
    for (uint32_t i = 0;; i++) {
        uint32_t left = len - i;
        uint32_t b0 = left > 0 ? segs_byte(s, n, i) : 0, b1 = left > 1 ? segs_byte(s, n, i + 1) : 0, b2 = left > 2 ? segs_byte(s, n, i + 2) : 0;
        if (left >= 3 && b0 == 0xEF && b1 == 0xBB && b2 == 0xBF) return false;
        if (left >= 2 && b0 == 0xFE && b1 == 0x0F) return false;
        if (i == 8) return false;
        if (left == 0) return false;
        if (b0 == 0) return true;
        if (b0 & 128) return true;
    }
}
EB_DEV bool mem_binarish(const uint8_t* p, uint32_t len) { Seg s = seg_copy(p, len); return segs_binarish(&s, 1, len); }

// does the first `len` bytes of the script equal p[0,len)?  (hd(Mll) == hd(Ll), reference
// src/erlamsa_mutations.erl:1278.)  Identity copies are skipped, the rest is compared by all lanes.
EB_DEV bool segs_equal_prefix(const Seg* s, int n, const uint8_t* p, uint32_t len) {
    uint32_t pos = 0; int l = lane_id(); uint32_t diff = 0;
    for (int k = 0; k < n && pos < len; k++) {
        uint32_t sl = s[k].len; if (pos + sl > len) sl = len - pos;
        uint32_t kind = s[k].kind();
        if (kind == SEG_COPY) {
            const uint8_t* src = (const uint8_t*)(uintptr_t)s[k].src;
            if (src != p + pos) for (uint32_t i = l; i < sl; i += 32) diff |= (uint32_t)(src[i] ^ p[pos + i]);
        } else if (kind == SEG_INLINE) {
            for (uint32_t i = l; i < sl; i += 32) diff |= (uint32_t)(((s[k].src >> (8 * i)) & 0xff) ^ p[pos + i]);
        } else if (kind == SEG_REPEAT) {
            const uint8_t* src = (const uint8_t*)(uintptr_t)s[k].src; uint32_t u = s[k].arg();
            for (uint32_t i = l; i < sl; i += 32) diff |= (uint32_t)(src[i % u] ^ p[pos + i]);
        } else {
            uint32_t b = s[k].arg() & 0xff;
            for (uint32_t i = l; i < sl; i += 32) diff |= (uint32_t)(b ^ p[pos + i]);
        }
        pos += sl;
        if (__any_sync(0xffffffffu, diff != 0)) return false;
    }
    return true;
}

// write the script's bytes to dst (cooperative)
EB_DEV void segs_write(const Seg* s, int n, uint8_t* dst) {
    int l = lane_id();
    for (int k = 0; k < n; k++) {
        uint32_t sl = s[k].len;
        switch (s[k].kind()) {
        case SEG_COPY: warp_copy(dst, (const uint8_t*)(uintptr_t)s[k].src, sl); break;
        case SEG_INLINE: if ((uint32_t)l < sl) dst[l] = (uint8_t)(s[k].src >> (8 * l)); break;
        case SEG_REPEAT: { const uint8_t* src = (const uint8_t*)(uintptr_t)s[k].src; uint32_t u = s[k].arg(); for (uint32_t i = l; i < sl; i += 32) dst[i] = src[i % u]; break; }
        default: warp_fill(dst, (uint8_t)s[k].arg(), sl);
        }
        dst += sl;
    }
    __syncwarp();
}

// single-pass mode: execute a script into its output slot with streaming copies; sources inside the (read-only)
// corpus [ro_lo, ro_hi) take the non-coherent load path, scratch written by this kernel takes plain loads
EB_DEV void segs_write_stream(JobQ* q, const Seg* s, int n, uint8_t* dst, const uint8_t* ro_lo, const uint8_t* ro_hi) {
    int l = lane_id();
    for (int k = 0; k < n; k++) {
        uint32_t sl = s[k].len;
        switch (s[k].kind()) {
        case SEG_COPY: {
            const uint8_t* src = (const uint8_t*)(uintptr_t)s[k].src;
            post_copy(q, dst, src, sl, src >= ro_lo && src + sl <= ro_hi);
            break;
        }
        case SEG_INLINE: if ((uint32_t)l < sl) dst[l] = (uint8_t)(s[k].src >> (8 * l)); break;
        case SEG_REPEAT: {
            const uint8_t* src = (const uint8_t*)(uintptr_t)s[k].src; uint32_t u = s[k].arg();
            if (u >= 512) {   // long unit: every repetition is a streaming copy of its own
                bool nc = src >= ro_lo && src + u <= ro_hi;
                for (uint32_t o = 0; o < sl; o += u) post_copy(q, dst + o, src, sl - o < u ? sl - o : u, nc);
            } else for (uint32_t i = l; i < sl; i += 32) dst[i] = src[i % u];
            break;
        }
        default: warp_fill(dst, (uint8_t)s[k].arg(), sl);
        }
        dst += sl;
    }
    __syncwarp();
}

// append to the output edit script; when the script is full it is folded into one scratch buffer
EB_DEV void o_push(CaseCtx& c, Seg s) {
    WarpState* ws = c.ws;
    EB_RECONVERGE();
    if (s.len == 0) return;
    int n = ws->noseg;
    if (n > 0 && s.kind() == SEG_COPY && ws->oseg[n - 1].kind() == SEG_COPY && ws->oseg[n - 1].src + ws->oseg[n - 1].len == s.src
        && (uint64_t)ws->oseg[n - 1].len + s.len < 0x80000000ull) {
        ws->oseg[n - 1].len += s.len; ws->olen += s.len; return;
    }
    if (n >= MAX_OSEG) {
        if (ws->olen > c.bp->max_case_out) { ws->status = CASE_OVERFLOW; ws->reason = 5; return; }
        uint8_t* buf = scratch_alloc(c, ws->olen);
        if (!buf) return;
        segs_write(ws->oseg, n, buf);
        uint64_t left = ws->olen; n = 0;
        while (left) { uint32_t ch = left > 0x40000000ull ? 0x40000000u : (uint32_t)left; ws->oseg[n++] = seg_copy(buf, ch); buf += ch; left -= ch; }
    }
    ws->oseg[n] = s; ws->noseg = n + 1; ws->olen += s.len;
}

}  // namespace eb
