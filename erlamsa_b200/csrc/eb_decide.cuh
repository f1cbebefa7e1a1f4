// erlamsa_b200 -- the decide kernel: one warp runs one test case's whole decision pipeline.
//
// Mirrors, per case I (reference file:line):
//   thread seed        erlamsa_main.erl:179-183   gen_predictable_seed on the parent stream (jump-ahead)
//   generator          erlamsa_gen.erl:43-178   direct (+ finish tail), random stream, file / stdin / jump streams (lazy)
//   pattern            erlamsa_patterns.erl:266-443   od / nd / bu / sk / co / nu state machine
//   scheduler          erlamsa_mutations.erl:1234-1280   weighted permutation, try until hd(Ll) changes
// and leaves an edit script (list of Seg) + output length per case. No payload bytes are moved
// here except when a later mutation round needs the previous round's result materialised.
#pragma once
#include "eb_mutators.cuh"

namespace eb {

// ------------------------------------------------------------------ active block list
EB_DEV uint32_t active_count(const WarpState* ws) {
    uint32_t n = 0;
    if (ws->vhead) n += ws->vchunked ? ws->vlen / AVG_BLOCK_SIZE + 1 : 1;
    for (int i = 0; i < ws->nruns; i++) n += ws->runs[i].cnt;
    return n;
}
EB_DEV bool active_is_single_empty(const WarpState* ws) {   // Ll =:= [<<>>]
    if (active_count(ws) != 1) return false;
    return ws->vhead ? ws->vlen == 0 : ws->runs[0].len == 0;
}
EB_DEV void runs_insert_front(WarpState* ws, Blk b) {
    EB_RECONVERGE();
    if (b.cnt == 0) return;
    if (ws->nruns >= MAX_RUNS) { ws->status = CASE_OVERFLOW; ws->reason = 4; return; }
    for (int i = ws->nruns; i > 0; i--) ws->runs[i] = ws->runs[i - 1];
    ws->runs[0] = b; ws->nruns++;
}
EB_DEV void runs_push_back(WarpState* ws, Blk b) {
    EB_RECONVERGE();
    if (b.cnt == 0) return;
    if (ws->nruns >= MAX_RUNS) { ws->status = CASE_OVERFLOW; ws->reason = 4; return; }
    ws->runs[ws->nruns++] = b;
}
EB_DEV void pop_head(WarpState* ws) {
    EB_RECONVERGE();
    if (ws->runs[0].cnt > 1) { ws->runs[0].p += ws->runs[0].len; ws->runs[0].cnt--; return; }
    for (int i = 1; i < ws->nruns; i++) ws->runs[i - 1] = ws->runs[i];
    ws->nruns--;
}
// materialise the virtual head into scratch and put its block(s) at the front of the run table
EB_DEV void realize_virtual(CaseCtx& c) {
    WarpState* ws = c.ws;
    if (!ws->vhead) return;
    uint8_t* buf = scratch_alloc(c, ws->vlen);
    ws->vhead = 0;
    if (!buf) return;
    segs_write(ws->vseg, ws->nvseg, buf);
    if (ws->vchunked) {
        uint32_t k = ws->vlen / AVG_BLOCK_SIZE, r = ws->vlen - k * AVG_BLOCK_SIZE;
        Blk last; last.p = buf + (uint64_t)k * AVG_BLOCK_SIZE; last.len = r; last.cnt = 1; runs_insert_front(ws, last);
        Blk full; full.p = buf; full.len = AVG_BLOCK_SIZE; full.cnt = k; runs_insert_front(ws, full);
    } else {
        Blk b; b.p = buf; b.len = ws->vlen; b.cnt = 1; runs_insert_front(ws, b);
    }
}
EB_DEV void emit_head(CaseCtx& c) {
    WarpState* ws = c.ws;
    if (ws->vhead && !ws->vchunked) { for (int i = 0; i < ws->nvseg; i++) o_push(c, ws->vseg[i]); ws->vhead = 0; return; }
    realize_virtual(c);
    if (ws->status != CASE_OK || ws->nruns == 0) return;
    o_push(c, seg_copy(ws->runs[0].p, ws->runs[0].len));
    pop_head(ws);
}
EB_DEV void emit_all(CaseCtx& c) {
    WarpState* ws = c.ws;
    if (ws->vhead) { for (int i = 0; i < ws->nvseg; i++) o_push(c, ws->vseg[i]); ws->vhead = 0; }
    for (int i = 0; i < ws->nruns; i++) {
        uint64_t tot = (uint64_t)ws->runs[i].len * ws->runs[i].cnt; const uint8_t* p = ws->runs[i].p;
        while (tot) { uint32_t ch = tot > 0x40000000ull ? 0x40000000u : (uint32_t)tot; o_push(c, seg_copy(p, ch)); p += ch; tot -= ch; }
    }
    ws->nruns = 0;
}
// split/1, reference src/erlamsa_patterns.erl:45-60: an oversize head block is cut into pieces (with draws)
EB_DEV void split_big(CaseCtx& c) {
    WarpState* ws = c.ws;
    realize_virtual(c);
    if (ws->status != CASE_OK || ws->nruns == 0) return;
    if (ws->runs[0].len <= ABSMAX_BINARY_BLOCK) return;
    const uint8_t* p = ws->runs[0].p; uint32_t left = ws->runs[0].len;
    pop_head(ws);
    Blk pieces[16]; int np = 0;
    while (left > ABSMAX_BINARY_BLOCK) {
        uint32_t as = ABSMAXHALF_BINARY_BLOCK + (uint32_t)c.rng.rand(ABSMAXHALF_BINARY_BLOCK) - 1;
        if (np >= 15) { ws->status = CASE_OVERFLOW; ws->reason = 6; return; }
        pieces[np].p = p; pieces[np].len = as; pieces[np].cnt = 1; np++;
        p += as; left -= as;
    }
    pieces[np].p = p; pieces[np].len = left; pieces[np].cnt = 1; np++;
    for (int i = np - 1; i >= 0; i--) runs_insert_front(ws, pieces[i]);
}

// Philox counter slots: (round << 8) | who, who = mutator id, or one of these
constexpr uint32_t SLOT_SCHED = 0xFF, SLOT_PATTERN = 0xFE;

// ------------------------------------------------------------------ scheduler: one mux_fuzzers round
EB_DEV double adjust_priority(double pri, double delta) {   // :1238-1242
    if (delta == 0.0) return pri;
    return fmax(2.0, fmin(10.0, pri + delta));
}
template <bool FULL>
EB_DEV void mux_fuzzers(CaseCtx& c) {
    WarpState* ws = c.ws; Rng& g = c.rng;
    if (active_count(ws) == 0 || active_is_single_empty(ws)) return;
    realize_virtual(c);
    if (ws->status != CASE_OK) return;
    const uint8_t* p = ws->runs[0].p; uint32_t n = ws->runs[0].len;
    if (ws->runs[0].cnt > 1) { c.has_next = 1; c.next_p = p + n; c.next_n = n; }
    else if (ws->nruns > 1) { c.has_next = 1; c.next_p = ws->runs[1].p; c.next_n = ws->runs[1].len; }
    else { c.has_next = 0; c.next_p = nullptr; c.next_n = 0; }
    int nr = ws->nrows;
    const uint32_t rnd = ++ws->round;
    g.set_slot((rnd << 8) | SLOT_SCHED);
    // weighted_permutations/1 :1244-1250: key_i = rand(trunc(Score*Pri)), stable sort by key descending
    for (int i = 0; i < nr; i++) ws->keys[i] = (uint32_t)g.rand((uint64_t)trunc(ws->rows[i].score * (double)ws->rows[i].pri));
    for (int i = 0; i < nr; i++) {
        uint32_t k = ws->keys[i]; int j = i - 1;
        // order[] holds row indices sorted so far; insert i after every entry with key >= k
        while (j >= 0 && ws->keys[ws->order[j]] < k) { ws->order[j + 1] = ws->order[j]; j--; }
        ws->order[j + 1] = (uint8_t)i;
    }
    int nt = 0;
    for (int t = 0; t < nr; t++) {
        bool big = n > ABSMAX_BINARY_BLOCK;   // :1269-1270 -- the node under the cursor is dropped from the list
        bool changed = false;
        MutResult r; r.kind = RES_SAME; r.delta = 0; r.rechunk = 0; r.consumed_next = 0;
        if (!big) {
            MutRow row = ws->rows[ws->order[t]];
            temp_reset(c);
            g.set_slot((rnd << 8) | (uint32_t)row.fn);
            unsigned long long t_m0 = 0;
            if (c.ar.mut_ns) asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t_m0));
            if (FULL) mut_apply(c, row, p, n, r); else mut_apply_light(c, row, p, n, r);
            if (c.ar.mut_ns && lane_id() == 0) { unsigned long long t_m1; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t_m1)); atomicAdd(&c.ar.mut_ns[2 * row.fn], t_m1 - t_m0); atomicAdd(&c.ar.mut_ns[2 * row.fn + 1], 1ull); }
            if (r.kind == RES_UNSUPPORTED) ws->status = CASE_UNSUPPORTED;
            if (ws->status != CASE_OK) return;
            row.score = adjust_priority(row.score, r.delta);
            ws->tried[nt++] = row;
            if (r.kind == RES_SEGS) {
                uint32_t first = (r.rechunk && ws->tlen >= AVG_BLOCK_SIZE) ? AVG_BLOCK_SIZE : ws->tlen;
                changed = !(first == n && segs_equal_prefix(ws->tseg, ws->ntseg, p, n));
            } else if (r.kind == RES_RUNS) {
                Seg s0 = seg_copy(ws->rrun[0].p, ws->rrun[0].len);
                changed = !(ws->rrun[0].len == n && segs_equal_prefix(&s0, 1, p, n));
            }
            EB_RECONVERGE();
            if (!changed) { ws->n_failed++; continue; }
            if (r.kind == RES_SEGS && ws->tlen > c.bp->max_case_out) { ws->status = CASE_OVERFLOW; ws->reason = 5; return; }
            if (ws->n_used < 16) ws->used[ws->n_used] = row.name;
            ws->n_used++;
        }
        // new scheduler list: reversed(tried) ++ untried tail (in permutation order)
        int tail = nr - (t + 1);
        for (int j = 0; j < tail; j++) ws->tried[nt + j] = ws->rows[ws->order[t + 1 + j]];
        for (int j = 0; j < nt / 2; j++) { MutRow x = ws->tried[j]; ws->tried[j] = ws->tried[nt - 1 - j]; ws->tried[nt - 1 - j] = x; }
        ws->nrows = nt + tail;
        for (int j = 0; j < ws->nrows; j++) ws->rows[j] = ws->tried[j];
        if (big) return;
        // commit: the head block becomes the virtual result
        pop_head(ws);
        if (r.consumed_next && ws->nruns > 0) pop_head(ws);
        if (r.kind == RES_RUNS) {
            for (int j = ws->rrun_n - 1; j >= 0; j--) runs_insert_front(ws, ws->rrun[j]);
            return;
        }
        ws->vhead = 1; ws->vchunked = r.rechunk; ws->nvseg = ws->ntseg; ws->vlen = ws->tlen;
        for (int j = 0; j < ws->ntseg; j++) ws->vseg[j] = ws->tseg[j];
        return;
    }
    // every mutator failed: mux_fuzzers(Out) -- the tried list reversed
    for (int j = 0; j < nt / 2; j++) { MutRow x = ws->tried[j]; ws->tried[j] = ws->tried[nt - 1 - j]; ws->tried[nt - 1 - j] = x; }
    for (int j = 0; j < nt; j++) ws->rows[j] = ws->tried[j];
    ws->nrows = nt;
}

// ------------------------------------------------------------------ generator
EB_DEV const uint8_t* random_block_dev(CaseCtx& c, uint32_t n) {   // random_block/1: draw i lands at byte n-1-i
    uint8_t* buf = scratch_alloc(c, n);
    if (!buf) return nullptr;
    // thirty-two draws at a time: lane l owns draws l, l+32, ... of the AS183 stream (x_{k+32} = x_k * a^32 mod p).
    // One case in ~65 000 gets a `finish` tail of up to 32 KiB; drawn one by one it held its whole CTA round for
    // milliseconds and showed up as 5-10 ms outliers among 4.0 ms steps on C3.
    random_block_fill(c, buf, n);
    return buf;
}
// finish/1 :43-51 after `len` bytes of stream: true when it adds a random tail block (false: no tail, or the scratch arena is out)
EB_DEV bool finish_block(CaseCtx& c, uint64_t len, Blk& tb) {
    Rng& g = c.rng;
    uint64_t x = g.rand(len + 1);
    if (x != len) return false;
    uint64_t bits = (uint64_t)g.rand_range(1, 16);
    uint32_t nlen = (uint32_t)g.rand(1ull << bits);
    if (!nlen) return false;
    const uint8_t* t = random_block_dev(c, nlen);
    if (!t) return false;
    tb.p = t; tb.len = nlen; tb.cnt = 1;
    return true;
}
EB_DEV void finish_tail(CaseCtx& c, uint64_t len) {
    Blk tb;
    if (finish_block(c, len, tb)) runs_push_back(c.ws, tb);
}
// ------------------------------------------------------------------ jump generator (reference src/erlamsa_gen.erl:123-150)
// Block cutter of stream_port/5 over n bytes, 32 rand_block_size draws per step: lane l evaluates draw `done + l` of the stream
// (AS183: its own state x * a^(done + l), stepped by a^32; Philox: uniform_philox_at), an inclusive scan says where each block
// ends, and the first lane whose block does not fit ends the stream. It draws from a COPY of `g`: `draws` (full blocks + 1, the
// same draws as the serial loop) is how far the caller's stream has to advance. With want < nfull the walk stops at block
// `want` and returns its place (the replay that finds a picked block without keeping the block list anywhere).
struct JumpCut { uint32_t nfull, pos; uint64_t draws; uint32_t at, len; };
EB_DEV JumpCut jump_cut(const Rng& g, const BatchParams* bp, uint32_t n, uint32_t want) {
    const int l = lane_id();
    JumpCut r; r.nfull = 0; r.pos = 0; r.draws = 0; r.at = 0; r.len = 0;
    Rng mine = g;
    if (g.mode == 0) mine.jump((uint64_t)l);
    const uint32_t s1 = modpow_u32<30269>(AS_M1, 31), s2 = modpow_u32<30307>(AS_M2, 31), s3 = modpow_u32<30323>(AS_M3, 31);
    for (;;) {
        double u;
        if (g.mode == 0) {
            u = mine.uniform_as183();
            mine.a1 = (int32_t)(((uint32_t)mine.a1 * s1) % 30269u); mine.a2 = (int32_t)(((uint32_t)mine.a2 * s2) % 30307u); mine.a3 = (int32_t)(((uint32_t)mine.a3 * s3) % 30323u);
        } else u = g.uniform_philox_at(g.local + (uint32_t)r.draws + (uint32_t)l);
        uint64_t x = (uint64_t)trunc(u * (double)bp->rbs_bound);                 // rand(rbs_bound)
        uint64_t w = x > (uint64_t)bp->rbs_min ? x : (uint64_t)bp->rbs_min;      // rand_block_size :55-56
        uint64_t end = w;
        for (int o = 1; o < 32; o <<= 1) { uint64_t y = __shfl_up_sync(0xffffffffu, end, o); if (l >= o) end += y; }
        unsigned miss = __ballot_sync(0xffffffffu, (uint64_t)r.pos + end > (uint64_t)n);
        uint32_t nfit = miss ? (uint32_t)(__ffs(miss) - 1) : 32u;
        if (want < r.nfull + nfit) {
            int j = (int)(want - r.nfull);
            uint64_t e = __shfl_sync(0xffffffffu, end, j), wj = __shfl_sync(0xffffffffu, w, j);
            r.at = r.pos + (uint32_t)(e - wj); r.len = (uint32_t)wj;
            return r;
        }
        if (nfit) r.pos += (uint32_t)__shfl_sync(0xffffffffu, end, (int)nfit - 1);
        r.nfull += nfit;
        if (miss) { r.draws += nfit + 1; return r; }
        r.draws += 32;
    }
}
// one file of jump_somewhere/2: the whole stream (every block-size draw, then finish/1), then erand over its blocks.
// false: the case ends here (an empty block list: the worker dies; or the scratch arena is out)
EB_DEV bool jump_pick(CaseCtx& c, const uint8_t* p, uint32_t n, const uint8_t*& d, uint32_t& dn) {
    WarpState* ws = c.ws; Rng& g = c.rng;
    const Rng saved = g;
    JumpCut cut = jump_cut(g, c.bp, n, 0xffffffffu);
    if (g.mode == 0) g.jump(cut.draws); else g.philox_skip((uint32_t)cut.draws);
    uint32_t rest = n - cut.pos;
    Blk tail; bool has_tail = finish_block(c, n, tail);
    if (ws->status != CASE_OK) return false;
    uint64_t nb = (uint64_t)cut.nfull + (rest ? 1 : 0) + (has_tail ? 1 : 0);
    if (nb == 0) { ws->status = CASE_DIED; return false; }   // rand_elem([]) is [], size([]) raises
    uint64_t k = g.erand(nb) - 1;
    if (k < cut.nfull) { JumpCut b = jump_cut(saved, c.bp, n, (uint32_t)k); d = p + b.at; dn = b.len; }
    else if (k == cut.nfull && rest) { d = p + cut.pos; dn = rest; }
    else { d = tail.p; dn = tail.len; }
    return true;
}
// jump_somewhere/2 :123-132: a block of each file, then S1, S2, L1, L2; the block list becomes the one block
// Data1[S1, S1+L1) ++ Data2[S2, S2+L2), materialised in scratch
EB_DEV void force_jump(CaseCtx& c) {
    WarpState* ws = c.ws; Rng& g = c.rng;
    // blockscale < 1/512: rand_block_size can be 0, and a zero-size block never ends the stream (the reference loops)
    if (c.bp->rbs_min == 0) { ws->status = CASE_UNSUPPORTED; ws->reason = 12; return; }
    const uint8_t *d1, *d2; uint32_t n1, n2;
    if (!jump_pick(c, ws->lz_p, ws->lz_n, d1, n1)) return;
    if (!jump_pick(c, ws->lz_p2, ws->lz_n2, d2, n2)) return;
    uint64_t s1 = g.rand(n1), s2 = g.rand(n2);
    uint64_t l1 = g.erand(n1 - s1), l2 = g.erand(n2 - s2);
    uint8_t* buf = scratch_alloc(c, l1 + l2);
    if (!buf) return;
    warp_copy(buf, d1 + s1, l1); warp_copy(buf + l1, d2 + s2, l2);
    __syncwarp();
    Blk b; b.p = buf; b.len = (uint32_t)(l1 + l2); b.cnt = 1; runs_push_back(ws, b);
}
// file / stdin generators (reference src/erlamsa_gen.erl:59-121): port_stream/2 returns an UNFORCED stream, so the blocks
// (stream_port/5: full blocks of the wanted size, a new rand_block_size after each, the short rest last) and the finish/1
// tail come into being at the pattern's first uncons/2 -- after the pattern's own first draws (SURVEY.md appendix A, W1'')
EB_DEV void force_stream(CaseCtx& c) {
    WarpState* ws = c.ws; Rng& g = c.rng; const BatchParams* bp = c.bp;
    if (!ws->lazy) return;
    ws->lazy = 0;
    if (bp->generator == 4) { force_jump(c); return; }
    const uint8_t* p = ws->lz_p; uint32_t n = ws->lz_n, pos = 0;
    uint64_t r0 = g.rand((uint64_t)bp->rbs_bound);
    uint32_t wanted = (uint32_t)(r0 > (uint64_t)bp->rbs_min ? r0 : (uint64_t)bp->rbs_min);
    while (n - pos >= wanted && ws->status == CASE_OK) {
        Blk b; b.p = p + pos; b.len = wanted; b.cnt = 1;
        // consecutive blocks of one size share a run
        if (ws->nruns > 0 && ws->runs[ws->nruns - 1].len == wanted && ws->runs[ws->nruns - 1].p + (uint64_t)wanted * ws->runs[ws->nruns - 1].cnt == b.p) ws->runs[ws->nruns - 1].cnt++;
        else runs_push_back(ws, b);
        pos += wanted;
        uint64_t r = g.rand((uint64_t)bp->rbs_bound);
        wanted = (uint32_t)(r > (uint64_t)bp->rbs_min ? r : (uint64_t)bp->rbs_min);
    }
    if (ws->status != CASE_OK) return;
    if (pos < n) { Blk b; b.p = p + pos; b.len = n - pos; b.cnt = 1; runs_push_back(ws, b); }
    finish_tail(c, n);
}
EB_DEV void generate(CaseCtx& c, const uint8_t* blob, uint32_t blen, const uint8_t* data, const uint64_t* off) {
    WarpState* ws = c.ws; Rng& g = c.rng; const BatchParams* bp = c.bp;
    ws->nruns = 0; ws->vhead = 0; ws->lazy = 0;
    if (bp->generator == 2 || bp->generator == 3) {
        if (bp->generator == 2) {   // file_streamer :106-121: the case picks its file, P = erand(N)
            uint64_t pi = g.erand(bp->n_blobs) - 1;
            blob = data + off[pi]; blen = (uint32_t)(off[pi + 1] - off[pi]);
        }
        ws->lazy = 1; ws->lz_p = blob; ws->lz_n = blen;
        return;
    }
    if (bp->generator == 4) {       // jump_streamer :135-150: P1, P2 = erand(N) now, the block at the first uncons
        uint64_t p1 = g.erand(bp->n_blobs) - 1, p2 = g.erand(bp->n_blobs) - 1;
        ws->lazy = 1;
        ws->lz_p = data + off[p1]; ws->lz_n = (uint32_t)(off[p1 + 1] - off[p1]);
        ws->lz_p2 = data + off[p2]; ws->lz_n2 = (uint32_t)(off[p2 + 1] - off[p2]);
        return;
    }
    if (bp->generator == 0) {   // direct_generator + finish
        (void)g.rand((uint64_t)bp->rbs_bound);
        Blk b; b.p = blob; b.len = blen; b.cnt = 1; runs_push_back(ws, b);
        uint64_t x = g.rand((uint64_t)blen + 1);
        if (x == blen) {
            uint64_t bits = (uint64_t)g.rand_range(1, 16);
            uint32_t nlen = (uint32_t)g.rand(1ull << bits);
            if (nlen) { const uint8_t* t = random_block_dev(c, nlen); if (t) { Blk tb; tb.p = t; tb.len = nlen; tb.cnt = 1; runs_push_back(ws, tb); } }
        }
    } else {                    // random_stream
        for (;;) {
            uint32_t n = (uint32_t)g.rand_range(32, (int64_t)bp->rbs_bound);
            const uint8_t* t = random_block_dev(c, n);
            if (!t || ws->status != CASE_OK) return;
            Blk tb; tb.p = t; tb.len = n; tb.cnt = 1; runs_push_back(ws, tb);
            if (ws->status != CASE_OK) return;
            uint64_t ip = (uint64_t)g.rand_range(1, 100);
            if (g.rand(ip) == 0) break;
        }
    }
}

// ------------------------------------------------------------------ sizer / checksum wrappers (patterns sz, cs)
// checksum of output bytes [from, olen) of the (virtual) output edit script
EB_DEV uint32_t oseg_checksum(CaseCtx& c, uint64_t from, bool crc) {
    WarpState* ws = c.ws; int l = lane_id();
    uint64_t pos = 0; uint32_t x = 0; uint32_t acc = 0;
    for (int k = 0; k < ws->noseg; k++) {
        Seg s = ws->oseg[k]; uint64_t b = pos, e = pos + s.len; pos = e;
        if (e <= from) continue;
        uint32_t o = b < from ? (uint32_t)(from - b) : 0; uint32_t len = s.len - o;
        if (!crc) {
            uint32_t y = 0;
            if (s.kind() == SEG_COPY) { const uint8_t* q = (const uint8_t*)(uintptr_t)s.src + o; for (uint32_t i = l; i < len; i += 32) y ^= q[i]; }
            else for (uint32_t i = l; i < len; i += 32) y ^= segs_byte(&s, 1, o + i);
            x ^= y;
        } else {
            uint32_t cs;
            if (s.kind() == SEG_COPY) cs = warp_crc32((const uint8_t*)(uintptr_t)s.src + o, len);
            else { uint32_t r = 0xffffffffu; for (uint32_t i = 0; i < len; i++) r = crc32_byte(r, segs_byte(&s, 1, o + i)); cs = ~r; }
            if (len) acc = crc_combine(acc, cs, len);
        }
    }
    if (crc) return acc;
    for (int o = 16; o; o >>= 1) x ^= __shfl_xor_sync(0xffffffffu, x, o);
    return x & 0xff;
}
// overwrite `nb` output bytes at offset `at` (a placeholder emitted earlier) with `bytes` (little-endian packed)
EB_DEV void oseg_patch(CaseCtx& c, uint64_t at, uint64_t bytes, uint32_t nb) {
    WarpState* ws = c.ws; uint64_t pos = 0;
    for (int k = 0; k < ws->noseg; k++) {
        Seg& s = ws->oseg[k]; uint64_t b = pos, e = pos + s.len; pos = e;
        if (at < b || at >= e) continue;
        if (s.kind() == SEG_INLINE && at == b && s.len == nb) { s.src = bytes; return; }
        if (s.kind() == SEG_COPY && at + nb <= e) {   // the script was folded into scratch meanwhile: patch the bytes in place
            uint8_t* q = (uint8_t*)(uintptr_t)s.src + (at - b);
            if ((uint32_t)lane_id() < nb) q[lane_id()] = (uint8_t)(bytes >> (8 * lane_id()));
            __syncwarp(); return;
        }
        ws->status = CASE_OVERFLOW; ws->reason = 10; return;
    }
}
// unwind innermost first: sz patches its length field with the size of everything emitted since, then emits the
// bytes that followed the blob; cs appends the checksum of the new blob (rebuild_blob / recalc_csum)
EB_DEV void unwind_wrappers(CaseCtx& c) {
    WarpState* ws = c.ws;
    while (ws->nwrap > 0 && ws->status == CASE_OK) {
        WarpState::Wrap w = ws->wrap[--ws->nwrap];
        if (w.kind == 1) {
            uint64_t newlen = ws->olen - w.mark;
            oseg_patch(c, w.field_pos, enc_field(newlen, w.bits, w.big != 0), w.bits / 8);
            o_push(c, seg_copy(w.tail_p, w.tail_n));
        } else {
            uint32_t v = oseg_checksum(c, w.mark, w.kind == 3);
            if (w.kind == 3) o_push(c, seg_inline(enc_field(v, 32, true), 4)); else o_push(c, seg_inline(v, 1));
        }
    }
}
EB_DEV bool looks_like_zip(const uint8_t* p, uint32_t n) {   // an end-of-central-directory signature anywhere
    uint32_t hit = 0;
    for (uint32_t i = lane_id(); i + 4 <= n; i += 32) hit |= (p[i] == 'P' && p[i + 1] == 'K' && p[i + 2] == 5 && p[i + 3] == 6) ? 1u : 0u;
    return __any_sync(0xffffffffu, hit != 0);
}
EB_DEV bool maybe_compressed(const uint8_t* p, uint32_t n) {   // gzip magic or a plausible zlib header
    if (n < 2) return false;
    uint32_t a = p[0], b = p[1];
    if (a == 0x1f && b == 0x8b) return true;
    return (a & 15) == 8 && (a >> 4) <= 7 && ((a << 8) | b) % 31 == 0;
}

// ------------------------------------------------------------------ pattern state machine
enum { CONT_OD = 0, CONT_ND = 1, CONT_BU = 2, CONT_PAT = 3 };

__host__ EB_DEV bool pat_supported(int id) { return id >= 0 && id < P_COUNT; }

// FULL false: od nd bu co nu only (the host never launches that flavour with another pattern selected)
template <bool FULL>
EB_DEV void run_case_machine(CaseCtx& c, int pat) {
    WarpState* ws = c.ws; Rng& g = c.rng;
    int cont = CONT_OD, next = 0;
    for (int guard = 0; guard < 100000 && ws->status == CASE_OK; guard++) {
        // ---- pattern dispatch
        uint64_t ip = 0;
        if (pat == P_NU) { force_stream(c); split_big(c); emit_all(c); return; }
        if (pat == P_CO) { if (g.erand(2) == 1) { force_stream(c); split_big(c); emit_all(c); return; } pat = P_OD; }
        if (pat == P_OD || pat == P_ND || pat == P_BU) {
            cont = pat == P_OD ? CONT_OD : pat == P_ND ? CONT_ND : CONT_BU;
            // mutate_once/4 :267-278
            if (!ws->lazy && active_is_single_empty(ws)) { ws->vhead = 0; ws->nruns = 0; return; }
            ip = g.rand(INITIAL_IP);
            force_stream(c);
            if (ws->status != CASE_OK) return;
            if (active_count(ws) == 0) {
                // an empty block list (an empty file without a finish/1 tail): mutate_once/4 hands [] to the continuation (:274-277).
                // od writes nothing; nd flips its coin and may come back here; bu would call the mutator on [] and then on the
                // binary it returns, which has no clause: the worker dies
                if (cont == CONT_OD) return;
                if (cont == CONT_ND) { if (g.rand_occurs_fixed(4, 5)) { pat = P_ND; continue; } return; }
                ws->status = CASE_DIED; return;
            }
            split_big(c);
        } else if (!FULL) { ws->status = CASE_UNSUPPORTED; return;
        } else if (pat == P_SK) {
            // make_complex_pat + mutate_once_skipper :148-161,352-361
            next = (int)g.rand_elem_idx(P_COUNT);
            ip = g.rand(INITIAL_IP);
            force_stream(c);
            if (ws->status != CASE_OK) return;
            if (active_count(ws) == 0) { ws->status = CASE_DIED; return; }
            realize_virtual(c);
            if (ws->status != CASE_OK) return;
            uint32_t n0 = ws->runs[0].len;
            uint32_t len = (uint32_t)g.rand((uint64_t)(n0 / 2));
            o_push(c, seg_copy(ws->runs[0].p, len));
            Blk tail; tail.p = ws->runs[0].p + len; tail.len = n0 - len; tail.cnt = 1;
            pop_head(ws); runs_insert_front(ws, tail);
            split_big(c);
            cont = CONT_PAT;
        } else if (pat == P_SZ || pat == P_CS) {
            // make_complex_pat + mutate_once_sizer :83-111 / mutate_once_csum :117-144
            next = (int)g.rand_elem_idx(P_COUNT);
            ip = g.rand(INITIAL_IP);
            force_stream(c);
            if (ws->status != CASE_OK) return;
            if (active_count(ws) == 0) { ws->status = CASE_DIED; return; }
            realize_virtual(c);
            if (ws->status != CASE_OK) return;
            const uint8_t* p0 = ws->runs[0].p; uint32_t n0 = ws->runs[0].len;
            temp_reset(c);
            if (ws->nwrap >= 8) { ws->status = CASE_OVERFLOW; ws->reason = 9; return; }
            WarpState::Wrap w; w.tail_p = nullptr; w.tail_n = 0; w.bits = 0; w.big = 0; w.field_pos = 0;
            bool found = false; uint32_t b0 = 0, bl = 0;
            if (pat == P_SZ) {
                Sizer e; found = lens_pick(c, p0, n0, e);
                if (found) {
                    uint32_t fb = e.size_bits / 8; b0 = e.a + fb; bl = (uint32_t)e.len;
                    o_push(c, seg_copy(p0, e.a));
                    w.kind = 1; w.bits = e.size_bits; w.big = e.big; w.field_pos = ws->olen;
                    o_push(c, seg_inline(0, fb));
                    w.tail_p = p0 + b0 + bl; w.tail_n = n0 - b0 - bl;
                }
            } else {
                Csum e; found = csum_pick(c, p0, n0, e);
                if (found) { b0 = e.plen; bl = e.blen; o_push(c, seg_copy(p0, e.plen)); w.kind = e.crc ? 3 : 2; }
            }
            if (ws->status != CASE_OK) return;
            if (found) {
                w.mark = ws->olen;
                EB_RECONVERGE();
                ws->wrap[ws->nwrap++] = w;
                Blk blob; blob.p = p0 + b0; blob.len = bl; blob.cnt = 1;
                pop_head(ws); runs_insert_front(ws, blob);
            }
            split_big(c);
            cont = CONT_PAT;
        } else if (pat == P_AR) {
            // mutate_once_archiver :167-214 on data that is not a ZIP archive: all blocks are glued into one
            next = (int)g.rand_elem_idx(P_COUNT);
            ip = g.rand(INITIAL_IP);
            force_stream(c);
            if (ws->status != CASE_OK) return;
            if (active_count(ws) == 0) { ws->status = CASE_DIED; return; }
            realize_virtual(c);
            if (ws->status != CASE_OK) return;
            if (active_count(ws) > 1) {
                uint64_t tot = 0; for (int i = 0; i < ws->nruns; i++) tot += (uint64_t)ws->runs[i].len * ws->runs[i].cnt;
                if (tot > c.bp->max_case_out) { ws->status = CASE_OVERFLOW; ws->reason = 5; return; }
                uint8_t* buf = scratch_alloc(c, tot);
                if (!buf) return;
                uint8_t* wq = buf;
                for (int i = 0; i < ws->nruns; i++) { uint64_t l = (uint64_t)ws->runs[i].len * ws->runs[i].cnt; warp_copy(wq, ws->runs[i].p, l); wq += l; }
                __syncwarp();
                ws->nruns = 0; Blk all; all.p = buf; all.len = (uint32_t)tot; all.cnt = 1; runs_push_back(ws, all);
            }
            if (looks_like_zip(ws->runs[0].p, ws->runs[0].len)) { ws->status = CASE_UNSUPPORTED; return; }
            split_big(c);
            cont = CONT_PAT;
        } else if (pat == P_CP) {
            // mutate_once_compressed :217-260 on data that is neither gzip nor zlib: plain mutate_once_loop
            next = (int)g.rand_elem_idx(P_COUNT);
            ip = g.rand(INITIAL_IP);
            force_stream(c);
            if (ws->status != CASE_OK) return;
            if (active_count(ws) == 0) { ws->status = CASE_DIED; return; }
            realize_virtual(c);
            if (ws->status != CASE_OK) return;
            if (maybe_compressed(ws->runs[0].p, ws->runs[0].len)) { ws->status = CASE_UNSUPPORTED; return; }
            split_big(c);
            cont = CONT_PAT;
        } else { ws->status = CASE_UNSUPPORTED; return; }
        if (ws->status != CASE_OK) return;
        // ---- mutate_once_loop :283-296
        for (;;) {
            uint64_t x = g.rand(ip);
            if (x == 0 || active_count(ws) == 1) break;
            emit_head(c);
            if (ws->status != CASE_OK) return;
        }
        mux_fuzzers<FULL>(c);
        if (ws->status != CASE_OK) return;
        g.set_slot((ws->round << 8) | SLOT_PATTERN);
        // ---- continuation
        if (cont == CONT_OD) { emit_all(c); return; }
        if (cont == CONT_ND) {
            if (g.rand_occurs_fixed(4, 5)) { pat = P_ND; continue; }
            emit_all(c); return;
        }
        if (cont == CONT_BU) {   // pat_burst_cont :332-343
            for (int nb = 1;; nb++) {
                bool pr = g.rand_occurs_fixed(4, 5);
                if (!(pr || nb < 2)) break;
                mux_fuzzers<FULL>(c);
                if (ws->status != CASE_OK) return;
                g.set_slot((ws->round << 8) | SLOT_PATTERN);
            }
            emit_all(c); return;
        }
        pat = next;   // CONT_PAT: the continuation pattern runs on the result list
    }
}

// ------------------------------------------------------------------ kernel
struct DecideArgs {
    const uint8_t* data; const uint64_t* off; Arenas ar;
    CaseOut* cases; uint64_t* out_len; uint64_t* out_sz16; MetaDev* meta;
    // single-pass (fused) mode
    int fused; uint8_t* out; uint64_t out_capacity; const uint64_t* slot_off; uint64_t* out_off;
    uint64_t ovf_base; unsigned long long* ovf_used; uint64_t data_bytes;
};
// case_list: a follow-up launch over the cases a previous launch had to flag for lack of arena space re-runs exactly
// those case numbers (same seeds, same slots; what outgrows the slot goes to the overflow region as before)
struct FusedArgs { int fused; uint8_t* out; uint64_t out_capacity; const uint64_t* slot_off; uint64_t* out_off; uint64_t ovf_base; unsigned long long* ovf_used; uint64_t data_bytes;
                   const uint32_t* case_list; uint64_t n_list; unsigned long long* case_counter; int deciders; int fronts; int front_depth; int tma_workers; };

// slot sizes for the single-pass mode: input length + slack, 16-byte aligned (the common mutations change a
// case by a few bytes; anything bigger spills to the overflow region). fixed != 0: every slot has that size (the jump
// generator, whose result is a slice of two blocks and has nothing to do with blob (I-1) mod n)
__global__ void __launch_bounds__(256) eb_slot_sizes(const uint64_t* __restrict__ off, uint64_t first_case, uint64_t n_blobs, uint64_t n_cases, uint64_t fixed, uint64_t* __restrict__ sz16) {
    uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_cases) return;
    if (fixed) { sz16[k] = fixed; return; }
    uint64_t b = (first_case - 1 + k) % n_blobs;
    uint64_t len = off[b + 1] - off[b];
    uint64_t slack = len / 16; if (slack < 256) slack = 256; if (slack > 65536) slack = 65536;
    sz16[k] = align16(len + slack);
}

#ifndef EB_CASE_THREADS
#define EB_CASE_THREADS 1024
#endif
constexpr int CASE_THREADS = EB_CASE_THREADS;   // threads per CTA = the register budget the per-case program is compiled for (64 at 1024)
constexpr int PW_BITS = 48;

// one test case, start to finish, decided by one warp (bulk byte work goes to the CTA's workers through q)
template <bool FULL>
EB_DEV void decide_one_case(WarpState* ws, const BatchParams& bp, const DecideArgs& a, uint64_t k, int32_t pa1, int32_t pa2, int32_t pa3, JobQ* q, uint32_t temp_slot) {
    const uint8_t* data = a.data; const uint64_t* off = a.off; const Arenas& ar = a.ar;
    CaseOut* cases = a.cases; uint64_t* out_len = a.out_len; uint64_t* out_sz16 = a.out_sz16; MetaDev* meta = a.meta;
    unsigned long long t_begin = 0;
    if (ar.case_usec) asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t_begin));
    {
        uint64_t I = bp.first_case + k;                 // the reference's 1-based case number
        uint64_t b = (I - 1) % bp.n_blobs;
        const uint8_t* blob = data + off[b]; uint32_t blen = (uint32_t)(off[b + 1] - off[b]);
        CaseCtx c; c.ws = ws; c.bp = &bp; c.ar = ar; c.q = q;
        c.temp_base = ar.temp ? ar.temp + (uint64_t)temp_slot * ar.temp_per_warp : nullptr;
        c.temp_used = 0; c.temp_floor = 0; c.snand_kind = bp.snand_kind;
        // thread seed: three erand(99999) at parent draw index 3*(I-1) (the caller keeps the parent state there)
        Rng par; par.mode = 0; par.a1 = pa1; par.a2 = pa2; par.a3 = pa3; par.draws = 0; par.key = 0; par.ctr_hi = 0;
        int64_t ts0 = (int64_t)par.erand(99999), ts1 = (int64_t)par.erand(99999), ts2 = (int64_t)par.erand(99999);
        c.rng.mode = bp.rng_mode; c.rng.key = bp.philox_key; c.rng.ctr_hi = I;
        c.rng.seed(ts0, ts1, ts2);
        ws->donor = (uint64_t)(ts0 * 31 + ts1 * 17 + ts2);
        ws->round = 0; c.rng.set_slot(SLOT_PATTERN);
        // fresh per-case state (CurMuta is not carried between cases, reference src/erlamsa_main.erl:223-235)
        ws->status = CASE_OK; ws->reason = 0; ws->n_used = 0; ws->n_failed = 0; ws->noseg = 0; ws->olen = 0;
        ws->st_n[0] = ws->st_n[1] = 0; ws->fo_has = 0; ws->nwrap = 0; ws->rrun_n = 0; ws->ntseg = 0; ws->tlen = 0; ws->nvseg = 0; ws->vlen = 0; ws->vchunked = 0;
        for (int i = 0; i < 16; i++) ws->used[i] = -1;
        ws->nrows = bp.n_rows;
        for (int i = 0; i < bp.n_rows; i++) { MutRow r; r.score = (double)bp.row_score[i]; r.pri = bp.row_pri[i]; r.name = bp.row_id[i]; r.fn = bp.row_id[i]; r.pad = 0; ws->rows[i] = r; }
        __syncwarp();
        generate(c, blob, blen, data, off);
        int pat = -1;
        if (ws->status == CASE_OK) {
            // mux_patterns :438-443 + choose_pri (reference src/erlamsa_utils.erl:155-160)
            int64_t x = (int64_t)c.rng.rand((uint64_t)bp.pat_sum);
            for (int i = 0; i < bp.n_pats; i++) { if (x == 0 || x < bp.pat_pri[i]) { pat = bp.pat_id[i]; break; } x -= bp.pat_pri[i]; }
            if (pat < 0) ws->status = CASE_DIED; else run_case_machine<FULL>(c, pat);
            if (FULL && ws->status == CASE_OK) unwind_wrappers(c);
        }
        if (ws->status == CASE_OK && ws->olen > bp.max_case_out) { ws->status = CASE_OVERFLOW; ws->reason = 5; }
        // a flagged case outputs its input unchanged -- except under jump, whose slots are not sized from the input: nothing
        if (ws->status == CASE_UNSUPPORTED || ws->status == CASE_OVERFLOW) { ws->noseg = 0; ws->olen = 0; if (bp.generator != 4) o_push(c, seg_copy(blob, blen)); }
        if (ws->status == CASE_DIED) { ws->noseg = 0; ws->olen = 0; }
        __syncwarp();
        unsigned long long sb = 0; int ns = ws->noseg;
        if (a.fused) {
            // single-pass mode: the output slot of case k was fixed before the kernel (prefix sum over INPUT sizes +
            // slack), so the warp that decided the case executes its edit script right away; results that outgrow
            // the slot go to the overflow region behind the slots
            uint64_t s0 = a.slot_off[k], cap = a.slot_off[k + 1] - s0;
            uint64_t dsto = s0;
            if (ws->olen > cap) {
                // bump allocation by compare-and-swap: the fill level only ever advances by GRANTED requests, so a
                // follow-up launch over the flagged cases continues exactly behind the bytes that are in use
                unsigned long long o = ~0ull, need = align16(ws->olen);
                if (lane_id() == 0) {
                    unsigned long long cur = *(volatile unsigned long long*)a.ovf_used;
                    while (a.ovf_base + cur + need <= a.out_capacity) {
                        unsigned long long prev = atomicCAS(a.ovf_used, cur, cur + need);
                        if (prev == cur) { o = cur; break; }
                        cur = prev;
                    }
                }
                o = __shfl_sync(0xffffffffu, o, 0);
                if (o == ~0ull) {   // no room: flag the case, emit the input unchanged (always fits its slot; jump: nothing)
                    if (lane_id() == 0) atomicOr(ar.overflow, 4u);
                    ws->status = CASE_OVERFLOW; ws->reason = 11; ws->noseg = 0; ws->olen = 0; if (bp.generator != 4) o_push(c, seg_copy(blob, blen)); ns = ws->noseg;
                } else dsto = a.ovf_base + o;
            }
            segs_write_stream(q, ws->oseg, ws->noseg, a.out + dsto, data, data + a.data_bytes);
            if (lane_id() == 0) { a.out_off[k] = dsto; out_len[k] = ws->olen; }
        } else {
            // two-pass mode: publish the edit script for the apply kernel
            if (lane_id() == 0 && ns > 0) sb = atomicAdd(ar.segs_used, (unsigned long long)ns);
            sb = __shfl_sync(0xffffffffu, sb, 0);
            if (sb + ns > ar.segs_cap) { if (lane_id() == 0) atomicOr(ar.overflow, 2u); ns = 0; ws->olen = 0; ws->status = CASE_OVERFLOW; ws->reason = 7; }
            for (int i = lane_id(); i < ns; i += 32) ar.segs[sb + i] = ws->oseg[i];
        }
        if (lane_id() == 0 && ws->status != CASE_OK && ar.flagged) atomicAdd(&ar.flagged[ws->status - 1], 1ull);
        if (lane_id() == 0) {
            if (ar.case_status) ar.case_status[k] = (uint8_t)(ws->status | (ws->reason << 4));
            if (ar.case_usec) { unsigned long long t_end; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t_end)); ar.case_usec[k] = (uint32_t)((t_end - t_begin) / 1000ull); }
            if (!a.fused) {
                CaseOut co; co.seg_begin = sb; co.nseg = (uint32_t)ns; co.status = ws->status; co.out_len = ws->olen; co.pad = 0;
                cases[k] = co; out_len[k] = ws->olen; out_sz16[k] = align16(ws->olen);
            }
            if (meta) {
                MetaDev m; m.pattern = pat; m.generator = bp.generator; m.n_used = ws->n_used; m.n_failed = ws->n_failed;
                for (int i = 0; i < 16; i++) m.used[i] = ws->used[i];
                m.draws = c.rng.draws; m.status = (int32_t)ws->status; m.pad = (int32_t)ws->reason; m.thread_seed[0] = ts0; m.thread_seed[1] = ts1; m.thread_seed[2] = ts2;
                meta[k] = m;
            }
        }
        __syncwarp();
    }
}

}  // namespace eb
