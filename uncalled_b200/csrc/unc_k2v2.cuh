// unc_k2v2.cuh -- the mapper's worker warps, second structure (included by unc_device.cuh).
//
// Same results as unc_k2_workers_exact (the first structure, the exact-ties kernels' worker): the reference's
// map_next (src/mapper.cpp:433-663) minus the seed clustering, which the tracker warp runs.  What changed
// is how an event's work is laid out on the CTA:
//
//   * FM index: a GPU-side Occ layout (DevIndex::occ2: 32-byte blocks = 4 x u32 cumulative counts + 64
//     two-bit BWT symbols, one sector per row) and ONE popcount sweep that yields Occ(k, c) for all four
//     bases, so that the warp executes the same instructions whichever bases its lanes want.
//   * extension: a lane owns a PARENT while thresholds and FM ranges are computed, then a CHILD while the
//     records are written (the chunk's children are staged in shared memory and re-dealt to the lanes), so
//     the record-writing code runs once per 32 children instead of five times per 32 parents.
//   * child sort: children sorted by fm_start are grouped by k-mer, and the k-mers' FM ranges are disjoint
//     and ordered (DevIndex::krank).  So the children are counted per k-mer during the extension, scattered
//     into k-mer buckets (one pass), and every bucket is sorted on its own by ONE warp: buckets of <= 32
//     keys by ranking in registers, larger ones by a warp-private LSD radix sort on the bits the bucket's
//     span needs.  No CTA-wide radix passes.
//   * dedup / gap sources / child seeds (src/mapper.cpp:527-603) work on k-mer runs, which are now exactly
//     the buckets: a warp walks its bucket with the run state in registers; the positions of the sources
//     and seeds come from one prefix sum over the buckets' counts.  No per-chunk aggregates, no look-back.
//   * 8 CTA barriers per event instead of ~20.
#pragma once

#define K2V2_STAGE_BYTES (K2_CH_SLOTS * 8u + K2_CH_SLOTS)   /* per worker warp: (start, end) + (lane | j<<5) of a chunk's children */

// ---- Occ for all four bases at once ------------------------------------------------------------------

// occ2 block j covers BWT positions [64j, 64j+64): counts of A,C,G,T before the block, then the 64 symbols
// (4 x u32, 16 symbols each, first symbol in the top two bits -- the .bwt file's own packing).
// Built from the bwa layout (submods/bwa/bwt.c:107-129: 128-position blocks of 4 x u64 counts + 8 x u32).
UNC_DEV void unc_occ2_build_block(const uint4 *bwt, u32 j, uint4 *out) {
    const uint4 *p = bwt + ((size_t) (j >> 1) << 2);
    const uint4 b0 = p[0], b1 = p[1];
    uint4 cnt = make_uint4(b0.x, b0.z, b1.x, b1.z);        // low words of the u64 counts
    const uint4 lo = p[2], hi = p[3];
    if (j & 1u) {
        const u32 w[4] = {lo.x, lo.y, lo.z, lo.w};
        for (int i = 0; i < 4; i++) {
            const u32 h = w[i] >> 1, m = 0x55555555u;
            const u32 c3 = (u32) d_popc(h & w[i] & m), c2 = (u32) d_popc(h & ~w[i] & m), c1 = (u32) d_popc(~h & w[i] & m);
            cnt.x += 16u - c1 - c2 - c3; cnt.y += c1; cnt.z += c2; cnt.w += c3;
        }
    }
    out[(size_t) j * 2] = cnt;
    out[(size_t) j * 2 + 1] = (j & 1u) ? hi : lo;
}

// Occ(., c) for c = 0..3 at position p (0..63, inclusive) of an occ2 block already in registers
UNC_DEV void unc_occ2_all(const uint4 cnt, const uint4 sym, u32 p, u32 o[4]) {
    u32 c1 = 0, c2 = 0, c3 = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const u32 w = i == 0 ? sym.x : i == 1 ? sym.y : i == 2 ? sym.z : sym.w;
        int n = (int) p + 1 - 16 * i;                       // symbols of this word at or before p
        n = n < 0 ? 0 : (n > 16 ? 16 : n);
        const u32 m = n == 0 ? 0u : (0x55555555u & (0xFFFFFFFFu << (32 - 2 * n)));
        const u32 h = w >> 1;
        c3 += (u32) d_popc(h & w & m); c2 += (u32) d_popc(h & ~w & m); c1 += (u32) d_popc(~h & w & m);
    }
    o[0] = cnt.x + (p + 1u - c1 - c2 - c3); o[1] = cnt.y + c1; o[2] = cnt.z + c2; o[3] = cnt.w + c3;
}

// ---- sort keys -----------------------------------------------------------------------------------------
// key = (fm_start, fm_end, seed_prob bits, seedable | move_count << 1 | k-mer's position in a merged group << 6 | record index << 14)
// order: fm_start, fm_end, seed_prob, record index (= emission order) -- reference src/mapper.cpp:866-871 plus
// the documented tie-break.  seed_prob is compared through a monotone integer image of the float so that the
// order is total whatever the bits are (a NaN cannot make two keys claim one rank); -0 counts as +0.
UNC_DEV u32 k2v2_fkey(u32 bits) {
    if (bits == 0x80000000u) bits = 0u;
    return (bits & 0x80000000u) ? ~bits : (bits | 0x80000000u);
}
UNC_DEV bool k2v2_less(u32 ax, u32 ay, u32 az, u32 aw, u32 bx, u32 by, u32 bz, u32 bw) {
    const u64 ha = ((u64) ax << 32) | ay, hb = ((u64) bx << 32) | by;
    const u64 la = ((u64) k2v2_fkey(az) << 32) | (aw >> 14), lb = ((u64) k2v2_fkey(bz) << 32) | (bw >> 14);
    return ha < hb || (ha == hb && la < lb);
}
// the same order on keys whose seed_prob word already holds k2v2_fkey(seed_prob) and whose w holds the record index only
UNC_DEV bool k2v2_less_pre(u32 ax, u32 ay, u32 af, u32 ar, u32 bx, u32 by, u32 bf, u32 br) {
    const u64 ha = ((u64) ax << 32) | ay, hb = ((u64) bx << 32) | by;
    const u64 la = ((u64) af << 32) | ar, lb = ((u64) bf << 32) | br;
    return ha < hb || (ha == hb && la < lb);
}

// One k-mer bucket [o, o+n) of `keys`, n > 32, sorted by ONE warp: LSD radix on (fm_start - lo) over the bits
// the bucket's span needs, then runs of equal fm_start ordered by (fm_end, seed_prob, record index).
// `tmp` is the ping-pong partner of `keys` (same index range), `hist` 256 warp-private counters.
// The sorted keys end in `keys`.
UNC_DEV
void k2v2_sort_big(uint4 *keys, uint4 *tmp, u32 o, u32 n, u32 lo, u32 span_bits, u32 *hist) {
    const int lane = w_lane();
    const u32 lt = w_lanemask_lt();
    const u32 npass = (span_bits + 7u) >> 3;
    uint4 *src = keys + o, *dst = tmp + o;
    const u32 nch = (n + 31u) >> 5;
    for (u32 pass = 0; pass < npass; pass++) {
        const u32 sb = pass * 8u;
        for (u32 b = (u32) lane; b < 256u; b += 32u) hist[b] = 0;
        w_sync();
        for (u32 c = 0; c < nch; c++) {
            const u32 g = c * 32u + (u32) lane;
            if (g < n) s_atomic_add(&hist[((src[g].x - lo) >> sb) & 255u], 1u);
        }
        w_sync();
        {   // exclusive scan of the 256 counters: 8 consecutive bins per lane
            u32 v[8], sum = 0;
#pragma unroll
            for (int i = 0; i < 8; i++) { v[i] = hist[(u32) lane * 8u + (u32) i]; sum += v[i]; }
            u32 tot, run = w_exscan(sum, &tot);
#pragma unroll
            for (int i = 0; i < 8; i++) { hist[(u32) lane * 8u + (u32) i] = run; run += v[i]; }
        }
        w_sync();
        for (u32 c = 0; c < nch; c++) {
            const u32 g = c * 32u + (u32) lane;
            const bool a = g < n;
            uint4 k = make_uint4(0, 0, 0, 0);
            if (a) k = src[g];
            const u32 dg = a ? (((k.x - lo) >> sb) & 255u) : 256u + (u32) lane;   // inactive lanes: unique digit
            const u32 peers = w_match(dg);
            const u32 rank = (u32) d_popc(peers & lt);
            const int leader = d_ffs(peers) - 1;
            u32 bpos = 0;
            if (a && lane == leader) { bpos = hist[dg]; hist[dg] = bpos + (u32) d_popc(peers); }
            w_sync();                              // the next chunk's leaders read these counters
            bpos = w_shfl(bpos, leader);
            if (a) dst[bpos + rank] = k;
        }
        w_sync();
        uint4 *t = src; src = dst; dst = t;
    }
    if (src != keys + o) {                          // odd number of passes: bring the keys home
        for (u32 g = (u32) lane; g < n; g += 32u) dst[g] = src[g];
        w_sync();
        src = keys + o;
    }
    // runs of equal fm_start: insertion sort by the run's head lane (rare and short)
    for (u32 c = 0; c < nch; c++) {
        const u32 g = c * 32u + (u32) lane;
        const bool a = g < n;
        u32 s = 0, px = 0, nx = 0;
        if (a) { s = src[g].x; if (g > 0) px = src[g - 1].x; if (g + 1 < n) nx = src[g + 1].x; }
        const bool head = a && (g == 0 || px != s) && (g + 1 < n && nx == s);
        if (head) {
            u32 e = g + 1;
            while (e < n && src[e].x == s) e++;
            for (u32 i = g + 1; i < e; i++) {
                const uint4 key = src[i];
                u32 j = i;
                while (j > g) {
                    const uint4 q = src[j - 1];
                    if (!k2v2_less(key.x, key.y, key.z, key.w, q.x, q.y, q.z, q.w)) break;
                    src[j] = q;
                    j--;
                }
                src[j] = key;
            }
        }
        w_sync();
    }
}

// What 32 consecutive lanes of sorted keys contribute to the dedup walk (reference src/mapper.cpp:527-603; the
// restatement's :1153-1194).  Every lane holds one key of some k-mer bucket (= one k-mer run); `head` marks the
// lanes where a bucket's keys start in this pass, `first` the first key of a bucket overall.
struct K2V2Walk {
    bool dup, begin_v, after_v, seed;
    u32 as, ae;          // the after-source's range
    u32 m_b, m_a, m_seed;
};
// cur = this lane's key, (nx, ny) = fm range of the key after it in the same bucket (valid iff has_next),
// kr / prob_ok = the bucket's k-mer range and whether the k-mer may get sources.  use_carry (uniform): all
// active lanes belong to one bucket that started in an earlier pass whose max fm_end so far is carry_mx.
// *mx_last = the running max at lane 31.
UNC_DEV K2V2Walk k2v2_walk(const uint4 cur, u32 nx, u32 ny, bool a, bool has_next, bool head, bool first, bool use_carry,
                           u32 carry_mx, bool prob_ok, uint2 kr, u32 *mx_last) {
    const int lane = w_lane();
    K2V2Walk r;
    r.dup = has_next && nx == cur.x && ny == cur.y;
    u32 mx = a ? cur.y : 0u;                          // segmented inclusive prefix max of fm_end
    bool hd = head || !a;
    for (int d = 1; d < 32; d <<= 1) {
        const u32 omx = w_shfl_up(mx, d), ohd = w_shfl_up(hd ? 1u : 0u, d);
        if (lane >= d && !hd) { mx = omx > mx ? omx : mx; hd = ohd != 0; }
    }
    if (use_carry) mx = mx > carry_mx ? mx : carry_mx;
    *mx_last = w_shfl(mx, 31);
    r.begin_v = a && first && prob_ok && kr.x <= cur.x - 1u;
    r.as = mx + 1u;
    r.ae = has_next ? nx - 1u : kr.y;
    r.after_v = a && !r.dup && prob_ok && r.as <= r.ae;
    r.seed = a && !r.dup && (cur.w & 1u);
    r.m_b = w_ballot(r.begin_v); r.m_a = w_ballot(r.after_v); r.m_seed = w_ballot(r.seed);
    return r;
}

// Small buckets (<= 32 keys) are handled several at a time: a PACK is a run of consecutive small buckets of one
// 32-rank group with at most 32 keys in all, one key per lane.
struct K2V2Pack {
    bool a;              // this lane holds a key
    u32 bl;              // lane (of the group) whose bucket the key belongs to
    u32 start, pos, n;   // first pack lane of that bucket, position of the key in it, its size
};
// cnt = size of this lane's bucket if it is a small one, else 0; P = exclusive prefix of cnt over the lanes;
// *remaining = lanes whose buckets are not packed yet (non-zero on entry)
UNC_DEV K2V2Pack k2v2_next_pack(u32 cnt, u32 P, u32 *remaining) {
    const int lane = w_lane();
    const int s = d_ffs(*remaining) - 1;
    const u32 Ps = w_shfl(P, s);
    const bool fits = ((*remaining >> lane) & 1u) && (P + cnt - Ps <= 32u);
    const u32 in_pack = w_ballot(fits);               // a prefix of `remaining` (P is non-decreasing); never empty
    *remaining &= ~in_pack;
    const int e = 31 - d_clz(in_pack);
    const u32 T = w_shfl(P + cnt, e) - Ps;
    K2V2Pack k;
    k.a = (u32) lane < T;
    k.bl = (u32) s; k.start = 0;
    u32 m = in_pack;
    while (m) {                                        // the last bucket that starts at or before this lane
        const int b = d_ffs(m) - 1;
        m &= m - 1;
        const u32 sb = w_shfl(P, b) - Ps;
        if ((u32) lane >= sb) { k.bl = (u32) b; k.start = sb; }
    }
    k.pos = (u32) lane - k.start;
    k.n = w_shfl(cnt, (int) k.bl);
    return k;
}
UNC_DEV u32 k2v2_segmask(u32 start, u32 n) { return (n >= 32u ? 0xFFFFFFFFu : ((1u << n) - 1u)) << start; }

// bucket rank -> index in the K2V2 per-bucket arrays: rank 32g + i sits at i*32 + g, so that a lane that owns 32
// consecutive ranks (the prefix sums) and a warp that reads one rank per lane... both touch distinct banks or one
UNC_DEV u32 k2v2_slot(u32 rank) { return ((rank & 31u) << 5) | (rank >> 5); }

// the next group of 32 bucket ranks for this warp (two sweeps of 32 groups: see phase C2)
UNC_DEV u32 k2v2_grab(u32 *counter) {
    u32 g = 0;
    if (w_lane() == 0) g = s_atomic_add(counter, 1u);
    return w_shfl(g, 0);
}

// <= 32 keys of one bucket sorted in place by one warp: every key ranked among the others, dealt out in order
UNC_DEV void k2v2_sort_small(uint4 *keys, u32 n, uint4 *sst) {
    const int lane = w_lane();
    const bool a = (u32) lane < n;
    uint4 k = make_uint4(0, 0, 0, 0);
    if (a) k = keys[lane];
    u32 rnk = 0;
    const u32 kf = k2v2_fkey(k.z), kr_ = k.w >> 14;
    for (u32 j = 0; j < n; j++) {
        const u32 jx = w_shfl(k.x, (int) j), jy = w_shfl(k.y, (int) j), jf = w_shfl(kf, (int) j), jr = w_shfl(kr_, (int) j);
        if (k2v2_less_pre(jx, jy, jf, jr, k.x, k.y, kf, kr_)) rnk++;
    }
    if (a) sst[rnk] = k;
    w_sync();
    if (a) keys[lane] = sst[lane];
    w_sync();
}

// The dedup walk over the sorted keys of a MERGED group's bucket (k-mers whose FM ranges overlap): the reference's
// loop statement by statement (src/mapper.cpp:527-603; the restatement's :1153-1194), by ONE lane -- the k-mer
// runs interleave here, so nothing about them is known in advance.  EMIT == false: count the bucket's gap sources
// and child seeds and note, per k-mer, how many sources precede its first run (D0 derives the sources_added_
// flags from that); EMIT == true: write the sources, order entries and seed rows at their final places.
struct K2V2Emit {
    uint4 *next; uint2 *hist_e; u32 *onext; uint2 *rlist;
    u32 S0, nc, maxp, n_ended_rows, rl_cap, pos0;      // pos0: sorted position of the bucket's first key
    u32 src_before, seeds_before;
};
// Called by the whole warp: the keys pass through the warp's staging area 32 at a time (a lane walking them straight
// from global memory pays two dependent loads per key: measured as the tail of both bucket phases), lane 0 walks.
template <bool EMIT>
UNC_DEV u32 k2v2_walk_merged(const DevIndex &ix, K2Shared *sh, const uint4 *keys, u32 n, u32 moff, float source_prob,
                             const K2V2Emit &E, u32 *pend_steps, u32 *pend_blocks, uint4 *sst) {
    K2V2 *v2 = &sh->v2;
    const u32 lane = (u32) w_lane();
    u32 nsrc = 0, nseed = 0, prev_sub = 0xFFFFFFFFu, un_st = 1, un_en = 0;      // the walk's state (lane 0)
  for (u32 g0 = 0; g0 < n; g0 += 32u) {
    const u32 cnt = n - g0 < 32u ? n - g0 : 32u;
    if (lane < cnt) sst[lane] = keys[g0 + lane];
    if (lane == 0 && g0 + cnt < n) sst[32] = keys[g0 + cnt];                     // the key after the window
    w_sync();
    if (lane == 0)
    for (u32 j = 0; j < cnt; j++) {
        const u32 i = g0 + j;
        const uint4 cur = sst[j];
        const u32 sub = (cur.w >> 6) & 0xFFu, kmer = v2->t.mk[moff + sub];
        const uint2 kr = sh->tb.kmer_range[kmer];
        const float pk = sh->probs[kmer];
        const bool ok = pk >= source_prob;
        if (sub != prev_sub) {
            if (!EMIT && v2->mfirst[moff + sub] == 0xFFFFu) v2->mfirst[moff + sub] = (u16) nsrc;
            if (ok) {
                if (kr.x <= cur.x - 1u) {
                    const u32 sidx = E.src_before + nsrc;
                    if (EMIT && E.nc + sidx < E.maxp) {
                        write_source(E.next, E.hist_e, E.S0 + E.nc + sidx, kr.x, cur.x - 1u, kmer, pk);
                        E.onext[E.nc + sidx] = E.S0 + E.nc + sidx;
                    }
                    nsrc++;
                }
                un_st = cur.y + 1u; un_en = kr.y;
            }
        }
        prev_sub = sub;
        const bool has_next = i + 1u < n;
        uint4 nxt = make_uint4(0, 0, 0, 0);
        if (has_next) nxt = sst[j + 1u];
        const bool dup = has_next && nxt.x == cur.x && nxt.y == cur.y;
        const u32 rec = cur.w >> 14;
        if (EMIT) E.onext[E.pos0 + i] = rec | (dup ? UNC_INVALID : 0u);
        if (dup) continue;
        if (ok) {
            u32 src_st = un_st, src_en = un_en;
            if (has_next && ((nxt.w >> 6) & 0xFFu) == sub) {
                src_en = nxt.x - 1u;
                if (un_st <= nxt.y) un_st = nxt.y + 1u;
            }
            if (src_st <= src_en) {
                const u32 sidx = E.src_before + nsrc;
                if (EMIT && E.nc + sidx < E.maxp) {
                    write_source(E.next, E.hist_e, E.S0 + E.nc + sidx, src_st, src_en, kmer, pk);
                    E.onext[E.nc + sidx] = E.S0 + E.nc + sidx;
                }
                nsrc++;
            }
        }
        if (cur.w & 1u) {
            if (EMIT) {
                d_atomic_or(&((u32 *) (E.next + (size_t) rec * 2))[3], 0x80000000u);   // sa_checked_
                const u32 ri = E.n_ended_rows + E.seeds_before + nseed;
                if (ri < E.rl_cap) E.rlist[ri] = make_uint2(ix.seq_len - unc_sa_lookup(ix, cur.x, pend_steps, pend_blocks), (cur.w >> 1) & 0x1Fu);
                else sh->wk_overflow = 1;
            }
            nseed++;
        }
    }
    w_sync();
  }
    return w_shfl(nsrc | (nseed << 16), 0);
}

// exclusive prefix of the bucket counts (one warp): lane i owns ranks 32i .. 32i+31 = slots j*32 + i
UNC_DEV void k2v2_bucket_offsets(K2V2 *v2) {
    const u32 lane = (u32) w_lane();
    u32 sum = 0;
#pragma unroll 1
    for (u32 j = 0; j < 32; j++) sum += v2->kcnt[j * 32u + lane];
    u32 tot, run = w_exscan(sum, &tot);
#pragma unroll 1
    for (u32 j = 0; j < 32; j++) {
        const u32 sl = j * 32u + lane, v = v2->kcnt[sl];
        v2->koff[sl] = run;
        v2->kcnt[sl] = run;                              // becomes the scatter cursor
        run += v;
    }
}

template <bool STREAM, bool FLAGS>
UNC_DEV void unc_k2_workers_v2(const DevIndex &ix, const DevParams &p, const DevBatch &B, const DevWork &W,
                               K2Shared *sh, u32 r, u32 n_first, u32 n_limit) {
    const int lane = w_lane();
    const u32 wt = (u32) c_tid() - 32u, nwt = (u32) c_nthreads() - 32u;   // worker thread index / count
    const u32 ww = wt >> 5, nwk = nwt >> 5;                               // worker warp index / count
    const K2Tables *tb = &sh->tb;
    K2V2 *v2 = &sh->v2;
    const u32 maxp = p.max_paths;
    const u32 S0 = ((maxp + 31u) >> 5) * K2_CH_SLOTS;                     // record index of the first source
    const size_t gen_recs = (size_t) S0 + maxp;
    const float scale = B.scale[r], shift = B.shift[r];
    const float *events = B.events + (size_t) r * B.ev_stride;
    const float source_prob = tb->thresh[0];
    u64 n_children = 0, n_sources = 0;                 // committed (events confirmed by the tracker)
    u32 pend_children = 0, pend_sources = 0;           // of the event in flight
    u32 my_blocks = 0, my_steps = 0, pend_blocks = 0, pend_steps = 0;
    u32 prev_size = 0, gen = 0, event_i = n_first;
    if (STREAM) {                                      // resume: the previous chunk's last generation is in the slot
        const DevMapState *ms = B.mstate + B.chan[r];
        if (ms->started) { prev_size = ms->prev_size; gen = ms->gen; }
    }
    const u32 lt = w_lanemask_lt();
    uint2 *stage_r = (uint2 *) (sh->v2_stage + (size_t) ww * K2V2_STAGE_BYTES);
    u8 *stage_m = (u8 *) (stage_r + K2_CH_SLOTS);
    u32 *whist = sh->hist_cur + (size_t) ww * 256u;    // warp-private radix counters (big buckets)
    PT_DECL
    PT_WDECL

    for (; event_i < n_limit; event_i++) {
        PT_MARK(9)
        const float event = f_add(f_mul(scale, events[event_i - n_first]), shift);
        PT_MARK(7)

        // ---- A. pore-model probabilities (reference src/mapper.cpp:443-445); clear the bucket counters
        if (FLAGS && wt < 32u) sh->flags_prev[wt] = sh->flags[wt];      // what the read ends with if this event is discarded
        for (u32 k = wt; k < UNC_NKMER; k += nwt) {
            sh->probs[k] = unc_match_prob(event, d_ldg(ix.lv_mean + k), d_ldg(ix.lv_var2 + k), d_ldg(ix.lognorm + k));
            v2->kcnt[k] = 0; v2->kagg[k] = 0;
        }
        for (u32 j = ww; j < 32; j += nwk) {              // k-mers that may get a fresh source (reference src/mapper.cpp:611-614)
            const u32 k = j * 32 + (u32) lane;
            const float pk = unc_match_prob(event, d_ldg(ix.lv_mean + k), d_ldg(ix.lv_var2 + k), d_ldg(ix.lognorm + k));
            const uint2 kr = tb->kmer_range[k];
            const u32 m = w_ballot(pk >= source_prob && kr.x <= kr.y);
            if (lane == 0) v2->fresh_cand[j] = m;
        }
        if (wt == 0) { v2->grab[0] = 0; v2->grab[1] = 0; v2->n_units = 0; }
        if (wt < K2V2_MAX_MERGED) v2->mfirst[wt] = 0xFFFFu;
        PT_MARK(0)
        c_sync_sub(1, (int) nwt);
        PT_FENCE
        PT_MARK(16)

        uint4 *prev = W.paths + (size_t) gen * gen_recs * 2, *next = W.paths + (size_t) (gen ^ 1u) * gen_recs * 2;
        uint2 *hist_e = W.hist + (size_t) (event_i % UNC_NGEN) * gen_recs;
        const u32 *oprev = W.order + (size_t) gen * maxp;
        u32 *onext = W.order + (size_t) (gen ^ 1u) * maxp;
        uint4 *ckA = W.ckey, *ckB = W.ckey + maxp, *cks = W.cks;
        uint2 *rlist = W.rlist + (size_t) (event_i & 1u) * W.rl_cap;

        // ---- B. extend every previous path (reference src/mapper.cpp:455-524): chunk c of 32 parents writes its
        //      children, in emission order, to records / keys [c*160, c*160+count)
        const u32 nch_prev = (prev_size + 31u) >> 5;
        {
            // software pipeline per warp: the order entry of chunk c+2*nwk is loaded (and its record line requested),
            // the record of chunk c+nwk is loaded (and the Occ block of its row start-1 requested), chunk c is consumed
            u32 oi_n = UNC_INVALID, oi_nn = UNC_INVALID; uint4 q0_n = make_uint4(0, 0, 0, 0); uint2 q1_n = make_uint2(0, 0);   // q1: (seed_prob, C)
            if (ww < nch_prev) {
                const u32 pi = ww * 32u + (u32) lane;
                if (pi < prev_size) oi_n = oprev[pi];
                if (!(oi_n & UNC_INVALID)) { const uint4 *pr = prev + (size_t) oi_n * 2; q0_n = pr[0]; q1_n = *(const uint2 *) (pr + 1); }
            }
            if (ww + nwk < nch_prev) {
                const u32 pi = (ww + nwk) * 32u + (u32) lane;
                if (pi < prev_size) oi_nn = oprev[pi];
                if (!(oi_nn & UNC_INVALID)) d_prefetch(prev + (size_t) oi_nn * 2);
            }
            for (u32 c = ww; c < nch_prev; c += nwk) {
                const u32 oi = oi_n;
                const uint4 q0 = q0_n; const uint2 q1 = q1_n;
                const bool valid = !(oi & UNC_INVALID);
                oi_n = oi_nn;
                if (c + nwk < nch_prev && !(oi_n & UNC_INVALID)) {
                    const uint4 *pr = prev + (size_t) oi_n * 2;
                    q0_n = pr[0]; q1_n = *(const uint2 *) (pr + 1);
                }
                oi_nn = UNC_INVALID;
                if (c + 2u * nwk < nch_prev) {
                    const u32 pi = (c + 2u * nwk) * 32u + (u32) lane;
                    if (pi < prev_size) oi_nn = oprev[pi];
                    if (!(oi_nn & UNC_INVALID)) d_prefetch(prev + (size_t) oi_nn * 2);
                }
                // -- parent per lane: thresholds, wanted bases, FM ranges of the four neighbours
                const u32 st = q0.x, en = q0.y, kmer = q0.z & UNC_KMASK, plen = (q0.z >> 16) & 0xFFu, stays = (q0.z >> 24) & 0xFFu;
                const u32 moves = q0.w & UNC_PATH_MASK, sa_checked = q0.w >> 31;
                u32 want = 0, cmask = 0;
                if (valid) {
                    const float thr = tb->thresh[32 + d_clz(en - st + 1u)];
                    if (stays < p.max_consec_stay && sh->probs[kmer] >= thr) cmask = 1u;
#pragma unroll
                    for (u32 b = 0; b < 4; b++)
                        if (!(sh->probs[((kmer << 2) & UNC_KMASK) | b] < thr)) want |= 1u << b;   // `if (prob < thresh) continue;`
                }
                if (cmask) stage_r[(u32) lane * 5u] = make_uint2(st, en);
                if (want) {
                    // BwaIndex::get_neighbor (reference src/bwa_index.hpp:158-162) over bwt_2occ (submods/bwa/bwt.c:132-163)
                    // for all four bases: ns = L2[c] + Occ(start-1, c) + 1, ne = L2[c] + Occ(end, c)
                    const u32 k0 = st - 1u, l0 = en;
                    const u32 kk = k0 - (k0 >= ix.primary), ll = l0 - (l0 >= ix.primary);
                    const bool l_is_end = (l0 == ix.seq_len);
                    const uint4 *bk = ix.occ2 + ((size_t) (kk >> 6) << 1);
                    const uint4 kc = d_ldg(bk), ks = d_ldg(bk + 1);
                    uint4 lc = kc, ls = ks;
                    if (!l_is_end && (ll >> 6) != (kk >> 6)) {
                        const uint4 *bl = ix.occ2 + ((size_t) (ll >> 6) << 1);
                        lc = d_ldg(bl); ls = d_ldg(bl + 1);
                    }
                    pend_blocks += 1u + ((!l_is_end && (ll >> 7) != (kk >> 7)) ? 1u : 0u);   // in the reference's 128-row blocks
                    u32 ok[4], ol[4];
                    unc_occ2_all(kc, ks, kk & 63u, ok);
                    unc_occ2_all(lc, ls, ll & 63u, ol);
                    if (l_is_end) { ol[0] = ix.L2[1] - ix.L2[0]; ol[1] = ix.L2[2] - ix.L2[1]; ol[2] = ix.L2[3] - ix.L2[2]; ol[3] = ix.L2[4] - ix.L2[3]; }
                    // a valid child's range goes to the parent's fixed staging slot lane*5 + 1 + base at once
#pragma unroll
                    for (u32 b = 0; b < 4; b++) {
                        const u32 nsb = ix.L2[b] + ok[b] + 1u, neb = ix.L2[b] + ol[b];
                        if (((want >> b) & 1u) && nsb <= neb) { cmask |= 2u << b; stage_r[(u32) lane * 5u + 1u + b] = make_uint2(nsb, neb); }
                    }
                }
                const u32 cc = (u32) d_popc(cmask);
                u32 total;
                const u32 off = w_exscan(cc, &total);
                // a childless, not yet SA-checked path may end here with seeds
                // (reference src/mapper.cpp:513-519 -> update_seeds(path, true), is_seed_valid :842-863)
                bool ended = false;
                const u32 mc = (u32) d_popc(moves);
                if (valid && cc == 0 && !sa_checked) {
                    const u32 len = en - st + 1u;
                    ended = plen == UNC_SEED_LEN && u2f(q1.x) >= p.min_seed_prob &&
                            ((len == 1 && (moves & 1u) && (float) ((plen - mc) & 0xFFu) <= f_mul(p.max_stay_frac, 22.0f)) ||
                             (len <= p.max_rep_copy && mc >= p.min_rep_len));
                }
                const u32 m_ended = w_ballot(ended);
                if (ended) W.elist[(size_t) c * 32 + (u32) d_popc(m_ended & lt)] = make_uint4(st, en, mc, off);
                if (lane == 0) { sh->bcnt[c] = total; sh->ecnt[c] = (u32) d_popc(m_ended); }
                // -- the chunk's children in emission order: (parent lane | child index << 5), then one child per lane
                {
                    u32 pos = off;
#pragma unroll
                    for (u32 j = 0; j < 5; j++)
                        if ((cmask >> j) & 1u) { stage_m[pos] = (u8) ((u32) lane | (j << 5)); pos++; }
                }
                w_sync();
                for (u32 t0 = 0; t0 < total; t0 += 32u) {
                    const u32 t = t0 + (u32) lane;
                    const bool act = t < total;
                    u32 m = 0; uint2 rg = make_uint2(0, 0);
                    if (act) { m = stage_m[t]; rg = stage_r[(m & 31u) * 5u + (m >> 5)]; }
                    const int L = (int) (m & 31u);
                    const u32 j = m >> 5;                                         // 0 = stay, 1..4 = move with base j-1
                    const u32 pz = w_shfl(q0.z, L), pw = w_shfl(q0.w, L), pC = w_shfl(q1.y, L), poi = w_shfl(oi, L);
                    if (act) {
                        const u32 pk = pz & UNC_KMASK, ppl = (pz >> 16) & 0xFFu, pst = (pz >> 24) & 0xFFu;
                        const u32 ckm = j == 0 ? pk : (((pk << 2) & UNC_KMASK) | (j - 1u));
                        const float pb = sh->probs[ckm];
                        const u32 move = j > 0 ? 1u : 0u;
                        const u32 nlen = ppl + (ppl < UNC_SEED_LEN ? 1u : 0u);
                        u32 nmoves = (((pw & UNC_PATH_MASK) << 1) | move) & UNC_PATH_MASK;
                        const u32 nstays = move ? 0u : pst + 1u;
                        const float newC = f_add(u2f(pC), pb);
                        const u32 ci = c * K2_CH_SLOTS + t;
                        float sp = 0.0f;
                        bool seedable = false;
                        if (ppl == UNC_SEED_LEN) {
                            // seed_prob = (C(e) - C(e-22)) / 22 needs the ancestor 22 generations back: deferred
                            nmoves |= UNC_PATH_TAIL;
                            W.wlist[s_atomic_add(&sh->wl_cnt, 1u)] = make_uint4(ci, poi, f2u(newC), nmoves);
                        } else {
                            sp = f_div(newC, (float) nlen);
                            // is_seed_valid(path_ended = false) of the child (reference src/mapper.cpp:842-863)
                            const u32 cmc = (u32) d_popc(nmoves);
                            seedable = nlen == UNC_SEED_LEN && sp >= p.min_seed_prob && rg.x == rg.y && (nmoves & 1u) &&
                                       (float) ((nlen - cmc) & 0xFFu) <= f_mul(p.max_stay_frac, 22.0f);
                        }
                        const u32 spb = f2u(sp);
                        next[(size_t) ci * 2] = make_uint4(rg.x, rg.y, ckm | (nlen << 16) | (nstays << 24), nmoves | (pw & 0x80000000u));
                        next[(size_t) ci * 2 + 1] = make_uint4(spb, f2u(newC), 0u, 0u);
                        hist_e[ci] = make_uint2(f2u(newC), poi);
                        cks[ci] = make_uint4(rg.x, rg.y, spb, ckm | (seedable ? 1u << 10 : 0u) | ((u32) d_popc(nmoves) << 11));
                        s_atomic_add(&v2->kcnt[v2->t.kslot[ckm]], 1u);
                    }
                }
                if (c + nwk < nch_prev && !(oi_n & UNC_INVALID)) {      // the next chunk's Occ block (row start-1), requested early
                    const u32 k0n = q0_n.x - 1u;
                    d_prefetch(ix.occ2 + ((size_t) ((k0n - (k0n >= ix.primary)) >> 6) << 1));
                }
                w_sync();                                       // the staging area is rewritten by the next chunk
            }
        }
        PT_MARK(1)
        c_sync_sub(1, (int) nwt);
        PT_FENCE
        PT_MARK(17)
        // ---- B1 + B2a + B2b, concurrently.  Worker warp 0: exclusive scan of the chunk counts (restores the
        //      global emission order and gives the buffer cap, reference src/mapper.cpp:480-482,507-509,521-523:
        //      extension stops when max_paths children exist), then the seed rows of ended paths.  The last worker
        //      warp: bucket offsets.  The others: deferred seed_prob of children whose parent was already seed_len
        //      long -- C(e-22) is the C of the ancestor 22 generations back (21 parent hops from the parent).
        if (ww == 0) {
            {   // every lane owns a run of consecutive chunks: its sum, one warp scan, its running prefix
                const u32 per = (nch_prev + 31u) >> 5, c_lo = (u32) lane * per, c_hi = c_lo + per < nch_prev ? c_lo + per : nch_prev;
                u32 sum = 0;
#pragma unroll 1
                for (u32 c = c_lo; c < c_hi; c++) sum += sh->bcnt[c];
                u32 tot, run = w_exscan(sum, &tot);
#pragma unroll 1
                for (u32 c = c_lo; c < c_hi; c++) { const u32 v = sh->bcnt[c]; sh->bcnt[c] = run; run += v; }
                if (lane == 0) sh->bc[2] = tot;
            }
            w_sync();
            // seed rows of ended paths, in parent order.  A parent counts only if the buffer was not yet full when
            // the sequential scan reached it (children before it < max_paths).
            u32 rows = 0;
            for (u32 i0 = 0; i0 < nch_prev; i0 += 32) {
                u32 ec = i0 + (u32) lane < nch_prev ? sh->ecnt[i0 + lane] : 0u;
                u32 m = w_ballot(ec != 0);
                while (m) {
                    int l = d_ffs(m) - 1;
                    m &= m - 1;
                    u32 c = i0 + (u32) l, n = w_shfl(ec, l), base = sh->bcnt[c];
                    for (u32 j = 0; j < n; j++) {
                        uint4 e = W.elist[(size_t) c * 32 + j];
                        if (base + e.w < maxp) {
                            u32 len = e.y - e.x + 1u;
                            if (rows + len <= W.rl_cap) {
                                for (u32 i = (u32) lane; i < len; i += 32) rlist[rows + i] = make_uint2(e.x + i, e.z | 0x100u);
                            } else sh->wk_overflow = 1;
                            rows += len;
                        }
                    }
                }
            }
            if (lane == 0) sh->bc[3] = rows;
        }
        if (ww == nwk - 1u) {
            // bucket offsets, assuming the buffer cap does not cut this event's children (else redone below)
            k2v2_bucket_offsets(v2);
        }
        if (ww != 0 || nwk == 1) {
            const u32 bt = nwk == 1 ? wt : wt - 32u, nbt = nwk == 1 ? nwt : nwt - 32u;
            const u32 nwl = *(volatile u32 *) &sh->wl_cnt;
            for (u32 i = bt; i < nwl; i += nbt) {
                uint4 w = W.wlist[i];
                u32 idx = w.y;
                for (u32 j = 1; j <= 21; j++)
                    idx = W.hist[(size_t) ((event_i + UNC_NGEN - j) % UNC_NGEN) * gen_recs + idx].y;
                float oldC = u2f(W.hist[(size_t) ((event_i + UNC_NGEN - 22u) % UNC_NGEN) * gen_recs + idx].x);
                float sp = f_div(f_sub(u2f(w.z), oldC), 22.0f);
                uint4 key = cks[w.x];
                u32 cmc = (u32) d_popc(w.w);
                bool seedable = sp >= p.min_seed_prob && key.x == key.y && (w.w & 1u) &&
                                (float) ((UNC_SEED_LEN - cmc) & 0xFFu) <= f_mul(p.max_stay_frac, 22.0f);
                key.z = f2u(sp);
                if (seedable) key.w |= 1u << 10;
                cks[w.x] = key;
                next[(size_t) w.x * 2 + 1].x = f2u(sp);
            }
        }
        PT_MARK(10)
        c_sync_sub(1, (int) nwt);
        PT_FENCE
        PT_MARK(26)
        if (wt == 0) sh->wl_cnt = 0;
        const u32 nc_total = nch_prev ? sh->bc[2] : 0u;
        const u32 nc = nc_total < maxp ? nc_total : maxp;
        if (nc_total > maxp) {
            // the cap cut the children (chunk order = emission order): take the dropped ones -- emission index >= max_paths,
            // all in the last chunks -- out of the bucket counts instead of counting everything again.  kagg is still zero.
            for (u32 c = ww; c < nch_prev; c += nwk) {
                const u32 base = sh->bcnt[c], end = c + 1 < nch_prev ? sh->bcnt[c + 1] : nc_total;
                if (end <= nc) continue;
                for (u32 i = (base < nc ? nc - base : 0u) + (u32) lane; base + i < end; i += 32)
                    s_atomic_add(&v2->kagg[v2->t.kslot[cks[(size_t) c * K2_CH_SLOTS + i].w & UNC_KMASK]], 1u);
            }
            c_sync_sub(1, (int) nwt);
            if (ww == 0) {
                // counts = differences of the offsets the optimistic scan left, minus the dropped; then the offsets again
                const u32 l = (u32) lane;
#pragma unroll 1
                for (u32 j = 0; j < 32; j++) {
                    const u32 sl = j * 32u + l;                                         // rank 32*l + j
                    const u32 nxt = j < 31u ? v2->koff[sl + 32u] : (l < 31u ? v2->koff[l + 1u] : nc_total);
                    v2->kcnt[sl] = nxt - v2->koff[sl] - v2->kagg[sl];
                    v2->kagg[sl] = 0;
                }
                w_sync();
                k2v2_bucket_offsets(v2);
            }
            c_sync_sub(1, (int) nwt);
        }
        PT_MARK(12)
        u32 n_rows = sh->bc[3];
        if (n_rows > W.rl_cap) n_rows = W.rl_cap;
        const u32 n_ended_rows = n_rows;
        pend_children = nc;

        if (nc > 0) {
            // ---- C1. scatter the keys into their k-mer buckets (any order inside a bucket: the record index is
            //          part of the key); each warp takes the chunks it extended
            uint4 kpre = make_uint4(0, 0, 0, 0);                     // the first 32 keys of the warp's next chunk, requested early
            if (ww < nch_prev) {
                const u32 b0 = sh->bcnt[ww], e0 = ww + 1 < nch_prev ? sh->bcnt[ww + 1] : nc_total;
                if (b0 + (u32) lane < e0 && b0 + (u32) lane < nc) kpre = cks[(size_t) ww * K2_CH_SLOTS + (u32) lane];
            }
            for (u32 c = ww; c < nch_prev; c += nwk) {
                const u32 base = sh->bcnt[c];
                if (base >= nc) break;                              // later chunks lie beyond the max_paths cut
                const u32 end = c + 1 < nch_prev ? sh->bcnt[c + 1] : nc_total;
                const uint4 kcur = kpre;
                if (c + nwk < nch_prev) {
                    const u32 bn = sh->bcnt[c + nwk], en = c + nwk + 1 < nch_prev ? sh->bcnt[c + nwk + 1] : nc_total;
                    if (bn + (u32) lane < en && bn + (u32) lane < nc) kpre = cks[(size_t) (c + nwk) * K2_CH_SLOTS + (u32) lane];
                }
                for (u32 i = (u32) lane; base + i < end && base + i < nc; i += 32) {
                    const u32 ci = c * K2_CH_SLOTS + i;
                    uint4 key = i < 32u ? kcur : cks[ci];
                    const u32 km = key.w & UNC_KMASK;
                    const u32 bk = v2->t.kslot[km];
                    key.w = ((key.w >> 10) & 0x3Fu) | ((u32) v2->t.ksub[km] << 6) | (ci << 14);   // seedable | move_count << 1 | sub << 6 | record index << 14
                    ckA[s_atomic_add(&v2->kcnt[bk], 1u)] = key;
                }
            }
            PT_MARK(2)
            c_sync_sub(1, (int) nwt);
            PT_FENCE
            PT_MARK(18)
            PT_WB

            // ---- C2. sort every bucket and count what its dedup walk will emit.  Buckets are handed out 32 ranks (one
            //          group) at a time: first sweep the large buckets (> 32 keys, one warp each, radix), second sweep
            //          the small ones, packed several to a warp pass.
            uint4 *csum = W.elist;                                     // per 32-key chunk of a large bucket: what D1 needs to take it alone
            for (;;) {
                const u32 gi = k2v2_grab(&v2->grab[0]);
                if (gi >= 96u) break;
                const u32 grp = gi & 31u;
                const u32 sl = (u32) lane * 32u + grp;                 // slot of rank 32*grp + lane
                const u32 bo = v2->koff[sl], bn = v2->kcnt[sl] - bo;
                const u32 meta = v2->t.gmeta[grp * 32u + (u32) lane];
                if (gi < 64u) {
                    // sweeps 0 and 1: the largest buckets (> 256 keys) start first, then the other large ones (longest job first)
                    const bool huge_sweep = gi < 32u;
                    u32 todo_m = huge_sweep ? w_ballot(meta != 0 && bn > 0) : 0u;
                    while (todo_m) {                                  // merged groups: sort, then one lane walks the bucket
                        const int l = d_ffs(todo_m) - 1;
                        todo_m &= todo_m - 1;
                        const u32 o = w_shfl(bo, l), n = w_shfl(bn, l), moff = w_shfl(meta, l) >> 8;
                        if (n <= 32u) k2v2_sort_small(ckA + o, n, (uint4 *) stage_r);
                        else {
                            u32 lo = 0xFFFFFFFFu, hi = 0;
                            for (u32 g = (u32) lane; g < n; g += 32u) { const u32 x = ckA[o + g].x; lo = x < lo ? x : lo; hi = x > hi ? x : hi; }
                            hi = w_max(hi);
                            lo = ~w_max(~lo);
                            k2v2_sort_big(ckA, ckB, o, n, lo, 32u - (u32) d_clz(hi - lo), whist);
                        }
                        {
                            K2V2Emit E;
                            E.src_before = 0; E.seeds_before = 0;
                            const u32 agg = k2v2_walk_merged<false>(ix, sh, ckA + o, n, moff, source_prob, E, &pend_steps, &pend_blocks, (uint4 *) stage_r);
                            if (lane == 0) v2->kagg[(u32) l * 32u + grp] = agg;
                        }
                    }
                    u32 todo = w_ballot(meta == 0 && (huge_sweep ? bn > 256u : (bn > 32u && bn <= 256u)));
                    while (todo) {
                        const int l = d_ffs(todo) - 1;
                        todo &= todo - 1;
                        const u32 o = w_shfl(bo, l), n = w_shfl(bn, l);
                        const u32 kmer = v2->t.gkmer[grp * 32u + (u32) l];
                        u32 ubase = 0;                                 // this bucket's chunks in the unit list
                        if (lane == 0) ubase = s_atomic_add(&v2->n_units, (n + 31u) >> 5);
                        ubase = w_shfl(ubase, 0);
                        const uint2 kr = tb->kmer_range[kmer];
                        const bool prob_ok = sh->probs[kmer] >= source_prob;
                        // span of the bucket's fm_start values -> radix passes
                        u32 lo = 0xFFFFFFFFu, hi = 0;
                        for (u32 g = (u32) lane; g < n; g += 32u) { const u32 x = ckA[o + g].x; lo = x < lo ? x : lo; hi = x > hi ? x : hi; }
                        hi = w_max(hi);
                        lo = ~w_max(~lo);
                        k2v2_sort_big(ckA, ckB, o, n, lo, 32u - (u32) d_clz(hi - lo), whist);
                        u32 carry_mx = 0, n_src = 0, n_seed = 0;
                        for (u32 g0 = 0; g0 < n; g0 += 32u) {
                            const u32 g = g0 + (u32) lane;
                            const bool a = g < n, has_next = g + 1u < n;
                            uint4 cur = make_uint4(0, 0, 0, 0); u32 nx = 0, ny = 0;
                            if (a) cur = ckA[o + g];
                            if (has_next) { const uint4 t = ckA[o + g + 1u]; nx = t.x; ny = t.y; }
                            // the chunk as a unit of the emit phase: max fm_end and the bucket's counts before it, bucket slot | chunk
                            if (lane == 0) csum[ubase + (g0 >> 5)] = make_uint4(carry_mx, n_src, n_seed, ((u32) l * 32u + grp) | ((g0 >> 5) << 10));
                            u32 mxo;
                            const K2V2Walk wk = k2v2_walk(cur, nx, ny, a, has_next, g == 0, g == 0, g0 != 0, carry_mx, prob_ok, kr, &mxo);
                            carry_mx = mxo;
                            n_src += (u32) d_popc(wk.m_b) + (u32) d_popc(wk.m_a);
                            n_seed += (u32) d_popc(wk.m_seed);
                        }
                        if (lane == 0) v2->kagg[(u32) l * 32u + grp] = n_src | (n_seed << 16);
                    }
                } else {
                    const u32 cnt = (bn > 0 && bn <= 32u && meta == 0) ? bn : 0u;
                    u32 tot;
                    const u32 P = w_exscan(cnt, &tot);
                    u32 remaining = w_ballot(cnt != 0);
                    while (remaining) {
                        const K2V2Pack pk = k2v2_next_pack(cnt, P, &remaining);
                        const u32 addr = w_shfl(bo, (int) pk.bl) + pk.pos;
                        uint4 k = make_uint4(0, 0, 0, 0);
                        if (pk.a) k = ckA[addr];
                        // rank every key among the keys of its bucket, deal the keys out in sorted order
                        const u32 maxn = w_max(pk.a ? pk.n : 0u);
                        u32 rnk = 0;
                        const u32 kf = k2v2_fkey(k.z), kri = k.w >> 14;
                        for (u32 q = 0; q < maxn; q++) {
                            const int src = (int) ((pk.start + q) & 31u);
                            const u32 jx = w_shfl(k.x, src), jy = w_shfl(k.y, src), jf = w_shfl(kf, src), jr = w_shfl(kri, src);
                            if (pk.a && q < pk.n && k2v2_less_pre(jx, jy, jf, jr, k.x, k.y, kf, kri)) rnk++;
                        }
                        uint4 *sst = (uint4 *) stage_r;
                        if (pk.a) sst[pk.start + rnk] = k;
                        w_sync();
                        uint4 cur = make_uint4(0, 0, 0, 0);
                        if (pk.a) { cur = sst[lane]; ckA[addr] = cur; }
                        w_sync();
                        const u32 nx = w_shfl_down(cur.x, 1), ny = w_shfl_down(cur.y, 1);
                        const u32 kmer = v2->t.gkmer[grp * 32u + pk.bl];
                        const uint2 kr = tb->kmer_range[kmer];
                        const bool prob_ok = sh->probs[kmer] >= source_prob;
                        u32 mxo;
                        const K2V2Walk wk = k2v2_walk(cur, nx, ny, pk.a, pk.a && pk.pos + 1u < pk.n, pk.pos == 0, pk.pos == 0, false, 0u,
                                                      prob_ok, kr, &mxo);
                        const u32 sm = k2v2_segmask(pk.start, pk.n);
                        if (pk.a && pk.pos == 0)
                            v2->kagg[pk.bl * 32u + grp] = ((u32) d_popc(wk.m_b & sm) + (u32) d_popc(wk.m_a & sm)) | ((u32) d_popc(wk.m_seed & sm) << 16);
                    }
                }
            }
            PT_WE(1)
            PT_MARK(3)
            c_sync_sub(1, (int) nwt);
            PT_FENCE
            PT_MARK(19)
            PT_WR(1, 15, 20)
        }

        // ---- D0 + S1, concurrently.  Worker warp 0: prefix sum of the buckets' (sources, seeds), the sources_added_
        //      flags the run starts set (reference src/mapper.cpp:560-562), and the plan of the fresh sources
        //      (reference :605-624).  The other warps: suffix-array look-ups of the ended paths' seed rows
        //      (reference :673-681: sa_end = fmi.size() - fmi.sa(s)).
        if (ww == 0) {
            // lane i owns ranks 32i .. 32i+31 (slots j*32 + i): its sum, a warp scan of the sums, its running prefix
            u32 sum = 0;
#pragma unroll 1
            for (u32 j = 0; j < 32; j++) sum += v2->kagg[j * 32u + (u32) lane];
            u32 ts, tq;
            const u32 es = w_exscan(sum & 0xFFFFu, &ts), eq = w_exscan(sum >> 16, &tq);
            u32 run = es | (eq << 16);                       // sources | seeds << 16 before the bucket
#pragma unroll 1
            for (u32 j = 0; j < 32; j++) {
                const u32 sl = j * 32u + (u32) lane, v = v2->kagg[sl];
                v2->kagg[sl] = run;
                // sources_added_[kmer] is set at a run start while the buffer is not full
                if (nc > 0 && v2->kcnt[sl] != v2->koff[sl]) {
                    const u32 meta = v2->t.gmeta[(u32) lane * 32u + j];
                    if (meta == 0) {
                        const u32 kmer = v2->t.gkmer[(u32) lane * 32u + j];
                        if (sh->probs[kmer] >= source_prob && nc + (run & 0xFFFFu) < maxp) s_atomic_or(&sh->flags[kmer >> 5], 1u << (kmer & 31u));
                    } else {
                        for (u32 m = 0; m < (meta & 0xFFu); m++) {        // every k-mer of the merged group that has a run
                            const u32 f = v2->mfirst[(meta >> 8) + m], kmer = v2->t.mk[(meta >> 8) + m];
                            if (f != 0xFFFFu && sh->probs[kmer] >= source_prob && nc + (run & 0xFFFFu) + f < maxp)
                                s_atomic_or(&sh->flags[kmer >> 5], 1u << (kmer & 31u));
                        }
                    }
                }
                run = ((run & 0xFFFFu) + (v & 0xFFFFu)) | (((run >> 16) + (v >> 16)) << 16);
            }
            w_sync();
            const u32 tot_src = ts;
            const u32 ns_added = nc + tot_src > maxp ? maxp - nc : tot_src;
            const u32 nn0 = nc + ns_added;
            const u32 my_mask = v2->fresh_cand[lane] & ~sh->flags[lane];   // word `lane` of the fresh-source walk
            u32 tot_add;
            const u32 my_pre = w_exscan((u32) d_popc(my_mask), &tot_add);
            v2->fresh_mask[lane] = my_mask;
            v2->fresh_before[lane] = nn0 + my_pre;           // fill level when the serial walk reaches word `lane`
            if (lane == 0) {
                sh->bc[1] = nn0 + tot_add < maxp ? nn0 + tot_add : maxp;
                sh->bc[6] = tq;
            }
        }
        if (ww != 0 || nwk == 1) {
            const u32 bt = nwk == 1 ? wt : wt - 32u, nbt = nwk == 1 ? nwt : nwt - 32u;
            for (u32 i = bt; i < n_ended_rows; i += nbt) {
                uint2 e = rlist[i];
                e.x = ix.seq_len - unc_sa_lookup(ix, e.x, &pend_steps, &pend_blocks);
                rlist[i] = e;
            }
        }
        PT_MARK(11)
        c_sync_sub(1, (int) nwt);
        PT_FENCE
        PT_MARK(27)
        PT_WB
        const u32 n_child_seeds = nc > 0 ? sh->bc[6] : 0u;
        n_rows = n_ended_rows + n_child_seeds;
        if (n_rows > W.rl_cap) n_rows = W.rl_cap;

        // ---- D1. dedup, gap sources, child seeds (reference src/mapper.cpp:527-603): every bucket is one k-mer run.  Work is
        //      handed out through one counter: first the 32-key chunks of the large buckets, one at a time and in any order
        //      (C2 left each chunk its running max and counts), then the groups' merged buckets and packs of small ones.
        if (nc > 0) {
            const uint4 *csum = W.elist;
            const u32 n_units = *(volatile u32 *) &v2->n_units;
            for (;;) {
                const u32 gi = k2v2_grab(&v2->grab[1]);
                if (gi >= n_units + 32u) break;
                if (gi < n_units) {
                    const uint4 u = csum[gi];
                    const u32 sl_u = u.w & 1023u, g0 = (u.w >> 10) << 5;
                    const u32 o = v2->koff[sl_u], n = v2->kcnt[sl_u] - o, pre = v2->kagg[sl_u];
                    const u32 kmer = v2->t.gkmer[((sl_u & 31u) << 5) | (sl_u >> 5)];
                    const uint2 kr = tb->kmer_range[kmer];
                    const float pkm = sh->probs[kmer];
                    const bool prob_ok = pkm >= source_prob;
                    const u32 pos = g0 + (u32) lane;
                    const bool a = pos < n, has_next = pos + 1u < n;
                    uint4 cur = make_uint4(0, 0, 0, 0);
                    if (a) cur = ckA[o + pos];
                    u32 nx = w_shfl_down(cur.x, 1), ny = w_shfl_down(cur.y, 1);
                    if (lane == 31 && has_next) { const uint4 t = ckA[o + pos + 1u]; nx = t.x; ny = t.y; }
                    u32 mxo;
                    const K2V2Walk wk = k2v2_walk(cur, nx, ny, a, has_next, pos == 0, pos == 0, g0 != 0, u.x, prob_ok, kr, &mxo);
                    const u32 sidx = (pre & 0xFFFFu) + u.y + (u32) d_popc(wk.m_b & lt) + (u32) d_popc(wk.m_a & lt);   // sources before this element
                    if (wk.begin_v && nc + sidx < maxp) {
                        write_source(next, hist_e, S0 + nc + sidx, kr.x, cur.x - 1u, kmer, pkm);
                        onext[nc + sidx] = S0 + nc + sidx;
                    }
                    const u32 sidx2 = sidx + (wk.begin_v ? 1u : 0u);
                    if (wk.after_v && nc + sidx2 < maxp) {
                        write_source(next, hist_e, S0 + nc + sidx2, wk.as, wk.ae, kmer, pkm);
                        onext[nc + sidx2] = S0 + nc + sidx2;
                    }
                    const u32 rec = cur.w >> 14;
                    if (a) onext[o + pos] = rec | (wk.dup ? UNC_INVALID : 0u);
                    if (wk.seed) {                                     // update_seeds(child, false)
                        d_atomic_or(&((u32 *) (next + (size_t) rec * 2))[3], 0x80000000u);   // sa_checked_
                        const u32 ri = n_ended_rows + (pre >> 16) + u.z + (u32) d_popc(wk.m_seed & lt);
                        if (ri < W.rl_cap)
                            rlist[ri] = make_uint2(ix.seq_len - unc_sa_lookup(ix, cur.x, &pend_steps, &pend_blocks), (cur.w >> 1) & 0x1Fu);
                        else sh->wk_overflow = 1;
                    }
                    continue;
                }
                const u32 grp = gi - n_units;
                const u32 sl = (u32) lane * 32u + grp;
                const u32 bo = v2->koff[sl], bn = v2->kcnt[sl] - bo, bpre = v2->kagg[sl];
                const u32 meta = v2->t.gmeta[grp * 32u + (u32) lane];
                u32 todo_m = w_ballot(meta != 0 && bn > 0);
                while (todo_m) {                                      // merged groups: one lane walks the sorted bucket
                    const int l = d_ffs(todo_m) - 1;
                    todo_m &= todo_m - 1;
                    {
                        const u32 o_m = w_shfl(bo, l), n_m = w_shfl(bn, l), pre_m = w_shfl(bpre, l), mt_m = w_shfl(meta, l);
                        K2V2Emit E;
                        E.next = next; E.hist_e = hist_e; E.onext = onext; E.rlist = rlist;
                        E.S0 = S0; E.nc = nc; E.maxp = maxp; E.n_ended_rows = n_ended_rows; E.rl_cap = W.rl_cap; E.pos0 = o_m;
                        E.src_before = pre_m & 0xFFFFu; E.seeds_before = pre_m >> 16;
                        k2v2_walk_merged<true>(ix, sh, ckA + o_m, n_m, mt_m >> 8, source_prob, E, &pend_steps, &pend_blocks, (uint4 *) stage_r);
                    }
                }
                const u32 cnt = (bn > 0 && bn <= 32u && meta == 0) ? bn : 0u;
                u32 tot;
                const u32 P = w_exscan(cnt, &tot);
                u32 remaining = w_ballot(cnt != 0);
                while (remaining) {
                    const K2V2Pack pk = k2v2_next_pack(cnt, P, &remaining);
                    const u32 kmer = v2->t.gkmer[grp * 32u + pk.bl];
                    const uint2 kr = tb->kmer_range[kmer];
                    const float pkm = sh->probs[kmer];
                    const bool prob_ok = pkm >= source_prob;
                    const u32 pre = w_shfl(bpre, (int) pk.bl), o = w_shfl(bo, (int) pk.bl);
                    uint4 cur = make_uint4(0, 0, 0, 0);
                    if (pk.a) cur = ckA[o + pk.pos];
                    const u32 nx = w_shfl_down(cur.x, 1), ny = w_shfl_down(cur.y, 1);
                    u32 mxo;
                    const K2V2Walk wk = k2v2_walk(cur, nx, ny, pk.a, pk.a && pk.pos + 1u < pk.n, pk.pos == 0, pk.pos == 0, false, 0u, prob_ok,
                                                  kr, &mxo);
                    const u32 sm = k2v2_segmask(pk.start, pk.n);
                    const u32 sidx = (pre & 0xFFFFu) + (u32) d_popc(wk.m_b & lt & sm) + (u32) d_popc(wk.m_a & lt & sm);   // sources before this element
                    if (wk.begin_v && nc + sidx < maxp) {
                        write_source(next, hist_e, S0 + nc + sidx, kr.x, cur.x - 1u, kmer, pkm);
                        onext[nc + sidx] = S0 + nc + sidx;
                    }
                    const u32 sidx2 = sidx + (wk.begin_v ? 1u : 0u);
                    if (wk.after_v && nc + sidx2 < maxp) {
                        write_source(next, hist_e, S0 + nc + sidx2, wk.as, wk.ae, kmer, pkm);
                        onext[nc + sidx2] = S0 + nc + sidx2;
                    }
                    const u32 rec = cur.w >> 14;
                    if (pk.a) onext[o + pk.pos] = rec | (wk.dup ? UNC_INVALID : 0u);
                    // update_seeds(child, false): unique, move-headed, full-length, probable paths
                    if (wk.seed) {
                        d_atomic_or(&((u32 *) (next + (size_t) rec * 2))[3], 0x80000000u);   // sa_checked_
                        const u32 ri = n_ended_rows + (pre >> 16) + (u32) d_popc(wk.m_seed & lt & sm);
                        if (ri < W.rl_cap)
                            rlist[ri] = make_uint2(ix.seq_len - unc_sa_lookup(ix, cur.x, &pend_steps, &pend_blocks), (cur.w >> 1) & 0x1Fu);
                        else sh->wk_overflow = 1;
                    }
                }
            }
        }
        PT_WE(2)
        // ---- E. fresh sources for every sufficiently probable k-mer without one (reference src/mapper.cpp:605-624):
        //      word j (32 k-mers) by warp j % nwk, positions and the buffer-full cut from worker warp 0's plan
        for (u32 j = ww; j < 32; j += nwk) {
            const u32 before = v2->fresh_before[j];
            if (before >= maxp) continue;                         // never visited: its flags stay as they are
            const u32 k = j * 32 + (u32) lane;
            const u32 fw = sh->flags[j];
            u32 m_add = v2->fresh_mask[j];
            const u32 room = maxp - before;
            u32 visited = 0xFFFFFFFFu;
            if ((u32) d_popc(m_add) >= room) {
                // the room-th add fills the buffer; k-mers after it are never visited
                u32 mm = m_add;
                for (u32 q = 1; q < room; q++) mm &= mm - 1;
                int last = d_ffs(mm) - 1;
                visited = last == 31 ? 0xFFFFFFFFu : ((2u << last) - 1u);
                m_add &= visited;
            }
            const u32 rank = (u32) d_popc(m_add & lt);
            if ((m_add >> lane) & 1u) {
                const uint2 kr = tb->kmer_range[k];
                write_source(next, hist_e, S0 + before + rank, kr.x, kr.y, k, sh->probs[k]);
                onext[before + rank] = S0 + before + rank;
            }
            w_sync();
            if (lane == 0) sh->flags[j] = fw & ~visited;
        }
        if (wt == 0) *(volatile u32 *) &sh->n_rows[event_i & 1u] = n_rows;
        PT_WARR(3)
        PT_MARK(5)
        // ---- hand the event's seeds to the tracker; learn the outcome of the previous event
        c_sync();                                                     // X_e
        PT_WREL(0)
        PT_FENCE
        PT_MARK(6)
        PT_WR(2, 21, 22)
        PT_WLAG(3, 23, 24)
        PT_WLAG(0, 13, 14)
        PT_WTRK(3, 25)
        const u32 nn = sh->bc[1];
        pend_sources = nn - nc;
        const u32 v = event_i > n_first ? *(volatile u32 *) &sh->verdict[(event_i - 1u) & 1u] : 0u;
        if (v) {                                                      // event_i's work is discarded: the Mapper returned
            if (FLAGS && wt < 32u) sh->flags[wt] = sh->flags_prev[wt];   // after event_i - 1 (reference src/mapper.cpp:633-651)
            break;
        }
        n_children += pend_children; n_sources += pend_sources;
        my_blocks += pend_blocks; my_steps += pend_steps;
        pend_children = pend_sources = pend_blocks = pend_steps = 0;
        prev_size = nn;
        gen ^= 1u;
        PT_MARK(8)
    }
    if (STREAM && wt == 0) { DevMapState *ms = B.mstate + B.chan[r]; ms->prev_size = prev_size; ms->gen = gen; }
    PT_FLUSH(B, r)
    for (int d = 16; d > 0; d >>= 1) { my_blocks += w_shfl(my_blocks, lane ^ d); my_steps += w_shfl(my_steps, lane ^ d); }
    if (lane == 0) { s_atomic_add(&sh->cnt_blocks, my_blocks); s_atomic_add(&sh->cnt_steps, my_steps); }
    if (wt == 0) {
        sh->tot_children[0] = (u32) n_children; sh->tot_children[1] = (u32) (n_children >> 32);
        sh->tot_sources[0] = (u32) n_sources; sh->tot_sources[1] = (u32) (n_sources >> 32);
    }
    c_sync();                                                         // Y: final barrier
}
