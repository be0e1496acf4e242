// unc_device.cuh -- device code of the B200-native `uncalled map` hot path.
//
//   K1  unc_k1_read()      thread-per-read event detection + whole-read normalisation stats
//                          (reference src/event_detector.cpp:83-319, src/normalizer.cpp:31-44)
//   K2  unc_k2_map_read()  CTA-per-read mapper: pore-model scoring, FM-index path extension,
//                          child sort/dedup, gap + fresh sources, seed clustering, PAF coords
//                          (reference src/mapper.cpp:433-728, src/seed_tracker.cpp:56-262,
//                           submods/bwa/bwt.c:53-163)
//
// Written against unc_warp.cuh so the same source runs under nvcc (sm_100a) and under the
// CPU warp emulator used by the tests.  All arithmetic that the reference performs in
// float/double is spelled with explicit round-to-nearest operations (no FMA contraction).
#pragma once
#include "unc_warp.cuh"

typedef uint8_t u8;
typedef uint16_t u16;
typedef uint32_t u32;
typedef int32_t i32;
typedef uint64_t u64;

#define UNC_NKMER 1024
#define UNC_KMASK 0x3FFu
#define UNC_SEED_LEN 22u
#define UNC_NGEN 24u            /* generations of (C, parent) history kept: need e-22 .. e */
#define UNC_PATH_MASK 0x3FFFFFu
#define UNC_PATH_TAIL 0x200000u
#define UNC_INVALID 0x80000000u /* flag in the order[] array: path invalidated by dedup */
#define UNC_BLK 32u             /* seed-cluster block capacity (one entry per lane) */

// ------------------------------------------------------------------ device image

struct DevIndex {
    const uint4 *bwt;      // 64-byte Occ blocks as in the .bwt file: 4 x u64 counts, 8 x u32 BWT words
    const u32 *sa;         // sampled SA (every 32 rows) narrowed to u32; sa[0] = 0xFFFFFFFF
    const u32 *sa_full;    // optional: bwt_sa(k) for every row k, expanded on the device at index load
    const uint2 *kmer_range;  // 1024 x (start, end) FM ranges
    const float *lv_mean, *lv_var2, *lognorm;  // pore model tables (complement order)
    const float *thresh;   // 64 probability thresholds indexed by clzll(range length)
    u32 primary, seq_len;
    u32 L2[5];
    u32 start_bits;        // bits needed to represent seq_len (radix-sort passes)
    // GPU-side layouts derived at index load (unc_k2v2.cuh):
    const uint4 *occ2;     // 32-byte Occ blocks: 4 x u32 counts before the block + 64 two-bit BWT symbols
    const struct K2V2Tab *kt;   // k-mer buckets of the child sort
};

// K-mer buckets of the child sort (unc_k2v2.cuh).  Children sorted by fm_start are grouped by k-mer because the
// k-mers' FM ranges are ordered and disjoint -- except where BwaIndex::get_base_range's start (L2[b], not L2[b]+1:
// reference src/bwa_index.hpp:172-174) lets a k-mer's range begin on the LAST row of its predecessor's.  K-mers
// whose ranges overlap share one bucket ("merged group"; a handful per index, two k-mers each in practice), and
// a key carries its k-mer's position in the group (sub).
#define K2V2_MAX_MERGED 64u     /* k-mers in merged groups, all groups together */
struct alignas(16) K2V2Tab {
    u16 kslot[UNC_NKMER];   // k-mer -> slot of its group in the per-bucket arrays (group rank r sits at (r&31)*32 + (r>>5))
    u16 gkmer[UNC_NKMER];   // group rank -> its k-mer (single-k-mer groups)
    u16 gmeta[UNC_NKMER];   // group rank -> 0, or (offset into mk) << 8 | members for a merged group
    u16 mk[K2V2_MAX_MERGED];   // the merged groups' k-mers, in FM order
    u8 ksub[UNC_NKMER];     // k-mer -> its position in its group
};

// L2[c] through selects: a dynamically indexed member would force the whole kernel-parameter
// struct into local memory (LDL on the extension loop's critical path)
UNC_DEV u32 unc_L2(const DevIndex &ix, u32 c) {
    return c == 0 ? ix.L2[0] : c == 1 ? ix.L2[1] : c == 2 ? ix.L2[2] : c == 3 ? ix.L2[3] : ix.L2[4];
}

struct DevParams {
    u32 max_rep_copy, max_paths, max_consec_stay, max_events, min_rep_len;
    float max_stay_frac, min_seed_prob;
    u32 min_map_len;
    float min_mean_conf, min_top_conf;
    float threshold1, threshold2, peak_height, min_mean, max_mean;
    float bp_per_sec, sample_rate;
    float tgt_mean, tgt_stdv;   // model means mean / stdv (normaliser target)
};

struct DevReadDesc {
    u64 offset;
    u32 n_samples, dtype;
    float cal_range, cal_offset, cal_digit;
    u32 pad;
};

struct DevRec {   // == unc_paf_rec
    i32 mapped, fwd, rid, status;
    u32 n_events, events_used, matches, n_clusters;
    u64 rd_len, rd_st, rd_en, rf_st, rf_en, rf_len;
    u64 n_children, n_sources, n_occ_blocks, n_sa_steps, n_seeds;
};

struct DevBatch {
    const void *samples;
    u64 samples_bytes;   // extent of the sample buffer (bulk copies never read past it)
    const DevReadDesc *reads;
    u32 n_reads;
    u32 *k1_queue;       // atomic read counter of the event-detection kernel
    u32 *k1_flags;       // per read: 1 = redo with the serial routine (exactness condition failed)
    u32 *k1_stats;       // optional (may be null): tiles, FSM re-run rounds, re-run lanes, flagged reads
    // streaming (k2_map_stream only): item r continues the read of channel chan[r] from mstate[chan[r]]
    struct DevMapState *mstate;
    const u32 *chan;
    // K1 outputs
    float *events;       // n_reads x ev_stride valid event means (raw, un-normalised)
    float *normed;       // optional (may be null): normalised means
    u32 ev_stride;
    u32 *n_events;
    float *scale, *shift, *mean_event_len;
    // K2
    u32 *queue;          // atomic read counter
    DevRec *out;
    unsigned long long *dbg;  // optional (may be null): 8 phase-cycle counters per read (UNC_PHASE_TIMING builds)
    const u64 *seq_offsets;  // .ann offsets / lens for translate_loc
    const u32 *seq_lens;
    u32 n_seqs;
    u64 l_pac;
    // ordered mode (unc_map_batch_ordered; both optional): read r starts with the sources_added_ words
    // flags_in[32r..32r+32) instead of a clear set and leaves its final ones in flags_out[32r..32r+32)
    const u32 *flags_in = nullptr;
    u32 *flags_out = nullptr;
};

struct DevWork {   // per-slot (per-CTA) workspaces; slot s uses [s*stride, (s+1)*stride)
    uint4 *paths;      // 2 generations x (ceil(max_paths/32)*160 chunk-local child slots + max_paths sources) x 2 uint4
    uint2 *hist;       // 24 generations x the same record index space: (cumulative log-prob C, parent record index)
    uint4 *wlist;      // ceil(max_paths/32)*160 deferred window look-ups: (child idx, parent idx, C bits, moves)
    uint4 *ckey;       // 2 x max_paths uint4 (radix ping-pong, compact)
    uint4 *cks;        // ceil(max_paths/32)*160 chunk-local sort keys written by the extension phase
    uint4 *elist;      // ceil(max_paths/32)*32 chunk-local ended-path entries (start, end, moves, children before)
    u32 *order;        // 2 x max_paths: logical path order -> record index (| UNC_INVALID)
    uint2 *rlist;      // 2 x rl_cap (double buffered by event parity) seed rows: (FM row -> ref end, move_count | ended<<8)
    uint4 *clu;        // max_blocks x 32 x 2 uint4
    uint4 *dir;        // max_blocks
    u32 max_blocks, rl_cap;
};

// ------------------------------------------------------------------ pore model

// reference src/pore_model.hpp:163-165: float subtract, double square/divide/subtract, one
// rounding to float.
UNC_DEV float unc_match_prob(float samp, float mean, float var2, float lognorm) {
    float d = f_sub(samp, mean);
    double dd = (double) d;
    double q = d_div(-d_mul(dd, dd), (double) var2);
    return (float) d_sub(q, (double) lognorm);
}

// ------------------------------------------------------------------ FM index

// count of 2-bit symbols equal to c in y (reference submods/bwa/bwt.c:98-105), as match bits
UNC_DEV u64 unc_match_bits(u64 y, u32 c) {
    return (((c & 2) ? y : ~y) >> 1) & ((c & 1) ? y : ~y) & 0x5555555555555555ull;
}

// Occ(k, c) for a row k that is NOT seq_len and NOT (u64)-1, given its 64-byte block already
// in registers (b0,b1 = counts; b2,b3 = BWT words).  kk = k - (k >= primary).
// Equivalent to reference submods/bwa/bwt.c:107-129 (masking the match bits of the partial
// word instead of the data removes the need for the c==0 correction).
UNC_DEV u32 unc_occ_in_block(uint4 b0, uint4 b1, uint4 b2, uint4 b3, u32 kk, u32 c) {
    u32 cnt = (c == 0) ? b0.x : (c == 1) ? b0.z : (c == 2) ? b1.x : b1.z;  // low words of the u64 counts
    u32 q = (kk & 127u) >> 5;  // index of the 64-bit word holding symbol kk
    u64 w0 = ((u64) b2.x << 32) | b2.y, w1 = ((u64) b2.z << 32) | b2.w;
    u64 w2 = ((u64) b3.x << 32) | b3.y, w3 = ((u64) b3.z << 32) | b3.w;
    u64 part = ~((1ull << ((~kk & 31u) << 1)) - 1ull);
    u64 m0 = q > 0 ? ~0ull : part;
    u64 m1 = q > 1 ? ~0ull : (q == 1 ? part : 0ull);
    u64 m2 = q > 2 ? ~0ull : (q == 2 ? part : 0ull);
    u64 m3 = q == 3 ? part : 0ull;
    cnt += d_popcll(unc_match_bits(w0, c) & m0);
    cnt += d_popcll(unc_match_bits(w1, c) & m1);
    cnt += d_popcll(unc_match_bits(w2, c) & m2);
    cnt += d_popcll(unc_match_bits(w3, c) & m3);
    return cnt;
}

// Same count, reading the block's words from memory as they are needed (L1-resident after the first
// touch) instead of holding the 64-byte block in 16 registers: the register-lean extension loop uses it.
UNC_DEV u32 unc_occ_at(const uint4 *blk, u32 kk, u32 c) {
    u32 cnt = d_ldg((const u32 *) blk + 2u * c);            // low word of the u64 cumulative count of base c
    const u32 q = (kk & 127u) >> 5;                            // index of the 64-bit word holding symbol kk
    const uint2 *wp = (const uint2 *) (blk + 2);
    for (u32 i = 0; i <= q; i++) {
        const uint2 v = d_ldg(wp + i);
        const u64 w = ((u64) v.x << 32) | v.y;
        const u64 m = i < q ? ~0ull : ~((1ull << ((~kk & 31u) << 1)) - 1ull);
        cnt += (u32) d_popcll(unc_match_bits(w, c) & m);
    }
    return cnt;
}

struct OccBlock { uint4 b0, b1, b2, b3; };

UNC_DEV OccBlock unc_load_block(const DevIndex &ix, u32 kk) {
    const uint4 *p = ix.bwt + ((size_t) (kk >> 7) << 2);
    OccBlock b;
    b.b0 = d_ldg(p); b.b1 = d_ldg(p + 1); b.b2 = d_ldg(p + 2); b.b3 = d_ldg(p + 3);
    return b;
}

// bwt_occ (reference submods/bwa/bwt.c:107-129) for a single row
UNC_DEV u32 unc_occ(const DevIndex &ix, u32 k, u32 c, u32 *n_blocks) {
    if (k == ix.seq_len) return unc_L2(ix, c + 1) - unc_L2(ix, c);
    if (k == 0xFFFFFFFFu) return 0;
    u32 kk = k - (k >= ix.primary);
    OccBlock b = unc_load_block(ix, kk);
    (*n_blocks)++;
    return unc_occ_in_block(b.b0, b.b1, b.b2, b.b3, kk, c);
}

// One backward-search step for all four bases at once: BwaIndex::get_neighbor
// (reference src/bwa_index.hpp:158-162) over bwt_2occ (submods/bwa/bwt.c:132-163).
// `want` has bit b set for each base whose range is needed; on return bit b of the result is
// set iff base b yields a valid (non-empty) range, stored in ns[b]..ne[b].
// Paths always have start >= 1.  Instead of two Occ values per base, the symbols of rows
// (k, l] are counted first: only bases that occur there have a non-empty range (for a
// unique path that is exactly one base), and only for those the prefix Occ(k, c) is needed:
//   ns = L2[c] + Occ(k,c) + 1,  ne = L2[c] + Occ(l,c) = ns + count_c(k,l] - 1.
// `pre` (optional): the Occ block of row start-1, already fetched (staged by cp.async in the extension loop)
UNC_DEV u32 unc_neighbors(const DevIndex &ix, u32 start, u32 end, u32 want, u32 ns[4], u32 ne[4], u32 *n_blocks,
                          const OccBlock *pre = nullptr) {
    u32 k = start - 1, l = end;
    u32 kk = k - (k >= ix.primary), ll = l - (l >= ix.primary);
    bool l_is_end = (l == ix.seq_len);
    OccBlock bk = pre ? *pre : unc_load_block(ix, kk);
    (*n_blocks)++;
    u32 valid = 0;
    if (!l_is_end && (ll >> 5) == (kk >> 5)) {
        // rows k and l fall into the same 64-bit BWT word: count symbols of (kk, ll] directly
        u32 q = (kk & 127u) >> 5;
        u32 hi = q == 0 ? bk.b2.x : q == 1 ? bk.b2.z : q == 2 ? bk.b3.x : bk.b3.z;
        u32 lo = q == 0 ? bk.b2.y : q == 1 ? bk.b2.w : q == 2 ? bk.b3.y : bk.b3.w;
        u64 w = ((u64) hi << 32) | lo;
        u64 le_k = ~((1ull << ((~kk & 31u) << 1)) - 1ull), le_l = ~((1ull << ((~ll & 31u) << 1)) - 1ull);
        u64 between = le_l & ~le_k;
#pragma unroll
        for (u32 c = 0; c < 4; c++) {
            if (!((want >> c) & 1u)) continue;
            u32 cnt = (u32) d_popcll(unc_match_bits(w, c) & between);
            if (cnt == 0) continue;
            u32 ok = unc_occ_in_block(bk.b0, bk.b1, bk.b2, bk.b3, kk, c);
            ns[c] = unc_L2(ix, c) + ok + 1;
            ne[c] = ns[c] + cnt - 1;
            valid |= 1u << c;
        }
        return valid;
    }
    OccBlock bl = bk;
    if (!l_is_end && (ll >> 7) != (kk >> 7)) { bl = unc_load_block(ix, ll); (*n_blocks)++; }
#pragma unroll
    for (u32 c = 0; c < 4; c++) {
        if (!((want >> c) & 1u)) continue;
        u32 ok = unc_occ_in_block(bk.b0, bk.b1, bk.b2, bk.b3, kk, c);
        u32 ol = l_is_end ? (unc_L2(ix, c + 1) - unc_L2(ix, c)) : unc_occ_in_block(bl.b0, bl.b1, bl.b2, bl.b3, ll, c);
        ns[c] = unc_L2(ix, c) + ok + 1;
        ne[c] = unc_L2(ix, c) + ol;
        if (ns[c] <= ne[c]) valid |= 1u << c;
    }
    return valid;
}

// bwt_sa (reference submods/bwa/bwt.c:86-96) with bwt_invPsi (:53-59); sa_intv == 32
UNC_DEV u32 unc_sa(const DevIndex &ix, u32 k, u32 *n_steps, u32 *n_blocks) {
    u32 steps = 0;
    while (k & 31u) {
        ++steps;
        u32 x = k - (k > ix.primary);
        const u32 *wp = (const u32 *) ix.bwt + (((size_t) (x >> 7)) << 4) + 8 + ((x & 0x7fu) >> 4);
        u32 c = (d_ldg(wp) >> ((~x & 0xfu) << 1)) & 3u;
        u32 r = unc_L2(ix, c) + unc_occ(ix, k, c, n_blocks);
        k = (k == ix.primary) ? 0u : r;
    }
    *n_steps += steps;
    return steps + d_ldg(ix.sa + (k >> 5));
}

// SA lookup as the mapper uses it: one load when the expanded table exists, else the LF walk
UNC_DEV u32 unc_sa_lookup(const DevIndex &ix, u32 k, u32 *n_steps, u32 *n_blocks) {
    if (ix.sa_full) return d_ldg(ix.sa_full + k);
    return unc_sa(ix, k, n_steps, n_blocks);
}

// The 1024 k-mer FM ranges (reference src/bwa_index.hpp:124-132): get_base_range(head) -- whose
// start is L2[b], NOT L2[b]+1 (:172-174) -- followed by four get_neighbor steps.
UNC_DEV uint2 unc_kmer_range_compute(const DevIndex &ix, u32 kmer) {
    u32 head = (kmer >> 8) & 3u;
    u32 st = unc_L2(ix, head), en = unc_L2(ix, head + 1);
    u32 nb = 0;
    for (u32 i = 1; i < 5; i++) {
        u32 base = (kmer >> (2 * (4 - i))) & 3u;
        u32 ok = unc_occ(ix, st - 1u, base, &nb), ol = unc_occ(ix, en, base, &nb);
        st = unc_L2(ix, base) + ok + 1u;
        en = unc_L2(ix, base) + ol;
    }
    return make_uint2(st, en);
}

// ------------------------------------------------------------------ K1: events + normalisation

struct DevDetector {
    u32 masked_to;
    i32 peak_pos;
    float peak_value;
    int valid_peak;
};

// reference src/event_detector.cpp:174-219 (compute_tstat), exact mixed precision
UNC_DEV float unc_tstat(const double *sum, const double *sumsq, u32 t, u32 buf_mid, u32 w) {
    const float wf = (float) w;
    if (t <= 2 * w) return 0.0f;
    u32 i = buf_mid % 13u, st = (buf_mid - w) % 13u, en = (buf_mid + w) % 13u;
    double sum1 = d_sub(sum[i], sum[st]);
    double sumsq1 = d_sub(sumsq[i], sumsq[st]);
    float sum2 = (float) d_sub(sum[en], sum[i]);
    float sumsq2 = (float) d_sub(sumsq[en], sumsq[i]);
    float mean1 = (float) d_div(sum1, (double) wf);
    float mean2 = f_div(sum2, wf);
    float m1sq = f_mul(mean1, mean1), m2sq = f_mul(mean2, mean2);
    float q2 = f_div(sumsq2, wf);
    double cv = d_sub(d_add(d_sub(d_div(sumsq1, (double) wf), (double) m1sq), (double) q2), (double) m2sq);
    float combined_var = (float) cv;
    combined_var = fmaxf(combined_var, 1.17549435e-38f);
    float delta = f_sub(mean2, mean1);
    return f_div(fabsf(delta), f_sqrt(f_div(combined_var, wf)));
}

// reference src/event_detector.cpp:221-279 (peak_detect).  `is_short` selects the branch that
// lets the short detector mask/reset the long one.
UNC_DEV bool unc_peak(DevDetector &d, DevDetector &longd, bool is_short, float cur, u32 buf_mid, u32 wlen,
                      float threshold, float peak_height) {
    if (d.masked_to >= buf_mid) return false;
    if (d.peak_pos == -1) {
        if (cur < d.peak_value) {
            d.peak_value = cur;
        } else if (f_sub(cur, d.peak_value) > peak_height) {
            d.peak_value = cur;
            d.peak_pos = (i32) buf_mid;
        }
    } else {
        if (cur > d.peak_value) {
            d.peak_value = cur;
            d.peak_pos = (i32) buf_mid;
        }
        if (is_short) {
            if (d.peak_value > threshold) {
                longd.masked_to = (u32) d.peak_pos + wlen;
                longd.peak_pos = -1;
                longd.peak_value = 3.402823466e+38f;
                longd.valid_peak = 0;
            }
        }
        if (f_sub(d.peak_value, cur) > peak_height && d.peak_value > threshold) d.valid_peak = 1;
        if (d.valid_peak && (buf_mid - (u32) d.peak_pos) > wlen / 2) {
            d.peak_pos = -1;
            d.peak_value = cur;
            d.valid_peak = 0;
            return true;
        }
    }
    return false;
}

struct DevEvdt {
    double sum[13], sumsq[13];
    u32 t, evt_st;
    double evt_st_sum, evt_st_sumsq;
    float len_sum;
    u32 total_events;
    DevDetector sd, ld;
};

UNC_DEV void unc_evdt_reset(DevEvdt &e) {
    for (int i = 0; i < 13; i++) { e.sum[i] = 0.0; e.sumsq[i] = 0.0; }
    e.t = 1;
    e.evt_st = 0;
    e.evt_st_sum = e.evt_st_sumsq = 0.0;
    e.len_sum = 0.0f;
    e.total_events = 0;
    e.sd.masked_to = 0; e.sd.peak_pos = -1; e.sd.peak_value = 3.402823466e+38f; e.sd.valid_peak = 0;
    e.ld = e.sd;
}

// reference src/event_detector.cpp:83-112 (add_sample) + :296-319 (create_event).
// Returns true and sets *mean when a valid event (min_mean <= mean <= max_mean) is emitted.
UNC_DEV bool unc_evdt_add(DevEvdt &e, const DevParams &p, float s, float *mean_out) {
    u32 t_mod = e.t % 13u;
    u32 prev = t_mod > 0 ? t_mod - 1 : 12u;
    float ss = f_mul(s, s);
    e.sum[t_mod] = d_add(e.sum[prev], (double) s);
    e.sumsq[t_mod] = d_add(e.sumsq[prev], (double) ss);
    e.t++;
    u32 buf_mid = e.t - 6u - 1u;
    float t1 = unc_tstat(e.sum, e.sumsq, e.t, buf_mid, 3u);
    float t2 = unc_tstat(e.sum, e.sumsq, e.t, buf_mid, 6u);
    bool p1 = unc_peak(e.sd, e.ld, true, t1, buf_mid, 3u, p.threshold1, p.peak_height);
    bool p2 = unc_peak(e.ld, e.ld, false, t2, buf_mid, 6u, p.threshold2, p.peak_height);
    if (!(p1 || p2)) return false;
    u32 evt_en = buf_mid - 3u + 1u;
    u32 eb = evt_en % 13u;
    u32 length = (u32) (float) (evt_en - e.evt_st);
    float mean = (float) d_div(d_sub(e.sum[eb], e.evt_st_sum), (double) length);
    e.evt_st = evt_en;
    e.evt_st_sum = e.sum[eb];
    e.evt_st_sumsq = e.sumsq[eb];
    e.len_sum = f_add(e.len_sum, (float) length);
    e.total_events++;
    *mean_out = mean;
    return mean >= p.min_mean && mean <= p.max_mean;
}

// calibrated pA sample i of a read (reference src/read_buffer.cpp:239-242 for raw i16 input)
UNC_DEV float unc_sample(const void *samples, const DevReadDesc &rd, u32 i) {
    if (rd.dtype == 0) return d_ldg((const float *) samples + rd.offset + i);
    u16 raw = (u16) d_ldg((const int16_t *) samples + rd.offset + i);
    return f_div(f_mul(rd.cal_range, f_add((float) raw, rd.cal_offset)), rd.cal_digit);
}

// One read, one thread.  Writes the read's valid event means, their count, the normaliser's
// scale/shift (reference src/normalizer.cpp:31-44 + :114-118) and mean_event_len
// (reference src/event_detector.cpp:151-153).
UNC_DEV void unc_k1_read(const DevBatch &B, const DevParams &p, u32 r) {
    DevReadDesc rd = B.reads[r];
    DevEvdt e;
    unc_evdt_reset(e);
    float *ev = B.events + (size_t) r * B.ev_stride;
    u32 ne = 0;
    for (u32 i = 0; i < rd.n_samples; i++) {
        float mean;
        if (unc_evdt_add(e, p, unc_sample(B.samples, rd, i), &mean)) ev[ne++] = mean;
    }
    B.n_events[r] = ne;
    B.mean_event_len[r] = f_div(e.len_sum, (float) e.total_events);
    float scale = 0.0f, shift = 0.0f;
    if (ne > 0) {
        double mean = 0.0;
        for (u32 i = 0; i < ne; i++) mean = d_add(mean, (double) ev[i]);
        mean = d_div(mean, (double) ne);
        double varsum = 0.0;
        for (u32 i = 0; i < ne; i++) {
            double d = d_sub((double) ev[i], mean);
            varsum = d_add(varsum, d_mul(d, d));
        }
        scale = (float) d_div((double) p.tgt_stdv, d_sqrt(d_div(varsum, (double) ne)));
        shift = (float) d_sub((double) p.tgt_mean, d_mul((double) scale, mean));
        if (B.normed) {
            float *nm = B.normed + (size_t) r * B.ev_stride;
            for (u32 i = 0; i < ne; i++) nm[i] = f_add(f_mul(scale, ev[i]), shift);
        }
    }
    B.scale[r] = scale;
    B.shift[r] = shift;
}

// ------------------------------------------------------------------ streaming: persistent mapper state
// What Mapper keeps between map_chunk calls of one read (reference src/mapper.hpp:205-236): the path
// buffers, event_i_, the seed tracker -- here the per-channel workspace slot plus these scalars.
struct DevMapState {
    u32 prev_size, gen, event_i, started;     // started == 0: new read (Mapper::reset, src/mapper.cpp:218-246)
    u32 flags[32];                            // sources_added_: persists across the reads of a channel (src/mapper.cpp:88)
    u32 t_nb, t_n_alloc, t_n_live, t_n_lens, t_top1, t_top2, t_overflow;
    float t_len_sum;
    u32 t_max_map[6];
    u32 pad[2];
};

struct DevWorkStrides {
    size_t paths, hist, ckey, cks, elist, order, rlist, clu, dir;
};

// ------------------------------------------------------------------ K2: seed tracker

// A cluster entry is two uint4:  A = (ren_start, evt_en, ref_st, ren_end)  B = (evt_st, total_len, 0, 0)
// std::set order (reference src/seed_tracker.cpp:97-102): ren_start descending, evt_en descending.
UNC_DEV bool clu_less(u32 as, u32 ae, u32 bs, u32 be) { return as > bs || (as == bs && ae > be); }

struct Clu { u32 ren_start, evt_en, ref_st, ren_end, evt_st, total_len; };

#if defined(UNC_PHASE_TIMING) && !defined(UNC_EMUL)
UNC_DEV long long trk_clock() { long long v; asm volatile("mov.u64 %0, %%clock64;" : "=l"(v) :: "memory"); return v; }
#define PT_TRK0(t) (t).pt_t = trk_clock();
#define PT_TRK(t, i) { const long long _n = trk_clock(); (t).pt[i] += (unsigned long long) (_n - (t).pt_t); (t).pt_t = _n; }
#else
#define PT_TRK0(t)
#define PT_TRK(t, i)
#endif
struct Tracker {     // all fields warp-uniform (replicated in every lane)
    uint4 *blocks;   // slot base: block b entry i at blocks[(b*32 + i)*2 + {0,1}]
    uint4 *dir;      // sorted directory: (first ren_start, first evt_en, block id, count) -- in shared memory while it fits
    uint4 *dir_glob; // its home in the slot's workspace (== dir once it has outgrown the shared copy, or when there is none)
    u32 dir_cap;     // entries the shared copy holds
#if defined(UNC_PHASE_TIMING) && !defined(UNC_EMUL)
    unsigned long long pt[3]; long long pt_t;   // phase-timing builds: cycles in search / scan / update of add_seed
#endif
    u32 nb, n_alloc, max_blocks;
    u32 n_live, n_lens, top1, top2;
    float len_sum;
    Clu max_map;
    u32 overflow;
};

UNC_DEV void trk_reset(Tracker &t) {
    t.nb = 0; t.n_alloc = 0; t.n_live = 0; t.n_lens = 0; t.top1 = 0; t.top2 = 0;
    t.len_sum = 0.0f;
    t.max_map.ren_start = 1; t.max_map.ren_end = 0; t.max_map.ref_st = 0;
    t.max_map.evt_st = 1; t.max_map.evt_en = 0; t.max_map.total_len = 0;  // NULL_ALN
    t.overflow = 0;
}

UNC_DEV Clu trk_load(const Tracker &t, u32 blk, u32 i) {
    uint4 a = t.blocks[((size_t) blk * UNC_BLK + i) * 2], b = t.blocks[((size_t) blk * UNC_BLK + i) * 2 + 1];
    Clu c; c.ren_start = a.x; c.evt_en = a.y; c.ref_st = a.z; c.ren_end = a.w; c.evt_st = b.x; c.total_len = b.y;
    return c;
}
UNC_DEV void trk_store(const Tracker &t, u32 blk, u32 i, const Clu &c) {
    t.blocks[((size_t) blk * UNC_BLK + i) * 2] = make_uint4(c.ren_start, c.evt_en, c.ref_st, c.ren_end);
    t.blocks[((size_t) blk * UNC_BLK + i) * 2 + 1] = make_uint4(c.evt_st, c.total_len, 0, 0);
}

// Global lower_bound of key (ks, ke): returns directory index d and position pos inside
// block d (pos may equal the block's count => the bound is the first entry of block d+1).
// On return *cnt_out = count of block d, and `mine` holds entry `lane` of block d (if lane < count).
UNC_DEV void trk_lower_bound(const Tracker &t, u32 ks, u32 ke, u32 *d_out, u32 *pos_out, u32 *blk_out, u32 *cnt_out,
                             Clu *mine) {
    int lane = w_lane();
    // number of directory entries whose first key is < key
    u32 lo = 0, hi = t.nb, c = 0;
    for (;;) {
        u32 span = hi - lo;
        if (span == 0) { c = lo; break; }
        u32 step = (span + 31u) / 32u;
        u32 idx = lo + (u32) lane * step;
        bool less = false;
        if (idx < hi) { uint4 e = t.dir[idx]; less = clu_less(e.x, e.y, ks, ke); }
        u32 nl = (u32) d_popc(w_ballot(less));
        if (step == 1) { c = lo + nl; break; }
        if (nl == 0) { c = lo; break; }
        u32 nlo = lo + (nl - 1) * step + 1;
        u32 nhi = lo + nl * step; if (nhi > hi) nhi = hi;
        lo = nlo; hi = nhi;
    }
    u32 d = c > 0 ? c - 1 : 0;
    uint4 de = t.dir[d];
    u32 blk = de.z, cnt = de.w;
    Clu m; m.ren_start = 0; m.evt_en = 0; m.ref_st = 0; m.ren_end = 0; m.evt_st = 0; m.total_len = 0;
    if ((u32) lane < cnt) m = trk_load(t, blk, (u32) lane);
    const bool less = (u32) lane < cnt && clu_less(m.ren_start, m.evt_en, ks, ke);
    *pos_out = (u32) d_popc(w_ballot(less));
    *d_out = d; *blk_out = blk; *cnt_out = cnt; *mine = m;
}

// room for one more directory entry: a directory that outgrows its shared-memory copy moves to the workspace for good
UNC_DEV void trk_dir_reserve(Tracker &t) {
    if (t.dir != t.dir_glob && t.nb + 1u > t.dir_cap) {
        for (u32 i = (u32) w_lane(); i < t.nb; i += 32u) t.dir_glob[i] = t.dir[i];
        w_sync();
        t.dir = t.dir_glob;
    }
}
// shift directory entries [from, nb) up by one (warp memmove, top-down)
UNC_DEV void trk_dir_open(Tracker &t, u32 from) {
    int lane = w_lane();
    u32 n = t.nb - from;  // entries to move
    for (u32 done = 0; done < n; done += 32) {
        u32 chunk_hi = t.nb - done;                 // exclusive
        u32 idx = chunk_hi - 1 - (u32) lane;        // process from the top
        bool act = ((u32) lane < n - done) && ((u32) lane < 32);
        uint4 e = make_uint4(0, 0, 0, 0);
        if (act) e = t.dir[idx];
        w_sync();
        if (act) t.dir[idx + 1] = e;
        w_sync();
    }
}
// remove directory entry d (shift [d+1, nb) down by one)
UNC_DEV void trk_dir_close(Tracker &t, u32 d) {
    int lane = w_lane();
    for (u32 base = d + 1; base < t.nb; base += 32) {
        u32 idx = base + (u32) lane;
        bool act = idx < t.nb;
        uint4 e = make_uint4(0, 0, 0, 0);
        if (act) e = t.dir[idx];
        w_sync();
        if (act) t.dir[idx - 1] = e;
        w_sync();
    }
    t.nb--;
}

// std::set::erase of entry (d, pos)
UNC_DEV void trk_erase(Tracker &t, u32 d, u32 pos) {
    int lane = w_lane();
    uint4 de = t.dir[d];
    u32 blk = de.z, cnt = de.w;
    Clu m; m.ren_start = 0; m.evt_en = 0;
    bool have = (u32) lane < cnt;
    if (have) m = trk_load(t, blk, (u32) lane);
    w_sync();
    if (have && (u32) lane > pos) trk_store(t, blk, (u32) lane - 1, m);
    w_sync();
    cnt--;
    t.n_live--;
    if (cnt == 0) {
        trk_dir_close(t, d);
    } else {
        // new first key: entry that is now at slot 0
        u32 src = pos == 0 ? 1u : 0u;
        u32 fs = w_shfl(m.ren_start, (int) src), fe = w_shfl(m.evt_en, (int) src);
        if (lane == 0) t.dir[d] = make_uint4(fs, fe, blk, cnt);
        w_sync();
    }
}

// What trk_lower_bound found for a key: directory index, position in the block, the block and its entries (one per lane)
struct TrkBound { u32 d, pos, blk, cnt; Clu m; };

// std::set::insert (unique keys): returns false when an equivalent key is already present.  `known` = the lower bound
// of c's key in the set as it is now (the caller has searched for exactly this key), or null.
UNC_DEV bool trk_insert_unique(Tracker &t, const Clu &c, const TrkBound *known = nullptr) {
    int lane = w_lane();
    if (t.nb == 0) {
        if (t.n_alloc >= t.max_blocks) { t.overflow = 1; return false; }
        u32 blk = t.n_alloc++;
        if (lane == 0) { trk_store(t, blk, 0, c); t.dir[0] = make_uint4(c.ren_start, c.evt_en, blk, 1); }
        w_sync();
        t.nb = 1; t.n_live++;
        return true;
    }
    for (;;) {
        u32 d, pos, blk, cnt; Clu m;
        if (known) { d = known->d; pos = known->pos; blk = known->blk; cnt = known->cnt; m = known->m; known = nullptr; }
        else trk_lower_bound(t, c.ren_start, c.evt_en, &d, &pos, &blk, &cnt, &m);
        // element at the bound
        u32 bs, be; bool have_bound = true;
        if (pos < cnt) { bs = w_shfl(m.ren_start, (int) pos); be = w_shfl(m.evt_en, (int) pos); }
        else if (d + 1 < t.nb) { uint4 nx = t.dir[d + 1]; bs = nx.x; be = nx.y; }
        else { have_bound = false; bs = be = 0; }
        if (have_bound && bs == c.ren_start && be == c.evt_en) return false;
        if (cnt < UNC_BLK) {
            w_sync();
            if ((u32) lane < cnt && (u32) lane >= pos) trk_store(t, blk, (u32) lane + 1, m);
            if (lane == 0) trk_store(t, blk, pos, c);
            w_sync();
            u32 fs = pos == 0 ? c.ren_start : w_shfl(m.ren_start, 0);
            u32 fe = pos == 0 ? c.evt_en : w_shfl(m.evt_en, 0);
            if (lane == 0) t.dir[d] = make_uint4(fs, fe, blk, cnt + 1);
            w_sync();
            t.n_live++;
            return true;
        }
        // full block: split the upper half into a new block, then retry
        if (t.n_alloc >= t.max_blocks) { t.overflow = 1; return false; }
        u32 nblk = t.n_alloc++;
        if (lane >= 16) trk_store(t, nblk, (u32) lane - 16, m);
        w_sync();
        trk_dir_reserve(t);
        trk_dir_open(t, d + 1);
        u32 s16 = w_shfl(m.ren_start, 16), e16 = w_shfl(m.evt_en, 16);
        u32 s0 = w_shfl(m.ren_start, 0), e0 = w_shfl(m.evt_en, 0);
        if (lane == 0) {
            t.dir[d] = make_uint4(s0, e0, blk, 16);
            t.dir[d + 1] = make_uint4(s16, e16, nblk, 16);
        }
        w_sync();
        t.nb++;
    }
}

// std::multiset<u32> all_lens_: only its size and two largest values are ever read
// (reference src/seed_tracker.cpp:129-143).  Values only arrive by insert(v) or by replacing
// one instance of `oldv` with a strictly larger `newv` (:199-203), so the top two can be
// maintained exactly without storing the multiset.
UNC_DEV void lens_insert(Tracker &t, u32 v) {
    t.n_lens++;
    if (v > t.top1) { t.top2 = t.top1; t.top1 = v; }
    else if (v > t.top2) t.top2 = v;
}
UNC_DEV void lens_replace(Tracker &t, u32 oldv, u32 newv) {
    if (oldv == t.top1) { t.top1 = newv; }                       // top2 unchanged (other copy or smaller)
    else if (oldv == t.top2) { if (newv > t.top1) { t.top2 = t.top1; t.top1 = newv; } else t.top2 = newv; }
    else { if (newv > t.top1) { t.top2 = t.top1; t.top1 = newv; } else if (newv > t.top2) t.top2 = newv; }
}

// SeedCluster::update (reference src/seed_tracker.cpp:56-73), growth truncated to u8
UNC_DEV void clu_update(Clu &a, const Clu &ns) {
    u32 growth = 0;
    if (ns.ren_start < a.ren_end) {
        if (ns.ren_end > a.ren_end) {
            growth = (ns.ren_end - a.ren_end) & 0xFFu;
            a.ren_start = ns.ren_start; a.ren_end = ns.ren_end;
        } else {
            a.ren_start = ns.ren_start;
        }
    } else {
        growth = ns.total_len & 0xFFu;
        a.ren_start = ns.ren_start; a.ren_end = ns.ren_end;
    }
    a.evt_en = ns.evt_en;
    a.total_len += growth;
}

// SeedTracker::add_seed (reference src/seed_tracker.cpp:157-232), executed cooperatively by
// the warp with uniform control flow.
UNC_DEV void trk_add_seed(Tracker &t, const DevParams &p, u32 ref_en, u32 ref_len, u32 evt) {
    Clu ns;
    ns.ren_start = ref_en - ref_len + 1; ns.ren_end = ref_en; ns.ref_st = ns.ren_start;
    ns.evt_st = evt; ns.evt_en = evt; ns.total_len = ref_len;
    const u32 e2 = evt, r2 = ns.ren_start;
    bool found = false; u32 md = 0, mpos = 0, best_len = 0;

    TrkBound lb;                                   // where the new seed's own key would go: the scan starts there
    bool have_lb = false;
    PT_TRK0(t)
    if (t.nb > 0) {
        u32 d, pos, blk, cnt; Clu m;
        trk_lower_bound(t, ns.ren_start, ns.evt_en, &d, &pos, &blk, &cnt, &m);
        PT_TRK(t, 0)
        lb.d = d; lb.pos = pos; lb.blk = blk; lb.cnt = cnt; lb.m = m; have_lb = true;
        int lane = w_lane();
        bool broke = false;
        u32 first = pos;
        while (!broke && d < t.nb) {
            bool valid = (u32) lane < cnt && (u32) lane >= first;
            u32 e1 = m.evt_en, r1 = m.ren_start;
            bool inr = valid && e1 <= e2 && (r2 - r1) <= (e2 - e1) && (r2 - r1) >= (e2 - e1) / 12u;
            bool brk = valid && (r2 - r1) >= e2;
            u32 m_inr = w_ballot(inr), m_brk = w_ballot(brk);
            u32 cand = m_inr | m_brk;
            while (cand) {
                int l = d_ffs(cand) - 1;
                cand &= cand - 1;
                bool matched = false;
                if ((m_inr >> l) & 1u) {
                    u32 tl = w_shfl(m.total_len, l);
                    if (!found || best_len < tl) { found = true; best_len = tl; md = d; mpos = (u32) l; matched = true; }
                }
                if (!matched && ((m_brk >> l) & 1u)) { broke = true; break; }
            }
            if (broke) break;
            d++;
            if (d < t.nb) {
                uint4 de = t.dir[d];
                blk = de.z; cnt = de.w; first = 0;
                if ((u32) lane < cnt) m = trk_load(t, blk, (u32) lane);
            }
        }
    }

    PT_TRK(t, 1)
    if (found) {
        // the matched cluster's block: still in registers when it is the block the scan started in
        const int lane = w_lane();
        u32 blk, cnt; Clu mm;
        if (md == lb.d) { blk = lb.blk; cnt = lb.cnt; mm = lb.m; }
        else {
            uint4 de = t.dir[md];
            blk = de.z; cnt = de.w;
            mm.ren_start = 0; mm.evt_en = 0; mm.ref_st = 0; mm.ren_end = 0; mm.evt_st = 0; mm.total_len = 0;
            if ((u32) lane < cnt) mm = trk_load(t, blk, (u32) lane);
        }
        Clu a;
        a.ren_start = w_shfl(mm.ren_start, (int) mpos); a.evt_en = w_shfl(mm.evt_en, (int) mpos); a.ref_st = w_shfl(mm.ref_st, (int) mpos);
        a.ren_end = w_shfl(mm.ren_end, (int) mpos); a.evt_st = w_shfl(mm.evt_st, (int) mpos); a.total_len = w_shfl(mm.total_len, (int) mpos);
        u32 prev_len = a.total_len;
        clu_update(a, ns);
        if (a.total_len != prev_len) {
            t.len_sum = f_add(t.len_sum, (float) (a.total_len - prev_len));
            lens_replace(t, prev_len, a.total_len);
            if (a.total_len >= p.min_map_len && a.total_len > t.max_map.total_len) t.max_map = a;
        }
        // erase + insert (reference src/seed_tracker.cpp:205-213).  The key only moves towards the front of the set
        // (ren_start never decreases; with it equal, evt_en does not); while it stays behind its predecessor the
        // cluster keeps its place and is rewritten where it is.  An equal predecessor (the insert would fail) and the
        // first entry of a later block take the general path.
        bool in_place = false;
        if (mpos > 0) {
            const u32 ps = w_shfl(mm.ren_start, (int) mpos - 1), pe = w_shfl(mm.evt_en, (int) mpos - 1);
            in_place = clu_less(ps, pe, a.ren_start, a.evt_en);
        } else in_place = md == 0;
        if (in_place) {
            w_sync();
            if (lane == 0) {
                trk_store(t, blk, mpos, a);
                if (mpos == 0) t.dir[md] = make_uint4(a.ren_start, a.evt_en, blk, cnt);
            }
            w_sync();
        } else {
            trk_erase(t, md, mpos);
            trk_insert_unique(t, a);
        }
    } else {
        lens_insert(t, ns.total_len);
        t.len_sum = f_add(t.len_sum, (float) ns.total_len);
        if (ns.total_len >= p.min_map_len && ns.total_len > t.max_map.total_len) t.max_map = ns;
        trk_insert_unique(t, ns, have_lb ? &lb : nullptr);
    }
    PT_TRK(t, 2)
}

// SeedTracker::get_final + check_map_conf (reference src/seed_tracker.cpp:129-143,259-262)
UNC_DEV bool trk_get_final(const Tracker &t, const DevParams &p) {
    if (t.max_map.total_len < p.min_map_len || t.n_lens < 2) return false;
    float mean_len = f_div(t.len_sum, (float) t.n_live);
    float second_len = (float) t.top2;
    float sl = (float) t.max_map.total_len;
    return (p.min_mean_conf > 0 && f_div(sl, mean_len) >= p.min_mean_conf) ||
           (p.min_top_conf > 0 && f_div(sl, second_len) >= p.min_top_conf);
}


// ------------------------------------------------------------------ K2: mapper (one CTA per read)
//
// Warp 0 of the CTA is the TRACKER: it owns the seed-cluster set (sequential by nature) and
// runs one event behind the other warps.  Warps 1.. are WORKERS: per event they score the 1024
// k-mers, extend all paths, sort the children, dedup + emit sources, and look up the suffix
// array for the event's seeds, which they hand to the tracker through a double-buffered list.
// The workers come in two structures.  unc_k2_workers_v2 (unc_k2v2.cuh) runs k2_map, k2_map_ord
// and k2_map_stream.  unc_k2_workers_exact below runs the exact-ties kernels: it extends chunks
// of 32 paths per warp into chunk-local slots (emission order restored by a scan), radix-sorts
// the children, and re-sorts an event's children with the reference's pdqsort when two of them
// tie.
//
// Path record = 2 uint4 (32 B):
//   q0 = (fm_start, fm_end, kmer | length<<16 | consec_stays<<24, event_moves | sa_checked<<31)
//   q1 = (seed_prob bits, C = cumulative log-prob since the path's source, 0, 0)
// The reference's 23-float prob_sums_ window (src/mapper.cpp:792-801) is only ever read at its two
// ends: C(e-1) to extend and C(e-22) once the path is seed_len long.  C(e-1) is the parent's C.
// C(e-22) is the C of the ancestor 22 generations back, found through hist[generation % 24][idx] =
// (C, parent idx); only ~2 % of children have a full-length parent, and those look-ups are
// deferred to a separate pass so the extension loop never waits on the 22-hop walk.
// Sort key (ckey) = (fm_start, fm_end, seed_prob bits, kmer | seedable<<10 | move_count<<11 | emission idx<<16)
#define K2_MAXCH 1024u     /* chunks of 32 paths (max_paths <= 32767) */
#define K2_CH_SLOTS 160u   /* 32 parents x at most 5 children */
#define K2_V2_DYN_BYTES (16u + K2_MAXSEG * (K2_CH_SLOTS * 8u + K2_CH_SLOTS))   /* per-warp child staging of unc_k2v2.cuh */
#define K2_RBITS 8u        /* radix digit width of the child sort */
#define K2_RB 256u
#define K2_MAXSEG 16u      /* max worker warps (sort segments) */
#define K2_DYN_PER_CHUNK 24u   /* pre 8 + agg 8 + bcnt 4 + ecnt 4 bytes of dynamic shared memory per 32 paths */
/* dynamic shared memory of a mapper CTA: the struct, the per-chunk arrays, the per-warp child staging */
#define K2_SMEM_BYTES(maxp) (sizeof(K2Shared) + 16 + (size_t) (((maxp) + 31) / 32) * K2_DYN_PER_CHUNK + 32 + K2_V2_DYN_BYTES)
struct K2Tables {
    uint2 kmer_range[UNC_NKMER];
    float thresh[64];
};
struct K2V2 {              // second worker structure (unc_k2v2.cuh)
    K2V2Tab t;
    u32 kcnt[UNC_NKMER];   // per k-mer bucket: children counted during the extension, then the scatter cursor (= bucket end)
    u32 koff[UNC_NKMER];   // bucket start in the sorted key array
    u32 kagg[UNC_NKMER];   // (gap sources | child seeds << 16) of the bucket, then their exclusive prefix
    u32 fresh_cand[32], fresh_mask[32], fresh_before[32];   // fresh-source candidates / plan per 32-k-mer word
    u32 grab[2];           // bucket hand-out counters (sort pass, emit pass)
    u32 n_units;           // 32-key chunks of large buckets listed for the emit pass (W.elist)
    u16 mfirst[K2V2_MAX_MERGED];   // per merged-group k-mer: gap sources of its bucket before its first run (0xFFFF: no run)
#if defined(UNC_PHASE_TIMING) && !defined(UNC_EMUL)
    u32 pt_dur[4][K2_MAXSEG];      // phase-timing builds: every worker warp's own time in B / C2 / D1 / E of the event
#endif
};
struct K2Shared {          // per CTA
    K2Tables tb;
    float probs[UNC_NKMER];
    u32 flags[32];         // sources_added_ bits (reference src/mapper.cpp:88), kmer k -> word k>>5
    u32 flags_prev[32];    // the flags as the previous event left them (restored when the event in flight is discarded)
    u32 hist_cur[K2_RB * K2_MAXSEG];    // [digit][segment]
    u32 hist_next[K2_RB * K2_MAXSEG];
    // per-chunk arrays carved from dynamic shared memory (ceil(max_paths/32) entries each)
    uint2 *agg;            // D1 aggregates of the k-mer run structure
    u64 *pre;              // D2 look-back prefix words: (epoch<<2 | state) << 32 | sources | seeds<<16
    u32 *bcnt, *ecnt;      // children per chunk (then exclusive prefix), ended paths per chunk
    K2V2 v2;
    unsigned char *v2_stage;   // K2V2_STAGE_BYTES per worker warp (dynamic shared memory)
    u32 bc[8];             // CTA broadcast scalars
    u32 scan_tmp[32];
    u32 n_rows[2];         // worker -> tracker: seed rows of event e in rlist[e & 1]
    u32 verdict[2];        // tracker -> workers: outcome of event e in verdict[e & 1]
    u32 wk_overflow;
    u32 wl_cnt;            // deferred window look-ups of the event in flight
    u32 cnt_blocks, cnt_steps;
    u32 tot_children[2], tot_sources[2];   // u64 as two words, written by a worker at the end
};

#include "unc_pdqsort.cuh"
#ifdef UNC_EMUL
static unsigned long g_emu_tie_stats[2];   // test statistics of the exact-ties path (emulator builds only)
#endif

// exclusive scan over the K2_RB*K2_MAXSEG sort counters by the worker threads:
// dst[i] = sum(src[0..i)); src := 0.   wt = worker thread index, nwt = worker thread count.
UNC_DEV void k2_wk_exscan_bins(K2Shared *sh, u32 *src, u32 *dst, u32 wt, u32 nwt) {
    const u32 n = K2_RB * K2_MAXSEG;
    const u32 per = (n + nwt - 1) / nwt;
    const u32 lo = wt * per < n ? wt * per : n, hi = lo + per < n ? lo + per : n;
    u32 sum = 0;
    for (u32 j = lo; j < hi; j++) sum += src[j];
    u32 wtot, woff = w_exscan(sum, &wtot);
    if (w_lane() == 31) sh->scan_tmp[wt >> 5] = wtot;
    c_sync_sub(1, (int) nwt);
    if (wt < 32) {
        u32 v = wt < (nwt >> 5) ? sh->scan_tmp[wt] : 0, t;
        u32 e = w_exscan(v, &t);
        sh->scan_tmp[wt] = e;
    }
    c_sync_sub(1, (int) nwt);
    u32 run = sh->scan_tmp[wt >> 5] + woff;
    for (u32 j = lo; j < hi; j++) {
        u32 cnt = src[j];
        dst[j] = run;
        src[j] = 0;
        run += cnt;
    }
    c_sync_sub(1, (int) nwt);
}

// PathBuffer::make_source (reference src/mapper.cpp:751-772): prob_sums_ = {0, prob}
UNC_DEV void write_source(uint4 *rec, uint2 *hist_e, u32 idx, u32 st, u32 en, u32 kmer, float prob) {
    rec[(size_t) idx * 2] = make_uint4(st, en, kmer | (1u << 16), 1u);
    rec[(size_t) idx * 2 + 1] = make_uint4(f2u(prob), f2u(prob), 0u, 0u);
    hist_e[idx] = make_uint2(f2u(prob), 0xFFFFFFFFu);
}

// Mapper::event_to_bp (reference src/mapper.cpp:703-706)
UNC_DEV u32 unc_event_to_bp(u32 evt_i, bool last, float mean_event_len, float bp_per_samp) {
    float v = f_add(f_mul(f_mul((float) evt_i, mean_event_len), bp_per_samp), (float) (last ? 4 : 0));
    return f_to_u32_x86(v);
}

// stage the pore model, k-mer FM ranges and thresholds in shared memory (once per CTA)
UNC_DEV void unc_k2_cta_setup(const DevIndex &ix, const DevParams &p, K2Shared *sh) {
    const u32 n_slots = (p.max_paths + 31u) >> 5;
    if (c_tid() == 0) {   // dynamic shared memory follows the struct
        char *base = (char *) ((((size_t) (sh + 1)) + 15) & ~(size_t) 15);
        sh->pre = (u64 *) base; base += (size_t) n_slots * 8;
        sh->agg = (uint2 *) base; base += (size_t) n_slots * 8;
        sh->bcnt = (u32 *) base; base += (size_t) n_slots * 4;
        sh->ecnt = (u32 *) base;
        sh->v2_stage = (unsigned char *) sh->pre + (size_t) n_slots * K2_DYN_PER_CHUNK + 8;
        sh->v2_stage = (unsigned char *) ((((size_t) sh->v2_stage) + 15) & ~(size_t) 15);
    }
    c_sync();
    for (u32 k = (u32) c_tid(); k < UNC_NKMER; k += (u32) c_nthreads()) {
        sh->tb.kmer_range[k] = ix.kmer_range[k];
    }
    for (u32 k = (u32) c_tid(); k < 64; k += (u32) c_nthreads()) sh->tb.thresh[k] = ix.thresh[k];
    for (u32 k = (u32) c_tid(); k < (u32) (sizeof(K2V2Tab) / 4); k += (u32) c_nthreads()) ((u32 *) &sh->v2.t)[k] = ((const u32 *) ix.kt)[k];
    for (u32 c = (u32) c_tid(); c < n_slots; c += (u32) c_nthreads()) sh->pre[c] = 0;
    c_sync();
}

// The read's result record (one lane): reference src/mapper.cpp:631-653 (get_final -> set_ref_loc), :708-728,
// bwa_index.hpp:213-220
UNC_DEV void unc_k2_write_record(const DevIndex &ix, const DevParams &p, const DevBatch &B, K2Shared *sh, u32 r,
                                 const Tracker &trk, u32 verdict, u32 final_event, u64 n_seeds) {
    const float mel = B.mean_event_len[r];
    const float bp_per_samp = f_div(p.bp_per_sec, p.sample_rate);
    DevRec o;
    o.mapped = 0; o.fwd = 0; o.rid = -1; o.status = verdict == 2u ? -7 : 0;
    o.n_events = B.n_events[r]; o.events_used = final_event; o.matches = 0; o.n_clusters = trk.n_live;
    o.rd_len = f_to_u64(f_mul((float) (u64) B.reads[r].n_samples, bp_per_samp));
    o.rd_st = o.rd_en = o.rf_st = o.rf_en = o.rf_len = 0;
    if (verdict == 1u) {
        const Clu &sc = trk.max_map;
        bool fwd = sc.ref_st < ix.seq_len / 2u;
        u64 sa_st = fwd ? (u64) sc.ref_st : (u64) ix.seq_len - ((u64) sc.ren_end + 4u);
        o.rd_st = unc_event_to_bp(sc.evt_st - UNC_SEED_LEN, false, mel, bp_per_samp);
        o.rd_en = unc_event_to_bp(sc.evt_en, true, mel, bp_per_samp);
        o.rd_len = unc_event_to_bp(final_event, true, mel, bp_per_samp);
        // bns_pos2rid (reference submods/bwa/bntseq.c:354-368)
        int rid = -1;
        if ((long long) sa_st < (long long) B.l_pac) {
            int left = 0, mid = 0, right = (int) B.n_seqs;
            while (left < right) {
                mid = (left + right) >> 1;
                if (sa_st >= B.seq_offsets[mid]) {
                    if (mid == (int) B.n_seqs - 1) break;
                    if (sa_st < B.seq_offsets[mid + 1]) break;
                    left = mid + 1;
                } else right = mid;
            }
            rid = mid;
        }
        u64 rf_st = 0, rf_len = 0;
        if (rid >= 0) { rf_st = sa_st - B.seq_offsets[rid]; rf_len = B.seq_lens[rid]; }
        o.mapped = 1; o.fwd = fwd ? 1 : 0; o.rid = rid;
        o.rf_st = rf_st; o.rf_len = rf_len;
        o.rf_en = rf_st + ((u64) sc.ren_end - (u64) sc.ref_st + 5u);
        o.matches = (sc.total_len + 4u) & 0xFFFFu;
    }
    o.n_children = ((u64) sh->tot_children[1] << 32) | sh->tot_children[0];
    o.n_sources = ((u64) sh->tot_sources[1] << 32) | sh->tot_sources[0];
    o.n_seeds = n_seeds;
    o.n_occ_blocks = sh->cnt_blocks; o.n_sa_steps = sh->cnt_steps;
    B.out[r] = o;
}

#if defined(UNC_PHASE_TIMING) && !defined(UNC_EMUL)
// cycle counter with a compiler memory barrier, so that loads/stores of a phase are not scheduled across a mark
UNC_DEV long long pt_clock() { long long v; asm volatile("mov.u64 %0, %%clock64;" : "=l"(v) :: "memory"); return v; }
#define PT_DECL unsigned long long pt_acc[32]; for (int _i = 0; _i < 32; _i++) pt_acc[_i] = 0; long long pt_t = pt_clock();
// timeline of one read: events UNC_PT_TRACE_E0 .. +8, every warp's clock at every mark (behind the per-read counters)
#define UNC_PT_TRACE_READ 40u
#define UNC_PT_TRACE_E0 60u
#define UNC_PT_TRACE_BYTES (8u * 16u * 32u * 8u)
#define PT_TRACE(ev, i, t) if ((B).dbg && r == UNC_PT_TRACE_READ && (ev) - UNC_PT_TRACE_E0 < 8u && (c_tid() & 31) == 0) \
        (B).dbg[(size_t) (B).n_reads * 64 + ((size_t) ((ev) - UNC_PT_TRACE_E0) * 16 + (c_tid() >> 5)) * 32 + (i)] = (unsigned long long) (t);
#define PT_MARK(i) { long long _n = pt_clock(); pt_acc[i] += (unsigned long long) (_n - pt_t); pt_t = _n; PT_TRACE(event_i, i, _n) }
// two observers per read: thread 0 of worker warp 0 (which also runs the single-warp sections: chunk scan,
// ended rows, fresh sources) -> counters 0..7, and lane 0 of the LAST worker warp (never runs them, so its
// barrier waits expose them) -> counters 16..31.  Marks 0..6 = phases A..X, 8 = verdict + bookkeeping after the event
// barrier, 9 = loop back-edge, 7 = the event's load and scaling (8 + 9 + 7 = the former "loop head")
#define PT_FLUSH(B, r) if ((B).dbg && (wt == 0 || wt == nwt - 32u)) { for (int _i = 0; _i < (wt == 0 ? 32 : 28); _i++) (B).dbg[(size_t) (r) * 64 + (wt == 0 ? 0 : 32) + _i] = pt_acc[_i]; }
// A warp leaves BAR.SYNC.DEFER_BLOCKING before the barrier completes and stalls at its next memory instruction, so a clock
// read right behind a barrier does not contain the wait.  PT_FENCE = the same barrier once more (nobody can arrive at it
// before the first has completed): the read behind it does.  PT_WB / PT_WE(ph): every worker warp times its own share of
// a phase; PT_WR(ph, s_max, s_mean): after the next barrier the observer adds the slowest warp's and the mean time.
#define PT_FENCE c_sync_sub(1, (int) nwt);
#define PT_WDECL long long pt_w0 = 0;
#define PT_WB pt_w0 = pt_clock();
#define PT_WE(ph) if (lane == 0) v2->pt_dur[ph][ww] = (u32) (pt_clock() - pt_w0);
#define PT_WARR(ph) if (lane == 0) v2->pt_dur[ph][ww] = (u32) pt_clock(); w_sync(); s_atomic_max(&v2->pt_dur[ph][ww], (u32) pt_clock());   /* arrival of the warp's last lane at the barrier that follows */
#define PT_WREL(ph) if (lane == 0 && *(volatile u32 *) &v2->grab[0] != 0xFFFFFFFFu) { const long long _t = pt_clock(); v2->pt_dur[ph][ww] = (u32) _t; PT_TRACE(event_i, 30, _t) }      /* the warp's release from the barrier before */
#define PT_WLAG(ph, s_last, s_first) if (wt == 0) { const u32 _now = (u32) pt_clock(); u32 _mn = 0xFFFFFFFFu, _mx = 0; for (u32 _w = 0; _w < nwk; _w++) { \
        const u32 _d = _now - *(volatile u32 *) &v2->pt_dur[ph][_w]; _mn = _d < _mn ? _d : _mn; _mx = _d > _mx ? _d : _mx; } pt_acc[s_last] += _mn; pt_acc[s_first] += _mx; }
#define PT_WTRK(ph, s) if (wt == 0) pt_acc[s] += (u32) pt_clock() - *(volatile u32 *) &v2->pt_dur[ph][K2_MAXSEG - 2 + (event_i & 1u)];
#define PT_WR(ph, s_max, s_mean) if (wt == 0) { u32 _mx = 0, _sm = 0; for (u32 _w = 0; _w < nwk; _w++) { const u32 _d = *(volatile u32 *) &v2->pt_dur[ph][_w]; \
        _mx = _d > _mx ? _d : _mx; _sm += _d; } pt_acc[s_max] += _mx; pt_acc[s_mean] += _sm / nwk; }
#else
#define PT_DECL
#define PT_MARK(i)
#define PT_FLUSH(B, r)
#define PT_FENCE
#define PT_WDECL
#define PT_WB
#define PT_WE(ph)
#define PT_WARR(ph)
#define PT_WLAG(ph, s_last, s_first)
#define PT_WTRK(ph, s)
#define PT_WREL(ph)
#define PT_WR(ph, s_max, s_mean)
#endif

// ---- tracker warp (warp 0): reference src/mapper.cpp:513-519,601 (update_seeds order),
//      :631-653 (get_final -> set_ref_loc), :708-728, bwa_index.hpp:213-220
template <bool STREAM>
UNC_DEV void unc_k2_tracker(const DevIndex &ix, const DevParams &p, const DevBatch &B, const DevWork &W,
                            K2Shared *sh, u32 r, u32 n_first, u32 n_limit, uint4 *dir_smem, u32 dir_smem_cap) {
    const int lane = w_lane();
    Tracker trk;
    trk.blocks = W.clu; trk.dir_glob = W.dir; trk.max_blocks = W.max_blocks;
    trk.dir = dir_smem ? dir_smem : W.dir; trk.dir_cap = dir_smem ? dir_smem_cap : 0u;   // the directory's fast copy (searched for every seed)
    trk_reset(trk);
    DevMapState *ms = nullptr;
    if (STREAM) {
        ms = B.mstate + B.chan[r];
        if (ms->started) {                          // continue the read: the cluster store lives in the channel's slot
            trk.nb = ms->t_nb; trk.n_alloc = ms->t_n_alloc; trk.n_live = ms->t_n_live; trk.n_lens = ms->t_n_lens;
            trk.top1 = ms->t_top1; trk.top2 = ms->t_top2; trk.overflow = ms->t_overflow; trk.len_sum = ms->t_len_sum;
            trk.max_map.ren_start = ms->t_max_map[0]; trk.max_map.evt_en = ms->t_max_map[1]; trk.max_map.ref_st = ms->t_max_map[2];
            trk.max_map.ren_end = ms->t_max_map[3]; trk.max_map.evt_st = ms->t_max_map[4]; trk.max_map.total_len = ms->t_max_map[5];
            if (trk.dir != trk.dir_glob) {          // the directory as the previous chunk left it
                if (trk.nb <= trk.dir_cap) { for (u32 j = (u32) lane; j < trk.nb; j += 32u) trk.dir[j] = trk.dir_glob[j]; w_sync(); }
                else trk.dir = trk.dir_glob;
            }
        }
    }
    u32 verdict = 0, i = n_first, final_event = n_limit;
    u64 n_seeds = 0;
#if defined(UNC_PHASE_TIMING) && !defined(UNC_EMUL)
    trk.pt[0] = trk.pt[1] = trk.pt[2] = 0;
#endif
    for (;;) {
#if defined(UNC_PHASE_TIMING) && !defined(UNC_EMUL)
        if (lane == 0) *(volatile u32 *) &sh->v2.pt_dur[3][K2_MAXSEG - 2 + (i & 1u)] = (u32) pt_clock();   // the tracker's arrival at the event barrier
        PT_TRACE(i, 0, pt_clock())
#endif
        c_sync();                                  // b_i: workers finished event i (or this is the final barrier)
        if (i == n_limit) break;
        if (verdict) { c_sync(); break; }          // event i is discarded; final barrier
        const uint2 *rl = W.rlist + (size_t) (i & 1u) * W.rl_cap;
#if defined(UNC_PHASE_TIMING) && !defined(UNC_EMUL)
        const long long trk_t0 = pt_clock();
        PT_TRACE(i, 1, trk_t0)
#endif
        const u32 n = *(volatile u32 *) &sh->n_rows[i & 1u];
#if defined(UNC_PHASE_TIMING) && !defined(UNC_EMUL)
        PT_TRACE(i, 2, pt_clock())
        PT_TRACE(i, 4, n)
#endif
        // seed clustering is sequential: ended paths' seeds (event i-1) in parent order, then the
        // children's (event i) in sorted order
        for (u32 j0 = 0; j0 < n; j0 += 32u) {         // 32 rows per load
            uint2 mine = make_uint2(0, 0);
            if (j0 + (u32) lane < n) mine = rl[j0 + (u32) lane];
            const u32 nj = n - j0 < 32u ? n - j0 : 32u;
            for (u32 j = 0; j < nj; j++) {
                const u32 ex = w_shfl(mine.x, (int) j), ey = w_shfl(mine.y, (int) j);
                trk_add_seed(trk, p, ex, ey & 0xFFu, (ey & 0x100u) ? i - 1u : i);
            }
        }
        n_seeds += n;
        u32 v = (trk.overflow || *(volatile u32 *) &sh->wk_overflow) ? 2u : (trk_get_final(trk, p) ? 1u : 0u);
        if (v) { verdict = v; final_event = i; }
        if (lane == 0) *(volatile u32 *) &sh->verdict[i & 1u] = v;
#if defined(UNC_PHASE_TIMING) && !defined(UNC_EMUL)
        PT_TRACE(i, 3, pt_clock())
#endif
        i++;
    }
    if (STREAM && trk.dir != trk.dir_glob) { for (u32 j = (u32) lane; j < trk.nb; j += 32u) trk.dir_glob[j] = trk.dir[j]; w_sync(); }
    if (STREAM && lane == 0) {                      // what the next map_chunk of this read resumes from
        ms->t_nb = trk.nb; ms->t_n_alloc = trk.n_alloc; ms->t_n_live = trk.n_live; ms->t_n_lens = trk.n_lens;
        ms->t_top1 = trk.top1; ms->t_top2 = trk.top2; ms->t_overflow = trk.overflow; ms->t_len_sum = trk.len_sum;
        ms->t_max_map[0] = trk.max_map.ren_start; ms->t_max_map[1] = trk.max_map.evt_en; ms->t_max_map[2] = trk.max_map.ref_st;
        ms->t_max_map[3] = trk.max_map.ren_end; ms->t_max_map[4] = trk.max_map.evt_st; ms->t_max_map[5] = trk.max_map.total_len;
        ms->event_i = final_event;
        ms->started = 1;
    }
#if defined(UNC_PHASE_TIMING) && !defined(UNC_EMUL)
    if (B.dbg && lane == 0) { unsigned long long *d = B.dbg + (size_t) r * 64 + 60; d[0] = trk.pt[0]; d[1] = trk.pt[1]; d[2] = trk.pt[2]; d[3] = n_seeds; }
#endif
    // all workers have passed the final barrier: their counters are in shared memory
    if (lane == 0) unc_k2_write_record(ix, p, B, sh, r, trk, verdict, final_event, n_seeds);
}


// ---- worker warps: reference src/mapper.cpp:433-663 (map_next) minus the seed clustering
//
// No inter-warp ordering on the hot loops: phase B writes each chunk's children to chunk-local
// ("sparse") slots, a small scan + key compaction restores the emission order afterwards; phase D
// resolves the k-mer-run carry from per-chunk aggregates and the source/seed positions with a
// decoupled look-back prefix sum.

UNC_DEV u32 k2_pre_pack(u32 epoch, u32 state) { return (epoch << 2) | state; }

// The exact-ties worker.  The sources_added_ words are an input / output of the read: it keeps what the previous
// event left, so that an event that is discarded because the read mapped one event earlier leaves no trace in them.
template <bool STREAM>
UNC_DEV void unc_k2_workers_exact(const DevIndex &ix, const DevParams &p, const DevBatch &B, const DevWork &W,
                                  K2Shared *sh, u32 r, u32 n_first, u32 n_limit, u32 *epoch_io) {
    const int lane = w_lane();
    const u32 wt = (u32) c_tid() - 32u, nwt = (u32) c_nthreads() - 32u;   // worker thread index / count
    const u32 ww = wt >> 5, nwk = nwt >> 5;                               // worker warp index / count
    const K2Tables *tb = &sh->tb;
    const u32 maxp = p.max_paths;
    const u32 S0 = ((maxp + 31u) >> 5) * K2_CH_SLOTS;                     // record index of the first source
    const size_t gen_recs = (size_t) S0 + maxp;
    const float scale = B.scale[r], shift = B.shift[r];
    const float *events = B.events + (size_t) r * B.ev_stride;
    const float source_prob = tb->thresh[0];
    u64 n_children = 0, n_sources = 0;                 // committed (events confirmed by the tracker)
    u32 pend_children = 0, pend_sources = 0;           // of the event in flight
    u32 my_blocks = 0, my_steps = 0, pend_blocks = 0, pend_steps = 0;
    u32 epoch = *epoch_io;
    u32 prev_size = 0, gen = 0, event_i = n_first;
    if (STREAM) {                                      // resume: the previous chunk's last generation is in the slot
        const DevMapState *ms = B.mstate + B.chan[r];
        if (ms->started) { prev_size = ms->prev_size; gen = ms->gen; }
    }
    const u32 npass = (ix.start_bits + K2_RBITS - 1) / K2_RBITS;
    const u32 lt = w_lanemask_lt();
    PT_DECL

    for (; event_i < n_limit; event_i++) {
        PT_MARK(9)
        const float event = f_add(f_mul(scale, events[event_i - n_first]), shift);
        PT_MARK(7)

        // ---- A. pore-model probabilities (reference src/mapper.cpp:443-445)
        if (wt < 32u) sh->flags_prev[wt] = sh->flags[wt];               // what the read ends with if this event is discarded
        for (u32 k = wt; k < UNC_NKMER; k += nwt)
            sh->probs[k] = unc_match_prob(event, d_ldg(ix.lv_mean + k), d_ldg(ix.lv_var2 + k), d_ldg(ix.lognorm + k));
        c_sync_sub(1, (int) nwt);
        PT_MARK(0)

        uint4 *prev = W.paths + (size_t) gen * gen_recs * 2, *next = W.paths + (size_t) (gen ^ 1u) * gen_recs * 2;
        uint2 *hist_e = W.hist + (size_t) (event_i % UNC_NGEN) * gen_recs;
        const u32 *oprev = W.order + (size_t) gen * maxp;
        u32 *onext = W.order + (size_t) (gen ^ 1u) * maxp;
        uint4 *ckA = W.ckey, *ckB = W.ckey + maxp, *cks = W.cks;
        uint2 *rlist = W.rlist + (size_t) (event_i & 1u) * W.rl_cap;

        // ---- B. extend every previous path (reference src/mapper.cpp:455-524): chunk c of 32
        //      parents writes its children, in emission order, to records/keys [c*160, c*160+count)
        const u32 nch_prev = (prev_size + 31u) >> 5;
        {
            // software prefetch of the next chunk's order entry + record head
            u32 oi_n = UNC_INVALID; uint4 q0_n = make_uint4(0, 0, 0, 0), q1_n = make_uint4(0, 0, 0, 0);
            const u32 c_first = ww;
            if (c_first < nch_prev) {
                u32 pi = c_first * 32 + (u32) lane;
                if (pi < prev_size) oi_n = oprev[pi];
                if (!(oi_n & UNC_INVALID)) { const uint4 *pr = prev + (size_t) oi_n * 2; q0_n = pr[0]; q1_n = pr[1]; }
            }
            for (u32 c = c_first; c < nch_prev; c += nwk) {
                const u32 cn = c + nwk;
                const u32 oi = oi_n;
                const uint4 q0 = q0_n, q1 = q1_n;
                const bool valid = !(oi & UNC_INVALID);
                if (cn < nch_prev) {
                    u32 pi = cn * 32 + (u32) lane;
                    oi_n = pi < prev_size ? oprev[pi] : UNC_INVALID;
                    if (!(oi_n & UNC_INVALID)) { const uint4 *pr = prev + (size_t) oi_n * 2; q0_n = pr[0]; q1_n = pr[1]; }
                }
                u32 st = q0.x, en = q0.y, kmer = q0.z & UNC_KMASK, plen = (q0.z >> 16) & 0xFFu, stays = (q0.z >> 24) & 0xFFu;
                u32 moves = q0.w & UNC_PATH_MASK, sa_checked = q0.w >> 31;
                u32 want = 0; bool stay_ok = false;
                float cprob[5]; u32 cst[5], cen[5], ckm[5];
                if (valid) {
                    u32 len = en - st + 1u;
                    float thr = tb->thresh[32 + d_clz(len)];
                    float pk = sh->probs[kmer];
                    stay_ok = stays < p.max_consec_stay && pk >= thr;
                    cprob[0] = pk; cst[0] = st; cen[0] = en; ckm[0] = kmer;
#pragma unroll
                    for (u32 b = 0; b < 4; b++) {
                        u32 nk = ((kmer << 2) & UNC_KMASK) | b;
                        float pb = sh->probs[nk];
                        ckm[b + 1] = nk; cprob[b + 1] = pb;
                        if (!(pb < thr)) want |= 1u << b;   // `if (prob < thresh) continue;`
                    }
                }
                u32 cmask = stay_ok ? 1u : 0u;
                if (want) {
                    u32 ns[4], ne[4];
                    u32 ok = unc_neighbors(ix, st, en, want, ns, ne, &pend_blocks);
#pragma unroll
                    for (u32 b = 0; b < 4; b++)
                        if ((ok >> b) & 1u) { cmask |= 2u << b; cst[b + 1] = ns[b]; cen[b + 1] = ne[b]; }
                }
                u32 cc = (u32) d_popc(cmask), total;
                u32 off = w_exscan(cc, &total);
                // a childless, not yet SA-checked path may end here with seeds
                // (reference src/mapper.cpp:513-519 -> update_seeds(path, true), is_seed_valid :842-863)
                bool ended = false;
                u32 mc = (u32) d_popc(moves);
                if (valid && cc == 0 && !sa_checked) {
                    u32 len = en - st + 1u;
                    ended = plen == UNC_SEED_LEN && u2f(q1.x) >= p.min_seed_prob &&
                            ((len == 1 && (moves & 1u) && (float) ((plen - mc) & 0xFFu) <= f_mul(p.max_stay_frac, 22.0f)) ||
                             (len <= p.max_rep_copy && mc >= p.min_rep_len));
                }
                u32 m_ended = w_ballot(ended);
                if (ended) W.elist[(size_t) c * 32 + (u32) d_popc(m_ended & lt)] = make_uint4(st, en, mc, off);
                if (lane == 0) { sh->bcnt[c] = total; sh->ecnt[c] = (u32) d_popc(m_ended); }
                if (valid && cc > 0) {
                    const float prevC = u2f(q1.y);
                    u32 ci = c * K2_CH_SLOTS + off;
#pragma unroll
                    for (u32 j = 0; j < 5; j++) {
                        if (!((cmask >> j) & 1u)) continue;
                        u32 move = j > 0 ? 1u : 0u;
                        u32 nlen = plen + (plen < UNC_SEED_LEN ? 1u : 0u);
                        u32 nmoves = ((moves << 1) | move) & UNC_PATH_MASK;
                        u32 nstays = move ? 0u : stays + 1u;
                        float newC = f_add(prevC, cprob[j]);
                        float sp = 0.0f;
                        bool seedable = false;
                        if (plen == UNC_SEED_LEN) {
                            // seed_prob = (C(e) - C(e-22)) / 22 needs the ancestor 22 generations back: deferred
                            nmoves |= UNC_PATH_TAIL;
                            W.wlist[s_atomic_add(&sh->wl_cnt, 1u)] = make_uint4(ci, oi, f2u(newC), nmoves);
                        } else {
                            sp = f_div(newC, (float) nlen);
                            // is_seed_valid(path_ended = false) of the child (reference src/mapper.cpp:842-863)
                            u32 cmc = (u32) d_popc(nmoves);
                            seedable = nlen == UNC_SEED_LEN && sp >= p.min_seed_prob && cst[j] == cen[j] && (nmoves & 1u) &&
                                       (float) ((nlen - cmc) & 0xFFu) <= f_mul(p.max_stay_frac, 22.0f);
                        }
                        u32 spb = f2u(sp);
                        next[(size_t) ci * 2] = make_uint4(cst[j], cen[j], ckm[j] | (nlen << 16) | (nstays << 24), nmoves | (sa_checked << 31));
                        next[(size_t) ci * 2 + 1] = make_uint4(spb, f2u(newC), 0u, 0u);
                        hist_e[ci] = make_uint2(f2u(newC), oi);
                        cks[ci] = make_uint4(cst[j], cen[j], spb, ckm[j] | (seedable ? 1u << 10 : 0u) | ((u32) d_popc(nmoves) << 11) | (ci << 16));
                        ci++;
                    }
                }
            }
        }
        c_sync_sub(1, (int) nwt);
        // ---- B1 + B2a, concurrently.  Worker warp 0: exclusive scan of the chunk counts (restores the
        //      global emission order and gives the buffer cap, reference src/mapper.cpp:480-482,507-509,
        //      521-523: extension stops when max_paths children exist).  The other worker warps:
        //      deferred seed_prob of children whose parent was already seed_len long -- C(e-22) is the C
        //      of the ancestor 22 generations back (21 parent hops from the parent), a serial chain of
        //      dependent loads that now overlaps the (equally serial) scan.
        if (ww == 0) {
            u32 carry = 0;
            for (u32 i0 = 0; i0 < nch_prev; i0 += 32) {
                u32 v = i0 + (u32) lane < nch_prev ? sh->bcnt[i0 + lane] : 0u, t;
                u32 ex = w_exscan(v, &t);
                if (i0 + (u32) lane < nch_prev) sh->bcnt[i0 + lane] = carry + ex;
                carry += t;
            }
            if (lane == 0) sh->bc[2] = carry;
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
        c_sync_sub(1, (int) nwt);
        if (wt == 0) sh->wl_cnt = 0;
        PT_MARK(1)

        // ---- B2. ended-path seed rows and compaction of the sort keys into emission order
        const u32 nc_total = nch_prev ? sh->bc[2] : 0u;
        const u32 nc = nc_total < maxp ? nc_total : maxp;
        const u32 nch = (nc + 31u) >> 5;
        const u32 seg_ch = nch ? (nch + nwk - 1) / nwk : 1u, seg_len = seg_ch * 32u;
        if (ww == 0) {
            // seed rows of ended paths, in parent order.  A parent counts only if the buffer was not
            // yet full when the sequential scan reached it (children before it < max_paths).
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
        {
            // compact the chunk-local keys into emission order: each warp copies the chunks it
            // extended (their keys are still in its L1) to [bcnt[c], bcnt[c+1]) -- coalesced on both
            // sides -- and counts the first radix digit for the destination's sort segment
            for (u32 c = ww; c < nch_prev; c += nwk) {
                const u32 base = sh->bcnt[c];
                if (base >= nc) break;                              // later chunks lie beyond the max_paths cut
                const u32 end = c + 1 < nch_prev ? sh->bcnt[c + 1] : nc_total;
                u32 seg = base / seg_len, bound = (seg + 1u) * seg_len;
                for (u32 i = (u32) lane; base + i < end; i += 32) {
                    const u32 di = base + i;
                    if (di < nc) {
                        uint4 key = cks[(size_t) c * K2_CH_SLOTS + i];
                        ckA[di] = key;
                        while (di >= bound) { seg++; bound += seg_len; }
                        s_atomic_add(&sh->hist_next[(key.x & (K2_RB - 1u)) * K2_MAXSEG + seg], 1u);
                    }
                }
            }
        }
        c_sync_sub(1, (int) nwt);
        u32 n_rows = sh->bc[3];
        if (n_rows > W.rl_cap) n_rows = W.rl_cap;
        const u32 n_ended_rows = n_rows;
        pend_children = nc;
        PT_MARK(2)

        u32 ns_added = 0;   // sources appended after the children
        u32 n_child_seeds = 0;
        if (nc > 0) {
            // ---- C. order children by (fm_start, fm_end, seed_prob, emission index)
            //         (reference src/mapper.cpp:531 pdqsort + operator< :866-871): LSD radix sort on
            //         fm_start, 8-bit digits; worker warp w owns the w-th contiguous segment of the
            //         array in every pass, so the scatter is stable without inter-warp ordering
            uint4 *src = ckA, *dst = ckB;
            const u32 c_lo = ww * seg_ch, c_hi = (c_lo + seg_ch < nch) ? c_lo + seg_ch : nch;
            // keep the keys in emission order (the array the reference sorts) in the chunk-local key buffer, which is
            // idle until the next event's extension
            for (u32 i = wt; i < nc; i += nwt) cks[i] = ckA[i];
            if (wt == 0) sh->bc[5] = 0;
            for (u32 pass = 0; pass < npass; pass++) {
                const u32 sb = pass * K2_RBITS;
                k2_wk_exscan_bins(sh, sh->hist_next, sh->hist_cur, wt, nwt);
                uint4 kn = make_uint4(0, 0, 0, 0), kn2 = make_uint4(0, 0, 0, 0);
                if (c_lo < c_hi && c_lo * 32 + (u32) lane < nc) kn = src[c_lo * 32 + (u32) lane];
                if (c_lo + 1 < c_hi && (c_lo + 1) * 32 + (u32) lane < nc) kn2 = src[(c_lo + 1) * 32 + (u32) lane];
                for (u32 c = c_lo; c < c_hi; c++) {
                    u32 g = c * 32 + (u32) lane;
                    bool a = g < nc;
                    uint4 k = kn;
                    kn = kn2;
                    if (c + 2 < c_hi && g + 64 < nc) kn2 = src[g + 64];
                    u32 dg = a ? ((k.x >> sb) & (K2_RB - 1u)) : K2_RB + (u32) lane;  // inactive lanes: unique digit
                    u32 peers = w_match(dg);
                    u32 rank = (u32) d_popc(peers & lt);
                    int leader = d_ffs(peers) - 1;
                    u32 bpos = 0;
                    if (a && lane == leader) {
                        bpos = sh->hist_cur[dg * K2_MAXSEG + ww];
                        sh->hist_cur[dg * K2_MAXSEG + ww] = bpos + (u32) d_popc(peers);
                    }
                    w_sync();                      // the next chunk's leaders read these counters
                    bpos = w_shfl(bpos, leader);
                    if (a) {
                        u32 pos = bpos + rank;
                        dst[pos] = k;
                        if (pass + 1 < npass)
                            s_atomic_add(&sh->hist_next[((k.x >> (sb + K2_RBITS)) & (K2_RB - 1u)) * K2_MAXSEG + pos / seg_len], 1u);
                    }
                }
                c_sync_sub(1, (int) nwt);
                uint4 *tmp = src; src = dst; dst = tmp;
            }
            // runs of equal fm_start: order by (fm_end, seed_prob, emission index).  Run heads are
            // found chunk-wise (one coalesced load per 32 keys, neighbours by shuffle); the rare
            // runs are then insertion-sorted by their head lane.
            {
                uint4 kq = make_uint4(0, 0, 0, 0); u32 bx = 0, ax = 0;   // key, fm_start before / after the chunk
                if (ww < nch) {
                    u32 g0 = ww * 32 + (u32) lane;
                    if (g0 < nc) kq = src[g0];
                    if (lane == 0 && g0 > 0) bx = src[g0 - 1].x;
                    if (lane == 31 && g0 + 1 < nc) ax = src[g0 + 1].x;
                }
                for (u32 c = ww; c < nch; c += nwk) {
                    const u32 g = c * 32 + (u32) lane;
                    const uint4 k = kq; const u32 bxc = bx, axc = ax;
                    if (c + nwk < nch) {
                        u32 gn = g + nwk * 32;
                        if (gn < nc) kq = src[gn];
                        if (lane == 0) bx = src[gn - 1].x;
                        if (lane == 31 && gn + 1 < nc) ax = src[gn + 1].x;
                    }
                    u32 px = w_shfl_up(k.x, 1), nx = w_shfl_down(k.x, 1);
                    if (lane == 0) px = bxc;
                    if (lane == 31) nx = axc;
                    const u32 s = k.x;
                    bool head = g < nc && (g == 0 || px != s) && (g + 1 < nc && nx == s);
                    if (head) {
                        u32 e = g + 1;
                        while (e < nc && src[e].x == s) e++;
                        for (u32 i = g + 1; i < e; i++) {
                            uint4 key = src[i];
                            float kp = u2f(key.z);
                            u32 j = i;
                            while (j > g) {
                                uint4 o = src[j - 1];
                                float op = u2f(o.z);
                                bool gt = o.y > key.y || (o.y == key.y && (kp < op || (!(op < kp) && (o.w >> 16) > (key.w >> 16))));
                                if (!gt) break;
                                src[j] = o;
                                j--;
                            }
                            src[j] = key;
                        }
                    }
                }
            }
            // Children that operator< does not separate are now adjacent.  Without any, the sorted order is unique
            // and this one is the reference's; with one, only running the reference's own unstable sort tells where
            // equal children end up (unc_pdqsort.cuh): one thread sorts the saved emission-order copy.
            c_sync_sub(1, (int) nwt);
            for (u32 i = wt; i + 1u < nc; i += nwt) {
                const uint4 k0 = src[i], k1 = src[i + 1u];
                if (!pq_less(k0, k1) && !pq_less(k1, k0)) *(volatile u32 *) &sh->bc[5] = 1u;
            }
            c_sync_sub(1, (int) nwt);
            PT_MARK(3)
            const uint4 *sk = src;   // sorted keys
#ifdef UNC_EMUL
            if (wt == 0) { g_emu_tie_stats[0]++; g_emu_tie_stats[1] += sh->bc[5]; }   // events sorted / with a tie
#endif
            if (*(volatile u32 *) &sh->bc[5]) {
                const u32 cap = ((maxp + 31u) >> 5) * K2_CH_SLOTS;
                if (wt == 0 && !unc_pdq_sort(cks, nc, cks + nc, cap - nc)) s_atomic_or(&sh->wk_overflow, 1u);
                c_sync_sub(1, (int) nwt);
                sk = cks;
            }

            // ---- D. dedup, gap sources, child seeds (reference src/mapper.cpp:527-603).
            // D1: per-chunk aggregate of the k-mer run structure: (max fm_end of the trailing run,
            //     first k-mer | last k-mer << 11 | whole-chunk-is-one-run << 22)
            uint4 d1n = make_uint4(0, 0, 0, 0);
            if (ww < nch && ww * 32 + (u32) lane < nc) d1n = sk[ww * 32 + (u32) lane];
            for (u32 c = ww; c < nch; c += nwk) {
                u32 g = c * 32 + (u32) lane;
                bool a = g < nc;
                u32 kmer = UNC_NKMER + 1u, endv = 0;
                if (a) { kmer = d1n.w & UNC_KMASK; endv = d1n.y; }
                if (c + nwk < nch && g + nwk * 32 < nc) d1n = sk[g + nwk * 32];
                u32 pk = w_shfl_up(kmer, 1);
                bool lhead = lane == 0 || kmer != pk || !a;
                u32 m_lhead = w_ballot(lhead), m_act = w_ballot(a);
                u32 mx = endv; bool hd = lhead;
                for (int d = 1; d < 32; d <<= 1) {
                    u32 omx = w_shfl_up(mx, d); u32 ohd = w_shfl_up(hd ? 1u : 0u, d);
                    if (lane >= d && !hd) { mx = omx > mx ? omx : mx; hd = ohd != 0; }
                }
                int last = 31 - d_clz(m_act);   // last active lane (m_act != 0)
                u32 kl = w_shfl(kmer, last), ml = w_shfl(mx, last), kf = w_shfl(kmer, 0);
                bool single = (m_lhead & m_act & ~1u) == 0;
                if (lane == 0) sh->agg[c] = make_uint2(ml, kf | (kl << 11) | (single ? 1u << 22 : 0u));
            }
            c_sync_sub(1, (int) nwt);
            // D2: everything else; source / seed positions from a decoupled look-back prefix sum
            epoch++;
            uint4 d2c = make_uint4(0, 0, 0, 0), d2n = make_uint4(0, 0, 0, 0);
            if (ww < nch) {
                u32 g0 = ww * 32 + (u32) lane;
                if (g0 < nc) d2c = sk[g0];
                if (g0 + 1 < nc) d2n = sk[g0 + 1];
            }
            for (u32 c = ww; c < nch; c += nwk) {
                u32 g = c * 32 + (u32) lane;
                bool a = g < nc;
                uint4 cur = make_uint4(0, 0, 0, 0), nxt = make_uint4(0, 0, 0, 0);
                if (a) cur = d2c;
                bool has_next = a && g + 1 < nc;
                if (has_next) nxt = d2n;
                if (c + nwk < nch) {
                    u32 gn = g + nwk * 32;
                    if (gn < nc) d2c = sk[gn];
                    if (gn + 1 < nc) d2n = sk[gn + 1];
                }
                u32 kmer = a ? (cur.w & UNC_KMASK) : UNC_NKMER + 1u;
                bool same_next = has_next && (nxt.w & UNC_KMASK) == kmer;
                bool dup = has_next && nxt.x == cur.x && nxt.y == cur.y;
                bool prob_ok = a && sh->probs[kmer & UNC_KMASK] >= source_prob;
                uint2 kr = tb->kmer_range[kmer & UNC_KMASK];
                u32 pk = w_shfl_up(kmer, 1);
                bool seed = a && !dup && ((cur.w >> 10) & 1u);
                u32 m_seed = w_ballot(seed);
                bool lhead = lane == 0 || kmer != pk || !a;
                u32 m_lhead = w_ballot(lhead);
                u32 mx = cur.y; bool hd = lhead;
                for (int d = 1; d < 32; d <<= 1) {
                    u32 omx = w_shfl_up(mx, d); u32 ohd = w_shfl_up(hd ? 1u : 0u, d);
                    if (lane >= d && !hd) { mx = omx > mx ? omx : mx; hd = ohd != 0; }
                }
                u32 first_head = (m_lhead & ~1u) ? (u32) d_ffs(m_lhead & ~1u) - 1u : 32u;
                bool in_lead = a && (u32) lane < first_head;
                // carry of the leading run: does it continue the previous chunk's trailing run, and
                // what is the max fm_end over that run's earlier elements?
                u32 cont = 0, cmax = 0;
                if (lane == 0 && c > 0) {
                    uint2 ag = sh->agg[c - 1];
                    if (((ag.y >> 11) & 0x7FFu) == kmer) {
                        cont = 1; cmax = ag.x;
                        u32 pc = c - 1;
                        while (pc > 0 && ((ag.y >> 22) & 1u)) {            // that chunk was a single run: look further back
                            uint2 pg = sh->agg[pc - 1];
                            if (((pg.y >> 11) & 0x7FFu) != (ag.y & 0x7FFu)) break;
                            cmax = pg.x > cmax ? pg.x : cmax;
                            ag = pg; pc--;
                        }
                    }
                }
                cont = w_shfl(cont, 0); cmax = w_shfl(cmax, 0);
                if (in_lead && cont) mx = mx > cmax ? mx : cmax;
                bool run_start = a && (lane == 0 ? !cont : (kmer != pk));
                bool begin_v = run_start && prob_ok && kr.x <= cur.x - 1u;
                u32 as = mx + 1u, ae = same_next ? nxt.x - 1u : kr.y;
                bool after_v = a && !dup && prob_ok && as <= ae;
                u32 m_b = w_ballot(begin_v), m_a = w_ballot(after_v);
                const u32 mine = ((u32) d_popc(m_b) + (u32) d_popc(m_a)) | ((u32) d_popc(m_seed) << 16);   // sources | seeds<<16
                // decoupled look-back: exclusive prefix of `mine` over the preceding chunks
                u32 excl = 0;
                if (c == 0) {
                    if (lane == 0) s_store_u64(&sh->pre[0], ((u64) k2_pre_pack(epoch, 2u) << 32) | mine);
                } else {
                    if (lane == 0) s_store_u64(&sh->pre[c], ((u64) k2_pre_pack(epoch, 1u) << 32) | mine);
                    int look = (int) c;
                    for (;;) {
                        int j = look - 1 - lane;
                        u64 w = 0;
                        if (j >= 0) {
                            for (;;) {
                                w = s_load_u64(&sh->pre[j]);
                                if ((u32) (w >> 34) == (epoch & 0x3FFFFFFFu)) break;
                                w_spin();
                            }
                        }
                        u32 state = (u32) (w >> 32) & 3u, val = (u32) w;
                        u32 mP = w_ballot(j >= 0 && state == 2u);
                        u32 upto = mP ? (u32) d_ffs(mP) : 32u;            // lanes [0, upto) contribute
                        u32 contrib = (j >= 0 && (u32) lane < upto) ? val : 0u;
                        for (int d = 16; d > 0; d >>= 1) contrib += w_shfl(contrib, lane ^ d);
                        excl += contrib;
                        if (mP) break;
                        look -= 32;
                        if (look <= 0) break;
                    }
                    if (lane == 0) s_store_u64(&sh->pre[c], ((u64) k2_pre_pack(epoch, 2u) << 32) | (excl + mine));
                }
                const u32 ns_before = excl & 0xFFFFu, seeds_before = excl >> 16;
                u32 off = (u32) d_popc(m_b & lt) + (u32) d_popc(m_a & lt);
                u32 sidx = ns_before + off;    // sources (that would be) added before this element
                // sources_added_[kmer] is set at a run start while the buffer is not full
                if (run_start && prob_ok && nc + sidx < maxp) s_atomic_or(&sh->flags[kmer >> 5], 1u << (kmer & 31u));
                if (begin_v && nc + sidx < maxp) {
                    write_source(next, hist_e, S0 + nc + sidx, kr.x, cur.x - 1u, kmer, sh->probs[kmer]);
                    onext[nc + sidx] = S0 + nc + sidx;
                }
                u32 sidx2 = sidx + (begin_v ? 1u : 0u);
                if (after_v && nc + sidx2 < maxp) {
                    write_source(next, hist_e, S0 + nc + sidx2, as, ae, kmer, sh->probs[kmer]);
                    onext[nc + sidx2] = S0 + nc + sidx2;
                }
                u32 emit = cur.w >> 16;
                if (a) onext[g] = emit | (dup ? UNC_INVALID : 0u);
                // update_seeds(child, false): unique, move-headed, full-length, probable paths
                if (seed) {
                    d_atomic_or(&((u32 *) (next + (size_t) emit * 2))[3], 0x80000000u);   // sa_checked_
                    u32 ri = n_ended_rows + seeds_before + (u32) d_popc(m_seed & lt);
                    if (ri < W.rl_cap) rlist[ri] = make_uint2(cur.x, (cur.w >> 11) & 0x1Fu);
                    else sh->wk_overflow = 1;
                }
            }
            c_sync_sub(1, (int) nwt);
            PT_MARK(4)
            {
                u32 fin = (u32) s_load_u64(&sh->pre[nch - 1]);
                u32 tot_src = fin & 0xFFFFu;
                ns_added = nc + tot_src > maxp ? maxp - nc : tot_src;
                n_child_seeds = fin >> 16;
            }
        }
        n_rows = n_ended_rows + n_child_seeds;
        if (n_rows > W.rl_cap) n_rows = W.rl_cap;
        u32 nn = nc + ns_added;

        // ---- S. suffix-array lookups for all seed rows of the event
        //         (reference src/mapper.cpp:673-681: sa_end = fmi.size() - fmi.sa(s))
        for (u32 i = wt; i < n_rows; i += nwt) {
            uint2 e = rlist[i];
            e.x = ix.seq_len - unc_sa_lookup(ix, e.x, &pend_steps, &pend_blocks);
            rlist[i] = e;
        }
        if (ww == 0) {
            // ---- E. fresh sources for every sufficiently probable k-mer without one
            //         (reference src/mapper.cpp:605-624)
            for (u32 j = 0; j < 32 && nn < maxp; j++) {
                u32 k = j * 32 + (u32) lane;
                u32 fw = sh->flags[j];
                uint2 kr = tb->kmer_range[k];
                float pk = sh->probs[k];
                bool add = !((fw >> lane) & 1u) && pk >= source_prob && kr.x <= kr.y;
                u32 m_add = w_ballot(add);
                u32 room = maxp - nn;
                u32 visited = 0xFFFFFFFFu;
                if ((u32) d_popc(m_add) >= room) {
                    // the room-th add fills the buffer; k-mers after it are never visited
                    u32 mm = m_add;
                    for (u32 q = 1; q < room; q++) mm &= mm - 1;
                    int last = d_ffs(mm) - 1;
                    visited = last == 31 ? 0xFFFFFFFFu : ((2u << last) - 1u);
                    m_add &= visited;
                }
                u32 rank = (u32) d_popc(m_add & lt);
                if ((m_add >> lane) & 1u) {
                    write_source(next, hist_e, S0 + nn + rank, kr.x, kr.y, k, pk);
                    onext[nn + rank] = S0 + nn + rank;
                }
                w_sync();
                if (lane == 0) sh->flags[j] = fw & ~visited;
                nn += (u32) d_popc(m_add);
            }
            if (lane == 0) { sh->bc[1] = nn; *(volatile u32 *) &sh->n_rows[event_i & 1u] = n_rows; }
        }
        PT_MARK(5)
        // ---- hand the event's seeds to the tracker; learn the outcome of the previous event
        c_sync();                                                     // X_e
        PT_MARK(6)
        nn = sh->bc[1];
        pend_sources = nn - nc;
        const u32 v = event_i > n_first ? *(volatile u32 *) &sh->verdict[(event_i - 1u) & 1u] : 0u;
        if (v) {                                                      // event_i's work is discarded: the Mapper returned
            if (wt < 32u) sh->flags[wt] = sh->flags_prev[wt];            // after event_i - 1 (reference src/mapper.cpp:633-651)
            break;
        }
        n_children += pend_children; n_sources += pend_sources;
        my_blocks += pend_blocks; my_steps += pend_steps;
        pend_children = pend_sources = pend_blocks = pend_steps = 0;
        prev_size = nn;
        gen ^= 1u;
        PT_MARK(8)
    }
    *epoch_io = epoch;
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

#include "unc_k2v2.cuh"

// One read mapped by one CTA.  reference src/mapper.cpp:188-200 (map_read); with STREAM, one map_chunk's
// worth of events of a read in progress (:381-431), resumed from and saved to the channel's DevMapState.
template <bool STREAM, bool EXACT, bool FLAGS>
UNC_DEV void unc_k2_map_read(const DevIndex &ix, const DevParams &p, const DevBatch &B, const DevWork &W,
                             K2Shared *sh, u32 r, u32 *epoch_io) {
    const u32 tid = (u32) c_tid();
    const u32 n_ev = B.n_events[r];
    u32 n_first = 0;
    if (STREAM) {
        const DevMapState *ms = B.mstate + B.chan[r];
        if (ms->started) n_first = ms->event_i;
        if (tid < 32) sh->flags[tid] = ms->flags[tid];
    } else {
        if (tid < 32) sh->flags[tid] = (FLAGS && B.flags_in) ? B.flags_in[(size_t) r * 32 + tid] : 0u;
    }
    const u32 n_limit = n_first + n_ev < p.max_events ? n_first + n_ev : (n_first < p.max_events ? p.max_events : n_first);
    if (tid == 0) {
        sh->cnt_blocks = 0; sh->cnt_steps = 0; sh->wk_overflow = 0; sh->wl_cnt = 0;
        sh->verdict[0] = sh->verdict[1] = 0; sh->n_rows[0] = sh->n_rows[1] = 0; sh->bc[1] = 0;
    }
    for (u32 b = tid; b < K2_RB * K2_MAXSEG; b += (u32) c_nthreads()) sh->hist_next[b] = 0;
    c_sync();
    if (EXACT) {   // the exact-ties worker sorts with the radix counters: the tracker's directory stays in global memory
        if (tid < 32) unc_k2_tracker<STREAM>(ix, p, B, W, sh, r, n_first, n_limit, nullptr, 0u);
        else unc_k2_workers_exact<STREAM>(ix, p, B, W, sh, r, n_first, n_limit, epoch_io);
    } else {       // the second structure leaves the radix counters free: they hold the directory's fast copy
        if (tid < 32) unc_k2_tracker<STREAM>(ix, p, B, W, sh, r, n_first, n_limit, (uint4 *) sh->hist_next, K2_RB * K2_MAXSEG / 4u);
        else unc_k2_workers_v2<STREAM, FLAGS>(ix, p, B, W, sh, r, n_first, n_limit);
    }
    c_sync();
    if (STREAM && tid < 32) B.mstate[B.chan[r]].flags[tid] = sh->flags[tid];
    if (!STREAM && FLAGS && B.flags_out && tid < 32) B.flags_out[(size_t) r * 32 + tid] = sh->flags[tid];
}

// Ordered mode (unc_ordered_logic.hpp): would k-mer k get a fresh source at read r's FIRST event if its
// sources_added_ flag were clear?  This is phase E's `add` test for event 0 (reference src/mapper.cpp:611-614) on
// the event value the event loop computes.  A read's first event has no children, so the flags it starts from act
// only through these k-mers: two initial flag sets that agree on them give the same mapping.
UNC_DEV bool unc_event0_cand(const DevIndex &ix, const DevParams &p, const DevBatch &B, u32 r, u32 k) {
    if (B.n_events[r] == 0 || p.max_events == 0) return false;
    const float event = f_add(f_mul(B.scale[r], B.events[(size_t) r * B.ev_stride]), B.shift[r]);
    const uint2 kr = ix.kmer_range[k];
    return unc_match_prob(event, d_ldg(ix.lv_mean + k), d_ldg(ix.lv_var2 + k), d_ldg(ix.lognorm + k)) >= ix.thresh[0] &&
           kr.x <= kr.y;
}

UNC_DEV DevWork unc_work_slot(const DevWork &W0, const DevWorkStrides &S, size_t slot) {
    DevWork W;
    W.paths = W0.paths + slot * S.paths;
    W.hist = W0.hist + slot * S.hist;
    W.wlist = W0.wlist + slot * S.cks;
    W.ckey = W0.ckey + slot * S.ckey;
    W.cks = W0.cks + slot * S.cks;
    W.elist = W0.elist + slot * S.elist;
    W.order = W0.order + slot * S.order;
    W.rlist = W0.rlist + slot * S.rlist;
    W.clu = W0.clu + slot * S.clu;
    W.dir = W0.dir + slot * S.dir;
    W.max_blocks = W0.max_blocks;
    W.rl_cap = W0.rl_cap;
    return W;
}

// Persistent CTA body: stage the tables, then pull reads from the global queue.
// Needs at least 2 warps (tracker + >= 1 worker) and at most 1 + K2_MAXSEG.
// EXACT: the exact-ties kernel (the reference's unstable child sort reproduced, unc_pdqsort.cuh)
template <bool EXACT = false, bool FLAGS = false>
UNC_DEV void unc_k2_cta_main(const DevIndex &ix, const DevParams &p, const DevBatch &B, const DevWork &W, K2Shared *sh) {
    unc_k2_cta_setup(ix, p, sh);
    u32 epoch = 0;
    for (;;) {
        if (c_tid() == 0) sh->bc[0] = d_atomic_add(B.queue, 1u);
        c_sync();
        u32 r = sh->bc[0];
        c_sync();
        if (r >= B.n_reads) break;
        unc_k2_map_read<false, EXACT, FLAGS>(ix, p, B, W, sh, r, &epoch);
    }
}

// Streaming variant: every item continues a read in the workspace slot of its CHANNEL.
template <bool EXACT = false>
UNC_DEV void unc_k2_cta_main_stream(const DevIndex &ix, const DevParams &p, const DevBatch &B, const DevWork &W0,
                                    const DevWorkStrides &S, K2Shared *sh) {
    unc_k2_cta_setup(ix, p, sh);
    u32 epoch = 0;
    for (;;) {
        if (c_tid() == 0) sh->bc[0] = d_atomic_add(B.queue, 1u);
        c_sync();
        u32 r = sh->bc[0];
        c_sync();
        if (r >= B.n_reads) break;
        const DevWork W = unc_work_slot(W0, S, B.chan[r]);
        unc_k2_map_read<true, EXACT, true>(ix, p, B, W, sh, r, &epoch);
    }
}
