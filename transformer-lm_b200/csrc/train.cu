// train.cu -- BPE training on the device: pretoken hash-count, word list, initial pair table,
// persistent cooperative merge loop.  Entry points: bpe_train*, bpe_count_* (include/bpe_sm100.h).
//
// Reference being replaced: models/tokenizer/train.py:142-231 (see each kernel for the exact lines).
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <unordered_set>
#include "kernels.h"
#include "ctx.h"
#include "merge.cuh"
#include "hashtab.cuh"
#include <cooperative_groups/reduce.h>

// =============================================================================================
// 1. Pretoken counting  (extract_subword_frequencies, train.py:16-28)
//
// The short, medium and long pretoken tables of hashtab.cuh in HBM, payload = the count (64-bit atomics).  Long keys with
// META_POOL_BIT address the persistent pool (imported / re-homed words), others the text arena of the current shard.
// =============================================================================================
struct CountTables : PtTables {
    // slot of the k-th unique short / medium / long word (k = value of counters[0] / [7] / [1] when it was claimed): everything that
    // walks the words (re-homing, export, word list, table growth) walks these lists instead of scanning the tables' capacity, which
    // is sized for the worst case (every pretoken of a batch new) and mostly empty
    u32 *slist, *mlist, *llist;
    ulonglong2 *hot; u64 *hcnt; u64 hot_nb;      // hot table (see below): hot_nb buckets of two 16-byte keys, counts apart; 0 = none
    u64 *counters;                               // [0]=n_short [1]=n_long [2]=long_bytes [3]=overflow [4]=n_pretokens [5]=too_long
                                                 // [6]=an owned pretoken ran past the trusted part of the right halo [7]=n_medium
};
struct WordCounts { u64 n_short, n_medium, n_long; };

struct CountState {
    DevBuf stab, mtab, ltab, slist, mlist, llist, pool, counters, hot;
    u64 scap = 0, mcap = 0, lcap = 0, pool_used = 0;
    u64 hot_nb = 0, hot_seen = 0;                // buckets of the hot table; pretokens counted when it was last built
    int hot_builds = 0;
    bool active = false;
    u64 n_pretokens = 0;
    u64 n_rehomed = 0;                           // long words [0, n_rehomed) of the list have their bytes in the pool
};

// count `delta` more occurrences of a word: a claim appends the slot to the tier's list; the count is never read
__device__ __forceinline__ void short_add(const CountTables &t, u64 key, u64 delta) {
    short_find_or_claim<false>(t, key, t.counters,
        [&](u64 s) { t.slist[atomicAdd(&t.counters[0], 1ull)] = (u32)s; atomicAdd(&t.stab[s].val, delta); },
        [&](u64 s, u64) { atomicAdd(&t.stab[s].val, delta); });
}
__device__ __forceinline__ void medium_add(const CountTables &t, u64 k0, u64 k1, u64 delta) {
    medium_find_or_claim<false>(t, k0, k1, t.counters,
        [&](u64 s) { t.mlist[atomicAdd(&t.counters[7], 1ull)] = (u32)s; atomicAdd(&t.medtab[s].val, delta); },
        [&](u64 s, u64) { atomicAdd(&t.medtab[s].val, delta); });
}
__device__ __forceinline__ void long_add(const CountTables &t, const uint8_t *p, u32 len, u64 off_meta, u64 delta) {
    long_find_or_claim<false>(t, p, len, off_meta, t.counters,
        [&](u64 s) {
            t.llist[atomicAdd(&t.counters[1], 1ull)] = (u32)s;
            atomicAdd(&t.counters[2], (u64)len);
            atomicAdd(&t.ltab[s].val, delta);
        },
        [&](u64 s, u64) { atomicAdd(&t.ltab[s].val, delta); });
}

// Counting straight from the text and its start bits (no per-pretoken offset array, no scan).  A warp takes 32 consecutive 16-byte
// chunks (512 bytes of text, coalesced 16-byte loads, the next step's loads in flight) per step, steps handed out by a ticket
// counter; the step's start bits are compacted into a list of positions in shared memory and the pretokens are taken 32 at a time,
// a lane each (details at the kernel).  For every pretoken: length = next position - position (pretokens that run past the bits
// the step holds look it up in the bit array), the first 16 bytes are cut out of the staged text with aligned loads and funnel
// shifts (no byte loops, no unaligned loads).
//   * pretokens of <= 7 bytes are counted in the CTA's shared-memory table (natural-language text is Zipfian: without it the few
//     hottest words serialise hundreds of millions of same-address L2 atomics);
//   * what misses there, and every longer pretoken, goes to the warp's queues (compacted with ballots; the queue lengths are
//     warp-uniform registers: no atomics, no CTA barrier anywhere in the loop): keys (short: k0 = key, k1 = 0; medium: k0, k1)
//     and long pretokens (offset | len << 32).  A drain takes whole groups of 64 keys, two per lane with their probes in flight
//     together: hot table first, the big tables for what misses it.
// The shared-memory table is flushed to the HBM table when the CTA is done.
// One CTA of 1 024 threads per SM with a 1 024-slot table.  Measured on the 11 GB OWT-shape corpus (count stage, ms) with the hot
// table behind it: 2 CTAs x 512 threads x 4 096 slots 48.4; 1 x 1 024 threads: 8 192 slots 47.0, 4 096 43.8, 2 048 44.4, 1 024 42.0,
// 512 44.0, 256 45.2 (TinyStories shape 2 GiB: 8.2 / 8.1 / 8.0 / 8.3 / 8.0 / 8.5 / 8.3).  The table only has to absorb the few hundred
// words whose same-address L2 atomics would serialise; everything else is as cheap in the L2-resident hot table.
#ifndef CNT_NT
#define CNT_NT 1024
#endif
#ifndef CNT_SMEM_LG
#define CNT_SMEM_LG 10
#endif
#define CNT_SMEM_SLOTS (1u << CNT_SMEM_LG)
#ifndef CNT_SMEM_PROBES
#define CNT_SMEM_PROBES 2u
#endif
#define CNT_WARPS (CNT_NT / 32u)
#define CNT_QCAP 96u                             // entries of the warp's key queue
#define CNT_QDRAIN 64u                           // drained when it reaches this (a round of 32 pretokens adds <= 32)
#define CNT_QL_CAP 64u
#define CNT_QL_DRAIN 32u
#define CNT_WARP_SMEM (CNT_QCAP * 16u + CNT_QL_CAP * 8u + 528u + 1040u)    // queues, staged text, staged positions
#define CNT_DYN_SMEM ((size_t)CNT_SMEM_SLOTS * 12 + (size_t)CNT_WARPS * CNT_WARP_SMEM)

// queues of a warp: qe = keys of short pretokens that missed the shared-memory table (k0 = key, k1 = 0) and of medium ones
// (k0, k1 != 0); ql = long pretokens (offset from base | len << 32)
struct CountQueues { ulonglong2 *qe; u64 *ql; u32 n, nl; };

// The HOT TABLE.  A probe into the big tables is one random 32-byte sector and its 128-byte L2 line to itself (the tables are
// sized for the worst case and mostly empty).  Measured on B200 (tools/bench_l2_random.cu, bench_l2_mix.cu): L2 keeps ~0.5 M such
// lines; a random read + RED pair that misses it runs at 16-20 G pairs/s, one that hits at 60-110 G/s -- and counting 11 GB of
// web-like text sends 1.1 G pairs to the tables, most of them to words that are neither among the few the shared-memory table
// holds nor rare.  So once enough text has been seen, the words counted at least T times are copied into a DENSE table of their
// own, probed first: a bucket is ONE 32-byte sector holding two 16-byte keys (short and medium words alike: k1 = 0 for a short
// one), the counts sit in an array beside it -- at most ~1 M words, 50 MB: it stays in L2.  A word whose bucket is full stays with
// the big tables, so a probe is exactly one sector: no chains, no claims, all lanes of a warp finish together.  The counts are added
// back to the big tables whenever somebody needs those (count_hot_flush).

// Drain the warp's queues: whole groups of 64 keys (everything when `all`), two per lane with their probes in flight together;
// every long entry.
__device__ __forceinline__ void count_drain(const CountTables &t, CountQueues &q, u64 base, u32 lane, bool all) {
    const u32 dn = all ? q.n : q.n & ~63u;
    __syncwarp();
    for (u32 e0 = 0; e0 < dn; e0 += 64u) {
        const bool ha = e0 + lane < dn, hb = e0 + 32u + lane < dn;
        ulonglong2 ka = make_ulonglong2(0, 0), kb = ka;
        if (ha) ka = q.qe[e0 + lane];
        if (hb) kb = q.qe[e0 + 32u + lane];
        bool ta = ha, tb = hb;                   // still to be added to the big tables
        if (t.hot_nb) {
            const u64 ba = hot_bucket(t.hot_nb, ka.x, ka.y), bb = hot_bucket(t.hot_nb, kb.x, kb.y);
            const int ia = ha ? hot_find(t.hot, ba, ka.x, ka.y) : -1, ib = hb ? hot_find(t.hot, bb, kb.x, kb.y) : -1;
            if (ia >= 0) { atomicAdd(&t.hcnt[2 * ba + ia], 1ull); ta = false; }
            if (ib >= 0) { atomicAdd(&t.hcnt[2 * bb + ib], 1ull); tb = false; }
        }
        if (ta) { if (ka.y == 0) short_add(t, ka.x, 1); else medium_add(t, ka.x, ka.y, 1); }
        if (tb) { if (kb.y == 0) short_add(t, kb.x, 1); else medium_add(t, kb.x, kb.y, 1); }
    }
    for (u32 e = lane; e < q.nl; e += 32u) {
        const u64 ent = q.ql[e];
        const u64 off = base + (u32)ent;
        long_add(t, t.text + off, (u32)(ent >> 32), off, 1);
    }
    q.nl = 0;
    // the remainder (< 64 keys) moves to the front
    const u32 r = q.n - dn;
    ulonglong2 v0 = make_ulonglong2(0, 0), v1 = v0;
    if (dn && lane < r) v0 = q.qe[dn + lane];
    if (dn && lane + 32u < r) v1 = q.qe[dn + 32u + lane];
    __syncwarp();
    if (dn && lane < r) q.qe[lane] = v0;
    if (dn && lane + 32u < r) q.qe[32u + lane] = v1;
    q.n = r;
    __syncwarp();
}

// chunks [c_lo, c_hi) (16 bytes each, absolute positions 16 c); `base` <= 16 c_lo is what the 32-bit offsets of the long queue count from.
// A warp step = 32 consecutive chunks.  The lanes first COMPACT the step's start bits into a list of positions in shared memory
// (warp scan of the popcounts; the 512 + 16 bytes of text are staged beside it), then take the list 32 pretokens at a time: a lane
// per pretoken, every lane busy, where a lane per chunk left half of them idle (3.5 starts per chunk on average, 7-8 in the fullest
// chunk of a step).  Length = next position - position; the first 16 bytes of the pretoken = five aligned words of the staged text
// and four funnel shifts.
#ifndef CNT_TICKET
#define CNT_TICKET 8u                            // steps (of 512 bytes) per ticket
#endif
#define CNT_STAGE_TEXT 528u                      // 32 chunks + the 16 bytes after them
#define CNT_STAGE_POS 520u                       // up to 512 starts + the sentinel (first start after the step), 16-bit each
#define CNT_POS_OWNED 0x8000u                    // the pretoken starts inside [own_begin, own_end) of this launch's chunks
#define CNT_POS_UNKNOWN 0xFFFFu                  // sentinel: no start within the bits the last lane holds
// SKIP_SP (training with split_special_tokens): spstart marks the first byte of every special-token occurrence.  Such a start
// still ends the pretoken before it, but is not counted itself: the occurrence is no word.
template <bool SKIP_SP>
__device__ __forceinline__ void count_pretokens(const CountTables &t, const u32 *__restrict__ flags, const u32 *__restrict__ spstart,
                                                u64 c_lo, u64 c_hi, u64 n, u64 base, u64 own_begin, u64 own_end, u64 trust_end) {
    extern __shared__ __align__(16) unsigned char cnt_smem[];
    const u32 lane = lane_id(), warp = threadIdx.x >> 5;
    u64 *s_key = reinterpret_cast<u64 *>(cnt_smem);                                        // shared-memory table: keys ...
    u32 *s_cnt = reinterpret_cast<u32 *>(s_key + CNT_SMEM_SLOTS);                          // ... and counts
    unsigned char *wq = cnt_smem + (size_t)CNT_SMEM_SLOTS * 12 + (size_t)warp * CNT_WARP_SMEM;
    CountQueues q;
    q.qe = reinterpret_cast<ulonglong2 *>(wq); q.ql = reinterpret_cast<u64 *>(wq + CNT_QCAP * 16u);
    q.n = q.nl = 0;
    u32 *s_text = reinterpret_cast<u32 *>(wq + CNT_QCAP * 16u + CNT_QL_CAP * 8u);
    unsigned short *s_pos = reinterpret_cast<unsigned short *>(wq + CNT_QCAP * 16u + CNT_QL_CAP * 8u + CNT_STAGE_TEXT);
    for (u32 i = threadIdx.x; i < CNT_SMEM_SLOTS; i += CNT_NT) { s_key[i] = 0; s_cnt[i] = 0; }
    __syncthreads();
    u64 n_tok = 0;
    const u32 lt = (1u << lane) - 1u;
    const u64 n_fw = (n + 31) >> 5;              // flag words that hold bits of the text
    // Steps are handed out CNT_TICKET at a time by a ticket counter (a warp that met expensive pretokens simply takes fewer tickets:
    // with a fixed assignment a fifth of all stall samples sat at the barrier that ends the launch); the warp holds the ticket it
    // works on and the next one, so that the loads of the next step can always be issued a step ahead.
    const u64 n_steps = (c_hi - c_lo + 31) / 32;
    u64 tk_cur = 0, tk_next = 0;
    if (lane == 0) { tk_cur = atomicAdd(&t.counters[16], 1ull); tk_next = atomicAdd(&t.counters[16], 1ull); }
    tk_cur = __shfl_sync(0xffffffffu, tk_cur, 0); tk_next = __shfl_sync(0xffffffffu, tk_next, 0);
    u32 sub = 0;                                 // step within the current ticket
    u64 c = c_lo + (tk_cur * CNT_TICKET) * 32u + lane;
    // loads of a step: the chunk (lane 31: also the 16 bytes after it; the arena is padded), the two flag words that hold its
    // 48..64-bit window.  Chunks past c_hi are loaded as well while they are text: their start bits end the last pretokens of the range
    uint4 A = make_uint4(0, 0, 0, 0), B = A; u32 f0 = 0, f1 = 0, g0 = 0;
    if (tk_cur * CNT_TICKET < n_steps && c * 16u < n) {
        const uint4 *tp = reinterpret_cast<const uint4 *>(t.text + c * 16u);
        A = __ldcs(tp); if (lane == 31) B = __ldcs(tp + 1);
        const u64 w = c >> 1; f0 = __ldcs(flags + w); f1 = w + 1 < n_fw ? __ldcs(flags + w + 1) : 0u;
        if (SKIP_SP) g0 = __ldcs(spstart + w);
    }
    while (tk_cur * CNT_TICKET + sub < n_steps) {
        c = c_lo + (tk_cur * CNT_TICKET + sub) * 32u + lane;
        // the step after this one: the next of the ticket, or the first of the next ticket (whose successor is fetched now)
        u64 cn;
        if (sub + 1 < CNT_TICKET) { sub++; cn = c + 32u; }
        else {
            sub = 0; tk_cur = tk_next;
            if (lane == 0) tk_next = atomicAdd(&t.counters[16], 1ull);
            tk_next = __shfl_sync(0xffffffffu, tk_next, 0);
            cn = c_lo + (tk_cur * CNT_TICKET) * 32u + lane;
        }
        const u64 p0 = c * 16u, step_p0 = (c - lane) * 16u;
        u64 F = (((u64)f1 << 32) | f0) >> (u32)(p0 & 16u);           // bit i: a pretoken starts at byte p0 + i (>= 48 bits)
        const u32 sp = SKIP_SP ? g0 >> (u32)(p0 & 16u) : 0u;          // bit i: a special-token occurrence starts at byte p0 + i
        reinterpret_cast<uint4 *>(s_text)[lane] = A;
        if (lane == 31) reinterpret_cast<uint4 *>(s_text)[32] = B;
        // the next step's loads
        {
            if (cn - lane < c_hi && cn * 16u < n) {
                const uint4 *tp = reinterpret_cast<const uint4 *>(t.text + cn * 16u);
                A = __ldcs(tp); if (lane == 31) B = __ldcs(tp + 1);
                const u64 w = cn >> 1; f0 = __ldcs(flags + w); f1 = w + 1 < n_fw ? __ldcs(flags + w + 1) : 0u;
                if (SKIP_SP) g0 = __ldcs(spstart + w);
            } else { f0 = 0; f1 = 0; }
        }
        if (p0 + 64 > n) F = p0 < n ? F & ((1ull << (n - p0)) - 1ull) : 0ull;   // bits past the end of the text do not count
        const u32 mall = (u32)F & 0xFFFFu;       // every start of the chunk
        // the starts this launch counts: chunks of the range, positions inside [own_begin, own_end), no special occurrence
        u32 m = c < c_hi ? mall : 0u;
        if (SKIP_SP) m &= ~sp;
        if (p0 < own_begin) m = own_begin - p0 >= 16 ? 0u : m & ~((1u << (u32)(own_begin - p0)) - 1u);
        if (p0 + 16 > own_end) m = own_end <= p0 ? 0u : m & ((1u << (u32)(own_end - p0)) - 1u);
        n_tok += __popc(m);
        // ---- compaction: positions of the step's starts, in text order ----
        u32 incl = __popc(mall);
#pragma unroll
        for (u32 d = 1; d < 32; d <<= 1) { const u32 o = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += o; }
        const u32 T = __shfl_sync(0xffffffffu, incl, 31);
        {
            u32 o = incl - __popc(mall), mm = mall;
            while (mm) {
                const u32 j = __ffs(mm) - 1u; mm &= mm - 1u;
                s_pos[o++] = (unsigned short)((lane * 16u + j) | (((m >> j) & 1u) ? CNT_POS_OWNED : 0u));
            }
            if (lane == 31) {                    // the sentinel: the first start after the step, if the window shows it
                const u32 nx = (u32)__ffsll((long long)(F >> 16));
                s_pos[T] = (unsigned short)(nx ? 512u + nx - 1u : CNT_POS_UNKNOWN);
            }
        }
        __syncwarp();
        // ---- the pretokens, 32 at a time ----
        for (u32 i0 = 0; i0 < T; i0 += 32u) {
            const u32 i = i0 + lane;
            const u32 pe = i < T ? s_pos[i] : 0u, pn = i < T ? s_pos[i + 1] : 0u;
            const bool act = (pe & CNT_POS_OWNED) != 0;
            const u32 pos = pe & 0x7FFFu;
            u32 len = (pn & 0x7FFFu) - pos;
            if (act && pn == CNT_POS_UNKNOWN) {  // no further start in sight: a long pretoken, or the last one of the text
                const u64 e = flags_next_start(flags, step_p0 + pos + 1, n) - (step_p0 + pos);
                if (e > MAX_TOKEN_LEN) { t.counters[5] = 1; len = MAX_TOKEN_LEN; } else len = (u32)e;
            }
            if (act && step_p0 + pos + len > trust_end) t.counters[6] = 1;
            // bytes pos .. pos + 15 of the staged text
            const u32 w = pos >> 2, sh = (pos & 3u) * 8u;
            const u32 Y0 = s_text[w], Y1 = s_text[w + 1], Y2 = s_text[w + 2], Y3 = s_text[w + 3], Y4 = s_text[w + 4];
            const u64 k0 = (u64)__funnelshift_r(Y0, Y1, sh) | ((u64)__funnelshift_r(Y1, Y2, sh) << 32);
            const u64 k1 = (u64)__funnelshift_r(Y2, Y3, sh) | ((u64)__funnelshift_r(Y3, Y4, sh) << 32);
            bool q_s = act && len <= SHORT_MAX;
            const bool q_m = act && len > SHORT_MAX && len <= MED_MAX, q_l = act && len > MED_MAX;
            const u64 key = (k0 & low_bytes_mask(len)) | ((u64)len << 56);               // (short pretokens)
            if (q_s) {
                u32 slot = (((u32)key ^ (u32)(key >> 32)) * 0x9E3779B1u) >> (32 - CNT_SMEM_LG);   // cheap hash for the shared-memory table
#pragma unroll
                for (u32 pr = 0; pr < CNT_SMEM_PROBES; pr++) {
                    u64 kk = s_key[slot];
                    if (kk == 0) { const u64 old = atomicCAS(&s_key[slot], 0ull, key); kk = old ? old : key; }
                    if (kk == key) { atomicAdd(&s_cnt[slot], 1u); q_s = false; break; }
                    slot = (slot + 1) & (CNT_SMEM_SLOTS - 1);
                }
            }
            const u32 me = __ballot_sync(0xffffffffu, q_s || q_m), ml = __ballot_sync(0xffffffffu, q_l);
            if (q_s) q.qe[q.n + __popc(me & lt)] = make_ulonglong2(key, 0ull);
            if (q_m) q.qe[q.n + __popc(me & lt)] = make_ulonglong2(k0, (len > 8 ? k1 & low_bytes_mask(len - 8) : 0ull) | ((u64)len << 56));
            if (q_l) q.ql[q.nl + __popc(ml & lt)] = (step_p0 + pos - base) | ((u64)len << 32);
            q.n += __popc(me); q.nl += __popc(ml);
            if (q.n >= CNT_QDRAIN || q.nl >= CNT_QL_DRAIN) count_drain(t, q, base, lane, false);
        }
        __syncwarp();                            // the staged text and positions are free for the next step
    }
    count_drain(t, q, base, lane, true);
    // one atomic per warp for the occurrence counter
    for (int d = 16; d; d >>= 1) n_tok += __shfl_down_sync(0xffffffffu, n_tok, d);
    if (lane == 0 && n_tok) atomicAdd(&t.counters[4], n_tok);
    __syncthreads();
    for (u32 i = threadIdx.x; i < CNT_SMEM_SLOTS; i += CNT_NT)
        if (s_cnt[i]) short_add(t, s_key[i], (u64)s_cnt[i]);
}
__global__ void __launch_bounds__(CNT_NT, 1024 / CNT_NT) k_count_pretokens(CountTables t, const u32 *__restrict__ flags, u64 c_lo, u64 c_hi, u64 n, u64 base,
                                                              u64 own_begin, u64 own_end, u64 trust_end) {
    count_pretokens<false>(t, flags, nullptr, c_lo, c_hi, n, base, own_begin, own_end, trust_end);
}
__global__ void __launch_bounds__(CNT_NT, 1024 / CNT_NT) k_count_pretokens_split(CountTables t, const u32 *__restrict__ flags, const u32 *__restrict__ spstart,
                                                                    u64 c_lo, u64 c_hi, u64 n, u64 base, u64 own_begin, u64 own_end, u64 trust_end) {
    count_pretokens<true>(t, flags, spstart, c_lo, c_hi, n, base, own_begin, own_end, trust_end);
}

// upper bound of new unique words a range of flag words can create: its number of start bits
__global__ void __launch_bounds__(256) k_popc_ranges(const u32 *__restrict__ flags, u64 n_words, u64 words_per_range,
                                                    u64 *__restrict__ out) {
    u64 r = blockIdx.y;
    u64 lo = r * words_per_range, hi = lo + words_per_range;
    if (hi > n_words) hi = n_words;
    u64 c = 0;
    for (u64 w = lo + (u64)blockIdx.x * blockDim.x + threadIdx.x; w < hi; w += (u64)gridDim.x * blockDim.x) c += __popc(flags[w]);
    for (int d = 16; d; d >>= 1) c += __shfl_down_sync(0xffffffffu, c, d);
    if (lane_id() == 0 && c) atomicAdd(&out[r], c);
}

// ---- hot table: histogram of the counts, build, flush ------------------------------------------------------------------
#define HOT_HIST 64
__global__ void __launch_bounds__(256) k_hot_hist(CountTables t, u64 n_short, u64 n_medium, u64 *__restrict__ hist /* [HOT_HIST] */) {
    __shared__ u32 s_h[HOT_HIST];
    if (threadIdx.x < HOT_HIST) s_h[threadIdx.x] = 0;
    __syncthreads();
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_short + n_medium; i += (u64)gridDim.x * blockDim.x) {
        const u64 c = i < n_short ? t.stab[t.slist[i]].val : t.medtab[t.mlist[i - n_short]].val;
        atomicAdd(&s_h[c < HOT_HIST ? (u32)c : HOT_HIST - 1], 1u);
    }
    __syncthreads();
    if (threadIdx.x < HOT_HIST && s_h[threadIdx.x]) atomicAdd(&hist[threadIdx.x], (u64)s_h[threadIdx.x]);
}
// every short / medium word counted at least `thresh` times is placed in its bucket if one of the two slots is free
__global__ void __launch_bounds__(256) k_hot_build(CountTables t, u64 n_short, u64 n_medium, u64 thresh, u64 *__restrict__ placed) {
    u64 np = 0;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_short + n_medium; i += (u64)gridDim.x * blockDim.x) {
        u64 k0, k1, c;
        if (i < n_short) { const SSlot &e = t.stab[t.slist[i]]; k0 = e.key; k1 = 0; c = e.val; }
        else { const MSlot &e = t.medtab[t.mlist[i - n_short]]; k0 = e.k0; k1 = e.k1; c = e.val; }
        if (c < thresh) continue;
        if (hot_claim(t.hot, hot_bucket(t.hot_nb, k0, k1), k0, k1) >= 0) np++;
    }
    for (int d = 16; d; d >>= 1) np += __shfl_down_sync(0xffffffffu, np, d);
    if (lane_id() == 0 && np) atomicAdd(placed, np);
}
// counts of the hot table -> big tables (the keys stay, the counts restart at zero)
__global__ void __launch_bounds__(256) k_hot_flush(CountTables t) {
    for (u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x; s < 2 * t.hot_nb; s += (u64)gridDim.x * blockDim.x) {
        const u64 c = t.hcnt[s];
        if (!c) continue;
        t.hcnt[s] = 0;
        const ulonglong2 k = t.hot[s];
        if (k.y == 0) short_add(t, k.x, c); else medium_add(t, k.x, k.y, c);
    }
}

// ---- table growth: re-insert every word of an old table's list into a bigger table, at the same position of the new list ------
// (so counters[0], [7], [1] and [2] stay as they are)
__global__ void __launch_bounds__(256) k_rehash_short(const SSlot *__restrict__ otab, const u32 *__restrict__ olist, u64 n_old, CountTables t) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_old; i += (u64)gridDim.x * blockDim.x) {
        const SSlot &o = otab[olist[i]];
        t.slist[i] = (u32)short_insert_unique(t, o.key, o.val);
    }
}
__global__ void __launch_bounds__(256) k_rehash_medium(const MSlot *__restrict__ otab, const u32 *__restrict__ olist, u64 n_old, CountTables t) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_old; i += (u64)gridDim.x * blockDim.x) {
        const MSlot &o = otab[olist[i]];
        t.mlist[i] = (u32)medium_insert_unique(t, o.k0, o.k1, o.val);
    }
}
__global__ void __launch_bounds__(256) k_rehash_long(const LSlot *__restrict__ otab, const u32 *__restrict__ olist, u64 n_old, CountTables t) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_old; i += (u64)gridDim.x * blockDim.x) {
        const LSlot &o = otab[olist[i]];
        t.llist[i] = (u32)long_insert_unique(t, o.meta, o.hash, o.val);
    }
}

// ---- re-homing: copy representatives that still point into the text arena to the pool ---------
// (only the long words claimed since the last re-homing can point into the arena: list positions [first, n_long))
__global__ void __launch_bounds__(256) k_rehome_sizes(CountTables t, u64 first, u64 n_long, u64 *__restrict__ need /* [0] */) {
    u64 c = 0;
    for (u64 i = first + (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_long; i += (u64)gridDim.x * blockDim.x) {
        u64 m = t.ltab[t.llist[i]].meta;
        if (!((m >> META_LEN_BITS) & META_POOL_BIT)) c += m & META_LEN_MASK;
    }
    for (int d = 16; d; d >>= 1) c += __shfl_down_sync(0xffffffffu, c, d);
    if (lane_id() == 0 && c) atomicAdd(&need[0], c);
}
__global__ void __launch_bounds__(256) k_rehome_copy(CountTables t, u64 first, u64 n_long, uint8_t *__restrict__ pool, u64 *__restrict__ cursor) {
    for (u64 i = first + (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_long; i += (u64)gridDim.x * blockDim.x) {
        const u64 s = t.llist[i];
        u64 m = t.ltab[s].meta;
        if ((m >> META_LEN_BITS) & META_POOL_BIT) continue;
        u32 len = (u32)(m & META_LEN_MASK);
        u64 o = atomicAdd(cursor, (u64)len);
        const uint8_t *src = t.text + (m >> META_LEN_BITS);
        for (u32 k = 0; k < len; k++) pool[o + k] = src[k];
        t.ltab[s].meta = ((o | META_POOL_BIT) << META_LEN_BITS) | len;
    }
}

// ---- import of another rank's table: words = blob/offs/counts ---------------------------------
__global__ void __launch_bounds__(256) k_import_words(CountTables t, const uint8_t *__restrict__ blob_in_pool, u64 pool_base,
                                                     const u64 *__restrict__ offs, const i64 *__restrict__ counts, u64 n_words) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_words; i += (u64)gridDim.x * blockDim.x) {
        u64 o = offs[i]; u64 len = offs[i + 1] - o;
        const uint8_t *p = blob_in_pool + o;
        if (len == 0) continue;
        if (len <= MED_MAX) {
            u64 k0, k1;
            pretoken_key(p, (u32)len, k0, k1);
            if (k1 == 0) short_add(t, k0, (u64)counts[i]); else medium_add(t, k0, k1, (u64)counts[i]);
        } else if (len <= MAX_TOKEN_LEN) {
            long_add(t, p, (u32)len, (pool_base + o) | META_POOL_BIT, (u64)counts[i]);
        } else t.counters[5] = 1;
    }
}

// ---- the k-th unique word: short words first, then medium, then long (list order) -------------------------------------
struct WordRef { u32 len; u64 cnt; const uint8_t *src; uint8_t tmp[16]; };
__device__ __forceinline__ void word_at(const CountTables &t, const WordCounts &wc, u64 i, WordRef &w) {
    if (i < wc.n_short) {
        const SSlot &e = t.stab[t.slist[i]];
        const u64 k = e.key;
        w.len = (u32)(k >> 56); w.cnt = e.val;
        for (u32 j = 0; j < 8; j++) w.tmp[j] = (uint8_t)(k >> (8 * j));
        w.src = w.tmp;
    } else if (i < wc.n_short + wc.n_medium) {
        const MSlot &e = t.medtab[t.mlist[i - wc.n_short]];
        const u64 k0 = e.k0, k1 = e.k1;
        w.len = (u32)(k1 >> 56); w.cnt = e.val;
        for (u32 j = 0; j < 8; j++) { w.tmp[j] = (uint8_t)(k0 >> (8 * j)); w.tmp[8 + j] = (uint8_t)(k1 >> (8 * j)); }
        w.src = w.tmp;
    } else {
        const LSlot &e = t.ltab[t.llist[i - wc.n_short - wc.n_medium]];
        const u64 m = e.meta;
        w.len = (u32)(m & META_LEN_MASK); w.cnt = e.val; w.src = rep_ptr(t, m);
    }
}
__device__ __forceinline__ u32 word_len_at(const CountTables &t, const WordCounts &wc, u64 i) {
    if (i < wc.n_short) return (u32)(t.stab[t.slist[i]].key >> 56);
    if (i < wc.n_short + wc.n_medium) return (u32)(t.medtab[t.mlist[i - wc.n_short]].k1 >> 56);
    return (u32)(t.ltab[t.llist[i - wc.n_short - wc.n_medium]].meta & META_LEN_MASK);
}

// ---- export: (bytes, offs, counts) of every word ----------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_export_lens(CountTables t, WordCounts wc, u64 n_words, u32 *__restrict__ lens) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_words; i += (u64)gridDim.x * blockDim.x) lens[i] = word_len_at(t, wc, i);
}
__global__ void __launch_bounds__(256) k_export_write(CountTables t, WordCounts wc, u64 n_words, const u64 *__restrict__ byte_off,
                                                     uint8_t *__restrict__ blob, u64 *__restrict__ offs, i64 *__restrict__ counts) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_words; i += (u64)gridDim.x * blockDim.x) {
        WordRef w;
        word_at(t, wc, i, w);
        const u64 o = byte_off[i];
        offs[i] = o;
        for (u32 j = 0; j < w.len; j++) blob[o + j] = w.src[j];
        counts[i] = (i64)w.cnt;
    }
}

// =============================================================================================
// 2. Word list + initial pair statistics
//    encode_subwords (train.py:31-32) and calculate_byte_pair_frequencies (train.py:35-49)
// =============================================================================================

__device__ __forceinline__ bool equals_special(const uint8_t *p, u32 len, const uint8_t *sp_blob, const u32 *sp_offs, int n_sp) {
    for (int s = 0; s < n_sp; s++) {
        u32 o = sp_offs[s], l = sp_offs[s + 1] - o;
        if (l != len) continue;
        bool eq = true;
        for (u32 k = 0; k < len && eq; k++) eq = p[k] == sp_blob[o + k];     // (p may be a small local array: plain byte loop)
        if (eq) return true;
    }
    return false;
}

// Pretokens equal to a special token are dropped (train.py:25).  Words of one byte carry no pair and are
// skipped: they can never be touched by the merge loop.
__global__ void __launch_bounds__(256) k_build_words(CountTables t, WordCounts wc, Words W, const uint8_t *__restrict__ sp_blob,
                                                    const u32 *__restrict__ sp_offs, int n_sp) {
    const u64 n_unique = wc.n_short + wc.n_medium + wc.n_long;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_unique; i += (u64)gridDim.x * blockDim.x) {
        WordRef wr;
        word_at(t, wc, i, wr);
        const u32 l = wr.len; const uint8_t *src = wr.src; const u64 c = wr.cnt;
        if (l < 2 || c == 0) continue;
        if (n_sp && equals_special(src, l, sp_blob, sp_offs, n_sp)) continue;
        // word index and symbol space: one atomic per group of threads that arrive here together (12 M words would
        // otherwise serialise on three addresses)
        cg::coalesced_group g = cg::coalesced_threads();
        const u32 need = l + 1;                                            // one separator in front of every word
        const u32 pre = cg::exclusive_scan(g, need);
        const u32 lmax = cg::reduce(g, l, cg::greater<u32>());
        u64 w0 = 0, o0 = 0;
        if (g.thread_rank() == g.size() - 1) {
            w0 = atomicAdd(&W.counters[0], (u64)g.size());
            o0 = atomicAdd(&W.counters[1], (u64)(pre + need));
            atomicMax(&W.counters[2], (u64)lmax);
        }
        const u64 w = g.shfl(w0, g.size() - 1) + g.thread_rank();
        const u64 o = SYM_PAD + g.shfl(o0, g.size() - 1) + pre + 1;
        WordMeta wm; wm.off = (u32)o; wm.len = l; wm.cnt = (i64)c;
        W.meta[w] = wm;
        for (u32 j = 0; j < l; j++) W.sym[o + j] = src[j];                 // (the array was filled with SYM_SEP)
    }
}

// The dense byte-pair table straight from the count tables (what k_build_words + k_init_pair_counts compute, without
// materialising the words): the per-rank table of the multi-GPU linearity check.
__global__ void __launch_bounds__(256) k_dense_pairs(CountTables t, WordCounts wc, const uint8_t *__restrict__ sp_blob, const u32 *__restrict__ sp_offs,
                                                    int n_sp, u64 *__restrict__ dense /* 65536 */) {
    const u64 n_unique = wc.n_short + wc.n_medium + wc.n_long;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_unique; i += (u64)gridDim.x * blockDim.x) {
        WordRef wr;
        word_at(t, wc, i, wr);
        const u32 l = wr.len; const uint8_t *src = wr.src; const u64 c = wr.cnt;
        if (l < 2 || c == 0) continue;
        if (n_sp && equals_special(src, l, sp_blob, sp_offs, n_sp)) continue;
        u32 prev = src[0];
        for (u32 j = 1; j < l; j++) { const u32 cur = src[j]; atomicAdd(&dense[(prev << 8) | cur], c); prev = cur; }
    }
}

// The pair tables of the initial words are privatised per CTA: byte pairs are Zipfian (a few hundred addresses take most of the
// ~10^8 updates), and one global atomic per pair occurrence serialised on them (ncu: 4.7 ms at 1.7 % of the DRAM bandwidth and an IPC
// of 0.05).  Pairs of two ASCII bytes -- nearly all -- are counted in a direct-indexed shared-memory table [a][b] (128 x 128) and
// flushed with one global atomic per CTA and non-empty entry; pairs with a byte >= 0x80 go to the global tables directly.
#define IP_NT 1024
#define IP_PAIRS (128u * 128u)
#define IP_SMEM_COUNTS ((size_t)IP_PAIRS * 12)   // u64 counts + u32 occurrences
#define IP_SMEM_FILL ((size_t)IP_PAIRS * 8)      // u32 occurrences / cursors + u32 bases
__global__ void __launch_bounds__(IP_NT, 1) k_init_pair_counts(Words W, u64 n_words, u64 *__restrict__ dense /* 65536 */,
                                                              u32 *__restrict__ hist /* 65536 */) {
    extern __shared__ __align__(16) unsigned char ip_smem[];
    u64 *s_cnt = reinterpret_cast<u64 *>(ip_smem);
    u32 *s_occ = reinterpret_cast<u32 *>(s_cnt + IP_PAIRS);
    for (u32 i = threadIdx.x; i < IP_PAIRS; i += IP_NT) { s_cnt[i] = 0; s_occ[i] = 0; }
    __syncthreads();
    for (u64 w = (u64)blockIdx.x * IP_NT + threadIdx.x; w < n_words; w += (u64)gridDim.x * IP_NT) {
        const int32_t *s = W.sym + W.meta[w].off; u32 l = W.meta[w].len; u64 c = (u64)W.meta[w].cnt;
        if (l < 2) continue;
        u32 prev = (u32)s[0];
        for (u32 j = 1; j < l; j++) {
            const u32 cur = (u32)s[j];
            if ((prev | cur) < 128u) { const u32 i = (prev << 7) | cur; atomicAdd(&s_cnt[i], c); atomicAdd(&s_occ[i], 1u); }
            else { const u32 p = (prev << 8) | cur; atomicAdd(&dense[p], c); atomicAdd(&hist[p], 1u); }
            prev = cur;
        }
    }
    __syncthreads();
    for (u32 i = threadIdx.x; i < IP_PAIRS; i += IP_NT) {
        const u32 o = s_occ[i];
        if (!o) continue;
        const u32 p = ((i >> 7) << 8) | (i & 127u);
        atomicAdd(&dense[p], s_cnt[i]); atomicAdd(&hist[p], o);
    }
}
// single block: exclusive scan of hist[65536] -> csr_off[65537]; also resets hist to 0 for the fill pass
__global__ void __launch_bounds__(1024) k_csr_scan(u32 *__restrict__ hist, u32 *__restrict__ csr_off) {
    __shared__ u32 s_part[1024];
    u32 tid = threadIdx.x;
    u32 sum = 0;
    for (u32 k = 0; k < 64; k++) sum += hist[tid * 64 + k];
    s_part[tid] = sum;
    __syncthreads();
    if (tid == 0) { u32 a = 0; for (u32 i = 0; i < 1024; i++) { u32 v = s_part[i]; s_part[i] = a; a += v; } csr_off[65536] = a; }
    __syncthreads();
    u32 a = s_part[tid];
    for (u32 k = 0; k < 64; k++) { u32 v = hist[tid * 64 + k]; csr_off[tid * 64 + k] = a; a += v; hist[tid * 64 + k] = 0; }
}
// CSR fill, privatised the same way: a CTA walks ITS words twice (the same static assignment both times) -- first it counts its
// occurrences per ASCII pair in shared memory and reserves a range of every pair's CSR slice with one global atomic, then it writes
// the records at range start + a shared-memory cursor.  (The order of the records inside a pair's slice is arbitrary, as before.)
__global__ void __launch_bounds__(IP_NT, 1) k_csr_fill(Words W, u64 n_words, const u32 *__restrict__ csr_off, u32 *__restrict__ fill,
                                                      Rec *__restrict__ csr_rec) {
    extern __shared__ __align__(16) unsigned char ip_smem[];
    u32 *s_occ = reinterpret_cast<u32 *>(ip_smem), *s_base = s_occ + IP_PAIRS;
    for (u32 i = threadIdx.x; i < IP_PAIRS; i += IP_NT) s_occ[i] = 0;
    __syncthreads();
    for (u64 w = (u64)blockIdx.x * IP_NT + threadIdx.x; w < n_words; w += (u64)gridDim.x * IP_NT) {
        const int32_t *s = W.sym + W.meta[w].off; const u32 l = W.meta[w].len;
        if (l < 2) continue;
        u32 prev = (u32)s[0];
        for (u32 j = 1; j < l; j++) { const u32 cur = (u32)s[j]; if ((prev | cur) < 128u) atomicAdd(&s_occ[(prev << 7) | cur], 1u); prev = cur; }
    }
    __syncthreads();
    for (u32 i = threadIdx.x; i < IP_PAIRS; i += IP_NT) {
        const u32 o = s_occ[i];
        if (o) { const u32 p = ((i >> 7) << 8) | (i & 127u); s_base[i] = csr_off[p] + atomicAdd(&fill[p], o); s_occ[i] = 0; }
    }
    __syncthreads();
    for (u64 w = (u64)blockIdx.x * IP_NT + threadIdx.x; w < n_words; w += (u64)gridDim.x * IP_NT) {
        const u32 off = W.meta[w].off, l = W.meta[w].len;
        const i64 c = W.meta[w].cnt;
        const int32_t *s = W.sym + off;
        if (l < 2) continue;
        u32 prev = (u32)s[0];
        for (u32 j = 1; j < l; j++) {
            const u32 cur = (u32)s[j];
            u32 at;
            if ((prev | cur) < 128u) { const u32 i = (prev << 7) | cur; at = s_base[i] + atomicAdd(&s_occ[i], 1u); }
            else { const u32 p = (prev << 8) | cur; at = csr_off[p] + atomicAdd(&fill[p], 1u); }
            store_rec(&csr_rec[at], 0u, off + j - 1, c);
            prev = cur;
        }
    }
}

// =============================================================================================
// host orchestration
// =============================================================================================
static u64 g_merge_prof[32];
// Debug/profiling aid: per-phase nanoseconds and counters of the last merge loop (see MergeState::prof).
BPE_API void bpe_debug_merge_profile(unsigned long long out[32]) { for (int i = 0; i < 32; i++) out[i] = g_merge_prof[i]; }

struct TrainBufs {
    DevBuf sym, wmeta, wctr;
    DevBuf dense, hist, csr_off, csr_rec;
    DevBuf pkey, pcnt, bmax, bsec, dirty, tok_key, prof, step_prof, merge_cnt, log, log2, bk_lg, bk_start, bk_off, bk_scratch, log_rng, tok_off, tok_len, tok_bytes, bar, cta_prof, merges, ctr;
    void free_all(bpe_ctx *ctx) {
        for (DevBuf *b : {&sym, &wmeta, &wctr, &dense, &hist, &csr_off, &csr_rec, &pkey, &pcnt, &bmax, &bsec,
                          &dirty, &tok_key, &prof, &step_prof, &merge_cnt, &log, &log2, &bk_lg, &bk_start, &bk_off, &bk_scratch, &log_rng, &tok_off, &tok_len, &tok_bytes, &bar, &cta_prof, &merges, &ctr})
            bpe_buf_free(ctx, *b);
    }
};

static CountTables count_tables(bpe_ctx *ctx) {
    CountState *cs = ctx->count;
    CountTables t;
    t.stab = (SSlot *)cs->stab.p; t.scap = cs->scap;
    t.medtab = (MSlot *)cs->mtab.p; t.medcap = cs->mcap;
    t.ltab = (LSlot *)cs->ltab.p; t.lcap = cs->lcap;
    t.slist = (u32 *)cs->slist.p; t.mlist = (u32 *)cs->mlist.p; t.llist = (u32 *)cs->llist.p;
    t.hot = (ulonglong2 *)cs->hot.p; t.hot_nb = cs->hot_nb; t.hcnt = (u64 *)((ulonglong2 *)cs->hot.p + 2 * cs->hot_nb);
    t.text = ctx->text.p ? (const uint8_t *)ctx->text.p + BPE_PAD : nullptr;
    t.pool = (uint8_t *)cs->pool.p;
    t.counters = (u64 *)cs->counters.p;
    return t;
}

void count_state_free(bpe_ctx *ctx) {
    if (!ctx->count) return;
    CountState *cs = ctx->count;
    for (DevBuf *b : {&cs->stab, &cs->mtab, &cs->ltab, &cs->slist, &cs->mlist, &cs->llist, &cs->pool, &cs->counters, &cs->hot}) bpe_buf_free(ctx, *b);
    delete cs;
    ctx->count = nullptr;
}

static int count_tables_alloc(bpe_ctx *ctx, PtCaps cap) {
    const u64 scap = cap.s, mcap = cap.m, lcap = cap.l;
    CountState *cs = ctx->count;
    BPE_TRY(alloc_exact(ctx, cs->stab, scap * 16)); BPE_TRY(alloc_exact(ctx, cs->mtab, mcap * 32)); BPE_TRY(alloc_exact(ctx, cs->ltab, lcap * 32));
    BPE_TRY(alloc_exact(ctx, cs->slist, scap * 4)); BPE_TRY(alloc_exact(ctx, cs->mlist, mcap * 4)); BPE_TRY(alloc_exact(ctx, cs->llist, lcap * 4));   // (written before read: no clearing)
    cudaStream_t st = ctx->stream;
    CUDA_TRY(ctx, cudaMemsetAsync(cs->stab.p, 0, scap * 16, st)); CUDA_TRY(ctx, cudaMemsetAsync(cs->mtab.p, 0, mcap * 32, st));
    CUDA_TRY(ctx, cudaMemsetAsync(cs->ltab.p, 0, lcap * 32, st));
    cs->scap = scap; cs->mcap = mcap; cs->lcap = lcap;
    return BPE_OK;
}

BPE_API int bpe_count_begin(bpe_ctx *ctx) {
    if (!ctx) return BPE_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    if (!ctx->count) ctx->count = new CountState();
    CountState *cs = ctx->count;
    BPE_TRY(bpe_buf_reserve(ctx, cs->counters, 64 * sizeof(u64)));
    CUDA_TRY(ctx, cudaMemsetAsync(cs->counters.p, 0, 64 * sizeof(u64), ctx->stream));
    BPE_TRY(count_tables_alloc(ctx, pt_caps(0, 0, 0, 0, 0)));
    cs->pool_used = 0; cs->active = true; cs->n_pretokens = 0; cs->n_rehomed = 0;
    bpe_buf_free(ctx, cs->hot); cs->hot_nb = 0; cs->hot_seen = 0; cs->hot_builds = 0;
    return BPE_OK;
}

static int read_counters(bpe_ctx *ctx, u64 *out, int k) {
    u64 *host = (u64 *)ctx->pinned;
    CUDA_TRY(ctx, cudaMemcpyAsync(host, ctx->count->counters.p, k * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < k; i++) out[i] = host[i];
    return BPE_OK;
}

// Make sure the tables can absorb `new_short` more unique words of <= 7 bytes and `new_long` of >= 8 bytes (medium and long tables
// together) without exceeding 7/8 load.
// c = the counters as read by read_counters(ctx, c, 8).
static int count_ensure_capacity(bpe_ctx *ctx, const u64 *c, u64 new_short, u64 new_long) {
    CountState *cs = ctx->count;
    const u64 n_short = c[0], n_long = c[1], n_medium = c[7];
    const PtCaps need = pt_caps(n_short, n_medium, n_long, new_short, new_long);
    if (need.s <= cs->scap && need.m <= cs->mcap && need.l <= cs->lcap) return BPE_OK;
    // grow: move old tables aside, allocate, re-insert the words of the old lists
    CountState old_view = *cs;                   // shallow copy of the DevBufs
    cs->stab = DevBuf(); cs->mtab = DevBuf(); cs->ltab = DevBuf(); cs->slist = DevBuf(); cs->mlist = DevBuf(); cs->llist = DevBuf();
    int rc = count_tables_alloc(ctx, {std::max(need.s, cs->scap), std::max(need.m, cs->mcap), std::max(need.l, cs->lcap)});
    if (rc != BPE_OK) return rc;
    CountTables t = count_tables(ctx);
    auto grid_for = [&](u64 n) { return (unsigned)std::min<u64>((u64)ctx->sm_count * bpe_grid_mult(64), (n + 255) / 256); };
    if (n_short) KLAUNCH(k_rehash_short, grid_for(n_short), 256, 0, ctx->stream, (const SSlot *)old_view.stab.p, (const u32 *)old_view.slist.p, n_short, t);
    if (n_medium) KLAUNCH(k_rehash_medium, grid_for(n_medium), 256, 0, ctx->stream, (const MSlot *)old_view.mtab.p, (const u32 *)old_view.mlist.p, n_medium, t);
    if (n_long) KLAUNCH(k_rehash_long, grid_for(n_long), 256, 0, ctx->stream, (const LSlot *)old_view.ltab.p, (const u32 *)old_view.llist.p, n_long, t);
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    for (DevBuf *b : {&old_view.stab, &old_view.mtab, &old_view.ltab, &old_view.slist, &old_view.mlist, &old_view.llist}) bpe_buf_free(ctx, *b);
    static const bool prof = getenv("BPE_COUNT_PROFILE") != nullptr;     // (the growth tests read these notes)
    if (prof) fprintf(stderr, "  [count tables grow: short %llu -> %llu slots (%llu entries), medium %llu -> %llu (%llu), long %llu -> %llu (%llu)]\n",
                      (unsigned long long)old_view.scap, (unsigned long long)cs->scap, (unsigned long long)n_short,
                      (unsigned long long)old_view.mcap, (unsigned long long)cs->mcap, (unsigned long long)n_medium,
                      (unsigned long long)old_view.lcap, (unsigned long long)cs->lcap, (unsigned long long)n_long);
    return BPE_OK;
}

// Add the counts of the hot table back to the big tables (which then hold everything again).
static int count_hot_flush(bpe_ctx *ctx) {
    CountState *cs = ctx->count;
    if (!cs->hot_nb) return BPE_OK;
    CountTables t = count_tables(ctx);
    KLAUNCH(k_hot_flush, (unsigned)std::min<u64>((u64)ctx->sm_count * 16, (2 * cs->hot_nb + 255) / 256), 256, 0, ctx->stream, t);
    CUDA_TRY(ctx, cudaGetLastError());
    return BPE_OK;
}
// (Re)build the hot table from the counts so far: the words counted at least T times, T the smallest threshold that selects at most
// BPE_COUNT_HOT_MAX (default 1 M) words.  c = the counters as read by read_counters(ctx, c, 8).
static int count_hot_rebuild(bpe_ctx *ctx, const u64 *c) {
    CountState *cs = ctx->count;
    cudaStream_t st = ctx->stream;
    static const u64 hot_max = getenv("BPE_COUNT_HOT_MAX") ? (u64)atoll(getenv("BPE_COUNT_HOT_MAX")) : (1ull << 20);
    const u64 n_short = c[0], n_medium = c[7];
    BPE_TRY(count_hot_flush(ctx));
    bpe_buf_free(ctx, cs->hot); cs->hot_nb = 0;
    cs->hot_builds++; cs->hot_seen = c[4];
    // test knob: BPE_COUNT_HOT_TEST=1 builds the table however small the vocabulary is (the parity tests cover it with small corpora)
    static const bool hot_test = getenv("BPE_COUNT_HOT_TEST") != nullptr;
    if (!hot_max || (!hot_test && n_short + n_medium < (1u << 16))) return BPE_OK;   // small vocabularies stay in L2 as they are
    CountTables t = count_tables(ctx);
    u64 *hist = (u64 *)ctx->scratch.p + 16;
    CUDA_TRY(ctx, cudaMemsetAsync(hist, 0, HOT_HIST * sizeof(u64), st));
    const unsigned grid = (unsigned)std::min<u64>((u64)ctx->sm_count * 16, (n_short + n_medium + 255) / 256);
    KLAUNCH(k_hot_hist, grid, 256, 0, st, t, n_short, n_medium, hist);
    u64 *host = (u64 *)ctx->pinned;
    CUDA_TRY(ctx, cudaMemcpyAsync(host, hist, HOT_HIST * sizeof(u64), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    u64 n_hot;
    const u64 thresh = fit_threshold(host, HOT_HIST, hot_max, &n_hot);
    if (thresh >= HOT_HIST || (!hot_test && n_hot < 1024)) return BPE_OK;
    const u64 nb = n_hot + 64;                   // one bucket (two slots) per selected word: ~10 % of them find theirs full
    BPE_TRY(alloc_exact(ctx, cs->hot, nb * 48));
    CUDA_TRY(ctx, cudaMemsetAsync(cs->hot.p, 0, nb * 48, st));
    cs->hot_nb = nb;
    t = count_tables(ctx);
    CUDA_TRY(ctx, cudaMemsetAsync(hist, 0, sizeof(u64), st));
    KLAUNCH(k_hot_build, grid, 256, 0, st, t, n_short, n_medium, thresh, hist);
    CUDA_TRY(ctx, cudaGetLastError());
    static const bool prof = getenv("BPE_COUNT_PROFILE") != nullptr;
    if (prof) {
        CUDA_TRY(ctx, cudaMemcpyAsync(host, hist, sizeof(u64), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
        fprintf(stderr, "  [hot table: %llu words counted >= %llu times, %llu buckets, %llu placed, after %llu pretokens]\n", (unsigned long long)n_hot, (unsigned long long)thresh, (unsigned long long)nb, (unsigned long long)host[0], (unsigned long long)c[4]);
    }
    return BPE_OK;
}

#include <chrono>
static double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
#define COUNT_BATCH_BYTES (256ull << 20)

// Count the pretokens whose start lies in [own_begin, own_end) of the text currently in the arena
// (flags already computed).  spstart (split_special_tokens): the first bytes of the special-token occurrences, which are not counted.
static int count_current_text(bpe_ctx *ctx, u64 n, u64 own_begin, u64 own_end, u64 trust_end, const u32 *spstart = nullptr) {
    CountState *cs = ctx->count;
    cudaStream_t st = ctx->stream;
    if (own_end > n) own_end = n;
    if (own_begin >= own_end) return BPE_OK;
    u64 w_lo = own_begin / 32, w_hi = (own_end + 31) / 32;
    // (test knobs: BPE_COUNT_BATCH_KB = batch size, BPE_COUNT_HOT_AFTER = pretokens before the hot table is first built)
    static const u64 batch_bytes = getenv("BPE_COUNT_BATCH_KB") ? std::max<u64>(1, (u64)atoll(getenv("BPE_COUNT_BATCH_KB"))) << 10 : COUNT_BATCH_BYTES;
    static const u64 hot_after = getenv("BPE_COUNT_HOT_AFTER") ? (u64)atoll(getenv("BPE_COUNT_HOT_AFTER")) : (8ull << 20);
    const u64 words_per_batch = batch_bytes / 32;
    // start bits are counted per RANGE (a quarter of a batch): while no hot table exists the first batch is one range only, so that
    // the cold start -- every queued word a probe of the big tables -- lasts 64 MB instead of 256
    const u64 words_per_range = words_per_batch % 4 == 0 && words_per_batch >= 4 ? words_per_batch / 4 : words_per_batch;
    const u64 ranges_per_batch = words_per_batch / words_per_range;
    const u64 n_ranges = (w_hi - w_lo + words_per_range - 1) / words_per_range;
    // per-range upper bound of new uniques = number of start bits
    BPE_TRY(bpe_buf_reserve(ctx, ctx->tmp0, n_ranges * sizeof(u64)));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->tmp0.p, 0, n_ranges * sizeof(u64), st));
    {
        dim3 grid((unsigned)std::min<u64>(ctx->sm_count * 4, (words_per_range + 255) / 256), (unsigned)n_ranges);
        KLAUNCH(k_popc_ranges, grid, 256, 0, st, (const u32 *)ctx->flags.p + w_lo, w_hi - w_lo, words_per_range, (u64 *)ctx->tmp0.p);
    }
    std::vector<u64> rbound(n_ranges);
    CUDA_TRY(ctx, cudaMemcpyAsync(rbound.data(), ctx->tmp0.p, n_ranges * sizeof(u64), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    std::vector<u64> bstart{0}, bound;           // batches: first range index of each, start bits of each
    for (u64 r0 = 0; r0 < n_ranges;) {
        const u64 k = (r0 == 0 && cs->hot_builds == 0) ? 1 : ranges_per_batch, r1 = std::min(n_ranges, r0 + k);
        u64 sum = 0;
        for (u64 r = r0; r < r1; r++) sum += rbound[r];
        bound.push_back(sum); bstart.push_back(r1);
        r0 = r1;
    }
    const u64 n_batches = bound.size();
    u64 c[8];
    BPE_TRY(read_counters(ctx, c, 8));
    static const bool prof = getenv("BPE_COUNT_PROFILE") != nullptr;
    for (u64 bi = 0; bi < n_batches; bi++) {
        const double tb0 = prof ? now_ms() : 0;
        u64 b_lo = w_lo + bstart[bi] * words_per_range, b_hi = std::min(w_hi, w_lo + bstart[bi + 1] * words_per_range);
        u64 bytes = (b_hi - b_lo) * 32;
        BPE_TRY(count_ensure_capacity(ctx, c, bound[bi], std::min(bound[bi], bytes / (SHORT_MAX + 1) + 1)));
        CountTables t = count_tables(ctx);
        if (bound[bi]) {
            static const int cnt_ctas_per_sm = getenv("BPE_COUNT_CTAS") ? std::max(1, atoi(getenv("BPE_COUNT_CTAS"))) : (int)(1024 / CNT_NT);
            const u64 c_lo = b_lo * 2, c_hi = std::min(b_hi * 2, (n + 15) / 16);
            const u64 steps = (c_hi - c_lo + 32 * CNT_WARPS * CNT_TICKET - 1) / (32 * CNT_WARPS * CNT_TICKET);
            unsigned g2 = (unsigned)std::min<u64>((u64)ctx->sm_count * cnt_ctas_per_sm, std::max<u64>(steps, 1));
            CUDA_TRY(ctx, cudaMemsetAsync(t.counters + 16, 0, 8, st));
            static bool attr_set = false;
            if (!attr_set) {
                CUDA_TRY(ctx, cudaFuncSetAttribute((void *)k_count_pretokens, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CNT_DYN_SMEM));
                CUDA_TRY(ctx, cudaFuncSetAttribute((void *)k_count_pretokens_split, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CNT_DYN_SMEM));
                attr_set = true;
            }
            if (spstart)
                KLAUNCH(k_count_pretokens_split, g2, CNT_NT, CNT_DYN_SMEM, st, t, (const u32 *)ctx->flags.p, spstart, c_lo, c_hi, n, b_lo * 32, own_begin, own_end, trust_end);
            else
                KLAUNCH(k_count_pretokens, g2, CNT_NT, CNT_DYN_SMEM, st, t, (const u32 *)ctx->flags.p, c_lo, c_hi, n, b_lo * 32, own_begin, own_end, trust_end);
        }
        CUDA_TRY(ctx, cudaGetLastError());
        if (bi + 1 < n_batches) {
            BPE_TRY(read_counters(ctx, c, 8));
            // the hot table: built once enough text has been seen to tell frequent words from rare ones, rebuilt twice with better counts
            if ((cs->hot_builds == 0 && c[4] >= hot_after) || (cs->hot_builds >= 1 && cs->hot_builds < 3 && c[4] >= 4 * cs->hot_seen))
                BPE_TRY(count_hot_rebuild(ctx, c));
        }
        if (prof) { cudaStreamSynchronize(st); fprintf(stderr, "  [batch %llu: %llu pretokens] %.2f ms (tables %llu + %llu slots)\n", (unsigned long long)bi, (unsigned long long)bound[bi], now_ms() - tb0, (unsigned long long)cs->scap, (unsigned long long)cs->lcap); }
    }
    BPE_TRY(count_hot_flush(ctx));
    BPE_TRY(read_counters(ctx, c, 8));
    if (c[6]) return bpe_set_error(ctx, BPE_ERR_HALO, "a pretoken that starts in the owned range runs past the right halo");
    if (c[3]) return bpe_set_error(ctx, BPE_ERR_CAPACITY, "pretoken table overflow");
    if (c[5]) return bpe_set_error(ctx, BPE_ERR_UNSUPPORTED, "a pretoken longer than %u bytes", MAX_TOKEN_LEN);
    cs->n_pretokens = c[4];
    return BPE_OK;
}

// Copy long-word representatives out of the (transient) text arena into the persistent pool.
static int count_rehome(bpe_ctx *ctx) {
    CountState *cs = ctx->count;
    cudaStream_t st = ctx->stream;
    u64 c[2];
    BPE_TRY(read_counters(ctx, c, 2));
    const u64 n_long = c[1], first = cs->n_rehomed;
    if (n_long <= first) return BPE_OK;
    CountTables t = count_tables(ctx);
    u64 *scr = (u64 *)ctx->scratch.p + 8;
    CUDA_TRY(ctx, cudaMemsetAsync(scr, 0, 16, st));
    unsigned grid = (unsigned)std::min<u64>((u64)ctx->sm_count * bpe_grid_mult(64), (n_long - first + 255) / 256);
    KLAUNCH(k_rehome_sizes, grid, 256, 0, st, t, first, n_long, scr);
    u64 *host = (u64 *)ctx->pinned;
    CUDA_TRY(ctx, cudaMemcpyAsync(host, scr, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    u64 need = host[0];
    cs->n_rehomed = n_long;
    if (!need) return BPE_OK;
    if (cs->pool_used + need + 16 > cs->pool.cap) {  // (+ 16: the key loads read up to 15 bytes past a word)
        DevBuf nb;
        BPE_TRY(bpe_buf_reserve(ctx, nb, (cs->pool_used + need) * 2 + (1 << 20)));
        if (cs->pool_used) CUDA_TRY(ctx, cudaMemcpyAsync(nb.p, cs->pool.p, cs->pool_used, cudaMemcpyDeviceToDevice, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
        bpe_buf_free(ctx, cs->pool);
        cs->pool = nb;
        t = count_tables(ctx);
    }
    host[0] = cs->pool_used;
    CUDA_TRY(ctx, cudaMemcpyAsync(scr + 1, host, 8, cudaMemcpyHostToDevice, st));
    KLAUNCH(k_rehome_copy, grid, 256, 0, st, t, first, n_long, (uint8_t *)cs->pool.p, scr + 1);
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    cs->pool_used += need;
    return BPE_OK;
}

// ---- split_special_tokens (BPE_TRAIN_SPLIT_SPECIALS) ----------------------------------------------------------------------
// The text is split on the special-token occurrences as Tokenizer.segment splits it (leftmost match, longest special first: the
// encoder's k_special_candidates / k_special_resolve inside ctx_run_flags), every piece is pretokenised as a whole text, and the
// occurrences themselves are counted nowhere (k_count_pretokens_split).  The specials, longest first, on the host (exact cuts) and
// on the device.
struct SplitSpecials {
    std::vector<uint8_t> blob; std::vector<u32> offs{0};
    const uint8_t *blob_dev = nullptr; const u32 *offs_dev = nullptr; u32 max_len = 0;
    int n() const { return (int)offs.size() - 1; }
};
static int split_specials_upload(bpe_ctx *ctx, const uint8_t *blob, const u32 *offs, int n_sp, SplitSpecials &sp) {
    std::vector<int> order;
    for (int i = 0; i < n_sp; i++) order.push_back(i);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return offs[a + 1] - offs[a] > offs[b + 1] - offs[b]; });
    for (int i : order) { sp.blob.insert(sp.blob.end(), blob + offs[i], blob + offs[i + 1]); sp.offs.push_back((u32)sp.blob.size()); }
    return ctx_upload_specials(ctx, sp.blob.data(), sp.offs.data(), sp.n(), &sp.blob_dev, &sp.offs_dev, &sp.max_len);
}
// flags of the text in the arena with the specials split out (sp null: the default mode); the special starts the count skips, or null
static int run_flags_for_training(bpe_ctx *ctx, u64 *n_io, bool translate, const SplitSpecials *sp, const u32 **spstart,
                                  u64 err_lo = 0, u64 err_hi = ~0ull) {
    *spstart = nullptr;
    if (!sp) return ctx_run_flags(ctx, n_io, translate, nullptr, nullptr, 0, 0, err_lo, err_hi);
    BPE_TRY(ctx_run_flags(ctx, n_io, translate, sp->blob_dev, sp->offs_dev, sp->n(), sp->max_len, err_lo, err_hi));
    if (sp->max_len) *spstart = (const u32 *)ctx->spstart.p;
    return BPE_OK;
}
// flags & BPE_TRAIN_SPLIT_SPECIALS: the specials uploaded into `split`, which the counting paths then use; BPE_ERR_ARG for unknown bits
static int split_from_flags(bpe_ctx *ctx, int flags, const uint8_t *specials_blob, const uint32_t *special_offs, int n_specials,
                            SplitSpecials &split, const SplitSpecials **use) {
    *use = nullptr;
    if (!ctx || (flags & ~BPE_TRAIN_SPLIT_SPECIALS) || (n_specials > 0 && (!specials_blob || !special_offs))) return BPE_ERR_ARG;
    if (!(flags & BPE_TRAIN_SPLIT_SPECIALS)) return BPE_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    BPE_TRY(split_specials_upload(ctx, specials_blob, special_offs, n_specials, split));
    *use = &split;
    return BPE_OK;
}

// sp (split mode): the shard is one whole text, cut from the file at exact boundaries (own range = all of it, no halo).
static int count_add_shard(bpe_ctx *ctx, const uint8_t *text, u64 n, bool on_device, u64 own_begin, u64 own_end, int at_file_end,
                           const SplitSpecials *sp = nullptr) {
    if (!ctx || !ctx->count || !ctx->count->active || (!text && n) || own_begin > own_end || own_end > n) return BPE_ERR_ARG;
    if (sp && (own_begin != 0 || own_end != n)) return bpe_set_error(ctx, BPE_ERR_ARG, "with BPE_TRAIN_SPLIT_SPECIALS a shard is counted whole");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    static const bool prof = getenv("BPE_COUNT_PROFILE") != nullptr;     // debug aid: host-side wall time of the phases (synchronising)
    double t0 = 0, t1 = 0, t2 = 0, t3 = 0;
    if (prof) { cudaStreamSynchronize(ctx->stream); t0 = now_ms(); }
    BPE_TRY(ctx_load_text(ctx, text, n, on_device));
    u64 nn = n;
    // only ill-formed sequences that start in the owned range are this shard's to report
    const u32 *spstart;
    BPE_TRY(run_flags_for_training(ctx, &nn, false, sp, &spstart, own_begin, own_end));
    if (ctx->saw_cr) return bpe_set_error(ctx, BPE_ERR_NEWLINE, "the shard contains a carriage return");
    if (prof) { cudaStreamSynchronize(ctx->stream); t1 = now_ms(); }
    // start bits in the last 16 bytes of a shard that is cut mid-file lack their right context
    u64 trust_end = at_file_end || sp ? n : (n >= 16 ? n - 16 : 0);
    BPE_TRY(count_current_text(ctx, n, own_begin, own_end, trust_end, spstart));
    if (prof) { cudaStreamSynchronize(ctx->stream); t2 = now_ms(); }
    int rc = count_rehome(ctx);
    if (prof) { cudaStreamSynchronize(ctx->stream); t3 = now_ms(); fprintf(stderr, "[count_add_shard %.2f GB] load+flags %.2f ms, count %.2f ms, rehome %.2f ms\n", n / 1e9, t1 - t0, t2 - t1, t3 - t2); }
    return rc;
}
BPE_API int bpe_count_add_shard(bpe_ctx *ctx, const uint8_t *text_host, uint64_t n, uint64_t own_begin, uint64_t own_end,
                                int at_file_start, int at_file_end) {
    (void)at_file_start;                         // the halo bytes carry all the left context the stencil needs
    return count_add_shard(ctx, text_host, n, false, own_begin, own_end, at_file_end);
}
BPE_API int bpe_count_add_shard_dev(bpe_ctx *ctx, const uint8_t *text_dev, uint64_t n, uint64_t own_begin, uint64_t own_end,
                                    int at_file_start, int at_file_end) {
    (void)at_file_start;
    return count_add_shard(ctx, text_dev, n, true, own_begin, own_end, at_file_end);
}
static int count_add_shard_ex(bpe_ctx *ctx, const uint8_t *text, u64 n, bool on_device, u64 own_begin, u64 own_end, int at_file_end,
                              const uint8_t *specials_blob, const uint32_t *special_offs, int n_specials, int flags) {
    SplitSpecials sp; const SplitSpecials *split;
    BPE_TRY(split_from_flags(ctx, flags, specials_blob, special_offs, n_specials, sp, &split));
    return count_add_shard(ctx, text, n, on_device, own_begin, own_end, at_file_end, split);
}
BPE_API int bpe_count_add_shard_ex(bpe_ctx *ctx, const uint8_t *text_host, uint64_t n, uint64_t own_begin, uint64_t own_end,
                                   int at_file_start, int at_file_end, const uint8_t *specials_blob, const uint32_t *special_offs,
                                   int n_specials, int flags) {
    (void)at_file_start;
    return count_add_shard_ex(ctx, text_host, n, false, own_begin, own_end, at_file_end, specials_blob, special_offs, n_specials, flags);
}
BPE_API int bpe_count_add_shard_dev_ex(bpe_ctx *ctx, const uint8_t *text_dev, uint64_t n, uint64_t own_begin, uint64_t own_end,
                                       int at_file_start, int at_file_end, const uint8_t *specials_blob, const uint32_t *special_offs,
                                       int n_specials, int flags) {
    (void)at_file_start;
    return count_add_shard_ex(ctx, text_dev, n, true, own_begin, own_end, at_file_end, specials_blob, special_offs, n_specials, flags);
}

// lens[] and the byte offsets of the export live in tmp1 between export_size and export (n_words entries, not table capacity)
static int count_export_scan(bpe_ctx *ctx, WordCounts *wc_out, u64 *n_words_out, u64 *blob_bytes_out) {
    cudaStream_t st = ctx->stream;
    u64 c[8];
    BPE_TRY(read_counters(ctx, c, 8));
    const WordCounts wc{c[0], c[7], c[1]};
    const u64 n_words = c[0] + c[7] + c[1];
    CountTables t = count_tables(ctx);
    size_t lens_b = round_up((n_words + 1) * 4, 256), boff_b = round_up((n_words + 2) * 8, 256);
    size_t tmp_b = scan_tmp_elems_host(n_words + 1) * 8;
    BPE_TRY(bpe_buf_reserve(ctx, ctx->tmp1, lens_b + boff_b + tmp_b));
    u32 *lens = (u32 *)ctx->tmp1.p;
    u64 *boff = (u64 *)((uint8_t *)lens + lens_b);
    u64 *tmp = (u64 *)((uint8_t *)boff + boff_b);
    u64 *host = (u64 *)ctx->pinned;
    host[0] = 0;
    if (n_words) {
        unsigned grid = (unsigned)std::min<u64>((u64)ctx->sm_count * bpe_grid_mult(64), (n_words + 255) / 256);
        KLAUNCH(k_export_lens, grid, 256, 0, st, t, wc, n_words, lens);
        launch_scan_u32(lens, n_words, boff, tmp, st);
        CUDA_TRY(ctx, cudaGetLastError());
        CUDA_TRY(ctx, cudaMemcpyAsync(host, boff + n_words, 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
    }
    *wc_out = wc; *n_words_out = n_words; *blob_bytes_out = host[0];
    return BPE_OK;
}

BPE_API int bpe_count_export_size(bpe_ctx *ctx, uint64_t *n_words, uint64_t *blob_bytes) {
    if (!ctx || !ctx->count || !n_words || !blob_bytes) return BPE_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    WordCounts wc; u64 nw, nb;
    BPE_TRY(count_export_scan(ctx, &wc, &nw, &nb));
    *n_words = nw; *blob_bytes = nb;
    return BPE_OK;
}

static int count_export(bpe_ctx *ctx, uint8_t *blob, uint64_t *offs, int64_t *counts, bool to_device) {
    if (!ctx || !ctx->count || !offs) return BPE_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    WordCounts wc; u64 nw, nb;
    BPE_TRY(count_export_scan(ctx, &wc, &nw, &nb));
    cudaStream_t st = ctx->stream;
    CountTables t = count_tables(ctx);
    size_t lens_b = round_up((nw + 1) * 4, 256);
    u64 *boff = (u64 *)((uint8_t *)ctx->tmp1.p + lens_b);
    uint8_t *dblob; u64 *doffs; i64 *dcnt;
    if (to_device) { dblob = blob; doffs = (u64 *)offs; dcnt = (i64 *)counts; }
    else {
        size_t ob = round_up(nb + 1, 256), oo = round_up((nw + 1) * 8, 256), oc = round_up((nw + 1) * 8, 256);
        BPE_TRY(bpe_buf_reserve(ctx, ctx->tmp0, ob + oo + oc));
        dblob = (uint8_t *)ctx->tmp0.p; doffs = (u64 *)(dblob + ob); dcnt = (i64 *)(dblob + ob + oo);
    }
    if ((nb && !dblob) || (nw && !dcnt)) return BPE_ERR_ARG;
    if (nw) {
        unsigned grid = (unsigned)std::min<u64>((u64)ctx->sm_count * bpe_grid_mult(64), (nw + 255) / 256);
        KLAUNCH(k_export_write, grid, 256, 0, st, t, wc, nw, boff, dblob, doffs, dcnt);
        CUDA_TRY(ctx, cudaGetLastError());
    }
    if (to_device) {
        CUDA_TRY(ctx, cudaMemcpyAsync(doffs + nw, &nb, 8, cudaMemcpyHostToDevice, st));
    } else {
        if (nb) CUDA_TRY(ctx, cudaMemcpyAsync(blob, dblob, nb, cudaMemcpyDeviceToHost, st));
        if (nw) CUDA_TRY(ctx, cudaMemcpyAsync(offs, doffs, nw * 8, cudaMemcpyDeviceToHost, st));
        if (nw) CUDA_TRY(ctx, cudaMemcpyAsync(counts, dcnt, nw * 8, cudaMemcpyDeviceToHost, st));
    }
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    if (!to_device) offs[nw] = nb;
    return BPE_OK;
}
BPE_API int bpe_count_export(bpe_ctx *ctx, uint8_t *blob, uint64_t *offs, int64_t *counts) {
    return count_export(ctx, blob, offs, counts, false);
}
BPE_API int bpe_count_export_dev(bpe_ctx *ctx, uint8_t *blob_dev, uint64_t *offs_dev, int64_t *counts_dev) {
    return count_export(ctx, blob_dev, offs_dev, counts_dev, true);
}

static int count_import(bpe_ctx *ctx, const uint8_t *blob, const uint64_t *offs, const int64_t *counts, uint64_t n_words, u64 nb,
                        bool from_device) {
    if (!ctx || !ctx->count || !ctx->count->active || (n_words && (!offs || !counts))) return BPE_ERR_ARG;
    if (!n_words) return BPE_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CountState *cs = ctx->count;
    cudaStream_t st = ctx->stream;
    const cudaMemcpyKind kind = from_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    // blob goes straight into the pool (long words keep pointing at it)
    if (cs->pool_used + nb + 16 > cs->pool.cap) {  // (+ 16: the key loads read up to 15 bytes past a word)
        DevBuf nbuf;
        BPE_TRY(bpe_buf_reserve(ctx, nbuf, (cs->pool_used + nb) * 2 + (1 << 20)));
        if (cs->pool_used) CUDA_TRY(ctx, cudaMemcpyAsync(nbuf.p, cs->pool.p, cs->pool_used, cudaMemcpyDeviceToDevice, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
        bpe_buf_free(ctx, cs->pool);
        cs->pool = nbuf;
    }
    u64 base = cs->pool_used;
    if (nb) CUDA_TRY(ctx, cudaMemcpyAsync((uint8_t *)cs->pool.p + base, blob, nb, kind, st));
    cs->pool_used += nb;
    const u64 *doffs; const i64 *dcnt;
    if (from_device) { doffs = (const u64 *)offs; dcnt = (const i64 *)counts; }
    else {
        size_t ob = round_up((n_words + 1) * 8, 256);
        BPE_TRY(bpe_buf_reserve(ctx, ctx->tmp0, ob * 2));
        u64 *o = (u64 *)ctx->tmp0.p; i64 *c2 = (i64 *)((uint8_t *)ctx->tmp0.p + ob);
        CUDA_TRY(ctx, cudaMemcpyAsync(o, offs, (n_words + 1) * 8, cudaMemcpyHostToDevice, st));
        CUDA_TRY(ctx, cudaMemcpyAsync(c2, counts, n_words * 8, cudaMemcpyHostToDevice, st));
        doffs = o; dcnt = c2;
    }
    u64 c[8];
    BPE_TRY(read_counters(ctx, c, 8));
    BPE_TRY(count_ensure_capacity(ctx, c, n_words, 2 * n_words));   // (any mix of lengths: the bound for >= 16 bytes is half the one for >= 8)
    CountTables t = count_tables(ctx);
    unsigned grid = (unsigned)std::min<u64>((u64)ctx->sm_count * bpe_grid_mult(64), (n_words + 255) / 256);
    KLAUNCH(k_import_words, grid, 256, 0, st, t, (const uint8_t *)cs->pool.p + base, base, doffs, dcnt, n_words);
    CUDA_TRY(ctx, cudaGetLastError());
    BPE_TRY(read_counters(ctx, c, 8));
    if (c[3]) return bpe_set_error(ctx, BPE_ERR_CAPACITY, "pretoken table overflow on import");
    if (c[5]) return bpe_set_error(ctx, BPE_ERR_UNSUPPORTED, "an imported word is longer than %u bytes", MAX_TOKEN_LEN);
    return BPE_OK;
}
BPE_API int bpe_count_import(bpe_ctx *ctx, const uint8_t *blob, const uint64_t *offs, const int64_t *counts, uint64_t n_words) {
    return count_import(ctx, blob, offs, counts, n_words, n_words ? offs[n_words] : 0, false);
}
BPE_API int bpe_count_import_dev(bpe_ctx *ctx, const uint8_t *blob_dev, const uint64_t *offs_dev, const int64_t *counts_dev,
                                 uint64_t n_words, uint64_t blob_bytes) {
    return count_import(ctx, blob_dev, offs_dev, counts_dev, n_words, blob_bytes, true);
}

// Dense byte-pair table of the current counts (train.py:35-49 at merge-loop start).
BPE_API int bpe_count_pair_table(bpe_ctx *ctx, const uint8_t *specials_blob, const uint32_t *special_offs, int n_specials,
                                 int64_t *dense_out) {
    if (!ctx || !ctx->count || !dense_out || (n_specials > 0 && (!specials_blob || !special_offs))) return BPE_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const uint8_t *spb; const u32 *spo; u32 spmax;
    BPE_TRY(ctx_upload_specials(ctx, specials_blob, special_offs, n_specials, &spb, &spo, &spmax));
    DevBuf dense;
    struct G { bpe_ctx *c; DevBuf *b; ~G() { bpe_buf_free(c, *b); } } g{ctx, &dense};
    BPE_TRY(bpe_buf_reserve(ctx, dense, 65536 * 8));
    CUDA_TRY(ctx, cudaMemsetAsync(dense.p, 0, 65536 * 8, st));
    CountTables t = count_tables(ctx);
    u64 c[8];
    BPE_TRY(read_counters(ctx, c, 8));
    const WordCounts wc{c[0], c[7], c[1]};
    if (c[0] + c[7] + c[1]) {
        unsigned grid = (unsigned)std::min<u64>((u64)ctx->sm_count * bpe_grid_mult(64), (c[0] + c[7] + c[1] + 255) / 256);
        KLAUNCH(k_dense_pairs, grid, 256, 0, st, t, wc, spb, spo, n_specials, (u64 *)dense.p);
    }
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaMemcpyAsync(dense_out, dense.p, 65536 * 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    return BPE_OK;
}

BPE_API int bpe_train_set_live(bpe_ctx *ctx, int32_t *live_pairs, int capacity_merges) {
    if (!ctx || capacity_merges < 0) return BPE_ERR_ARG;
    if (live_pairs) {                            // the kernel writes it directly: it must be page-locked host memory
        cudaPointerAttributes a{};
        if (cudaPointerGetAttributes(&a, live_pairs) != cudaSuccess || a.type != cudaMemoryTypeHost) {
            cudaGetLastError();
            return bpe_set_error(ctx, BPE_ERR_ARG, "bpe_train_set_live: the buffer must be page-locked host memory (bpe_host_alloc)");
        }
    }
    ctx->live_pairs = live_pairs; ctx->live_cap = live_pairs ? capacity_merges : 0;
    return BPE_OK;
}

BPE_API int bpe_last_pair_table(bpe_ctx *ctx, int64_t *dense_out) {
    if (!ctx || !dense_out) return BPE_ERR_ARG;
    if (ctx->last_dense.size() != 65536) return bpe_set_error(ctx, BPE_ERR_ARG, "bpe_last_pair_table: no training call has built a pair table on this context");
    memcpy(dense_out, ctx->last_dense.data(), 65536 * 8);
    return BPE_OK;
}

// ---- merge phase ---------------------------------------------------------------------------------
static int run_merges(bpe_ctx *ctx, const uint8_t *sp_blob, const u32 *sp_offs, int n_sp, int n_merges,
                      int32_t *merge_pairs_out, int *n_done, bpe_train_stats *stats, EvTimer &tm, int ev_start) {
    cudaStream_t st = ctx->stream;
    CountState *cs = ctx->count;
    TrainBufs B;
    struct Guard { TrainBufs &b; bpe_ctx *c; ~Guard() { b.free_all(c); } } guard{B, ctx};
    u64 c[8];
    BPE_TRY(read_counters(ctx, c, 8));
    const WordCounts wc{c[0], c[7], c[1]};
    const u64 long_bytes = c[2];
    u64 max_words = wc.n_short + wc.n_medium + wc.n_long, max_syms = wc.n_short * SHORT_MAX + wc.n_medium * MED_MAX + long_bytes;
    const u64 sym_slots = max_syms + max_words + 2 * SYM_PAD;
    if (sym_slots >= (1ull << 32)) return bpe_set_error(ctx, BPE_ERR_UNSUPPORTED, "more than 2^32 symbols in unique words");
    const uint8_t *spb; const u32 *spo; u32 spmax;
    BPE_TRY(ctx_upload_specials(ctx, sp_blob, sp_offs, n_sp, &spb, &spo, &spmax));

    int ev_build0 = tm.mark();
    BPE_TRY(alloc_exact(ctx, B.sym, sym_slots * 4)); BPE_TRY(alloc_exact(ctx, B.wmeta, (max_words + 1) * sizeof(WordMeta)));
    BPE_TRY(alloc_exact(ctx, B.wctr, 64));
    CUDA_TRY(ctx, cudaMemsetAsync(B.sym.p, 0xFF, sym_slots * 4, st));           // SYM_SEP everywhere: padding and word separators
    CUDA_TRY(ctx, cudaMemsetAsync(B.wctr.p, 0, 64, st));
    Words W{(int32_t *)B.sym.p, (WordMeta *)B.wmeta.p, (u64 *)B.wctr.p};
    CountTables t = count_tables(ctx);
    if (max_words) {
        unsigned grid = (unsigned)std::min<u64>((u64)ctx->sm_count * bpe_grid_mult(64), (max_words + 255) / 256);
        KLAUNCH(k_build_words, grid, 256, 0, st, t, wc, W, spb, spo, n_sp);
        CUDA_TRY(ctx, cudaGetLastError());
    }
    u64 *host = (u64 *)ctx->pinned;
    CUDA_TRY(ctx, cudaMemcpyAsync(host, B.wctr.p, 24, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    u64 n_words = host[0], n_syms = host[1] - host[0], max_len = host[2];     // host[1] counts one separator per word

    BPE_TRY(alloc_exact(ctx, B.dense, 65536 * 8)); BPE_TRY(alloc_exact(ctx, B.hist, 65536 * 4));
    BPE_TRY(alloc_exact(ctx, B.csr_off, 65537 * 4)); BPE_TRY(alloc_exact(ctx, B.csr_rec, (n_syms + 1) * sizeof(Rec)));
    CUDA_TRY(ctx, cudaMemsetAsync(B.dense.p, 0, 65536 * 8, st)); CUDA_TRY(ctx, cudaMemsetAsync(B.hist.p, 0, 65536 * 4, st));
    unsigned wgrid = (unsigned)std::max<u64>(1, std::min<u64>((u64)ctx->sm_count, (n_words + IP_NT - 1) / IP_NT));
    static bool ip_attr = false;
    if (!ip_attr) {
        CUDA_TRY(ctx, cudaFuncSetAttribute((void *)k_init_pair_counts, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)IP_SMEM_COUNTS));
        CUDA_TRY(ctx, cudaFuncSetAttribute((void *)k_csr_fill, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)IP_SMEM_FILL));
        ip_attr = true;
    }
    KLAUNCH(k_init_pair_counts, wgrid, IP_NT, IP_SMEM_COUNTS, st, W, n_words, (u64 *)B.dense.p, (u32 *)B.hist.p);
    KLAUNCH(k_csr_scan, 1, 1024, 0, st, (u32 *)B.hist.p, (u32 *)B.csr_off.p);
    KLAUNCH(k_csr_fill, wgrid, IP_NT, IP_SMEM_FILL, st, W, n_words, (const u32 *)B.csr_off.p, (u32 *)B.hist.p, (Rec *)B.csr_rec.p);
    CUDA_TRY(ctx, cudaGetLastError());
    std::vector<u64> dense(65536);
    CUDA_TRY(ctx, cudaMemcpyAsync(dense.data(), B.dense.p, 65536 * 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    ctx->last_dense.assign(dense.begin(), dense.end());

    // pair table: sized for the keys we expect (initial pairs + a fraction of the symbols), grown x4 by
    // the host whenever the kernel reports it more than half full (all loop state lives in HBM, so the
    // persistent kernel is simply relaunched after the rehash).
    u64 n_pairs0 = 0;
    for (u64 v : dense) n_pairs0 += v != 0;
    // At least 2^22 slots (64 MB): every 64-slot block reports only its largest pair, so the several-merges-per-step rule needs
    // the top pairs in different blocks (a small table put the top 16 of a TinyStories-sized run into a few hundred blocks and the
    // hidden second-largest counts cut the batches short).  The grid is sized from the natural capacity, not from the floor.
    const u64 pcap_natural = next_pow2(std::max<u64>(1 << 12, std::max<u64>(8 * n_pairs0, n_syms / 8)));
    static const u64 pcap_floor = getenv("BPE_MERGE_PCAP_MIN") ? std::max<u64>(1 << 12, next_pow2(strtoull(getenv("BPE_MERGE_PCAP_MIN"), nullptr, 10))) : (1ull << 22);
    u64 pcap = std::max(pcap_natural, pcap_floor);
    MergeState M;
    memset(&M, 0, sizeof(M));
    M.W = W; M.n_words = (u32)n_words;
    auto alloc_pair_table = [&](u64 cap) -> int {
        M.pcap = cap; M.n_blocks = (u32)(cap / PB);
        BPE_TRY(alloc_exact(ctx, B.pkey, cap * 8)); BPE_TRY(alloc_exact(ctx, B.pcnt, cap * 8));
        BPE_TRY(alloc_exact(ctx, B.bmax, (u64)M.n_blocks * sizeof(Best))); BPE_TRY(alloc_exact(ctx, B.dirty, M.n_blocks));
        BPE_TRY(alloc_exact(ctx, B.bsec, (u64)M.n_blocks * 4));
        CUDA_TRY(ctx, cudaMemsetAsync(B.pkey.p, 0xFF, cap * 8, st)); CUDA_TRY(ctx, cudaMemsetAsync(B.pcnt.p, 0, cap * 8, st));
        CUDA_TRY(ctx, cudaMemsetAsync(B.dirty.p, 1, M.n_blocks, st));          // every block is rescanned in the first step
        CUDA_TRY(ctx, cudaMemsetAsync(B.bsec.p, 0, (u64)M.n_blocks * 4, st));
        M.pkey = (u64 *)B.pkey.p; M.pcnt = (i64 *)B.pcnt.p; M.bmax = (Best *)B.bmax.p; M.bsec = (u32 *)B.bsec.p; M.dirty = (uint8_t *)B.dirty.p;
        return BPE_OK;
    };
    BPE_TRY(alloc_pair_table(pcap));
    u64 log_cap = 2 * n_syms + 16;
    BPE_TRY(alloc_exact(ctx, B.log, log_cap * sizeof(Rec))); BPE_TRY(alloc_exact(ctx, B.log_rng, ((u64)n_merges + 2) * 16));
    u64 n_tok_max = 256 + (u64)n_merges;
    u64 tok_bytes_cap = 256 + (u64)n_merges * 2 * std::max<u64>(max_len, 1);
    if (tok_bytes_cap > (4ull << 30)) tok_bytes_cap = 4ull << 30;
    BPE_TRY(alloc_exact(ctx, B.tok_off, n_tok_max * 4)); BPE_TRY(alloc_exact(ctx, B.tok_len, n_tok_max * 4));
    BPE_TRY(alloc_exact(ctx, B.tok_key, n_tok_max * 8));
    BPE_TRY(alloc_exact(ctx, B.tok_bytes, tok_bytes_cap)); BPE_TRY(alloc_exact(ctx, B.merge_cnt, ((u64)n_merges + 1) * 8));
    BPE_TRY(alloc_exact(ctx, B.merges, ((u64)n_merges + 1) * 8)); BPE_TRY(alloc_exact(ctx, B.ctr, MG_CTR_WORDS * 8));
    BPE_TRY(alloc_exact(ctx, B.prof, 256)); CUDA_TRY(ctx, cudaMemsetAsync(B.prof.p, 0, 256, st));
    CUDA_TRY(ctx, cudaMemsetAsync(B.log_rng.p, 0, ((u64)n_merges + 2) * 16, st));
    {   // byte tokens: bytes(i) = [i], rank(i) = i; counters
        std::vector<u32> toff(256), tlen(256, 1); std::vector<uint8_t> tb(256); std::vector<u64> tk(256);
        for (int i = 0; i < 256; i++) { toff[i] = i; tb[i] = (uint8_t)i; tk[i] = (u64)i << 56; }
        CUDA_TRY(ctx, cudaMemcpyAsync(B.tok_off.p, toff.data(), 1024, cudaMemcpyHostToDevice, st));
        CUDA_TRY(ctx, cudaMemcpyAsync(B.tok_len.p, tlen.data(), 1024, cudaMemcpyHostToDevice, st));
        CUDA_TRY(ctx, cudaMemcpyAsync(B.tok_key.p, tk.data(), 2048, cudaMemcpyHostToDevice, st));
        CUDA_TRY(ctx, cudaMemcpyAsync(B.tok_bytes.p, tb.data(), 256, cudaMemcpyHostToDevice, st));
        for (int i = 0; i < MG_CTR_WORDS; i++) host[i] = 0;
        host[4] = 256;
        CUDA_TRY(ctx, cudaMemcpyAsync(B.ctr.p, host, MG_CTR_WORDS * 8, cudaMemcpyHostToDevice, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
    }
    M.csr_off = (const u32 *)B.csr_off.p; M.csr_rec = (const Rec *)B.csr_rec.p;
    M.log = (Rec *)B.log.p; M.log_rng = (u64 *)B.log_rng.p; M.log_cap = log_cap;
    {
        u64 bk_cap = log_cap / 32 + (u64)(SORT_MAX_BK + 1) * 64 + 1024;
        // (test knob: a smaller pool of bucket offsets runs out within the run, and the later slices stay unsorted)
        if (const char *e = getenv("BPE_MERGE_SORTPOOL")) bk_cap = std::min<u64>(bk_cap, std::max<u64>(1, strtoull(e, nullptr, 10)));
        BPE_TRY(alloc_exact(ctx, B.log2, log_cap * sizeof(Rec))); BPE_TRY(alloc_exact(ctx, B.bk_lg, ((u64)n_merges + 2) * 4));
        BPE_TRY(alloc_exact(ctx, B.bk_start, ((u64)n_merges + 2) * 8)); BPE_TRY(alloc_exact(ctx, B.bk_off, bk_cap * 4));
        BPE_TRY(alloc_exact(ctx, B.bk_scratch, (u64)4 * SORT_MAX_BK * 4));
        CUDA_TRY(ctx, cudaMemsetAsync(B.bk_lg.p, 0, ((u64)n_merges + 2) * 4, st));
        M.log2 = (Rec *)B.log2.p; M.bk_lg = (u32 *)B.bk_lg.p; M.bk_start = (u64 *)B.bk_start.p; M.bk_off = (u32 *)B.bk_off.p;
        M.bk_off_cap = bk_cap; M.bk_scratch = (u32 *)B.bk_scratch.p;
    }
    M.tok_off = (u32 *)B.tok_off.p; M.tok_len = (u32 *)B.tok_len.p; M.tok_key = (u64 *)B.tok_key.p; M.tok_bytes = (uint8_t *)B.tok_bytes.p;
    M.tok_bytes_cap = tok_bytes_cap; M.merge_cnt_out = (i64 *)B.merge_cnt.p;
    M.live_pairs = ctx->live_pairs; M.live_cap = ctx->live_cap;
    M.merges_out = (int32_t *)B.merges.p; M.n_merges = n_merges; M.ctr = (u64 *)B.ctr.p; M.prof = (u64 *)B.prof.p;
    M.step_prof = nullptr;
    M.min_rec = 1;                                   // measured at 11 GB, same box: 32 -> 433 ms, 8 -> 418, 2 -> 409, 1 -> 406
    if (const char *e = getenv("BPE_MERGE_MINREC")) M.min_rec = (u32)std::max(1, std::min(32, atoi(e)));
    M.sort_min = 65536;                              // one pass of the apply phase covers 148 x 16 x 32 = 75 776 records
    if (const char *e = getenv("BPE_MERGE_SORTMIN")) M.sort_min = (u32)std::max(64, atoi(e));
    M.max_batch = MG_BATCH;                          // merges per grid step, at most (1 = the strictly sequential loop)
    if (const char *e = getenv("BPE_MERGE_BATCH")) M.max_batch = (u32)std::max(1, std::min((int)MG_BATCH, atoi(e)));
    if (getenv("BPE_CTA_PROFILE")) { BPE_TRY(alloc_exact(ctx, B.cta_prof, (u64)n_merges * 160 * 32)); CUDA_TRY(ctx, cudaMemsetAsync(B.cta_prof.p, 0, (u64)n_merges * 160 * 32, st)); M.cta_prof = (u64 *)B.cta_prof.p; }
    if (getenv("BPE_STEP_PROFILE")) { BPE_TRY(alloc_exact(ctx, B.step_prof, ((u64)n_merges + 1) * 16)); CUDA_TRY(ctx, cudaMemsetAsync(B.step_prof.p, 0, ((u64)n_merges + 1) * 16, st)); M.step_prof = (u32 *)B.step_prof.p; }

    // initial pair table from the dense 256x256 counts (same device-side insert as the merge loop uses)
    CUDA_TRY(ctx, cudaMemcpyToSymbolAsync(cM, &M, sizeof(M), 0, cudaMemcpyHostToDevice, st));
    KLAUNCH(k_insert_initial_pairs, 256, 256, 0, st, (const u64 *)B.dense.p);
    CUDA_TRY(ctx, cudaGetLastError());
    int ev_build1 = tm.mark();

    {
        int per_sm = 0;
        CUDA_TRY(ctx, cudaFuncSetAttribute((void *)k_merge_loop, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MG_DYN_SMEM));
        CUDA_TRY(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_merge_loop, MG_NT, MG_DYN_SMEM));
        if (per_sm < 1) return bpe_set_error(ctx, BPE_ERR_CUDA, "merge kernel does not fit on an SM");
    }
    const u64 bar_bytes = (u64)MG_MAX_CTAS * sizeof(BarSlot) + 512;   // gather slots, two counters
    BPE_TRY(alloc_exact(ctx, B.bar, bar_bytes));
    M.bar = (BarSlot *)B.bar.p; M.bar_ctr = (u32 *)(M.bar + MG_MAX_CTAS);
    u64 ctr[MG_CTR_WORDS] = {0};
    static const bool verbose = getenv("BPE_MERGE_VERBOSE") != nullptr;
    M.stop_at = n_merges;
    for (int round = 0; n_merges > 0 && round < 64; round++) {
        CUDA_TRY(ctx, cudaMemcpyToSymbolAsync(cM, &M, sizeof(M), 0, cudaMemcpyHostToDevice, st));
        CUDA_TRY(ctx, cudaMemsetAsync(B.bk_scratch.p, 0, (u64)4 * SORT_MAX_BK * 4, st));
        CUDA_TRY(ctx, cudaMemsetAsync(B.bar.p, 0, bar_bytes, st));   // epochs restart at 0
        // grid: one CTA per SM for big tables, fewer for small ones (cheaper barriers).  Measured at 11 GB with the counter
        // barrier, same box: G = 148: 449 ms, 112: 464, 96: 463, 80: 481, 64: 485, 48: 535.  (With the per-CTA flag barrier
        // that this replaced, 64 CTAs were the optimum: polling 148 slots cost more than the extra apply threads gave.)
        // Since a step applies several merges the small-table optimum moved up: TinyStories shape (98 K words, 4 M slots), G = 41 (what
        // the size rule gives): 23.3 ms, 74: 19.5, 96: 19.4, 120: 19.9, 148: 20.5; 11 GB OWT shape: 148: 139.6, 120: 150.9, 96: 160.3.
        int G = std::max(2, (int)std::min<u64>((u64)std::min(ctx->sm_count, (int)MG_MAX_CTAS),
                                               std::max<u64>(96, std::max<u64>(pcap_natural, M.pcap / 16) / PB / 256 + 1 + (n_words + 4095) / 4096)));
        if (const char *e = getenv("BPE_MERGE_G")) G = std::max(2, std::min(atoi(e), std::min(ctx->sm_count, (int)MG_MAX_CTAS)));
        g_bpe_launches++;
        CUDA_TRY(ctx, cudaLaunchCooperativeKernel((void *)k_merge_loop, dim3(G), dim3(MG_NT), nullptr, MG_DYN_SMEM, st));
        CUDA_TRY(ctx, cudaMemcpyAsync(host, B.ctr.p, MG_CTR_WORDS * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
        for (int i = 0; i < MG_CTR_WORDS; i++) ctr[i] = host[i];
        if (ctr[3] != MG_NEED_GROW) break;                            // done, pair table ran empty (train.py:184-185), or error
        // grow x4: the new table holds the same keys with the same counts (k_pairs_rehash); the counters carry over, the pending
        // pops (the last step's winners) included, and the relaunch rescans every block
        DevBuf okey = B.pkey, ocnt = B.pcnt;
        u64 ocap = M.pcap;
        B.pkey = DevBuf(); B.pcnt = DevBuf();
        int rc = alloc_pair_table(ocap * 4);
        if (rc != BPE_OK) { bpe_buf_free(ctx, okey); bpe_buf_free(ctx, ocnt); return rc; }
        if (verbose) fprintf(stderr, "  [pair table: %llu -> %llu slots at merge %llu, %llu keys]\n", (unsigned long long)ocap,
                             (unsigned long long)M.pcap, (unsigned long long)ctr[1], (unsigned long long)ctr[2]);
        host[3] = 0;
        CUDA_TRY(ctx, cudaMemcpyAsync((u64 *)B.ctr.p + 3, host + 3, 8, cudaMemcpyHostToDevice, st));
        ctr[3] = 0;
        unsigned rg = (unsigned)std::min<u64>((u64)ctx->sm_count * bpe_grid_mult(64), (ocap + 255) / 256);
        CUDA_TRY(ctx, cudaMemcpyToSymbolAsync(cM, &M, sizeof(M), 0, cudaMemcpyHostToDevice, st));
        KLAUNCH(k_pairs_rehash, rg, 256, 0, st, (const u64 *)okey.p, (const i64 *)ocnt.p, ocap);
        CUDA_TRY(ctx, cudaGetLastError());
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
        bpe_buf_free(ctx, okey); bpe_buf_free(ctx, ocnt);
    }
    int ev_merge1 = tm.mark();
    CUDA_TRY(ctx, cudaMemcpyAsync(g_merge_prof, B.prof.p, 256, cudaMemcpyDeviceToHost, st));
    if (M.cta_prof) {
        std::vector<u64> cp((size_t)n_merges * 160 * 4);
        CUDA_TRY(ctx, cudaMemcpyAsync(cp.data(), B.cta_prof.p, cp.size() * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
        if (FILE *f = fopen(getenv("BPE_CTA_PROFILE"), "wb")) { fwrite(cp.data(), 8, cp.size(), f); fclose(f); }
    }
    if (M.step_prof) {
        std::vector<u32> sp((size_t)n_merges * 4);
        CUDA_TRY(ctx, cudaMemcpyAsync(sp.data(), B.step_prof.p, sp.size() * 4, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
        if (FILE *f = fopen(getenv("BPE_STEP_PROFILE"), "wb")) { fwrite(sp.data(), 4, sp.size(), f); fclose(f); }
    }
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    if (ctr[3]) return bpe_set_error(ctx, BPE_ERR_CAPACITY, "merge loop table overflow (code %llu)", (unsigned long long)ctr[3]);
    int done = (int)ctr[1];
    if (done > 0) CUDA_TRY(ctx, cudaMemcpyAsync(merge_pairs_out, B.merges.p, (size_t)done * 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    *n_done = done;
    // SURVEY A-6: the reference identifies tokens by their byte string.  A merge with a positive count whose product bytes
    // already exist cannot occur (DESIGN.md section 8); the count is kept as an invariant check and the host raises on it.
    u64 dup_tokens = 0;
    if (done > 0) {
        std::vector<i64> mc(done);
        CUDA_TRY(ctx, cudaMemcpyAsync(mc.data(), B.merge_cnt.p, (size_t)done * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
        if (const char *dump = getenv("BPE_DUMP_MERGES")) {        // debug aid: (a, b, count) of every merge, for offline analysis
            if (FILE *f = fopen(dump, "wb")) {
                for (int k = 0; k < done; k++) { i64 rec[3] = {merge_pairs_out[2 * k], merge_pairs_out[2 * k + 1], mc[k]}; fwrite(rec, 8, 3, f); }
                fclose(f);
            }
        }
        std::vector<std::string> sym(256);
        std::unordered_set<std::string> seen;
        for (int i = 0; i < 256; i++) { sym[i] = std::string(1, (char)i); seen.insert(sym[i]); }
        for (int k = 0; k < done; k++) {
            std::string t = sym[merge_pairs_out[2 * k]] + sym[merge_pairs_out[2 * k + 1]];
            if (!seen.insert(t).second && mc[k] > 0) dup_tokens++;
            sym.push_back(std::move(t));
        }
    }
    int ev_end = tm.mark();
    if (stats) {
        stats->n_unique = n_words; stats->n_symbols = n_syms; stats->n_pairs_initial = n_pairs0;
        stats->n_pairs_final = ctr[2]; stats->log_records = ctr[0]; stats->duplicate_tokens = dup_tokens;
        stats->n_pretokens = cs->n_pretokens; stats->sum_live_pairs = ctr[7]; stats->merge_steps = ctr[12];
        stats->ms_build = tm.ms(ev_build0, ev_build1); stats->ms_merge = tm.ms(ev_build1, ev_merge1);
        stats->ms_total = tm.ms(ev_start, ev_end);
    }
    return BPE_OK;
}

static int train_impl(bpe_ctx *ctx, const uint8_t *text, u64 n, bool text_is_device, const uint8_t *sp_blob, const u32 *sp_offs,
                      int n_sp, int n_merges, int32_t *merge_pairs_out, int *n_done, bpe_train_stats *stats, const SplitSpecials *split = nullptr) {
    if (!ctx || (!text && n) || !n_done || (n_merges > 0 && !merge_pairs_out) || (n_sp > 0 && (!sp_blob || !sp_offs))) return BPE_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    *n_done = 0;
    if (stats) memset(stats, 0, sizeof(*stats));
    if (n_merges < 0) n_merges = 0;
    EvTimer tm(ctx);
    int e0 = tm.mark();
    BPE_TRY(ctx_load_text(ctx, text, n, text_is_device));
    int e1 = tm.mark();
    u64 nn = n;
    const u32 *spstart;
    BPE_TRY(run_flags_for_training(ctx, &nn, true, split, &spstart));
    int e2 = tm.mark();
    BPE_TRY(bpe_count_begin(ctx));
    BPE_TRY(count_current_text(ctx, nn, 0, nn, nn, spstart));
    int e3 = tm.mark();
    int rc = run_merges(ctx, sp_blob, sp_offs, n_sp, n_merges, merge_pairs_out, n_done, stats, tm, e0);
    if (stats) {
        stats->n_bytes = nn;
        stats->ms_h2d = tm.ms(e0, e1); stats->ms_pretok = tm.ms(e1, e2); stats->ms_count = tm.ms(e2, e3);
    }
    ctx->count->active = false;
    return rc;
}

// Host entry point for big inputs: the text is uploaded in chunks (each with a small halo, exactly like a rank's shard in
// the multi-GPU path) on a copy stream while the previous chunk is pretokenised and counted.  Returns 1 when the input
// needs the one-piece path instead (a carriage return: newline translation shifts offsets; or a pretoken longer than the halo).
#define TRAIN_PIPE_MIN (96ull << 20)
#define TRAIN_PIPE_CHUNK (256ull << 20)
#define TRAIN_HALO_LEFT 64ull
#define TRAIN_HALO_RIGHT (64ull << 10)
static u64 align_cut_host(const uint8_t *t, u64 n, u64 pos) {       // largest position <= pos that does not split a UTF-8 sequence
    if (pos >= n) return n;
    for (int k = 0; k < 3 && pos > 0 && (t[pos] & 0xC0u) == 0x80u; k++) pos--;
    return pos;
}
// Split mode (split != null): special-token resolution at a cut can depend on context further left than any fixed halo (chains of
// overlapping candidates), so the chunks are cut only at exact boundaries (exact_cut_host, as the encoder's pipeline) and each one is
// counted as a whole text.  A nominal cut with no exact boundary within TRAIN_CUT_WINDOW after it is skipped: that chunk grows.
#define TRAIN_CUT_WINDOW (8ull << 20)
static int count_host_pipelined(bpe_ctx *ctx, const uint8_t *text, u64 n, bpe_train_stats *stats, float *ms_pretok, float *ms_count,
                                const SplitSpecials *split = nullptr) {
    BPE_TRY(ctx_pipeline_init(ctx));
    cudaStream_t st = ctx->stream;
    std::vector<u64> cut{0};
    for (u64 p = TRAIN_PIPE_CHUNK; p + TRAIN_PIPE_CHUNK / 2 < n; p += TRAIN_PIPE_CHUNK) {
        if (!split) { cut.push_back(align_cut_host(text, n, p)); continue; }
        const u64 c = exact_cut_host(text, n, p, TRAIN_CUT_WINDOW, split->blob.data(), split->offs.data(), split->n());
        if (c) cut.push_back(c);
    }
    cut.push_back(n);
    const size_t m = cut.size() - 1;
    auto range = [&](size_t k, u64 *rlo, u64 *rhi) {
        if (split) { *rlo = cut[k]; *rhi = cut[k + 1]; return; }
        *rlo = align_cut_host(text, n, cut[k] > TRAIN_HALO_LEFT ? cut[k] - TRAIN_HALO_LEFT : 0);
        *rhi = align_cut_host(text, n, std::min(n, cut[k + 1] + TRAIN_HALO_RIGHT));
    };
    u64 max_len = 0;
    for (size_t k = 0; k < m; k++) { u64 a, b; range(k, &a, &b); max_len = std::max(max_len, b - a); }
    DevBuf *tbuf[2] = {&ctx->text, &ctx->text_alt};
    auto upload = [&](size_t k, DevBuf &dst) -> int {
        u64 a, b; range(k, &a, &b);
        BPE_TRY(ctx_prepare_arena(ctx, dst, max_len, ctx->s_in));
        if (b - a < max_len) CUDA_TRY(ctx, cudaMemsetAsync((uint8_t *)dst.p + BPE_PAD + (b - a), BPE_BYTE_PAD, max_len - (b - a), ctx->s_in));
        CUDA_TRY(ctx, cudaMemcpyAsync((uint8_t *)dst.p + BPE_PAD, text + a, b - a, cudaMemcpyHostToDevice, ctx->s_in));
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_in[k & 1], ctx->s_in));
        return BPE_OK;
    };
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    BPE_TRY(upload(0, *tbuf[0]));
    int rc = BPE_OK;
    for (size_t k = 0; k < m && rc == BPE_OK; k++) {
        const int cur = (int)(k & 1);
        u64 a, b; range(k, &a, &b);
        if (k + 1 < m) { rc = upload(k + 1, *tbuf[cur ^ 1]); if (rc != BPE_OK) break; }
        if (cur == 1) std::swap(ctx->text, ctx->text_alt);
        CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_in[cur], 0));
        EvTimer tm(ctx, 8);
        int e0 = tm.mark();
        u64 nn = b - a;
        const u32 *spstart;
        rc = run_flags_for_training(ctx, &nn, false, split, &spstart, cut[k] - a, cut[k + 1] - a);
        int e1 = tm.mark();
        if (rc == BPE_OK && ctx->saw_cr) rc = 1;
        if (rc == BPE_OK) {
            rc = count_current_text(ctx, b - a, cut[k] - a, cut[k + 1] - a, b == n || split ? b - a : (b - a >= 16 ? b - a - 16 : 0), spstart);
            if (rc == BPE_ERR_HALO) rc = 1;
        }
        int e2 = tm.mark();
        if (rc == BPE_OK) rc = count_rehome(ctx);
        if (rc == BPE_OK) { *ms_pretok += tm.ms(e0, e1); *ms_count += tm.ms(e1, e2); }
        if (cur == 1) std::swap(ctx->text, ctx->text_alt);
        if (rc == BPE_ERR_UTF8) ctx->err_detail += (int64_t)a;
    }
    cudaStreamSynchronize(ctx->s_in);
    (void)stats;
    return rc;
}

static int train_host(bpe_ctx *ctx, const uint8_t *text_host, uint64_t n, const uint8_t *specials_blob, const uint32_t *special_offs,
                      int n_specials, int n_merges, int32_t *merge_pairs_out, int *n_done, bpe_train_stats *stats, const SplitSpecials *split) {
    if (n >= TRAIN_PIPE_MIN && ctx && text_host && n_done && (n_merges <= 0 || merge_pairs_out) && (n_specials <= 0 || (specials_blob && special_offs))) {
        CUDA_TRY(ctx, cudaSetDevice(ctx->device));
        *n_done = 0;
        if (stats) memset(stats, 0, sizeof(*stats));
        if (n_merges < 0) n_merges = 0;
        EvTimer tm(ctx);
        int e0 = tm.mark();
        BPE_TRY(bpe_count_begin(ctx));
        float ms_pretok = 0, ms_count = 0;
        int rc = count_host_pipelined(ctx, text_host, n, stats, &ms_pretok, &ms_count, split);
        if (rc == BPE_OK) {
            rc = run_merges(ctx, specials_blob, special_offs, n_specials, n_merges, merge_pairs_out, n_done, stats, tm, e0);
            if (stats) { stats->n_bytes = n; stats->ms_h2d = 0; stats->ms_pretok = ms_pretok; stats->ms_count = ms_count; }
            ctx->count->active = false;
            return rc;
        }
        ctx->count->active = false;
        if (rc != 1) return rc;                   // (1 = needs the one-piece path below)
    }
    return train_impl(ctx, text_host, n, false, specials_blob, special_offs, n_specials, n_merges, merge_pairs_out, n_done, stats, split);
}
BPE_API int bpe_train(bpe_ctx *ctx, const uint8_t *text_host, uint64_t n, const uint8_t *specials_blob,
                      const uint32_t *special_offs, int n_specials, int n_merges, int32_t *merge_pairs_out, int *n_done,
                      bpe_train_stats *stats) {
    return train_host(ctx, text_host, n, specials_blob, special_offs, n_specials, n_merges, merge_pairs_out, n_done, stats, nullptr);
}
BPE_API int bpe_train_dev(bpe_ctx *ctx, const uint8_t *text_dev, uint64_t n, const uint8_t *specials_blob,
                          const uint32_t *special_offs, int n_specials, int n_merges, int32_t *merge_pairs_out, int *n_done,
                          bpe_train_stats *stats) {
    return train_impl(ctx, text_dev, n, true, specials_blob, special_offs, n_specials, n_merges, merge_pairs_out, n_done, stats);
}
BPE_API int bpe_train_ex(bpe_ctx *ctx, const uint8_t *text_host, uint64_t n, const uint8_t *specials_blob,
                         const uint32_t *special_offs, int n_specials, int n_merges, int32_t *merge_pairs_out, int *n_done,
                         bpe_train_stats *stats, int flags) {
    SplitSpecials sp; const SplitSpecials *split;
    BPE_TRY(split_from_flags(ctx, flags, specials_blob, special_offs, n_specials, sp, &split));
    return train_host(ctx, text_host, n, specials_blob, special_offs, n_specials, n_merges, merge_pairs_out, n_done, stats, split);
}
BPE_API int bpe_train_dev_ex(bpe_ctx *ctx, const uint8_t *text_dev, uint64_t n, const uint8_t *specials_blob,
                             const uint32_t *special_offs, int n_specials, int n_merges, int32_t *merge_pairs_out, int *n_done,
                             bpe_train_stats *stats, int flags) {
    SplitSpecials sp; const SplitSpecials *split;
    BPE_TRY(split_from_flags(ctx, flags, specials_blob, special_offs, n_specials, sp, &split));
    return train_impl(ctx, text_dev, n, true, specials_blob, special_offs, n_specials, n_merges, merge_pairs_out, n_done, stats, split);
}
BPE_API int bpe_train_from_counts(bpe_ctx *ctx, const uint8_t *specials_blob, const uint32_t *special_offs, int n_specials,
                                  int n_merges, int32_t *merge_pairs_out, int *n_done, bpe_train_stats *stats) {
    if (!ctx || !ctx->count || !n_done || (n_merges > 0 && !merge_pairs_out)) return BPE_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    *n_done = 0;
    if (stats) memset(stats, 0, sizeof(*stats));
    if (n_merges < 0) n_merges = 0;
    EvTimer tm(ctx);
    int e0 = tm.mark();
    int rc = run_merges(ctx, specials_blob, special_offs, n_specials, n_merges, merge_pairs_out, n_done, stats, tm, e0);
    ctx->count->active = false;
    return rc;
}
