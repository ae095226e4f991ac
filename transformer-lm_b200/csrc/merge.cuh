// merge.cuh -- the BPE merge loop as one persistent cooperative kernel that applies SEVERAL merges per grid step.
//
// Reference: the loop at models/tokenizer/train.py:183-228:
//     best = max(byte_pair_frequencies, key=lambda x: (byte_pair_frequencies[x], x))        187-189
//     for every word indexed under best: left-to-right rewrite + 4 count updates             192-224
//     pop best from both dicts, merges.append(best)                                          226-228
//
// Device data structures
//   pair table   open addressing, key = a<<32|b, 64-bit count.  A key lives from its first touch
//                (defaultdict semantics: counts may be 0) until it is merged (count = CNT_DEAD).
//   argmax       every PB slots form a block with a cached maximum and an upper bound of its second-largest count; an
//                update marks its block dirty, so a step rescans only the blocks that changed.  The cached values of the
//                blocks a CTA owns live in its shared memory for the whole launch (written through for the next one).
//   tie-break    (count, (bytes_a, bytes_b)) with python's bytes ordering.  Each token keeps its
//                first 8 bytes as a big-endian integer (tok_key): comparing the integers decides
//                almost every tie; equal prefixes fall back to lengths / a byte loop.
//   words        symbols never move: a merge writes the new token over its left operand and a tombstone over the
//                right one, so an occurrence is addressed by the position of its left symbol for ever.
//   token_indices  one record (neighbour, position, word count) per pair OCCURRENCE.  Pairs of two initial bytes:
//                CSR built once; any other pair (p,q): every occurrence is created in the step that created the
//                younger of p,q, so it is found in that step's slice of an append-only log (bucket-sorted by
//                neighbour when large).  Stale records are harmless (the symbols are re-checked, like the
//                reference re-checks its stale index entries, train.py:196-200).  One warp per occurrence in most
//                steps: no per-word serialisation, no divergence between sites.
//
// Several merges per step (the loop is latency-bound: two grid barriers and ~10 dependent memory round trips per step, whatever
// the step does).  Every CTA reports its best TWO pairs and a bound H on the count of everything else it owns; every CTA then
// derives the same sorted candidate list d1 >= d2 >= ... and applies the longest prefix d1..dr (r <= MG_BATCH) with
//   (1) for i < j: the second token of dj is not the first token of di, and the first token of dj is not the second token of di
//       (dj is neither of the form (x, a_i) nor (b_i, y)); no a == b unless r == 1,
//   (2) count(dr) > count(d(r+1)) and count(dr) > H.
// Why this is exactly the reference's next r merges: merge i only decrements pairs (x, a_i) and (b_i, y) and creates pairs that
// contain its new token.  By (1) no dj is decremented by an earlier merge of the step and no occurrence of dj shares a symbol with
// an occurrence of di (the merges may share tokens otherwise: (a,b) and (a,c) do not interact).  A new pair (x, new_i) is counted
// at most count(x, a_i) times, and (x, a_i) is not a later dj by (1), cannot occur after an earlier dj = (x, a_i) took all its
// occurrences, and otherwise has, by (2), a count below count(dr): so every pair created or changed during the step stays strictly
// below count(dr), the reference's max() picks d1, .., dr in this order, and the pair it picks next is again the maximum of the
// table after the step.
// Adjacent sites of different merges of a step are resolved as the reference's sequence would: a site of merge j sees the
// occurrences of merges i < j already merged and those of merges i > j untouched (apply_site).
#pragma once
#include <cooperative_groups.h>
#include <cooperative_groups/scan.h>
#include "common.cuh"

namespace cg = cooperative_groups;

// slot hash of the pair table: 32-bit multiplies only (the apply path computes four of these per site)
__device__ __forceinline__ u32 pair_hash(u64 key) {
    u32 h = ((u32)(key >> 32) * 0x9E3779B1u) ^ ((u32)key * 0x85EBCA77u);
    h ^= h >> 16; h *= 0x7FEB352Du; h ^= h >> 15;
    return h;
}

#define PAIR_EMPTY 0xFFFFFFFFFFFFFFFFull
#define CNT_DEAD ((i64)0x8000000000000000ll)     // key was popped from the dict (train.py:226)
#define CNT_DEAD_LIMIT ((i64)0xC000000000000000ll) // counts below this are "popped (+ later deltas)"
#define PB 64u                                   // pair-table slots per block (one rescan = two slots per lane)
#define MG_NT 512
#define MG_NEED_GROW 8ull                        // ctr[3] code: pair table more than half full, host must grow it
#ifndef MG_BATCH
#ifndef MG_BATCH
#define MG_BATCH 15u                             // merges per step, at most (<= 30).  Measured at 11 GB with the relaxed rule: 15 -> 143 ms, 20 -> 150, 24 -> 155, 30 -> 164 (fewer steps, but every extra merge of a step costs ~1.5 us of rescans and apply work)
#endif
#endif

struct __align__(16) WordMeta {
    u32 off, len;        // word w occupies sym[off, off+len) at build time
    i64 cnt;             // word frequency
};
// Symbol array: every word is preceded by one SYM_SEP; the array starts and ends with SYM_PAD separators, so the
// neighbour scans of apply_site never need a bounds check.  Values: >= 0 live symbol, SYM_SEP word boundary,
// <= -2 tombstone written by merge step (-v - 2).
#define SYM_SEP (-1)
#define SYM_PAD 32u
struct Words {
    int32_t *sym;
    WordMeta *meta;
    u64 *counters;       // [0]=n_words [1]=sym slots used (symbols + one separator per word) [2]=max_len
};
// index record: one pair occurrence.  x = neighbour token (bit 31: the neighbour is on the right), pos = position of
// the occurrence's left symbol, cnt = frequency of the word it lies in
struct __align__(16) Rec { u32 x, pos; i64 cnt; };
__device__ __forceinline__ Rec load_rec(const Rec *p) {
    uint4 v = *reinterpret_cast<const uint4 *>(p);
    Rec r; r.x = v.x; r.pos = v.y; r.cnt = (i64)(((u64)v.w << 32) | v.z); return r;
}
__device__ __forceinline__ void store_rec(Rec *p, u32 x, u32 pos, i64 cnt) {
    *reinterpret_cast<uint4 *>(p) = make_uint4(x, pos, (u32)cnt, (u32)((u64)cnt >> 32));
}

// candidate of the argmax: count, pair key, and the 8-byte prefix keys of both tokens (so that almost every
// tie is broken in registers, without dependent loads)
struct __align__(32) Best { i64 cnt; u64 key; u64 ka; u64 kb; };
#define BEST_NONE Best{CNT_DEAD, PAIR_EMPTY, 0, 0}
// whole-struct 2 x 128-bit accesses (otherwise the compiler loads .cnt first and the rest behind a branch:
// two dependent round trips instead of one)
__device__ __forceinline__ Best load_best(const Best *p) {
    const uint4 *q = reinterpret_cast<const uint4 *>(p);
    uint4 lo = q[0], hi = q[1];
    Best b;
    b.cnt = (i64)(((u64)lo.y << 32) | lo.x); b.key = ((u64)lo.w << 32) | lo.z;
    b.ka = ((u64)hi.y << 32) | hi.x; b.kb = ((u64)hi.w << 32) | hi.z;
    return b;
}
__device__ __forceinline__ void store_best(Best *p, const Best &b) {
    uint4 *q = reinterpret_cast<uint4 *>(p);
    q[0] = make_uint4((u32)b.cnt, (u32)((u64)b.cnt >> 32), (u32)b.key, (u32)(b.key >> 32));
    q[1] = make_uint4((u32)b.ka, (u32)(b.ka >> 32), (u32)b.kb, (u32)(b.kb >> 32));
}
// Upper bound of the second-largest count of a block as 32 bits: 0 = "no second key" (a real bound of 0 means the same to
// the batching rule, which needs count > bound), saturated = "unknown, assume huge".
#define SEC_SAT 0xFFFFFFFFu
__device__ __forceinline__ u32 sec_pack(i64 c) { return c <= 0 ? 0u : (c >= (i64)SEC_SAT ? SEC_SAT : (u32)c); }
__device__ __forceinline__ i64 sec_unpack(u32 s) { return s == SEC_SAT ? (i64)0x7FFFFFFFFFFFFFFFll : (i64)s; }

struct MergeState {
    Words W; u32 n_words;
    u64 *pkey; i64 *pcnt; u64 pcap;
    Best *bmax; u32 *bsec; uint8_t *dirty; u32 n_blocks;
    const u32 *csr_off; const Rec *csr_rec;
    // log_rng[2t], [2t+1] = slice of the log written by the STEP that contained merge t (all merges of a step share it)
    Rec *log; u64 *log_rng; u64 log_cap;
    // big log slices are bucket-sorted by hash(neighbour) into log2 right after the step that wrote them:
    // bk_lg[t] = log2(buckets) (0 = slice left unsorted), bk_start[t] = first of its buckets+1 offsets in bk_off
    Rec *log2; u32 *bk_lg; u64 *bk_start; u32 *bk_off; u64 bk_off_cap; u32 *bk_scratch;   // bk_scratch: 2 x (hist, cursor) x SORT_MAX_BK
    u32 *tok_off; u32 *tok_len; u64 *tok_key; uint8_t *tok_bytes; u64 tok_bytes_cap;
    struct BarSlot *bar; u32 *bar_ctr;            // gather slots / the two barrier counters (128 B apart) of k_merge_loop, zeroed before every launch
    int stop_at;                                 // this launch runs merges [ctr[1], stop_at)
    u32 max_batch;                               // merges per step, <= MG_BATCH (BPE_MERGE_BATCH)
    int32_t *merges_out; i64 *merge_cnt_out; int n_merges;
    int32_t *live_pairs; int live_cap;           // page-locked HOST memory (or null): the merges as they are made, for the host to follow (bpe_train_set_live)
    // [0]=log cursor [1]=n_done (next merge) [2]=pair keys created [3]=status flags [4]=tok bytes cursor
    // [5]=keys popped [6]=number of keys still to be popped (the last step's winners, in [16..16+MG_BATCH))
    // [7]=sum over merges of the live pair-table keys (the reference's max() scans that many dict entries, train.py:187-189;
    //     merges of one step are all charged [2] - [5] at the start of the step)
    // [8]=words rewritten (all steps) [9]=bk_off pool cursor [10]=slices sorted
    // [12]=grid steps taken
    u64 *ctr;
    // profile (ns / counts): [0]=phase1 [1]=sync1 [2]=apply [3]=sync2 on CTA 0; [4]=token CTA work; [5]=index records scanned;
    // [6]=words rewritten; [7]=steps; [9]=dirty blocks rescanned
    u64 *prof;
    u32 sort_min;     // log slices with fewer records are left unsorted and scanned whole (BPE_MERGE_SORTMIN)
    u32 min_rec;      // smallest number of records dealt to a warp per pass of the apply phase (BPE_MERGE_MINREC)
    u64 *cta_prof;    // optional (profile builds): per step and CTA {start, arrive1, exit1, arrive2}
    u32 *step_prof;   // optional per-step trace: 4 x u32 per step (phase1+sync1 ns, apply+sync2 ns, records scanned, words rewritten so far)
};
#define MG_CTR_WORDS 64
#define MG_CTR_PENDING 16                        // .. 16 + MG_BATCH <= 64

// The loop state lives in constant memory: helpers are real (non-inlined) functions so that the persistent
// kernel stays small enough for the instruction caches -- every step runs each code path only once, so a
// large inlined kernel is instruction-fetch bound.
__constant__ MergeState cM;

#ifdef BPE_MERGE_PROFILE
__device__ __forceinline__ u64 gtime_ns() { u64 t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define PROF_ADD(i, v) atomicAdd(&cM.prof[i], (u64)(v))
#else
__device__ __forceinline__ u64 gtime_ns() { return 0; }
#define PROF_ADD(i, v) do { } while (0)
#endif

__device__ __forceinline__ int bytes_cmp_dev(const uint8_t *x, u32 nx, const uint8_t *y, u32 ny) {
    u32 m = nx < ny ? nx : ny;
    for (u32 i = 0; i < m; i++) { if (x[i] != y[i]) return x[i] < y[i] ? -1 : 1; }
    return nx < ny ? -1 : (nx > ny ? 1 : 0);
}
// python: bytes(p) > bytes(q) for two tokens whose 8-byte prefix keys are equal (rare slow path)
__device__ __noinline__ bool tok_greater_slow(u32 p, u32 q) {
    PROF_ADD(8, 1);
    u32 lp = cM.tok_len[p], lq = cM.tok_len[q];
    if (lp <= 8 && lq <= 8) return lp > lq;      // equal zero-padded prefixes: the shorter one is a prefix of the longer
    return bytes_cmp_dev(cM.tok_bytes + cM.tok_off[p], lp, cM.tok_bytes + cM.tok_off[q], lq) > 0;
}
// Tie-break of two candidates with equal counts: python's ((bytes_a, bytes_b)) tuple order.
__device__ __forceinline__ bool best_tie_greater(u64 xkey, u64 xka, u64 xkb, u64 ykey, u64 yka, u64 ykb) {
    u32 xa = (u32)(xkey >> 32), ya = (u32)(ykey >> 32);
    if (xa != ya) return xka != yka ? xka > yka : tok_greater_slow(xa, ya);
    u32 xb = (u32)xkey, yb = (u32)ykey;
    if (xb == yb) return false;
    return xkb != ykb ? xkb > ykb : tok_greater_slow(xb, yb);
}
// (count, (bytes_a, bytes_b)) ordering of train.py:187-189
// (a real function: the persistent kernel is instruction-fetch bound -- every step walks through most of its code once, far more
// than the 32 KB instruction cache of an SM holds -- so the comparison exists once, not once per call site)
__device__ __noinline__ bool best_tie_greater_ni(u64 xkey, u64 xka, u64 xkb, u64 ykey, u64 yka, u64 ykb) { return best_tie_greater(xkey, xka, xkb, ykey, yka, ykb); }
__device__ __forceinline__ bool best_greater(const Best &x, const Best &y) {
    if (x.cnt != y.cnt) return x.cnt > y.cnt;
    if (x.cnt == CNT_DEAD) return false;
    return best_tie_greater_ni(x.key, x.ka, x.kb, y.key, y.ka, y.kb);
}
// butterfly reduction with the full comparison (handles every tie): the slow path of warp_best
__device__ __noinline__ Best warp_best_butterfly(Best b) {
#pragma unroll 1
    for (int d = 16; d; d >>= 1) {
        Best o;
        o.cnt = __shfl_xor_sync(0xffffffffu, b.cnt, d);
        o.key = __shfl_xor_sync(0xffffffffu, b.key, d);
        o.ka = __shfl_xor_sync(0xffffffffu, b.ka, d);
        o.kb = __shfl_xor_sync(0xffffffffu, b.kb, d);
        if (best_greater(o, b)) b = o;
    }
    return b;
}
// warp-wide maximum of v over the lanes in `active` (0 elsewhere), two redux.sync steps
__device__ __forceinline__ u64 warp_max_u64(u64 v, bool active) {
    const u32 hi = active ? (u32)(v >> 32) : 0u;
    const u32 mh = __reduce_max_sync(0xffffffffu, hi);
    const u32 lo = (active && hi == mh) ? (u32)v : 0u;
    const u32 ml = __reduce_max_sync(0xffffffffu, lo);
    return ((u64)mh << 32) | ml;
}
// warp-wide maximum of signed counts (CNT_DEAD = "nothing")
__device__ __forceinline__ i64 warp_max_cnt(i64 c) { return (i64)(warp_max_u64((u64)c ^ 0x8000000000000000ull, true) ^ 0x8000000000000000ull); }
// Warp arg-max under the (count, (bytes_a, bytes_b)) order; every lane returns the winner.  The common cases -- a
// unique maximal count, or ties decided by the 8-byte prefix keys -- take a few redux / ballot steps instead of a
// five-round butterfly of 256-bit shuffles; anything subtler (equal prefixes of different tokens) falls back to it.
__device__ __noinline__ Best warp_best(Best b) {
    // counts: CNT_DEAD (most negative) marks "no candidate"; bias to unsigned order
    const u64 bc = (u64)b.cnt ^ 0x8000000000000000ull;
    const u64 mc = warp_max_u64(bc, true);
    if (mc == 0) return BEST_NONE;               // every lane is empty
    u32 t = __ballot_sync(0xffffffffu, bc == mc);
    if (t & (t - 1)) {                           // tie on the count: first tokens by prefix key
        const bool in1 = (t >> lane_id()) & 1u;
        const u64 ma = warp_max_u64(b.ka, in1);
        const u32 t2 = __ballot_sync(0xffffffffu, in1 && b.ka == ma);
        if (t2 & (t2 - 1)) {
            const bool in2 = (t2 >> lane_id()) & 1u;
            const u32 a0 = __shfl_sync(0xffffffffu, (u32)(b.key >> 32), __ffs(t2) - 1);
            if (__ballot_sync(0xffffffffu, in2 && (u32)(b.key >> 32) != a0)) return warp_best_butterfly(b);   // equal prefix, different tokens
            const u64 mb = warp_max_u64(b.kb, in2);
            const u32 t3 = __ballot_sync(0xffffffffu, in2 && b.kb == mb);
            if (t3 & (t3 - 1)) {
                const u32 b0 = __shfl_sync(0xffffffffu, (u32)b.key, __ffs(t3) - 1);
                const bool in3 = (t3 >> lane_id()) & 1u;
                if (__ballot_sync(0xffffffffu, in3 && (u32)b.key != b0)) return warp_best_butterfly(b);
            }
            t = t3;
        } else t = t2;
    }
    const int src = __ffs(t) - 1;
    Best r;
    r.cnt = __shfl_sync(0xffffffffu, b.cnt, src); r.key = __shfl_sync(0xffffffffu, b.key, src);
    r.ka = __shfl_sync(0xffffffffu, b.ka, src); r.kb = __shfl_sync(0xffffffffu, b.kb, src);
    return r;
}

// The two largest candidates a thread / warp / CTA has seen, and an upper bound h of the counts of everything else it has seen.
struct Top2 { Best m1, m2; i64 h; };
__device__ __forceinline__ Top2 top2_none() { Top2 t; t.m1 = BEST_NONE; t.m2 = BEST_NONE; t.h = CNT_DEAD; return t; }
__device__ __forceinline__ void top2_add(Top2 &t, const Best &e) {
    if (e.cnt == CNT_DEAD) return;
    if (e.cnt < t.m2.cnt) { if (e.cnt > t.h) t.h = e.cnt; return; }
    if (best_greater(e, t.m1)) { if (t.m2.cnt > t.h) t.h = t.m2.cnt; t.m2 = t.m1; t.m1 = e; }
    else if (best_greater(e, t.m2)) { if (t.m2.cnt > t.h) t.h = t.m2.cnt; t.m2 = e; }
    else if (e.cnt > t.h) t.h = e.cnt;
}
// Reduce the lanes' Top2 to the warp's (returned in every lane).
__device__ __forceinline__ Top2 warp_top2(Top2 t) {
    Top2 r;
    r.m1 = warp_best(t.m1);
    if (r.m1.cnt != CNT_DEAD && t.m1.key == r.m1.key) { t.m1 = t.m2; t.m2 = BEST_NONE; }
    r.m2 = warp_best(t.m1);
    if (r.m2.cnt != CNT_DEAD && t.m1.key == r.m2.key) { t.m1 = t.m2; t.m2 = BEST_NONE; }
    i64 h = t.h;
    if (t.m1.cnt > h) h = t.m1.cnt;              // (m2 <= m1 in every lane, and CNT_DEAD is the smallest value)
    r.h = warp_max_cnt(h);
    return r;
}

// The merges of the current step, identical in every CTA (shared memory).
struct __align__(16) Batch {
    u64 key[MG_BATCH]; i64 cnt[MG_BATCH];
    u64 lo[MG_BATCH], pre[MG_BATCH + 1];         // index range of merge j: src[j][lo[j] .. lo[j] + pre[j+1] - pre[j])
    const Rec *src[MG_BATCH];
    u32 a[MG_BATCH], b[MG_BATCH], want[MG_BATCH]; // want: neighbour the records are filtered by (0xFFFFFFFF: no filter, CSR slice)
    u32 r;
};
#define WANT_ANY 0xFFFFFFFFu

// A pair-table slot changed: its block must be rescanned before the next arg-max.
__device__ __forceinline__ void mark_dirty(u64 slot) { cM.dirty[(u32)(slot / PB)] = 1; }

// frequencies[key] += delta with defaultdict semantics (train.py:36,65-78): a missing key is created.
// The count update is a fire-and-forget reduction; a popped key that is touched again is repaired by
// the next rescan of its block (see rescan_block).  (s, k) = first probe slot and the key read there.
__device__ __noinline__ void pair_add_from(u64 key, i64 delta, u64 s, u64 k) {
    const u64 mask = cM.pcap - 1;
    for (u64 probes = 0; probes < cM.pcap; probes++) {
        if (k == PAIR_EMPTY) k = atomicCAS(&cM.pkey[s], PAIR_EMPTY, key);
        if (k == PAIR_EMPTY) { atomicAdd(&cM.ctr[2], 1ull); k = key; }       // our CAS claimed the slot
        if (k == key) {
            atomicAdd((u64 *)&cM.pcnt[s], (u64)delta);
            mark_dirty(s);
            return;
        }
        s = (s + 1) & mask;
        k = cM.pkey[s];
    }
    cM.ctr[3] = 1;                                // table full
}
__device__ __forceinline__ void pair_add(u32 a, u32 b, i64 delta) {
    u64 key = ((u64)a << 32) | b;
    u64 s = pair_hash(key) & (cM.pcap - 1);
    pair_add_from(key, delta, s, cM.pkey[s]);
}

// Apply merge j of the step, (a,b) -> nw = nw0 + j, at the occurrence whose left symbol sits at position p (word frequency c):
// one merge site of the left-to-right scan of train.py:196-224 with update_frequencies_after_merge (52-78), merge_subwords
// (132-139) and create_new_token_indices (107-129).
//
// All sites of a step run concurrently, so every thread reasons about the state AT THE START OF THE STEP, which it can always
// reconstruct: a symbol equal to nw0 + i was a_i, the tombstone of merge i of this step was b_i.  The reference's sequential
// semantics in those terms:
//   * a record is a site iff its symbols are (a,b) and -- for a == b (only in steps of one merge), inside a run of a's -- it
//     sits at an even offset from the start of the run (non-overlapping, left to right: aaaa -> [aa, aa], aaa -> [aa, a]);
//   * the left neighbour is the already merged token when the occurrence directly to the left is a site of merge i <= j
//     (abab: the second site sees (nw, a), decrements it and creates (nw, nw)); when it is a site of a merge i > j, or no site,
//     it is the plain symbol;
//   * the right neighbour is the merged token when the occurrence directly to the right is a site of a merge i < j, and the
//     unmerged symbol otherwise (the same merge's scan has not reached it yet, a later merge has not happened yet);
//   * both new pairs are indexed, even if the right one is merged away later in the same step (stale, harmless).
__device__ __noinline__ void apply_site(u32 p, i64 c, u32 j, int step0, u32 nw0, const Batch *B) {
    int32_t *s = cM.W.sym;
    const int32_t ia = (int32_t)B->a[j], ib = (int32_t)B->b[j], inw = (int32_t)(nw0 + j);
    const int32_t tomb_hi = -(step0 + 2);                                     // tombstones of this step: tomb_hi - i for merge i
    const int32_t dead_now = tomb_hi - (int32_t)j;
#define ORIG(e) ((e) >= (int32_t)nw0 ? (int32_t)B->a[(e) - (int32_t)nw0] : ((e) <= tomb_hi ? (int32_t)B->b[tomb_hi - (e)] : (e)))   /* value at the start of the step */
#define WAS_LIVE(e) ((e) >= 0 || (e) <= tomb_hi)                            /* live at the start of the step */
#define OLD_TOMB(e) ((e) < SYM_SEP && (e) > tomb_hi)                         /* tombstone of an earlier step */
    // the four symbols around p are loaded together (one round trip in the common case of no old tombstones)
    int32_t vl = s[p - 1];
    const int32_t e0 = s[p];
    int32_t vb = s[p + 1], vr = s[p + 2];
    if (!WAS_LIVE(e0) || ORIG(e0) != ia) return;                           // stale record
    u32 pb = p + 1;
    while (OLD_TOMB(vb)) { pb++; vb = s[pb]; }
    if (!WAS_LIVE(vb) || ORIG(vb) != ib) return;                           // stale record
    // ---- left context ----
    bool has_l = false; u32 left = 0, pos_l = 0;
    u32 q = p - 1;
    while (OLD_TOMB(vl)) { q--; vl = s[q]; }
    if (ia == ib) {
        // run of a's ending just before p: its length decides whether p starts a site
        u32 n_left = 0, second = p;                                        // position of the second nearest a on the left
        while (WAS_LIVE(vl) && ORIG(vl) == ia) {
            n_left++;
            if (n_left == 2) second = q;
            q--; vl = s[q];
            while (OLD_TOMB(vl)) { q--; vl = s[q]; }
        }
        if (n_left & 1u) return;                                           // the a at p is the right half of the previous site
        if (n_left) { has_l = true; left = (u32)inw; pos_l = second; }
        else if (vl != SYM_SEP) { has_l = true; left = (u32)ORIG(vl); pos_l = q; }
    } else if (vl != SYM_SEP) {
        const int32_t o1 = ORIG(vl);
        has_l = true; left = (u32)o1; pos_l = q;
        // (.., a_i, b_i, [a, b]): when the occurrence on the left is a site of a merge i <= j it is merged before this one
        // (several merges of the step may have the same second token: the symbol further left decides which one it is)
        bool looked = false; u32 q2 = q - 1; int32_t o2 = SYM_SEP;
        for (u32 i = 0; i <= j; i++) {
            if ((int32_t)B->b[i] != o1) continue;
            if (!looked) {
                int32_t v2 = s[q2];
                while (OLD_TOMB(v2)) { q2--; v2 = s[q2]; }
                o2 = WAS_LIVE(v2) ? ORIG(v2) : SYM_SEP;
                looked = true;
            }
            if (o2 == (int32_t)B->a[i]) { left = nw0 + i; pos_l = q2; break; }
        }
    }
    // ---- right context: the symbol as it was, unless it starts a site of an EARLIER merge of this step ----
    u32 qr = pb + 1;
    if (pb != p + 1) vr = s[qr];
    while (OLD_TOMB(vr)) { qr++; vr = s[qr]; }
    const bool has_r = vr != SYM_SEP;
    u32 right = has_r ? (u32)ORIG(vr) : 0;
    if (has_r) {
        bool looked = false; int32_t o3 = SYM_SEP;
        for (u32 i = 0; i < j; i++) {
            if (B->a[i] != right) continue;
            if (!looked) {
                u32 q3 = qr + 1;
                int32_t v3 = s[q3];
                while (OLD_TOMB(v3)) { q3++; v3 = s[q3]; }
                o3 = WAS_LIVE(v3) ? ORIG(v3) : SYM_SEP;
                looked = true;
            }
            if (o3 == (int32_t)B->b[i]) { right = nw0 + i; break; }
        }
    }
    const u32 a = (u32)ia, b = (u32)ib, nw = (u32)inw;
    // ---- the four dict updates of update_frequencies_after_merge.  (left, nw) and (nw, right) contain the token made in
    // this step, so they are not in the table unless another site of this step put them there: their first probe is the
    // claiming CAS itself, issued together with the read probes of the two old keys and the log allocation ----
    const u64 mask = cM.pcap - 1;
    const u64 k0 = ((u64)left << 32) | a, k1 = ((u64)left << 32) | nw, k2 = ((u64)b << 32) | right, k3 = ((u64)nw << 32) | right;
    const u64 s0 = pair_hash(k0) & mask, s1 = pair_hash(k1) & mask, s2 = pair_hash(k2) & mask, s3 = pair_hash(k3) & mask;
    u64 v0 = 0, v1 = 0, v2 = 0, v3 = 0;
    if (has_l) { v0 = cM.pkey[s0]; v1 = atomicCAS(&cM.pkey[s1], PAIR_EMPTY, k1); }
    if (has_r) { v2 = cM.pkey[s2]; v3 = atomicCAS(&cM.pkey[s3], PAIR_EMPTY, k3); }
    // index records of the two new pairs: one atomic per group of threads that arrive here together
    const u32 n_rec = (u32)has_l + (u32)has_r;
    u64 li = 0;
    {
        const u32 act = __activemask();
        const u32 ml = __ballot_sync(act, has_l), mr = __ballot_sync(act, has_r);
        const u32 lt = (1u << lane_id()) - 1u;
        const u32 pre = __popc(ml & lt) + __popc(mr & lt), tot = __popc(ml) + __popc(mr);
        const int leader = __ffs(act) - 1;
        u64 base = 0;
        if ((int)lane_id() == leader && tot) base = atomicAdd(&cM.ctr[0], (u64)tot);
        li = __shfl_sync(act, base, leader) + pre;
    }
    const bool log_ok = li + n_rec <= cM.log_cap;
    if (!log_ok) cM.ctr[3] = 2;
    s[p] = inw; s[pb] = dead_now;                                          // merge_subwords: positions never move
    if (log_ok) {
        if (has_l) { store_rec(&cM.log[li], left, pos_l, c); li++; }        // (left, nw) at the position of `left`
        if (has_r) store_rec(&cM.log[li], 0x80000000u | right, p, c);       // (nw, right) at p
    }
    // The four probe sequences advance together: one loop whose trip count is the longest of the four (in the warp), with
    // the loads / CASes of an iteration in flight at the same time -- not four loops one after the other.
    // vj = what the probe of key j at slot sj returned; casj: that probe was a claiming CAS (PAIR_EMPTY = claimed by us).
    {
        u64 kk[4] = {k0, k1, k2, k3}, ss[4] = {s0, s1, s2, s3}, vv[4] = {v0, v1, v2, v3};
        const i64 dd[4] = {-c, c, -c, c};
        u32 cas = 0xAu;                                                    // keys 1 and 3 start with a claiming CAS
        u32 pend = (has_l ? 3u : 0u) | (has_r ? 12u : 0u);
        for (u64 probes = 0; pend && probes <= cM.pcap; probes++) {
#pragma unroll
            for (u32 t = 0; t < 4; t++) {
                if (!((pend >> t) & 1u)) continue;
                u64 k = vv[t];
                if (k == PAIR_EMPTY) {
                    if (!((cas >> t) & 1u)) {                              // empty slot seen by a read probe: claim it
                        vv[t] = atomicCAS(&cM.pkey[ss[t]], PAIR_EMPTY, kk[t]);
                        cas |= 1u << t;
                        continue;
                    }
                    atomicAdd(&cM.ctr[2], 1ull);                           // our CAS claimed the slot
                    k = kk[t];
                }
                if (k == kk[t]) {
                    atomicAdd((u64 *)&cM.pcnt[ss[t]], (u64)dd[t]);
                    mark_dirty(ss[t]);
                    pend &= ~(1u << t);
                    continue;
                }
                ss[t] = (ss[t] + 1) & mask;
                vv[t] = ((cas >> t) & 1u) ? atomicCAS(&cM.pkey[ss[t]], PAIR_EMPTY, kk[t]) : cM.pkey[ss[t]];
            }
        }
        if (pend) cM.ctr[3] = 1;                                           // table full
    }
    PROF_ADD(6, 1);
#undef ORIG
#undef WAS_LIVE
#undef OLD_TOMB
}

// Rescan the PB slots of one block with a full warp.  Pops the winners of the previous step (prev[0..n_prev)) when it meets
// them and repairs popped keys that were touched again (count = CNT_DEAD + deltas  ->  deltas).  Returns the block's maximum
// and, in sec, the bound of its second-largest count.
__device__ __noinline__ Best rescan_block(u32 blk, const u64 *prev, u32 n_prev, u32 &sec) {
    Best bst = BEST_NONE;
    i64 other = CNT_DEAD;                         // largest count this lane saw apart from bst
    const u64 sbase = (u64)blk * PB;
    u64 keys[PB / 32]; i64 cnts[PB / 32]; u64 kas[PB / 32], kbs[PB / 32];
#pragma unroll
    for (u32 k = 0; k < PB / 32; k++) { keys[k] = cM.pkey[sbase + k * 32 + lane_id()]; cnts[k] = cM.pcnt[sbase + k * 32 + lane_id()]; }
#pragma unroll
    for (u32 k = 0; k < PB / 32; k++) {          // second round trip: prefix keys of both tokens of every live slot
        bool live = keys[k] != PAIR_EMPTY;
        kas[k] = live ? cM.tok_key[(u32)(keys[k] >> 32)] : 0;
        kbs[k] = live ? cM.tok_key[(u32)keys[k]] : 0;
    }
#pragma unroll
    for (u32 k = 0; k < PB / 32; k++) {
        Best c;
        c.key = keys[k]; c.cnt = cnts[k]; c.ka = kas[k]; c.kb = kbs[k];
        if (c.key == PAIR_EMPTY) continue;
        bool popped = false;
        for (u32 i = 0; i < n_prev; i++) popped |= c.key == prev[i];
        if (popped) { cM.pcnt[sbase + k * 32 + lane_id()] = CNT_DEAD; continue; }
        if (c.cnt == CNT_DEAD) continue;
        if (c.cnt < CNT_DEAD_LIMIT) { c.cnt = (i64)((u64)c.cnt - (u64)CNT_DEAD); cM.pcnt[sbase + k * 32 + lane_id()] = c.cnt; }
        if (best_greater(c, bst)) { other = bst.cnt; bst = c; }
        else other = c.cnt > other ? c.cnt : other;
    }
    const Best w = warp_best(bst);
    const i64 rest = (w.cnt != CNT_DEAD && bst.key == w.key) ? other : (bst.cnt > other ? bst.cnt : other);
    sec = sec_pack(warp_max_cnt(rest));
    return w;
}

// source array of an index range: 0 = log, 1 = bucket-sorted copy, 2 = CSR of the initial byte pairs
#define T_SRC(code) ((code) == 2 ? cM.csr_rec : ((code) == 1 ? (const Rec *)cM.log2 : (const Rec *)cM.log))
#define SORT_MAX_LG 12u                          // at most 4096 buckets
#define SORT_MAX_BK (1u << SORT_MAX_LG)
__device__ __forceinline__ u32 bucket_of(u32 x, u32 lg) { return (x * 0x9E3779B1u) >> (32u - lg); }

// Index range of a pair (a,b) -- token_indices[best_pair] of train.py:192 -- is looked up in select_batch: pairs of two initial
// bytes in the CSR; any other pair in the log slice of the step that made its younger token, in the bucket of its other token
// when that slice was sorted.
// Bucket-sort the slice [lo, lo + n) of the log by hash(record.x) into log2 (same offsets) and publish the bucket
// offsets for the r merges [step0, step0 + r) that wrote it.  Called by every thread of every CTA between two steps; `sync` is
// the grid barrier.  s_scan: SORT_MAX_BK u32 of shared memory.  parity alternates so that the scratch of the previous sort can
// be cleared here.
// Both passes go through SHARED-MEMORY histograms: neighbour tokens are Zipfian, so a tenth of a slice's records can share one
// bucket, and one global atomic per record serialised on those few addresses (ncu: 31 % of all stall samples of the merge loop sat in
// this function).  Pass 1: every CTA counts its records (record i belongs to thread i mod gstride in both passes) per bucket in
// shared memory and reserves its part of every bucket with ONE global atomic per (CTA, non-empty bucket).  Pass 2: slot = bucket
// start + the CTA's part + a shared-memory cursor.  s_h / s_base: SORT_MAX_BK u32 of shared memory each.
template <typename SyncFn>
__device__ __forceinline__ void sort_slice(int step0, u32 r, u64 lo, u32 n, u32 parity, bool leader_cta, u64 gthread, u64 gstride,
                                           u32 *s_scan, u32 *s_wsum, u32 *s_h, u32 *s_base, SyncFn sync) {
    u32 lg = 4;
    while ((64u << lg) < n && lg < SORT_MAX_LG) lg++;
    const u32 nbk = 1u << lg;
    const u32 tid = threadIdx.x;
    u32 *hist = cM.bk_scratch + (size_t)parity * 2 * SORT_MAX_BK;
    u32 *other = cM.bk_scratch + (size_t)(parity ^ 1u) * 2 * SORT_MAX_BK;
    for (u32 i = tid; i < nbk; i += MG_NT) s_h[i] = 0;
    __syncthreads();
    {
        u64 i = gthread;
        for (; i + 3 * gstride < n; i += 4 * gstride) {              // four records in flight per thread
            const u32 x0 = cM.log[lo + i].x, x1 = cM.log[lo + i + gstride].x, x2 = cM.log[lo + i + 2 * gstride].x, x3 = cM.log[lo + i + 3 * gstride].x;
            atomicAdd(&s_h[bucket_of(x0, lg)], 1u); atomicAdd(&s_h[bucket_of(x1, lg)], 1u);
            atomicAdd(&s_h[bucket_of(x2, lg)], 1u); atomicAdd(&s_h[bucket_of(x3, lg)], 1u);
        }
        for (; i < n; i += gstride) atomicAdd(&s_h[bucket_of(cM.log[lo + i].x, lg)], 1u);
    }
    __syncthreads();
    for (u32 i = tid; i < nbk; i += MG_NT) { const u32 c = s_h[i]; s_base[i] = c ? atomicAdd(&hist[i], c) : 0u; s_h[i] = 0; }
    for (u64 i = gthread; i < 2 * SORT_MAX_BK; i += gstride) other[i] = 0;       // last used two barriers ago
    sync();
    // exclusive scan of the histogram, redundantly in every CTA
    const u32 per = (nbk + MG_NT - 1) / MG_NT;   // <= 8
    u32 v[8], sum = 0;
#pragma unroll
    for (u32 k = 0; k < 8; k++) { u32 i = tid * per + k; v[k] = (k < per && i < nbk) ? hist[i] : 0; sum += v[k]; }
    u32 inc = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { u32 t = __shfl_up_sync(0xffffffffu, inc, d); if (lane_id() >= (u32)d) inc += t; }
    if (lane_id() == 31) s_wsum[tid >> 5] = inc;
    __syncthreads();
    if (tid < 32) {
        u32 x = tid < MG_NT / 32 ? s_wsum[tid] : 0, xi = x;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { u32 t = __shfl_up_sync(0xffffffffu, xi, d); if (tid >= (u32)d) xi += t; }
        s_wsum[tid] = xi - x;
    }
    __syncthreads();
    u32 base = inc - sum + s_wsum[tid >> 5];
    u64 pool = 0;
    if (leader_cta) pool = cM.ctr[9];
#pragma unroll
    for (u32 k = 0; k < 8; k++) {
        u32 i = tid * per + k;
        if (k < per && i < nbk) { s_scan[i] = base; if (leader_cta) cM.bk_off[pool + i] = base; base += v[k]; }
    }
    if (leader_cta && tid == 0) {
        cM.bk_off[pool + nbk] = n; cM.ctr[9] = pool + nbk + 1; cM.ctr[10] += 1;
        for (u32 j = 0; j < r; j++) { cM.bk_start[step0 + j] = pool; cM.bk_lg[step0 + j] = lg; }
    }
    __syncthreads();
    {
        u64 i = gthread;
        for (; i + gstride < n; i += 2 * gstride) {                  // two records in flight per thread
            const uint4 r0 = *reinterpret_cast<const uint4 *>(&cM.log[lo + i]), r1 = *reinterpret_cast<const uint4 *>(&cM.log[lo + i + gstride]);
            const u32 b0 = bucket_of(r0.x, lg), b1 = bucket_of(r1.x, lg);
            *reinterpret_cast<uint4 *>(&cM.log2[lo + s_scan[b0] + s_base[b0] + atomicAdd(&s_h[b0], 1u)]) = r0;
            *reinterpret_cast<uint4 *>(&cM.log2[lo + s_scan[b1] + s_base[b1] + atomicAdd(&s_h[b1], 1u)]) = r1;
        }
        for (; i < n; i += gstride) {
            const uint4 rec = *reinterpret_cast<const uint4 *>(&cM.log[lo + i]);
            const u32 bk = bucket_of(rec.x, lg);
            *reinterpret_cast<uint4 *>(&cM.log2[lo + s_scan[bk] + s_base[bk] + atomicAdd(&s_h[bk], 1u)]) = rec;
        }
    }
    sync();
}

// ---- apply the merges of the step at every occurrence indexed under their pairs: the r index slices form one list of
// B->pre[r] records, spread over `gstride` threads ----
__device__ __forceinline__ bool fetch_rec(const Batch *B, u64 g, Rec &rec, u32 &j) {
    j = 0;
    while (g >= B->pre[j + 1]) j++;
    rec = load_rec(&B->src[j][B->lo[j] + (g - B->pre[j])]);
    return B->want[j] == WANT_ANY || rec.x == B->want[j];
}
__device__ __forceinline__ void apply_batch(int step0, u32 nw0, const Batch *B, u64 gthread, u64 gstride) {
    const u64 total = B->pre[B->r];
    if (gthread == 0) PROF_ADD(5, total);
    for (u64 g = gthread; g < total; g += 2 * gstride) {                  // 2 records in flight per thread
        Rec r0, r1; u32 j0, j1 = 0;
        const bool ok0 = fetch_rec(B, g, r0, j0);
        const bool h1 = g + gstride < total;
        const bool ok1 = h1 && fetch_rec(B, g + gstride, r1, j1);
        if (ok0) apply_site(r0.pos, r0.cnt, j0, step0, nw0, B);
        if (ok1) apply_site(r1.pos, r1.cnt, j1, step0, nw0, B);
    }
}

// ---- grid-wide synchronisation of k_merge_loop (all CTAs are co-resident: cooperative launch) ------------------------
// Counter barrier: every CTA adds 1 to one global counter with release semantics and ONE lane polls that word with acquire
// loads until it reaches (barriers so far) x (CTAs).  Measured against the alternatives at 11 GB (same box): per-CTA flags
// polled by a warp 514 ms (five acquire loads per lane per poll, 148 pollers), cooperative_groups::grid.sync 581 ms,
// fence + relaxed stores / polls 580 ms, this 481 ms.
//  * grid_barrier: the barrier alone.
//  * grid_gather:  barrier + all-gather of the per-CTA candidates: a CTA stores its two best pairs and its bound H in its slot
//    before it arrives; after the barrier warp 0 of every CTA loads all slots and derives the same batch of merges.
// Slot of a CTA: w[0..3] best pair, w[4..7] second best, w[8] bound of everything else.
struct __align__(128) BarSlot { u64 w[16]; };
#define MG_MAX_CTAS 160u
__device__ __forceinline__ u32 ld_acquire_u32(const u32 *p) { u32 v; asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }
__device__ __forceinline__ void red_release_add_u32(u32 *p, u32 v) { asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
// warp 0 only; the CTA barriers around it extend the ordering to the other warps
__device__ __forceinline__ void counter_arrive_wait(u32 *counter, u32 target) {
    if (threadIdx.x == 0) {
        red_release_add_u32(counter, 1u);
        while ((int)(ld_acquire_u32(counter) - target) < 0) { }
    }
    __syncwarp();
}
// Called by all threads of the CTA.
__device__ __forceinline__ void grid_barrier(u32 *counter, u32 G, u32 epoch, u64 *tp = nullptr) {
    __syncthreads();
#ifdef BPE_MERGE_PROFILE
    if (tp && threadIdx.x == 0) tp[0] = gtime_ns();
#endif
    if (threadIdx.x < 32) counter_arrive_wait(counter, epoch * G);
    __syncthreads();
}

// After the gather barrier: all CTAs' candidates (s_c[0 .. 2G): entry 2i is CTA i's best pair, 2i + 1 its second best) -> the
// merges of this step in *B (see the header of this file for the rule).  Two stages, both exact under the full
// (count, (bytes, bytes)) order:
//   rank_bests    (threads 0 .. 2G) the rank of every CTA's best pair among all CTAs' best pairs.  One of the MG_BATCH + 1
//                 greatest candidates overall is either a best pair of rank <= MG_BATCH or the second best of such a CTA, so
//                 those CTAs' pairs are copied to s_surv[2 * rank + {0, 1}] and nothing else matters.
//   select_batch  (warp 0) ranks the <= 2 (MG_BATCH + 1) survivors against each other, which yields d1 >= d2 >= ..., and applies
//                 the rule with one lane per candidate.
#define MG_SURV (2u * (MG_BATCH + 1u))
__device__ __noinline__ bool best_greater_ni(const Best *x, const Best *y) { return best_greater(*x, *y); }
// All warps of the CTA: warp w ranks the best pairs of CTAs [w * per, (w + 1) * per) against all G best pairs, which its lanes hold
// in registers (five per lane): a candidate costs five compares per lane and two warp reductions.  Pairs of equal count are
// compared in full only for candidates that can still be among the first MG_BATCH + 1.
__device__ __forceinline__ void rank_bests(const Best *s_c, const i64 *s_cnt, Best *s_surv, u32 G) {
    const u32 lane = lane_id(), warp = threadIdx.x >> 5;
    const u32 per = (G + MG_NT / 32 - 1) / (MG_NT / 32);
    i64 cj[MG_MAX_CTAS / 32];
#pragma unroll
    for (u32 m = 0; m < MG_MAX_CTAS / 32; m++) { const u32 j = lane + 32 * m; cj[m] = j < G ? s_cnt[2 * j] : CNT_DEAD; }
#pragma unroll 1
    for (u32 k = 0; k < per; k++) {
        const u32 i = warp * per + k;
        if (i >= G) break;
        const i64 ci = s_cnt[2 * i];
        if (ci == CNT_DEAD) continue;
        u32 gt = 0, eq = 0;
#pragma unroll
        for (u32 m = 0; m < MG_MAX_CTAS / 32; m++) { gt += cj[m] > ci; eq += cj[m] == ci; }
        gt = __reduce_add_sync(0xffffffffu, gt);
        eq = __reduce_add_sync(0xffffffffu, eq);   // (counts the pair itself)
        if (gt <= MG_BATCH && eq > 1) {
            u32 extra = 0;
#pragma unroll 1
            for (u32 m = 0; m < MG_MAX_CTAS / 32; m++) {
                const u32 j = lane + 32 * m;
                if (j < G && j != i && s_cnt[2 * j] == ci && best_greater_ni(&s_c[2 * j], &s_c[2 * i])) extra++;
            }
            gt += __reduce_add_sync(0xffffffffu, extra);
        }
        if (lane == 0 && gt <= MG_BATCH) { s_surv[2 * gt] = s_c[2 * i]; s_surv[2 * gt + 1] = s_c[2 * i + 1]; }
    }
}
// warp 0; H: bound of every pair that is not a candidate; max_r: upper limit of merges for this step
__device__ __noinline__ void select_batch(const Best *s_surv, Best *s_sorted, i64 H, Batch *B, u32 max_r) {
    const u32 lane = threadIdx.x;
    // rank of the survivors among themselves (a lane holds survivors lane and lane + 32): counts first, the (bytes, bytes)
    // comparison only on ties
    const Best e = lane < MG_SURV ? s_surv[lane] : BEST_NONE;
    const Best e2 = lane + 32 < MG_SURV ? s_surv[lane + 32] : BEST_NONE;
    u32 rank = 0, rank2 = 0;
#pragma unroll 1
    for (u32 m = 0; m < MG_SURV; m++) {
        const i64 cm = s_surv[m].cnt;
        if (cm > e.cnt) rank++;
        else if (cm == e.cnt && cm != CNT_DEAD && m != lane && best_greater_ni(&s_surv[m], &s_surv[lane])) rank++;
        if (MG_SURV > 32) {
            if (cm > e2.cnt) rank2++;
            else if (cm == e2.cnt && cm != CNT_DEAD && m != lane + 32 && best_greater_ni(&s_surv[m], &s_surv[lane + 32])) rank2++;
        }
    }
    if (lane <= MG_BATCH) s_sorted[lane] = BEST_NONE;
    __syncwarp();
    if (e.cnt != CNT_DEAD && rank <= MG_BATCH) s_sorted[rank] = e;
    if (MG_SURV > 32 && e2.cnt != CNT_DEAD && rank2 <= MG_BATCH) s_sorted[rank2] = e2;
    __syncwarp();
    const Best d = lane <= MG_BATCH ? s_sorted[lane] : BEST_NONE;           // lane t holds d(t+1)
    const u32 a = (u32)(d.key >> 32), b = (u32)d.key;
    // first half of the index-range lookup of every candidate, in flight while the rule is evaluated (winner_range, split)
    const u32 wT = a > b ? a : b;
    const bool have = d.cnt != CNT_DEAD, csr = wT < 256;
    u64 r_lo = 0, r_hi = 0, st0 = 0; u32 lg = 0;
    if (have) {
        if (csr) { const u32 pp = (a << 8) | b; r_lo = cM.csr_off[pp]; r_hi = cM.csr_off[pp + 1]; }
        else {
            const u32 t = wT - 256;
            const ulonglong2 rg = *reinterpret_cast<const ulonglong2 *>(&cM.log_rng[2 * (u64)t]);
            r_lo = rg.x; r_hi = rg.y; lg = cM.bk_lg[t]; st0 = cM.bk_start[t];
        }
    }
    const bool sq0 = __shfl_sync(0xffffffffu, a == b, 0);
    bool bad = !have || (lane > 0 && (a == b || sq0));                        // a == b goes alone
#pragma unroll 1
    for (u32 i = 0; i < MG_BATCH; i++) {
        const u32 ai = __shfl_sync(0xffffffffu, a, i), bi = __shfl_sync(0xffffffffu, b, i);
        if (i < lane) bad |= ai == b || bi == a;  // this pair is (x, a_i) or (b_i, y): merge i changes its count
    }
    const u32 first_bad = __ffs(__ballot_sync(0xffffffffu, bad || lane >= max_r)) - 1;   // d1 .. d(first_bad) do not interact
    const i64 next = __shfl_down_sync(0xffffffffu, d.cnt, 1);
    const bool strict = have && d.cnt > H && (next == CNT_DEAD || d.cnt > next);   // d1 .. d(lane+1) may go together
    const u32 ends = __ballot_sync(0xffffffffu, lane < first_bad && strict);
    u32 good = ends ? 32u - __clz(ends) : 0u;
    const bool any = __shfl_sync(0xffffffffu, have, 0);
    if (good == 0 && any && max_r > 0) good = 1;  // the maximum alone is always the reference's next merge
    // index ranges of the merges, one lane each
    u64 n = 0;
    if (lane < good) {
        const u32 want = b >= a ? a : (0x80000000u | b);
        u32 code = csr ? 2u : 0u;
        if (!csr && lg) {                         // bucket-sorted slice: the bucket of the neighbour
            const u64 st = st0 + bucket_of(want, lg);
            const u64 base = r_lo;
            r_lo = base + cM.bk_off[st]; r_hi = base + cM.bk_off[st + 1]; code = 1u;
        }
        B->a[lane] = a; B->b[lane] = b; B->key[lane] = d.key; B->cnt[lane] = d.cnt;
        B->lo[lane] = r_lo; B->src[lane] = T_SRC(code);
        B->want[lane] = csr ? WANT_ANY : want;
        n = r_hi - r_lo;
    }
    u64 inc = n;
#pragma unroll
    for (int k = 1; k < 32; k <<= 1) { const u64 t = __shfl_up_sync(0xffffffffu, inc, k); if (lane >= (u32)k) inc += t; }
    if (lane < good) B->pre[lane + 1] = inc;
    if (lane == 0) { B->pre[0] = 0; B->r = good; }
}

__device__ __forceinline__ uint4 ldcg_v4(const void *p) { return __ldcg(reinterpret_cast<const uint4 *>(p)); }
// Called by all threads of the CTA; `mine` (the CTA's two best pairs and its bound) is read from lane 0 of warp 0.
// s_c / s_cnt: 2 * MG_MAX_CTAS candidates, s_h: MG_NT / 32 words, s_surv: MG_SURV + MG_BATCH + 1 candidates.
__device__ __forceinline__ void grid_gather(BarSlot *slots, u32 *counter, u32 G, u32 epoch, const Top2 &mine, Best *s_c, i64 *s_cnt, i64 *s_h,
                                            Best *s_surv, Batch *B, u32 max_r, u64 *tp = nullptr) {
    __syncthreads();
#ifdef BPE_MERGE_PROFILE
    if (tp && threadIdx.x == 0) tp[0] = gtime_ns();
#endif
    if (threadIdx.x < 32) {
        if (threadIdx.x == 0) {
            u64 *w = slots[blockIdx.x].w;
            store_best(reinterpret_cast<Best *>(w), mine.m1);
            store_best(reinterpret_cast<Best *>(w + 4), mine.m2);
            w[8] = (u64)mine.h;
        }
        counter_arrive_wait(counter, epoch * G);
    }
    __syncthreads();
#ifdef BPE_MERGE_PROFILE
    const bool pt = tp && threadIdx.x == 0 && blockIdx.x == 0;
    u64 q0 = pt ? gtime_ns() : 0;
#endif
    // one candidate per thread: a single round trip for the whole gather
    const u32 tid = threadIdx.x;
    i64 h = CNT_DEAD;
    if (tid < 2 * G) {
        const u64 *w = slots[tid >> 1].w + 4 * (tid & 1u);
        const uint4 lo = ldcg_v4(w), hi = ldcg_v4(w + 2);
        if (!(tid & 1u)) h = (i64)__ldcg(slots[tid >> 1].w + 8);
        Best b;
        b.cnt = (i64)(((u64)lo.y << 32) | lo.x); b.key = ((u64)lo.w << 32) | lo.z;
        b.ka = ((u64)hi.y << 32) | hi.x; b.kb = ((u64)hi.w << 32) | hi.z;
        s_c[tid] = b; s_cnt[tid] = b.cnt;
    }
    if (tid >= MG_NT - MG_SURV) s_surv[tid - (MG_NT - MG_SURV)] = BEST_NONE;
    h = warp_max_cnt(h);
    if (lane_id() == 0) s_h[tid >> 5] = h;
    __syncthreads();
#ifdef BPE_MERGE_PROFILE
    u64 q1 = pt ? gtime_ns() : 0;
#endif
    rank_bests(s_c, s_cnt, s_surv, G);
    __syncthreads();
#ifdef BPE_MERGE_PROFILE
    u64 q2 = pt ? gtime_ns() : 0;
#endif
    if (tid < 32) {
        i64 hh = tid < MG_NT / 32 ? s_h[tid] : CNT_DEAD;
        hh = warp_max_cnt(hh);
        select_batch(s_surv, s_surv + MG_SURV, hh, B, max_r);
    }
    __syncthreads();
#ifdef BPE_MERGE_PROFILE
    if (tp && threadIdx.x == 0) tp[1] = gtime_ns();
    if (pt) { u64 q3 = gtime_ns(); cM.prof[10] += q0 - tp[0]; cM.prof[11] += q1 - q0; cM.prof[12] += q2 - q1; cM.prof[13] += q3 - q2; }
#endif
}

// ---- token bookkeeping: bytes and prefix keys of the new tokens, outputs (one CTA, all its threads; warp j = merge j) ------
// live: ctr[2] at the start of the step (the apply CTAs claim keys while this runs: reading ctr[2] here would depend on timing)
__device__ __forceinline__ void token_bookkeeping(int step0, u32 nw0, const Batch *B, u32 *s_off, u64 live) {
    const u32 tid = threadIdx.x, lane = lane_id(), warp = tid >> 5;
    const u32 r = B->r;
    if (warp == 0) {
        u32 ln = 0;
        if (lane < r) ln = cM.tok_len[B->a[lane]] + cM.tok_len[B->b[lane]];
        u32 inc = ln;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const u32 t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= (u32)d) inc += t; }
        if (lane < r) s_off[lane] = inc - ln;
        if (lane == r - 1) s_off[MG_BATCH] = inc;
    }
    const u64 cur = cM.ctr[4];
    __syncthreads();
    const u64 total = s_off[MG_BATCH];
    if (cur + total > cM.tok_bytes_cap) { if (tid == 0) cM.ctr[3] = 4; }
    else {
        for (u32 j = warp; j < r; j += MG_NT / 32) {
            const u32 a = B->a[j], b = B->b[j], nw = nw0 + j;
            const u32 la = cM.tok_len[a], lb = cM.tok_len[b], ln = la + lb;
            const u64 at = cur + s_off[j];
            uint8_t *dst = cM.tok_bytes + at;
            const uint8_t *pa = cM.tok_bytes + cM.tok_off[a], *pb = cM.tok_bytes + cM.tok_off[b];
            for (u32 i = lane; i < ln; i += 32) dst[i] = i < la ? pa[i] : pb[i - la];
            if (lane == 0) {
                // first 8 bytes of a+b from the operands' zero-padded big-endian prefix keys
                u64 nkey = cM.tok_key[a];
                if (la < 8) nkey |= cM.tok_key[b] >> (8 * la);
                cM.tok_off[nw] = (u32)at; cM.tok_len[nw] = ln; cM.tok_key[nw] = nkey;
                const int step = step0 + (int)j;
                cM.merges_out[2 * step] = (int32_t)a; cM.merges_out[2 * step + 1] = (int32_t)b;
                cM.merge_cnt_out[step] = B->cnt[j];
                // one posted 8-byte store per merge, no fence (a system-scope fence per step cost 2.5 us of a 24 us step): the host
                // pre-fills the buffer with -1 and takes an entry as complete when it is non-negative
                if (cM.live_pairs && step < cM.live_cap)
                    *reinterpret_cast<volatile long long *>(cM.live_pairs + 2 * step) = (long long)(((u64)b << 32) | a);
            }
            // make sure the winner's block is rescanned so the key gets popped
            if (lane == 1) {
                const u64 key = B->key[j], mask = cM.pcap - 1;
                u64 s = pair_hash(key) & mask;
                while (cM.pkey[s] != key) s = (s + 1) & mask;
                mark_dirty(s);
            }
        }
        if (tid == 0) {
            cM.ctr[4] = cur + total;
            cM.ctr[1] = (u64)(step0 + (int)r);
            const u64 popped = cM.ctr[5];
            cM.ctr[7] += (u64)r * (live - popped) - (u64)r * (r - 1) / 2; cM.ctr[5] = popped + r;
            cM.ctr[12] += 1;
        }
    }
}

// ---- shared-memory copy of the cached block maxima a CTA owns (structure of arrays: conflict-free 8-byte accesses) ----
#define MG_CACHE_ITERS 4u                        // chunks (of 64 blocks) per warp kept in shared memory; more are read from bmax
#define MG_CACHE_N (MG_CACHE_ITERS * (MG_NT / 32) * 64u)
#define MG_LIST_CAP 2048u                        // dirty blocks a CTA lists per step; the overflow is rescanned by the owning warp
#define MG_DYN_SMEM ((size_t)MG_CACHE_N * 36 + (size_t)MG_LIST_CAP * 4 + (size_t)SORT_MAX_BK * 8)    // cached block maxima, dirty list, the sort's two histograms
struct BmaxCache { i64 *cnt; u64 *key, *ka, *kb; u32 *sec; };
__device__ __forceinline__ BmaxCache bmax_cache(unsigned char *base) {
    BmaxCache c;
    c.cnt = reinterpret_cast<i64 *>(base); c.key = reinterpret_cast<u64 *>(base) + MG_CACHE_N;
    c.ka = c.key + MG_CACHE_N; c.kb = c.ka + MG_CACHE_N; c.sec = reinterpret_cast<u32 *>(c.kb + MG_CACHE_N);
    return c;
}
__device__ __forceinline__ void cache_store(const BmaxCache &c, u32 i, const Best &b, u32 sec) { c.cnt[i] = b.cnt; c.key[i] = b.key; c.ka[i] = b.ka; c.kb[i] = b.kb; c.sec[i] = sec; }
__device__ __forceinline__ void cache_consider(const BmaxCache &c, u32 i, Top2 &mine) {
    const i64 s2 = sec_unpack(c.sec[i]);
    if (s2 > mine.h) mine.h = s2;
    const i64 n = c.cnt[i];
    if (n == CNT_DEAD) return;
    if (n < mine.m2.cnt) { if (n > mine.h) mine.h = n; return; }
    Best o; o.cnt = n; o.key = c.key[i]; o.ka = c.ka[i]; o.kb = c.kb[i];
    top2_add(mine, o);
}

__global__ void __launch_bounds__(MG_NT) k_merge_loop() {
    __shared__ Best s_w1[MG_NT / 32], s_w2[MG_NT / 32];
    __shared__ i64 s_wh[MG_NT / 32];
    __shared__ Best s_c[2 * MG_MAX_CTAS];
    __shared__ i64 s_cnt[2 * MG_MAX_CTAS], s_h[MG_NT / 32];
    __shared__ Best s_surv[MG_SURV + MG_BATCH + 1];
    __shared__ Batch s_B;
    __shared__ u64 s_status[2];
    __shared__ u32 s_scan[SORT_MAX_BK];
    __shared__ u32 s_wsum[32];                   // (sort_slice writes all 32 entries)
    __shared__ u32 s_off[MG_BATCH + 1];
    __shared__ u32 s_nd;                         // dirty blocks listed in this step
    extern __shared__ __align__(16) unsigned char mg_smem[];
    const u32 tid = threadIdx.x, lane = lane_id(), warp = tid >> 5;
    const u32 G = gridDim.x;
    u32 n_sorts = 0;
    u32 epoch = 0, gepoch = 0;                   // barriers / gathers passed in this launch (the slots start at 0)
    const u32 warps_per_cta = MG_NT / 32;
    const u32 gwarp = blockIdx.x * warps_per_cta + warp, total_warps = G * warps_per_cta;
    const bool token_cta = blockIdx.x == G - 1;
    const u32 apply_ctas = G - 1;
    const int first_step = (int)cM.ctr[1];
    // winners of the previous step: popped lazily during the rescans of this step (they stay in s_B until the next gather)
    if (tid == 0) {
        const u32 np = (u32)cM.ctr[6];
        s_B.r = np <= MG_BATCH ? np : 0;
        for (u32 i = 0; i < s_B.r; i++) s_B.key[i] = cM.ctr[MG_CTR_PENDING + i];
        s_nd = 0;
    }
    if (tid < 2 * MG_MAX_CTAS) { s_c[tid] = BEST_NONE; s_cnt[tid] = CNT_DEAD; }
    // The cached block maxima of the chunks this CTA owns stay in shared memory for the whole launch (chunk (it, warp) =
    // 64 blocks starting at (it * total_warps + gwarp) * 64); bmax / bsec in global memory are written through for the next launch.
    const BmaxCache sc = bmax_cache(mg_smem);
    u32 *s_list = reinterpret_cast<u32 *>(mg_smem + (size_t)MG_CACHE_N * 36);
    u32 *s_sort_h = s_list + MG_LIST_CAP, *s_sort_base = s_sort_h + SORT_MAX_BK;
    const u32 n_iter = (cM.n_blocks + total_warps * 64 - 1) / (total_warps * 64);
    for (u32 it = 0; it < n_iter && it < MG_CACHE_ITERS; it++) {
        const u32 base = (it * total_warps + gwarp) * 64, i0 = (it * warps_per_cta + warp) * 64 + lane;
        const bool in0 = base + lane < cM.n_blocks, in1 = base + 32 + lane < cM.n_blocks;
        cache_store(sc, i0, in0 ? load_best(&cM.bmax[base + lane]) : BEST_NONE, in0 ? cM.bsec[base + lane] : 0u);
        cache_store(sc, i0 + 32, in1 ? load_best(&cM.bmax[base + 32 + lane]) : BEST_NONE, in1 ? cM.bsec[base + 32 + lane] : 0u);
    }
    __syncthreads();

    int step = first_step;
    while (step < cM.stop_at) {
        // status flags are written before the barrier that ends a step and read here (uniform across the grid); the loads
        // overlap with the dirty-flag loads of phase 1A and are checked behind its CTA barrier
        u64 st_err = 0, st_keys = 0;
        if (tid == 0) { st_err = *((volatile u64 *)&cM.ctr[3]); st_keys = *((volatile u64 *)&cM.ctr[2]); }
        // ---- phase 1: rescan dirty blocks, reduce cached block maxima to two candidates per CTA ----
        // log cursor at the start of the step (a slot of its own per step: a fast CTA 0 must not overwrite the value the
        // others still have to read after the barrier that ends the previous step)
        if (blockIdx.x == 0 && tid == 0) cM.log_rng[2 * (u64)step] = *((volatile u64 *)&cM.ctr[0]);
#ifdef BPE_MERGE_PROFILE
        const bool prof_thread = tid == 0 && (blockIdx.x == 0 || token_cta);
        u64 *ctp = cM.cta_prof ? cM.cta_prof + ((size_t)step * G + blockIdx.x) * 4 : nullptr;
        if (ctp && tid == 0) ctp[0] = gtime_ns();
#else
        const bool prof_thread = false;
        u64 *ctp = nullptr;
#endif
        u64 t0 = prof_thread ? gtime_ns() : 0;
        const u32 n_prev = s_B.r;
        const u64 *prev = s_B.key;
        // A: collect the dirty blocks of this CTA's chunks in a shared list (any warp of the CTA may rescan them)
        for (u32 it = 0; it < n_iter; it++) {
            const u32 base = (it * total_warps + gwarp) * 64;
            const u32 b0 = base + lane, b1 = base + 32 + lane;
            const bool d0 = b0 < cM.n_blocks && cM.dirty[b0], d1 = b1 < cM.n_blocks && cM.dirty[b1];
            const u32 dlo = __ballot_sync(0xffffffffu, d0), dhi = __ballot_sync(0xffffffffu, d1);
            if (dlo | dhi) {
                const u32 nlo = __popc(dlo), n = nlo + __popc(dhi);
                u32 pos = 0;
                if (lane == 0) pos = atomicAdd(&s_nd, n);
                pos = __shfl_sync(0xffffffffu, pos, 0);
                const u32 lt = (1u << lane) - 1u;
                const u32 e0 = pos + __popc(dlo & lt), e1 = pos + nlo + __popc(dhi & lt);
                if (d0 && e0 < MG_LIST_CAP) s_list[e0] = b0;
                if (d1 && e1 < MG_LIST_CAP) s_list[e1] = b1;
                if (pos + n > MG_LIST_CAP) {     // list full (huge tables, first step): this warp rescans the rest itself
                    u64 dm = (u64)__ballot_sync(0xffffffffu, d0 && e0 >= MG_LIST_CAP) | ((u64)__ballot_sync(0xffffffffu, d1 && e1 >= MG_LIST_CAP) << 32);
                    while (dm) {
                        const u32 l2 = __ffsll((long long)dm) - 1; dm &= dm - 1;
                        u32 sec;
                        const Best bst = rescan_block(base + l2, prev, n_prev, sec);
                        if (lane == 0) {
                            store_best(&cM.bmax[base + l2], bst); cM.bsec[base + l2] = sec; cM.dirty[base + l2] = 0;
                            if (it < MG_CACHE_ITERS) cache_store(sc, (it * warps_per_cta + warp) * 64 + l2, bst, sec);
                        }
                    }
                }
            }
        }
        if (tid == 0) { s_status[0] = st_err; s_status[1] = st_keys; }
        __syncthreads();
        if (s_status[0]) break;
        if (s_status[1] * 2 > cM.pcap) {         // table over half full: hand back to the host to grow it
            grid_barrier(cM.bar_ctr, G, ++epoch);
            if (blockIdx.x == 0 && tid == 0) cM.ctr[3] = MG_NEED_GROW;
            break;
        }
        // B: the CTA's warps share the rescans evenly
        {
            const u32 nd = s_nd < MG_LIST_CAP ? s_nd : MG_LIST_CAP;
            for (u32 e = warp; e < nd; e += warps_per_cta) {
                const u32 blk = s_list[e];
                u32 sec;
                const Best bst = rescan_block(blk, prev, n_prev, sec);
                if (lane == 0) {
                    store_best(&cM.bmax[blk], bst); cM.bsec[blk] = sec; cM.dirty[blk] = 0; PROF_ADD(9, 1);
                    const u32 chunk = blk >> 6, it = chunk / total_warps, w = chunk - it * total_warps - blockIdx.x * warps_per_cta;
                    if (it < MG_CACHE_ITERS) cache_store(sc, (it * warps_per_cta + w) * 64 + (blk & 63u), bst, sec);
                }
            }
        }
        __syncthreads();
        if (tid == 0) s_nd = 0;                  // (next written in phase A of the next step)
        // C: the two largest of the cached block maxima this warp owns (shared memory; global for chunks beyond the cache)
        Top2 mine = top2_none();
        for (u32 it = 0; it < n_iter; it++) {
            if (it < MG_CACHE_ITERS) {
                const u32 i0 = (it * warps_per_cta + warp) * 64 + lane;
                cache_consider(sc, i0, mine);
                cache_consider(sc, i0 + 32, mine);
            } else {
                const u32 base = (it * total_warps + gwarp) * 64;
                const u32 b0 = base + lane, b1 = base + 32 + lane;
                if (b0 < cM.n_blocks) { const i64 s2 = sec_unpack(cM.bsec[b0]); if (s2 > mine.h) mine.h = s2; top2_add(mine, load_best(&cM.bmax[b0])); }
                if (b1 < cM.n_blocks) { const i64 s2 = sec_unpack(cM.bsec[b1]); if (s2 > mine.h) mine.h = s2; top2_add(mine, load_best(&cM.bmax[b1])); }
            }
        }
        mine = warp_top2(mine);
        if (lane == 0) { s_w1[warp] = mine.m1; s_w2[warp] = mine.m2; s_wh[warp] = mine.h; }
        __syncthreads();
        Top2 cta = top2_none();
        if (warp == 0) {
            // 32 candidates, one per lane: the best of warp l in lane l, its second best in lane 16 + l
            Top2 t = top2_none();
            t.m1 = lane < warps_per_cta ? s_w1[lane] : s_w2[lane - warps_per_cta];
            t.h = lane < warps_per_cta ? s_wh[lane] : CNT_DEAD;
            cta = warp_top2(t);
        }
        u64 t1 = prof_thread ? gtime_ns() : 0;
        // ---- barrier + all-gather of the CTA candidates: every CTA derives the same merges for this step ----
        const u32 max_r = min(cM.max_batch, (u32)(cM.stop_at - step));
        grid_gather(cM.bar, cM.bar_ctr + 32, G, ++gepoch, cta, s_c, s_cnt, s_h, s_surv, &s_B, max_r, ctp ? ctp + 1 : nullptr);
        u64 t2 = prof_thread ? gtime_ns() : 0;
        const u32 r = s_B.r;
        if (r == 0) break;                       // len(byte_pair_frequencies) == 0 (train.py:184-185)
        const u32 nw0 = 256 + (u32)step;         // symbol ids of the new tokens: nw0 + j = a_j + b_j (train.py:190)
        const u64 n_rec = s_B.pre[r];
        // Every key this step can create contains one of its new tokens: (x, nw0 + j) or (nw0 + j, y) with x, y < nw0 + r, and a
        // site claims at most two of them.  When that bound could take the table past three quarters full, hand back to the host
        // before anything is applied (the check at the start of the step leaves only the keys already in the table as headroom,
        // and one step can claim more).  The winners of the previous step were popped in phase B, so none is left pending; the
        // relaunch derives this step's merges again.
        {
            const u64 bound = min(2 * n_rec, 2ull * r * (nw0 + r));
            if ((s_status[1] + bound) * 4 > cM.pcap * 3) {
                __syncthreads();
                if (tid == 0) { s_B.r = 0; if (blockIdx.x == 0) cM.ctr[3] = MG_NEED_GROW; }
                break;
            }
        }

        if (token_cta) token_bookkeeping(step, nw0, &s_B, s_off, s_status[1]);
        // Records are dealt to the warps of all apply CTAs R at a time, R as small as one pass over the slices allows (but not
        // below cM.min_rec): a step with a few hundred occurrences runs a few lanes on every SM instead of sixteen full warps on
        // one SM, with less divergence between the sites that share a warp.
        else {
            const u64 aw = (u64)apply_ctas * warps_per_cta;
            u32 R = 32;
            while (R > cM.min_rec && n_rec <= aw * (R >> 1)) R >>= 1;
            if (lane < R) apply_batch(step, nw0, &s_B, ((u64)warp * apply_ctas + blockIdx.x) * R + lane, aw * R);
        }
        u64 t3 = prof_thread ? gtime_ns() : 0;
        u64 tp2[2];
        grid_barrier(cM.bar_ctr, G, ++epoch, ctp ? tp2 : nullptr);
        if (ctp && tid == 0) ctp[3] = tp2[0];
        // the slice of the log this step wrote belongs to all its merges
        const u64 lb = *((volatile u64 *)&cM.log_rng[2 * (u64)step]), cur = *((volatile u64 *)&cM.ctr[0]);
        if (blockIdx.x == 0 && tid < r) { cM.log_rng[2 * (u64)(step + (int)tid)] = lb; cM.log_rng[2 * (u64)(step + (int)tid) + 1] = cur; }
        if (n_rec * 2 >= cM.sort_min) {          // heuristic: about two records per index entry visited
            const u64 pool = *((volatile u64 *)&cM.ctr[9]);
            if (cur - lb >= cM.sort_min && cur <= cM.log_cap && pool + SORT_MAX_BK + 1 <= cM.bk_off_cap) {
                sort_slice(step, r, lb, (u32)(cur - lb), n_sorts & 1u, blockIdx.x == 0, (u64)blockIdx.x * MG_NT + tid, (u64)G * MG_NT, s_scan, s_wsum,
                           s_sort_h, s_sort_base, [&]() { grid_barrier(cM.bar_ctr, G, ++epoch); });
                n_sorts++;
            }
        }
        if (prof_thread) {
            u64 t4 = gtime_ns();
            if (blockIdx.x == 0) {
                cM.prof[0] += t1 - t0; cM.prof[1] += t2 - t1; cM.prof[2] += t3 - t2; cM.prof[3] += t4 - t3; cM.prof[7] += 1;
                if (cM.step_prof) {
                    cM.step_prof[4 * step] = (u32)(t2 - t0); cM.step_prof[4 * step + 1] = (u32)(t4 - t2);
                    cM.step_prof[4 * step + 2] = (u32)cM.prof[5]; cM.step_prof[4 * step + 3] = r;
                }
            }
            if (token_cta) cM.prof[4] += t3 - t2;
        }
        step += (int)r;
    }
    // the winners of the last step are still to be popped: by the next launch, or dropped by the table rebuild
    __syncthreads();
    if (blockIdx.x == 0 && tid == 0) {
        cM.ctr[6] = s_B.r;
        for (u32 i = 0; i < s_B.r; i++) cM.ctr[MG_CTR_PENDING + i] = s_B.key[i];
    }
}

__global__ void __launch_bounds__(256) k_insert_initial_pairs(const u64 *__restrict__ dense) {
    u32 p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < 65536 && dense[p]) pair_add(p >> 8, p & 255u, (i64)dense[p]);
}

// Table growth: copy every key of the old table with its count as it is.  Popped keys stay as tombstones (CNT_DEAD, or CNT_DEAD
// plus later deltas, which the next rescan repairs) and the last step's winners stay pending (ctr[6]): the grown table holds
// exactly the keys of the old one, ctr[2] and ctr[5] keep their meaning, and the relaunch -- which rescans every block in its
// first step -- pops the pending winners like a launch on a table that never grew.
__global__ void __launch_bounds__(256) k_pairs_rehash(const u64 *__restrict__ okey, const i64 *__restrict__ ocnt, u64 ocap) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < ocap; i += (u64)gridDim.x * blockDim.x) {
        const u64 k = okey[i];
        if (k == PAIR_EMPTY) continue;
        const i64 c = ocnt[i];
        u64 mask = cM.pcap - 1, s = pair_hash(k) & mask;
        for (;;) {
            if (cM.pkey[s] == PAIR_EMPTY && atomicCAS(&cM.pkey[s], PAIR_EMPTY, k) == PAIR_EMPTY) { cM.pcnt[s] = c; break; }
            s = (s + 1) & mask;
        }
    }
}
