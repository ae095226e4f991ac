// encode.cu -- Tokenizer.encode / decode on the device.  Entry points: bpe_tok_*, bpe_encode*, bpe_decode.
//
// Reference being replaced: models/tokenizer/tokenizer.py:111-138 (encode), 63-90 (segment / pretokenize),
// 92-109 (merge), 155-157 (decode).
//
// Pipeline of one bpe_encode call (all stages on the context's stream), per batch of 256 MB of text:
//   1. special-token split + GPT-2 pretoken start flags            (pretok.cu, shared with training), pretoken ordinals per
//                     512-byte group
//   2. k_enc_lookup   straight from the text and its start bits: every pretoken occurrence gets its cached value -- from the
//                     CTA's shared-memory image of the most looked-up short pretokens, else from the dense L2-resident hot table,
//                     else from the tokenizer's device-resident pretoken -> token-ids cache (open addressing, exact keys: short,
//                     medium and long tables); unseen pretokens claim a slot there and are queued
//   3. k_enc_bpe_short / k_enc_bpe   the queued (new unique) pretokens: the merges in rank order through the pair -> rank table
//                     (repeatedly the lowest-ranked adjacent pair, all its non-overlapping occurrences left to right); one thread
//                     per pretoken of <= 32 bytes (row_bpe), one warp per longer one (warp_bpe)
//   (BPE-dropout only: k_enc_drop_starts, then k_enc_drop_short / k_enc_drop_warp -- row_bpe and
//                     warp_bpe with dropped candidates -- replace the value of every occurrence whose segmentation can change with its
//                     own BPE-dropout result, bypassing the cache)
//   4. k_enc_scan_emit  tokens per pretoken -> exclusive offsets -> ids scattered to the uint16 / int32 output, in one
//                     pass (single-pass scan with decoupled look-back)
// The reference re-runs BPE for every occurrence (no memoisation, tokenizer.py:118-136); the result per
// pretoken is a pure function of its bytes, so caching by exact bytes cannot change the output.
#include <algorithm>
#include "kernels.h"
#include "ctx.h"
#include "hashtab.cuh"
#include "scan.cuh"

#define REF_LONG 0x80000000u
#define REF_MED 0x40000000u
#define REF_SLOT(r) ((r) & 0x3FFFFFFFu)

// cached value of a pretoken (u64):
//   tag = v >> 60
//   0..3   that many ids inline, 20 bits each at bits 0, 20, 40
//   4      ids in the id pool: bits 59..24 = offset, bits 23..0 = count
//   5      KeyError: bits 31..0 = offending symbol (bit 31 set: index of a special token instead)
//   13     (per-occurrence array only, batch encode) document boundary: bits 39..0 = index of the document it ends, in the chunk
//   14     (per-occurrence array only) not computed when looked up: bits 31..0 = cache slot reference
//   15     not computed yet
#define VAL_NONE 0xFFFFFFFFFFFFFFFFull
#define VAL_FWD 14ull
#define VAL_TAG(v) ((u32)((v) >> 60))
#define VAL_EXT 4ull
#define VAL_ERR 5ull
#define VAL_DOC 13ull
#define VAL_DOC_MASK ((1ull << 40) - 1)
#define INLINE_ID_LIMIT (1u << 20)
#define RANK_NONE 0xFFFFFFFFFFFFFFFFull
#define MKEY_EMPTY 0xFFFFFFFFFFFFFFFFull

// the pretoken cache: the tables of hashtab.cuh, payload = the cached value (VAL_NONE in an empty slot).  Key and value share a slot,
// so a lookup brings the value in with the key (one 32-byte sector); pool = persistent key bytes of long pretokens.
struct EncTables : PtTables {
    const ulonglong2 *mtab; u64 mmask;           // pair -> {key = a<<32|b, (rank << 32) | result symbol}
    const int32_t *mpairs;                       // operand symbols of merge j
    const int32_t *sym_to_id;
    u32 *ipool;                                  // token ids of pretokens with more than 3 tokens
    u32 *todo;                                   // slots claimed in this batch (REF_LONG = long table)
    // hot table (see k_enc_hot_build): hot_nb buckets of two 16-byte keys (one sector), their cached values in hval; 0 = none
    const ulonglong2 *hot; const u64 *hval; u64 hot_nb;
    const ulonglong2 *sm_img;                    // LK_SM_SLOTS x {key, value}: image of the lookup kernel's shared-memory value cache (or null)
    u32 *scnt, *mcnt;                            // per-slot hit counters (short, medium) while the cache is being sampled for the hot table (else null)
    // [0]=n_short [1]=n_long [2]=todo count [3]=table overflow [4]=key pool cursor [5]=ipool cursor [6]=pretoken too long
    // [7]=smallest ordinal (in the text of the call) of a pretoken whose value is a KeyError  [8]=n_medium  [9]=step tickets of the lookup kernel
    u64 *ctr;
    // document boundaries of a batch encode (all null for bpe_encode): bit per arena byte, boundaries before every 512-byte group,
    // id_offs[j] = index of the first id after document j of the chunk (id_base + its offset in the chunk's output)
    const u32 *bmask; const u64 *bpre; u64 *id_offs; u64 id_base;
};

// ---- pair -> rank ---------------------------------------------------------------------------------
__device__ __forceinline__ u64 rank_lookup(const EncTables &t, u32 a, u32 b) {
    u64 key = ((u64)a << 32) | b;
    u64 s = mix64(key) & t.mmask;
    for (;;) {
        ulonglong2 e = __ldg(&t.mtab[s]);
        if (e.x == key) return e.y;
        if (e.x == MKEY_EMPTY) return RANK_NONE;
        s = (s + 1) & t.mmask;
    }
}

__global__ void __launch_bounds__(256) k_enc_build_ranks(ulonglong2 *__restrict__ mtab, u64 mmask, const int32_t *__restrict__ pairs,
                                                        const int32_t *__restrict__ result, int n_merges) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_merges) return;
    int32_t a = pairs[2 * j], b = pairs[2 * j + 1];
    if (a < 0 || b < 0) return;
    u64 key = ((u64)(u32)a << 32) | (u32)b;
    u64 s = mix64(key) & mmask;
    for (;;) {                                   // keys are distinct (the host drops superseded duplicates)
        u64 old = atomicCAS(&mtab[s].x, MKEY_EMPTY, key);
        if (old == MKEY_EMPTY) { mtab[s].y = ((u64)(u32)j << 32) | (u32)result[j]; return; }
        s = (s + 1) & mmask;
    }
}

// ---- pretoken cache: lookup or claim -----------------------------------------------------------------
// Returns the cached value of the pretoken, or (VAL_FWD << 60 | slot reference) when it is not computed yet (a value read early can
// only be "not computed yet", which yields a forward reference that is resolved after the BPE kernels: correct either way).  A claim
// counts the new key and queues its slot for the BPE kernels; a sampled lookup (scnt / mcnt set) bumps the slot's hit counter.
__device__ __forceinline__ u64 enc_short_get(const EncTables &t, u64 key) {
    return short_find_or_claim<true>(t, key, t.ctr,
        [&](u64 s) {
            atomicAdd(&t.ctr[0], 1ull);
            t.todo[atomicAdd(&t.ctr[2], 1ull)] = (u32)s;
            if (t.scnt) atomicAdd(&t.scnt[s], 1u);
            return (VAL_FWD << 60) | (u32)s;
        },
        [&](u64 s, u64 v) { if (t.scnt) atomicAdd(&t.scnt[s], 1u); return v != VAL_NONE ? v : ((VAL_FWD << 60) | (u32)s); });
}
__device__ __forceinline__ u64 enc_med_get(const EncTables &t, u64 k0, u64 k1) {
    return medium_find_or_claim<true>(t, k0, k1, t.ctr,
        [&](u64 s) {
            atomicAdd(&t.ctr[8], 1ull);
            t.todo[atomicAdd(&t.ctr[2], 1ull)] = (u32)s | REF_MED;
            if (t.mcnt) atomicAdd(&t.mcnt[s], 1u);
            return (VAL_FWD << 60) | (u32)s | REF_MED;
        },
        [&](u64 s, u64 v) { if (t.mcnt) atomicAdd(&t.mcnt[s], 1u); return v != VAL_NONE ? v : ((VAL_FWD << 60) | (u32)s | REF_MED); });
}
__device__ __forceinline__ u64 enc_long_get(const EncTables &t, const uint8_t *p, u32 len, u64 off_meta) {
    return long_find_or_claim<true>(t, p, len, off_meta, t.ctr,
        [&](u64 s) {
            atomicAdd(&t.ctr[1], 1ull);
            t.todo[atomicAdd(&t.ctr[2], 1ull)] = (u32)s | REF_LONG;
            return (VAL_FWD << 60) | (u32)s | REF_LONG;
        },
        [&](u64 s, u64 v) { return v != VAL_NONE ? v : ((VAL_FWD << 60) | (u32)s | REF_LONG); });
}

// ---- hot table ---------------------------------------------------------------------------------------------------------
// A probe into the cache tables is a random 32-byte sector with a 128-byte L2 line to itself (they are sized for the worst case and
// mostly empty): L2 keeps ~0.5 M such lines, and a lookup that misses it runs at the DRAM random-access rate (~40 G/s on B200,
// tools/bench_l2_random.cu) -- which is what bulk encoding ran at.  So the pretokens of <= 15 bytes that the first big batch after a
// cache reset looked up most often (per-slot hit counters, that batch only) are copied, with their values, into a dense table that
// stays in L2: a bucket is one sector holding two 16-byte keys (k0 = bytes 0-7, k1 = bytes 8-14 | len << 56; k1 = 0 and k0 = the
// short-table key for <= 7 bytes), the values sit in an array beside it.  A key whose bucket is full simply stays with the big
// tables, so a probe is exactly one sector.  Values are immutable once computed, so the copy never goes stale.

// ---- lookup: straight from the text and its start bits -------------------------------------------------------------------
// vals[ordinal of the pretoken in the batch] = its cached value when the cache has it, else a forward reference to its slot
// (resolved after the BPE kernels).  Same walk as the count stage of training (train.cu, k_count_pretokens): a lane owns one
// 16-byte chunk -- its 32-byte text window in registers, a 64-bit window of start bits -- and walks the chunk's start bits; a warp
// takes 32 consecutive chunks per step.  Three levels:
//   1. pretokens of <= 7 bytes: the CTA's shared-memory copy of the value cache image (the ~3 000 most looked-up short pretokens
//      of the sampled batch, read-only: LDS and compare, no global traffic) -- six lookups in ten end here;
//   2. what misses there and pretokens of 8..15 bytes go to the warp's queue and are drained in whole groups of 64 with all lanes:
//      one probe of the hot table (one sector, L2-resident), value from the array beside it;
//   3. what misses that, and pretokens of >= 16 bytes: the big tables (lookup or claim, enc_short_get / enc_long_get).
#define LK_NT 1024
#define LK_WARPS (LK_NT / 32u)
#ifndef LK_SM_LG
#define LK_SM_LG 12
#endif
#define LK_SM_SLOTS (1u << LK_SM_LG)
#ifndef LK_SM_FILL_NUM
#define LK_SM_FILL_NUM 6u                         // eighths of the image that may be filled
#endif
#ifndef LK_SM_PROBES
#define LK_SM_PROBES 2u
#endif
#ifndef LK_TICKET
#define LK_TICKET 8u                             // steps (of 512 bytes) per ticket
#endif
#define LK_QCAP 96u                              // entries of the warp's key queue
#define LK_QDRAIN 64u                            // drained when it reaches this (a round of the bit loop adds <= 32)
#define LK_QL_CAP 64u
#define LK_QL_DRAIN 32u
#define LK_WARP_SMEM (LK_QCAP * 24u + LK_QL_CAP * 12u)
#define LK_DYN_SMEM ((size_t)LK_SM_SLOTS * 16 + (size_t)LK_WARPS * LK_WARP_SMEM)
__device__ __forceinline__ u32 enc_sm_slot(u64 key) { return (((u32)key ^ (u32)(key >> 32)) * 0x9E3779B1u) >> (32 - LK_SM_LG); }

// queues of a warp: qe = keys (k0, k1; k1 = 0: a short pretoken, k0 its key) with qx = (ordinal, offset from base);
// ql = long pretokens (offset from base | len << 32) with qlo = ordinal
struct LookupQueues { ulonglong2 *qe; uint2 *qx; u64 *ql; u32 *qlo; u32 n, nl; };

__device__ __forceinline__ u64 enc_queued_get(const EncTables &t, ulonglong2 k, uint2 x, u64 base) {
    (void)x; (void)base;
    return k.y == 0 ? enc_short_get(t, k.x) : enc_med_get(t, k.x, k.y);
}
__device__ __forceinline__ void lookup_drain(const EncTables &t, LookupQueues &q, u64 base, u64 *__restrict__ vals, u32 lane, bool all) {
    const u32 dn = all ? q.n : q.n & ~63u;
    __syncwarp();
    for (u32 e0 = 0; e0 < dn; e0 += 64u) {
        const bool ha = e0 + lane < dn, hb = e0 + 32u + lane < dn;
        ulonglong2 ka = make_ulonglong2(0, 0), kb = ka;
        uint2 xa = make_uint2(0, 0), xb = xa;
        if (ha) { ka = q.qe[e0 + lane]; xa = q.qx[e0 + lane]; }
        if (hb) { kb = q.qe[e0 + 32u + lane]; xb = q.qx[e0 + 32u + lane]; }
        bool ta = ha, tb = hb;                   // still to be looked up in the big tables
        u64 va = 0, vb = 0;
        if (t.hot_nb) {
            const u64 ba = hot_bucket(t.hot_nb, ka.x, ka.y), bb = hot_bucket(t.hot_nb, kb.x, kb.y);
            const int ia = ha ? hot_find(t.hot, ba, ka.x, ka.y) : -1, ib = hb ? hot_find(t.hot, bb, kb.x, kb.y) : -1;
            if (ia >= 0) { va = __ldg(&t.hval[2 * ba + ia]); ta = false; }
            if (ib >= 0) { vb = __ldg(&t.hval[2 * bb + ib]); tb = false; }
        }
        if (ta) va = enc_queued_get(t, ka, xa, base);
        if (tb) vb = enc_queued_get(t, kb, xb, base);
        if (ha) __stcs(&vals[xa.x], va);         // (streaming stores: the value array is written once and read once -- it must not push the hot table out of L2)
        if (hb) __stcs(&vals[xb.x], vb);
    }
    for (u32 e = lane; e < q.nl; e += 32u) {
        const u64 ent = q.ql[e];
        const u64 pos = base + (u32)ent;
        __stcs(&vals[q.qlo[e]], enc_long_get(t, t.text + pos, (u32)(ent >> 32), pos));
    }
    q.nl = 0;
    // the remainder (< 64 keys) moves to the front
    const u32 r = q.n - dn;
    ulonglong2 k0 = make_ulonglong2(0, 0), k1 = k0; uint2 x0 = make_uint2(0, 0), x1 = x0;
    if (dn && lane < r) { k0 = q.qe[dn + lane]; x0 = q.qx[dn + lane]; }
    if (dn && lane + 32u < r) { k1 = q.qe[dn + 32u + lane]; x1 = q.qx[dn + 32u + lane]; }
    __syncwarp();
    if (dn && lane < r) { q.qe[lane] = k0; q.qx[lane] = x0; }
    if (dn && lane + 32u < r) { q.qe[32u + lane] = k1; q.qx[32u + lane] = x1; }
    q.n = r;
    __syncwarp();
}

// chunks [c_lo, c_hi) (16 bytes each, absolute positions 16 c; c_lo a multiple of 32); pre[g] = ordinal of the first pretoken of the
// g-th group of 32 chunks (absolute), ord0 = ordinal of the batch's first pretoken, base = 16 c_lo
// DOCS (batch encode): a pretoken that starts on a boundary bit is a document boundary, value VAL_DOC | document index (boundary
// bits before the step's group + the warp's lanes before this one + the chunk's bits before the pretoken); it never touches the cache.
template <bool DOCS>
__global__ void __launch_bounds__(LK_NT, 1) k_enc_lookup(EncTables t, const u32 *__restrict__ flags, const u64 *__restrict__ pre, u64 ord0,
                                                        u64 c_lo, u64 c_hi, u64 n, u64 base, u64 *__restrict__ vals) {
    extern __shared__ __align__(16) unsigned char lk_smem[];
    const u32 lane = lane_id(), warp = threadIdx.x >> 5;
    ulonglong2 *s_kv = reinterpret_cast<ulonglong2 *>(lk_smem);                            // {key, value} image of the value cache
    unsigned char *wq = lk_smem + (size_t)LK_SM_SLOTS * 16 + (size_t)warp * LK_WARP_SMEM;
    LookupQueues q;
    q.qe = reinterpret_cast<ulonglong2 *>(wq); q.qx = reinterpret_cast<uint2 *>(wq + LK_QCAP * 16u);
    q.ql = reinterpret_cast<u64 *>(wq + LK_QCAP * 24u); q.qlo = reinterpret_cast<u32 *>(wq + LK_QCAP * 24u + LK_QL_CAP * 8u);
    q.n = q.nl = 0;
    for (u32 i = threadIdx.x; i < LK_SM_SLOTS; i += LK_NT) s_kv[i] = t.sm_img ? t.sm_img[i] : make_ulonglong2(0, 0);
    __syncthreads();
    const u32 lt = (1u << lane) - 1u;
    const u64 n_fw = (n + 31) >> 5;              // flag words that hold bits of the text
    // steps (32 chunks) are handed out LK_TICKET at a time by a ticket counter: a warp that met expensive pretokens takes fewer
    const u64 n_steps = (c_hi - c_lo + 31) / 32;
    for (;;) {
        u64 tk = 0;
        if (lane == 0) tk = atomicAdd(&t.ctr[9], 1ull);
        tk = __shfl_sync(0xffffffffu, tk, 0);
        if (tk * LK_TICKET >= n_steps) break;
    for (u32 sub = 0; sub < LK_TICKET && tk * LK_TICKET + sub < n_steps; sub++) {
        const u64 c = c_lo + (tk * LK_TICKET + sub) * 32u + lane;
        const bool live = c < c_hi;
        const u64 p0 = c * 16u;
        uint4 A = make_uint4(0, 0, 0, 0), B = A; u32 f0 = 0, f1 = 0, bm = 0;
        const u64 ordg = __ldcs(pre + ((c - lane) >> 5));            // (one word per step, the same for all lanes)
        if (live) {
            const uint4 *tp = reinterpret_cast<const uint4 *>(t.text + p0);
            A = __ldcs(tp); B = __ldcs(tp + 1);
            const u64 w = c >> 1; f0 = __ldcs(flags + w); f1 = w + 1 < n_fw ? __ldcs(flags + w + 1) : 0u;
            if (DOCS) bm = (__ldcs(t.bmask + w) >> (u32)(p0 & 16u)) & 0xFFFFu;
        }
        u64 docc = 0;                            // index of the first document boundary of the chunk
        if (DOCS) {
            u32 bi = __popc(bm);
#pragma unroll
            for (u32 d = 1; d < 32; d <<= 1) { const u32 o = __shfl_up_sync(0xffffffffu, bi, d); if (lane >= d) bi += o; }
            docc = __ldcs(t.bpre + ((c - lane) >> 5)) + bi - __popc(bm);
        }
        const u32 W0 = A.x, W1 = A.y, W2 = A.z, W3 = A.w, W4 = B.x, W5 = B.y, W6 = B.z, W7 = B.w;
        u64 F = (((u64)f1 << 32) | f0) >> (u32)(p0 & 16u);           // bit i: a pretoken starts at byte p0 + i (>= 48 bits)
        if (p0 + 64 > n) F = p0 < n ? F & ((1ull << (n - p0)) - 1ull) : 0ull;   // bits past the end of the text do not count
        const u32 mall = live ? (u32)F & 0xFFFFu : 0u;
        // ordinal of the chunk's first pretoken in the batch: the step's + the start bits of the lanes before this one
        u32 incl = __popc(mall);
#pragma unroll
        for (u32 d = 1; d < 32; d <<= 1) { const u32 o = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += o; }
        const u32 ordc = (u32)(ordg - ord0) + incl - __popc(mall);
        u32 m = mall;
        while (__any_sync(0xffffffffu, m != 0)) {
            const bool act = m != 0;
            const u32 j = act ? __ffs(m) - 1u : 0u;
            m &= m - 1u;
            const u32 ord = ordc + __popc(mall & ((1u << j) - 1u));
            const u64 rest = F >> (j + 1u);
            u32 len = (u32)__ffsll((long long)rest);
            const bool isb = DOCS && act && ((bm >> j) & 1u);
            if (isb) __stcs(&vals[ord], (VAL_DOC << 60) | (docc + __popc(bm & ((1u << j) - 1u))));
            if (act && !isb && len == 0) {               // no further start in the window: a long pretoken, or the last one of the text
                const u64 e = flags_next_start(flags, p0 + j + 1, n) - (p0 + j);
                if (e > MAX_TOKEN_LEN) { t.ctr[6] = 1; len = MAX_TOKEN_LEN; } else len = (u32)e;
            }
            // bytes j .. j + 15 of the 32-byte window
            const u32 qd = j >> 2, sh = (j & 3u) * 8u;
            const bool q2 = qd & 2u, q1 = qd & 1u;
            const u32 X0 = q2 ? W2 : W0, X1 = q2 ? W3 : W1, X2 = q2 ? W4 : W2, X3 = q2 ? W5 : W3, X4 = q2 ? W6 : W4, X5 = q2 ? W7 : W5;
            const u32 Y0 = q1 ? X1 : X0, Y1 = q1 ? X2 : X1, Y2 = q1 ? X3 : X2, Y3 = q1 ? X4 : X3, Y4 = q1 ? X5 : X4;
            const u64 k0 = (u64)__funnelshift_r(Y0, Y1, sh) | ((u64)__funnelshift_r(Y1, Y2, sh) << 32);
            const u64 k1 = (u64)__funnelshift_r(Y2, Y3, sh) | ((u64)__funnelshift_r(Y3, Y4, sh) << 32);
            bool q_s = act && !isb && len <= SHORT_MAX;
            const bool q_m = act && !isb && len > SHORT_MAX && len <= MED_MAX, q_l = act && !isb && len > MED_MAX;
            const u64 key = (k0 & low_bytes_mask(len)) | ((u64)len << 56);               // (short pretokens)
            if (q_s) {
                u32 slot = enc_sm_slot(key);
#pragma unroll
                for (u32 pr = 0; pr < LK_SM_PROBES; pr++) {
                    const ulonglong2 kv = s_kv[slot];
                    if (kv.x == key) { __stcs(&vals[ord], kv.y); q_s = false; break; }
                    slot = (slot + 1) & (LK_SM_SLOTS - 1);
                }
            }
            const u32 me = __ballot_sync(0xffffffffu, q_s || q_m), ml = __ballot_sync(0xffffffffu, q_l);
            const u32 qi = q.n + __popc(me & lt);
            if (q_s) q.qe[qi] = make_ulonglong2(key, 0ull);
            if (q_m) q.qe[qi] = make_ulonglong2(k0, (len > 8 ? k1 & low_bytes_mask(len - 8) : 0ull) | ((u64)len << 56));
            if (q_s || q_m) q.qx[qi] = make_uint2(ord, (u32)(p0 + j - base));
            if (q_l) { const u32 li = q.nl + __popc(ml & lt); q.ql[li] = (p0 + j - base) | ((u64)len << 32); q.qlo[li] = ord; }
            q.n += __popc(me); q.nl += __popc(ml);
            if (q.n >= LK_QDRAIN || q.nl >= LK_QL_DRAIN) lookup_drain(t, q, base, vals, lane, false);
        }
    }
    }
    lookup_drain(t, q, base, vals, lane, true);
}

// ---- BPE of one pretoken: the rank loop, shared by the cache kernels and the BPE-dropout kernels -------------------------------
// Repeatedly the lowest-ranked adjacent pair through the pair -> rank table (tokenizer.py:128-131), and every non-overlapping
// occurrence of it, left to right (Tokenizer.merge, tokenizer.py:92-109).  Two forms: row_bpe, one thread over a shared-memory row
// (pretokens of <= 32 bytes), and warp_bpe, one warp over the tokens in place in the id pool (longer ones).
// DROP (BPE-dropout, spec below at EncDrop): a round also leaves out the candidate pairs that DropOcc::drops, takes the lowest rank
// among the pairs that are left and merges exactly those of its occurrences; for that every token carries the byte offset of its
// first byte in the occurrence (to[]).  The deterministic instances have neither the test nor the offsets.
__device__ __forceinline__ u64 splitmix64(u64 z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
struct DropOcc {                                 // BPE-dropout of one occurrence (see drop_occ)
    u64 thr, h_doc, off0;                        // threshold, mix(mix(seed) ^ doc), the occurrence's byte offset in its document
    // is the pair whose left token starts at byte o of the occurrence dropped in merge round `round`?
    __device__ __forceinline__ bool drops(u64 o, u32 round) const { return (splitmix64(splitmix64(h_doc ^ (off0 + o)) ^ round) >> 32) < thr; }
};

__device__ __forceinline__ u64 warp_min_u64(u64 v) {
#pragma unroll
    for (int d = 16; d; d >>= 1) { u64 o = __shfl_xor_sync(0xffffffffu, v, d); v = o < v ? o : v; }
    return v;
}
// positions that start a merge when the matches of (a, a) overlap: left to right, non-overlapping
// (Tokenizer.merge, tokenizer.py:92-109: after a match the scan resumes two tokens further)
__device__ __forceinline__ u32 resolve_heads_same(u32 m, u32 prev_head) {
    u32 heads = 0, prev = prev_head;
    for (int i = 0; i < 32; i++) {
        u32 h = ((m >> i) & 1u) & (prev ^ 1u);
        heads |= h << i;
        prev = h;
    }
    return heads;
}

// One thread: the n (<= 32) symbols in sym[], the ranks of the adjacent pairs kept up to date in rk[] (after a merge only the pairs
// next to a merged token change).  Returns the number of tokens left in sym[].
template <bool DROP>
__device__ __forceinline__ u32 row_bpe(const EncTables &t, u32 *sym, u32 *rk, uint8_t *to, u32 n, const DropOcc &x) {
    if constexpr (DROP) for (u32 i = 0; i < n; i++) to[i] = (uint8_t)i;
    for (u32 i = 0; i + 1 < n; i++) rk[i] = (u32)(rank_lookup(t, sym[i], sym[i + 1]) >> 32);
    for (u32 round = 0; n > 1; round++) {
        // the lowest-ranked candidate pair; cand = the candidates (DROP only: otherwise every pair is one)
        u32 best = 0xFFFFFFFFu, bi = 0, cand = 0;
        for (u32 i = 0; i + 1 < n; i++) {
            if constexpr (DROP) {
                if (rk[i] == 0xFFFFFFFFu || x.drops(to[i], round)) continue;
                cand |= 1u << i;
            }
            if (rk[i] < best) { best = rk[i]; bi = i; }
        }
        if (best == 0xFFFFFFFFu) break;
        const u32 a = sym[bi], b = sym[bi + 1], res = (u32)rank_lookup(t, a, b);
        // its candidates, left to right, non-overlapping (equal rank <=> same pair)
        u32 o = 0, merged = 0;
        for (u32 i = 0; i < n; o++) {
            if (i + 1 < n && rk[i] == best && (!DROP || ((cand >> i) & 1u))) {
                sym[o] = res; merged |= 1u << o;
                if constexpr (DROP) to[o] = to[i];
                i += 2;
            } else {
                sym[o] = sym[i]; rk[o] = rk[i];
                if constexpr (DROP) to[o] = to[i];
                i += 1;
            }
        }
        n = o;
        for (u32 i = 0; i + 1 < n; i++)
            if ((merged >> i) & 3u) rk[i] = (u32)(rank_lookup(t, sym[i], sym[i + 1]) >> 32);
    }
    return n;
}

// The value of the n tokens in sym[] (their ids go through rk[]); a token missing from the vocabulary is a KeyError
// (tokenizer.py:135).  Up to 3 ids below INLINE_ID_LIMIT go into the value, more go to the id pool at pool_off(n).
template <typename PoolOff>
__device__ __forceinline__ u64 row_value(const EncTables &t, const u32 *sym, u32 *rk, u32 n, PoolOff pool_off) {
    u64 value = 0;
    bool bad = false, big = false;
    for (u32 i = 0; i < n && !bad; i++) {
        const int32_t id = t.sym_to_id[sym[i]];
        if (id < 0) { bad = true; value = (VAL_ERR << 60) | sym[i]; }
        else { big |= (u32)id >= INLINE_ID_LIMIT; rk[i] = (u32)id; }
    }
    if (!bad) {
        if (n <= 3 && !big) {
            value = (u64)n << 60;
            if (n > 0) value |= (u64)rk[0];
            if (n > 1) value |= (u64)rk[1] << 20;
            if (n > 2) value |= (u64)rk[2] << 40;
        } else {
            const u64 off = pool_off(n);
            for (u32 i = 0; i < n; i++) t.ipool[off + i] = rk[i];
            value = (VAL_EXT << 60) | (off << 24) | n;
        }
    }
    return value;
}

// One warp: the n bytes at src, as tokens in place in w = t.ipool + off, which holds their ids at the end; to[] (DROP only) sits
// beside w.  Returns the value.
template <bool DROP>
__device__ __forceinline__ u64 warp_bpe(const EncTables &t, const uint8_t *src, u32 *w, u32 *to, u32 n, u64 off, const DropOcc &x, u32 lane) {
    for (u32 i = lane; i < n; i += 32) {
        w[i] = src[i];
        if constexpr (DROP) to[i] = i;
    }
    __syncwarp();
    for (u32 round = 0; n > 1; round++) {
        u64 best = RANK_NONE;
        for (u32 b0 = 0; b0 + 1 < n; b0 += 32) {
            u32 i = b0 + lane;
            if (i + 1 < n) { u64 r = rank_lookup(t, w[i], w[i + 1]); if (r < best && !(DROP && x.drops(to[i], round))) best = r; }
        }
        best = warp_min_u64(best);
        if (best == RANK_NONE) break;
        const u32 j = (u32)(best >> 32), res = (u32)best;
        const u32 a = (u32)t.mpairs[2 * j], b = (u32)t.mpairs[2 * j + 1];
        u32 out = 0, carry = 0;
        for (u32 b0 = 0; b0 < n; b0 += 32) {
            u32 i = b0 + lane;
            u32 cur = i < n ? w[i] : 0xFFFFFFFFu, nx = i + 1 < n ? w[i + 1] : 0xFFFFFFFFu, ci = DROP && i < n ? to[i] : 0u;
            u32 m = __ballot_sync(0xffffffffu, cur == a && nx == b && !(DROP && x.drops(ci, round)));
            // only the matches of (a, a) can overlap: a match of (a, b), a != b, ends in b, which starts no match
            u32 heads = a == b ? resolve_heads_same(m, carry) : m;
            u32 valid = __ballot_sync(0xffffffffu, i < n);
            u32 kept = valid & ~((heads << 1) | carry);
            carry = heads >> 31;
            u32 val = ((heads >> lane) & 1u) ? res : cur;
            u32 pos = out + __popc(kept & ((1u << lane) - 1u));
            __syncwarp();
            if ((kept >> lane) & 1u) {
                w[pos] = val;
                if constexpr (DROP) to[pos] = ci;
            }
            out += __popc(kept);
            __syncwarp();
        }
        n = out;
    }
    // ids in place; a token missing from the vocabulary is a KeyError (tokenizer.py:135)
    u32 bad_idx = 0xFFFFFFFFu;
    for (u32 i = lane; i < n; i += 32) if (t.sym_to_id[w[i]] < 0 && i < bad_idx) bad_idx = i;
    for (int d = 16; d; d >>= 1) { u32 o = __shfl_xor_sync(0xffffffffu, bad_idx, d); bad_idx = o < bad_idx ? o : bad_idx; }
    if (bad_idx != 0xFFFFFFFFu) return (VAL_ERR << 60) | w[bad_idx];
    for (u32 i = lane; i < n; i += 32) w[i] = (u32)t.sym_to_id[w[i]];
    return (VAL_EXT << 60) | (off << 24) | n;
}

// ---- BPE of the queued pretokens of <= 32 bytes: one THREAD each ---------------------------------------------------
// (one warp per pretoken leaves three quarters of the lanes idle on the typical 4-10 byte pretoken: 1 380 warp
// instructions per pretoken measured.)  Symbols and the ranks of the adjacent pairs live in a private shared-memory row.
#define BPT_NT 128
#define BPT_MAX 32u
// Two instances: pretokens of <= 15 bytes (short and medium table entries -- 98 % of the new pretokens of web-like text) with rows of
// 16 symbols, i.e. half the shared memory and twice the resident threads of the 32-symbol instance that takes the long-table entries
// of 16..32 bytes (the kernel waits on dependent L2 lookups of pair ranks: occupancy is what it needs).
template <u32 ROW, bool LONGS>
__global__ void __launch_bounds__(BPT_NT) k_enc_bpe_short(EncTables t, u64 n_todo) {
    __shared__ u32 s_sym[BPT_NT][ROW + 1];
    __shared__ u32 s_ids[BPT_NT][ROW + 1];
    u32 *sym = s_sym[threadIdx.x], *rk = s_ids[threadIdx.x];
    for (u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x; q < n_todo; q += (u64)gridDim.x * blockDim.x) {
        const u32 ref = t.todo[q];
        const bool is_long = ref & REF_LONG, is_med = ref & REF_MED;
        if (is_long != LONGS) continue;          // the other instance's
        const u32 slot = REF_SLOT(ref);
        u32 n;
        if (is_med) {
            const u64 k0 = t.medtab[slot].k0, k1 = t.medtab[slot].k1;
            n = (u32)(k1 >> 56);
            for (u32 i = 0; i < n; i++) sym[i] = (u32)(((i < 8 ? k0 >> (8 * i) : k1 >> (8 * (i - 8)))) & 0xFFu);
        } else if (is_long) {
            const u64 m = t.ltab[slot].meta;
            n = (u32)(m & META_LEN_MASK);
            if (n > BPT_MAX) continue;           // the warp kernel's
            const uint8_t *src = rep_ptr(t, m);
            // move the key bytes out of the (transient) text arena into the persistent key pool
            const u64 ko = atomicAdd(&t.ctr[4], (u64)n);
            for (u32 i = 0; i < n; i++) { const u32 b = src[i]; t.pool[ko + i] = (uint8_t)b; sym[i] = b; }
            t.ltab[slot].meta = ((ko | META_POOL_BIT) << META_LEN_BITS) | n;
        } else {
            const u64 k = t.stab[slot].key;
            n = (u32)(k >> 56);
            for (u32 i = 0; i < n; i++) sym[i] = (u32)((k >> (8 * i)) & 0xFFu);
        }
        n = row_bpe<false>(t, sym, rk, nullptr, n, DropOcc{});
        const u64 value = row_value(t, sym, rk, n, [&](u32 c) { return (u64)atomicAdd(&t.ctr[5], (u64)c); });
        if (is_med) t.medtab[slot].val = value; else if (is_long) t.ltab[slot].val = value; else t.stab[slot].val = value;
    }
}

// ---- the long-table entries of more than BPT_MAX bytes: one warp each, tokens in place in the id pool ----
// (every entry of up to BPT_MAX bytes, short and medium ones included, is k_enc_bpe_short's)
__global__ void __launch_bounds__(256) k_enc_bpe(EncTables t, u64 n_todo) {
    const u32 lane = lane_id();
    const u64 gwarp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((u64)gridDim.x * blockDim.x) >> 5;
    for (u64 q = gwarp; q < n_todo; q += nwarps) {
        const u32 ref = t.todo[q];
        if (!(ref & REF_LONG)) continue;
        const u32 slot = REF_SLOT(ref);
        const u64 m = t.ltab[slot].meta;
        const u32 len = (u32)(m & META_LEN_MASK);
        if (len <= BPT_MAX) continue;
        const uint8_t *src = rep_ptr(t, m);
        // move the key bytes out of the (transient) text arena into the persistent key pool
        u64 ko = 0;
        if (lane == 0) ko = atomicAdd(&t.ctr[4], (u64)len);
        ko = __shfl_sync(0xffffffffu, ko, 0);
        for (u32 i = lane; i < len; i += 32) t.pool[ko + i] = src[i];
        __syncwarp();
        if (lane == 0) t.ltab[slot].meta = ((ko | META_POOL_BIT) << META_LEN_BITS) | len;
        u64 off = 0;
        if (lane == 0) off = atomicAdd(&t.ctr[5], (u64)len);
        off = __shfl_sync(0xffffffffu, off, 0);
        const u64 value = warp_bpe<false>(t, t.pool + ko, t.ipool + off, nullptr, len, off, DropOcc{}, lane);
        if (lane == 0) t.ltab[slot].val = value;
    }
}

__device__ __forceinline__ u64 enc_value(const EncTables &t, u32 ref) {
    return (ref & REF_LONG) ? t.ltab[REF_SLOT(ref)].val : (ref & REF_MED) ? t.medtab[REF_SLOT(ref)].val : t.stab[ref].val;
}
__device__ __forceinline__ u32 value_count(u64 v) {
    u32 tag = VAL_TAG(v);
    return tag <= 3 ? tag : (tag == VAL_EXT ? (u32)(v & 0xFFFFFFu) : 0);
}

// ---- fused: tokens per pretoken -> exclusive offsets -> ids, in ONE pass (single-pass scan with decoupled look-back) -------
// The three kernels above read the per-occurrence values twice and round-trip a count and an offset array through HBM
// (~45 B per pretoken); this one reads each value once and writes only the ids (8 B + 2 B per token).  A CTA takes the next
// tile from a ticket counter (tiles start in order, so the look-back cannot wait on a tile that has not been scheduled),
// counts its tokens, publishes {status, sum} in one 64-bit word, adds up its predecessors' words until it meets an
// inclusive prefix, and emits its ids at that offset.
#ifndef SE_NT
#define SE_NT 512
#endif
#ifndef SE_ITEMS
#define SE_ITEMS 8
#endif
#define SE_TILE (SE_NT * SE_ITEMS)
#ifndef SE_STAGE
#define SE_STAGE 10240u                          // ids staged per tile (40 KB); OWT-shape text averages ~5 700 per tile (512 x 8 pretokens: 19.0 -> 17.1 ms per 10 GB against 256 x 8)
#endif
#define SE_AGG (1ull << 62)
#define SE_INCL (2ull << 62)
#define SE_VAL(x) ((x) & ((1ull << 62) - 1))
__device__ __forceinline__ u64 warp_sum_u64(u64 v) {
#pragma unroll
    for (int d = 16; d; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    return v;
}
template <typename OutT, bool kEmit>
__global__ void __launch_bounds__(SE_NT) k_enc_scan_emit(EncTables t, const u64 *__restrict__ vals, u64 n_items, u64 ord_base,
                                                        u64 *tile_state, u32 *ticket, OutT *__restrict__ out, u64 out_base, u64 cap,
                                                        u64 *__restrict__ total_out) {
    __shared__ u32 s_tile;
    __shared__ u32 s_warp[33];
    __shared__ u64 s_prefix;
    if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const u32 tile = s_tile;
    const u64 first = (u64)tile * SE_TILE + (u64)threadIdx.x * SE_ITEMS;
    u64 v[SE_ITEMS];
    u32 sum = 0;
    if (first + SE_ITEMS <= n_items) {           // 16-byte loads (vals is 16-byte aligned and `first` a multiple of SE_ITEMS): a sector is fetched by two instructions, not four
#pragma unroll
        for (u32 k = 0; k < SE_ITEMS; k += 2) { const ulonglong2 w = __ldcs(reinterpret_cast<const ulonglong2 *>(vals + first + k)); v[k] = w.x; v[k + 1] = w.y; }
    } else {
#pragma unroll
        for (u32 k = 0; k < SE_ITEMS; k++) v[k] = first + k < n_items ? __ldcs(&vals[first + k]) : 0;
    }
#pragma unroll
    for (u32 k = 0; k < SE_ITEMS; k++) {
        if (first + k >= n_items) continue;
        if (VAL_TAG(v[k]) == VAL_FWD) v[k] = enc_value(t, (u32)v[k]);                             // computed by the BPE kernels meanwhile
        if (VAL_TAG(v[k]) == VAL_ERR) atomicMin(&t.ctr[7], ord_base + first + k);                 // KeyError: the first failing pretoken in text order
        sum += value_count(v[k]);
    }
    u32 tot;
    const u32 ex = block_excl_scan_u32(sum, &tot, s_warp);
    // A thread owns SE_ITEMS consecutive pretokens, i.e. ~11 consecutive ids: written straight to global memory, the 32 lanes
    // of a store instruction would hit ~22 different sectors with 2 bytes each.  The ids of the tile are staged in shared
    // memory instead and copied out with consecutive threads on consecutive ids (tiles with more ids than the stage holds
    // -- long pool-resident values -- take the direct path).  The staging needs only the offsets INSIDE the tile, so the warps
    // do it while warp 0 looks back for the tile's global offset (a third of all stall samples sat behind that look-back).
    __shared__ u32 s_ids[SE_STAGE];
    const bool staged = kEmit && tot <= SE_STAGE;
    auto stage_ids = [&]() {
        u32 o = ex;
#pragma unroll
        for (u32 k = 0; k < SE_ITEMS; k++) {
            const u32 tag = VAL_TAG(v[k]);
            if (tag <= 3) {
                for (u32 q = 0; q < tag; q++) s_ids[o++] = (u32)((v[k] >> (20 * q)) & 0xFFFFFu);
            } else if (tag == VAL_EXT) {
                const u32 *src = t.ipool + ((v[k] >> 24) & 0xFFFFFFFFFull);
                const u32 c = (u32)(v[k] & 0xFFFFFFu);
                for (u32 q = 0; q < c; q++) s_ids[o++] = src[q];
            }
        }
    };
    if (threadIdx.x >= 32 && staged) stage_ids();
    if (threadIdx.x < 32) {
        const u32 lane = threadIdx.x;
        u64 run = 0;
        if (tile > 0) {
            if (lane == 0) *((volatile u64 *)&tile_state[tile]) = SE_AGG | (u64)tot;
            long long j = (long long)tile - 1;
            for (;;) {
                const long long idx = j - lane;
                u64 w = idx >= 0 ? *((volatile u64 *)&tile_state[idx]) : SE_INCL;
                while (__any_sync(0xffffffffu, (w >> 62) == 0)) { if (idx >= 0 && (w >> 62) == 0) w = *((volatile u64 *)&tile_state[idx]); }
                const u32 m = __ballot_sync(0xffffffffu, (w >> 62) == 2);
                if (m) {
                    const u32 stop = __ffs(m) - 1;                       // nearest tile with an inclusive prefix
                    run += warp_sum_u64(lane <= stop ? SE_VAL(w) : 0);
                    break;
                }
                run += warp_sum_u64(SE_VAL(w));
                j -= 32;
            }
        }
        if (lane == 0) {
            *((volatile u64 *)&tile_state[tile]) = SE_INCL | (run + tot);
            s_prefix = run;
            if ((u64)(tile + 1) * SE_TILE >= n_items) *total_out = run + tot;
        }
        if (staged) stage_ids();
    }
    __syncthreads();
    if (t.id_offs) {                             // batch encode: a document boundary holds where the next document's ids start
        u64 o = t.id_base + out_base + s_prefix + ex;
#pragma unroll
        for (u32 k = 0; k < SE_ITEMS; k++) {
            if (VAL_TAG(v[k]) == VAL_DOC) t.id_offs[v[k] & VAL_DOC_MASK] = o;
            o += value_count(v[k]);
        }
    }
    if (!kEmit) return;
    const u64 tile_dst = out_base + s_prefix;
    if (staged) {
        for (u32 j = threadIdx.x; j < tot; j += SE_NT) { const u64 d = tile_dst + j; if (d < cap) __stcs(&out[d], (OutT)s_ids[j]); }
        return;
    }
    u64 dst = tile_dst + ex;
#pragma unroll
    for (u32 k = 0; k < SE_ITEMS; k++) {
        const u32 tag = VAL_TAG(v[k]);
        if (tag <= 3) {
            for (u32 q = 0; q < tag; q++) { if (dst < cap) out[dst] = (OutT)((v[k] >> (20 * q)) & 0xFFFFFu); dst++; }
        } else if (tag == VAL_EXT) {
            const u32 *src = t.ipool + ((v[k] >> 24) & 0xFFFFFFFFFull);
            const u32 c = (u32)(v[k] & 0xFFFFFFu);
            for (u32 q = 0; q < c; q++) { if (dst < cap) out[dst] = (OutT)src[q]; dst++; }
        }
    }
}

// ---- BPE-dropout (bpe_encode_ex with dropout > 0): every pretoken occurrence gets its own random BPE ----------
// Spec (include/bpe_sm100.h): candidate pair (i, i+1) of merge round t is dropped when (u(seed, doc, off_i, t) >> 32) < thr, with
// u = mix(mix(mix(mix(seed) ^ doc) ^ off) ^ t), mix = the splitmix64 finalizer, off_i = byte offset in the document of token i's first
// byte.  The round takes the lowest rank among the pairs that are left and merges, left to right and non-overlapping, exactly those of
// its occurrences that were not dropped.  The result depends on the occurrence, so it never goes to the cache: the stage runs after the
// cache BPE kernels and replaces vals[ordinal] of the batch, with ids (when they do not fit the value) in the id pool's unused tail.
struct EncDrop {
    u64 thr;                                     // 0 < thr <= 2^32
    u64 seed_mix;                                // mix(seed)
    u64 lo;                                      // where the chunk starts in the caller's text
    const u64 *doffs; u64 da;                    // batch encode: the caller's document offsets, the chunk's first document (else null, 0)
    const u32 *skip;                             // special-token starts and document boundaries (or null): their values stay
    const u64 *starts;                           // byte offset in the arena of every pretoken of the batch
    u32 *loff;                                   // per byte from the batch start: token offsets of the warp kernel's pretokens
    u64 ibase;                                   // id pool offset of the batch start's scratch (one id per byte)
};

// set bits before arena byte p of a bitmask with one bit per byte, from its counts before every 512-byte group (pre) and the words of
// p's group; mask needs the word that holds p
__device__ __forceinline__ u64 bits_before(const u32 *__restrict__ mask, const u64 *__restrict__ pre, u64 p) {
    const u64 w = p >> 5;
    u64 j = pre[w >> 4];
    for (u64 k = w & ~15ull; k < w; k++) j += __popc(mask[k]);
    return j + __popc(mask[w] & ((1u << (p & 31)) - 1u));
}

// mix(mix(seed) ^ doc) and the offset in its document of the pretoken at arena byte p
__device__ __forceinline__ DropOcc drop_occ(const EncTables &t, const EncDrop &d, u64 p) {
    if (!d.doffs) return {d.thr, splitmix64(d.seed_mix), d.lo + p};
    const u64 j = bits_before(t.bmask, t.bpre, p);   // document boundaries before p
    return {d.thr, splitmix64(d.seed_mix ^ (d.da + j)), d.lo + p - j - d.doffs[d.da + j]};   // (arena -> caller position: minus the boundary bytes before it)
}

// starts[ordinal - ord0] = arena offset of every pretoken starting in flag words [w_lo, w_hi)
__global__ void __launch_bounds__(256) k_enc_drop_starts(const u32 *__restrict__ flags, const u64 *__restrict__ pre, u64 ord0, u64 w_lo, u64 w_hi,
                                                        u64 *__restrict__ starts) {
    for (u64 w = w_lo + (u64)blockIdx.x * blockDim.x + threadIdx.x; w < w_hi; w += (u64)gridDim.x * blockDim.x) {
        u32 bits = flags[w];
        if (!bits) continue;
        u64 o = pre[w >> 4] - ord0;
        for (u64 k = w & ~15ull; k < w; k++) o += __popc(flags[k]);
        while (bits) { const u32 j = __ffs(bits) - 1; bits &= bits - 1; starts[o++] = w * 32 + j; }
    }
}

// One thread per occurrence of <= 32 bytes (row_bpe in the row layout of k_enc_bpe_short, plus each token's byte offset); longer ones
// that need redoing are queued (t.todo, count in ctr[10]) for k_enc_drop_warp.  An occurrence keeps its cached value when it is a special
// token or a document boundary, or when that value already has one token per byte: no pair had a rank, and dropout only removes candidates.
__global__ void __launch_bounds__(BPT_NT) k_enc_drop_short(EncTables t, EncDrop d, const u32 *__restrict__ flags, u64 n, u64 base, u64 bound,
                                                          u64 *__restrict__ vals) {
    __shared__ u32 s_sym[BPT_NT][BPT_MAX + 1];
    __shared__ u32 s_rk[BPT_NT][BPT_MAX + 1];
    __shared__ uint8_t s_off[BPT_NT][BPT_MAX + 1];
    u32 *sym = s_sym[threadIdx.x], *rk = s_rk[threadIdx.x];
    for (u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x; q < bound; q += (u64)gridDim.x * blockDim.x) {
        u64 v = vals[q];
        if (VAL_TAG(v) == VAL_DOC) continue;
        const u64 p = d.starts[q];
        if (d.skip && ((d.skip[p >> 5] >> (p & 31)) & 1u)) continue;
        const u64 e = q + 1 < bound ? d.starts[q + 1] : flags_next_start(flags, p + 1, n);
        const u32 len = (u32)(e - p);
        if (VAL_TAG(v) == VAL_FWD) v = enc_value(t, (u32)v);
        if (VAL_TAG(v) != VAL_ERR && value_count(v) == len) continue;
        if (len > BPT_MAX) { const u64 k = atomicAdd(&t.ctr[10], 1ull); t.todo[k] = (u32)q; continue; }
        for (u32 i = 0; i < len; i++) sym[i] = t.text[p + i];
        const u32 nt = row_bpe<true>(t, sym, rk, s_off[threadIdx.x], len, drop_occ(t, d, p));
        vals[q] = row_value(t, sym, rk, nt, [&](u32) { return d.ibase + (p - base); });
    }
}

// The queued occurrences of > 32 bytes: warp_bpe, one warp each, symbols in place in the id pool scratch, token offsets beside them
// in d.loff.
__global__ void __launch_bounds__(256) k_enc_drop_warp(EncTables t, EncDrop d, const u32 *__restrict__ flags, u64 n, u64 base, u64 bound,
                                                      u64 *__restrict__ vals) {
    const u32 lane = lane_id();
    const u64 gwarp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((u64)gridDim.x * blockDim.x) >> 5;
    const u64 n_q = t.ctr[10];
    for (u64 k = gwarp; k < n_q; k += nwarps) {
        const u64 q = t.todo[k];
        const u64 p = d.starts[q];
        const u64 e = q + 1 < bound ? d.starts[q + 1] : flags_next_start(flags, p + 1, n);
        const u64 io = d.ibase + (p - base);
        const u64 value = warp_bpe<true>(t, t.text + p, t.ipool + io, d.loff + (p - base), (u32)(e - p), io, drop_occ(t, d, p), lane);
        if (lane == 0) vals[q] = value;
    }
}

// ---- token offsets (bpe_encode_ex with with_offsets): a span of the input for every token --------------------------
// Spec (include/bpe_sm100.h): the tokens of a pretoken occurrence tile its bytes in order; each but the last is as long as its vocabulary
// entry (tok->vlen), the last ends where the pretoken ends.  So a special-token occurrence -- one id, whatever that id is -- spans the
// special's bytes.  Per batch, after the emit kernel: the pretoken starts (k_enc_drop_starts), the token count of every pretoken and its
// exclusive scan (the index of its first token), then one thread per pretoken writes {start, end} of its tokens next to their ids.
// Characters: lead bytes ((b & 0xC0) != 0x80) before a byte, counted from a bit per arena byte and its count per 512-byte group;
// a token's start is the index of the character holding its first byte, its end one past that of the character holding its last byte.
struct EncOffs {
    int chars;                                   // BPE_OFF_CHARS: character indices, else byte offsets
    long long *out;                              // {start, end} of every token of the chunk, in the order of its ids
    u64 lo;                                      // where the chunk starts in the caller's text
    const u64 *doffs; u64 da;                    // batch encode: the caller's document offsets, the chunk's first document (else null, 0)
    u64 carry;                                   // characters of the chunk's first document before lo
    const u32 *lmask; const u64 *lpre;           // lead-byte bit per arena byte (words up to 16 (groups + 1)), count before every 512-byte group
    const u32 *vlen; u64 n_dense;                // byte length of every vocabulary id
    const u64 *starts, *tpre;                    // per batch: arena offset of every pretoken, index of its first token in the batch
};

// lmask[w] = lead-byte bits of arena bytes 32 w .. 32 w + 31 (none past n), for w < n_words
__global__ void __launch_bounds__(256) k_enc_lead_bits(const uint8_t *__restrict__ text, u64 n, u64 n_words, u32 *__restrict__ lmask) {
    for (u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += (u64)gridDim.x * blockDim.x) {
        u32 m = 0;
        if (w * 32 < n) {
            const uint4 *p = reinterpret_cast<const uint4 *>(text + w * 32);
            const uint4 a = p[0], b = p[1];
            const u32 x[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
            for (int k = 0; k < 8; k++) {
                const u32 l = ~((x[k] >> 7) & ~(x[k] >> 6)) & 0x01010101u;      // bit 0 of every byte: not a continuation byte 10xxxxxx
                m |= ((l | (l >> 7) | (l >> 14) | (l >> 21)) & 0xFu) << (4 * k);
            }
            if (n - w * 32 < 32) m &= (1u << (n - w * 32)) - 1u;
        }
        lmask[w] = m;
    }
}

// cnt[q] = tokens of pretoken q of the batch; forward references are resolved in vals (the emit kernel has read them)
__global__ void __launch_bounds__(256) k_enc_off_count(EncTables t, u64 *__restrict__ vals, u64 bound, u32 *__restrict__ cnt) {
    for (u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x; q < bound; q += (u64)gridDim.x * blockDim.x) {
        u64 v = vals[q];
        if (VAL_TAG(v) == VAL_FWD) { v = enc_value(t, (u32)v); vals[q] = v; }
        cnt[q] = value_count(v);
    }
}

// o.out[out_base + o.tpre[q] + k] = span of token k of pretoken q (below cap); n = arena bytes, flags = pretoken starts
template <bool CHARS>
__global__ void __launch_bounds__(256) k_enc_offsets(EncTables t, EncOffs o, const u32 *__restrict__ flags, const u64 *__restrict__ vals, u64 n,
                                                    u64 bound, u64 out_base, u64 cap) {
    longlong2 *out = reinterpret_cast<longlong2 *>(o.out);
    for (u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x; q < bound; q += (u64)gridDim.x * blockDim.x) {
        const u64 v = vals[q];
        const u32 c = value_count(v);
        if (!c) continue;                        // a document boundary (or a KeyError: the call fails)
        const u64 p = o.starts[q], e = q + 1 < bound ? o.starts[q + 1] : flags_next_start(flags, p + 1, n);
        // its document: j boundaries before p; arena -> document coordinates (all mod 2^64)
        const u64 j = t.bmask ? bits_before(t.bmask, t.bpre, p) : 0;
        const u64 bbase = o.lo - j - (o.doffs ? o.doffs[o.da + j] : 0);
        u64 cbase = 0, lc = 0;                   // lc = lead bytes before the token
        if (CHARS) {
            cbase = j ? 0 - bits_before(o.lmask, o.lpre, o.doffs[o.da + j] - o.lo + j) : o.carry;
            lc = bits_before(o.lmask, o.lpre, p);
        }
        const u32 *pool = t.ipool + ((v >> 24) & 0xFFFFFFFFFull);
        const u64 dst = out_base + o.tpre[q];
        u64 s = p;
        for (u32 k = 0; k < c; k++) {
            u64 end = e;
            if (k + 1 < c) {
                const u32 id = VAL_TAG(v) <= 3 ? (u32)((v >> (20 * k)) & 0xFFFFFu) : pool[k];
                end = min(e, s + (id < o.n_dense ? o.vlen[id] : 1u));
            }
            longlong2 span;
            if (CHARS) {
                const u64 le = bits_before(o.lmask, o.lpre, end);
                const u64 lead = (o.lmask[s >> 5] >> (s & 31)) & 1u;
                span = make_longlong2((long long)(lc + lead - 1 + cbase), (long long)(le + cbase));
                lc = le;
            } else {
                span = make_longlong2((long long)(s + bbase), (long long)(end + bbase));
            }
            if (dst + k < cap) out[dst + k] = span;
            s = end;
        }
    }
}

// *host = lead bytes in arena bytes [a, b)
__global__ void k_enc_lead_span(const u32 *__restrict__ lmask, const u64 *__restrict__ lpre, u64 a, u64 b, u64 *host) {
    *host = bits_before(lmask, lpre, b) - bits_before(lmask, lpre, a);
    __threadfence_system();
}

// ---- hot table: histogram of the sampled hit counts, build ----------------------------------------------------------
#define ENC_HOT_HIST 64
__global__ void __launch_bounds__(256) k_enc_hot_hist(EncTables t, u64 *__restrict__ hist /* [ENC_HOT_HIST] */) {
    __shared__ u32 s_h[ENC_HOT_HIST];
    if (threadIdx.x < ENC_HOT_HIST) s_h[threadIdx.x] = 0;
    __syncthreads();
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < t.scap + t.medcap; i += (u64)gridDim.x * blockDim.x) {
        const u32 c = i < t.scap ? t.scnt[i] : t.mcnt[i - t.scap];
        if (c) atomicAdd(&s_h[c < ENC_HOT_HIST ? c : ENC_HOT_HIST - 1], 1u);
    }
    __syncthreads();
    if (threadIdx.x < ENC_HOT_HIST && s_h[threadIdx.x]) atomicAdd(&hist[threadIdx.x], (u64)s_h[threadIdx.x]);
}
// every cached pretoken of <= 15 bytes looked up at least `thresh` times whose value is computed: into its bucket if a slot is free
__global__ void __launch_bounds__(256) k_enc_hot_build(EncTables t, ulonglong2 *__restrict__ hot, u64 *__restrict__ hval, u64 nb, u32 thresh) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < t.scap + t.medcap; i += (u64)gridDim.x * blockDim.x) {
        u64 k0, k1, v;
        if (i < t.scap) {
            if (t.scnt[i] < thresh) continue;
            k0 = t.stab[i].key; k1 = 0; v = t.stab[i].val;
            if (k0 == 0) continue;
        } else {
            const u64 s = i - t.scap;
            if (t.mcnt[s] < thresh) continue;
            k0 = t.medtab[s].k0; k1 = t.medtab[s].k1; v = t.medtab[s].val;
            if ((k0 | k1) == 0) continue;
        }
        if (v == VAL_NONE || VAL_TAG(v) == VAL_FWD) continue;
        const u64 b = hot_bucket(nb, k0, k1);
        const int w = hot_claim(hot, b, k0, k1);
        if (w >= 0) hval[2 * b + w] = v;
    }
}

// ---- image of the lookup kernel's shared-memory value cache: the most looked-up short pretokens of the sampled batch ----
__device__ __forceinline__ u32 log_bucket(u32 c) {                   // 8 buckets per power of two
    if (c < 8) return c;
    const u32 lz = 31u - __clz(c);
    return (lz - 2u) * 8u + ((c >> (lz - 3u)) & 7u);
}
__global__ void __launch_bounds__(256) k_enc_sm_hist(EncTables t, u64 *__restrict__ hist /* [256] */) {
    __shared__ u32 s_h[256];
    s_h[threadIdx.x] = 0;
    __syncthreads();
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < t.scap; i += (u64)gridDim.x * blockDim.x) {
        const u32 c = t.scnt[i];
        if (c) atomicAdd(&s_h[log_bucket(c)], 1u);
    }
    __syncthreads();
    if (s_h[threadIdx.x]) atomicAdd(&hist[threadIdx.x], (u64)s_h[threadIdx.x]);
}
__global__ void __launch_bounds__(256) k_enc_sm_build(EncTables t, ulonglong2 *__restrict__ img, u32 min_bucket) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < t.scap; i += (u64)gridDim.x * blockDim.x) {
        const u32 c = t.scnt[i];
        if (!c || log_bucket(c) < min_bucket) continue;
        const u64 key = t.stab[i].key, v = t.stab[i].val;
        if (key == 0 || v == VAL_NONE || VAL_TAG(v) == VAL_FWD) continue;
        u32 slot = enc_sm_slot(key);
        for (u32 pr = 0; pr < LK_SM_PROBES; pr++) {
            if (atomicCAS(&img[slot].x, 0ull, key) == 0ull) { img[slot].y = v; break; }
            slot = (slot + 1) & (LK_SM_SLOTS - 1);
        }
    }
}

// ---- cache maintenance ---------------------------------------------------------------------------------
// growth: every key of an old table into the bigger one
__global__ void __launch_bounds__(256) k_enc_rehash_short(const SSlot *__restrict__ otab, u64 ocap, EncTables t) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < ocap; i += (u64)gridDim.x * blockDim.x)
        if (otab[i].key) short_insert_unique(t, otab[i].key, otab[i].val);
}
__global__ void __launch_bounds__(256) k_enc_rehash_long(const LSlot *__restrict__ otab, u64 ocap, EncTables t) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < ocap; i += (u64)gridDim.x * blockDim.x)
        if (otab[i].meta != META_EMPTY) long_insert_unique(t, otab[i].meta, otab[i].hash, otab[i].val);
}
__global__ void __launch_bounds__(256) k_enc_rehash_med(const MSlot *__restrict__ otab, u64 ocap, EncTables t) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < ocap; i += (u64)gridDim.x * blockDim.x)
        if ((otab[i].k0 | otab[i].k1) != 0) medium_insert_unique(t, otab[i].k0, otab[i].k1, otab[i].val);
}

// empty tables: short {0, VAL_NONE}, medium {0, 0, VAL_NONE, 0}, long {META_EMPTY, 0, VAL_NONE, 0}
__global__ void __launch_bounds__(256) k_enc_clear_tables(EncTables t) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < t.scap; i += (u64)gridDim.x * blockDim.x) {
        *reinterpret_cast<ulonglong2 *>(&t.stab[i]) = make_ulonglong2(0ull, VAL_NONE);
    }
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < t.lcap; i += (u64)gridDim.x * blockDim.x) {
        ulonglong2 *q = reinterpret_cast<ulonglong2 *>(&t.ltab[i]);
        q[0] = make_ulonglong2(META_EMPTY, 0ull); q[1] = make_ulonglong2(VAL_NONE, 0ull);
    }
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < t.medcap; i += (u64)gridDim.x * blockDim.x) {
        ulonglong2 *q = reinterpret_cast<ulonglong2 *>(&t.medtab[i]);
        q[0] = make_ulonglong2(0ull, 0ull); q[1] = make_ulonglong2(VAL_NONE, 0ull);
    }
}

// Special tokens are pretokens of their own (tokenizer.py:119-122): pre-insert them with their id into the empty tables.
// Their bytes sit at the start of the key pool (sp_offs are offsets into it).  Of specials with the same bytes the first one counts.
__global__ void k_enc_insert_specials(EncTables t, const u32 *__restrict__ sp_offs, const long long *__restrict__ sp_ids, int n_sp) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_sp) return;
    u32 o = sp_offs[i], len = sp_offs[i + 1] - o;
    if (len == 0) return;
    const uint8_t *p = t.pool + o;
    for (int j = 0; j < i; j++)
        if (sp_offs[j + 1] - sp_offs[j] == len && bytes_equal(t.pool + sp_offs[j], p, len)) return;
    long long id = sp_ids[i];
    u64 v;
    if (id < 0) v = (VAL_ERR << 60) | 0x80000000ull | (u32)i;
    else if ((u64)id < INLINE_ID_LIMIT) v = (1ull << 60) | (u64)id;
    else { u64 q = atomicAdd(&t.ctr[5], 1ull); t.ipool[q] = (u32)id; v = (VAL_EXT << 60) | (q << 24) | 1ull; }
    if (len <= MED_MAX) {
        u64 k0, k1;
        pretoken_key(p, len, k0, k1);
        if (k1 == 0) { short_insert_unique(t, k0, v); atomicAdd(&t.ctr[0], 1ull); }
        else { medium_insert_unique(t, k0, k1, v); atomicAdd(&t.ctr[8], 1ull); }
    } else {
        long_insert_unique(t, (((u64)o | META_POOL_BIT) << META_LEN_BITS) | len, hash_long(p, len), v);
        atomicAdd(&t.ctr[1], 1ull);
    }
}

// ---- decode ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_dec_lens(const long long *__restrict__ ids, u64 n, const u32 *__restrict__ vlen, long long n_dense,
                                                 u32 *__restrict__ lens, u64 *__restrict__ bad) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        long long id = ids[i];
        u32 l = (id >= 0 && id < n_dense) ? vlen[id] : 0xFFFFFFFFu;
        if (l == 0xFFFFFFFFu) { atomicMin(bad, i); l = 0; }
        lens[i] = l;
    }
}
__global__ void __launch_bounds__(256) k_dec_copy(const long long *__restrict__ ids, u64 n, const u64 *__restrict__ voff,
                                                 const uint8_t *__restrict__ vblob, const u32 *__restrict__ lens,
                                                 const u64 *__restrict__ off, uint8_t *__restrict__ out, u64 cap) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        u32 l = lens[i];
        if (!l) continue;
        const uint8_t *src = vblob + voff[ids[i]];
        u64 o = off[i];
        for (u32 k = 0; k < l; k++) if (o + k < cap) out[o + k] = src[k];
    }
}

// =============================================================================================
// host side
// =============================================================================================
struct bpe_tok {
    bpe_ctx *ctx = nullptr;
    int n_merges = 0, n_syms = 0, n_sp = 0;
    long long max_id = -1, n_dense = 0;
    DevBuf mtab, mpairs, sym_to_id;              // merge tables
    u64 mcap = 0;
    DevBuf vlen, voff, vblob;                    // decode tables
    DevBuf sp_offs, sp_ids;                      // specials (device); their bytes open the key pool
    std::vector<uint8_t> sp_blob_h; std::vector<u32> sp_offs_h;
    std::vector<uint8_t> sym_blob_h; std::vector<u64> sym_offs_h;
    u32 sp_max_len = 0;
    // pretoken cache
    DevBuf stab, medtab, ltab, kpool, ipool, todo, ctr;
    u64 scap = 0, medcap = 0, lcap = 0;
    bool cache_ready = false;
    DevBuf hot, samp, sm_img;                    // hot table (keys then values); sampling counters of the batch that feeds it; shared-memory cache image
    u64 hot_nb = 0;
    bool hot_built = false, sampling = false;
    std::vector<uint8_t> key_error;              // bytes of the last KeyError key
    DevBuf drop;                                 // BPE-dropout scratch of a batch: pretoken offsets, token offsets of long pretokens
    DevBuf offs_text, offs_batch, offs_out[2];   // token offsets: lead-byte bits of a chunk; pretoken starts and token scan of a batch; spans of a chunk
    int doc_sep = -1;                            // boundary byte of the batch encode (-1: every candidate occurs in a special)
};

// grow keeping the first `used` bytes
static int grow_keep(bpe_ctx *ctx, DevBuf &b, size_t need, size_t used) {
    if (need <= b.cap) return BPE_OK;
    DevBuf nb;
    BPE_TRY(bpe_buf_reserve(ctx, nb, need + need / 2));
    if (used && b.p) {
        cudaError_t e = cudaMemcpyAsync(nb.p, b.p, used, cudaMemcpyDeviceToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) { bpe_buf_free(ctx, nb); return bpe_set_error(ctx, BPE_ERR_CUDA, "pool copy: %s", cudaGetErrorString(e)); }
    }
    bpe_buf_free(ctx, b);
    b = nb;
    return BPE_OK;
}

static EncTables enc_tables(bpe_tok *tok) {
    EncTables t;
    t.mtab = (const ulonglong2 *)tok->mtab.p; t.mmask = tok->mcap - 1;
    t.mpairs = (const int32_t *)tok->mpairs.p; t.sym_to_id = (const int32_t *)tok->sym_to_id.p;
    t.stab = (SSlot *)tok->stab.p; t.scap = tok->scap;
    t.medtab = (MSlot *)tok->medtab.p; t.medcap = tok->medcap;
    t.ltab = (LSlot *)tok->ltab.p; t.lcap = tok->lcap;
    t.text = tok->ctx->text.p ? (const uint8_t *)tok->ctx->text.p + BPE_PAD : nullptr;
    t.pool = (uint8_t *)tok->kpool.p; t.ipool = (u32 *)tok->ipool.p; t.todo = (u32 *)tok->todo.p;
    t.ctr = (u64 *)tok->ctr.p;
    t.hot = (const ulonglong2 *)tok->hot.p; t.hot_nb = tok->hot_nb; t.hval = (const u64 *)((const ulonglong2 *)tok->hot.p + 2 * tok->hot_nb);
    t.sm_img = tok->hot_built ? (const ulonglong2 *)tok->sm_img.p : nullptr;
    t.scnt = tok->sampling ? (u32 *)tok->samp.p : nullptr; t.mcnt = tok->sampling ? (u32 *)tok->samp.p + tok->scap : nullptr;
    t.bmask = nullptr; t.bpre = nullptr; t.id_offs = nullptr; t.id_base = 0;
    return t;
}

static int cache_tables_alloc(bpe_tok *tok, PtCaps cap) {
    bpe_ctx *ctx = tok->ctx;
    const u64 scap = cap.s, medcap = cap.m, lcap = cap.l;
    BPE_TRY(alloc_exact(ctx, tok->stab, scap * sizeof(SSlot)));
    BPE_TRY(alloc_exact(ctx, tok->medtab, medcap * sizeof(MSlot)));
    BPE_TRY(alloc_exact(ctx, tok->ltab, lcap * sizeof(LSlot)));
    tok->scap = scap; tok->medcap = medcap; tok->lcap = lcap;
    EncTables t = enc_tables(tok);
    KLAUNCH(k_enc_clear_tables, (unsigned)std::min<u64>((u64)ctx->sm_count * bpe_grid_mult(64), (std::max(scap, std::max(medcap, lcap)) + 255) / 256), 256, 0, ctx->stream, t);
    CUDA_TRY(ctx, cudaGetLastError());
    return BPE_OK;
}

// (Re)initialise the pretoken cache: empty tables, the specials pre-inserted with their ids.
static int cache_reset(bpe_tok *tok) {
    bpe_ctx *ctx = tok->ctx;
    cudaStream_t st = ctx->stream;
    BPE_TRY(bpe_buf_reserve(ctx, tok->ctr, 64 * sizeof(u64)));
    BPE_TRY(cache_tables_alloc(tok, pt_caps(0, 0, 0, 0, 0)));
    size_t spb = tok->sp_blob_h.size();
    BPE_TRY(bpe_buf_reserve(ctx, tok->kpool, std::max<size_t>(spb, 1) + (1 << 20)));
    BPE_TRY(bpe_buf_reserve(ctx, tok->ipool, ((size_t)tok->n_sp + (1 << 18)) * 4));
    u64 *host = (u64 *)ctx->pinned;
    for (int i = 0; i < 16; i++) host[i] = 0;
    host[4] = spb; host[7] = ~0ull;
    CUDA_TRY(ctx, cudaMemcpyAsync(tok->ctr.p, host, 128, cudaMemcpyHostToDevice, st));
    if (spb) CUDA_TRY(ctx, cudaMemcpyAsync(tok->kpool.p, tok->sp_blob_h.data(), spb, cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));    // host[] is reused below
    if (tok->n_sp > 0) {
        EncTables t = enc_tables(tok);
        KLAUNCH(k_enc_insert_specials, (tok->n_sp + 63) / 64, 64, 0, st, t, (const u32 *)tok->sp_offs.p, (const long long *)tok->sp_ids.p, tok->n_sp);
        CUDA_TRY(ctx, cudaGetLastError());
    }
    tok->cache_ready = true;
    bpe_buf_free(ctx, tok->hot); bpe_buf_free(ctx, tok->sm_img); tok->hot_nb = 0; tok->hot_built = false; tok->sampling = false;
    return BPE_OK;
}

// Build the hot table from the hit counters of the batch just looked up (values are final: the BPE kernels have run).
#define ENC_HOT_MIN_BATCH (8ull << 20)           // pretokens a batch needs for its hit counts to mean something
static int cache_build_hot(bpe_tok *tok) {
    bpe_ctx *ctx = tok->ctx;
    cudaStream_t st = ctx->stream;
    static const u64 hot_max = getenv("BPE_ENC_HOT_MAX") ? (u64)atoll(getenv("BPE_ENC_HOT_MAX")) : (1ull << 20);
    EncTables t = enc_tables(tok);               // (sampling still on: t.scnt / t.lcnt point at the counters)
    tok->sampling = false; tok->hot_built = true;
    if (!hot_max) { bpe_buf_free(ctx, tok->samp); return BPE_OK; }
    u64 *hist = (u64 *)ctx->scratch.p + 16;
    CUDA_TRY(ctx, cudaMemsetAsync(hist, 0, ENC_HOT_HIST * sizeof(u64), st));
    const unsigned grid = (unsigned)std::min<u64>((u64)ctx->sm_count * 16, (tok->scap + tok->medcap + 255) / 256);
    KLAUNCH(k_enc_hot_hist, grid, 256, 0, st, t, hist);
    u64 *host = (u64 *)ctx->pinned;
    CUDA_TRY(ctx, cudaMemcpyAsync(host, hist, ENC_HOT_HIST * sizeof(u64), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    u64 n_hot;
    const u64 thresh = fit_threshold(host, ENC_HOT_HIST, hot_max, &n_hot);
    static const bool hot_test = getenv("BPE_ENC_HOT_TEST") != nullptr;       // test knob: build it however few pretokens qualify
    if (thresh < ENC_HOT_HIST && (hot_test || n_hot >= 1024)) {
        const u64 nb = n_hot + 64;
        BPE_TRY(alloc_exact(ctx, tok->hot, nb * 48));
        CUDA_TRY(ctx, cudaMemsetAsync(tok->hot.p, 0, nb * 48, st));
        KLAUNCH(k_enc_hot_build, grid, 256, 0, st, t, (ulonglong2 *)tok->hot.p, (u64 *)((ulonglong2 *)tok->hot.p + 2 * nb), nb, (u32)thresh);
        CUDA_TRY(ctx, cudaGetLastError());
        tok->hot_nb = nb;
        static const bool prof = getenv("BPE_ENC_PROFILE") != nullptr;
        if (prof) fprintf(stderr, "  [encoder hot table: %llu pretokens looked up >= %llu times in the sampled batch, %llu buckets]\n", (unsigned long long)n_hot, (unsigned long long)thresh, (unsigned long long)nb);
    }
    // image of the lookup kernel's shared-memory cache: the most looked-up short pretokens, about three quarters of its slots
    {
        u64 *h2 = (u64 *)ctx->scratch.p + 16;
        CUDA_TRY(ctx, cudaMemsetAsync(h2, 0, 256 * sizeof(u64), st));
        const unsigned g = (unsigned)std::min<u64>((u64)ctx->sm_count * 16, (tok->scap + 255) / 256);
        KLAUNCH(k_enc_sm_hist, g, 256, 0, st, t, h2);
        CUDA_TRY(ctx, cudaMemcpyAsync(host, h2, 256 * sizeof(u64), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
        u64 acc;
        const u32 min_bucket = (u32)fit_threshold(host, 256, LK_SM_SLOTS * LK_SM_FILL_NUM / 8, &acc);
        BPE_TRY(alloc_exact(ctx, tok->sm_img, (size_t)LK_SM_SLOTS * 16));
        CUDA_TRY(ctx, cudaMemsetAsync(tok->sm_img.p, 0, (size_t)LK_SM_SLOTS * 16, st));
        if (min_bucket < 256) KLAUNCH(k_enc_sm_build, g, 256, 0, st, t, (ulonglong2 *)tok->sm_img.p, min_bucket);
        CUDA_TRY(ctx, cudaGetLastError());
    }
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    bpe_buf_free(ctx, tok->samp);
    return BPE_OK;
}

static int cache_read_ctr(bpe_tok *tok, u64 *out, int k) {
    bpe_ctx *ctx = tok->ctx;
    u64 *host = (u64 *)ctx->pinned;
    launch_peek(host, (const u64 *)tok->ctr.p, k, ctx->stream);
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < k; i++) out[i] = host[i];
    return BPE_OK;
}

// c = the counters (cache_read_ctr(tok, c, 9)); the batch can add up to new_short pretokens of <= 7 bytes and new_long longer ones
static int cache_ensure_capacity(bpe_tok *tok, const u64 *c, u64 new_short, u64 new_long) {
    bpe_ctx *ctx = tok->ctx;
    const PtCaps need = pt_caps(c[0], c[8], c[1], new_short, new_long);
    if (need.s >= (1ull << 30) || need.m >= (1ull << 30) || need.l >= (1ull << 30)) return bpe_set_error(ctx, BPE_ERR_CAPACITY, "pretoken cache would exceed 2^30 slots");
    if (need.s <= tok->scap && need.m <= tok->medcap && need.l <= tok->lcap) return BPE_OK;
    DevBuf ostab = tok->stab, omtab = tok->medtab, oltab = tok->ltab;
    u64 oscap = tok->scap, omcap = tok->medcap, olcap = tok->lcap;
    tok->stab = DevBuf(); tok->medtab = DevBuf(); tok->ltab = DevBuf();
    int rc = cache_tables_alloc(tok, {std::max(need.s, tok->scap), std::max(need.m, tok->medcap), std::max(need.l, tok->lcap)});
    if (rc == BPE_OK) {
        EncTables t = enc_tables(tok);
        auto grid_for = [&](u64 cap) { return (unsigned)std::min<u64>((u64)ctx->sm_count * bpe_grid_mult(64), (cap + 255) / 256); };
        KLAUNCH(k_enc_rehash_short, grid_for(oscap), 256, 0, ctx->stream, (const SSlot *)ostab.p, oscap, t);
        KLAUNCH(k_enc_rehash_med, grid_for(omcap), 256, 0, ctx->stream, (const MSlot *)omtab.p, omcap, t);
        KLAUNCH(k_enc_rehash_long, grid_for(olcap), 256, 0, ctx->stream, (const LSlot *)oltab.p, olcap, t);
        cudaError_t e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = bpe_set_error(ctx, BPE_ERR_CUDA, "cache rehash: %s", cudaGetErrorString(e));
    }
    for (DevBuf *b : {&ostab, &omtab, &oltab}) bpe_buf_free(ctx, *b);
    static const bool prof = getenv("BPE_ENC_PROFILE") != nullptr;       // (the growth tests read these notes)
    if (prof && rc == BPE_OK)
        fprintf(stderr, "  [encoder cache grow: short %llu -> %llu slots (%llu entries), medium %llu -> %llu (%llu), long %llu -> %llu (%llu)]\n",
                (unsigned long long)oscap, (unsigned long long)tok->scap, (unsigned long long)c[0], (unsigned long long)omcap,
                (unsigned long long)tok->medcap, (unsigned long long)c[8], (unsigned long long)olcap, (unsigned long long)tok->lcap,
                (unsigned long long)c[1]);
    return rc;
}

BPE_API int bpe_tok_create(bpe_ctx *ctx, const int32_t *merge_pairs, const int32_t *merge_result, int n_merges,
                           const int32_t *sym_to_id, const uint8_t *sym_blob, const uint64_t *sym_offs, int n_syms,
                           const uint8_t *vocab_blob, const uint64_t *vocab_offs, const int64_t *vocab_ids, int64_t n_vocab,
                           const uint8_t *specials_blob, const uint32_t *special_offs, const int64_t *special_ids, int n_specials,
                           bpe_tok **out) {
    if (out) *out = nullptr;
    if (!ctx || !out || n_merges < 0 || n_syms < 256 || !sym_to_id || !sym_offs || (n_merges > 0 && (!merge_pairs || !merge_result)) ||
        n_vocab < 0 || (n_vocab > 0 && (!vocab_offs || !vocab_ids)) || n_specials < 0 ||
        (n_specials > 0 && (!specials_blob || !special_offs || !special_ids)))
        return BPE_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    for (int j = 0; j < n_merges; j++) {
        int32_t a = merge_pairs[2 * j], b = merge_pairs[2 * j + 1];
        if ((a < 0) != (b < 0) || a >= n_syms || b >= n_syms || (a >= 0 && (merge_result[j] < 0 || merge_result[j] >= n_syms)))
            return bpe_set_error(ctx, BPE_ERR_ARG, "merge %d refers to a symbol outside [0, %d)", j, n_syms);
    }
    bpe_tok *tok = new bpe_tok();
    tok->ctx = ctx; tok->n_merges = n_merges; tok->n_syms = n_syms; tok->n_sp = n_specials;
    struct Guard { bpe_tok *t; bool ok = false; ~Guard() { if (!ok) bpe_tok_destroy(t); } } guard{tok};
    cudaStream_t st = ctx->stream;
    // merge tables
    tok->mcap = next_pow2(std::max<u64>(1024, (u64)n_merges * 2 + 2));
    BPE_TRY(bpe_buf_reserve(ctx, tok->mtab, tok->mcap * 16));
    BPE_TRY(bpe_buf_reserve(ctx, tok->mpairs, std::max<size_t>((size_t)n_merges * 8, 8)));
    BPE_TRY(bpe_buf_reserve(ctx, tok->sym_to_id, (size_t)n_syms * 4));
    DevBuf res;
    BPE_TRY(bpe_buf_reserve(ctx, res, std::max<size_t>((size_t)n_merges * 4, 4)));
    struct ResGuard { bpe_ctx *c; DevBuf &b; ~ResGuard() { bpe_buf_free(c, b); } } rg{ctx, res};
    CUDA_TRY(ctx, cudaMemsetAsync(tok->mtab.p, 0xFF, tok->mcap * 16, st));
    if (n_merges) {
        CUDA_TRY(ctx, cudaMemcpyAsync(tok->mpairs.p, merge_pairs, (size_t)n_merges * 8, cudaMemcpyHostToDevice, st));
        CUDA_TRY(ctx, cudaMemcpyAsync(res.p, merge_result, (size_t)n_merges * 4, cudaMemcpyHostToDevice, st));
        KLAUNCH(k_enc_build_ranks, (n_merges + 255) / 256, 256, 0, st, (ulonglong2 *)tok->mtab.p, tok->mcap - 1, (const int32_t *)tok->mpairs.p,
                (const int32_t *)res.p, n_merges);
        CUDA_TRY(ctx, cudaGetLastError());
    }
    CUDA_TRY(ctx, cudaMemcpyAsync(tok->sym_to_id.p, sym_to_id, (size_t)n_syms * 4, cudaMemcpyHostToDevice, st));
    tok->sym_offs_h.assign(sym_offs, sym_offs + n_syms + 1);
    if (sym_blob && sym_offs[n_syms]) tok->sym_blob_h.assign(sym_blob, sym_blob + sym_offs[n_syms]);
    long long max_id = -1;
    for (int s = 0; s < n_syms; s++) max_id = std::max<long long>(max_id, sym_to_id[s]);
    // specials
    if (n_specials) {
        tok->sp_offs_h.assign(special_offs, special_offs + n_specials + 1);
        tok->sp_blob_h.assign(specials_blob, specials_blob + special_offs[n_specials]);
        for (int i = 0; i < n_specials; i++) {
            tok->sp_max_len = std::max(tok->sp_max_len, special_offs[i + 1] - special_offs[i]);
            max_id = std::max<long long>(max_id, special_ids[i]);
        }
        BPE_TRY(bpe_buf_reserve(ctx, tok->sp_offs, (size_t)(n_specials + 1) * 4));
        BPE_TRY(bpe_buf_reserve(ctx, tok->sp_ids, (size_t)n_specials * 8));
        CUDA_TRY(ctx, cudaMemcpyAsync(tok->sp_offs.p, special_offs, (size_t)(n_specials + 1) * 4, cudaMemcpyHostToDevice, st));
        CUDA_TRY(ctx, cudaMemcpyAsync(tok->sp_ids.p, special_ids, (size_t)n_specials * 8, cudaMemcpyHostToDevice, st));
    }
    tok->max_id = max_id;
    // the batch encode's boundary byte: an ASCII value that occurs in no special token, so that no special-token match can cross a
    // boundary (it would have to contain the byte); never '\r', which the flags kernel reports as a carriage return
    {
        bool used[128] = {false};
        used['\r'] = true;
        for (uint8_t b : tok->sp_blob_h) if (b < 128) used[b] = true;
        for (int b = 0; b < 128 && tok->doc_sep < 0; b++) if (!used[b]) tok->doc_sep = b;
    }
    // decode tables: dense id -> (offset, length)
    long long n_dense = 0;
    for (int64_t i = 0; i < n_vocab; i++) {
        if (vocab_ids[i] < 0) continue;
        n_dense = std::max<long long>(n_dense, vocab_ids[i] + 1);
    }
    if (n_dense > (1ll << 28)) return bpe_set_error(ctx, BPE_ERR_UNSUPPORTED, "vocab ids up to %lld: decode table too sparse", n_dense);
    tok->n_dense = n_dense;
    {
        std::vector<u32> vlen((size_t)std::max<long long>(n_dense, 1), 0xFFFFFFFFu);
        std::vector<u64> voff((size_t)std::max<long long>(n_dense, 1), 0);
        for (int64_t i = 0; i < n_vocab; i++) {
            if (vocab_ids[i] < 0) continue;
            vlen[vocab_ids[i]] = (u32)(vocab_offs[i + 1] - vocab_offs[i]);   // later entries win, like a dict
            voff[vocab_ids[i]] = vocab_offs[i];
        }
        size_t vb = n_vocab ? (size_t)vocab_offs[n_vocab] : 0;
        BPE_TRY(bpe_buf_reserve(ctx, tok->vlen, vlen.size() * 4)); BPE_TRY(bpe_buf_reserve(ctx, tok->voff, voff.size() * 8));
        BPE_TRY(bpe_buf_reserve(ctx, tok->vblob, std::max<size_t>(vb, 1)));
        CUDA_TRY(ctx, cudaMemcpyAsync(tok->vlen.p, vlen.data(), vlen.size() * 4, cudaMemcpyHostToDevice, st));
        CUDA_TRY(ctx, cudaMemcpyAsync(tok->voff.p, voff.data(), voff.size() * 8, cudaMemcpyHostToDevice, st));
        if (vb) CUDA_TRY(ctx, cudaMemcpyAsync(tok->vblob.p, vocab_blob, vb, cudaMemcpyHostToDevice, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));    // the host vectors go out of scope
    }
    BPE_TRY(cache_reset(tok));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    guard.ok = true;
    *out = tok;
    return BPE_OK;
}

BPE_API void bpe_tok_destroy(bpe_tok *tok) {
    if (!tok) return;
    if (tok->ctx) { cudaSetDevice(tok->ctx->device); cudaStreamSynchronize(tok->ctx->stream); }
    for (DevBuf *b : {&tok->mtab, &tok->mpairs, &tok->sym_to_id, &tok->vlen, &tok->voff, &tok->vblob, &tok->sp_offs, &tok->sp_ids,
                      &tok->stab, &tok->medtab, &tok->ltab, &tok->kpool, &tok->ipool, &tok->todo, &tok->ctr, &tok->hot, &tok->samp, &tok->sm_img, &tok->drop,
                      &tok->offs_text, &tok->offs_batch, &tok->offs_out[0], &tok->offs_out[1]})
        bpe_buf_free(tok->ctx, *b);
    delete tok;
}

BPE_API int bpe_tok_cache_reset(bpe_tok *tok) {
    if (!tok) return BPE_ERR_ARG;
    CUDA_TRY(tok->ctx, cudaSetDevice(tok->ctx->device));
    BPE_TRY(cache_reset(tok));
    CUDA_TRY(tok->ctx, cudaStreamSynchronize(tok->ctx->stream));
    return BPE_OK;
}

BPE_API int bpe_tok_saw_cr(bpe_tok *tok) { return tok && tok->ctx && tok->ctx->saw_cr_encode ? 1 : 0; }

BPE_API int bpe_tok_key_error(bpe_tok *tok, uint8_t *buf, uint64_t cap, uint64_t *len) {
    if (!tok || !len) return BPE_ERR_ARG;
    *len = tok->key_error.size();
    if (buf) memcpy(buf, tok->key_error.data(), (size_t)std::min<u64>(cap, tok->key_error.size()));
    return BPE_OK;
}

#define ENC_BATCH_BYTES (256ull << 20)
#define ENC_CACHE_MAX_ENTRIES (384ull << 20)

// Document boundaries of a batch encode's chunk: bit per arena byte; id_offs[j] gets id_base + the offset of the first id after
// the chunk's document j.
struct DocBounds { const u32 *bmask; u64 *id_offs; u64 id_base; };

// Encode the n bytes in the context's text arena into out_dev (device pointer, may be null: count only).
// *n_out = number of tokens (may exceed dev_cap; only dev_cap are written).  stats, when given, are ADDED to.
// drop (BPE-dropout, or null): its thr, seed_mix, lo, doffs and da; the rest is filled in per batch.
// offs (token offsets, or null; needs out_dev): its chars, out, lo, doffs, da and carry; on return carry = that of the next chunk, whose first
// document starts at arena byte next_ds (next_keep: it is this chunk's first one, which continues).
static int encode_core(bpe_tok *tok, u64 n, int out_dtype, void *out_dev, u64 dev_cap, uint64_t *n_out, bpe_encode_stats *stats,
                       const DocBounds *docs = nullptr, const EncDrop *drop = nullptr, EncOffs *offs = nullptr, u64 next_ds = 0,
                       bool next_keep = false) {
    bpe_ctx *ctx = tok->ctx;
    cudaStream_t st = ctx->stream;
    *n_out = 0;
    EvTimer tm(ctx, 8);                           // (the callers' timers use events 0..7)
    int e1 = tm.mark();
    const uint8_t *spb; const u32 *spo; u32 spmax;
    BPE_TRY(ctx_upload_specials(ctx, tok->sp_blob_h.data(), tok->sp_offs_h.data(), tok->n_sp, &spb, &spo, &spmax));
    u64 nn = n;
    BPE_TRY(ctx_run_flags(ctx, &nn, false, spb, spo, tok->n_sp, spmax, 0, ~0ull, docs ? docs->bmask : nullptr));
    ctx->saw_cr_encode |= ctx->saw_cr;
    // ordinal of the first pretoken of every GROUP of 16 flag words (512 bytes of text = one warp step of the lookup kernel, which
    // gets the ordinals inside a step from a warp scan): a scan over N / 512 entries instead of N / 32
    const u64 nw = (n + 31) / 32, ng = (nw + 15) / 16;
    size_t cnt_b = round_up((ng + 1) * sizeof(u32), 256), pre_b = round_up((ng + 2) * sizeof(u64), 256);
    const size_t bpre_b = docs ? pre_b : 0;
    BPE_TRY(bpe_buf_reserve(ctx, ctx->tmp0, cnt_b + pre_b + bpre_b + scan_tmp_elems_host(ng) * sizeof(u64)));
    u32 *cnt = (u32 *)ctx->tmp0.p;
    u64 *pre = (u64 *)((uint8_t *)ctx->tmp0.p + cnt_b);
    u64 *bpre = (u64 *)((uint8_t *)ctx->tmp0.p + cnt_b + pre_b);
    u64 *scan_tmp = (u64 *)((uint8_t *)ctx->tmp0.p + cnt_b + pre_b + bpre_b);
    launch_popc_words16((const u32 *)ctx->flags.p, ng, cnt, ctx->sm_count, st);
    launch_scan_u32(cnt, ng, pre, scan_tmp, st);
    if (docs) {                                  // the same per group for the boundary bits: document index of a boundary
        launch_popc_words16(docs->bmask, ng, cnt, ctx->sm_count, st);
        launch_scan_u32(cnt, ng, bpre, scan_tmp, st);
    }
    EncOffs o{};
    if (offs) {                                  // lead-byte bits and their count per group: character indices
        o = *offs;
        const u64 lw = 16 * (ng + 1);
        BPE_TRY(bpe_buf_reserve(ctx, tok->offs_text, lw * sizeof(u32) + (ng + 2) * sizeof(u64)));
        u32 *lmask = (u32 *)tok->offs_text.p;
        u64 *lpre = (u64 *)(lmask + lw);
        KLAUNCH(k_enc_lead_bits, (unsigned)std::min<u64>((u64)ctx->sm_count * 16, (lw + 255) / 256), 256, 0, st,
                (const uint8_t *)ctx->text.p + BPE_PAD, n, lw, lmask);
        launch_popc_words16(lmask, ng, cnt, ctx->sm_count, st);
        launch_scan_u32(cnt, ng, lpre, scan_tmp, st);
        o.lmask = lmask; o.lpre = lpre;
        o.vlen = (const u32 *)tok->vlen.p; o.n_dense = (u64)tok->n_dense;
    }
    CUDA_TRY(ctx, cudaGetLastError());
    // (test knobs: BPE_ENC_BATCH_KB = batch size, BPE_ENC_HOT_MIN = pretokens a batch needs to be sampled for the hot table,
    // BPE_ENC_CACHE_MAX = cache entries above which the cache is dropped between two batches)
    static const u64 batch_bytes = getenv("BPE_ENC_BATCH_KB") ? std::max<u64>(1, (u64)atoll(getenv("BPE_ENC_BATCH_KB"))) << 10 : ENC_BATCH_BYTES;
    static const u64 hot_min_batch = getenv("BPE_ENC_HOT_MIN") ? (u64)atoll(getenv("BPE_ENC_HOT_MIN")) : ENC_HOT_MIN_BATCH;
    static const u64 cache_max = getenv("BPE_ENC_CACHE_MAX") ? (u64)atoll(getenv("BPE_ENC_CACHE_MAX")) : ENC_CACHE_MAX_ENTRIES;
    static const bool prof = getenv("BPE_ENC_PROFILE") != nullptr;
    const u64 words_per_batch = batch_bytes / 32;
    // batch boundaries (flag words).  While the hot table is still to be built the first batch is a small one (64 MB: enough pretokens
    // to sample), so that the cold start -- every lookup a probe of the big tables -- is over after a quarter of a normal batch.
    std::vector<u64> bw{0};
    if (nw) {
        u64 w = std::min(nw, tok->hot_built ? words_per_batch : std::min<u64>(words_per_batch, (64ull << 20) / 32));
        bw.push_back(w);
        while (w < nw) { w = std::min(nw, w + words_per_batch); bw.push_back(w); }
    }
    const u64 n_batches = bw.size() - 1;
    std::vector<u64> ord(n_batches + 1, 0);
    {
        u64 *host = (u64 *)ctx->pinned;          // (kernel writes into page-locked memory: no copy engine, see launch_peek)
        if ((n_batches + 1) * 8 > ctx->pinned_cap) return bpe_set_error(ctx, BPE_ERR_UNSUPPORTED, "text too large for one call (%llu batches)", (unsigned long long)n_batches);
        for (u64 b = 0; b <= n_batches; b++) launch_peek(host + b, pre + (bw[b] + 15) / 16, 1, st);   // (boundaries are multiples of 16 words, or the end)
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
        for (u64 b = 0; b <= n_batches; b++) ord[b] = host[b];
    }
    int e2 = tm.mark();
    const u64 n_pretok = ord[n_batches];
    if (!tok->cache_ready) BPE_TRY(cache_reset(tok));

    float ms_lookup = 0, ms_bpe = 0, ms_emit = 0;
    u64 total_tokens = 0, new_unique = 0;
    u64 c[16];
    cudaEvent_t evs[4];
    for (auto &e : evs) CUDA_TRY(ctx, cudaEventCreate(&e));
    struct EvGuard { cudaEvent_t *e; ~EvGuard() { for (int i = 0; i < 4; i++) cudaEventDestroy(e[i]); } } evg{evs};
    for (u64 b = 0; b < n_batches; b++) {
        const u64 b_lo = bw[b], b_hi = bw[b + 1];
        const u64 bound = ord[b + 1] - ord[b];
        const u64 bytes = (b_hi - b_lo) * 32;
        BPE_TRY(cache_read_ctr(tok, c, 9));
        if (c[0] + c[1] + c[8] + bound > cache_max && c[0] + c[1] + c[8] > (u64)tok->n_sp) {
            if (prof) fprintf(stderr, "  [encoder cache reset: %llu entries + up to %llu new > %llu, before batch %llu of %llu]\n",
                              (unsigned long long)(c[0] + c[1] + c[8]), (unsigned long long)bound, (unsigned long long)cache_max,
                              (unsigned long long)b, (unsigned long long)n_batches);
            BPE_TRY(cache_reset(tok));
            BPE_TRY(cache_read_ctr(tok, c, 9));
        }
        BPE_TRY(cache_ensure_capacity(tok, c, bound, std::min(bound, bytes / (SHORT_MAX + 1) + 1)));
        BPE_TRY(grow_keep(ctx, tok->kpool, c[4] + bytes + 64, c[4]));
        BPE_TRY(grow_keep(ctx, tok->ipool, (c[5] + bytes + 64) * 4, c[5] * 4));
        BPE_TRY(bpe_buf_reserve(ctx, tok->todo, std::max<size_t>(bound * 4, 16)));
        // per-pretoken values of the batch; tile states of the scan
        const u64 n_tiles = (bound + SE_TILE - 1) / SE_TILE;
        size_t slot_b = round_up((bound + 1) * 8, 256), st_b = round_up((n_tiles + 4) * 8, 256);          // tile states, ticket, batch total
        BPE_TRY(bpe_buf_reserve(ctx, ctx->tmp1, slot_b + st_b));
        u64 *vals = (u64 *)ctx->tmp1.p;
        u64 *stmp = (u64 *)((uint8_t *)ctx->tmp1.p + slot_b);
        CUDA_TRY(ctx, cudaMemsetAsync((u64 *)tok->ctr.p + 2, 0, 8, st));
        if (!tok->hot_built && bound >= hot_min_batch) {      // this batch's lookups are counted per slot; the hot table follows it
            BPE_TRY(bpe_buf_reserve(ctx, tok->samp, (tok->scap + tok->medcap) * 4));
            CUDA_TRY(ctx, cudaMemsetAsync(tok->samp.p, 0, (tok->scap + tok->medcap) * 4, st));
            tok->sampling = true;
        }
        EncTables t = enc_tables(tok);
        if (docs) { t.bmask = docs->bmask; t.bpre = bpre; t.id_offs = docs->id_offs; t.id_base = docs->id_base; }
        const u64 base = b_lo * 32;
        CUDA_TRY(ctx, cudaEventRecord(evs[0], st));
        if (bound) {
            const u64 c_lo = b_lo * 2, c_hi = std::min(b_hi * 2, (n + 15) / 16);
            const u64 steps = (c_hi - c_lo + 32 * LK_WARPS * LK_TICKET - 1) / (32 * LK_WARPS * LK_TICKET);
            CUDA_TRY(ctx, cudaMemsetAsync((u64 *)tok->ctr.p + 9, 0, 8, st));
            static bool attr_set = false;
            if (!attr_set) {
                CUDA_TRY(ctx, cudaFuncSetAttribute((void *)k_enc_lookup<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LK_DYN_SMEM));
                CUDA_TRY(ctx, cudaFuncSetAttribute((void *)k_enc_lookup<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LK_DYN_SMEM));
                attr_set = true;
            }
            const unsigned lgrid = (unsigned)std::max<u64>(1, std::min<u64>((u64)ctx->sm_count, steps));
            if (docs) KLAUNCH(k_enc_lookup<true>, lgrid, LK_NT, LK_DYN_SMEM, st, t, (const u32 *)ctx->flags.p, pre, ord[b], c_lo, c_hi, n, base, vals);
            else KLAUNCH(k_enc_lookup<false>, lgrid, LK_NT, LK_DYN_SMEM, st, t, (const u32 *)ctx->flags.p, pre, ord[b], c_lo, c_hi, n, base, vals);
        }
        CUDA_TRY(ctx, cudaGetLastError());
        CUDA_TRY(ctx, cudaEventRecord(evs[1], st));
        BPE_TRY(cache_read_ctr(tok, c, 8));
        if (c[3]) return bpe_set_error(ctx, BPE_ERR_CAPACITY, "pretoken cache overflow");
        if (c[6]) return bpe_set_error(ctx, BPE_ERR_UNSUPPORTED, "a pretoken longer than %u bytes", MAX_TOKEN_LEN);
        const u64 n_todo = c[2];
        new_unique += n_todo;
        if (n_todo) {
            unsigned g2 = (unsigned)std::min<u64>((u64)ctx->sm_count * bpe_grid_mult(64), (n_todo + 7) / 8);
            unsigned g1 = (unsigned)std::min<u64>((u64)ctx->sm_count * bpe_grid_mult(64), (n_todo + BPT_NT - 1) / BPT_NT);
            KLAUNCH((k_enc_bpe_short<16u, false>), g1, BPT_NT, 0, st, t, n_todo);
            KLAUNCH((k_enc_bpe_short<BPT_MAX, true>), g1, BPT_NT, 0, st, t, n_todo);
            KLAUNCH(k_enc_bpe, g2, 256, 0, st, t, n_todo);
            CUDA_TRY(ctx, cudaGetLastError());
        }
        if (tok->sampling) BPE_TRY(cache_build_hot(tok));
        if (drop && bound) {                     // BPE-dropout: every occurrence's own BPE replaces its cached value
            BPE_TRY(cache_read_ctr(tok, c, 6));  // id pool cursor after the cache BPE: the batch's id scratch starts there
            const u64 span = std::min<u64>(n - base, bytes + MAX_TOKEN_LEN);      // (the batch's last pretoken may run past its end)
            BPE_TRY(grow_keep(ctx, tok->ipool, (c[5] + span) * 4, c[5] * 4));
            t.ipool = (u32 *)tok->ipool.p;
            const size_t starts_b = round_up(bound * 8, 256);
            BPE_TRY(bpe_buf_reserve(ctx, tok->drop, starts_b + span * 4));
            EncDrop d = *drop;
            d.skip = tok->n_sp > 0 && spmax > 0 ? (const u32 *)ctx->spstart.p : docs ? docs->bmask : nullptr;
            d.starts = (const u64 *)tok->drop.p;
            d.loff = (u32 *)((uint8_t *)tok->drop.p + starts_b);
            d.ibase = c[5];
            CUDA_TRY(ctx, cudaMemsetAsync((u64 *)tok->ctr.p + 10, 0, 8, st));
            const unsigned gmax = (unsigned)((u64)ctx->sm_count * bpe_grid_mult(64));
            KLAUNCH(k_enc_drop_starts, (unsigned)std::min<u64>(gmax, (b_hi - b_lo + 255) / 256), 256, 0, st, (const u32 *)ctx->flags.p, pre, ord[b],
                    b_lo, b_hi, (u64 *)tok->drop.p);
            KLAUNCH(k_enc_drop_short, (unsigned)std::min<u64>(gmax, (bound + BPT_NT - 1) / BPT_NT), BPT_NT, 0, st, t, d, (const u32 *)ctx->flags.p,
                    n, base, bound, vals);
            KLAUNCH(k_enc_drop_warp, (unsigned)ctx->sm_count * 8, 256, 0, st, t, d, (const u32 *)ctx->flags.p, n, base, bound, vals);
            CUDA_TRY(ctx, cudaGetLastError());
        }
        CUDA_TRY(ctx, cudaEventRecord(evs[2], st));
        // tokens per pretoken -> offsets -> ids, one pass
        u64 *host = (u64 *)ctx->pinned;
        {
            u64 *tile_state = stmp, *total_dev = stmp + n_tiles + 2;
            u32 *ticket = (u32 *)(stmp + n_tiles + 1);
            CUDA_TRY(ctx, cudaMemsetAsync(stmp, 0, (n_tiles + 4) * 8, st));
            const bool emit = out_dev && total_tokens < dev_cap;
            if (bound) {
                if (!emit) KLAUNCH((k_enc_scan_emit<uint16_t, false>), (unsigned)n_tiles, SE_NT, 0, st, t, vals, bound, ord[b], tile_state, ticket, (uint16_t *)nullptr, total_tokens, dev_cap, total_dev);
                else if (out_dtype == BPE_DTYPE_U16) KLAUNCH((k_enc_scan_emit<uint16_t, true>), (unsigned)n_tiles, SE_NT, 0, st, t, vals, bound, ord[b], tile_state, ticket, (uint16_t *)out_dev, total_tokens, dev_cap, total_dev);
                else KLAUNCH((k_enc_scan_emit<int32_t, true>), (unsigned)n_tiles, SE_NT, 0, st, t, vals, bound, ord[b], tile_state, ticket, (int32_t *)out_dev, total_tokens, dev_cap, total_dev);
            }
            CUDA_TRY(ctx, cudaGetLastError());
            launch_peek(host, total_dev, 1, st);
        }
        if (offs && bound) {                     // token offsets, while the batch's values are resident
            const size_t starts_b = round_up(bound * 8, 256), cnt_b2 = round_up(bound * 4, 256), tpre_b = round_up((bound + 1) * 8, 256);
            BPE_TRY(bpe_buf_reserve(ctx, tok->offs_batch, starts_b + cnt_b2 + tpre_b + scan_tmp_elems_host(bound) * sizeof(u64)));
            uint8_t *ob = (uint8_t *)tok->offs_batch.p;
            u64 *starts = (u64 *)ob, *tpre = (u64 *)(ob + starts_b + cnt_b2), *otmp = (u64 *)(ob + starts_b + cnt_b2 + tpre_b);
            u32 *ocnt = (u32 *)(ob + starts_b);
            const unsigned gmax = (unsigned)((u64)ctx->sm_count * bpe_grid_mult(64));
            const unsigned gq = (unsigned)std::min<u64>(gmax, (bound + 255) / 256);
            KLAUNCH(k_enc_drop_starts, (unsigned)std::min<u64>(gmax, (b_hi - b_lo + 255) / 256), 256, 0, st, (const u32 *)ctx->flags.p, pre, ord[b],
                    b_lo, b_hi, starts);
            KLAUNCH(k_enc_off_count, gq, 256, 0, st, t, vals, bound, ocnt);
            launch_scan_u32(ocnt, bound, tpre, otmp, st);
            o.starts = starts; o.tpre = tpre;
            if (o.chars) KLAUNCH(k_enc_offsets<true>, gq, 256, 0, st, t, o, (const u32 *)ctx->flags.p, vals, n, bound, total_tokens, dev_cap);
            else KLAUNCH(k_enc_offsets<false>, gq, 256, 0, st, t, o, (const u32 *)ctx->flags.p, vals, n, bound, total_tokens, dev_cap);
            CUDA_TRY(ctx, cudaGetLastError());
        }
        launch_peek(host + 1, (u64 *)tok->ctr.p + 7, 1, st);
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
        const u64 batch_tokens = host[0], err_ord = host[1];
        if (err_ord != ~0ull) {
            // KeyError (tokenizer.py:120,135): report the key of the first failing pretoken in text order.  Its byte offset: the
            // flag word that holds that ordinal (binary search in the scanned word counts), then the matching start bit.
            u64 hv[2] = {0, 0};
            u64 lo = 0, hi = ng;                 // largest group g with pre[g] <= err_ord
            while (hi - lo > 1) {
                const u64 mid = lo + (hi - lo) / 2; u64 pm = 0;
                CUDA_TRY(ctx, cudaMemcpy(&pm, pre + mid, 8, cudaMemcpyDeviceToHost));
                if (pm <= err_ord) lo = mid; else hi = mid;
            }
            u64 hpre = 0; u32 hfl[16];
            CUDA_TRY(ctx, cudaMemcpy(&hpre, pre + lo, 8, cudaMemcpyDeviceToHost));
            CUDA_TRY(ctx, cudaMemcpy(hfl, (const u32 *)ctx->flags.p + 16 * lo, sizeof(hfl), cudaMemcpyDeviceToHost));
            u64 err_pos = 16 * lo * 32, skip = err_ord - hpre;
            for (int k = 0; k < 16; k++) {
                const u64 pc = (u64)__builtin_popcount(hfl[k]);
                if (skip >= pc) { skip -= pc; continue; }
                u32 f = hfl[k];
                while (skip--) f &= f - 1;
                err_pos = (16 * lo + k) * 32 + (u64)__builtin_ctz(f);
                break;
            }
            CUDA_TRY(ctx, cudaMemcpy(&hv[0], vals + (err_ord - ord[b]), 8, cudaMemcpyDeviceToHost));
            if (VAL_TAG(hv[0]) == VAL_FWD) {     // a forward reference: the value sits in the slot
                const u32 ref = (u32)hv[0];
                const void *src = (ref & REF_LONG) ? (const void *)&((const LSlot *)tok->ltab.p)[REF_SLOT(ref)].val
                                : (ref & REF_MED) ? (const void *)&((const MSlot *)tok->medtab.p)[REF_SLOT(ref)].val
                                                  : (const void *)&((const SSlot *)tok->stab.p)[ref].val;
                CUDA_TRY(ctx, cudaMemcpy(&hv[0], src, 8, cudaMemcpyDeviceToHost));
            }
            u32 sym = (u32)hv[0];
            tok->key_error.clear();
            if (sym & 0x80000000u) {
                u32 i = sym & 0x7FFFFFFFu;
                if ((int)i < tok->n_sp) tok->key_error.assign(tok->sp_blob_h.begin() + tok->sp_offs_h[i], tok->sp_blob_h.begin() + tok->sp_offs_h[i + 1]);
            } else if ((int)sym < tok->n_syms && !tok->sym_blob_h.empty()) {
                tok->key_error.assign(tok->sym_blob_h.begin() + tok->sym_offs_h[sym], tok->sym_blob_h.begin() + tok->sym_offs_h[sym + 1]);
            }
            u64 reset7 = ~0ull;
            CUDA_TRY(ctx, cudaMemcpy((u64 *)tok->ctr.p + 7, &reset7, 8, cudaMemcpyHostToDevice));
            ctx->err_detail = (int64_t)err_pos;
            return bpe_set_error(ctx, BPE_ERR_KEY, "KeyError: a token of the pretoken at byte %llu is not in the vocabulary", (unsigned long long)err_pos);
        }
        CUDA_TRY(ctx, cudaEventRecord(evs[3], st));
        CUDA_TRY(ctx, cudaEventSynchronize(evs[3]));
        float f;
        cudaEventElapsedTime(&f, evs[0], evs[1]); ms_lookup += f;
        cudaEventElapsedTime(&f, evs[1], evs[2]); ms_bpe += f;
        cudaEventElapsedTime(&f, evs[2], evs[3]); ms_emit += f;
        total_tokens += batch_tokens;
    }
    if (offs) {                                  // characters of the next chunk's first document in this one
        u64 *host = (u64 *)ctx->pinned;
        KLAUNCH(k_enc_lead_span, 1, 1, 0, st, o.lmask, o.lpre, next_keep ? 0 : std::min(next_ds, n), n, host);
        CUDA_TRY(ctx, cudaGetLastError());
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
        offs->carry = (next_keep ? offs->carry : 0) + host[0];
    }
    int e3 = tm.mark();
    *n_out = total_tokens;
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    if (stats) {
        stats->n_bytes += n; stats->n_pretokens += n_pretok; stats->n_tokens += total_tokens; stats->cache_new_unique += new_unique;
        stats->ms_pretok += tm.ms(e1, e2); stats->ms_lookup += ms_lookup; stats->ms_bpe += ms_bpe;
        stats->ms_emit += ms_emit; stats->ms_total += tm.ms(e1, e3);
    }
    return BPE_OK;
}

static int encode_check_args(bpe_tok *tok, const uint8_t *text, u64 n, int out_dtype, uint64_t *n_out) {
    if (!tok || (!text && n) || !n_out || (out_dtype != BPE_DTYPE_U16 && out_dtype != BPE_DTYPE_I32)) return BPE_ERR_ARG;
    bpe_ctx *ctx = tok->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    if (out_dtype == BPE_DTYPE_U16 && tok->max_id > 65535)
        return bpe_set_error(ctx, BPE_ERR_ARG, "vocabulary ids go up to %lld: they do not fit uint16 output", tok->max_id);
    *n_out = 0;
    return BPE_OK;
}

#define ENC_PIPE_CHUNK (256ull << 20)
#define ENC_PIPE_MIN (96ull << 20)
#define ENC_CUT_WINDOW (8ull << 20)

static u64 find_exact_cut(const bpe_tok *tok, const uint8_t *t, u64 n, u64 nominal) {
    return exact_cut_host(t, n, nominal, ENC_CUT_WINDOW, tok->sp_blob_h.data(), tok->sp_offs_h.data(), tok->n_sp);
}

// ---- batch encode: a chunk of documents into the text arena, one boundary byte after every document that ends in it ----------
// ends[j] - lo = where document j ends in the chunk (ascending, 0..len).  Byte i of the chunk goes to i + #{j : ends[j] - lo <= i},
// the boundary after document j to ends[j] - lo + j, which also sets its bit in bmask (zeroed by the caller).  A warp takes 512
// bytes at a time, 32 consecutive bytes per instruction; the boundaries inside them (usually none) come from a binary search.
__device__ __forceinline__ u64 ends_lower_bound(const u64 *__restrict__ e, u64 lo, u64 hi, u64 x) {      // first index with e >= x
    while (lo < hi) { const u64 m = (lo + hi) >> 1; if (__ldg(&e[m]) < x) lo = m + 1; else hi = m; }
    return lo;
}
__global__ void __launch_bounds__(256) k_enc_expand_docs(const uint8_t *__restrict__ src, u64 len, const u64 *__restrict__ ends, u64 n_ends,
                                                        u64 lo, uint8_t *__restrict__ arena, u32 *__restrict__ bmask, uint8_t sep) {
    const u32 lane = lane_id();
    const u64 gw = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((u64)gridDim.x * blockDim.x) >> 5;
    for (u64 w0 = gw * 512; w0 < len; w0 += nw * 512) {
        const u64 r = ends_lower_bound(ends, 0, n_ends, lo + w0), r1 = ends_lower_bound(ends, r, n_ends, lo + w0 + 512);
        for (u32 k = 0; k < 16; k++) {
            const u64 i = w0 + k * 32 + lane;
            if (i >= len) break;
            const u64 rank = r1 > r ? ends_lower_bound(ends, r, r1, lo + i + 1) : r;
            arena[i + rank] = src[i];
        }
    }
    for (u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x; j < n_ends; j += (u64)gridDim.x * blockDim.x) {
        const u64 p = ends[j] - lo + j;
        arena[p] = sep;
        atomicOr(&bmask[p >> 5], 1u << (p & 31));
    }
}

// A pipeline chunk: bytes [lo, hi) of the caller's text; documents [da, db) end inside it.
struct EncChunk { u64 lo, hi, da, db; };

// The pipeline's chunks: cut at a document end near every multiple of the nominal size; a document that runs well past it is cut
// at an exact boundary inside it (find_exact_cut on the document alone), or else stays whole.  bpe_encode: one document.
static std::vector<EncChunk> doc_chunks(const bpe_tok *tok, const uint8_t *t, u64 n, const uint64_t *doc_offs, u64 n_docs, u64 chunk) {
    std::vector<EncChunk> out;
    u64 lo = 0, d = 0;
    while (n >= ENC_PIPE_MIN && n - lo > chunk + chunk / 2) {
        const u64 target = lo + chunk;
        const u64 j = (u64)(std::upper_bound(doc_offs + 1 + d, doc_offs + 1 + n_docs, target) - (doc_offs + 1));   // docs [d, j) end <= target
        const u64 e = j > d ? doc_offs[j] : lo;
        u64 hi, nd;
        if (e >= lo + chunk / 2) { hi = e; nd = j; }
        else {
            const u64 ds = doc_offs[j], c = find_exact_cut(tok, t + ds, doc_offs[j + 1] - ds, target - ds);   // (ds < target: j does not end by it)
            if (c && ds + c > lo) { hi = ds + c; nd = j; }
            else if (e > lo) { hi = e; nd = j; }
            else if (doc_offs[j + 1] == n) break;    // the rest is this document: one piece
            else { hi = doc_offs[j + 1]; nd = j + 1; }
        }
        out.push_back({lo, hi, d, nd});
        lo = hi; d = nd;
    }
    out.push_back({lo, n, d, n_docs});
    return out;
}

// ---- host entry points: chunks cut at exact boundaries, double-buffered so that the upload of chunk k+1 and the download of
// chunk k-1 run while chunk k is encoded.  doc_offs (batch encode) or null (one document).
//   one document: a chunk is uploaded straight into the arena the kernels read next (the two arenas alternate)
//   batch encode: a chunk is uploaded as it is into one of two staging buffers; on the compute stream k_enc_expand_docs moves it
//                 into the arena with a boundary byte after every document and sets the boundary bitmask
// drop: BPE-dropout (thr and seed_mix set), or null.  offs_out (with out): the tokens' spans in `unit` (BPE_OFF_*), downloaded with the ids.
static int encode_pipeline(bpe_tok *tok, const uint8_t *text_host, uint64_t n, const uint64_t *doc_offs, uint64_t n_docs, int out_dtype,
                           void *out, uint64_t cap, uint64_t *n_out, uint64_t *id_offs_out, bpe_encode_stats *stats,
                           const EncDrop *drop = nullptr, int unit = BPE_OFF_BYTES, int64_t *offs_out = nullptr) {
    BPE_TRY(encode_check_args(tok, text_host, n, out_dtype, n_out));
    bpe_ctx *ctx = tok->ctx;
    cudaStream_t st = ctx->stream;
    ctx->saw_cr_encode = false;
    if (stats) memset(stats, 0, sizeof(*stats));
    const size_t esz = out_dtype == BPE_DTYPE_U16 ? 2 : 4;
    u64 chunk = ENC_PIPE_CHUNK;
    if (const char *e = getenv("BPE_ENCODE_CHUNK_MB")) chunk = std::max<u64>(1, strtoull(e, nullptr, 10)) << 20;
    const uint64_t one_doc[2] = {0, n};
    const std::vector<EncChunk> chunks = doc_offs ? doc_chunks(tok, text_host, n, doc_offs, n_docs, chunk)
                                                  : doc_chunks(tok, text_host, n, one_doc, 1, chunk);
    const size_t m = chunks.size();
    BPE_TRY(ctx_pipeline_init(ctx));
    u64 *id_dev = nullptr;
    if (doc_offs) {                              // document offsets up; id offsets come back in the second half of the buffer
        BPE_TRY(bpe_buf_reserve(ctx, ctx->doc_offs, (n_docs + 1) * 16));
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->doc_offs.p, doc_offs, (n_docs + 1) * 8, cudaMemcpyHostToDevice, st));
        id_dev = (u64 *)ctx->doc_offs.p + (n_docs + 1);
    }
    EvTimer tm(ctx);
    int e0 = tm.mark();
    DevBuf *tbuf[2] = {&ctx->text, &ctx->text_alt};     // one document: the two arenas
    DevBuf *sbuf[2] = {&ctx->text_alt, &ctx->doc_stage};   // batch encode: the two staging buffers (the arena is ctx->text)
    DevBuf *obuf[2] = {&ctx->out_a, &ctx->out_b};
    u64 max_chunk = 0;
    for (const EncChunk &c : chunks) max_chunk = std::max(max_chunk, c.hi - c.lo);
    auto upload = [&](size_t k, DevBuf &dst) -> int {     // chunk k -> arena (staging buffer) dst, on the copy-in stream
        const u64 len = chunks[k].hi - chunks[k].lo;
        if (doc_offs) BPE_TRY(bpe_buf_reserve(ctx, dst, std::max<u64>(max_chunk, 16)));
        else {
            BPE_TRY(ctx_prepare_arena(ctx, dst, m > 1 ? max_chunk : len, ctx->s_in));
            if (m > 1 && len < max_chunk)         // bytes between this chunk's end and the arena padding must read as padding
                CUDA_TRY(ctx, cudaMemsetAsync((uint8_t *)dst.p + BPE_PAD + len, BPE_BYTE_PAD, max_chunk - len, ctx->s_in));
        }
        uint8_t *p = (uint8_t *)dst.p + (doc_offs ? 0 : BPE_PAD);
        if (len) CUDA_TRY(ctx, cudaMemcpyAsync(p, text_host + chunks[k].lo, len, cudaMemcpyHostToDevice, ctx->s_in));
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_in[k & 1], ctx->s_in));
        return BPE_OK;
    };
    // (the compute stream must not run ahead of pool (re)allocations done for the other buffer: everything below that
    // touches a buffer is ordered by events, and every chunk ends with a host-side synchronisation of the compute stream)
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    BPE_TRY(upload(0, doc_offs ? *sbuf[0] : *tbuf[0]));
    u64 total = 0, char_carry = 0;
    int rc = BPE_OK;
    const bool want_offs = out && offs_out;
    for (size_t k = 0; k < m && rc == BPE_OK; k++) {
        const int cur = (int)(k & 1);
        const EncChunk &ch = chunks[k];
        const u64 len = ch.hi - ch.lo;
        if (k + 1 < m) { rc = upload(k + 1, doc_offs ? *sbuf[cur ^ 1] : *tbuf[cur ^ 1]); if (rc != BPE_OK) break; }
        const bool swap = !doc_offs && cur == 1;
        if (swap) std::swap(ctx->text, ctx->text_alt);            // the arena the kernels read is always ctx->text
        CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_in[cur], 0));
        void *odev = nullptr;
        if (out) {
            rc = bpe_buf_reserve(ctx, *obuf[cur], std::max<size_t>((m > 1 ? max_chunk : len) * esz, 16));
            if (rc != BPE_OK) { if (swap) std::swap(ctx->text, ctx->text_alt); break; }
            if (want_offs) rc = bpe_buf_reserve(ctx, tok->offs_out[cur], std::max<size_t>((m > 1 ? max_chunk : len) * 16, 16));
            if (rc != BPE_OK) { if (swap) std::swap(ctx->text, ctx->text_alt); break; }
            CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_out[cur], 0));   // its previous download has finished
            odev = obuf[cur]->p;
        }
        // token offsets: the chunk's place in the caller's text; the next chunk's first document (ch.db) starts in this one unless none ends here
        EncOffs och{};
        const uint64_t *dofs = doc_offs ? doc_offs : one_doc;
        if (want_offs) {
            och.chars = unit == BPE_OFF_CHARS; och.out = (long long *)tok->offs_out[cur].p; och.lo = ch.lo; och.da = ch.da; och.carry = char_carry;
            och.doffs = doc_offs ? (const u64 *)ctx->doc_offs.p : nullptr;
        }
        EncOffs *op = want_offs ? &och : nullptr;
        const bool next_keep = ch.db == ch.da;
        const u64 next_ds = next_keep ? 0 : dofs[ch.db] - ch.lo + (doc_offs ? ch.db - ch.da : 0);
        uint64_t nt = 0;
        EncDrop dch{};                           // the chunk's place in the caller's text, for the dropout offsets
        if (drop) { dch = *drop; dch.lo = ch.lo; dch.da = ch.da; dch.doffs = doc_offs ? (const u64 *)ctx->doc_offs.p : nullptr; }
        const EncDrop *dp = drop ? &dch : nullptr;
        if (doc_offs) {
            const u64 nb = ch.db - ch.da, an = len + nb;            // a boundary byte after each document that ends here
            rc = ctx_prepare_arena(ctx, ctx->text, an);
            if (rc == BPE_OK) rc = bpe_buf_reserve(ctx, ctx->doc_bmask, flag_words(an) * sizeof(u32));
            if (rc != BPE_OK) break;
            CUDA_TRY(ctx, cudaMemsetAsync(ctx->doc_bmask.p, 0, flag_words(an) * sizeof(u32), st));
            const unsigned g = (unsigned)std::max<u64>(1, std::min<u64>((u64)ctx->sm_count * 16, std::max((len + 4095) / 4096, (nb + 255) / 256)));
            KLAUNCH(k_enc_expand_docs, g, 256, 0, st, (const uint8_t *)sbuf[cur]->p, len, (const u64 *)ctx->doc_offs.p + ch.da + 1, nb, ch.lo,
                    (uint8_t *)ctx->text.p + BPE_PAD, (u32 *)ctx->doc_bmask.p, (uint8_t)tok->doc_sep);
            CUDA_TRY(ctx, cudaGetLastError());
            const DocBounds db{(const u32 *)ctx->doc_bmask.p, id_dev + ch.da + 1, total};
            rc = encode_core(tok, an, out_dtype, odev, len, &nt, stats, &db, dp, op, next_ds, next_keep);
            if (rc == BPE_ERR_UTF8 || rc == BPE_ERR_KEY) {      // arena offset -> offset in the caller's text: minus the boundaries before it
                const u64 p = (u64)ctx->err_detail;
                u64 a = 0, b = nb;                              // boundaries j < a lie before p (boundary j sits at ends[j] - lo + j)
                while (a < b) { const u64 mid = (a + b) / 2; if (doc_offs[ch.da + 1 + mid] - ch.lo + mid < p) a = mid + 1; else b = mid; }
                ctx->err_detail = (int64_t)(ch.lo + p - a);
                bpe_set_error(ctx, rc, rc == BPE_ERR_UTF8 ? "invalid UTF-8 at byte offset %llu of the batch"
                                                          : "KeyError: a token of the pretoken at byte %llu of the batch is not in the vocabulary",
                              (unsigned long long)ctx->err_detail);
            }
            if (rc != BPE_OK) break;
        } else {
            rc = encode_core(tok, len, out_dtype, odev, len, &nt, stats, nullptr, dp, op, next_ds, next_keep);
            if (swap) std::swap(ctx->text, ctx->text_alt);
            if (rc != BPE_OK) { ctx->err_detail += (int64_t)ch.lo; break; }
        }
        if (out && total < cap) {
            const u64 w = std::min<u64>(nt, cap - total);
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_done, st));
            CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->s_out, ctx->ev_done, 0));
            if (w) CUDA_TRY(ctx, cudaMemcpyAsync((uint8_t *)out + total * esz, odev, w * esz, cudaMemcpyDeviceToHost, ctx->s_out));
            if (w && want_offs) CUDA_TRY(ctx, cudaMemcpyAsync(offs_out + 2 * total, och.out, w * 16, cudaMemcpyDeviceToHost, ctx->s_out));
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_out[cur], ctx->s_out));
        }
        total += nt;
        char_carry = och.carry;
    }
    cudaStreamSynchronize(ctx->s_in);
    cudaStreamSynchronize(ctx->s_out);
    if (rc != BPE_OK) return rc;
    int e1 = tm.mark();
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    *n_out = total;
    if (doc_offs) {
        id_offs_out[0] = 0;
        if (n_docs) CUDA_TRY(ctx, cudaMemcpy(id_offs_out + 1, id_dev + 1, n_docs * 8, cudaMemcpyDeviceToHost));
    }
    if (stats) {
        stats->ms_total = tm.ms(e0, e1); stats->ms_h2d = 0; stats->ms_d2h = 0;
        stats->n_bytes -= n_docs; stats->n_pretokens -= n_docs;     // (the boundaries)
    }
    if (out && total > cap) return bpe_set_error(ctx, BPE_ERR_TOO_SMALL, "need room for %llu ids", (unsigned long long)total);
    return BPE_OK;
}

BPE_API int bpe_encode(bpe_tok *tok, const uint8_t *text_host, uint64_t n, int out_dtype, void *out, uint64_t cap, uint64_t *n_out,
                       bpe_encode_stats *stats) {
    return bpe_encode_ex(tok, text_host, n, nullptr, out_dtype, out, cap, n_out, stats);
}

// Arguments are checked in the order include/bpe_sm100.h gives, every option's checks only when it is used.
BPE_API int bpe_encode_ex(bpe_tok *tok, const uint8_t *text_host, uint64_t n, const bpe_encode_opts *opts, int out_dtype, void *out,
                          uint64_t cap, uint64_t *n_out, bpe_encode_stats *stats) {
    if (!tok) return BPE_ERR_ARG;
    bpe_ctx *ctx = tok->ctx;
    const bpe_encode_opts o = opts ? *opts : bpe_encode_opts{};
    if (o.with_offsets) {
        if (o.offset_unit != BPE_OFF_BYTES && o.offset_unit != BPE_OFF_CHARS)
            return bpe_set_error(ctx, BPE_ERR_ARG, "unknown offset unit %d", o.offset_unit);
        if (out && !o.offs_out) return bpe_set_error(ctx, BPE_ERR_ARG, "offs_out is null");
    }
    // BPE-dropout: thr(p) = 2^32 for p = 1, else floor(p * 2^32) (exact in binary64); p outside [0, 1] or NaN is BPE_ERR_ARG.
    // thr = 0 (p = 0, or p below 2^-32) drops nothing: the deterministic pipeline runs.
    if (!(o.dropout >= 0.0 && o.dropout <= 1.0)) return bpe_set_error(ctx, BPE_ERR_ARG, "dropout probability must be in [0, 1]");
    EncDrop d{};
    d.thr = o.dropout == 1.0 ? (1ull << 32) : (u64)(o.dropout * 4294967296.0);
    u64 z = o.seed + 0x9E3779B97F4A7C15ull;      // mix(seed), as splitmix64 on the device
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    d.seed_mix = z ^ (z >> 31);
    if (o.doc_offs || o.n_docs) {
        const uint64_t *doc_offs = o.doc_offs, n_docs = o.n_docs;
        if (!n_out || !o.id_offs_out || !doc_offs) return BPE_ERR_ARG;
        for (uint64_t j = 0; j < n_docs; j++)
            if (doc_offs[j] > doc_offs[j + 1]) return bpe_set_error(ctx, BPE_ERR_ARG, "bpe_encode_ex: document offsets must not decrease");
        if (n_docs ? (doc_offs[0] != 0 || doc_offs[n_docs] != n) : n != 0)
            return bpe_set_error(ctx, BPE_ERR_ARG, "bpe_encode_ex: document offsets must run from 0 to n");
        if (n_docs && tok->doc_sep < 0)
            return bpe_set_error(ctx, BPE_ERR_UNSUPPORTED, "bpe_encode_ex: every ASCII byte but '\\r' occurs in a special token (no boundary byte)");
        if (n_docs == 0) {
            BPE_TRY(encode_check_args(tok, text_host, 0, out_dtype, n_out));
            if (stats) memset(stats, 0, sizeof(*stats));
            o.id_offs_out[0] = 0;
            return BPE_OK;
        }
    }
    return encode_pipeline(tok, text_host, n, o.doc_offs, o.n_docs, out_dtype, out, cap, n_out, o.id_offs_out, stats, d.thr ? &d : nullptr,
                           o.offset_unit, o.with_offsets ? o.offs_out : nullptr);
}

BPE_API int bpe_encode_dev(bpe_tok *tok, const uint8_t *text_dev, uint64_t n, int out_dtype, void *out_dev, uint64_t cap, uint64_t *n_out,
                           bpe_encode_stats *stats) {
    BPE_TRY(encode_check_args(tok, text_dev, n, out_dtype, n_out));
    bpe_ctx *ctx = tok->ctx;
    ctx->saw_cr_encode = false;
    if (stats) memset(stats, 0, sizeof(*stats));
    EvTimer tm(ctx);
    int e0 = tm.mark();
    BPE_TRY(ctx_load_text(ctx, text_dev, n, true));
    int e1 = tm.mark();
    BPE_TRY(encode_core(tok, n, out_dtype, out_dev, cap, n_out, stats));
    if (stats) { stats->ms_h2d = tm.ms(e0, e1); stats->ms_total += stats->ms_h2d; }
    if (out_dev && *n_out > cap) return bpe_set_error(ctx, BPE_ERR_TOO_SMALL, "need room for %llu ids", (unsigned long long)*n_out);
    return BPE_OK;
}

// byte offset of the first token of every sequence: boff[j] = off[seq[j]] (seq[n_seq] = n gives the total)
__global__ void __launch_bounds__(256) k_dec_seq_offsets(const u64 *__restrict__ off, const u64 *__restrict__ seq, u64 n_seq1, u64 *__restrict__ boff) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n_seq1) boff[j] = off[seq[j]];
}

static int decode_core(bpe_tok *tok, const int64_t *ids_host, uint64_t n, uint8_t *out, uint64_t cap, uint64_t *n_out,
                       const uint64_t *seq_offs_host, uint64_t n_seq, uint64_t *byte_offs_host) {
    if (!tok || (!ids_host && n) || !n_out) return BPE_ERR_ARG;
    bpe_ctx *ctx = tok->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    *n_out = 0;
    if (n == 0) return BPE_OK;
    size_t ids_b = round_up(n * 8, 256), len_b = round_up((n + 1) * 4, 256), off_b = round_up((n + 2) * 8, 256);
    BPE_TRY(bpe_buf_reserve(ctx, ctx->tmp0, ids_b + len_b + off_b + scan_tmp_elems_host(n) * 8));
    long long *ids = (long long *)ctx->tmp0.p;
    u32 *lens = (u32 *)((uint8_t *)ctx->tmp0.p + ids_b);
    u64 *off = (u64 *)((uint8_t *)ctx->tmp0.p + ids_b + len_b);
    u64 *tmp = (u64 *)((uint8_t *)ctx->tmp0.p + ids_b + len_b + off_b);
    u64 *scr = (u64 *)ctx->scratch.p;
    u64 *host = (u64 *)ctx->pinned;
    host[0] = ~0ull;
    CUDA_TRY(ctx, cudaMemcpyAsync(scr, host, 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(ids, ids_host, n * 8, cudaMemcpyHostToDevice, st));
    unsigned grid = (unsigned)std::min<u64>((u64)ctx->sm_count * bpe_grid_mult(64), (n + 255) / 256);
    KLAUNCH(k_dec_lens, grid, 256, 0, st, ids, n, (const u32 *)tok->vlen.p, tok->n_dense, lens, scr);
    launch_scan_u32(lens, n, off, tmp, st);
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaStreamSynchronize(st));    // host[0] was the upload source
    CUDA_TRY(ctx, cudaMemcpyAsync(host, scr, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(host + 1, off + n, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    if (host[0] != ~0ull) {
        ctx->err_detail = (int64_t)host[0];
        return bpe_set_error(ctx, BPE_ERR_KEY, "KeyError: id at index %llu is not in the vocabulary", (unsigned long long)host[0]);
    }
    u64 total = host[1];
    *n_out = total;
    if (n_seq && byte_offs_host) {               // byte offsets of the sequences (bpe_decode_batch)
        BPE_TRY(bpe_buf_reserve(ctx, ctx->tmp2, round_up((n_seq + 1) * 16, 256)));
        u64 *seq = (u64 *)ctx->tmp2.p, *boff = seq + (n_seq + 1);
        CUDA_TRY(ctx, cudaMemcpyAsync(seq, seq_offs_host, (n_seq + 1) * 8, cudaMemcpyHostToDevice, st));
        KLAUNCH(k_dec_seq_offsets, (unsigned)((n_seq + 1 + 255) / 256), 256, 0, st, off, seq, n_seq + 1, boff);
        CUDA_TRY(ctx, cudaGetLastError());
        CUDA_TRY(ctx, cudaMemcpyAsync(byte_offs_host, boff, (n_seq + 1) * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
    }
    if (!out) return BPE_OK;
    u64 m = std::min<u64>(total, cap);
    if (m) {
        BPE_TRY(bpe_buf_reserve(ctx, ctx->tmp1, m));
        KLAUNCH(k_dec_copy, grid, 256, 0, st, ids, n, (const u64 *)tok->voff.p, (const uint8_t *)tok->vblob.p, lens, off, (uint8_t *)ctx->tmp1.p, m);
        CUDA_TRY(ctx, cudaGetLastError());
        CUDA_TRY(ctx, cudaMemcpyAsync(out, ctx->tmp1.p, m, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
    }
    return total > cap ? bpe_set_error(ctx, BPE_ERR_TOO_SMALL, "need room for %llu bytes", (unsigned long long)total) : BPE_OK;
}

BPE_API int bpe_decode(bpe_tok *tok, const int64_t *ids_host, uint64_t n, uint8_t *out, uint64_t cap, uint64_t *n_out) {
    return decode_core(tok, ids_host, n, out, cap, n_out, nullptr, 0, nullptr);
}

BPE_API int bpe_decode_batch(bpe_tok *tok, const int64_t *ids_host, uint64_t n, const uint64_t *seq_offs_host, uint64_t n_seq,
                             uint8_t *out, uint64_t cap, uint64_t *n_out, uint64_t *byte_offs_host) {
    if (!tok || !n_out || (n_seq && (!seq_offs_host || !byte_offs_host))) return BPE_ERR_ARG;
    bpe_ctx *ctx = tok->ctx;
    for (uint64_t j = 0; j < n_seq; j++)
        if (seq_offs_host[j] > seq_offs_host[j + 1]) return bpe_set_error(ctx, BPE_ERR_ARG, "bpe_decode_batch: sequence offsets must not decrease");
    if (n_seq && (seq_offs_host[0] != 0 || seq_offs_host[n_seq] != n)) return bpe_set_error(ctx, BPE_ERR_ARG, "bpe_decode_batch: sequence offsets must run from 0 to n");
    if (n == 0) {
        *n_out = 0;
        for (uint64_t j = 0; j <= n_seq && n_seq; j++) byte_offs_host[j] = 0;
        return BPE_OK;
    }
    return decode_core(tok, ids_host, n, out, cap, n_out, seq_offs_host, n_seq, byte_offs_host);
}
