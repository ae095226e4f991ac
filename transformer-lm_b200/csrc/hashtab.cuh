// hashtab.cuh -- the pretoken tables of training (train.cu: counts) and encoding (encode.cu: cached values): the one statement of
// their slot format, probes, growth policy and hot table (DESIGN.md section 3).
#pragma once
#include <algorithm>
#include "common.cuh"

// Three open-addressing tables keyed by the pretoken's bytes, linear probing from a home slot, every slot {key, 64-bit payload}
// (a count in training, a cached value in the encoder):
//   short  (<= SHORT_MAX bytes)  {key, payload}, 16 B: the key IS the token -- bytes little-endian in the low 56 bits, length in
//                                the top byte -- so one 64-bit CAS claims and publishes a slot and equality is an integer compare.
//   medium (.. MED_MAX bytes)    {k0, k1, payload, pad}, 32 B: k0 = bytes 0-7, k1 = bytes 8-14 | len << 56, claimed and published
//                                by one 128-bit CAS; a lookup costs one 32-byte sector like a short one.
//   long   (> MED_MAX bytes)     {meta, hash, payload, pad}, 32 B: meta = (offset:40 | len:24) of a representative copy of the bytes
//                                (offset bit 39 set: in the pool, else in the text arena), claimed by CAS; the 64-bit hash is
//                                published after it as a filter, and every hit is confirmed by comparing the bytes.
// An empty slot has key 0, k0 = k1 = 0, meta = 0 (a real key carries its length, >= 1 and >= 16), whatever its payload.
#define SHORT_MAX 7u
#define MED_MAX 15u
#define META_EMPTY 0ull
#define META_LEN_BITS 24
#define META_LEN_MASK ((1ull << META_LEN_BITS) - 1)
#define META_POOL_BIT (1ull << 39)
#define MAX_TOKEN_LEN ((1u << META_LEN_BITS) - 2)

struct __align__(16) SSlot { u64 key, val; };
struct __align__(32) MSlot { u64 k0, k1, val, pad; };
struct __align__(32) LSlot { u64 meta, hash, val, pad; };

// device view of the three tables and of the bytes long keys point at
struct PtTables {
    SSlot *stab; u64 scap;
    MSlot *medtab; u64 medcap;
    LSlot *ltab; u64 lcap;
    const uint8_t *text;                         // payload of the current text arena
    uint8_t *pool;                               // persistent bytes of long keys
};

// Capacities (powers of two) that keep every table at most 7/8 full after a batch that can add new_short pretokens of <= 7 bytes
// and new_long longer ones to the uniques it holds; with no uniques, the initial sizes.
struct PtCaps { u64 s, m, l; };
static inline PtCaps pt_caps(u64 n_short, u64 n_medium, u64 n_long, u64 new_short, u64 new_long) {
    return {next_pow2(std::max<u64>(1 << 16, (n_short + new_short) * 8 / 7 + 64)),
            next_pow2(std::max<u64>(1 << 14, (n_medium + new_long) * 8 / 7 + 64)),
            // pretokens of >= 16 bytes: at most bytes / 16 of them in a batch, i.e. half of the bound for >= 8 bytes
            next_pow2(std::max<u64>(1 << 14, (n_long + (new_long + 1) / 2) * 8 / 7 + 64))};
}

// Smallest k >= 2 such that buckets k .. n - 1 of a histogram hold at most `cap` entries together (n: not even bucket n - 1 fits);
// *taken = what they hold.  Selects the words of the hot tables and of the encoder's shared-memory image.
static inline u64 fit_threshold(const u64 *hist, int n, u64 cap, u64 *taken) {
    u64 sum = 0, k = (u64)n;
    for (int j = n - 1; j >= 2; j--) { if (sum + hist[j] > cap) break; sum += hist[j]; k = (u64)j; }
    *taken = sum;
    return k;
}

#ifdef __CUDACC__
// 8 bytes at an arbitrary address through aligned 64-bit loads (up to 15 bytes past p are touched: every buffer
// these helpers see -- text arena, key pools -- is padded accordingly).  Byte loops cost ~4 instructions per byte
// and diverge on the length; this is ~8 instructions per 8 bytes.
__device__ __forceinline__ u64 load8_unaligned(const uint8_t *p) {
    const u64 *q = reinterpret_cast<const u64 *>(reinterpret_cast<uintptr_t>(p) & ~(uintptr_t)7);
    const u32 sh = (u32)(reinterpret_cast<uintptr_t>(p) & 7u) * 8u;
    const u64 lo = q[0], hi = q[1];
    return sh ? (lo >> sh) | (hi << (64u - sh)) : lo;
}
__device__ __forceinline__ u64 low_bytes_mask(u32 n_bytes) { return n_bytes >= 8 ? ~0ull : ((1ull << (8u * n_bytes)) - 1ull); }

__device__ __forceinline__ u64 hash_long(const uint8_t *p, u32 len) {
    u64 h = 0x9E3779B97F4A7C15ull ^ len;
    u32 i = 0;
    for (; i + 8 <= len; i += 8) {
        h = (h ^ load8_unaligned(p + i)) * 0x9FB21C651E98DF25ull;
        h ^= h >> 29;
    }
    const u64 v = i < len ? load8_unaligned(p + i) & low_bytes_mask(len - i) : 0;
    h = (h ^ v) * 0x9FB21C651E98DF25ull;
    return mix64(h) | 1ull;                      // never 0 ("hash not published yet")
}

__device__ __forceinline__ bool bytes_equal(const uint8_t *a, const uint8_t *b, u32 len) {
    u32 i = 0;
    for (; i + 8 <= len; i += 8) if (load8_unaligned(a + i) != load8_unaligned(b + i)) return false;
    if (i < len) return ((load8_unaligned(a + i) ^ load8_unaligned(b + i)) & low_bytes_mask(len - i)) == 0;
    return true;
}

// key of a pretoken of 1..MED_MAX bytes: a short one's in k0 with k1 = 0, a medium one's in (k0, k1)
__device__ __forceinline__ void pretoken_key(const uint8_t *p, u32 len, u64 &k0, u64 &k1) {
    k0 = load8_unaligned(p) & low_bytes_mask(len);
    if (len <= SHORT_MAX) { k0 |= (u64)len << 56; k1 = 0; }
    else k1 = (len > 8 ? load8_unaligned(p + 8) & low_bytes_mask(len - 8) : 0ull) | ((u64)len << 56);
}

__device__ __forceinline__ const uint8_t *rep_ptr(const PtTables &t, u64 meta) {
    const u64 off = meta >> META_LEN_BITS;
    return (off & META_POOL_BIT) ? t.pool + (off & ~META_POOL_BIT) : t.text + off;
}

// 128-bit compare-and-swap on a 16-byte aligned address: returns the old value in (lo, hi)
__device__ __forceinline__ void cas128(u64 *addr, u64 cmp_lo, u64 cmp_hi, u64 new_lo, u64 new_hi, u64 &lo, u64 &hi) {
    asm volatile("{\n .reg .b128 c, n, d;\n mov.b128 c, {%3, %4};\n mov.b128 n, {%5, %6};\n atom.global.cas.b128 d, [%2], c, n;\n mov.b128 {%0, %1}, d;\n}"
                 : "=l"(lo), "=l"(hi) : "l"(addr), "l"(cmp_lo), "l"(cmp_hi), "l"(new_lo), "l"(new_hi) : "memory");
}

// hash of a 16-byte key: home slot of the medium table, bucket of the hot table
__device__ __forceinline__ u64 key16_hash(u64 k0, u64 k1) { return mix64(k0 ^ (k1 * 0x9E3779B97F4A7C15ull)); }
__device__ __forceinline__ u64 short_home(const PtTables &t, u64 key) { return mix64(key) & (t.scap - 1); }
__device__ __forceinline__ u64 medium_home(const PtTables &t, u64 k0, u64 k1) { return key16_hash(k0, k1) & (t.medcap - 1); }
__device__ __forceinline__ u64 long_home(const PtTables &t, u64 hash) { return hash & (t.lcap - 1); }

// ---- find or claim ------------------------------------------------------------------------------------------------------
// The probe of each tier.  claimed(s) runs in the one thread whose CAS claimed slot s for the key (in the long tier after the hash is
// published); hit(s, v) in every thread that finds the key already there.  With VAL, v is the payload, read in the same round trip
// as the key (of a key claimed in the same kernel it can be the empty slot's payload); without, the payload is not read and v = 0.
// Both return what the probe returns.  When the probe has seen every slot taken, ctr[3] (the overflow flag of both callers) is set
// and R() returned.
template <bool VAL, class Claimed, class Hit>
__device__ __forceinline__ auto short_find_or_claim(const PtTables &t, u64 key, u64 *ctr, Claimed claimed, Hit hit) {
    const u64 mask = t.scap - 1;
    u64 s = short_home(t, key);
    for (u64 probes = 0; probes < t.scap; probes++) {
        u64 k, v = 0;
        if (VAL) { const ulonglong2 kv = *reinterpret_cast<const ulonglong2 *>(&t.stab[s]); k = kv.x; v = kv.y; }
        else k = t.stab[s].key;
        if (k == 0) {
            const u64 old = atomicCAS(&t.stab[s].key, 0ull, key);
            if (old == 0) return claimed(s);
            k = old;
        }
        if (k == key) return hit(s, v);
        s = (s + 1) & mask;
    }
    ctr[3] = 1;
    return decltype(hit(0ull, 0ull))();
}

template <bool VAL, class Claimed, class Hit>
__device__ __forceinline__ auto medium_find_or_claim(const PtTables &t, u64 k0, u64 k1, u64 *ctr, Claimed claimed, Hit hit) {
    const u64 mask = t.medcap - 1;
    u64 s = medium_home(t, k0, k1);
    for (u64 probes = 0; probes < t.medcap; probes++) {
        const ulonglong2 kk = *reinterpret_cast<const ulonglong2 *>(&t.medtab[s]);
        const u64 v = VAL ? t.medtab[s].val : 0;  // (same sector)
        u64 a = kk.x, b = kk.y;
        if ((a | b) == 0) {                      // (k1 carries the length: a real key is never all zero)
            cas128(&t.medtab[s].k0, 0, 0, k0, k1, a, b);
            if ((a | b) == 0) return claimed(s);
        }
        if (a == k0 && b == k1) return hit(s, v);
        s = (s + 1) & mask;
    }
    ctr[3] = 1;
    return decltype(hit(0ull, 0ull))();
}

// p = bytes of the occurrence, off_meta = its offset in the space meta addresses (text, or pool with META_POOL_BIT)
template <bool VAL, class Claimed, class Hit>
__device__ __forceinline__ auto long_find_or_claim(const PtTables &t, const uint8_t *p, u32 len, u64 off_meta, u64 *ctr,
                                                   Claimed claimed, Hit hit) {
    const u64 h = hash_long(p, len);
    const u64 mask = t.lcap - 1;
    u64 s = long_home(t, h);
    const u64 mine = (off_meta << META_LEN_BITS) | len;
    for (u64 probes = 0; probes < t.lcap; probes++) {
        // meta and hash in one 16-byte load (with VAL the whole slot, one round trip)
        const ulonglong2 mh = *reinterpret_cast<const ulonglong2 *>(&t.ltab[s]);
        const ulonglong2 vp = VAL ? *(reinterpret_cast<const ulonglong2 *>(&t.ltab[s]) + 1) : make_ulonglong2(0, 0);
        u64 m = mh.x, hh = mh.y;
        if (m == META_EMPTY) {
            const u64 old = atomicCAS(&t.ltab[s].meta, META_EMPTY, mine);
            if (old == META_EMPTY) { t.ltab[s].hash = h; return claimed(s); }
            m = old;
            hh = *((volatile u64 *)&t.ltab[s].hash);
        }
        if ((m & META_LEN_MASK) == len && (hh == 0 || hh == h) && bytes_equal(rep_ptr(t, m), p, len)) return hit(s, vp.x);
        s = (s + 1) & mask;
    }
    ctr[3] = 1;
    return decltype(hit(0ull, 0ull))();
}

// ---- unique insert: a key known to be absent (table growth, the encoder's specials) -------------------------------------------
// The first free slot from home gets the key and the payload; returns the slot.
__device__ __forceinline__ u64 short_insert_unique(const PtTables &t, u64 key, u64 val) {
    const u64 mask = t.scap - 1;
    u64 s = short_home(t, key);
    while (!(t.stab[s].key == 0 && atomicCAS(&t.stab[s].key, 0ull, key) == 0)) s = (s + 1) & mask;
    t.stab[s].val = val;
    return s;
}
__device__ __forceinline__ u64 medium_insert_unique(const PtTables &t, u64 k0, u64 k1, u64 val) {
    const u64 mask = t.medcap - 1;
    for (u64 s = medium_home(t, k0, k1);; s = (s + 1) & mask) {
        if (t.medtab[s].k1 != 0) continue;       // (taken: a real k1 is never 0)
        u64 a, b;
        cas128(&t.medtab[s].k0, 0, 0, k0, k1, a, b);
        if ((a | b) == 0) { t.medtab[s].val = val; return s; }
    }
}
__device__ __forceinline__ u64 long_insert_unique(const PtTables &t, u64 meta, u64 hash, u64 val) {
    const u64 mask = t.lcap - 1;
    u64 s = long_home(t, hash);
    while (!(t.ltab[s].meta == META_EMPTY && atomicCAS(&t.ltab[s].meta, META_EMPTY, meta) == META_EMPTY)) s = (s + 1) & mask;
    t.ltab[s].hash = hash; t.ltab[s].val = val;
    return s;
}

// ---- hot table --------------------------------------------------------------------------------------------------------
// nb buckets of one 32-byte sector: two 16-byte keys (k0, k1; k1 = 0 for a short pretoken, k0 its key), payloads in an array beside
// it.  A key whose bucket is full stays with the big tables, so a probe is exactly one sector.
__device__ __forceinline__ u64 hot_bucket(u64 nb, u64 k0, u64 k1) { return ((key16_hash(k0, k1) >> 32) * nb) >> 32; }
// slot (0, 1) of bucket b that holds the key, else -1
__device__ __forceinline__ int hot_find(const ulonglong2 *hot, u64 b, u64 k0, u64 k1) {
    const ulonglong2 e0 = __ldg(&hot[2 * b]), e1 = __ldg(&hot[2 * b + 1]);
    return (e0.x == k0 && e0.y == k1) ? 0 : (e1.x == k0 && e1.y == k1) ? 1 : -1;
}
// the first free slot of bucket b gets the key (keys are distinct: no comparison); -1 when both are taken
__device__ __forceinline__ int hot_claim(ulonglong2 *hot, u64 b, u64 k0, u64 k1) {
    u64 x, y;
    cas128(&hot[2 * b].x, 0, 0, k0, k1, x, y);
    if ((x | y) == 0) return 0;
    cas128(&hot[2 * b + 1].x, 0, 0, k0, k1, x, y);
    return (x | y) == 0 ? 1 : -1;
}

__device__ __forceinline__ u64 flags_next_start(const u32 *__restrict__ flags, u64 from, u64 n) {
    // first start bit at position >= from (< n), else n
    if (from >= n) return n;
    u64 w = from >> 5;
    u32 cur = flags[w] & (0xFFFFFFFFu << (from & 31));
    for (;;) {
        if (cur) { u64 p = (w << 5) + (__ffs(cur) - 1); return p < n ? p : n; }
        w++;
        if ((w << 5) >= n) return n;
        cur = flags[w];
    }
}

#endif
