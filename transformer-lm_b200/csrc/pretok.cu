// pretok.cu -- kernels: UTF-8 validation + class + pretoken-start flags, universal-newline
// translation, special-token matching, bitmask -> offsets.
#include "pretok.cuh"
#include "scan.cuh"
#include "kernels.h"
#include "hashtab.cuh"

// ---------------------------------------------------------------------------------------------
// flags kernel: one pass over the text, a tile of PT_TILE bytes at a time.
//   staging   a tile and its two 16-byte neighbour chunks are ONE contiguous global range (the arena is padded on both sides):
//             one elected thread fetches it with a bulk asynchronous copy (cp.async.bulk, completion on an mbarrier) into one of
//             two shared-memory stages while the CTA works on the other one -- no LDG / STS instructions, no exposed load latency
//   phase 1   per 16-byte chunk a thread turns its ASCII bytes into one-hot class bytes through a shared-memory table; chunks
//             with bytes >= 0x80 are queued
//   phase 2   the queued chunks are patched densely, one thread each (characters decoded, validated and looked up in the Unicode
//             class table in shared memory).  Almost every warp holds a few non-ASCII bytes (1-2 % of natural text), so doing this
//             inline made every warp walk the long decode path with one or two active lanes.
//   phase 3   class bytes -> bit masks, start rules on 32-bit windows built with the neighbours' masks
// Output: 1 bit per byte (bit set = a pretoken starts on that byte).  Algorithmic HBM bytes: n read + n/8 written.
// ---------------------------------------------------------------------------------------------
#define PT_STAGE_BYTES (PT_TILE + 64u)           // [16 B of 0xFF][chunk before][PT_NT chunks][chunk after][16 B of 0xFF]
__device__ __forceinline__ u32 smem_u32(const void *p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(u64 *bar, u32 count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory"); }
__device__ __forceinline__ void bulk_load(void *dst_smem, const void *src_gmem, u32 bytes, u64 *bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(u64 *bar, u32 parity) {
    u32 done = 0;
    while (!done)
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
}

template <bool HAS_SP>
__global__ void __launch_bounds__(PT_NT) k_pretok_flags(const uint8_t *__restrict__ text, u64 n, u64 n_tiles,
                                                       const u32 *__restrict__ spmask, const u32 *__restrict__ spstart,
                                                       u32 *__restrict__ flags, u64 *__restrict__ err, u64 err_lo, u64 err_hi) {
    __shared__ PretokTables tb;
    __shared__ __align__(128) uint8_t s_stage[2][PT_STAGE_BYTES];
    __shared__ uint4 s_info[PT_NT + 2];          // class bytes, then masks, of [chunk before][PT_NT chunks][chunk after]
    __shared__ u32 s_hi[PT_NT + 2];
    __shared__ u32 s_q[PT_NT + 2];               // chunks with non-ASCII bytes
    __shared__ u32 s_nq;
    __shared__ __align__(8) u64 s_bar[2];
    const u32 tid = threadIdx.x;
    pretok_load_tables(&tb);
    for (u32 i = tid; i < 2 * 32; i += PT_NT) {  // the 16-byte guards of both stages (never overwritten by the copies)
        const u32 st = i >> 5, k = i & 31u;
        s_stage[st][k < 16 ? k : PT_STAGE_BYTES - 32 + k] = 0xFF;
    }
    if (tid == 0) { mbar_init(&s_bar[0], 1); mbar_init(&s_bar[1], 1); s_nq = 0; asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    __syncthreads();
    u32 k = 0;
    if (tid == 0 && blockIdx.x < n_tiles) bulk_load(&s_stage[0][16], text + (u64)blockIdx.x * PT_TILE - 16, PT_TILE + 32, &s_bar[0]);
    for (u64 tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, k++) {
        const u32 stg = k & 1u;
        const u64 tbeg = tile * PT_TILE;
        // the other stage was released by the barrier that ended the previous iteration
        if (tid == 0 && tile + gridDim.x < n_tiles) bulk_load(&s_stage[stg ^ 1u][16], text + (tile + gridDim.x) * PT_TILE - 16, PT_TILE + 32, &s_bar[stg ^ 1u]);
        mbar_wait(&s_bar[stg], (k >> 1) & 1u);
        const uint8_t *tx = s_stage[stg];
        // ---- phase 1: ASCII class bytes, queue of the chunks that need decoding ----
        {
            u32 hi; bool cr;
            s_info[tid + 1] = chunk_info_ascii(&tb, tx, 32u + tid * 16u, &hi, &cr);
            s_hi[tid + 1] = hi;
            if (cr) err[1] = 1;
            const u32 m = __ballot_sync(0xffffffffu, hi != 0);
            if (m) {
                u32 base = 0;
                if ((tid & 31u) == (u32)(__ffs(m) - 1)) base = atomicAdd(&s_nq, (u32)__popc(m));
                base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
                if (hi) s_q[base + __popc(m & ((1u << (tid & 31u)) - 1u))] = tid + 1;
            }
            if (tid >= PT_NT - 2) {              // halo chunks (validated by the tile that owns them)
                const u32 idx = tid == PT_NT - 2 ? 0u : PT_NT + 1u;
                u32 h2; bool cr2;
                s_info[idx] = chunk_info_ascii(&tb, tx, 16u + idx * 16u, &h2, &cr2);
                s_hi[idx] = h2;
                if (h2) s_q[atomicAdd(&s_nq, 1u)] = idx;
            }
        }
        __syncthreads();
        // ---- phase 2: non-ASCII characters, one queued chunk per thread ----
        {
            const u32 nq = s_nq;
            for (u32 e = tid; e < nq; e += PT_NT) {
                const u32 c = s_q[e];
                const u32 bad = chunk_patch_non_ascii(&tb, tx, 16u + c * 16u, s_hi[c], &s_info[c]);
                if (bad != 0xFFu && c >= 1 && c <= PT_NT) {
                    const u64 off = tbeg + (u64)(c - 1) * PT_CHUNK + bad;
                    if (off < n && off >= err_lo && off < err_hi) atomicMin(reinterpret_cast<u64 *>(&err[0]), off);
                }
            }
        }
        __syncthreads();
        // ---- phase 3: masks ----
        u32 m16 = 0, s16 = 0;
        uint4 mk = info_to_masks(s_info[tid + 1]);
        uint4 hk = make_uint4(0, 0, 0, 0);
        const u32 hidx = tid == PT_NT - 2 ? 0u : PT_NT + 1u;
        if (tid >= PT_NT - 2) hk = info_to_masks(s_info[hidx]);
        if (HAS_SP) {
            const u64 wi = (tbeg >> 5) + (tid >> 1);
            const u32 sh = (tid & 1u) * 16u;
            m16 = (spmask[wi] >> sh) & 0xFFFFu;
            s16 = (spstart[wi] >> sh) & 0xFFFFu;
            if (m16) mk = masks_apply_boundary(mk, m16);
            if (tid >= PT_NT - 2) {              // halo chunk = last chunk of the previous tile / first chunk of the next one
                u32 hm = 0;
                if (hidx != 0) hm = spmask[(tbeg >> 5) + (PT_NT >> 1)] & 0xFFFFu;
                else if (tile > 0) hm = (spmask[(tbeg >> 5) - 1] >> 16) & 0xFFFFu;
                if (hm) hk = masks_apply_boundary(hk, hm);
            }
        }
        __syncthreads();                         // every thread has read its class bytes: the array now takes the masks
        s_info[tid + 1] = mk;
        if (tid >= PT_NT - 2) s_info[hidx] = hk;
        if (tid == 0) s_nq = 0;
        __syncthreads();
        u32 bits = flags_from_masks(s_info[tid], s_info[tid + 1], s_info[tid + 2], tx, 32u + tid * 16u);
        if (HAS_SP) bits = (bits & ~m16) | s16;
        const u32 hi2 = __shfl_down_sync(0xffffffffu, bits, 1);
        if ((tid & 1u) == 0) flags[(tbeg >> 5) + (tid >> 1)] = bits | (hi2 << 16);
        __syncthreads();                         // the stage and the mask array are free for the next tile
    }
}

void launch_pretok_flags(const uint8_t *text, u64 n, const u32 *spmask, const u32 *spstart, u32 *flags, u64 *err,
                         u64 err_lo, u64 err_hi, int sm_count, cudaStream_t st) {
    u64 n_tiles = (n + PT_TILE - 1) / PT_TILE;
    if (n_tiles == 0) return;
    u64 grid = (u64)sm_count * bpe_grid_mult(64);
    if (grid > n_tiles) grid = n_tiles;
    if (spmask)
        KLAUNCH(k_pretok_flags<true>, (unsigned)grid, PT_NT, 0, st, text, n, n_tiles, spmask, spstart, flags, err, err_lo, err_hi);
    else
        KLAUNCH(k_pretok_flags<false>, (unsigned)grid, PT_NT, 0, st, text, n, n_tiles, nullptr, nullptr, flags, err, err_lo, err_hi);
}

int pretok_upload_tables() {
    cudaError_t e;
    e = cudaMemcpyToSymbol(c_uc_pages, bpe_uc_pages, sizeof(bpe_uc_pages)); if (e) return (int)e;
    e = cudaMemcpyToSymbol(c_uc_index, bpe_uc_index, sizeof(bpe_uc_index)); if (e) return (int)e;
    e = cudaMemcpyToSymbol(c_uc_ascii, bpe_uc_ascii, sizeof(bpe_uc_ascii)); if (e) return (int)e;
    return 0;
}

// ---------------------------------------------------------------------------------------------
// universal newlines ("\r\n" -> "\n", "\r" -> "\n"): text-mode open() in models/tokenizer/train.py:21-23.
// Rare slow path (taken only when the flags kernel saw a '\r'): count kept bytes per 4 KiB tile,
// scan, scatter.
// ---------------------------------------------------------------------------------------------
#define NL_NT 256
#define NL_TILE (NL_NT * 16)

__device__ __forceinline__ u32 nl_keep_mask(const uint8_t *text, u64 base, u64 n, uint8_t *vals) {
    // bit j set <=> byte base+j survives; vals[j] = translated byte
    u32 keep = 0;
    uint8_t prev = base > 0 ? text[base - 1] : 0;
#pragma unroll
    for (int j = 0; j < 16; j++) {
        u64 i = base + j;
        uint8_t b = i < n ? text[i] : 0;
        bool k = i < n && !(b == '\n' && prev == '\r');
        vals[j] = b == '\r' ? (uint8_t)'\n' : b;
        keep |= (k ? 1u : 0u) << j;
        prev = b;
    }
    return keep;
}

__global__ void __launch_bounds__(NL_NT) k_nl_count(const uint8_t *__restrict__ text, u64 n, u32 *__restrict__ tile_cnt) {
    __shared__ u32 s_warp[33];
    u64 base = (u64)blockIdx.x * NL_TILE + (u64)threadIdx.x * 16;
    uint8_t vals[16];
    u32 keep = nl_keep_mask(text, base, n, vals);
    u32 tot;
    block_excl_scan_u32(__popc(keep), &tot, s_warp);
    if (threadIdx.x == 0) tile_cnt[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(NL_NT) k_nl_scatter(const uint8_t *__restrict__ text, u64 n, const u64 *__restrict__ tile_off,
                                                     uint8_t *__restrict__ out) {
    __shared__ u32 s_warp[33];
    u64 base = (u64)blockIdx.x * NL_TILE + (u64)threadIdx.x * 16;
    uint8_t vals[16];
    u32 keep = nl_keep_mask(text, base, n, vals);
    u32 tot;
    u32 ex = block_excl_scan_u32(__popc(keep), &tot, s_warp);
    u64 o = tile_off[blockIdx.x] + ex;
#pragma unroll
    for (int j = 0; j < 16; j++)
        if ((keep >> j) & 1u) out[o++] = vals[j];
}

// tile_cnt: ceil(n/NL_TILE) u32; tile_off: that + 1 u64; scan_tmp: scan_tmp_elems(n_tiles) u64.
// *n_out_dev (device u64) = tile_off[n_tiles].
void launch_newline_translate(const uint8_t *text, u64 n, uint8_t *out, u32 *tile_cnt, u64 *tile_off, u64 *scan_tmp,
                              cudaStream_t st) {
    u64 nt = (n + NL_TILE - 1) / NL_TILE;
    if (nt == 0) { cudaMemsetAsync(tile_off, 0, sizeof(u64), st); return; }
    KLAUNCH(k_nl_count, (unsigned)nt, NL_NT, 0, st, text, n, tile_cnt);
    launch_excl_scan_u32_to_u64(tile_cnt, nt, tile_off, scan_tmp, st);
    KLAUNCH(k_nl_scatter, (unsigned)nt, NL_NT, 0, st, text, n, tile_off, out);
}
u64 newline_tiles(u64 n) { return (n + NL_TILE - 1) / NL_TILE; }

// ---------------------------------------------------------------------------------------------
// special tokens: Tokenizer.segment (models/tokenizer/tokenizer.py:63-66) = re.split on
// "(s1|s2|...)" with specials sorted longest first => leftmost match, longest special at that
// position, non-overlapping, scanning resumes after each match.
//   k_special_candidates: bit i of cand set <=> some special matches at byte i.
//   k_special_resolve:    chains of candidates closer than max_len are resolved left to right by the
//                         chain's first candidate; isolated candidates (the normal case) accept themselves.
// Output: spstart (first byte of an accepted occurrence), spmask (all bytes of accepted occurrences).
// ---------------------------------------------------------------------------------------------
struct SpecialsDev {
    const uint8_t *blob; const u32 *offs; int n; u32 max_len;
};

__device__ __forceinline__ int special_match_at(const uint8_t *text, u64 n, u64 i, const SpecialsDev &sp) {
    for (int s = 0; s < sp.n; s++) {             // longest first
        u32 o = sp.offs[s], l = sp.offs[s + 1] - o;
        if (l == 0 || i + l > n) continue;
        bool ok = true;
        for (u32 k = 0; k < l && ok; k++) ok = text[i + k] == sp.blob[o + k];
        if (ok) return s;
    }
    return -1;
}

__global__ void __launch_bounds__(256) k_special_candidates(const uint8_t *__restrict__ text, u64 n, SpecialsDev sp,
                                                           u32 *__restrict__ cand, u64 n_words) {
    __shared__ u32 s_first[8];                   // 256-bit set of first bytes of the specials
    __shared__ u32 s_fb[4], s_nfirst;            // the distinct first bytes when there are at most four (else s_nfirst = 5)
    if (threadIdx.x < 8) s_first[threadIdx.x] = 0;
    __syncthreads();
    for (u32 i = threadIdx.x; i < (u32)sp.n; i += blockDim.x) {
        u32 o = sp.offs[i];
        if (sp.offs[i + 1] > o) { u32 b = sp.blob[o]; atomicOr(&s_first[b >> 5], 1u << (b & 31)); }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        u32 k = 0;
        for (u32 b = 0; b < 256; b++)
            if ((s_first[b >> 5] >> (b & 31)) & 1u) { if (k < 4) s_fb[k] = b; k++; }
        for (u32 i = k; i < 4; i++) s_fb[i] = k ? s_fb[0] : 0xFFu;
        s_nfirst = k <= 4 ? (k ? k : 1u) : 5u;   // (no special with bytes at all: test for 0xFF, which never occurs)
    }
    __syncthreads();
    for (u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += (u64)gridDim.x * blockDim.x) {
        const uint4 *p = reinterpret_cast<const uint4 *>(text + w * 32);
        uint4 a = ld_stream_v4(p), b4 = ld_stream_v4(p + 1);
        u32 ws[8] = {a.x, a.y, a.z, a.w, b4.x, b4.y, b4.z, b4.w};
        u32 bits = 0;
        // with at most four distinct first bytes (the usual single "<" of "<|endoftext|>"): four SIMD byte tests per word decide
        // whether the 32 bytes hold a candidate at all -- the per-byte walk below then runs for one word in a few hundred
        if (s_nfirst <= 4) {
            bool any = false;
#pragma unroll
            for (int k = 0; k < 8; k++) {
                any |= has_byte(ws[k], s_fb[0]);
                if (s_nfirst > 1) any |= has_byte(ws[k], s_fb[1]);
                if (s_nfirst > 2) any |= has_byte(ws[k], s_fb[2]);
                if (s_nfirst > 3) any |= has_byte(ws[k], s_fb[3]);
            }
            if (!any) { cand[w] = 0; continue; }
        }
#pragma unroll
        for (int j = 0; j < 32; j++) {
            u32 b = (ws[j >> 2] >> ((j & 3) * 8)) & 0xFFu;
            if ((s_first[b >> 5] >> (b & 31)) & 1u) {
                u64 i = w * 32 + j;
                if (i < n && special_match_at(text, n, i, sp) >= 0) bits |= 1u << j;
            }
        }
        cand[w] = bits;
    }
}

__device__ __forceinline__ bool bit_get(const u32 *m, u64 i) { return (m[i >> 5] >> (i & 31)) & 1u; }
// first set bit at position >= from and < to, or ~0
__device__ __forceinline__ u64 bit_find_next(const u32 *m, u64 from, u64 to) {
    if (from >= to) return ~0ull;
    u64 w = from >> 5;
    u32 cur = m[w] & (0xFFFFFFFFu << (from & 31));
    for (;;) {
        if (cur) { u64 p = (w << 5) + (__ffs(cur) - 1); return p < to ? p : ~0ull; }
        w++;
        if ((w << 5) >= to) return ~0ull;
        cur = m[w];
    }
}
// last set bit at position in [from, to), or ~0
__device__ __forceinline__ u64 bit_find_last(const u32 *m, u64 from, u64 to) {
    u64 best = ~0ull;
    for (u64 p = bit_find_next(m, from, to); p != ~0ull; p = bit_find_next(m, p + 1, to)) best = p;
    return best;
}
__device__ __forceinline__ void bit_set_range(u32 *m, u64 from, u64 to) {
    for (u64 w = from >> 5; (w << 5) < to; w++) {
        u64 lo = w << 5;
        u32 mask = 0xFFFFFFFFu;
        if (from > lo) mask &= 0xFFFFFFFFu << (from - lo);
        if (to < lo + 32) mask &= 0xFFFFFFFFu >> (lo + 32 - to);
        atomicOr(&m[w], mask);
    }
}

__global__ void __launch_bounds__(256) k_special_resolve(const uint8_t *__restrict__ text, u64 n, SpecialsDev sp,
                                                        const u32 *__restrict__ cand, u64 n_words,
                                                        u32 *__restrict__ spstart, u32 *__restrict__ spmask) {
    for (u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += (u64)gridDim.x * blockDim.x) {
        u32 bits = cand[w];
        while (bits) {
            u32 j = __ffs(bits) - 1; bits &= bits - 1;
            u64 p = w * 32 + j;
            // chain head <=> no other candidate within max_len-1 bytes before p
            u64 lo = p >= sp.max_len - 1 ? p - (sp.max_len - 1) : 0;
            if (sp.max_len > 1 && bit_find_next(cand, lo, p) != ~0ull) continue;
            u64 reach = p;
            for (;;) {
                int s = special_match_at(text, n, p, sp);
                u32 len = sp.offs[s + 1] - sp.offs[s];
                atomicOr(&spstart[p >> 5], 1u << (p & 31));
                bit_set_range(spmask, p, p + len);
                u64 last_in = bit_find_last(cand, p + 1, p + len);   // suppressed candidates extend the chain
                if (last_in != ~0ull && last_in > reach) reach = last_in;
                if (p > reach) reach = p;
                u64 limit = reach + sp.max_len;                    // q belongs to this chain iff q - reach <= max_len-1
                if (limit > n) limit = n;
                u64 q = bit_find_next(cand, p + len, limit);
                if (q == ~0ull) break;
                reach = q; p = q;
            }
        }
    }
}

void launch_special_split(const uint8_t *text, u64 n, const uint8_t *sp_blob_dev, const u32 *sp_offs_dev, int n_sp,
                          u32 max_len, u32 *cand, u32 *spstart, u32 *spmask, u64 n_words, int sm_count, cudaStream_t st) {
    SpecialsDev sp{sp_blob_dev, sp_offs_dev, n_sp, max_len};
    u64 grid = (n_words + 255) / 256;
    u64 cap = (u64)sm_count * bpe_grid_mult(64);
    if (grid > cap) grid = cap;
    if (grid == 0) return;
    KLAUNCH(k_special_candidates, (unsigned)grid, 256, 0, st, text, n, sp, cand, n_words);
    KLAUNCH(k_special_resolve, (unsigned)grid, 256, 0, st, text, n, sp, cand, n_words, spstart, spmask);
}

// ---------------------------------------------------------------------------------------------
// bitmask -> ascending byte offsets (used by bpe_pretokenize and the encoder)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_popc_words(const u32 *__restrict__ flags, u64 n_words, u32 *__restrict__ cnt) {
    for (u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += (u64)gridDim.x * blockDim.x)
        cnt[w] = __popc(flags[w]);
}
__global__ void __launch_bounds__(256) k_flags_to_offsets(const u32 *__restrict__ flags, u64 n_words, const u64 *__restrict__ pre,
                                                         u64 *__restrict__ out, u64 cap) {
    for (u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += (u64)gridDim.x * blockDim.x) {
        u32 bits = flags[w];
        u64 o = pre[w];
        while (bits) {
            u32 j = __ffs(bits) - 1; bits &= bits - 1;
            if (o < cap) out[o] = w * 32 + j;
            o++;
        }
    }
}
__global__ void k_poke(u64 *dst, PokeVals vals, int n) { if (threadIdx.x < (u32)n) dst[threadIdx.x] = vals.v[threadIdx.x]; }
__global__ void k_peek(u64 *host_dst, const u64 *__restrict__ src, int n) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) host_dst[i] = src[i];
    __threadfence_system();
}
void launch_poke(u64 *dst, const PokeVals &vals, int n, cudaStream_t st) { KLAUNCH(k_poke, 1, 32, 0, st, dst, vals, n); }
void launch_peek(u64 *host_dst, const u64 *src, int n, cudaStream_t st) { KLAUNCH(k_peek, 1, 64, 0, st, host_dst, src, n); }

// cnt[g] = start bits in flag words [16 g, 16 g + 16) = pretokens that start in 512 bytes of text (one warp step of the encoder's
// lookup); the caller guarantees that the words up to the next multiple of 16 exist and are zero past the text
__global__ void __launch_bounds__(256) k_popc_words16(const u32 *__restrict__ flags, u64 n_groups, u32 *__restrict__ cnt) {
    for (u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x; g < n_groups; g += (u64)gridDim.x * blockDim.x) {
        const uint4 *p = reinterpret_cast<const uint4 *>(flags + 16 * g);
        u32 c = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) { const uint4 v = p[k]; c += __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w); }
        cnt[g] = c;
    }
}
void launch_popc_words16(const u32 *flags, u64 n_groups, u32 *cnt, int sm_count, cudaStream_t st) {
    u64 grid = (n_groups + 255) / 256, cap = (u64)sm_count * bpe_grid_mult(64);
    if (grid > cap) grid = cap;
    if (grid) KLAUNCH(k_popc_words16, (unsigned)grid, 256, 0, st, flags, n_groups, cnt);
}

void launch_popc_words(const u32 *flags, u64 n_words, u32 *cnt, int sm_count, cudaStream_t st) {
    u64 grid = (n_words + 255) / 256, capg = (u64)sm_count * bpe_grid_mult(64);
    if (grid > capg) grid = capg;
    if (grid) KLAUNCH(k_popc_words, (unsigned)grid, 256, 0, st, flags, n_words, cnt);
}
void launch_flags_to_offsets(const u32 *flags, u64 n_words, const u64 *pre, u64 *out, u64 cap, int sm_count, cudaStream_t st) {
    u64 grid = (n_words + 255) / 256, capg = (u64)sm_count * bpe_grid_mult(64);
    if (grid > capg) grid = capg;
    if (grid) KLAUNCH(k_flags_to_offsets, (unsigned)grid, 256, 0, st, flags, n_words, pre, out, cap);
}
__global__ void __launch_bounds__(256) k_copy_words2(const u32 *__restrict__ src, u32 *__restrict__ a, u32 *__restrict__ b, u64 n_words) {
    for (u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += (u64)gridDim.x * blockDim.x) { const u32 v = src[w]; a[w] = v; b[w] = v; }
}
void launch_copy_words2(const u32 *src, u32 *a, u32 *b, u64 n_words, int sm_count, cudaStream_t st) {
    u64 grid = (n_words + 255) / 256, capg = (u64)sm_count * bpe_grid_mult(64);
    if (grid > capg) grid = capg;
    if (grid) KLAUNCH(k_copy_words2, (unsigned)grid, 256, 0, st, src, a, b, n_words);
}
void launch_scan_u32(const u32 *in, u64 n, u64 *out, u64 *tmp, cudaStream_t st) { launch_excl_scan_u32_to_u64(in, n, out, tmp, st); }
size_t scan_tmp_elems_host(u64 n) { return scan_tmp_elems(n); }
