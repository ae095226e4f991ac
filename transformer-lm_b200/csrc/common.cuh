// common.cuh -- context, error plumbing and small device helpers shared by all kernels.
#pragma once
#include <cstdlib>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <string.h>
#include <string>
#include <vector>

#include "../../include/bpe_sm100.h"

#define BPE_API extern "C" __attribute__((visibility("default")))

typedef unsigned long long u64;
typedef long long i64;
typedef unsigned int u32;

// Text lives in a padded arena: PAD bytes of 0xFF (never valid UTF-8 => "boundary" class) on both
// sides of the payload so every stencil read is in-bounds without index checks.
#define BPE_PAD 64
#define BPE_BYTE_PAD 0xFF

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
};

struct bpe_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;                   // stream in use
    cudaStream_t own_stream = nullptr;               // the one the context created
    cudaEvent_t ev[16] = {};
    std::string err;
    int64_t err_detail = 0;
    // reusable device workspaces (grown on demand, never shrunk)
    DevBuf text;        // padded text arena
    DevBuf flags;       // pretoken-start bitmask, 1 bit per byte
    DevBuf spmask;      // bytes covered by a special-token occurrence (encode only)
    DevBuf spstart;     // first byte of an accepted special occurrence
    DevBuf scratch;     // small scalars: error words, counters
    DevBuf tmp0, tmp1, tmp2;
    DevBuf sp_dev;      // the special tokens last uploaded (blob + offsets), with a host copy to tell when they change
    std::vector<uint8_t> sp_cache_blob; std::vector<uint32_t> sp_cache_offs;
    // double buffering of the host-side entry points: second text arena / output buffers, copy streams, events
    DevBuf text_alt, out_a, out_b;
    DevBuf doc_bmask, doc_offs, doc_stage;   // batch encode: boundary bitmask; document / id offsets; second upload buffer
    cudaStream_t s_in = nullptr, s_out = nullptr;
    cudaEvent_t ev_in[2] = {}, ev_out[2] = {}, ev_done = nullptr;
    void *pinned = nullptr; size_t pinned_cap = 0;   // small pinned staging for scalar readbacks
    struct CountState *count = nullptr;              // pretoken count tables (count.cu)
    uint64_t mem_limit = 0;
    std::vector<DevBuf> pool;                        // cached free device buffers
    bool saw_cr_encode = false;                      // a '\r' anywhere in the text of the last bpe_encode / bpe_encode_dev call
    bool saw_cr = false;                             // the last flags pass met a '\r'
    int32_t *live_pairs = nullptr; int live_cap = 0;   // bpe_train_set_live: page-locked host buffer the merge loop writes as it goes
    std::vector<unsigned long long> last_dense;      // initial 256 x 256 byte-pair table of the last training call (bpe_last_pair_table)
};

int bpe_set_error(bpe_ctx *ctx, int code, const char *fmt, ...);
// Device buffers come from a per-context caching pool: cudaMalloc / cudaFree cost milliseconds per GB and
// synchronise the device, and every call of the library asks for the same sizes again.
int bpe_buf_reserve(bpe_ctx *ctx, DevBuf &b, size_t bytes);       // grow-only, contents NOT preserved
int bpe_buf_alloc(bpe_ctx *ctx, DevBuf &b, size_t bytes);         // (re)size to about `bytes` (may shrink), contents NOT preserved
static inline int alloc_exact(bpe_ctx *ctx, DevBuf &b, size_t bytes) { return bpe_buf_alloc(ctx, b, bytes ? bytes : 256); }   // (0 bytes: still a buffer)
void bpe_buf_free(bpe_ctx *ctx, DevBuf &b);                       // back to the pool
void bpe_pool_trim(bpe_ctx *ctx);                                 // cudaFree everything cached

#define CUDA_TRY(ctx, expr)                                                                      \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess)                                                                   \
            return bpe_set_error((ctx), _e == cudaErrorMemoryAllocation ? BPE_ERR_OOM : BPE_ERR_CUDA, \
                                 "%s:%d %s: %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
    } while (0)

#define BPE_TRY(expr)                 \
    do {                              \
        int _rc = (expr);             \
        if (_rc != BPE_OK) return _rc; \
    } while (0)

static inline size_t round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
// CTAs per SM of the grid-stride kernels (BPE_GRID_MULT overrides; measured per kernel, see DESIGN.md section 4)
static inline int bpe_grid_mult(int dflt) { static const int env = getenv("BPE_GRID_MULT") ? atoi(getenv("BPE_GRID_MULT")) : 0; return env > 0 ? env : dflt; }
static inline uint64_t next_pow2(uint64_t x) { uint64_t p = 1; while (p < x) p <<= 1; return p; }

// every kernel launch of the library goes through KLAUNCH so that launches can be counted (bench.py: gpu_launches)
extern unsigned long long g_bpe_launches;
#define KLAUNCH(kernel, grid, block, smem, stream, ...) \
    do { g_bpe_launches++; kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__); } while (0)

#ifdef __CUDACC__
__device__ __forceinline__ u64 mix64(u64 x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33;
    x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33; return x;
}
// 128-bit streaming load that does not pollute L1 (text is read once)
__device__ __forceinline__ uint4 ld_stream_v4(const void *p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ u32 lane_id() { return threadIdx.x & 31; }
#endif
