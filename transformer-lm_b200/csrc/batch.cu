// batch.cu -- token-array consumers next to the tokenizer (SURVEY 8f row 4).
//
//   bpe_batch_windows_dev   replaces the per-row Python loop of load_batch (models/util.py:37-57 of the reference):
//                           inputs[row] = dataset[idx : idx + ctx], targets[row] = dataset[idx + 1 : idx + ctx + 1],
//                           both as int64 (torch.long), for `batch` start indices chosen by the caller (the reference
//                           draws them with torch.randint on the host, so the caller keeps doing that: same generator,
//                           same batches).
//
//   bpe_pad_rows_dev        collates the ragged output of a batch encode (ids back to back, id offsets per document) into
//                           [rows][row_len] int64 ids, a uint8 attention mask and, optionally, [rows][row_len][2] spans: the
//                           padding / truncation of a tokenizer's padded-batch call, without a trip through host memory.
//
// Both are HBM-bound with one element per thread and consecutive threads on consecutive columns of a row, so reads and writes
// are coalesced.  k_batch_windows: 2 x 2 B read (the second read of a token hits L1/L2) and 16 B written per element.
// k_pad_rows: 4 B (+ 16 B of span) read per kept element and 9 B (+ 16 B) written per element.
#include <algorithm>
#include "kernels.h"
#include "ctx.h"

template <typename T>
__global__ void __launch_bounds__(256) k_batch_windows(const T *__restrict__ tok, const long long *__restrict__ starts, u32 batch,
                                                      u32 context, long long *__restrict__ x, long long *__restrict__ y) {
    const u64 total = (u64)batch * context;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (u64)gridDim.x * blockDim.x) {
        const u32 row = (u32)(i / context), col = (u32)(i - (u64)row * context);
        const T *p = tok + starts[row] + col;
        x[i] = (long long)p[0];
        y[i] = (long long)p[1];
    }
}

BPE_API int bpe_batch_windows_dev(bpe_ctx *ctx, const void *tokens_dev, int dtype, uint64_t n_tokens, const int64_t *starts_host,
                                  uint32_t batch, uint32_t context, int64_t *x_dev, int64_t *y_dev) {
    if (!ctx) return BPE_ERR_ARG;
    if ((!tokens_dev && n_tokens) || (!starts_host && batch) || (batch && context && (!x_dev || !y_dev)))
        return bpe_set_error(ctx, BPE_ERR_ARG, "bpe_batch_windows_dev: null argument");
    if (dtype != BPE_DTYPE_U16 && dtype != BPE_DTYPE_I32) return bpe_set_error(ctx, BPE_ERR_ARG, "bpe_batch_windows_dev: dtype must be BPE_DTYPE_U16 or BPE_DTYPE_I32");
    if (batch == 0 || context == 0) return BPE_OK;
    for (uint32_t r = 0; r < batch; r++)       // dataset[idx + 1 : idx + ctx + 1] must exist (the reference draws idx < len - ctx)
        if (starts_host[r] < 0 || (uint64_t)starts_host[r] + context + 1 > n_tokens) {
            ctx->err_detail = (int64_t)r;
            return bpe_set_error(ctx, BPE_ERR_ARG, "bpe_batch_windows_dev: window %u (start %lld, context %u) leaves the %llu tokens", r,
                                 (long long)starts_host[r], context, (unsigned long long)n_tokens);
        }
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    BPE_TRY(bpe_buf_reserve(ctx, ctx->tmp0, round_up((size_t)batch * 8, 256)));
    // (pageable source: cudaMemcpyAsync stages it before returning, the caller's array may be reused at once)
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->tmp0.p, starts_host, (size_t)batch * 8, cudaMemcpyHostToDevice, st));
    const u64 total = (u64)batch * context;
    const unsigned grid = (unsigned)std::min<u64>((u64)ctx->sm_count * bpe_grid_mult(64), (total + 255) / 256);
    if (dtype == BPE_DTYPE_U16)
        KLAUNCH(k_batch_windows<uint16_t>, grid, 256, 0, st, (const uint16_t *)tokens_dev, (const long long *)ctx->tmp0.p, batch, context, (long long *)x_dev, (long long *)y_dev);
    else
        KLAUNCH(k_batch_windows<int32_t>, grid, 256, 0, st, (const int32_t *)tokens_dev, (const long long *)ctx->tmp0.p, batch, context, (long long *)x_dev, (long long *)y_dev);
    CUDA_TRY(ctx, cudaGetLastError());
    // On the caller's stream (bpe_ctx_set_stream) the result is stream-ordered with the caller's other work and nothing waits
    // here; on the context's private stream the call returns with x / y complete.
    if (st == ctx->own_stream) CUDA_TRY(ctx, cudaStreamSynchronize(st));
    return BPE_OK;
}

// Row r's kept tokens are ids[offs[r] + t0 .. + k) with k = min(m, row_len), t0 = m - k under BPE_TRUNC_LEFT (else 0); they sit at
// columns [c0, c0 + k) with c0 = row_len - k under BPE_PAD_LEFT (else 0).
__global__ void __launch_bounds__(256) k_pad_rows(const int32_t *__restrict__ ids, const longlong2 *__restrict__ spans,
                                                 const unsigned long long *__restrict__ offs, u64 n_rows, u32 row_len, long long pad_id,
                                                 int flags, long long *__restrict__ ids_out, uint8_t *__restrict__ mask_out,
                                                 longlong2 *__restrict__ spans_out) {
    const u64 total = n_rows * row_len;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (u64)gridDim.x * blockDim.x) {
        const u64 row = i / row_len;
        const u32 col = (u32)(i - row * row_len);
        const u64 lo = offs[row], m = offs[row + 1] - lo;
        const u32 k = (u32)min(m, (u64)row_len);
        const u32 c0 = (flags & BPE_PAD_LEFT) ? row_len - k : 0;
        const bool kept = col >= c0 && col - c0 < k;
        long long id = pad_id;
        longlong2 sp = make_longlong2(0, 0);
        if (kept) {
            const u64 src = lo + ((flags & BPE_TRUNC_LEFT) ? m - k : 0) + (col - c0);
            id = ids[src];
            if (spans) sp = spans[src];
        }
        ids_out[i] = id;
        if (mask_out) mask_out[i] = kept;
        if (spans_out) spans_out[i] = sp;
    }
}

BPE_API int bpe_pad_rows_dev(bpe_ctx *ctx, const int32_t *ids_dev, uint64_t n_ids, const uint64_t *id_offs_host, uint64_t n_rows,
                             const int64_t *spans_dev, uint32_t row_len, int64_t pad_id, int flags, int64_t *ids_out_dev,
                             uint8_t *mask_out_dev, int64_t *spans_out_dev) {
    if (!ctx) return BPE_ERR_ARG;
    if ((!ids_dev && n_ids) || (!id_offs_host && n_rows) || (n_rows && row_len && !ids_out_dev))
        return bpe_set_error(ctx, BPE_ERR_ARG, "bpe_pad_rows_dev: null argument");
    if (flags & ~(BPE_PAD_LEFT | BPE_TRUNC_LEFT)) return bpe_set_error(ctx, BPE_ERR_ARG, "bpe_pad_rows_dev: unknown flag bits 0x%x", flags);
    if (!spans_dev != !spans_out_dev) return bpe_set_error(ctx, BPE_ERR_ARG, "bpe_pad_rows_dev: spans_dev and spans_out_dev go together");
    if (n_rows == 0 || row_len == 0) return BPE_OK;
    for (uint64_t r = 0; r < n_rows; r++)
        if (id_offs_host[r] > id_offs_host[r + 1] || id_offs_host[r + 1] > n_ids) {
            ctx->err_detail = (int64_t)r;
            return bpe_set_error(ctx, BPE_ERR_ARG, "bpe_pad_rows_dev: row %llu (ids %llu .. %llu) is not a range of the %llu ids",
                                 (unsigned long long)r, (unsigned long long)id_offs_host[r], (unsigned long long)id_offs_host[r + 1],
                                 (unsigned long long)n_ids);
        }
    if (n_ids) BPE_TRY(ctx_check_dev_ptr(ctx, ids_dev, "bpe_pad_rows_dev: ids_dev"));
    BPE_TRY(ctx_check_dev_ptr(ctx, ids_out_dev, "bpe_pad_rows_dev: ids_out_dev"));
    if (mask_out_dev) BPE_TRY(ctx_check_dev_ptr(ctx, mask_out_dev, "bpe_pad_rows_dev: mask_out_dev"));
    if (spans_dev) {
        if (n_ids) BPE_TRY(ctx_check_dev_ptr(ctx, spans_dev, "bpe_pad_rows_dev: spans_dev"));
        BPE_TRY(ctx_check_dev_ptr(ctx, spans_out_dev, "bpe_pad_rows_dev: spans_out_dev"));
        if ((uintptr_t)spans_dev % 16 || (uintptr_t)spans_out_dev % 16)
            return bpe_set_error(ctx, BPE_ERR_ARG, "bpe_pad_rows_dev: span pointers must be 16-byte aligned");
    }
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    BPE_TRY(bpe_buf_reserve(ctx, ctx->tmp0, round_up((size_t)(n_rows + 1) * 8, 256)));
    // (pageable source: cudaMemcpyAsync stages it before returning, the caller's array may be reused at once)
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->tmp0.p, id_offs_host, (size_t)(n_rows + 1) * 8, cudaMemcpyHostToDevice, st));
    const u64 total = n_rows * row_len;
    const unsigned grid = (unsigned)std::min<u64>((u64)ctx->sm_count * bpe_grid_mult(64), (total + 255) / 256);
    KLAUNCH(k_pad_rows, grid, 256, 0, st, ids_dev, (const longlong2 *)spans_dev, (const unsigned long long *)ctx->tmp0.p, (u64)n_rows,
            row_len, (long long)pad_id, flags, (long long *)ids_out_dev, mask_out_dev, (longlong2 *)spans_out_dev);
    CUDA_TRY(ctx, cudaGetLastError());
    if (st == ctx->own_stream) CUDA_TRY(ctx, cudaStreamSynchronize(st));   // (as bpe_batch_windows_dev)
    return BPE_OK;
}
