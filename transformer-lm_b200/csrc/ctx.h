// ctx.h -- host-side helpers shared by the API translation units.
#pragma once
#include "common.cuh"

int ctx_prepare_arena(bpe_ctx *ctx, DevBuf &buf, u64 n, cudaStream_t st = nullptr);
int ctx_pipeline_init(bpe_ctx *ctx);           // copy streams + events of the double-buffered host paths (lazy)
int ctx_load_text(bpe_ctx *ctx, const uint8_t *src, u64 n, bool src_is_device);
int ctx_upload_specials(bpe_ctx *ctx, const uint8_t *blob, const u32 *offs, int n_sp, const uint8_t **blob_dev,
                        const u32 **offs_dev, u32 *max_len);
int ctx_run_flags(bpe_ctx *ctx, u64 *n_io, bool translate_newlines, const uint8_t *sp_blob_dev, const u32 *sp_offs_dev,
                  int n_sp, u32 sp_max_len, u64 err_lo = 0, u64 err_hi = ~0ull, const u32 *bmask = nullptr);
void count_state_free(bpe_ctx *ctx);

struct EvTimer {                      // CUDA-event stage timer on the context's stream (nested timers take different bases)
    bpe_ctx *ctx; int next = 0;
    explicit EvTimer(bpe_ctx *c, int base = 0) : ctx(c), next(base) {}
    int mark() { cudaEventRecord(ctx->ev[next], ctx->stream); return next++; }
    float ms(int a, int b) { float t = 0; cudaEventElapsedTime(&t, ctx->ev[a], ctx->ev[b]); return t; }
};
