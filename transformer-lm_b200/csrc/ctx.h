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
// BPE_ERR_ARG (message "<what> is not device memory of device N") unless p is device memory of ctx's device.
int ctx_check_dev_ptr(bpe_ctx *ctx, const void *p, const char *what);
// A position in [nominal, min(n, nominal + window)) where cutting the text changes nothing on either side: the start of a
// special-token occurrence that no occurrence covers from the left (Tokenizer.segment splits there, tokenizer.py:63-66), or a
// single U+0020 between two ASCII non-space bytes that no occurrence covers (SURVEY B.2).  0 = none.  Specials longest first.
u64 exact_cut_host(const uint8_t *t, u64 n, u64 nominal, u64 window, const uint8_t *sp_blob, const u32 *sp_offs, int n_sp);

struct EvTimer {                      // CUDA-event stage timer on the context's stream (nested timers take different bases)
    bpe_ctx *ctx; int next = 0;
    explicit EvTimer(bpe_ctx *c, int base = 0) : ctx(c), next(base) {}
    int mark() { cudaEventRecord(ctx->ev[next], ctx->stream); return next++; }
    float ms(int a, int b) { float t = 0; cudaEventElapsedTime(&t, ctx->ev[a], ctx->ev[b]); return t; }
};
