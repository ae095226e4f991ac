// api.cu -- context management and the pretokenizer entry points of the C ABI (include/bpe_sm100.h).
#include "kernels.h"
#include "ctx.h"
#include "unicode_tables.h"

unsigned long long g_bpe_launches = 0;
BPE_API unsigned long long bpe_launch_count(void) { return g_bpe_launches; }

int bpe_set_error(bpe_ctx *ctx, int code, const char *fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) { ctx->err = buf; }
    return code;
}

static size_t pool_round(size_t bytes) { return bytes <= (1 << 20) ? round_up(bytes ? bytes : 1, 4096) : round_up(bytes, 1 << 20); }

static int pool_take(bpe_ctx *ctx, DevBuf &out, size_t want) {
    // smallest cached buffer that fits without wasting more than half
    int best = -1;
    for (int i = 0; i < (int)ctx->pool.size(); i++) {
        size_t c = ctx->pool[i].cap;
        if (c >= want && c <= 2 * want + (1 << 20) && (best < 0 || c < ctx->pool[best].cap)) best = i;
    }
    if (best >= 0) { out = ctx->pool[best]; ctx->pool.erase(ctx->pool.begin() + best); return BPE_OK; }
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {                       // give the cached buffers back to the driver and retry once
        cudaGetLastError();
        bpe_pool_trim(ctx);
        e = cudaMalloc(&p, want);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        return bpe_set_error(ctx, BPE_ERR_OOM, "cudaMalloc(%zu bytes) failed: %s", want, cudaGetErrorString(e));
    }
    out.p = p; out.cap = want;
    return BPE_OK;
}

void bpe_pool_trim(bpe_ctx *ctx) {
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (auto &b : ctx->pool) if (b.p) cudaFree(b.p);
    ctx->pool.clear();
}

void bpe_buf_free(bpe_ctx *ctx, DevBuf &b) {
    if (!b.p) { b.cap = 0; return; }
    if (ctx) {
        ctx->pool.push_back(b);
        if (ctx->pool.size() > 256) {            // bound the cache: drop the buffer that has waited longest (a training call alone holds ~40 buffers)
            cudaFree(ctx->pool.front().p);       // (cudaFree synchronises the device: nothing can still be using it)
            ctx->pool.erase(ctx->pool.begin());
        }
    } else cudaFree(b.p);
    b.p = nullptr; b.cap = 0;
}

int bpe_buf_reserve(bpe_ctx *ctx, DevBuf &b, size_t bytes) {
    if (bytes <= b.cap) return BPE_OK;
    bpe_buf_free(ctx, b);
    return pool_take(ctx, b, pool_round(bytes + bytes / 8));
}

int bpe_buf_alloc(bpe_ctx *ctx, DevBuf &b, size_t bytes) {
    size_t want = pool_round(bytes);
    if (b.cap >= want && b.cap <= 2 * want + (1 << 20)) return BPE_OK;
    bpe_buf_free(ctx, b);
    return pool_take(ctx, b, want);
}

BPE_API int bpe_version(void) { return 100; }
BPE_API const char *bpe_unicode_table_source(void) { return BPE_UNICODE_TABLE_SOURCE; }

BPE_API int bpe_ctx_create(int device, bpe_ctx **out) {
    if (!out) return BPE_ERR_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return BPE_ERR_NO_DEVICE; }
    if (device < 0 || device >= ndev) return BPE_ERR_ARG;
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return BPE_ERR_NO_DEVICE; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { cudaGetLastError(); return BPE_ERR_NO_DEVICE; }
    if (prop.major != 10) return BPE_ERR_NO_DEVICE;   // sm_100a cubin only: no other architecture, no CPU path
    bpe_ctx *ctx = new bpe_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return BPE_ERR_CUDA; }
    ctx->stream = ctx->own_stream;
    for (auto &e : ctx->ev) cudaEventCreate(&e);
    if (pretok_upload_tables() != 0) { delete ctx; return BPE_ERR_CUDA; }
    if (cudaMallocHost(&ctx->pinned, 1 << 16) != cudaSuccess) { delete ctx; return BPE_ERR_OOM; }
    ctx->pinned_cap = 1 << 16;
    if (bpe_buf_reserve(ctx, ctx->scratch, 4096) != BPE_OK) { delete ctx; return BPE_ERR_OOM; }
    *out = ctx;
    return BPE_OK;
}

void count_state_free(bpe_ctx *ctx);

BPE_API void bpe_ctx_destroy(bpe_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    count_state_free(ctx);
    if (ctx->s_in) { cudaStreamSynchronize(ctx->s_in); cudaStreamSynchronize(ctx->s_out); }
    for (DevBuf *b : {&ctx->text, &ctx->flags, &ctx->spmask, &ctx->spstart, &ctx->scratch, &ctx->tmp0, &ctx->tmp1, &ctx->tmp2, &ctx->sp_dev,
                      &ctx->text_alt, &ctx->out_a, &ctx->out_b, &ctx->doc_bmask, &ctx->doc_offs, &ctx->doc_stage})
        bpe_buf_free(ctx, *b);
    if (ctx->s_in) {
        cudaStreamDestroy(ctx->s_in); cudaStreamDestroy(ctx->s_out);
        for (auto &e : ctx->ev_in) if (e) cudaEventDestroy(e);
        for (auto &e : ctx->ev_out) if (e) cudaEventDestroy(e);
        if (ctx->ev_done) cudaEventDestroy(ctx->ev_done);
    }
    bpe_pool_trim(ctx);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    for (auto &e : ctx->ev) if (e) cudaEventDestroy(e);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

BPE_API const char *bpe_last_error(bpe_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }
BPE_API int64_t bpe_last_error_detail(bpe_ctx *ctx) { return ctx ? ctx->err_detail : 0; }
BPE_API int bpe_device_sync(bpe_ctx *ctx) {
    if (!ctx) return BPE_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return BPE_OK;
}

BPE_API int bpe_ctx_set_stream(bpe_ctx *ctx, void *cuda_stream) {
    if (!ctx) return BPE_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return BPE_OK;
}

BPE_API void *bpe_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
BPE_API void bpe_host_free(void *p) { if (p) cudaFreeHost(p); }

// ---------------------------------------------------------------------------------------------
// text arena
// ---------------------------------------------------------------------------------------------
int ctx_prepare_arena(bpe_ctx *ctx, DevBuf &buf, u64 n, cudaStream_t st) {
    if (!st) st = ctx->stream;
    BPE_TRY(bpe_buf_reserve(ctx, buf, arena_bytes(n)));
    uint8_t *a = (uint8_t *)buf.p;
    CUDA_TRY(ctx, cudaMemsetAsync(a, BPE_BYTE_PAD, BPE_PAD, st));
    CUDA_TRY(ctx, cudaMemsetAsync(a + BPE_PAD + n, BPE_BYTE_PAD, arena_bytes(n) - BPE_PAD - n, st));
    return BPE_OK;
}

int ctx_pipeline_init(bpe_ctx *ctx) {
    if (ctx->s_in) return BPE_OK;
    CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->s_in, cudaStreamNonBlocking));
    CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->s_out, cudaStreamNonBlocking));
    for (auto &e : ctx->ev_in) CUDA_TRY(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (auto &e : ctx->ev_out) CUDA_TRY(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->ev_done, cudaEventDisableTiming));
    return BPE_OK;
}

int ctx_load_text(bpe_ctx *ctx, const uint8_t *src, u64 n, bool src_is_device) {
    BPE_TRY(ctx_prepare_arena(ctx, ctx->text, n));
    if (n)
        CUDA_TRY(ctx, cudaMemcpyAsync((uint8_t *)ctx->text.p + BPE_PAD, src, n,
                                      src_is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, ctx->stream));
    return BPE_OK;
}

// Upload the specials (blob + offsets) into tmp2; returns device pointers and the longest length.
int ctx_upload_specials(bpe_ctx *ctx, const uint8_t *blob, const u32 *offs, int n_sp, const uint8_t **blob_dev,
                        const u32 **offs_dev, u32 *max_len) {
    *blob_dev = nullptr; *offs_dev = nullptr; *max_len = 0;
    if (n_sp <= 0) return BPE_OK;
    size_t blob_bytes = offs[n_sp];
    size_t offs_bytes = sizeof(u32) * (n_sp + 1);
    size_t offs_at = round_up(blob_bytes + 1, 16);
    // the same specials as last time (every chunk of a pipelined encode asks again): nothing to upload -- and nothing queued on the
    // copy engine behind the chunk that is being uploaded
    const bool same = ctx->sp_dev.p && ctx->sp_cache_blob.size() == blob_bytes && ctx->sp_cache_offs.size() == (size_t)n_sp + 1 &&
                      memcmp(ctx->sp_cache_offs.data(), offs, offs_bytes) == 0 && (blob_bytes == 0 || memcmp(ctx->sp_cache_blob.data(), blob, blob_bytes) == 0);
    if (!same) {
        ctx->sp_cache_blob.clear(); ctx->sp_cache_offs.clear();
        BPE_TRY(bpe_buf_reserve(ctx, ctx->sp_dev, offs_at + offs_bytes));
        if (blob_bytes) CUDA_TRY(ctx, cudaMemcpyAsync(ctx->sp_dev.p, blob, blob_bytes, cudaMemcpyHostToDevice, ctx->stream));
        CUDA_TRY(ctx, cudaMemcpyAsync((uint8_t *)ctx->sp_dev.p + offs_at, offs, offs_bytes, cudaMemcpyHostToDevice, ctx->stream));
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));           // (the caller's arrays may go away)
        ctx->sp_cache_blob.assign(blob, blob + blob_bytes); ctx->sp_cache_offs.assign(offs, offs + n_sp + 1);
    }
    for (int i = 0; i < n_sp; i++) if (offs[i + 1] - offs[i] > *max_len) *max_len = offs[i + 1] - offs[i];
    *blob_dev = (const uint8_t *)ctx->sp_dev.p;
    *offs_dev = (const u32 *)((uint8_t *)ctx->sp_dev.p + offs_at);
    return BPE_OK;
}

// Run validation + flags over the text currently in the arena (payload length *n).
//   translate_newlines: apply universal-newline translation when a '\r' is present (training path);
//                       *n is updated to the translated length.
//   specials: when n_sp > 0 the text is first split on the specials (encode path).
//   bmask: document boundaries of bpe_encode_batch (flag_words(n) words, or null): every set bit is a one-byte occurrence of
//          class B, like a special token -- the text before it sees the end of a text, the text after it the start of one.
// Leaves ctx->flags holding the start bitmask.  Synchronises the stream once (error words).
int ctx_run_flags(bpe_ctx *ctx, u64 *n_io, bool translate_newlines, const uint8_t *sp_blob_dev, const u32 *sp_offs_dev,
                  int n_sp, u32 sp_max_len, u64 err_lo, u64 err_hi, const u32 *bmask) {
    u64 n = *n_io;
    cudaStream_t st = ctx->stream;
    u64 *scr = (u64 *)ctx->scratch.p;
    u64 *host = (u64 *)ctx->pinned;
    for (int pass = 0; pass < 2; pass++) {
        const uint8_t *text = (const uint8_t *)ctx->text.p + BPE_PAD;
        u64 fw = flag_words(n);
        BPE_TRY(bpe_buf_reserve(ctx, ctx->flags, fw * sizeof(u32)));
        { PokeVals pv{}; pv.v[0] = ~0ull; pv.v[1] = 0; launch_poke(scr, pv, 2, st); }
        const u32 *spmask = nullptr, *spstart = nullptr;
        if (n_sp > 0 && sp_max_len > 0) {
            BPE_TRY(bpe_buf_reserve(ctx, ctx->spmask, fw * sizeof(u32)));
            BPE_TRY(bpe_buf_reserve(ctx, ctx->spstart, fw * sizeof(u32)));
            BPE_TRY(bpe_buf_reserve(ctx, ctx->tmp0, fw * sizeof(u32)));
            if (bmask) {                         // the special-token kernels OR their occurrences into the boundaries
                launch_copy_words2(bmask, (u32 *)ctx->spmask.p, (u32 *)ctx->spstart.p, fw, ctx->sm_count, st);
            } else {
                CUDA_TRY(ctx, cudaMemsetAsync(ctx->spmask.p, 0, fw * sizeof(u32), st));
                CUDA_TRY(ctx, cudaMemsetAsync(ctx->spstart.p, 0, fw * sizeof(u32), st));
            }
            CUDA_TRY(ctx, cudaMemsetAsync(ctx->tmp0.p, 0, fw * sizeof(u32), st));
            launch_special_split(text, n, sp_blob_dev, sp_offs_dev, n_sp, sp_max_len, (u32 *)ctx->tmp0.p,
                                 (u32 *)ctx->spstart.p, (u32 *)ctx->spmask.p, (n + 31) / 32, ctx->sm_count, st);
            spmask = (const u32 *)ctx->spmask.p; spstart = (const u32 *)ctx->spstart.p;
        } else if (bmask) {                      // boundaries only: they are both the occurrences and their first bytes
            spmask = bmask; spstart = bmask;
        }
        // words past the last tile stay zero
        u64 tiles_words = ((n + 4095) / 4096) * (4096 / 32);
        if (fw > tiles_words)
            CUDA_TRY(ctx, cudaMemsetAsync((u32 *)ctx->flags.p + tiles_words, 0, (fw - tiles_words) * sizeof(u32), st));
        launch_pretok_flags(text, n, spmask, spstart, (u32 *)ctx->flags.p, scr, err_lo, err_hi, ctx->sm_count, st);
        launch_peek(host, scr, 2, st);
        CUDA_TRY(ctx, cudaGetLastError());
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
        if (pass == 0 && host[0] != ~0ull) {
            ctx->err_detail = (int64_t)host[0];
            return bpe_set_error(ctx, BPE_ERR_UTF8, "invalid UTF-8 at byte offset %llu", (unsigned long long)host[0]);
        }
        if (pass == 0) ctx->saw_cr = host[1] != 0;
        if (!(translate_newlines && host[1] && pass == 0)) break;
        // universal newlines: compact into tmp1 (as a fresh arena), swap, redo the flags
        u64 nt = newline_tiles(n);
        BPE_TRY(ctx_prepare_arena(ctx, ctx->tmp1, n));
        size_t cnt_bytes = round_up(nt * sizeof(u32), 256), off_bytes = round_up((nt + 1) * sizeof(u64), 256);
        size_t tmp_bytes = scan_tmp_elems_host(nt) * sizeof(u64);
        BPE_TRY(bpe_buf_reserve(ctx, ctx->tmp0, cnt_bytes + off_bytes + tmp_bytes));
        u32 *tile_cnt = (u32 *)ctx->tmp0.p;
        u64 *tile_off = (u64 *)((uint8_t *)ctx->tmp0.p + cnt_bytes);
        u64 *scan_tmp = (u64 *)((uint8_t *)ctx->tmp0.p + cnt_bytes + off_bytes);
        launch_newline_translate(text, n, (uint8_t *)ctx->tmp1.p + BPE_PAD, tile_cnt, tile_off, scan_tmp, st);
        CUDA_TRY(ctx, cudaGetLastError());
        CUDA_TRY(ctx, cudaMemcpyAsync(host, tile_off + nt, 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
        u64 n2 = host[0];
        // bytes between n2 and n in the new arena must read as padding
        CUDA_TRY(ctx, cudaMemsetAsync((uint8_t *)ctx->tmp1.p + BPE_PAD + n2, BPE_BYTE_PAD, n - n2, st));
        std::swap(ctx->text, ctx->tmp1);
        n = n2;
    }
    *n_io = n;
    return BPE_OK;
}

BPE_API int bpe_utf8_validate(bpe_ctx *ctx, const uint8_t *text_host, uint64_t n) {
    if (!ctx || (!text_host && n)) return BPE_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    BPE_TRY(ctx_load_text(ctx, text_host, n, false));
    u64 nn = n;
    return ctx_run_flags(ctx, &nn, false, nullptr, nullptr, 0, 0);
}

BPE_API int bpe_pretokenize(bpe_ctx *ctx, const uint8_t *text_host, uint64_t n,
                            const uint8_t *specials_blob, const uint32_t *special_offs, int n_specials,
                            uint64_t *starts_out, uint64_t cap, uint64_t *n_out) {
    if (!ctx || (!text_host && n) || !n_out || (n_specials > 0 && (!specials_blob || !special_offs))) return BPE_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    BPE_TRY(ctx_load_text(ctx, text_host, n, false));
    const uint8_t *spb; const u32 *spo; u32 spmax;
    BPE_TRY(ctx_upload_specials(ctx, specials_blob, special_offs, n_specials, &spb, &spo, &spmax));
    u64 nn = n;
    BPE_TRY(ctx_run_flags(ctx, &nn, false, spb, spo, n_specials, spmax));
    u64 nw = (n + 31) / 32;
    size_t cnt_bytes = round_up((nw + 1) * sizeof(u32), 256), pre_bytes = round_up((nw + 2) * sizeof(u64), 256);
    BPE_TRY(bpe_buf_reserve(ctx, ctx->tmp0, cnt_bytes + pre_bytes + scan_tmp_elems_host(nw) * sizeof(u64)));
    u32 *cnt = (u32 *)ctx->tmp0.p;
    u64 *pre = (u64 *)((uint8_t *)ctx->tmp0.p + cnt_bytes);
    u64 *tmp = (u64 *)((uint8_t *)ctx->tmp0.p + cnt_bytes + pre_bytes);
    launch_popc_words((const u32 *)ctx->flags.p, nw, cnt, ctx->sm_count, st);
    launch_scan_u32(cnt, nw, pre, tmp, st);
    u64 *host = (u64 *)ctx->pinned;
    CUDA_TRY(ctx, cudaMemcpyAsync(host, pre + nw, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    u64 total = host[0];
    *n_out = total;
    if (!starts_out) return BPE_OK;
    u64 m = total < cap ? total : cap;
    if (m) {
        BPE_TRY(bpe_buf_reserve(ctx, ctx->tmp1, m * sizeof(u64)));
        launch_flags_to_offsets((const u32 *)ctx->flags.p, nw, pre, (u64 *)ctx->tmp1.p, m, ctx->sm_count, st);
        CUDA_TRY(ctx, cudaGetLastError());
        CUDA_TRY(ctx, cudaMemcpyAsync(starts_out, ctx->tmp1.p, m * sizeof(u64), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
    }
    return total > cap ? bpe_set_error(ctx, BPE_ERR_TOO_SMALL, "need room for %llu starts", (unsigned long long)total) : BPE_OK;
}
