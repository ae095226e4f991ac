// kernels.h -- host-callable launchers implemented across the .cu files.
#pragma once
#include "common.cuh"

// pretok.cu
int  pretok_upload_tables();
void launch_pretok_flags(const uint8_t *text, u64 n, const u32 *spmask, const u32 *spstart, u32 *flags, u64 *err,
                         u64 err_lo, u64 err_hi, int sm_count, cudaStream_t st);
void launch_newline_translate(const uint8_t *text, u64 n, uint8_t *out, u32 *tile_cnt, u64 *tile_off, u64 *scan_tmp,
                              cudaStream_t st);
u64  newline_tiles(u64 n);
void launch_special_split(const uint8_t *text, u64 n, const uint8_t *sp_blob_dev, const u32 *sp_offs_dev, int n_sp,
                          u32 max_len, u32 *cand, u32 *spstart, u32 *spmask, u64 n_words, int sm_count, cudaStream_t st);
void launch_popc_words(const u32 *flags, u64 n_words, u32 *cnt, int sm_count, cudaStream_t st);
void launch_popc_words16(const u32 *flags, u64 n_groups, u32 *cnt, int sm_count, cudaStream_t st);
void launch_flags_to_offsets(const u32 *flags, u64 n_words, const u64 *pre, u64 *out, u64 cap, int sm_count, cudaStream_t st);
void launch_copy_words2(const u32 *src, u32 *a, u32 *b, u64 n_words, int sm_count, cudaStream_t st);   // a[i] = b[i] = src[i]
void launch_scan_u32(const u32 *in, u64 n, u64 *out, u64 *tmp, cudaStream_t st);
size_t scan_tmp_elems_host(u64 n);
// Small control words WITHOUT the copy engines: while the pipelined entry points stream 256 MB chunks over PCIe, a 16-byte
// cudaMemcpyAsync on the compute stream queues behind the chunk in flight on the same copy engine and stalls the kernels after it
// for milliseconds (measured: upload and encode of bpe_encode ran one after the other, 280 ms instead of ~215 per 10 GB).
//   launch_poke: dst[0..n) = vals (device memory, n <= 8) by a one-thread kernel
//   launch_peek: host_dst[i] = src[idx ? idx[i] : i] -- the kernel writes straight into page-locked host memory (unified addressing);
//                valid after the stream has been synchronised
struct PokeVals { u64 v[8]; };
void launch_poke(u64 *dst, const PokeVals &vals, int n, cudaStream_t st);
void launch_peek(u64 *host_dst, const u64 *src, int n, cudaStream_t st);

// Geometry of the padded text arena (see common.cuh): payload at arena + BPE_PAD, 0xFF everywhere else,
// readable up to arena_bytes(n).
#define BPE_ARENA_ROUND 32768ull
static inline size_t arena_bytes(u64 n) { return (size_t)(BPE_PAD + round_up(n + 1, BPE_ARENA_ROUND) + BPE_ARENA_ROUND); }
static inline u64 flag_words(u64 n) { return round_up(n + 1, BPE_ARENA_ROUND) / 32 + 64; }
