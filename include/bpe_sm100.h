/*
 * bpe_sm100.h -- C ABI of libbpe_sm100.so: the byte-level BPE hot path of gashon/transformer-lm
 * as hand-written sm_100a CUDA kernels.
 *
 * The reference has no native layer (it is pure Python), so every entry point below replaces a
 * Python function; the reference interface each one stands in for is cited as path:line relative
 * to the reference repository root.  All functions are extern "C", take plain pointers and sizes,
 * return an int status (0 = BPE_OK, negative = error) and never throw across the ABI.
 * bpe_last_error(ctx) returns a human-readable message for the last failing call on that context.
 *
 * Threading: one in-flight call per bpe_ctx (callers serialise); different contexts are independent.
 * Ownership: the caller allocates every output buffer; the library owns only device memory.
 */
#ifndef BPE_SM100_H
#define BPE_SM100_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BPE_OK                 0
#define BPE_ERR_ARG           -1   /* bad argument */
#define BPE_ERR_CUDA          -2   /* CUDA runtime error, see bpe_last_error */
#define BPE_ERR_OOM           -3   /* device or host allocation failed */
#define BPE_ERR_UTF8          -4   /* input is not valid UTF-8; detail = byte offset of the first bad sequence */
#define BPE_ERR_KEY           -5   /* KeyError: byte string / id missing from vocab; detail describes it */
#define BPE_ERR_CAPACITY      -6   /* an internal table overflowed even after growing */
#define BPE_ERR_TOO_SMALL     -7   /* caller's output buffer too small; *n_out holds the required size */
#define BPE_ERR_UNSUPPORTED   -8   /* input outside what this build supports (e.g. a pretoken > 16 MiB) */
#define BPE_ERR_NO_DEVICE     -9   /* no usable sm_100 device: the library has NO CPU fallback */
#define BPE_ERR_HALO          -10  /* a pretoken owned by the shard runs past its right halo: retry with a larger halo */
#define BPE_ERR_NEWLINE       -11  /* the shard contains '\r': newline translation shifts offsets, use the unsharded path */

typedef struct bpe_ctx bpe_ctx;   /* one per process per GPU: device, streams, workspaces */
typedef struct bpe_tok bpe_tok;   /* device-resident tokenizer (merge ranks, vocab, pretoken cache) */

/* ---- context ------------------------------------------------------------------------------- */
int  bpe_version(void);
/* Unicode table provenance, e.g. "regex-2026.3.32" (the tables reproduce that module's \s \p{L} \p{N}). */
const char *bpe_unicode_table_source(void);
int  bpe_ctx_create(int device, bpe_ctx **out);
void bpe_ctx_destroy(bpe_ctx *ctx);
const char *bpe_last_error(bpe_ctx *ctx);
/* Numeric detail of the last error (UTF-8 error offset, offending id, ...). */
int64_t bpe_last_error_detail(bpe_ctx *ctx);
int  bpe_device_sync(bpe_ctx *ctx);
/* Run all of this context's work on the caller's CUDA stream (e.g. torch.cuda.current_stream().cuda_stream) so
 * that the caller's events and collectives order with it; NULL restores the context's own stream. */
int  bpe_ctx_set_stream(bpe_ctx *ctx, void *cuda_stream);
/* Number of CUDA kernels this library has launched in this process (bench.py reports it as gpu_launches). */
unsigned long long bpe_launch_count(void);
/* Page-locked host memory for inputs/outputs (H2D / D2H copies from it run at PCIe speed). */
void *bpe_host_alloc(size_t bytes);
void  bpe_host_free(void *p);

/* ---- text-mode read semantics -------------------------------------------------------------- */
/* Replaces open(path, "r", encoding="utf-8").read()'s strict decode: models/tokenizer/train.py:21-23.
 * Returns BPE_OK or BPE_ERR_UTF8 (detail = UnicodeDecodeError.start). */
int bpe_utf8_validate(bpe_ctx *ctx, const uint8_t *text_host, uint64_t n);

/* ---- pretokenizer -------------------------------------------------------------------------- */
/* Replaces pattern.finditer(text) with the GPT-2 pattern: models/tokenizer/train.py:143-146,21-23 and
 * models/tokenizer/tokenizer.py:26-27,68-77.  Writes the byte offset of every pretoken start
 * (ascending).  Two-call idiom: starts_out == NULL only reports *n_out.
 * With n_specials > 0 the text is first split on the special tokens (leftmost, longest first):
 * tokenizer.py:63-66; each special occurrence is reported as one pretoken. */
int bpe_pretokenize(bpe_ctx *ctx, const uint8_t *text_host, uint64_t n,
                    const uint8_t *specials_blob, const uint32_t *special_offs, int n_specials,
                    uint64_t *starts_out, uint64_t cap, uint64_t *n_out);

/* ---- training ------------------------------------------------------------------------------ */
typedef struct bpe_train_stats {
    uint64_t n_bytes;            /* bytes after newline translation */
    uint64_t n_pretokens;        /* total pretoken occurrences */
    uint64_t n_unique;           /* unique pretokens (words) */
    uint64_t n_symbols;          /* total symbols over unique words at merge-loop start */
    uint64_t n_pairs_initial;    /* distinct adjacent byte pairs at start */
    uint64_t n_pairs_final;      /* distinct pair keys ever created (popped ones included); independent of the pair table's size and growth */
    uint64_t log_records;        /* inverted-index records written by the merge loop */
    uint64_t duplicate_tokens;   /* positive-count merges whose product bytes already existed (SURVEY A-6): provably 0, kept as an invariant check */
    uint64_t sum_live_pairs;     /* sum over merges of the live pair-table keys (what the reference's max() scans), every merge of a
                                    grid step charged the count at the start of the step (so it does not depend on the timing of
                                    the step's own insertions, but does depend on how merges are batched into steps) */
    uint64_t merge_steps;        /* grid steps of the merge loop (a step applies up to 12 merges, see csrc/merge.cuh) */
    float ms_h2d;                /* host->device copy of the text */
    float ms_validate;           /* UTF-8 validation + CR scan */
    float ms_pretok;             /* boundary-flag kernel */
    float ms_count;              /* pretoken hash-count kernel */
    float ms_build;              /* word list, initial pair table, inverted index */
    float ms_merge;              /* merge loop */
    float ms_total;              /* whole call, device timeline */
} bpe_train_stats;

/* Replaces train_bpe(input_path, vocab_size, special_tokens): models/tokenizer/train.py:142-231
 * (pretokenise + count: 16-28; byte-pair counts + inverted index: 31-49; merge loop: 183-228).
 * text_host = raw file bytes (strict UTF-8 check and universal-newline translation happen on the
 * device, as the reference's text-mode read does).  specials: pretokens EQUAL to a special are
 * dropped (train.py:25); specials are not split out (SURVEY A-1).
 * n_merges = vocab_size - len(Vocab(special_tokens)) is computed by the host (train.py:183).
 * merge_pairs_out[2*k], [2*k+1] = symbol ids of merge k: 0..255 are bytes, 256+j is the product
 * of merge j.  *n_done <= n_merges (the loop stops early when the pair table is empty, 184-185).
 * stats may be NULL. */
int bpe_train(bpe_ctx *ctx, const uint8_t *text_host, uint64_t n,
              const uint8_t *specials_blob, const uint32_t *special_offs, int n_specials,
              int n_merges, int32_t *merge_pairs_out, int *n_done, bpe_train_stats *stats);
/* Same, text already resident on this context's device (device pointer, >= 64 readable bytes of
 * slack after n are NOT required; the library copies into its padded arena). */
int bpe_train_dev(bpe_ctx *ctx, const uint8_t *text_dev, uint64_t n,
                  const uint8_t *specials_blob, const uint32_t *special_offs, int n_specials,
                  int n_merges, int32_t *merge_pairs_out, int *n_done, bpe_train_stats *stats);

/* Training options of the _ex entry points (an unknown bit is BPE_ERR_ARG).
 * BPE_TRAIN_SPLIT_SPECIALS (train_bpe(..., split_special_tokens=True)): training splits the text on the special tokens before
 * counting, the way the tokenizer splits it before encoding.  Without it training is bpe_train exactly (SURVEY A-1).
 *   1. The input is validated as strict UTF-8 over all of it (same BPE_ERR_UTF8 and detail = the first invalid byte of the whole
 *      input), then universal newlines are translated (A-2).
 *   2. The translated text is split on the special-token occurrences as Tokenizer.segment splits it: leftmost match, longest
 *      special first (re.split on the escaped alternation sorted by length, descending; the order of the caller's list does not
 *      matter).  A special containing '\r' never matches: the text holds no '\r' after translation.  An empty special matches
 *      nothing (empty specials are unsupported, DESIGN.md section 8).
 *   3. Every piece between occurrences is pretokenised on its own with the GPT-2 pattern, as a whole text (\s+(?!\S) sees the
 *      end of the text before an occurrence).
 *   4. Occurrences are counted nowhere: they add no word and no pair, and no word or merge crosses one.  stats->n_pretokens
 *      counts the ordinary pretokens only.
 *   5. The merge loop and everything after it are unchanged (vocab layout A-3, dedupe A-5, tie-break A-10, zero-count tail A-7).
 * Consequences: no learned token contains a special token (a piece holds no whole occurrence of one), and a text in which no
 * special occurs trains exactly as without the flag. */
#define BPE_TRAIN_SPLIT_SPECIALS 1
int bpe_train_ex(bpe_ctx *ctx, const uint8_t *text_host, uint64_t n,
                 const uint8_t *specials_blob, const uint32_t *special_offs, int n_specials,
                 int n_merges, int32_t *merge_pairs_out, int *n_done, bpe_train_stats *stats, int flags);
int bpe_train_dev_ex(bpe_ctx *ctx, const uint8_t *text_dev, uint64_t n,
                     const uint8_t *specials_blob, const uint32_t *special_offs, int n_specials,
                     int n_merges, int32_t *merge_pairs_out, int *n_done, bpe_train_stats *stats, int flags);

/* Sharded training (one process per GPU; SURVEY 8e).  A rank counts the pretokens that START in its
 * byte range of the file, exports its (word, count) table, the host exchanges tables (NCCL all-gather
 * via torch.distributed), every rank imports the other ranks' tables and runs the replicated merge
 * loop.  Replaces extract_subword_frequencies on a shard: train.py:16-28.
 *   shard = text_host[0..n) = file bytes [lo - halo_l, hi + halo_r); own_begin/own_end are offsets
 *   INSIDE shard delimiting the owned range; pretokens starting in [own_begin, own_end) are counted
 *   (they may extend past own_end into the right halo).  The shard must be cut on code-point
 *   boundaries and contain no '\r' (the host takes the single-GPU path otherwise). */
int bpe_count_begin(bpe_ctx *ctx);
/* BPE_ERR_UTF8 reports only ill-formed sequences that START in the owned range (detail = offset inside the
 * shard); BPE_ERR_HALO / BPE_ERR_NEWLINE as described above.  at_file_end: the shard ends where the file ends
 * (the last pretoken may then end at n); at_file_start is informational. */
int bpe_count_add_shard(bpe_ctx *ctx, const uint8_t *text_host, uint64_t n,
                        uint64_t own_begin, uint64_t own_end, int at_file_start, int at_file_end);
int bpe_count_add_shard_dev(bpe_ctx *ctx, const uint8_t *text_dev, uint64_t n,
                            uint64_t own_begin, uint64_t own_end, int at_file_start, int at_file_end);
/* Same with the training options.  flags == 0 is bpe_count_add_shard (the specials are unused).  With BPE_TRAIN_SPLIT_SPECIALS
 * the shard is split on the specials (bpe_train_ex) and counted as one whole text: the host cuts the file only at exact
 * boundaries (the start of a special-token occurrence that no occurrence covers from the left, or a single U+0020 between two
 * ASCII non-space bytes that no occurrence covers), where splitting and pretokenisation on both sides do not depend on the other.
 * own_begin must be 0 and own_end n (BPE_ERR_ARG otherwise); there is no halo, BPE_ERR_HALO cannot occur. */
int bpe_count_add_shard_ex(bpe_ctx *ctx, const uint8_t *text_host, uint64_t n,
                           uint64_t own_begin, uint64_t own_end, int at_file_start, int at_file_end,
                           const uint8_t *specials_blob, const uint32_t *special_offs, int n_specials, int flags);
int bpe_count_add_shard_dev_ex(bpe_ctx *ctx, const uint8_t *text_dev, uint64_t n,
                               uint64_t own_begin, uint64_t own_end, int at_file_start, int at_file_end,
                               const uint8_t *specials_blob, const uint32_t *special_offs, int n_specials, int flags);
/* Export sizes, then the table itself: blob = concatenated word bytes, offs[n_words+1], counts[n_words]. */
int bpe_count_export_size(bpe_ctx *ctx, uint64_t *n_words, uint64_t *blob_bytes);
int bpe_count_export(bpe_ctx *ctx, uint8_t *blob, uint64_t *offs, int64_t *counts);
/* Same with device pointers (the buffers an NCCL all-gather then moves between ranks). */
int bpe_count_export_dev(bpe_ctx *ctx, uint8_t *blob_dev, uint64_t *offs_dev, int64_t *counts_dev);
/* Add another rank's table to this context's counts. */
int bpe_count_import(bpe_ctx *ctx, const uint8_t *blob, const uint64_t *offs, const int64_t *counts, uint64_t n_words);
int bpe_count_import_dev(bpe_ctx *ctx, const uint8_t *blob_dev, const uint64_t *offs_dev, const int64_t *counts_dev,
                         uint64_t n_words, uint64_t blob_bytes);
/* Dense 256x256 table of adjacent byte-pair counts over the words counted so far (pair (a,b) at [a*256+b]):
 * calculate_byte_pair_frequencies at merge-loop start, models/tokenizer/train.py:35-49.  It is linear in the
 * word counts, so the per-rank tables sum (NCCL all-reduce) to the table of the merged counts. */
int bpe_count_pair_table(bpe_ctx *ctx, const uint8_t *specials_blob, const uint32_t *special_offs, int n_specials,
                         int64_t *dense_out /* 65536, host */);
/* Merge loop over whatever has been counted/imported so far. */
int bpe_train_from_counts(bpe_ctx *ctx, const uint8_t *specials_blob, const uint32_t *special_offs, int n_specials,
                          int n_merges, int32_t *merge_pairs_out, int *n_done, bpe_train_stats *stats);
/* Live view of the merge loop (train.py:183-228 appends to `merges` one pair at a time; a host that has to turn the symbol ids into
 * its own objects -- the reference's `list[tuple[bytes, bytes]]` and vocab dict -- can do so WHILE the loop runs instead of after it).
 * During the merge loop of every later bpe_train / bpe_train_dev / bpe_train_from_counts call on this context the kernel stores merge
 * k's symbol ids into live_pairs[2k], [2k+1] with ONE 8-byte store as soon as the merge is made.  live_pairs must be page-locked host
 * memory (bpe_host_alloc) of capacity_merges entries; the caller fills it with -1 before the training call and treats an entry as
 * complete when it is non-negative (entries may become visible out of order).  merge_pairs_out of the training call remains the
 * authoritative result.  NULL switches it off. */
int bpe_train_set_live(bpe_ctx *ctx, int32_t *live_pairs, int capacity_merges);
/* The dense 256 x 256 byte-pair table (calculate_byte_pair_frequencies over single bytes, train.py:35-49) that the last
 * bpe_train / bpe_train_dev / bpe_train_from_counts call on this context built before its first merge: the multi-GPU path
 * checks it against the all-reduced per-rank tables of bpe_count_pair_table without building the table a second time. */
int bpe_last_pair_table(bpe_ctx *ctx, int64_t *dense_out /* [65536] */);

/* ---- tokenizer ----------------------------------------------------------------------------- */
/* Replaces Tokenizer.__init__ table building: models/tokenizer/tokenizer.py:12-38 and the per-call
 * inv_merges dict (115).  The reference identifies tokens by their byte strings; the host turns them into
 * integer symbols: 0..255 = single bytes, 256.. = every distinct byte string a+b over the merge list.
 *   merge_pairs[2*j], [2*j+1]   operand symbols of merge j (its rank is j), or -1,-1 for an entry that can
 *                               never apply (operand is not a symbol, or a later duplicate of the same pair
 *                               overrides it: {pair: i for i, pair in enumerate(merges)} keeps the LAST i)
 *   merge_result[j]             symbol of a+b
 *   sym_to_id[s]                vocab_inv[bytes(s)], or -1 when absent (KeyError when such a token is emitted,
 *                               tokenizer.py:135)
 *   sym_blob/sym_offs           bytes of every symbol (used to report the KeyError key)
 *   vocab_blob/offs/ids         id -> bytes table for decode (ids need not be dense)
 *   specials                    longest first; special_ids[i] = vocab_inv[special] (or -1 -> KeyError when met) */
int bpe_tok_create(bpe_ctx *ctx,
                   const int32_t *merge_pairs, const int32_t *merge_result, int n_merges,
                   const int32_t *sym_to_id, const uint8_t *sym_blob, const uint64_t *sym_offs, int n_syms,
                   const uint8_t *vocab_blob, const uint64_t *vocab_offs, const int64_t *vocab_ids, int64_t n_vocab,
                   const uint8_t *specials_blob, const uint32_t *special_offs, const int64_t *special_ids, int n_specials,
                   bpe_tok **out);
void bpe_tok_destroy(bpe_tok *tok);

#define BPE_DTYPE_U16 0
#define BPE_DTYPE_I32 1

typedef struct bpe_encode_stats {
    uint64_t n_bytes, n_pretokens, n_tokens;
    uint64_t cache_new_unique;   /* pretokens BPE-merged in this call (cache misses) */
    float ms_h2d, ms_pretok, ms_lookup, ms_bpe, ms_emit, ms_d2h, ms_total;
} bpe_encode_stats;

/* Replaces Tokenizer.encode(text): models/tokenizer/tokenizer.py:111-138 (segment 63-66, pretokenize
 * 79-90, merge 92-109).  text_host is UTF-8 (validated; BPE_ERR_UTF8 otherwise).  Two-call idiom:
 * out == NULL reports *n_out only; otherwise at most cap ids are written and BPE_ERR_TOO_SMALL is
 * returned if cap < *n_out.  BPE_ERR_KEY mirrors the KeyError of tokenizer.py:120,135:
 * bpe_tok_key_error() then yields the offending byte string.  BPE_DTYPE_U16 with an id > 65535
 * returns BPE_ERR_ARG (the reference's np.uint16 cast at models/tokenizer/encode.py:37 would wrap). */
int bpe_encode(bpe_tok *tok, const uint8_t *text_host, uint64_t n, int out_dtype,
               void *out, uint64_t cap, uint64_t *n_out, bpe_encode_stats *stats);
/* bpe_encode_ex: bpe_encode with options -- documents, BPE-dropout and token offsets, each independent of the others; opts == NULL,
 * or a zero-filled struct, is bpe_encode exactly.  BPE_ERR_ARG, checked in this order: a null tokenizer, an unknown offset_unit (with
 * offsets), a null offs_out (with offsets and out != NULL), dropout outside [0, 1] or NaN, then document offsets that are not as
 * described below (BPE_ERR_UNSUPPORTED after them when there is no boundary byte). */
typedef struct bpe_encode_opts {
    /* Documents: replaces [Tokenizer.encode(d) for d in docs]: models/tokenizer/tokenizer.py:111-138 once per document.
     * doc_offs == NULL: the text is one document (bpe_encode), n_docs must be 0 and id_offs_out is unused.  Otherwise
     * text_host holds n_docs UTF-8 documents back to back, document j = text[doc_offs[j] .. doc_offs[j+1])
     * (doc_offs[0] = 0, doc_offs[n_docs] = n, non-decreasing); an empty batch passes the one-element array {0}.  Writes the ids of
     * all documents back to back and id_offs_out[j] (n_docs + 1 entries, required) = index of document j's first id.  Same
     * size-query idiom, dtypes and errors as bpe_encode; BPE_ERR_UTF8 / BPE_ERR_KEY detail = byte offset in text_host.  Every
     * document is encoded on its own: no pretoken or special-token occurrence spans two documents, and UTF-8 validity is per
     * document.  The error reported is the first one the device meets: an invalid UTF-8 sequence anywhere in a pipeline chunk
     * (256 MB of documents) comes before a KeyError in it, so a caller that needs the first failing document in list order
     * re-encodes the documents before the invalid one (Tokenizer.encode_batch does).  BPE_ERR_UNSUPPORTED when every ASCII byte
     * but '\r' occurs in some special token (the boundary byte between documents must occur in none).  bpe_tok_saw_cr afterwards:
     * a '\r' in any document. */
    const uint64_t *doc_offs;
    uint64_t n_docs;
    uint64_t *id_offs_out;
    /* BPE-dropout (subword regularisation, Provilkov et al. 2020): dropout = p in (0, 1], the encode where every pretoken occurrence
     * gets its own random segmentation; p = 0 is the deterministic encode.  Same two-call idiom (out == NULL reports the same
     * *n_out), dtypes, errors, error details and bpe_tok_saw_cr as the deterministic calls; BPE_ERR_ARG when p is outside [0, 1] or
     * NaN.  The result is a pure function of (tokenizer, text, document split, p, seed): it does not depend on the pretoken cache or
     * on how the library cuts the text.
     *   mix(z): z += 0x9E3779B97F4A7C15; z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9; z = (z ^ (z >> 27)) * 0x94D049BB133111EB;
     *           return z ^ (z >> 31)                                                         (splitmix64 finalizer, all mod 2^64)
     *   u(seed, doc, off, t) = mix(mix(mix(mix(seed) ^ doc) ^ off) ^ t)
     *   thr(p) = 2^32 if p == 1 else floor(p * 2^32)
     *   dropped = (u(seed, doc, off, t) >> 32) < thr(p)
     * doc = the document's index (0 when doc_offs == NULL), off = byte offset in that document of the first byte of the candidate
     * pair's left token, t = the 0-based merge round within the pretoken occurrence.  BPE of one occurrence (the merge loop of
     * models/tokenizer/tokenizer.py:92-109,124-136 with candidates removed at random):
     *   tokens = the pretoken's bytes; t = 0
     *   loop: cand = { i : (tokens[i], tokens[i+1]) has a merge rank and not dropped(seed, doc, off_i, t) }
     *         if cand is empty: stop
     *         r = min rank over cand; scan i left to right: if i in cand and rank(i) == r: merge i, i+1 and i += 2, else i += 1
     *         t += 1
     *   ids = vocab_inv[token] for each token (a missing token is BPE_ERR_KEY, as in tokenizer.py:135)
     * Special-token occurrences are one id and never split.  p = 0 gives exactly the deterministic encode; p = 1 gives every
     * pretoken as single bytes.  Dropout can emit tokens deterministic BPE never does, so with a vocabulary that lacks an
     * intermediate merge product one of the two calls can raise a KeyError the other does not. */
    double dropout;
    uint64_t seed;
    /* Token offsets (with_offsets != 0): the ids of the same call without offsets, and for every token i its span [start_i, end_i)
     * of the input, offs_out[2 i], offs_out[2 i + 1] (int64, cap x 2 entries).  Same two-call idiom (out == NULL reports *n_out and
     * writes no offsets; otherwise offs_out must be given), dtypes, errors in the same order and error details; BPE_ERR_ARG for an
     * unknown offset_unit.
     *   BPE_OFF_BYTES  the bytes token i was produced from.  The spans tile the document in order (start_0 = 0, end_i = start_{i+1}, the last
     *                  end = its length).  The tokens of a pretoken occurrence tile it; each but its last is as long as its vocabulary entry
     *                  and the last ends where the pretoken ends.  So data[start:end] == vocab[id] for an ordinary token, and a special-token
     *                  occurrence spans the special's bytes whatever its id (also an id missing from the vocabulary or shared with another
     *                  token, SURVEY A-12).
     *   BPE_OFF_CHARS  Python str indices: start = index of the character that holds the token's first byte, end = one past the index of the
     *                  character that holds its last byte.  A token that splits a multi-byte character maps to the whole character, so the
     *                  spans of the tokens that share it overlap by one (as HF byte-level offsets do): text[start:end].encode() always
     *                  contains the token's bytes, and equals them when no character is split.
     * With documents: spans are relative to each document's start, as if it were encoded on its own.  The spans depend only on the
     * text, the document split, p and seed: not on the pretoken cache, how the library cuts the text, or the batch size. */
    int with_offsets;
    int offset_unit;
    int64_t *offs_out;
} bpe_encode_opts;
#define BPE_OFF_BYTES 0
#define BPE_OFF_CHARS 1
int bpe_encode_ex(bpe_tok *tok, const uint8_t *text_host, uint64_t n, const bpe_encode_opts *opts,
                  int out_dtype, void *out, uint64_t cap, uint64_t *n_out, bpe_encode_stats *stats);
/* 1 if the text of the last bpe_encode* call on this tokenizer's context held a carriage return (the flags kernel
 * sees every byte anyway).  Tokenizer.encode takes a str and keeps '\r' as it is; a caller that reads a FILE in text mode, like the
 * reference's bulk driver (models/tokenizer/encode.py:31-34, universal newlines), uses this instead of scanning the text on the host:
 * it translates and encodes the piece again in the rare case. */
int bpe_tok_saw_cr(bpe_tok *tok);
/* Device-resident variant: text_dev and out_dev are device pointers on the tokenizer's device. */
int bpe_encode_dev(bpe_tok *tok, const uint8_t *text_dev, uint64_t n, int out_dtype,
                   void *out_dev, uint64_t cap, uint64_t *n_out, bpe_encode_stats *stats);
int bpe_tok_key_error(bpe_tok *tok, uint8_t *buf, uint64_t cap, uint64_t *len);
/* Drop the device pretoken->ids cache (it is also dropped automatically when it fills). */
int bpe_tok_cache_reset(bpe_tok *tok);

/* Replaces the byte part of Tokenizer.decode(ids): b"".join(vocab[i] for i in ids),
 * models/tokenizer/tokenizer.py:155-157 (the host applies .decode("utf-8", errors="replace")).
 * BPE_ERR_KEY (detail = index into ids) when an id is not in the vocab. */
int bpe_decode(bpe_tok *tok, const int64_t *ids_host, uint64_t n, uint8_t *out, uint64_t cap, uint64_t *n_out);
/* Batched form for samplers that decode many sequences at once (models/transformer/decode.py:51 calls
 * tokenizer.decode once per generated sequence): ids_host holds n_seq sequences back to back, sequence j =
 * ids[seq_offs[j] .. seq_offs[j+1]) (seq_offs[0] = 0, seq_offs[n_seq] = n).  One decode of the concatenation;
 * byte_offs_host[j] (n_seq + 1 entries) = where sequence j starts in `out`.  Same size-query idiom and errors. */
int bpe_decode_batch(bpe_tok *tok, const int64_t *ids_host, uint64_t n, const uint64_t *seq_offs_host, uint64_t n_seq,
                     uint8_t *out, uint64_t cap, uint64_t *n_out, uint64_t *byte_offs_host);

/* ---- training-batch feeder (SURVEY 8f row 4) --------------------------------------------------
 * Replaces the per-row loop of load_batch, models/util.py:37-57: for r < batch and c < context
 *   x[r][c] = tokens[starts[r] + c],  y[r][c] = tokens[starts[r] + c + 1]      (int64, row-major)
 * tokens_dev: the encoder's uint16 / int32 id array resident in HBM (BPE_DTYPE_*), n_tokens entries;
 * starts_host: the `batch` start indices (the reference draws them with torch.randint(len - context) on
 * the host; the caller keeps doing that, so a given generator yields the same batches);
 * x_dev, y_dev: device buffers of batch * context int64.  BPE_ERR_ARG (detail = row) when a window leaves
 * the array. */
int bpe_batch_windows_dev(bpe_ctx *ctx, const void *tokens_dev, int dtype, uint64_t n_tokens, const int64_t *starts_host,
                          uint32_t batch, uint32_t context, int64_t *x_dev, int64_t *y_dev);

/* ---- synthetic corpora (bench/test infrastructure; SURVEY 8d) -------------------------------- */
#define BPE_SYNTH_TINYSTORIES 0
#define BPE_SYNTH_OWT         1
/* Fill out_dev[0..n) (device pointer) with deterministic synthetic UTF-8 text of the given shape.
 * The text is a pure function of (shape, seed, n); bpe_synth_host produces the identical bytes on
 * the CPU (same code compiled for the host) so CPU oracles can be fed the same input. */
int bpe_synth_dev(bpe_ctx *ctx, int shape, uint64_t seed, uint8_t *out_dev, uint64_t n);
int bpe_synth_host(int shape, uint64_t seed, uint8_t *out_host, uint64_t n);
/* Same, starting at 4096-byte block `first_block` of the corpus (a rank generates only its shard). */
int bpe_synth_dev_at(bpe_ctx *ctx, int shape, uint64_t seed, uint64_t first_block, uint8_t *out_dev, uint64_t n);
int bpe_synth_host_at(int shape, uint64_t seed, uint64_t first_block, uint8_t *out_host, uint64_t n);

#ifdef __cplusplus
}
#endif
#endif /* BPE_SM100_H */
