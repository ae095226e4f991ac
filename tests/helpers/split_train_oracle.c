/*
 * split_train_oracle.c -- CPU oracle of training with split_special_tokens (BPE_TRAIN_SPLIT_SPECIALS, spec in
 * include/bpe_sm100.h).  TEST INFRASTRUCTURE ONLY, built at test time by tests/helpers/split_train_oracle.py.
 *
 * It compiles the CPU oracle (oracle/bpe_oracle.c) into the same unit and reuses its UTF-8 check, newline translation, GPT-2
 * counter and trainer helpers; only the counting differs: the translated text is cut at the special-token occurrences with the
 * oracle's segmentation (orc_encode: leftmost match, specials longest first, scanning resumes after a match) and every piece is
 * counted on its own.  The occurrences are counted nowhere.
 */
#include "../../oracle/bpe_oracle.c"

/* The merge loop of orc_train_bpe (train.py:165-228) on words counted elsewhere: the oracle's code from the word list on, over
 * its own trainer helpers (freq_touch, add_token, pair_key_greater, ...).  orc_train_bpe counts the whole text itself, so its
 * loop cannot be handed the split-mode words; tests/test_train_split_cpu.py pins this copy to orc_train_bpe on texts without
 * special-token occurrences, where both modes must agree. */
static void train_from_words(const bmap *words_in, int n_merges, int32_t *merge_pairs, int *n_done) {
    const bmap words = *words_in;
    trainer T; memset(&T, 0, sizeof(T));
    T.tok_cap = 512; T.tok = xmalloc(T.tok_cap * sizeof(uint8_t *)); T.tok_len = xmalloc(T.tok_cap * sizeof(uint32_t));
    bmap_init(&T.tok_by_bytes, 1 << 12);
    for (int i = 0; i < 256; i++) {
        T.tok[i] = xmalloc(1); T.tok[i][0] = (uint8_t)i; T.tok_len[i] = 1;
        size_t s = bmap_get(&T.tok_by_bytes, T.tok[i], 1, 0, 1, NULL); T.tok_by_bytes.val[s] = i;
    }
    T.n_tok = 256;
    T.pairs_cap = 1024; T.pairs = xmalloc(T.pairs_cap * sizeof(pair_ent));
    T.pm_cap = 1 << 12; T.pm_key = xmalloc(T.pm_cap * sizeof(uint64_t)); T.pm_val = xmalloc(T.pm_cap * sizeof(int32_t));
    for (size_t i = 0; i < T.pm_cap; i++) T.pm_val[i] = -1;

    /* encode_subwords (train.py:31-32): word -> list of single-byte symbols */
    size_t W = words.cnt;
    int32_t **w = xmalloc(W * sizeof(int32_t *));
    uint32_t *wl = xmalloc(W * sizeof(uint32_t));
    int64_t *wf = xmalloc(W * sizeof(int64_t));
    for (size_t i = 0; i < W; i++) {
        size_t s = words.order[i];
        wl[i] = words.klen[s]; wf[i] = words.val[s];
        w[i] = xmalloc(sizeof(int32_t) * (wl[i] ? wl[i] : 1));
        for (uint32_t j = 0; j < wl[i]; j++) w[i][j] = words.pool[words.koff[s] + j];
    }
    /* calculate_byte_pair_frequencies (train.py:35-49) */
    for (size_t i = 0; i < W; i++)
        for (uint32_t j = 0; j + 1 < wl[i]; j++) {
            pair_ent *p = freq_touch(&T, w[i][j], w[i][j + 1]);
            p->count += wf[i];
            if (p->words.n == 0 || p->words.v[p->words.n - 1] != (int32_t)i) ivec_push(&p->words, (int32_t)i);
        }

    /* merge loop (train.py:183-228) */
    for (int step = 0; step < n_merges; step++) {
        /* len(byte_pair_frequencies) == 0 -> break (184-185); max over ALL keys incl. count 0 (187-189) */
        int32_t best = -1;
        for (size_t i = 0; i < T.n_pairs; i++) {
            if (!T.pairs[i].alive) continue;
            if (best < 0 || pair_key_greater(&T, &T.pairs[i], &T.pairs[best])) best = (int32_t)i;
        }
        if (best < 0) break;
        int32_t a = T.pairs[best].a, b = T.pairs[best].b;
        int32_t nw = add_token(&T, a, b);                 /* new_byte = a + b (190) */
        /* subword_indices = list(token_indices[best_pair].keys()) (192): snapshot */
        size_t nidx = T.pairs[best].words.n;
        int32_t *idx = xmalloc(sizeof(int32_t) * (nidx ? nidx : 1));
        memcpy(idx, T.pairs[best].words.v, sizeof(int32_t) * nidx);
        for (size_t q = 0; q < nidx; q++) {
            int32_t wi = idx[q];
            int32_t *sw = w[wi]; int64_t c = wf[wi];
            uint32_t bi = 0;
            while (wl[wi] >= 2 && bi < wl[wi] - 1) {      /* 196-224 */
                if (sw[bi] == a && sw[bi + 1] == b) {
                    /* update_frequencies_after_merge (52-78) on the not-yet-spliced word */
                    if (bi > 0) {
                        freq_touch(&T, sw[bi - 1], sw[bi])->count -= c;
                        freq_touch(&T, sw[bi - 1], nw)->count += c;
                    }
                    if (bi + 2 < wl[wi]) {
                        freq_touch(&T, sw[bi + 1], sw[bi + 2])->count -= c;
                        freq_touch(&T, nw, sw[bi + 2])->count += c;
                    }
                    /* update_token_indices (81-104) never deletes anything (SURVEY A-9) */
                    /* merge_subwords (132-139) */
                    sw[bi] = nw;
                    memmove(sw + bi + 1, sw + bi + 2, sizeof(int32_t) * (wl[wi] - bi - 2));
                    wl[wi]--;
                    /* create_new_token_indices (107-129) */
                    if (bi > 0) ivec_push(&freq_touch(&T, sw[bi - 1], sw[bi])->words, wi);
                    if (bi + 1 < wl[wi]) ivec_push(&freq_touch(&T, sw[bi], sw[bi + 1])->words, wi);
                }
                bi++;
            }
        }
        free(idx);
        /* pop best from both dicts (226-227), merges.append (228) */
        pair_ent *bp = &T.pairs[pm_find(&T, a, b, 0)];
        bp->alive = 0; bp->words.n = 0;
        merge_pairs[2 * step] = a; merge_pairs[2 * step + 1] = b;
        *n_done = step + 1;
    }

    for (size_t i = 0; i < W; i++) free(w[i]);
    free(w); free(wl); free(wf);
    for (size_t i = 0; i < T.n_pairs; i++) free(T.pairs[i].words.v);
    free(T.pairs); free(T.pm_key); free(T.pm_val);
    for (size_t i = 0; i < T.n_tok; i++) free(T.tok[i]);
    free(T.tok); free(T.tok_len); bmap_free(&T.tok_by_bytes);
}

/* the words of every piece of `text` (translated) between special occurrences; specials longest first */
static int split_count(const uint8_t *text, size_t n, const uint8_t *sp_blob, const uint32_t *sp_offs, int n_sp, bmap *m) {
    size_t seg_start = 0, i = 0;
    while (i <= n) {
        int hit = -1;
        if (i < n) for (int s = 0; s < n_sp; s++) {
            size_t l = sp_offs[s + 1] - sp_offs[s];
            if (l && i + l <= n && memcmp(text + i, sp_blob + sp_offs[s], l) == 0) { hit = s; break; }
        }
        if (hit >= 0 || i == n) {
            if (i > seg_start && count_pretokens(text + seg_start, i - seg_start, NULL, NULL, 0, m)) return -1;
            if (hit < 0) break;
            i += sp_offs[hit + 1] - sp_offs[hit];
            seg_start = i;
            continue;
        }
        i++;
    }
    return 0;
}

/* raw bytes -> validated, translated, split and counted words; -1 (*err_off) on invalid UTF-8 */
static int split_words(const uint8_t *text_in, uint64_t n_in, const uint8_t *sp_blob, const uint32_t *sp_offs, int n_sp,
                       bmap *m, int64_t *err_off) {
    int64_t bad = orc_utf8_validate(text_in, n_in);
    if (bad >= 0) { if (err_off) *err_off = bad; return -1; }
    uint8_t *text = xmalloc(n_in ? n_in : 1);
    uint64_t n = orc_universal_newlines(text_in, n_in, text);
    bmap_init(m, 1 << 12);
    split_count(text, n, sp_blob, sp_offs, n_sp, m);
    free(text);
    return 0;
}

/* The split-mode words of the raw bytes in first-occurrence order: returns their number (-1 on invalid UTF-8); with out_blob,
 * out_offs and out_counts (sized by a first call) fills them as orc_count_pretokens does. */
ORC_API int64_t orc_split_count(const uint8_t *text_in, uint64_t n_in, const uint8_t *sp_blob, const uint32_t *sp_offs, int n_sp,
                                uint8_t *out_blob, uint64_t *out_offs, int64_t *out_counts, uint64_t *blob_bytes) {
    bmap m;
    if (split_words(text_in, n_in, sp_blob, sp_offs, n_sp, &m, NULL)) return -1;
    if (blob_bytes) *blob_bytes = m.pool_n;
    if (out_blob && out_offs && out_counts) {
        uint64_t o = 0;
        for (size_t i = 0; i < m.cnt; i++) {
            size_t s = m.order[i];
            memcpy(out_blob + o, m.pool + m.koff[s], m.klen[s]);
            out_offs[i] = o; o += m.klen[s];
            out_counts[i] = m.val[s];
        }
        out_offs[m.cnt] = o;
    }
    int64_t r = (int64_t)m.cnt;
    bmap_free(&m);
    return r;
}

/* orc_train_bpe with split_special_tokens: the same outputs and error convention */
ORC_API int orc_split_train_bpe(const uint8_t *text_in, uint64_t n_in, const uint8_t *sp_blob, const uint32_t *sp_offs, int n_sp,
                                int n_merges, int32_t *merge_pairs, int *n_done, int64_t *err_off) {
    *n_done = 0;
    bmap words;
    if (split_words(text_in, n_in, sp_blob, sp_offs, n_sp, &words, err_off)) return -1;
    train_from_words(&words, n_merges, merge_pairs, n_done);
    bmap_free(&words);
    return 0;
}
