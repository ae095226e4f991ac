/*
 * dropout_oracle.c -- CPU oracle of BPE-dropout (bpe_encode_ex with dropout > 0, spec at bpe_encode_opts in include/bpe_sm100.h).
 * TEST INFRASTRUCTURE ONLY, built at test time by tests/helpers/dropout_oracle.py.
 *
 * It compiles the CPU oracle (oracle/bpe_oracle.c) into the same unit and reuses its tokenizer tables, segmentation and GPT-2
 * pretokenizer; only the per-pretoken merge loop differs: in round t the candidate pair at token i is dropped when
 * (mix(mix(mix(mix(seed) ^ doc) ^ off_i) ^ t) >> 32) < thr, off_i = byte offset of token i in the document.
 */
#include "../../oracle/bpe_oracle.c"

typedef struct { uint64_t thr, h_doc, off; } drop_args;      /* h_doc = mix(mix(seed) ^ doc); off = the pretoken's offset */

static uint64_t splitmix64(uint64_t z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

/* encode_pretoken of the oracle with dropped candidates: they take no part in the minimum and are not merged */
static int drop_pretoken(const orc_tok *t, const uint8_t *p, uint32_t len, lvec *out, const uint8_t **kerr_p, uint32_t *kerr_len,
                         const drop_args *d) {
    uint32_t *cut = xmalloc(sizeof(uint32_t) * (len + 1));           /* tokens are contiguous slices cut[i]..cut[i+1] */
    uint8_t *dropped = xmalloc(len ? len : 1);
    uint32_t nt = len;
    for (uint32_t i = 0; i <= len; i++) cut[i] = i;
    for (uint32_t round = 0; nt > 1; round++) {
        int64_t best_rank = -1;
        for (uint32_t i = 0; i + 1 < nt; i++) {
            dropped[i] = 0;
            size_t s = bmap_get((bmap *)&t->merges, p + cut[i], cut[i + 2] - cut[i], cut[i + 1] - cut[i], 0, NULL);
            if (s == (size_t)-1) continue;
            if ((splitmix64(splitmix64(d->h_doc ^ (d->off + cut[i])) ^ round) >> 32) < d->thr) { dropped[i] = 1; continue; }
            int64_t r = t->merges.val[s];
            if (best_rank < 0 || r < best_rank) best_rank = r;
        }
        if (best_rank < 0) break;
        /* left to right, non-overlapping: the undropped candidates of the best rank (equal rank <=> the same pair) */
        uint32_t o = 0, i = 0;
        while (i < nt) {
            int merge = 0;
            if (i + 1 < nt && !dropped[i]) {
                size_t s = bmap_get((bmap *)&t->merges, p + cut[i], cut[i + 2] - cut[i], cut[i + 1] - cut[i], 0, NULL);
                merge = s != (size_t)-1 && t->merges.val[s] == best_rank;
            }
            cut[o++] = cut[i];
            i += merge ? 2 : 1;
        }
        cut[o] = len; nt = o;
    }
    int rc = 0;
    for (uint32_t i = 0; i < nt; i++) {
        size_t s = bmap_get((bmap *)&t->vocab_inv, p + cut[i], cut[i + 1] - cut[i], 0, 0, NULL);
        if (s == (size_t)-1) { *kerr_p = p + cut[i]; *kerr_len = cut[i + 1] - cut[i]; rc = -2; break; }
        lvec_push(out, t->vocab_inv.val[s]);
    }
    free(cut); free(dropped);
    return rc;
}

/* encode_segment of the oracle (tokenizer.py:68-77) with the pretoken's offset in the document */
static int drop_segment(const orc_tok *t, const uint8_t *seg, size_t n, lvec *out, const uint8_t **kerr_p, uint32_t *kerr_len,
                        drop_args d /* off = the segment's */) {
    cptext ct;
    if (cptext_decode(seg, n, &ct)) return -1;
    size_t i = 0; int rc = 0;
    while (i < ct.n && rc == 0) {
        size_t l = gpt2_match_len(&ct, i);
        const uint8_t *p = seg + ct.off[i]; size_t blen = ct.off[i + l] - ct.off[i];
        drop_args dp = d; dp.off = d.off + ct.off[i];
        if (!is_special(p, blen, t->sp_blob, t->sp_offs, t->n_sp))
            rc = drop_pretoken(t, p, (uint32_t)blen, out, kerr_p, kerr_len, &dp);
        i += l;
    }
    cptext_free(&ct);
    return rc;
}

/* orc_encode (tokenizer.py:111-138) with BPE-dropout; text = document `doc`.  Returns 0; -1 invalid UTF-8; -2 KeyError
 * (kerr_off/kerr_len = the missing token within text); -3 p outside [0, 1] or NaN.  Two-call idiom as orc_encode. */
ORC_API int orc_encode_dropout(const orc_tok *t, const uint8_t *text, uint64_t n, double p, uint64_t seed, uint64_t doc,
                               int64_t *ids, uint64_t cap, uint64_t *n_out, uint64_t *kerr_off, uint32_t *kerr_len) {
    if (!(p >= 0.0 && p <= 1.0)) return -3;
    drop_args d;
    d.thr = p == 1.0 ? (1ull << 32) : (uint64_t)(p * 4294967296.0);
    d.h_doc = splitmix64(splitmix64(seed) ^ doc);
    d.off = 0;
    lvec out = {0};
    int rc = 0; const uint8_t *kp = NULL; uint32_t kl = 0;
    size_t seg_start = 0, i = 0;
    while (i <= n && rc == 0) {                  /* segment (tokenizer.py:63-66): specials longest first */
        int hit = -1;
        if (i < n) for (int s = 0; s < t->n_sp; s++) {
            size_t l = t->sp_offs[s + 1] - t->sp_offs[s];
            if (l && i + l <= n && memcmp(text + i, t->sp_blob + t->sp_offs[s], l) == 0) { hit = s; break; }
        }
        if (hit >= 0 || i == n) {
            d.off = seg_start;
            if (i > seg_start) rc = drop_segment(t, text + seg_start, i - seg_start, &out, &kp, &kl, d);
            if (rc) break;
            if (hit >= 0) {
                size_t l = t->sp_offs[hit + 1] - t->sp_offs[hit];
                size_t s = bmap_get((bmap *)&t->vocab_inv, text + i, (uint32_t)l, 0, 0, NULL);
                if (s == (size_t)-1) { kp = text + i; kl = (uint32_t)l; rc = -2; break; }
                lvec_push(&out, t->vocab_inv.val[s]);
                i += l; seg_start = i;
                continue;
            }
            break;
        }
        i++;
    }
    if (rc == -2 && kerr_off) { *kerr_off = (uint64_t)(kp - text); *kerr_len = kl; }
    *n_out = out.n;
    if (rc == 0 && ids) memcpy(ids, out.v, sizeof(int64_t) * (out.n < cap ? out.n : cap));
    free(out.v);
    return rc;
}

/* u(seed, doc, off, t) of the spec (its test vectors) */
ORC_API uint64_t orc_dropout_u(uint64_t seed, uint64_t doc, uint64_t off, uint64_t round) {
    return splitmix64(splitmix64(splitmix64(splitmix64(seed) ^ doc) ^ off) ^ round);
}
