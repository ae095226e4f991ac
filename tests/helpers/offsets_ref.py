"""Python reference of the token-offsets spec (bpe_encode_opts, include/bpe_sm100.h).  TEST INFRASTRUCTURE ONLY.

reference_offsets(otok, data, unit, ids=None) -> (ids, spans[n, 2]): segment `data` on the special tokens (leftmost, longest first), GPT-2
pretokens in between; the tokens of an occurrence tile it, each but the last as long as its vocabulary entry and the last up to the
occurrence's end, so a special-token occurrence spans the special's bytes whatever its id.  ids = None: every pretoken's ids from the
oracle on its own (deterministic BPE); otherwise `ids` (e.g. the dropout oracle's for the whole text) are split over the occurrences by
their vocabulary lengths.  "char" turns byte offsets into str indices with a count of UTF-8 lead bytes (chars_from_bytes)."""
from __future__ import annotations

import numpy as np

from oracle import oracle


def occurrences(data: bytes, specials) -> list[tuple[int, int, bool]]:
    """(start, end, is_special) of every pretoken occurrence of `data`, in order."""
    sp = sorted((s.encode() for s in specials), key=len, reverse=True)
    out, i = [], 0
    while i <= len(data):
        hit = None                               # the leftmost special occurrence from i; at a tie the longest (first in sp)
        for s in sp:
            k = data.find(s, i)
            if k >= 0 and (hit is None or k < hit[0]):
                hit = (k, s)
        end = hit[0] if hit else len(data)
        if end > i:
            st = oracle.pretokenize(data[i:end]) + [end - i]
            out += [(i + st[k], i + st[k + 1], False) for k in range(len(st) - 1)]
        if hit is None:
            return out
        out.append((end, end + len(hit[1]), True))
        i = end + len(hit[1])
    return out


def chars_from_bytes(data: bytes, spans: np.ndarray) -> np.ndarray:
    """Byte spans -> str index spans: start = index of the character holding the first byte, end = one past that of the last byte's."""
    lead = (np.frombuffer(data, dtype=np.uint8) & 0xC0) != 0x80
    before = np.zeros(len(data) + 1, dtype=np.int64)   # before[x] = characters that start before byte x
    np.cumsum(lead, out=before[1:])
    spans = np.asarray(spans, dtype=np.int64).reshape(-1, 2)
    return np.stack([before[spans[:, 0] + 1] - 1, before[spans[:, 1]]], axis=1)


def reference_offsets(otok, data: bytes, unit: str = "byte", ids=None) -> tuple[np.ndarray, np.ndarray]:
    vlen = {k: len(v) for k, v in otok.vocab.items() if isinstance(k, int) and isinstance(v, bytes)}
    given = None if ids is None else [int(x) for x in ids]
    out_ids, spans, pos = [], [], 0
    for s, e, is_sp in occurrences(data, otok.special_tokens):
        if is_sp:
            piece = [otok.vocab_inv[data[s:e]]] if given is None else given[pos: pos + 1]
        elif given is None:
            piece = otok.encode_bytes(data[s:e]).tolist()
        else:                                    # the ids whose vocabulary bytes make up this occurrence
            piece, k, filled = [], pos, 0
            while filled < e - s:
                piece.append(given[k]); filled += vlen[given[k]]; k += 1
            assert filled == e - s, (s, e, piece)
        pos += len(piece)
        x = s
        for k, tid in enumerate(piece):
            end = e if k + 1 == len(piece) else x + vlen[tid]
            spans.append((x, end))
            x = end
        out_ids += piece
    assert given is None or pos == len(given)
    spans = np.array(spans, dtype=np.int64).reshape(-1, 2)
    return np.array(out_ids, dtype=np.int64), chars_from_bytes(data, spans) if unit == "char" else spans
