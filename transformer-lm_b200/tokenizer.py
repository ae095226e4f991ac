"""Tokenizer host: mirrors models/tokenizer/tokenizer.py:11-167 of the reference.

    Tokenizer(vocab, merges, special_tokens).encode(str, *, dropout=0.0, seed=0) -> list[int]
                                            .encode_batch(Sequence[str]) -> list[list[int]]
                                            .encode_iterable(Iterable[str]) -> Iterator[int]
                                            .encode_with_offsets(str) -> (list[int], list[(start, end)])
                                            .decode(list[int]) -> str

encode / decode run on the GPU through the C ABI (bpe_tok_create / bpe_encode / bpe_decode in
include/bpe_sm100.h).  The host turns the reference's byte-string tokens into integer symbols once per
tokenizer; nothing here re-implements the algorithm on the CPU (there is no fallback).
"""
from __future__ import annotations

import ctypes as C
import os
import pickle
from typing import Iterable, Iterator, List, Sequence, Tuple

import numpy as np

from . import _lib
from .train import train_bpe

_CHUNK_CHARS = 1024 * 1024 * 2                   # tokenizer.py:145


def _pack_documents(texts: list) -> Tuple[np.ndarray, np.ndarray, UnicodeEncodeError | None]:
    """(UTF-8 bytes of all documents back to back as uint8, uint64 byte offsets (len + 1), None), or -- when item k is a str that
    cannot be encoded (a lone surrogate) -- the packing of the items before it and the error."""
    try:
        joined = "".join(texts)
    except TypeError:                            # some items are bytes
        joined = None
    if joined is not None and joined.isascii():  # one byte per character: no per-item encode
        lens = np.fromiter(map(len, texts), dtype=np.uint64, count=len(texts))
        parts, bad = [joined.encode("ascii")], None
    else:
        parts, bad = [], None
        for t in texts:
            if isinstance(t, str):
                try:
                    t = t.encode("utf-8")
                except UnicodeEncodeError as e:
                    bad = e
                    break
            parts.append(t)
        lens = np.fromiter(map(len, parts), dtype=np.uint64, count=len(parts))
    offs = np.zeros(lens.size + 1, dtype=np.uint64)
    np.cumsum(lens, out=offs[1:])
    return np.frombuffer(b"".join(parts), dtype=np.uint8), offs, bad


def _check_dropout(dropout, seed) -> Tuple[float, int]:
    """BPE-dropout arguments: a probability in [0, 1] and a seed in [0, 2**64)."""
    p = float(dropout)
    if not 0.0 <= p <= 1.0:                      # (also rejects NaN)
        raise ValueError("dropout must be a probability in [0, 1], got %r" % (dropout,))
    if isinstance(seed, bool) or not isinstance(seed, (int, np.integer)) or not 0 <= int(seed) < 2**64:
        raise ValueError("seed must be an integer in [0, 2**64), got %r" % (seed,))
    return p, int(seed)


_UNITS = {"byte": _lib.OFF_BYTES, "char": _lib.OFF_CHARS}


def _check_unit(unit) -> int:
    """Offset unit of the *_offsets calls: "byte" (offsets into the UTF-8 bytes) or "char" (Python str indices)."""
    if not isinstance(unit, str) or unit not in _UNITS:
        raise ValueError("unit must be 'byte' or 'char', got %r" % (unit,))
    return _UNITS[unit]


class Tokenizer:
    def __init__(self, vocab: dict[int, bytes], merges: List[Tuple[bytes, bytes]], special_tokens: List[str] | None = [], *, ctx=None):
        # same attribute names and the same (quirky) mutations as tokenizer.py:18-38
        self.vocab = vocab
        self.vocab_inv = {v: k for k, v in vocab.items()}
        self.merges = merges
        self.special_tokens = list(set(special_tokens or []))
        self.special_tokens.sort(key=len, reverse=True)
        for token in self.special_tokens:        # SURVEY A-12: key and value are swapped in the reference
            tb = token.encode("utf-8")
            if tb not in self.vocab_inv:
                self.vocab[tb] = len(self.vocab)
                self.vocab_inv[tb] = len(self.vocab) - 1
        self._ctx = ctx
        self._tok = None                         # bpe_tok*, built on first use
        self._sig = None
        self.last_stats: dict | None = None

    # ---- constructors (tokenizer.py:40-61) -------------------------------------------------------
    @classmethod
    def train_from_file(cls, filepath: str, vocab_size: int, special_tokens: List[str], *, split_special_tokens: bool = False):
        """split_special_tokens=True trains on the text split at the special tokens, as encode splits it (train.train_bpe)."""
        vocab, merges = train_bpe(filepath, vocab_size, special_tokens, split_special_tokens=split_special_tokens)
        return cls(vocab, merges, special_tokens)

    @classmethod
    def fit(cls, input_path: str, vocab_size: int, special_tokens: List[str], *, split_special_tokens: bool = False):
        vocab, merges = train_bpe(input_path, vocab_size, special_tokens, split_special_tokens=split_special_tokens)
        return cls(vocab, merges, special_tokens)

    @classmethod
    def from_files(cls, vocab_filepath: str, merges_filepath: str, special_tokens: List[str] = []) -> "Tokenizer":
        with open(vocab_filepath, "rb") as f:
            vocab = pickle.load(f)
        with open(merges_filepath, "rb") as f:
            merges = pickle.load(f)
        return cls(vocab, merges, special_tokens=special_tokens)

    def save(self, path: str, prefix: str = ""):
        os.makedirs(path, exist_ok=True)         # tokenizer.py:159-167: plain pickles of the two objects
        with open(os.path.join(path, prefix + "-vocab.pkl"), "wb+") as f:
            pickle.dump(self.vocab, f)
        with open(os.path.join(path, prefix + "-merges.pkl"), "wb+") as f:
            pickle.dump(self.merges, f)

    # ---- device tokenizer ------------------------------------------------------------------------
    def _signature(self):
        return (id(self.vocab), len(self.vocab), len(self.vocab_inv), id(self.merges), len(self.merges), tuple(self.special_tokens))

    def _tables(self):
        """Integer-symbol form of (merges, vocab_inv): symbols 0..255 are the single bytes, 256.. every distinct
        byte string a+b of the merge list (the reference identifies tokens by their bytes)."""
        sym_of = {bytes([i]): i for i in range(256)}
        sym_bytes = [bytes([i]) for i in range(256)]
        for a, b in self.merges:
            t = a + b
            if t not in sym_of:
                sym_of[t] = len(sym_bytes)
                sym_bytes.append(t)
        n = len(self.merges)
        last = {pair: j for j, pair in enumerate(self.merges)}      # inv_merges, tokenizer.py:115 (last duplicate wins)
        pairs = np.full((max(n, 1), 2), -1, dtype=np.int32)
        result = np.zeros(max(n, 1), dtype=np.int32)
        for j, (a, b) in enumerate(self.merges):
            sa, sb = sym_of.get(a), sym_of.get(b)
            if sa is None or sb is None or last[(a, b)] != j:
                continue                         # can never be adjacent / superseded by a later duplicate
            pairs[j, 0], pairs[j, 1] = sa, sb
            result[j] = sym_of[a + b]
        inv = self.vocab_inv
        sym_to_id = np.array([inv.get(t, -1) for t in sym_bytes], dtype=np.int64)
        return pairs, result, sym_bytes, sym_to_id

    def _device_tok(self):
        ctx = self._ctx or _lib.default_context()
        with ctx.lock:
            return self._device_tok_locked(ctx)

    def _device_tok_locked(self, ctx):
        sig = self._signature()
        if self._tok is not None and sig == self._sig:
            return self._tok
        self.close()
        L = _lib.lib()
        pairs, result, sym_bytes, sym_to_id = self._tables()
        if sym_to_id.size and (sym_to_id.max() >= 2**31 or sym_to_id.min() < -1):
            raise ValueError("token ids must fit int32")
        sym_to_id32 = sym_to_id.astype(np.int32)
        sym_blob, sym_offs = _lib.pack_blobs64(sym_bytes)
        items = [(k, v) for k, v in self.vocab.items() if isinstance(k, int) and isinstance(v, (bytes, bytearray))]
        v_blob, v_offs = _lib.pack_blobs64([bytes(v) for _, v in items])
        v_ids = np.array([k for k, _ in items] or [0], dtype=np.int64)
        sp_bytes = [s.encode("utf-8") for s in self.special_tokens]
        sp_blob, sp_offs = _lib.pack_blobs(sp_bytes)
        sp_ids = np.array([self.vocab_inv.get(b, -1) for b in sp_bytes] or [0], dtype=np.int64)
        h = C.c_void_p()
        rc = L.bpe_tok_create(ctx.handle, _lib.ptr(pairs), _lib.ptr(result), len(self.merges),
                              _lib.ptr(sym_to_id32), _lib.ptr(sym_blob), _lib.ptr(sym_offs), len(sym_bytes),
                              _lib.ptr(v_blob), _lib.ptr(v_offs), _lib.ptr(v_ids), len(items),
                              _lib.ptr(sp_blob), _lib.ptr(sp_offs), _lib.ptr(sp_ids), len(sp_bytes), C.byref(h))
        ctx.check(rc)
        self._tok, self._sig, self._tok_ctx = h, sig, ctx
        return h

    def close(self):
        if getattr(self, "_tok", None):
            if self._tok_ctx.handle:             # the tokenizer's device memory belongs to its (still open) context
                _lib.lib().bpe_tok_destroy(self._tok)
            self._tok = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _raise(self, ctx, rc: int, data: np.ndarray | None = None):
        L = _lib.lib()
        if rc == _lib.ERR_KEY and self._tok is not None:
            n = C.c_uint64(0)
            L.bpe_tok_key_error(self._tok, None, 0, C.byref(n))
            buf = np.zeros(max(n.value, 1), dtype=np.uint8)
            L.bpe_tok_key_error(self._tok, _lib.ptr(buf), n.value, C.byref(n))
            raise KeyError(buf[: n.value].tobytes())              # tokenizer.py:120,135
        if rc == _lib.ERR_UTF8 and data is not None:
            bytes(data).decode("utf-8")
        ctx.check(rc)

    # ---- encode (tokenizer.py:111-138) -------------------------------------------------------------
    def _encode_ex(self, data, dtype, out=None, *, docs=None, texts=None, drop=(0.0, 0), unit=None):
        """bpe_encode_ex of UTF-8 `data` into `out` (or a new array) of `dtype` (uint16 or int32): (ids, spans or None, id offsets or
        None).  docs: uint64 document offsets into `data` (a batch; `texts` are the items they came from, when known); drop: (p, seed)
        of BPE-dropout; unit: _lib.OFF_* for the int64 spans [n, 2] of the tokens."""
        tok = self._device_tok()
        ctx = self._tok_ctx
        L = _lib.lib()
        arr = _lib.as_u8(data)
        code = {np.dtype(np.uint16): _lib.DTYPE_U16, np.dtype(np.int32): _lib.DTYPE_I32}[np.dtype(dtype)]
        if out is None:
            out = np.empty(max(arr.size, 1), dtype=dtype)         # a token covers at least one byte
        opts = _lib.EncodeOpts(dropout=drop[0], seed=drop[1])
        spans = id_offs = None
        if docs is not None:
            id_offs = np.zeros(docs.size, dtype=np.uint64)
            opts.doc_offs, opts.n_docs, opts.id_offs_out = docs.ctypes.data, docs.size - 1, id_offs.ctypes.data
        if unit is not None:
            spans = np.empty((out.size, 2), dtype=np.int64)
            opts.with_offsets, opts.offset_unit, opts.offs_out = 1, unit, spans.ctypes.data
        n_out = C.c_uint64(0)
        stats = _lib.EncodeStats()
        with ctx.lock:
            rc = L.bpe_encode_ex(tok, _lib.ptr(arr) if arr.size else None, arr.size, C.byref(opts), code, _lib.ptr(out), out.size,
                                 C.byref(n_out), C.byref(stats))
            if rc == _lib.ERR_UTF8 and texts is not None:
                # the device reports invalid UTF-8 in a chunk before a KeyError in it: the documents before the invalid one
                # go first, then that document fails as its decode does
                k = int(np.searchsorted(docs, L.bpe_last_error_detail(ctx.handle), side="right")) - 1
                self._encode_ex(arr[: int(docs[k])], dtype, docs=docs[: k + 1], drop=drop)
                item = texts[k]
                if isinstance(item, (bytes, bytearray, memoryview)):
                    bytes(item).decode("utf-8")
            if rc != _lib.BPE_OK:
                self._raise(ctx, rc, arr if docs is None else None)
        self.last_stats = stats.as_dict()
        n = n_out.value
        return out[:n], None if spans is None else spans[:n], None if id_offs is None else id_offs.astype(np.int64)

    def encode_to_numpy(self, data, dtype=np.int32, *, dropout: float = 0.0, seed: int = 0) -> np.ndarray:
        """Token ids of UTF-8 `data` (bytes / uint8 array) as a numpy array of `dtype` (uint16 or int32).  dropout > 0: BPE-dropout
        (every pretoken occurrence merged with each candidate pair of each round dropped with that probability; a pure function of
        the text, dropout and seed -- see bpe_encode_opts in include/bpe_sm100.h)."""
        return self._encode_ex(data, dtype, drop=_check_dropout(dropout, seed))[0]

    def encode_offsets_to_numpy(self, data, dtype=np.int32, *, unit: str = "byte", dropout: float = 0.0,
                                seed: int = 0) -> Tuple[np.ndarray, np.ndarray]:
        """encode_to_numpy's ids and int64 spans [n, 2] of `data` in `unit` ("byte" or "char"), computed on the device in the same pass:
        token i came from data[start:end] ("byte"), or text[start:end] holds its bytes ("char"; a character that several tokens split
        belongs to each of them).  See bpe_encode_opts in include/bpe_sm100.h."""
        code_unit = _check_unit(unit)
        ids, spans, _ = self._encode_ex(data, dtype, drop=_check_dropout(dropout, seed), unit=code_unit)
        return ids, spans

    def encode_with_offsets(self, text: str, *, dropout: float = 0.0, seed: int = 0) -> Tuple[List[int], List[Tuple[int, int]]]:
        """encode(text)'s ids and the character span (start, end) of every token in `text` (encode_offsets_to_numpy, unit="char")."""
        ids, spans = self.encode_offsets_to_numpy(text.encode("utf-8"), np.int32, unit="char", dropout=dropout, seed=seed)
        return ids.tolist(), list(map(tuple, spans.tolist()))

    def encode_into(self, data, out: np.ndarray) -> int:
        """encode_to_numpy into a caller-owned array (uint16 or int32; page-locked for PCIe-speed downloads).  Returns the count."""
        n = self._encode_ex(data, out.dtype, out)[0].size
        self.last_saw_cr = bool(_lib.lib().bpe_tok_saw_cr(self._tok))
        return n

    def encode(self, text: str, *, dropout: float = 0.0, seed: int = 0) -> List[int]:
        """Token ids of `text`; dropout > 0 samples a BPE-dropout segmentation (see encode_to_numpy)."""
        dropout, seed = _check_dropout(dropout, seed)
        return self.encode_to_numpy(text.encode("utf-8"), np.int32, dropout=dropout, seed=seed).tolist()

    def encode_batch(self, texts: Sequence[str], *, dropout: float = 0.0, seed: int = 0) -> List[List[int]]:
        """[self.encode(t) for t in texts] -- the same ids, split the same way, the same first exception -- with one device pass
        over all documents (bpe_encode_ex with document offsets) instead of one pipeline per document.  With dropout > 0, document j
        is sampled as document j of the batch: encode(d, dropout=p, seed=s) == encode_batch([d], dropout=p, seed=s)[0]."""
        ids, offs = self.encode_batch_to_numpy(texts, np.int32, dropout=dropout, seed=seed)
        flat, o = ids.tolist(), offs.tolist()
        return [flat[o[j]: o[j + 1]] for j in range(len(o) - 1)]

    def encode_batch_to_numpy(self, texts: Sequence[str | bytes], dtype=np.int32, *, dropout: float = 0.0,
                              seed: int = 0) -> Tuple[np.ndarray, np.ndarray]:
        """Ids of every document back to back (uint16 or int32) and int64 offsets (len(texts) + 1): document j's ids are
        ids[offsets[j]:offsets[j + 1]].  A `bytes` item must be UTF-8; it fails as item.decode("utf-8") would.  Where several
        documents would fail, the error is that of the first one in list order, as in a loop over encode_to_numpy.  dropout > 0:
        BPE-dropout with the document's index in `texts` as its `doc`."""
        ids, _, offs = self._encode_batch(texts, dtype, _check_dropout(dropout, seed))
        return ids, offs

    def encode_batch_offsets_to_numpy(self, texts: Sequence[str | bytes], dtype=np.int32, *, unit: str = "byte", dropout: float = 0.0,
                                      seed: int = 0) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """encode_batch_to_numpy's ids and document offsets with the int64 span [n, 2] of every token in `unit` ("byte" / "char"),
        relative to its document's start: (ids, spans, offsets), and document j's tokens are [offsets[j], offsets[j + 1]).  Document j's
        spans are those of encode_offsets_to_numpy(texts[j]); the errors are those of encode_batch_to_numpy."""
        code_unit = _check_unit(unit)
        return self._encode_batch(texts, dtype, _check_dropout(dropout, seed), code_unit)

    def encode_batch_with_offsets(self, texts: Sequence[str], *, dropout: float = 0.0,
                                  seed: int = 0) -> List[Tuple[List[int], List[Tuple[int, int]]]]:
        """[self.encode_with_offsets(t) for t in texts] in one device pass (encode_batch_offsets_to_numpy, unit="char")."""
        ids, spans, o = self.encode_batch_offsets_to_numpy(texts, np.int32, unit="char", dropout=dropout, seed=seed)
        flat, sp, o = ids.tolist(), list(map(tuple, spans.tolist())), o.tolist()
        return [(flat[o[j]: o[j + 1]], sp[o[j]: o[j + 1]]) for j in range(len(o) - 1)]

    def _encode_batch(self, texts, dtype, drop, unit=None):
        """(ids, spans or None, id offsets) of the documents `texts`, with the errors of encode_batch_to_numpy."""
        texts = list(texts)
        blob, offs, bad = _pack_documents(texts)
        if bad is not None:                      # a str that cannot be encoded: the documents before it fail first, if any does
            self._encode_ex(blob, dtype, docs=offs, drop=drop)
            raise bad
        return self._encode_ex(blob, dtype, docs=offs, texts=texts, drop=drop, unit=unit)

    def encode_sharded(self, data, dtype=np.uint16, group=None):
        """Multi-GPU encode (one process per GPU, torch.distributed initialised): every rank passes the same UTF-8 `data`
        and gets (ids of its shard, global index of its first id, total ids); shards are cut at exact boundaries, so the
        ranks' arrays in rank order concatenate to encode(data).  See sharded_encode.py."""
        from .sharded_encode import encode_sharded
        return encode_sharded(self, data, dtype, group)

    def encode_iterable(self, iterable: Iterable[str]) -> Iterator[int]:
        # Chunk rule of tokenizer.py:140-153: concatenate items until the buffer holds >= 2 Mi CHARACTERS,
        # encode the buffer on its own, repeat until the iterable yields nothing (SURVEY A-13/A-14).
        #
        # Double-buffered (SURVEY 8f row 3): once the first id of chunk k has been handed out, chunk k + 1 is read from
        # the iterable (in the caller's thread: the iterable is never touched from another one) and its encode runs on a
        # worker thread -- ctypes releases the GIL for the C call -- while the caller consumes the ids of chunk k.  The
        # ids, their order and the chunk boundaries are those of the sequential loop; the only observable difference is
        # that the iterable is read one chunk ahead of the ids being consumed (never before the first id is out).
        def read_chunk():
            parts, chars = [], 0
            for line in iterable:
                parts.append(line)
                chars += len(line)
                if chars >= _CHUNK_CHARS:
                    break
            return "".join(parts) if chars else None

        def encode_list(text):
            return self.encode_to_numpy(text.encode("utf-8"), np.int32).tolist()

        text = read_chunk()
        if text is None:
            return
        ids = encode_list(text)
        pool = None
        try:
            while True:
                it = iter(ids)
                for first in it:
                    yield first
                    break
                nxt = read_chunk()
                fut = None
                if nxt is not None:
                    if pool is None:
                        from concurrent.futures import ThreadPoolExecutor
                        pool = ThreadPoolExecutor(max_workers=1, thread_name_prefix="bpe-encode-ahead")
                    fut = pool.submit(encode_list, nxt)
                yield from it
                if fut is None:
                    break
                ids = fut.result()                # re-raises KeyError / UnicodeDecodeError of that chunk here, in order
        finally:
            if pool is not None:
                pool.shutdown(wait=True)

    # ---- decode (tokenizer.py:155-157) -------------------------------------------------------------
    def decode_bytes(self, ids) -> bytes:
        tok = self._device_tok()
        ctx = self._tok_ctx
        L = _lib.lib()
        try:
            arr = np.ascontiguousarray(np.asarray(ids, dtype=np.int64).reshape(-1))
        except (OverflowError, TypeError, ValueError):
            raise KeyError(next(i for i in ids if i not in self.vocab))
        if arr.size == 0:
            return b""
        n_out = C.c_uint64(0)
        with ctx.lock:
            rc = L.bpe_decode(tok, _lib.ptr(arr), arr.size, None, 0, C.byref(n_out))
            if rc == _lib.ERR_KEY:
                raise KeyError(int(arr[L.bpe_last_error_detail(ctx.handle)]))
            ctx.check(rc)
            out = np.empty(max(n_out.value, 1), dtype=np.uint8)
            rc = L.bpe_decode(tok, _lib.ptr(arr), arr.size, _lib.ptr(out), out.size, C.byref(n_out))
            ctx.check(rc)
        return out[: n_out.value].tobytes()

    def decode(self, ids: List[int]) -> str:
        return self.decode_bytes(ids).decode("utf-8", errors="replace")

    def decode_batch(self, sequences) -> List[str]:
        """[self.decode(s) for s in sequences] with one device decode of the concatenation (bpe_decode_batch): what a
        sampler that generates many sequences needs (models/transformer/decode.py:51 decodes one at a time)."""
        seqs = [np.asarray(s, dtype=np.int64).reshape(-1) for s in sequences]
        if not seqs:
            return []
        tok = self._device_tok()
        ctx = self._tok_ctx
        L = _lib.lib()
        seq_offs = np.zeros(len(seqs) + 1, dtype=np.uint64)
        np.cumsum([s.size for s in seqs], out=seq_offs[1:])
        ids = np.ascontiguousarray(np.concatenate(seqs)) if int(seq_offs[-1]) else np.zeros(0, dtype=np.int64)
        byte_offs = np.zeros(len(seqs) + 1, dtype=np.uint64)
        n_out = C.c_uint64(0)
        with ctx.lock:
            args = (tok, _lib.ptr(ids) if ids.size else None, ids.size, _lib.ptr(seq_offs), len(seqs))
            rc = L.bpe_decode_batch(*args, None, 0, C.byref(n_out), _lib.ptr(byte_offs))
            if rc == _lib.ERR_KEY:
                raise KeyError(int(ids[L.bpe_last_error_detail(ctx.handle)]))
            ctx.check(rc)
            out = np.empty(max(n_out.value, 1), dtype=np.uint8)
            if n_out.value:
                ctx.check(L.bpe_decode_batch(*args, _lib.ptr(out), out.size, C.byref(n_out), _lib.ptr(byte_offs)))
        blob = out[: n_out.value].tobytes()
        bo = byte_offs.astype(np.int64)
        return [blob[bo[j]: bo[j + 1]].decode("utf-8", errors="replace") for j in range(len(seqs))]

    # ---- the reference's public helper methods (tokenizer.py:63-109), kept for callers that use them ----
    def segment(self, text: str) -> List[str]:
        """re.split on the specials with a capturing group: [text, special, text, ...] (tokenizer.py:63-66)."""
        if not self.special_tokens:
            return [text]
        from .pretok import pretoken_starts
        data = text.encode("utf-8")
        sp = set(s.encode("utf-8") for s in self.special_tokens)
        st = pretoken_starts(data, self.special_tokens, ctx=self._ctx).tolist() + [len(data)]
        out, cur = [], b""
        for i in range(len(st) - 1):
            piece = data[st[i]:st[i + 1]]
            if piece in sp:
                out.extend([cur.decode("utf-8"), piece.decode("utf-8")])
                cur = b""
            else:
                cur += piece
        out.append(cur.decode("utf-8"))
        return out

    def match(self, text: str) -> List[str]:
        from .pretok import pretokens
        return [m for m in pretokens(text, None, ctx=self._ctx) if m not in self.special_tokens]   # tokenizer.py:68-77

    def pretokenize(self, segments: List[str]) -> List[str]:
        matches = []
        for segment in segments:                 # tokenizer.py:79-90
            if segment == "":
                continue
            if segment in self.special_tokens:
                matches.append(segment)
            else:
                matches.extend(self.match(segment))
        return matches

    def merge(self, tokens: List[bytes], pair: Tuple[bytes, bytes], replacement: bytes) -> List[bytes]:
        # tokenizer.py:92-109: left to right, non-overlapping (host helper only; encode does this on the device)
        a, b = pair
        out: List[bytes] = []
        skip = False
        for k, tok in enumerate(tokens):
            if skip:
                skip = False
            elif tok == a and k + 1 < len(tokens) and tokens[k + 1] == b:
                out.append(replacement)
                skip = True
            else:
                out.append(tok)
        return out
