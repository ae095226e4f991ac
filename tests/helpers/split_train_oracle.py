"""CPU oracle of training with split_special_tokens (tests/helpers/split_train_oracle.c on top of oracle/bpe_oracle.c).
TEST INFRASTRUCTURE ONLY.

count_words(data, specials): the words the split mode counts in the raw bytes `data` (validated, newline-translated, split on
the specials, each piece counted whole).  train_bpe_on_bytes / train_bpe: oracle.train_bpe with split_special_tokens=True.
The library is compiled on first use into the temporary directory (the repository tree may be read-only), named by a hash of
its sources."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import pathlib
import subprocess
import tempfile

import numpy as np

from oracle import oracle

_HERE = pathlib.Path(__file__).resolve().parent
_ROOT = _HERE.parent.parent
_SOURCES = [_HERE / "split_train_oracle.c", _ROOT / "oracle" / "bpe_oracle.c", _ROOT / "transformer-lm_b200" / "csrc" / "unicode_tables.h"]
_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256(b"".join(p.read_bytes() for p in _SOURCES)).hexdigest()[:16]
        so = pathlib.Path(tempfile.gettempdir()) / ("bpe_split_train_oracle_%d_%s.so" % (os.getuid(), h))
        if not so.exists():
            tmp = so.with_suffix(".%d.tmp" % os.getpid())
            subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-fvisibility=hidden", "-std=gnu11", "-shared",
                                   "-o", str(tmp), str(_SOURCES[0])])
            os.replace(tmp, so)
        L = C.CDLL(str(so))
        vp = C.c_void_p
        L.orc_split_count.restype = C.c_int64
        L.orc_split_count.argtypes = [vp, C.c_uint64, vp, vp, C.c_int, vp, vp, vp, C.POINTER(C.c_uint64)]
        L.orc_split_train_bpe.restype = C.c_int
        L.orc_split_train_bpe.argtypes = [vp, C.c_uint64, vp, vp, C.c_int, C.c_int, vp, C.POINTER(C.c_int), C.POINTER(C.c_int64)]
        _lib = L
    return _lib


def _specials(special_tokens):
    """Tokenizer.segment's order: longest first (a special never matches where a longer one that extends it does)."""
    sp = sorted((s.encode("utf-8") for s in special_tokens), key=len, reverse=True)
    return oracle._pack_specials(sp) + (len(sp),)


def count_words(data: bytes, special_tokens: list[str]) -> dict[bytes, int]:
    a = oracle._buf(data)
    sb, so, ns = _specials(special_tokens)
    nb = C.c_uint64(0)
    n = lib().orc_split_count(oracle._ptr(a), len(data), oracle._ptr(sb), oracle._ptr(so), ns, None, None, None, C.byref(nb))
    if n < 0:
        raise ValueError("invalid utf-8")
    blob = np.zeros(max(nb.value, 1), dtype=np.uint8)
    offs = np.zeros(n + 1, dtype=np.uint64)
    cnts = np.zeros(max(n, 1), dtype=np.int64)
    lib().orc_split_count(oracle._ptr(a), len(data), oracle._ptr(sb), oracle._ptr(so), ns, oracle._ptr(blob), oracle._ptr(offs),
                          oracle._ptr(cnts), C.byref(nb))
    raw = blob.tobytes()
    return {raw[int(offs[i]):int(offs[i + 1])]: int(cnts[i]) for i in range(n)}


def train_bpe_on_bytes(data: bytes, vocab_size: int, special_tokens: list[str] = []):
    vocab = oracle._ref_vocab(list(special_tokens))
    n_merges = max(vocab_size - len(vocab), 0)
    a = oracle._buf(data)
    sb, so, ns = _specials(special_tokens)
    pairs = np.zeros((max(n_merges, 1), 2), dtype=np.int32)
    n_done = C.c_int(0)
    err = C.c_int64(-1)
    rc = lib().orc_split_train_bpe(oracle._ptr(a), len(data), oracle._ptr(sb), oracle._ptr(so), ns, n_merges, oracle._ptr(pairs),
                                   C.byref(n_done), C.byref(err))
    if rc == -1:
        data.decode("utf-8")                               # raises the UnicodeDecodeError of the default mode
        raise AssertionError("oracle flagged invalid UTF-8 at %d but CPython accepted it" % err.value)
    sym = [bytes([i]) for i in range(256)]
    merges = []
    seen = set(vocab.values())
    for k in range(n_done.value):
        x, y = sym[pairs[k, 0]], sym[pairs[k, 1]]
        merges.append((x, y))
        sym.append(x + y)
        if x + y not in seen:                              # Vocab.add_token dedupe (vocab.py:28-34)
            seen.add(x + y)
            vocab[len(vocab)] = x + y
    return vocab, merges


def train_bpe(input_path, vocab_size: int, special_tokens: list[str] = []):
    with open(input_path, "rb") as f:
        return train_bpe_on_bytes(f.read(), vocab_size, special_tokens)
