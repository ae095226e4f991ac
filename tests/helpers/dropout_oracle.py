"""CPU oracle of BPE-dropout (tests/helpers/dropout_oracle.c on top of oracle/bpe_oracle.c).  TEST INFRASTRUCTURE ONLY.

DropoutOracle is oracle.OracleTokenizer with encode_bytes(data, *, dropout=, seed=, doc=): the spec of bpe_encode_dropout
(include/bpe_sm100.h) for `data` as document `doc` of a batch; dropout = 0 is the oracle's plain encode.  The library is compiled
on first use into the temporary directory (the repository tree may be read-only), named by a hash of its sources."""
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
_SOURCES = [_HERE / "dropout_oracle.c", _ROOT / "oracle" / "bpe_oracle.c", _ROOT / "transformer-lm_b200" / "csrc" / "unicode_tables.h"]
_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256(b"".join(p.read_bytes() for p in _SOURCES)).hexdigest()[:16]
        so = pathlib.Path(tempfile.gettempdir()) / ("bpe_dropout_oracle_%d_%s.so" % (os.getuid(), h))
        if not so.exists():
            tmp = so.with_suffix(".%d.tmp" % os.getpid())
            subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-fvisibility=hidden", "-std=gnu11", "-shared",
                                   "-o", str(tmp), str(_SOURCES[0])])
            os.replace(tmp, so)
        L = C.CDLL(str(so))
        u64p, u32p = C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)
        L.orc_tok_create.restype = C.c_void_p
        L.orc_tok_create.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64,
                                     C.c_void_p, C.c_void_p, C.c_int]
        L.orc_tok_destroy.restype = None
        L.orc_tok_destroy.argtypes = [C.c_void_p]
        L.orc_encode_dropout.restype = C.c_int
        L.orc_encode_dropout.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_uint64, C.c_uint64, C.c_void_p,
                                         C.c_uint64, u64p, u64p, u32p]
        L.orc_dropout_u.restype = C.c_uint64
        L.orc_dropout_u.argtypes = [C.c_uint64] * 4
        _lib = L
    return _lib


def dropout_u(seed: int, doc: int, off: int, t: int) -> int:
    """u(seed, doc, off, t) of the BPE-dropout spec."""
    return lib().orc_dropout_u(seed, doc, off, t)


class DropoutOracle(oracle.OracleTokenizer):
    def _build(self):
        super()._build()
        vb, voffs, vids, mb, moffs, sb, so = self._keep       # the same tables, in this library's own tokenizer object
        self._hd = lib().orc_tok_create(oracle._ptr(vb), oracle._ptr(voffs), oracle._ptr(vids), len(voffs) - 1,
                                        oracle._ptr(mb), oracle._ptr(moffs), (len(moffs) - 1) // 2,
                                        oracle._ptr(sb), oracle._ptr(so), len(self.special_tokens))

    def __del__(self):
        if getattr(self, "_hd", None):
            lib().orc_tok_destroy(self._hd)
            self._hd = None
        super().__del__()

    def encode_bytes(self, data: bytes, *, dropout: float = 0.0, seed: int = 0, doc: int = 0) -> np.ndarray:
        if not dropout:
            return super().encode_bytes(data)
        a = oracle._buf(data)
        n_out, koff, klen = C.c_uint64(0), C.c_uint64(0), C.c_uint32(0)

        def run(ids, cap):
            return lib().orc_encode_dropout(self._hd, oracle._ptr(a), len(data), dropout, seed, doc, ids, cap, C.byref(n_out),
                                            C.byref(koff), C.byref(klen))
        rc = run(None, 0)
        if rc == -3:
            raise ValueError("dropout must be in [0, 1]")
        if rc == -2:
            raise KeyError(data[koff.value:koff.value + klen.value])
        if rc == -1:
            raise ValueError("invalid utf-8")
        out = np.zeros(max(n_out.value, 1), dtype=np.int64)
        run(oracle._ptr(out), n_out.value)
        return out[:n_out.value]
