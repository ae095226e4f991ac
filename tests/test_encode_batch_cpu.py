"""Host logic of Tokenizer.encode_batch / encode_batch_to_numpy without a device: packing the documents into one buffer with byte
offsets, the order of exceptions (the first failing document in list order), splitting the ids by the offsets, argument checks
of bpe_encode_ex with document offsets."""
import ctypes as C

import numpy as np
import pytest

import _bootstrap  # noqa: F401
from transformer_lm_b200 import _lib
from transformer_lm_b200.tokenizer import Tokenizer, _pack_documents


def _unpack(blob, offs):
    b = blob.tobytes()
    return [b[int(offs[j]): int(offs[j + 1])] for j in range(len(offs) - 1)]


@pytest.mark.parametrize("docs", [[], [""], ["a", "", "bc "], ["ab", "", ""], ["", "x"]])
def test_pack_ascii(docs):
    blob, offs, bad = _pack_documents(docs)
    assert bad is None and offs.dtype == np.uint64 and blob.dtype == np.uint8
    assert offs[0] == 0 and len(offs) == len(docs) + 1
    assert _unpack(blob, offs) == [d.encode() for d in docs]


def test_pack_non_ascii_and_bytes():
    docs = ["café", "", "中文\n", "\U0001F643", "plain"]
    blob, offs, bad = _pack_documents(docs)
    assert bad is None and _unpack(blob, offs) == [d.encode("utf-8") for d in docs]
    assert offs.tolist() == [0, 5, 5, 12, 16, 21]
    mixed = [b"ab\xff", "é", bytearray(b"xy"), b""]
    blob, offs, bad = _pack_documents(mixed)
    assert bad is None and _unpack(blob, offs) == [b"ab\xff", "é".encode(), b"xy", b""]


def test_pack_stops_at_a_lone_surrogate():
    blob, offs, bad = _pack_documents(["ok", "é", "bad \ud800", "later"])
    assert isinstance(bad, UnicodeEncodeError)
    assert _unpack(blob, offs) == [b"ok", "é".encode()]


class _FakeDevice:
    """_encode_ex stand-in for a batch: ids = the bytes of each document; a document holding b"K" is a KeyError."""

    def __call__(self, blob, dtype, *, docs, texts=None, drop=(0.0, 0), unit=None):
        parts = _unpack(blob, docs)
        for d in parts:
            if b"K" in d:
                raise KeyError(b"K")
        ids = np.frombuffer(b"".join(parts), dtype=np.uint8).astype(dtype)
        return ids, None, docs.astype(np.int64)


@pytest.fixture
def fake_tok(monkeypatch):
    tok = Tokenizer({i: bytes([i]) for i in range(256)}, [], [])
    monkeypatch.setattr(tok, "_encode_ex", _FakeDevice())
    return tok


def test_first_failing_document_in_list_order_raises(fake_tok):
    with pytest.raises(KeyError):
        fake_tok.encode_batch(["a", "K", "b \ud800"])             # the KeyError comes first in list order
    with pytest.raises(UnicodeEncodeError):
        fake_tok.encode_batch(["a", "b \ud800", "K"])
    with pytest.raises(UnicodeEncodeError):
        fake_tok.encode_batch(["\ud800"])


def test_ids_split_by_document_offsets(fake_tok):
    docs = ["ab", "", "cde", "", "f"]
    assert fake_tok.encode_batch(docs) == [list(d.encode()) for d in docs]
    assert fake_tok.encode_batch([]) == []
    ids, offs = fake_tok.encode_batch_to_numpy(["é", "x"], np.int32)
    assert offs.tolist() == [0, 2, 3] and ids.tolist() == list("é".encode()) + [120]
    assert fake_tok.encode_batch(iter(["a", "b"])) == [[97], [98]]          # any iterable of documents


def test_encode_ex_batch_rejects_null_tokenizer():
    L = _lib.lib()
    n_out = C.c_uint64(0)
    ids = np.zeros(2, dtype=np.uint64)
    offs = np.array([0, 3], dtype=np.uint64)
    blob = np.frombuffer(b"abc", dtype=np.uint8)
    opts = _lib.EncodeOpts(doc_offs=offs.ctypes.data, n_docs=1, id_offs_out=ids.ctypes.data)
    assert L.bpe_encode_ex(None, _lib.ptr(blob), 3, C.byref(opts), _lib.DTYPE_I32, None, 0, C.byref(n_out), None) == _lib.ERR_ARG
