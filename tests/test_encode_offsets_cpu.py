"""Token-offsets spec (include/bpe_sm100.h, bpe_encode_opts) on the CPU: the Python reference (tests/helpers/offsets_ref.py) against
the spec's invariants on fuzzed text, hand-worked cases (split characters, special tokens missing from the vocabulary or sharing an id with
an ordinary token, SURVEY A-12), and the argument checks of the Tokenizer methods and the C ABI."""
import ctypes as C
import random

import numpy as np
import pytest

import _bootstrap  # noqa: F401
from oracle import oracle
from tests.common import load_gpt2_fixture
from tests.helpers.offsets_ref import chars_from_bytes, reference_offsets
from transformer_lm_b200 import _lib
from transformer_lm_b200.tokenizer import Tokenizer

EOT = "<|endoftext|>"
ALPHA = ["a", "b", "t", "e", "s", " ", " ", "  ", "\n", "'s", "é", "中", "\U0001F643", "1", "00", ".", "the", " the", "ing", "tion",
         "aaaa", EOT, "<|", " tokenization", "é" * 9, "\U0001F468‍\U0001F469", "ß", "Zürich"]


@pytest.fixture(scope="module", params=[[EOT], []], ids=["eot", "plain"])
def gpt2(request):
    vocab, merges = load_gpt2_fixture()
    return oracle.OracleTokenizer(dict(vocab), list(merges), request.param)


def _fuzz_texts(seed):
    rnd = random.Random(seed)
    out = ["".join(rnd.choice(ALPHA) for _ in range(rnd.randint(0, 60))) for _ in range(40)]
    out.append(EOT + EOT + "x" + EOT)
    out.append("\U0001F643" * 20 + " " + "中文字符" * 10 + EOT + " résumé")
    return out


def _check_invariants(otok, text):
    data = text.encode()
    ids, spans = reference_offsets(otok, data, "byte")
    assert ids.tolist() == otok.encode_bytes(data).tolist()
    if len(ids):                                 # the spans tile the text in order
        assert spans[0, 0] == 0 and spans[-1, 1] == len(data)
        assert np.array_equal(spans[1:, 0], spans[:-1, 1]) and (spans[:, 1] > spans[:, 0]).all()
    else:
        assert data == b""
    sp = {s.encode() for s in otok.special_tokens}
    for t, (s, e) in zip(ids.tolist(), spans.tolist()):
        assert data[s:e] in sp or data[s:e] == otok.vocab[t]
    # the ids of the whole text split by vocabulary lengths give the same spans
    assert np.array_equal(reference_offsets(otok, data, "byte", ids=ids)[1], spans)
    chars = reference_offsets(otok, data, "char")[1]
    assert np.array_equal(chars, chars_from_bytes(data, spans))
    for (s, e), (cs, ce) in zip(spans.tolist(), chars.tolist()):
        got = text[cs:ce].encode()
        assert data[s:e] in got
        split = (s < len(data) and (data[s] & 0xC0) == 0x80) or (e < len(data) and (data[e] & 0xC0) == 0x80)
        assert split or got == data[s:e]


def test_reference_invariants_on_fuzzed_text(gpt2):
    for text in _fuzz_texts(5):
        _check_invariants(gpt2, text)


def _bytes_vocab(extra=()):
    vocab = {i: bytes([i]) for i in range(256)}
    vocab.update(extra)
    return vocab


def test_emoji_split_into_byte_tokens():
    otok = oracle.OracleTokenizer(_bytes_vocab(), [], [])
    text = "a\U0001F643b"                          # "a", the emoji (4 bytes, no merges: 4 tokens), "b"
    ids, b = reference_offsets(otok, text.encode(), "byte")
    assert ids.tolist() == [97, 0xF0, 0x9F, 0x99, 0x83, 98]
    assert b.tolist() == [[0, 1], [1, 2], [2, 3], [3, 4], [4, 5], [5, 6]]
    assert reference_offsets(otok, text.encode(), "char")[1].tolist() == [[0, 1], [1, 2], [1, 2], [1, 2], [1, 2], [2, 3]]


def test_two_byte_character_split_across_tokens():
    otok = oracle.OracleTokenizer(_bytes_vocab({256: b"x\xc3"}), [(b"x", b"\xc3")], [])
    text = "xé"                                  # one pretoken, bytes 78 C3 A9: "x" + the lead byte, then the continuation byte
    ids, b = reference_offsets(otok, text.encode(), "byte")
    assert ids.tolist() == [256, 0xA9] and b.tolist() == [[0, 2], [2, 3]]
    assert reference_offsets(otok, text.encode(), "char")[1].tolist() == [[0, 2], [1, 2]]    # both hold "é": they overlap by one


def test_special_missing_from_vocab():
    otok = oracle.OracleTokenizer(_bytes_vocab(), [], ["<s>"])
    assert otok.vocab_inv[b"<s>"] == 256 and 256 not in otok.vocab      # A-12: id len(vocab), no vocabulary bytes
    for unit in ("byte", "char"):
        ids, sp = reference_offsets(otok, "a<s>é".encode(), unit)
        assert ids.tolist() == [97, 256, 0xC3, 0xA9]
        assert sp.tolist() == ([[0, 1], [1, 4], [4, 5], [5, 6]] if unit == "byte" else [[0, 1], [1, 4], [4, 5], [4, 5]])


def test_special_id_shared_with_an_ordinary_token():
    otok = oracle.OracleTokenizer(_bytes_vocab({257: b"ab"}), [(b"a", b"b")], ["<s>"])
    assert otok.vocab_inv[b"<s>"] == 257 == otok.vocab_inv[b"ab"]    # A-12: len(vocab) - 1 after the insert collides with "ab"
    ids, sp = reference_offsets(otok, b"ab<s>abc", "byte")
    assert ids.tolist() == [257, 257, 257, 99]
    assert sp.tolist() == [[0, 2], [2, 5], [5, 7], [7, 8]]


BAD_UNITS = ["bytes", "chars", "", None, 1]


@pytest.mark.parametrize("unit", BAD_UNITS)
def test_tokenizer_rejects_unknown_unit(unit):
    vocab, merges = load_gpt2_fixture()
    tok = Tokenizer(vocab, merges, [EOT])          # (the checks come before any device work)
    with pytest.raises(ValueError):
        tok.encode_offsets_to_numpy(b"abc", np.int32, unit=unit)
    with pytest.raises(ValueError):
        tok.encode_batch_offsets_to_numpy(["abc"], np.int32, unit=unit)


@pytest.mark.parametrize("kw", [dict(dropout=-0.01), dict(dropout=1.01), dict(dropout=float("nan")), dict(dropout=0.1, seed=-1),
                                dict(dropout=0.1, seed=2**64), dict(dropout=0.1, seed=True)])
def test_tokenizer_rejects_bad_dropout(kw):
    vocab, merges = load_gpt2_fixture()
    tok = Tokenizer(vocab, merges, [EOT])
    for call in (lambda: tok.encode_with_offsets("abc", **kw), lambda: tok.encode_offsets_to_numpy(b"abc", np.int32, **kw),
                 lambda: tok.encode_batch_with_offsets(["abc"], **kw), lambda: tok.encode_batch_offsets_to_numpy(["abc"], np.int32, **kw)):
        with pytest.raises(ValueError):
            call()


def test_encode_ex_offsets_reject_null_tokenizer():
    L = _lib.lib()
    n = C.c_uint64(0)
    buf = np.zeros(4, dtype=np.int64)
    docs = np.zeros(1, dtype=np.uint64)                                   # an empty batch
    batch = dict(doc_offs=docs.ctypes.data, n_docs=0, id_offs_out=buf.ctypes.data)
    for opts in (_lib.EncodeOpts(with_offsets=1, offset_unit=_lib.OFF_BYTES),
                 _lib.EncodeOpts(with_offsets=1, offset_unit=_lib.OFF_CHARS, **batch),
                 _lib.EncodeOpts(dropout=0.5, seed=1, with_offsets=1, offset_unit=_lib.OFF_BYTES),
                 _lib.EncodeOpts(dropout=0.5, seed=1, with_offsets=1, offset_unit=_lib.OFF_BYTES, **batch)):
        assert L.bpe_encode_ex(None, None, 0, C.byref(opts), _lib.DTYPE_I32, None, 0, C.byref(n), None) == _lib.ERR_ARG
