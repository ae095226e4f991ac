"""GPU token offsets (bpe_encode_ex with offsets, alone or with documents and dropout, through Tokenizer.encode_offsets_to_numpy and
encode_batch_offsets_to_numpy): exact equality of ids and spans, in bytes and in characters, with the Python reference of the spec
(tests/helpers/offsets_ref.py) over the CPU oracles' ids; the ids equal those of the ids-only calls; batch spans equal the per-document
ones; independence from pipeline chunks and the pretoken cache; the same errors as the ids-only calls.

Spans above 2^32 are not run (a text of more than 4 GB and 16 bytes of spans per token).  Nothing on that path is 32-bit: arena
offsets, the chunk's place in the text and the character count carried from chunk to chunk are 64-bit on the device, and the chunked
run below (hundreds of 1 MB chunks) checks that the chunk base and the carried character count are added in."""
import ctypes as C
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

import _bootstrap  # noqa: F401
from oracle import oracle
from tests.helpers.offsets_ref import reference_offsets
from tests.test_gpu_encode_dropout import EOT, ROOT, _doc_lists, _pair, _texts
from tests.adapters import get_tokenizer
from tests.common import load_gpt2_fixture
from transformer_lm_b200 import _lib
from transformer_lm_b200.synth import synth_host

pytestmark = pytest.mark.gpu
UNITS = ["byte", "char"]
ALPHA = ["a", " the", "é", "中", "\U0001F643", "\U0001F468‍\U0001F469", "ß", " Zürich", "  ", "\n", EOT, "'s", "1", "00", "."]


@pytest.fixture(scope="module", params=["gpt2", "gpt2_plain", "corpus1000"])
def toks(request):
    return _pair(request.param)


@pytest.fixture(scope="module")
def gpt2():
    return _pair("gpt2")


def _wide_text(n, seed=1):
    rnd = np.random.default_rng(seed)
    return "".join(ALPHA[k] for k in rnd.integers(0, len(ALPHA), n)).encode()


def _all_texts():
    out = _texts()
    out["wide"] = _wide_text(200_000)            # 2-, 3- and 4-byte characters, split emoji, specials back to back
    return out


def _check(tok, otok, data, unit, dtypes=(np.int32,), **kw):
    drop = kw.get("dropout", 0.0)
    want_ids = otok.encode_bytes(data, dropout=drop, seed=kw.get("seed", 0)) if drop else otok.encode_bytes(data)
    want = reference_offsets(otok, data, unit, ids=want_ids)[1]
    for dtype in dtypes:
        ids, spans = tok.encode_offsets_to_numpy(data, dtype, unit=unit, **kw)
        assert np.array_equal(ids.astype(np.int64), want_ids) and np.array_equal(spans, want), dtype
    return ids


@pytest.mark.parametrize("unit", UNITS)
def test_offsets_match_reference(toks, unit):
    tok, otok = toks
    dtypes = (np.int32, np.uint16) if max(otok.vocab_inv.values()) < 65536 else (np.int32,)
    for name, data in _all_texts().items():
        ids = _check(tok, otok, data, unit, dtypes)
        assert np.array_equal(ids.astype(np.int64), tok.encode_to_numpy(data, np.int32)), name


@pytest.mark.parametrize("p", [0.1, 0.5, 1.0])
def test_dropout_offsets_match_reference(gpt2, p):
    tok, otok = gpt2
    for name, data in _all_texts().items():
        for unit in UNITS:
            ids = _check(tok, otok, data, unit, dropout=p, seed=3)
            assert np.array_equal(ids, tok.encode_to_numpy(data, np.int32, dropout=p, seed=3)), name


def test_hand_worked_cases():
    vocab = {i: bytes([i]) for i in range(256)}
    cases = [(dict(vocab), [], [], "a\U0001F643b", [[0, 1], [1, 2], [1, 2], [1, 2], [1, 2], [2, 3]]),
             ({**vocab, 256: b"x\xc3"}, [(b"x", b"\xc3")], [], "xé", [[0, 2], [1, 2]]),
             (dict(vocab), [], ["<s>"], "a<s>é", [[0, 1], [1, 4], [4, 5], [4, 5]]),
             ({**vocab, 257: b"ab"}, [(b"a", b"b")], ["<s>"], "ab<s>abc", [[0, 2], [2, 5], [5, 7], [7, 8]])]
    for v, m, sp, text, chars in cases:
        tok, otok = get_tokenizer(dict(v), list(m), sp), oracle.OracleTokenizer(dict(v), list(m), sp)
        for unit in UNITS:
            want_ids, want = reference_offsets(otok, text.encode(), unit)
            ids, spans = tok.encode_offsets_to_numpy(text.encode(), np.int32, unit=unit)
            assert ids.tolist() == want_ids.tolist() and spans.tolist() == want.tolist(), (text, unit)
        assert tok.encode_with_offsets(text) == (want_ids.tolist(), [tuple(c) for c in chars])


@pytest.mark.parametrize("unit", UNITS)
def test_batch_equals_per_document(toks, unit):
    tok, otok = toks
    for docs in _doc_lists() + [["", "a", "", "é\U0001F643", EOT, ""], [_wide_text(3000, s).decode() for s in range(50)]]:
        ids, spans, offs = tok.encode_batch_offsets_to_numpy(docs, np.int32, unit=unit)
        a, ao = tok.encode_batch_to_numpy(docs, np.int32)
        assert np.array_equal(ids, a) and np.array_equal(offs, ao)
        for j in range(0, len(docs), max(1, len(docs) // 200)):      # (one pipeline per document: a sample of the long lists)
            di, ds = tok.encode_offsets_to_numpy(docs[j].encode(), np.int32, unit=unit)
            assert np.array_equal(ids[offs[j]: offs[j + 1]], di) and np.array_equal(spans[offs[j]: offs[j + 1]], ds), j
    docs = [d.decode() for d in list(_all_texts().values())[:3]] + ["", "x"]
    got = tok.encode_batch_with_offsets(docs)
    assert got == [tok.encode_with_offsets(d) for d in docs]


def test_batch_dropout_offsets(gpt2):
    tok, otok = gpt2
    docs = _doc_lists()[0][:300] + [_wide_text(2000, s).decode() for s in range(20)]
    for unit in UNITS:
        ids, spans, offs = tok.encode_batch_offsets_to_numpy(docs, np.int32, unit=unit, dropout=0.3, seed=9)
        for j, d in enumerate(docs):
            want_ids = otok.encode_bytes(d.encode(), dropout=0.3, seed=9, doc=j)
            assert np.array_equal(ids[offs[j]: offs[j + 1]], want_ids), j
            assert np.array_equal(spans[offs[j]: offs[j + 1]], reference_offsets(otok, d.encode(), unit, ids=want_ids)[1]), j
    got = tok.encode_batch_with_offsets(docs[:5], dropout=0.3, seed=9)
    assert got[0] == tok.encode_with_offsets(docs[0], dropout=0.3, seed=9)    # document 0 is sampled as encode's


def test_many_tiny_and_empty_documents(gpt2):
    tok, otok = gpt2
    assert tok.encode_with_offsets("") == ([], [])
    assert tok.encode_batch_with_offsets([]) == []
    assert tok.encode_batch_with_offsets(["", "", ""]) == [([], [])] * 3
    words = ["", "a", " the", "ing", EOT, " tokenization", "é", "  ", "\U0001F643"]
    docs = [words[(j * 7919) % len(words)] + words[(j * 104729) % len(words)] for j in range(100_000)]
    for unit in UNITS:
        ids, spans, offs = tok.encode_batch_offsets_to_numpy(docs, np.int32, unit=unit)
        for j in list(range(0, 100_000, 997)) + [99_999]:
            want_ids, want = reference_offsets(otok, docs[j].encode(), unit)
            assert np.array_equal(ids[offs[j]: offs[j + 1]], want_ids) and np.array_equal(spans[offs[j]: offs[j + 1]], want), j


def test_cache_state_does_not_matter(gpt2):
    tok, _ = gpt2
    data = _all_texts()["synth_owt"]
    docs = _doc_lists()[3]
    L = _lib.lib()
    L.bpe_tok_cache_reset(tok._device_tok())
    cold = tok.encode_offsets_to_numpy(data, np.int32, unit="char")
    cold_b = tok.encode_batch_offsets_to_numpy(docs, np.int32, unit="char")
    warm = tok.encode_offsets_to_numpy(data, np.int32, unit="char")
    warm_b = tok.encode_batch_offsets_to_numpy(docs, np.int32, unit="char")
    L.bpe_tok_cache_reset(tok._device_tok())
    reset_b = tok.encode_batch_offsets_to_numpy(docs, np.int32, unit="char")
    for a, b in [(cold, warm), (cold_b, warm_b), (cold_b, reset_b)]:
        assert all(np.array_equal(x, y) for x, y in zip(a, b))


def _outcome(fn):
    try:
        fn()
        return ("ok",)
    except (KeyError, UnicodeError) as e:
        return (type(e), e.args)


def test_errors_match_ids_only_calls():
    vocab, merges = load_gpt2_fixture()
    vocab = dict(vocab)
    del vocab[next(k for k, v in vocab.items() if v == b" token")]   # deterministic BPE emits it in " token"
    tok = get_tokenizer(vocab, list(merges), [EOT])
    docs = ["hello", " world", " tokenization", " token", "more"]
    for kw in (dict(), dict(dropout=0.5, seed=1)):
        for unit in UNITS:
            a = _outcome(lambda: tok.encode_batch_to_numpy(docs, np.int32, **kw))
            b = _outcome(lambda: tok.encode_batch_offsets_to_numpy(docs, np.int32, unit=unit, **kw))
            assert a == b and (kw or a[0] is KeyError), (kw, unit, a)
            data = "".join(docs).encode()
            assert _outcome(lambda: tok.encode_to_numpy(data, np.int32, **kw)) == _outcome(
                lambda: tok.encode_offsets_to_numpy(data, np.int32, unit=unit, **kw))
    good = get_tokenizer(*load_gpt2_fixture(), [EOT])
    bad_docs = [["ok", b"fine \xff", "x"], ["ok", "lone \ud800 surrogate", "x"], [b"\xc3", "x", b"\xe2\x82"],
                ["a" * 100, " tokenization", b"bad \xc3\x28 utf-8"]]
    for docs in bad_docs:
        a = _outcome(lambda: good.encode_batch_to_numpy(docs, np.int32))
        b = _outcome(lambda: good.encode_batch_offsets_to_numpy(docs, np.int32, unit="char"))
        assert a == b and a[0] != "ok", docs
    data = b"abc \xe2\x82 def"
    assert _outcome(lambda: good.encode_to_numpy(data)) == _outcome(lambda: good.encode_offsets_to_numpy(data, unit="char"))


def test_encode_ex_unknown_unit_and_count_only(gpt2):
    tok, _ = gpt2
    L = _lib.lib()
    h = tok._device_tok()
    data = np.frombuffer(b"hello world", dtype=np.uint8)
    out = np.zeros(16, dtype=np.int32)
    spans = np.zeros((16, 2), dtype=np.int64)
    n = C.c_uint64(0)

    def encode_offsets(out, cap, unit, offs_out):
        opts = _lib.EncodeOpts(with_offsets=1, offset_unit=unit, offs_out=offs_out)
        return L.bpe_encode_ex(h, _lib.ptr(data), data.size, C.byref(opts), _lib.DTYPE_I32, out, cap, C.byref(n), None)

    for unit in (-1, 2, 99):
        assert encode_offsets(_lib.ptr(out), 16, unit, spans.ctypes.data) == _lib.ERR_ARG
    assert encode_offsets(_lib.ptr(out), 16, 0, None) == _lib.ERR_ARG
    assert encode_offsets(None, 0, 0, None) == _lib.BPE_OK
    assert n.value == 2
    assert encode_offsets(_lib.ptr(out), 1, 0, spans.ctypes.data) == _lib.ERR_TOO_SMALL
    assert spans[0].tolist() == [0, 5]


# More than 96 MB (shorter texts are never cut), with a non-ASCII document of 6 MB and others larger than a pipeline chunk
# (BPE_ENCODE_CHUNK_MB=1): the same ids and spans as with one chunk.
LARGE_CODE = """
    import hashlib, sys
    import numpy as np
    import _bootstrap
    from tests.test_gpu_encode_offsets import _large_inputs
    from tests.adapters import get_tokenizer
    from tests.common import load_gpt2_fixture
    tok = get_tokenizer(*load_gpt2_fixture(), ["<|endoftext|>"])
    docs, one, _ = _large_inputs()
    h = lambda *a: hashlib.sha256(b"".join(x.tobytes() for x in a)).hexdigest()
    for unit in ("byte", "char"):
        print(unit, h(*tok.encode_batch_offsets_to_numpy(docs, np.int32, unit=unit)),
              h(*tok.encode_offsets_to_numpy(one, np.int32, unit=unit, dropout=0.1, seed=2)))
"""


def _large_inputs():
    tiny = synth_host("tinystories", 1234, 100 << 20).tobytes().decode("utf-8", errors="ignore").split(EOT)
    owt = synth_host("owt", 77, 6 << 20).tobytes().decode("utf-8", errors="ignore")
    big = len(tiny) // 2
    docs = tiny[:big] + [owt, "x é", "", _wide_text(300_000, 4).decode()] + tiny[big:]
    return docs, EOT.join(docs).encode(), big


def test_chunk_boundaries(tmp_path):
    import hashlib
    e = dict(os.environ, BPE_ENCODE_CHUNK_MB="1", BPE_ENC_BATCH_KB="256")
    r = subprocess.run([sys.executable, "-c", textwrap.dedent(LARGE_CODE)], cwd=ROOT, env=e, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    chunked = {line.split()[0]: line.split()[1:] for line in r.stdout.splitlines()}
    vocab, merges = load_gpt2_fixture()
    tok, otok = get_tokenizer(dict(vocab), list(merges), [EOT]), oracle.OracleTokenizer(dict(vocab), list(merges), [EOT])
    docs, one, big = _large_inputs()
    h = lambda *a: hashlib.sha256(b"".join(x.tobytes() for x in a)).hexdigest()      # noqa: E731
    for unit in UNITS:
        ids, spans, offs = tok.encode_batch_offsets_to_numpy(docs, np.int32, unit=unit)
        assert h(ids, spans, offs) == chunked[unit][0], unit
        for j in (big, big + 3):                 # the non-ASCII documents of 6 and ~1 MB, against the reference
            want_ids = otok.encode_bytes(docs[j].encode())
            want = reference_offsets(otok, docs[j].encode(), unit, ids=want_ids)[1]
            assert np.array_equal(ids[offs[j]: offs[j + 1]], want_ids) and np.array_equal(spans[offs[j]: offs[j + 1]], want), (unit, j)
        assert spans[offs[big + 1]].tolist() == [0, 1]                    # "x é" starts again at 0
        ids, spans = tok.encode_offsets_to_numpy(one, np.int32, unit=unit, dropout=0.1, seed=2)
        assert h(ids, spans) == chunked[unit][1], unit
        assert spans[-1, 1] == (len(one) if unit == "byte" else len(one.decode()))
