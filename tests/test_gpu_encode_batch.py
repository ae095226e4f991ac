"""GPU parity of Tokenizer.encode_batch / encode_batch_to_numpy (bpe_encode_batch): many documents in one device pass must give
exactly [tok.encode(d) for d in docs] -- the same ids, the same split, the same first exception.  The expected value is the CPU
oracle per document (and the encode loop); the documents are chosen so that encoding their concatenation would differ."""
import ctypes as C
import os
import random
import subprocess
import sys
import textwrap

import numpy as np
import pytest

import _bootstrap  # noqa: F401
from oracle import oracle
from tests.adapters import get_tokenizer
from tests.common import FIXTURES_PATH, load_gpt2_fixture
from tests.test_gpu_tokenizer import ALPHA, _trained
from transformer_lm_b200 import _lib

pytestmark = pytest.mark.gpu

EOT = "<|endoftext|>"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _pair(which):
    if which == "gpt2":
        vocab, merges, sp = *load_gpt2_fixture(), [EOT]
    elif which == "gpt2_plain":
        vocab, merges, sp = *load_gpt2_fixture(), []
    else:
        vocab, merges, sp = *_trained(1000, [EOT]), [EOT]
    return get_tokenizer(dict(vocab), list(merges), sp), oracle.OracleTokenizer(dict(vocab), list(merges), sp)


@pytest.fixture(scope="module", params=["gpt2", "gpt2_plain", "corpus1000"])
def toks(request):
    return _pair(request.param)


@pytest.fixture(scope="module")
def gpt2():
    return _pair("gpt2")


def _document_lists():
    lists = []
    for name in ["corpus.en", "german.txt", "address.txt", "tinystories_sample.txt"]:
        text = (FIXTURES_PATH / name).read_text(encoding="utf-8")
        lists.append(text.splitlines(keepends=True))
        lists.append(text.split("\n\n"))
    lists.append((FIXTURES_PATH / "tinystories_sample.txt").read_text(encoding="utf-8").split(EOT))
    rnd = random.Random(5)
    lists.append(["".join(rnd.choice(ALPHA) for _ in range(rnd.randint(0, 60))) for _ in range(400)])
    return lists


def test_parity_on_document_lists(toks):
    tok, otok = toks
    for docs in _document_lists():
        got = tok.encode_batch(docs)
        assert got == [otok.encode(d) for d in docs]
    docs = _document_lists()[-1][:150]
    assert tok.encode_batch(docs) == [tok.encode(d) for d in docs]


HAZARDS = [("a  ", "b"), ("x ", "y"), ("don'", "t"), ("we'", "ve"), ("19", "99"), ("2", "000"), ("...", "..."), ("!?", "!?"),
           ("é", "t"), ("r", "ésumé"), ("Zür", "ich"), (" ", "é"), ("<|endo", "ftext|>"), ("\n", "\n")]


@pytest.mark.parametrize("a,b", HAZARDS)
def test_no_pretoken_crosses_a_document_boundary(gpt2, a, b):
    tok, otok = gpt2
    assert tok.encode(a + b) != tok.encode(a) + tok.encode(b)          # the test bites: the join tokenises differently
    assert tok.encode_batch([a, b]) == [otok.encode(a), otok.encode(b)]
    assert tok.encode_batch([b, a, b]) == [otok.encode(b), otok.encode(a), otok.encode(b)]


def test_specials_at_document_edges(gpt2):
    tok, otok = gpt2
    docs = [EOT, EOT + "a", "b" + EOT, "", EOT + EOT, " " + EOT + " ", "x" + EOT + "y", EOT[:5], EOT[5:]]
    assert tok.encode_batch(docs) == [otok.encode(d) for d in docs]


ALL_ASCII = "".join(chr(i) for i in range(128))


@pytest.mark.parametrize("specials", [["\x00"], ["\x00", "\n"], ["a\x00b", "\n\n", EOT], ["".join(chr(i) for i in range(64) if i != 13)]])
def test_boundary_byte_avoids_every_special(specials):
    vocab, merges = _trained(1000, [EOT])
    tok = get_tokenizer(dict(vocab), list(merges), specials)
    otok = oracle.OracleTokenizer(dict(vocab), list(merges), specials)
    docs = [ALL_ASCII, "\x00", "\x00\x01\x02", "\r\n", "\r", "\n", "a", "\x01" * 5, ALL_ASCII[::-1], "", "\x00 \x00"] + specials
    docs += [s[:1] for s in specials] + [s[1:] for s in specials]
    assert tok.encode_batch(docs) == [otok.encode(d) for d in docs]


def test_no_boundary_byte_left_is_unsupported():
    vocab = {i: bytes([i]) for i in range(256)}
    specials = [chr(i) for i in range(128) if i != 13]
    tok = get_tokenizer(dict(vocab), [], specials)
    with pytest.raises(_lib.BpeError) as e:
        tok.encode_batch(["a"])
    assert e.value.code == _lib.ERR_UNSUPPORTED
    assert tok.encode_batch([]) == []


def test_shapes(gpt2):
    tok, otok = gpt2
    assert tok.encode_batch([]) == []
    ids, offs = tok.encode_batch_to_numpy([])
    assert ids.size == 0 and offs.tolist() == [0] and offs.dtype == np.int64
    assert tok.encode_batch([""]) == [[]]
    assert tok.encode_batch(["", "", ""]) == [[], [], []]
    for docs in (["", "a b", "c"], ["a b", "", "c"], ["a b", "c", ""], ["", "a", "", "", "b", ""]):
        assert tok.encode_batch(docs) == [otok.encode(d) for d in docs]
    text = (FIXTURES_PATH / "german.txt").read_text(encoding="utf-8")
    assert tok.encode_batch([text]) == [tok.encode(text)]


def test_200k_tiny_documents(gpt2):
    tok, otok = gpt2
    rnd = random.Random(7)
    docs = ["".join(rnd.choice(ALPHA) for _ in range(rnd.randint(0, 4))) for _ in range(200_000)]
    memo = {}
    want = [memo[d] if d in memo else memo.setdefault(d, otok.encode(d)) for d in docs]
    assert tok.encode_batch(docs) == want


def _keyerror_tok():
    vocab = {i: bytes([i]) for i in range(256)}
    merges = [(b"a", b"b"), (b"ab", b"c")]                               # b"ab", b"abc" are not in the vocab
    return get_tokenizer(dict(vocab), list(merges), []), oracle.OracleTokenizer(dict(vocab), list(merges), [])


def test_keyerror_of_the_first_failing_document():
    tok, otok = _keyerror_tok()
    docs = ["xyz"] * 50 + ["q abc"] + ["zz"] * 10 + ["zab"] + ["x"] * 5
    with pytest.raises(KeyError) as e1:
        tok.encode_batch(docs)
    with pytest.raises(KeyError) as e2:
        [otok.encode(d) for d in docs]
    assert e1.value.args == e2.value.args == (b"abc",)
    with pytest.raises(KeyError) as e3:
        tok.encode_batch(docs[51:])
    assert e3.value.args == (b"ab",)
    assert tok.encode_batch(["xyz", "a b c"]) == [otok.encode("xyz"), otok.encode("a b c")]


def test_surrogate_and_keyerror_ordering():
    tok, _ = _keyerror_tok()
    with pytest.raises(KeyError):
        tok.encode_batch(["ok", "zab", "ok", "bad \ud800"])
    with pytest.raises(UnicodeEncodeError):
        tok.encode_batch(["ok", "bad \ud800", "zab"])


def test_per_document_utf8_validity(gpt2):
    tok, otok = gpt2
    docs = [b"ok ", b"abc\xe4\xb8", b"\xad rest"]                         # joined: valid ("abc" + U+4E2D + " rest")
    b"".join(docs).decode("utf-8")
    with pytest.raises(UnicodeDecodeError) as e:
        tok.encode_batch_to_numpy(docs)
    with pytest.raises(UnicodeDecodeError) as want:
        docs[1].decode("utf-8")
    assert (e.value.start, e.value.end, e.value.reason, e.value.object) == (want.value.start, want.value.end, want.value.reason, want.value.object)
    with pytest.raises(UnicodeDecodeError) as e:
        tok.encode_batch_to_numpy([b"ok", b"\xad rest"])
    assert e.value.object == b"\xad rest"
    ids, offs = tok.encode_batch_to_numpy([b"caf\xc3\xa9", "naïve", b""])
    assert [ids[offs[j]: offs[j + 1]].tolist() for j in range(3)] == [otok.encode("café"), otok.encode("naïve"), []]
    # C ABI: the detail is the offset of the bad sequence in the caller's text, boundary bytes not counted
    L = _lib.lib()
    h = tok._device_tok()
    blob = np.frombuffer(b"".join(docs), dtype=np.uint8)
    doc_offs = np.array([0, 3, 8, 14], dtype=np.uint64)
    out = np.empty(blob.size, dtype=np.int32)
    id_offs = np.zeros(4, dtype=np.uint64)
    n_out = C.c_uint64(0)
    rc = L.bpe_encode_batch(h, _lib.ptr(blob), blob.size, _lib.ptr(doc_offs), 3, _lib.DTYPE_I32, _lib.ptr(out), out.size,
                            C.byref(n_out), _lib.ptr(id_offs), None)
    assert rc == _lib.ERR_UTF8
    assert L.bpe_last_error_detail(tok._tok_ctx.handle) == 6


def test_keyerror_before_a_later_invalid_document():
    tok, _ = _keyerror_tok()
    with pytest.raises(KeyError):
        tok.encode_batch_to_numpy([b"ok", b"zab", b"\xff", b"q"])
    with pytest.raises(UnicodeDecodeError):
        tok.encode_batch_to_numpy([b"ok", b"\xff", b"zab"])


def test_c_abi_argument_checks(gpt2):
    tok, _ = gpt2
    L = _lib.lib()
    h = tok._device_tok()
    blob = np.frombuffer(b"abcdef", dtype=np.uint8)
    out = np.empty(8, dtype=np.int32)
    ids = np.zeros(3, dtype=np.uint64)
    n_out = C.c_uint64(0)
    for offs in ([0, 4, 3], [1, 3, 6], [0, 3, 5]):
        o = np.array(offs, dtype=np.uint64)
        assert L.bpe_encode_batch(h, _lib.ptr(blob), 6, _lib.ptr(o), 2, _lib.DTYPE_I32, _lib.ptr(out), 8, C.byref(n_out),
                                  _lib.ptr(ids), None) == _lib.ERR_ARG
    o = np.array([0, 3, 6], dtype=np.uint64)
    assert L.bpe_encode_batch(h, _lib.ptr(blob), 6, _lib.ptr(o), 2, _lib.DTYPE_I32, _lib.ptr(out), 8, C.byref(n_out), _lib.ptr(ids), None) == 0
    assert ids.tolist()[0] == 0 and ids.tolist()[2] == n_out.value
    assert L.bpe_encode_batch(h, _lib.ptr(blob), 6, _lib.ptr(o), 2, _lib.DTYPE_I32, None, 0, C.byref(n_out), _lib.ptr(ids), None) == 0
    assert ids.tolist()[2] == n_out.value                                 # size query: the offsets too


def test_uint16_refusal_and_agreement(gpt2):
    tok, _ = gpt2
    docs = (FIXTURES_PATH / "german.txt").read_text(encoding="utf-8").splitlines(keepends=True)
    a, oa = tok.encode_batch_to_numpy(docs, np.uint16)
    b, ob = tok.encode_batch_to_numpy(docs, np.int32)
    assert a.dtype == np.uint16 and b.dtype == np.int32
    assert a.astype(np.int64).tolist() == b.astype(np.int64).tolist() and oa.tolist() == ob.tolist()
    assert ob[0] == 0 and ob[-1] == len(b) and len(ob) == len(docs) + 1
    vocab = {i: bytes([i]) for i in range(256)}
    vocab[70000] = b"ab"
    big = get_tokenizer(vocab, [(b"a", b"b")], [])
    assert big.encode_batch(["abc", "ab"]) == [[70000, 99], [70000]]
    with pytest.raises(_lib.BpeError) as e1:
        big.encode_to_numpy(b"abc", np.uint16)
    with pytest.raises(type(e1.value)):
        big.encode_batch_to_numpy(["abc"], np.uint16)


def test_cache_interplay(gpt2):
    tok, _ = gpt2
    docs = (FIXTURES_PATH / "corpus.en").read_text(encoding="utf-8").split("\n\n")
    first = tok.encode_batch(docs)
    joined = "\n\n".join(docs)
    assert tok.encode(joined) == tok.encode(joined)
    _lib.lib().bpe_tok_cache_reset(tok._device_tok())
    assert tok.encode_batch(docs) == first
    assert tok.encode_batch(docs) == first


LARGE_CODE = """
    import random
    import numpy as np
    import _bootstrap
    from oracle import oracle
    from transformer_lm_b200.synth import synth_host
    from tests.adapters import get_tokenizer
    from tests.common import load_gpt2_fixture
    EOT = "<|endoftext|>"
    vocab, merges = load_gpt2_fixture()
    tok = get_tokenizer(dict(vocab), list(merges), [EOT])
    text = synth_host("tinystories", 1234, 128 << 20).tobytes().decode("utf-8", errors="ignore")
    docs = text.split(EOT)
    rnd = random.Random(3)
    big = " ".join(rnd.choice(["once", "upon", "a", "time", "Lily", "saw", "3", "dog."]) for _ in range(3_000_000))
    docs.insert(len(docs) // 2, big)                                   # one document larger than a pipeline chunk
    ids, offs = tok.encode_batch_to_numpy(docs, np.int32)
    # every document on its own == the joined text with <|endoftext|> between them (a special is a hard boundary), split at it
    want = tok.encode_to_numpy(EOT.join(docs).encode("utf-8"), np.int32)
    eot = 50256
    cuts = np.flatnonzero(want == eot)
    assert len(cuts) == len(docs) - 1, (len(cuts), len(docs))
    starts = np.concatenate([[0], cuts + 1]); ends = np.concatenate([cuts, [len(want)]])
    assert np.array_equal(np.delete(want, cuts), ids)
    assert np.array_equal(offs[:-1], starts - np.arange(len(docs))) and offs[-1] == len(ids)
    otok = oracle.OracleTokenizer(dict(vocab), list(merges), [EOT])
    for j in rnd.sample(range(len(docs)), 200):
        assert ids[offs[j]: offs[j + 1]].tolist() == otok.encode(docs[j]), j
    print("ok", len(docs), len(ids), tok.last_stats["ms_total"])
"""


def test_multi_batch_multi_chunk():
    e = dict(os.environ, BPE_ENC_BATCH_KB="4096", BPE_ENCODE_CHUNK_MB="8")
    r = subprocess.run([sys.executable, "-c", textwrap.dedent(LARGE_CODE)], cwd=ROOT, env=e, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert r.stdout.startswith("ok ")
