"""GPU parity of BPE-dropout (bpe_encode_dropout / bpe_encode_batch_dropout through Tokenizer.encode_to_numpy and
encode_batch_to_numpy): exact equality with the CPU dropout oracle (tests/helpers/dropout_oracle.c), with doc = the document's index in the batch;
independence from the pretoken cache, from batch and chunk boundaries; p = 0 is encode."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

import _bootstrap  # noqa: F401
from tests.helpers.dropout_oracle import DropoutOracle
from tests.adapters import get_tokenizer
from tests.common import FIXTURES_PATH, load_gpt2_fixture
from tests.test_gpu_tokenizer import _trained
from transformer_lm_b200 import _lib
from transformer_lm_b200.synth import synth_host

pytestmark = pytest.mark.gpu

EOT = "<|endoftext|>"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PS = [0.05, 0.1, 0.5, 1.0]
SEEDS = [0, 7, 2**64 - 1]


def _pair(which):
    if which == "gpt2":
        vocab, merges, sp = *load_gpt2_fixture(), [EOT]
    elif which == "gpt2_plain":
        vocab, merges, sp = *load_gpt2_fixture(), []
    else:
        vocab, merges, sp = *_trained(1000, [EOT]), [EOT]
    return get_tokenizer(dict(vocab), list(merges), sp), DropoutOracle(dict(vocab), list(merges), sp)


@pytest.fixture(scope="module", params=["gpt2", "gpt2_plain", "corpus1000"])
def toks(request):
    return _pair(request.param)


@pytest.fixture(scope="module")
def gpt2():
    return _pair("gpt2")


def _texts():
    out = {name: (FIXTURES_PATH / name).read_bytes() for name in ["corpus.en", "tinystories_sample.txt", "german.txt"]}
    out["synth_owt"] = synth_host("owt", 3, 3 << 20).tobytes().decode("utf-8", errors="ignore").encode()
    # pretokens at and around the row limits of the per-thread kernel (15 / 16 and 32 / 33 bytes) and long runs of one repeated
    # byte for the per-warp kernel; joined by spaces, every part but the first is a pretoken one byte longer (" " + the part)
    parts = ["a" * 33, "a" * 1000, " " * 777 + "x", "ab" * 500, "=" * 4097, "é" * 700, "x" * 32, "y" * 31, "z" * 64, "w" * 65,
             "q" * 14, "r" * 15, "s" * 16]
    out["long_pretokens"] = " ".join(parts).encode()
    return out


def _oracle(otok, data, p, seed, doc=0):
    try:
        return otok.encode_bytes(data, dropout=p, seed=seed, doc=doc)
    except KeyError as e:
        return ("KeyError", e.args[0])


def _device(tok, data, p, seed, dtype=np.int32):
    try:
        return tok.encode_to_numpy(data, dtype, dropout=p, seed=seed)
    except KeyError as e:
        return ("KeyError", e.args[0])


def _same(a, b):
    if isinstance(a, tuple) or isinstance(b, tuple):
        return a == b
    return np.array_equal(np.asarray(a, dtype=np.int64), np.asarray(b, dtype=np.int64))


@pytest.mark.parametrize("p", PS)
def test_encode_matches_oracle(toks, p):
    tok, otok = toks
    for name, data in _texts().items():
        for seed in SEEDS[:2] if name == "synth_owt" else SEEDS:
            want = _oracle(otok, data, p, seed)
            assert _same(_device(tok, data, p, seed), want), (name, seed)
            if max(otok.vocab_inv.values()) < 65536:
                assert _same(_device(tok, data, p, seed, np.uint16), want), (name, seed, "uint16")


def _doc_lists():
    ts = (FIXTURES_PATH / "tinystories_sample.txt").read_text(encoding="utf-8")
    en = (FIXTURES_PATH / "corpus.en").read_text(encoding="utf-8")
    synth = synth_host("tinystories", 4, 2 << 20).tobytes().decode("utf-8", errors="ignore")
    return [ts.split(EOT), en.split("\n\n"), en.splitlines(keepends=True)[:2000], synth.split(EOT)]


@pytest.mark.parametrize("p", PS)
def test_encode_batch_matches_oracle(toks, p):
    tok, otok = toks
    for k, docs in enumerate(_doc_lists()):
        for seed in SEEDS[:2]:
            for dtype in (np.int32, np.uint16) if max(otok.vocab_inv.values()) < 65536 else (np.int32,):
                ids, offs = tok.encode_batch_to_numpy(docs, dtype, dropout=p, seed=seed)
                assert offs.size == len(docs) + 1
                for j, d in enumerate(docs):
                    want = otok.encode_bytes(d.encode(), dropout=p, seed=seed, doc=j)
                    assert np.array_equal(ids[offs[j]: offs[j + 1]].astype(np.int64), want), (k, seed, j)
    docs = _doc_lists()[0]
    for j, d in enumerate(docs[:20]):                # encode(d) == encode_batch([d])[0]; the position in the batch matters
        assert tok.encode(d, dropout=p, seed=3) == tok.encode_batch([d], dropout=p, seed=3)[0]
        assert tok.encode_batch(docs[: j + 1], dropout=p, seed=3)[j] == otok.encode_bytes(d.encode(), dropout=p, seed=3, doc=j).tolist()


def test_p0_is_encode(toks):
    tok, _ = toks
    for data in _texts().values():
        assert np.array_equal(tok.encode_to_numpy(data, np.int32, dropout=0.0, seed=9), tok.encode_to_numpy(data, np.int32))
    for docs in _doc_lists():
        a, ao = tok.encode_batch_to_numpy(docs, np.int32, dropout=0.0, seed=9)
        b, bo = tok.encode_batch_to_numpy(docs, np.int32)
        assert np.array_equal(a, b) and np.array_equal(ao, bo)


def test_seed_determinism(gpt2):
    tok, _ = gpt2
    data = _texts()["synth_owt"]
    a = tok.encode_to_numpy(data, np.int32, dropout=0.1, seed=1)
    assert np.array_equal(a, tok.encode_to_numpy(data, np.int32, dropout=0.1, seed=1))
    assert not np.array_equal(a, tok.encode_to_numpy(data, np.int32, dropout=0.1, seed=2))
    docs = _doc_lists()[3]
    x = tok.encode_batch_to_numpy(docs, np.int32, dropout=0.1, seed=1)[0]
    assert np.array_equal(x, tok.encode_batch_to_numpy(docs, np.int32, dropout=0.1, seed=1)[0])
    assert not np.array_equal(x, tok.encode_batch_to_numpy(docs, np.int32, dropout=0.1, seed=2)[0])


def test_cache_state_does_not_matter(gpt2):
    tok, _ = gpt2
    data = _texts()["synth_owt"]
    docs = _doc_lists()[3]
    L = _lib.lib()
    L.bpe_tok_cache_reset(tok._device_tok())
    cold = tok.encode_to_numpy(data, np.int32, dropout=0.1, seed=4)
    cold_b = tok.encode_batch_to_numpy(docs, np.int32, dropout=0.1, seed=4)[0]
    tok.encode_to_numpy(data, np.int32)                                  # warm (deterministic values cached)
    assert np.array_equal(tok.encode_to_numpy(data, np.int32, dropout=0.1, seed=4), cold)
    assert np.array_equal(tok.encode_batch_to_numpy(docs, np.int32, dropout=0.1, seed=4)[0], cold_b)
    L.bpe_tok_cache_reset(tok._device_tok())
    assert np.array_equal(tok.encode_batch_to_numpy(docs, np.int32, dropout=0.1, seed=4)[0], cold_b)
    assert np.array_equal(tok.encode_to_numpy(data, np.int32, dropout=0.1, seed=4), cold)


def test_key_error_matches_oracle():
    vocab, merges = load_gpt2_fixture()
    vocab = dict(vocab)
    iz = next(k for k, v in vocab.items() if v == b"iz")
    del vocab[iz]                                # an intermediate product deterministic BPE never emits in " tokenization"
    tok, otok = get_tokenizer(dict(vocab), list(merges), [EOT]), DropoutOracle(dict(vocab), list(merges), [EOT])
    text = " tokenization"
    assert tok.encode(text) == otok.encode(text)
    with pytest.raises(KeyError) as e:
        tok.encode(text, dropout=0.5, seed=1)
    assert e.value.args[0] == b"iz"
    docs = ["hello world", " the cat", text * 3, " tokenization", "more"]
    for seed in range(6):
        first = None
        for j, d in enumerate(docs):             # the oracle's first failing document, in list order, and its key
            r = _oracle(otok, d.encode(), 0.5, seed, j)
            if isinstance(r, tuple):
                first = r
                break
        if first is None:
            got = tok.encode_batch(docs, dropout=0.5, seed=seed)
            assert got == [otok.encode_bytes(d.encode(), dropout=0.5, seed=seed, doc=j).tolist() for j, d in enumerate(docs)]
        else:
            with pytest.raises(KeyError) as e:
                tok.encode_batch(docs, dropout=0.5, seed=seed)
            assert e.value.args[0] == first[1], seed
        joined = "".join(docs).encode()
        assert _same(_device(tok, joined, 0.5, seed), _oracle(otok, joined, 0.5, seed))


def test_empty_and_many_tiny_documents(gpt2):
    tok, otok = gpt2
    assert tok.encode("", dropout=0.5, seed=1) == []
    assert tok.encode_batch([], dropout=0.5, seed=1) == []
    assert tok.encode_batch(["", "", ""], dropout=0.5, seed=1) == [[], [], []]
    words = ["", "a", " the", "ing", EOT, " tokenization", "é", "  "]
    docs = [words[(j * 7919) % len(words)] + words[(j * 104729) % len(words)] for j in range(100_000)]
    ids, offs = tok.encode_batch_to_numpy(docs, np.int32, dropout=0.5, seed=11)
    for j in list(range(0, 100_000, 997)) + [99_999]:
        assert ids[offs[j]: offs[j + 1]].tolist() == otok.encode_bytes(docs[j].encode(), dropout=0.5, seed=11, doc=j).tolist(), j


# A document larger than a pipeline chunk (BPE_ENCODE_CHUNK_MB) and many batches (BPE_ENC_BATCH_KB): the same ids as with one chunk.
LARGE_CODE = """
    import random, sys
    import numpy as np
    import _bootstrap
    from transformer_lm_b200.synth import synth_host
    from tests.adapters import get_tokenizer
    from tests.common import load_gpt2_fixture
    EOT = "<|endoftext|>"
    vocab, merges = load_gpt2_fixture()
    tok = get_tokenizer(dict(vocab), list(merges), [EOT])
    text = synth_host("tinystories", 1234, 100 << 20).tobytes().decode("utf-8", errors="ignore")
    docs = text.split(EOT)
    rnd = random.Random(3)
    big = " ".join(rnd.choice(["once", "upon", "a", "time", "Lily", "saw", "3", "dog."]) for _ in range(3_000_000))
    docs.insert(len(docs) // 2, big)
    ids, offs = tok.encode_batch_to_numpy(docs, np.int32, dropout=0.1, seed=5)
    one = tok.encode_to_numpy(EOT.join(docs).encode(), np.int32, dropout=0.1, seed=5)
    np.save(sys.argv[1] + "/ids.npy", ids); np.save(sys.argv[1] + "/offs.npy", offs); np.save(sys.argv[1] + "/one.npy", one)
    print("ok", len(docs), len(ids), tok.last_stats["ms_total"])
"""


def test_chunk_and_batch_boundaries(tmp_path):
    e = dict(os.environ, BPE_ENC_BATCH_KB="4096", BPE_ENCODE_CHUNK_MB="8")
    r = subprocess.run([sys.executable, "-c", textwrap.dedent(LARGE_CODE), str(tmp_path)], cwd=ROOT, env=e, capture_output=True,
                       text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert r.stdout.startswith("ok ")
    # the same in this process, with one pipeline chunk
    import random
    vocab, merges = load_gpt2_fixture()
    tok = get_tokenizer(dict(vocab), list(merges), [EOT])
    text = synth_host("tinystories", 1234, 100 << 20).tobytes().decode("utf-8", errors="ignore")
    docs = text.split(EOT)
    rnd = random.Random(3)
    big = " ".join(rnd.choice(["once", "upon", "a", "time", "Lily", "saw", "3", "dog."]) for _ in range(3_000_000))
    jb = len(docs) // 2
    docs.insert(jb, big)
    ids, offs = tok.encode_batch_to_numpy(docs, np.int32, dropout=0.1, seed=5)
    assert np.array_equal(np.load(tmp_path / "offs.npy"), offs)
    assert np.array_equal(np.load(tmp_path / "ids.npy"), ids)
    assert np.array_equal(np.load(tmp_path / "one.npy"), tok.encode_to_numpy(EOT.join(docs).encode(), np.int32, dropout=0.1, seed=5))
    otok = DropoutOracle(dict(vocab), list(merges), [EOT])
    assert np.array_equal(ids[offs[jb]: offs[jb + 1]], otok.encode_bytes(big.encode(), dropout=0.1, seed=5, doc=jb))
    for j in rnd.sample(range(len(docs)), 100):
        assert ids[offs[j]: offs[j + 1]].tolist() == otok.encode_bytes(docs[j].encode(), dropout=0.1, seed=5, doc=j).tolist(), j
