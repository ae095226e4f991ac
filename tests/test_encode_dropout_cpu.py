"""BPE-dropout spec (include/bpe_sm100.h, bpe_encode_dropout) on the CPU: its test vectors and worked example, the dropout oracle
(tests/helpers/dropout_oracle.c) against an independent Python restatement of the spec on fuzzed texts, and Tokenizer's argument
checks."""
import math
import random

import numpy as np
import pytest

import _bootstrap  # noqa: F401
from oracle import oracle
from tests.helpers.dropout_oracle import DropoutOracle, dropout_u
from tests.common import load_gpt2_fixture
from transformer_lm_b200.tokenizer import Tokenizer

EOT = "<|endoftext|>"
M64 = 2**64 - 1


# ---- the spec, restated -----------------------------------------------------------------------------------------------------
def mix(z):
    z = (z + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def u(seed, doc, off, t):
    return mix(mix(mix(mix(seed) ^ doc) ^ off) ^ t)


def thr(p):
    return 2**32 if p == 1 else math.floor(p * 2**32)


def bpe_dropout(word: bytes, off: int, ranks, p, seed, doc):
    toks, offs, t = [bytes([b]) for b in word], list(range(off, off + len(word))), 0
    while True:
        cand = {i for i in range(len(toks) - 1)
                if (toks[i], toks[i + 1]) in ranks and (u(seed, doc, offs[i], t) >> 32) >= thr(p)}
        if not cand:
            return toks
        r = min(ranks[toks[i], toks[i + 1]] for i in cand)
        nt, no, i = [], [], 0
        while i < len(toks):
            if i in cand and ranks[toks[i], toks[i + 1]] == r:
                nt.append(toks[i] + toks[i + 1]); no.append(offs[i]); i += 2
            else:
                nt.append(toks[i]); no.append(offs[i]); i += 1
        toks, offs, t = nt, no, t + 1


def encode_dropout(data: bytes, vocab_inv, ranks, specials, p, seed, doc=0):
    """Segment on the specials (leftmost, longest first), GPT-2 pretokens in between, BPE-dropout of every occurrence."""
    sp = sorted((s.encode() for s in specials), key=len, reverse=True)
    pieces, i, seg = [], 0, 0                    # (offset, bytes, is_special)
    while i <= len(data):
        hit = next((s for s in sp if i < len(data) and data.startswith(s, i)), None)
        if hit is not None or i == len(data):
            if i > seg:
                st = oracle.pretokenize(data[seg:i]) + [i - seg]
                pieces += [(seg + st[k], data[seg + st[k]: seg + st[k + 1]], False) for k in range(len(st) - 1)]
            if hit is None:
                break
            pieces.append((i, hit, True))
            i = seg = i + len(hit)
            continue
        i += 1
    ids = []
    for off, b, is_sp in pieces:
        for tok in [b] if is_sp else bpe_dropout(b, off, ranks, p, seed, doc):
            if tok not in vocab_inv:
                raise KeyError(tok)
            ids.append(vocab_inv[tok])
    return ids


# ---- fixtures ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module", params=[[EOT], []], ids=["eot", "plain"])
def gpt2(request):
    vocab, merges = load_gpt2_fixture()
    otok = DropoutOracle(dict(vocab), list(merges), request.param)
    ranks = {pair: i for i, pair in enumerate(merges)}
    return otok, ranks, request.param


ALPHA = ["a", "b", "t", "e", "s", " ", " ", "  ", "\n", "'s", "é", "中", "\U0001F643", "1", "00", ".", "the", " the", "ing", "tion",
         "aaaa", EOT, "<|", " tokenization", "é" * 9]


def _fuzz_texts(seed):
    rnd = random.Random(seed)
    out = ["".join(rnd.choice(ALPHA) for _ in range(rnd.randint(0, 40))) for _ in range(30)]
    out.append("a" * 37 + " " + "aa" * 20 + " x" + "b" * 33)         # runs of one byte: the (a, a) overlap rule, > 32 bytes
    out.append(" " + "".join(rnd.choice("abcdefghijklmnopqrstuvwxyz") for _ in range(1100)))   # a pretoken > 1 024 bytes
    out.append("Zürich " * 5 + "中文字符" * 10 + EOT + " résumé" + EOT)
    return out


def _oracle_ids(otok, text, p, seed, doc):
    try:
        return otok.encode_bytes(text.encode(), dropout=p, seed=seed, doc=doc).tolist()
    except KeyError as e:
        return ("KeyError", e.args[0])


def _restated_ids(otok, ranks, specials, text, p, seed, doc):
    try:
        return encode_dropout(text.encode(), otok.vocab_inv, ranks, specials, p, seed, doc)
    except KeyError as e:
        return ("KeyError", e.args[0])


# ---- tests ------------------------------------------------------------------------------------------------------------------
def test_vectors():
    assert mix(0) == 0xE220A8397B1DCDAF and mix(1) == 0x910A2DEC89025CC1
    for args, want in [((0, 0, 0, 0), 0x2130748AAAC80268), ((1, 2, 3, 4), 0xD55CCD4AEB3CCAFB),
                       ((M64, 7, 2**40 + 5, 9), 0x6DCA632AF2E3D87E)]:
        assert u(*args) == want
        assert dropout_u(*args) == want
    assert thr(0) == 0 and thr(1) == 2**32 and thr(0.5) == 2**31


def test_worked_example(gpt2):
    otok, ranks, specials = gpt2
    cases = {(0, 0): [" token", "ization"], (0.5, 0): [" ", "to", "ke", "n", "i", "za", "t", "i", "on"],
             (0.5, 1): [" t", "ok", "en", "iz", "at", "io", "n"], (1, 0): [chr(c) for c in b" tokenization"]}
    for (p, s), want in cases.items():
        want_ids = [otok.vocab_inv[w.encode()] for w in want]
        assert otok.encode_bytes(b" tokenization", dropout=p, seed=s).tolist() == want_ids
        assert _restated_ids(otok, ranks, specials, " tokenization", p, s, 0) == want_ids


@pytest.mark.parametrize("p", [0, 0.1, 0.5, 0.9, 1])
def test_oracle_matches_restatement(gpt2, p):
    otok, ranks, specials = gpt2
    for k, text in enumerate(_fuzz_texts(11)):
        for seed, doc in [(0, 0), (1, 3), (2**64 - 1, 2**40 + 7)]:
            if p in (0.1, 0.9) and len(text) > 1000 and seed:
                continue                         # (the restatement is slow on the 1 100-byte pretoken: one seed is enough)
            assert _oracle_ids(otok, text, p, seed, doc) == _restated_ids(otok, ranks, specials, text, p, seed, doc), (k, seed, doc)


def test_p0_is_encode_and_p1_is_bytes(gpt2):
    otok, _, specials = gpt2
    sp = set(s.encode() for s in specials)
    for text in _fuzz_texts(12):
        data = text.encode()
        assert otok.encode_bytes(data, dropout=0.0, seed=5, doc=2).tolist() == otok.encode_bytes(data).tolist()
        ids = otok.encode_bytes(data, dropout=1.0, seed=5, doc=2).tolist()
        if not sp:
            assert ids == [otok.vocab_inv[bytes([b])] for b in data]
        assert b"".join(otok.vocab[i] for i in ids) == data


def test_dropout_depends_on_seed_doc_and_offset(gpt2):
    otok, _, _ = gpt2
    data = " tokenization is the process of".encode() * 8
    runs = {tuple(otok.encode_bytes(data, dropout=0.5, seed=s, doc=d).tolist()) for s in range(3) for d in range(3)}
    assert len(runs) == 9
    # a word at offset 0 is cut as on its own; the same word further on is cut differently (the offsets differ)
    alone = otok.encode_bytes(b" tokenization", dropout=0.5, seed=0).tolist()
    both = otok.encode_bytes(b" tokenization tokenization", dropout=0.5, seed=0).tolist()
    assert both[: len(alone)] == alone and both[len(alone):] != alone


def test_key_error_from_a_missing_intermediate(gpt2):
    otok, ranks, specials = gpt2
    vocab, merges = load_gpt2_fixture()
    del vocab[otok.vocab_inv[b"iz"]]
    o2 = DropoutOracle(vocab, list(merges), specials)
    assert o2.encode_bytes(b" tokenization").tolist() == otok.encode_bytes(b" tokenization").tolist()   # deterministic BPE never makes "iz"
    with pytest.raises(KeyError) as e:
        o2.encode_bytes(b" tokenization", dropout=0.5, seed=1)
    assert e.value.args[0] == b"iz"
    assert _restated_ids(o2, ranks, specials, " tokenization", 0.5, 1, 0) == ("KeyError", b"iz")


def test_oracle_rejects_bad_p(gpt2):
    otok, _, _ = gpt2
    for p in (-0.1, 1.5, float("nan")):
        with pytest.raises(ValueError):
            otok.encode_bytes(b"abc", dropout=p)


@pytest.mark.parametrize("kw", [dict(dropout=-0.01), dict(dropout=1.01), dict(dropout=float("nan")), dict(dropout=float("inf")),
                                dict(dropout=0.1, seed=-1), dict(dropout=0.1, seed=2**64), dict(dropout=0.1, seed=1.5),
                                dict(dropout=0.1, seed=True)])
def test_tokenizer_argument_validation(kw):
    vocab, merges = load_gpt2_fixture()
    tok = Tokenizer(vocab, merges, [EOT])          # (the checks come before any device work)
    for call in (lambda: tok.encode("abc", **kw), lambda: tok.encode_to_numpy(b"abc", np.int32, **kw),
                 lambda: tok.encode_batch(["abc"], **kw), lambda: tok.encode_batch_to_numpy(["abc"], np.int32, **kw)):
        with pytest.raises(ValueError):
            call()
