"""The composition of the tier corpus (tests/helpers/tier_corpus.py) that the GPU tests of the pretoken tables run on, pinned through
the oracle's count.  Those tests only cover table growth with entries, the tier boundaries and the near-twin compares while the corpus
holds what is listed here: an edit of the generator that silently stops producing it fails on CPU."""
import collections

import pytest

import _bootstrap  # noqa: F401
from oracle import oracle
from tests.helpers import tier_corpus as tc


@pytest.fixture(scope="module")
def corpus():
    text, info = tc.tier_corpus(0)
    return text, info, oracle.count_pretokens(text, [])


def _tier(n):
    return 0 if n <= 7 else 1 if n <= 15 else 2


def test_every_placed_word_is_one_pretoken(corpus):
    text, info, count = corpus
    text.decode("utf-8")
    assert b"\r" not in text
    # the oracle finds exactly the words the generator placed (and the separators it put between whitespace runs)
    sep = {b" ws", b" end"}
    assert set(count) | sep == set(info["words"]) | set(tc.FREQUENT) | sep


def test_tier_sizes_grow_every_table(corpus):
    """Enough distinct pretokens in every tier that each table must grow with entries in it when the text arrives in pieces: the long
    table (2^14 slots at the start, grown at 7/8 load) needs more than ~14 000, the medium one alike, the short one (2^16) ~57 000
    together with a batch's bound."""
    _, _, count = corpus
    tiers = collections.Counter(_tier(len(k)) for k in count)
    assert tiers[2] >= 20000 and tiers[1] >= 25000 and tiers[0] >= 45000, tiers
    longs = [len(k) for k in count if len(k) > 15]
    assert sum(16 <= n <= 32 for n in longs) >= 5000 and sum(n > 32 for n in longs) >= 5000      # both BPE kernels of the encoder
    assert sum(n >= 4096 for n in longs) >= 30
    # designed counts: most words occur 1-4 times; a few very frequent ones feed the shared-memory and hot tables
    freq = sorted(count.values(), reverse=True)
    assert freq[len(tc.FREQUENT) - 1] >= 2000 and sum(1 <= c <= 4 for c in freq) >= 0.95 * len(freq)
    assert 1 in freq and 2 in freq and 3 in freq and 4 in freq


def test_edge_lengths_present_in_every_kind(corpus):
    _, info, count = corpus
    lens = collections.Counter(len(k) for k in count)
    for n in (1, 2, 3, 4, 5, 6) + tc.EDGE_LENGTHS:
        assert lens[n] >= 1, n
    for w in info["edges"]:
        assert count.get(w, 0) >= 1, (len(w), w[:20])
    kinds = {len(w): set() for w in info["edges"]}
    for w in info["edges"]:
        kinds[len(w)].add("space" if w.strip(b" \n\t") == b"" else "digits" if w[1:2].isdigit() else "other")
    assert all(len(k) >= 2 for n, k in kinds.items() if n > 1), kinds
    # multi-byte characters across the 8-byte key boundaries (byte 7/8 and 15/16 inside one character)
    across = collections.Counter()
    for k in count:
        s = k.decode("utf-8")
        pos = 0
        for ch in s:
            b = len(ch.encode("utf-8"))
            for edge in (8, 16):
                if b > 1 and pos < edge < pos + b:
                    across[(edge, b)] += 1
            pos += b
    for edge in (8, 16):
        for b in (2, 3, 4):
            assert across[(edge, b)] >= 10, (edge, b, across)
    assert any(b"\x00" in k and len(k) > 15 for k in count) and any(b"\x00" in k and len(k) <= 15 for k in count)


def test_near_twins_and_prefixes_present(corpus):
    _, info, count = corpus
    positions = collections.Counter()
    for a, b in info["twins"]:
        assert a != b and len(a) == len(b) and a in count and b in count
        diff = [i for i in range(len(a)) if a[i] != b[i]]
        assert len(diff) == 1
        positions[("last" if diff[0] == len(a) - 1 else diff[0], _tier(len(a)))] += 1
    for pos in ("last", 8, 15):
        assert positions[(pos, 1 if pos != 15 else 2)] + positions[(pos, 2)] >= 2, positions
    # long twins sharing their first 4 096 bytes, differing in the masked tail of the byte compare: every tail length 1..7
    tails = {len(a) % 8 for a, b in info["twins"] if len(a) > tc.LONG_TWIN_PREFIX and a[:tc.LONG_TWIN_PREFIX] == b[:tc.LONG_TWIN_PREFIX]
             and a[-1] != b[-1]}
    assert tails >= set(range(1, 8)), tails
    assert all(p in count for p in info["prefixes"]) and {_tier(len(p)) for p in info["prefixes"]} == {0, 1, 2}


def test_pretoken_positions_cover_the_count_kernel_steps(corpus):
    """Long pretokens start at every offset modulo 16 (a chunk of the count and lookup kernels) and cross the 512-byte steps."""
    text, _, _ = corpus
    starts = oracle.pretokenize(text) + [len(text)]
    mod16, crossing = set(), 0
    for s, e in zip(starts, starts[1:]):
        if e - s > 15:
            mod16.add(s % 16)
            crossing += (s // 512) != ((e - 1) // 512)
    assert mod16 == set(range(16)) and crossing >= 1000, (sorted(mod16), crossing)


def test_encoder_texts_composition():
    specials = [b"<|endoftext|>"]
    t1, t2, train = tc.encoder_texts(1, specials)
    c1, c2 = tc.encoder_pretokens(t1, specials), tc.encoder_pretokens(t2, specials)
    assert set(c1) <= set(c2)
    for tier in (1, 2):
        old = sum(_tier(len(k)) == tier for k in c1)
        new = sum(_tier(len(k)) == tier for k in c2 if k not in c1)
        assert new >= 2 * old, (tier, old, new)
    assert t1.count(specials[0]) == 300 and t2.count(specials[0]) == 300
    assert len(train) > 100000
