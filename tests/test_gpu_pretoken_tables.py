"""The pretoken tables of hashtab.cuh tested directly against the oracle: the count table of training (bpe_count_export) word for word,
and the encoder's cache through the number of entries every call adds (last_stats["cache_new_unique"]).

The merges of training and the ids of encoding hide most faults of a hash table: a long word counted 3 times instead of 4, or stored
twice with its count split, moves no merge; a cache entry that a rehash lost is claimed again and recomputed, and the ids stay right.
So the count table is compared with oracle.count_pretokens exactly, and the cache's new entries with the number of distinct pretokens
a call brings that the cache did not hold.  The text is the tier corpus (tests/helpers/tier_corpus.py): tens of thousands of distinct
pretokens in each of the three tiers, every tier and kernel boundary length, near-twins that differ in one byte.

Table growth with entries in it only happens between batches or calls, so the cases that must prove it ran go through a fresh
interpreter with the profile knobs set and read the library's growth notes ("[count tables grow: ...]", "[encoder cache grow: ...]")
from stderr, like test_gpu_capacity.py does with its pair-table notes: a case whose growth stopped happening fails."""
import os
import re
import subprocess
import sys
import textwrap

import numpy as np
import pytest

import _bootstrap  # noqa: F401
from oracle import oracle
from tests.helpers import tier_corpus as tc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAX_TOKEN_LEN = (1 << 24) - 2                   # hashtab.cuh: the length field of a long key holds up to 2^24 - 1
GROW_RE = r"\[%s grow: short (\d+) -> (\d+) slots \((\d+) entries\), medium (\d+) -> (\d+) \((\d+)\), long (\d+) -> (\d+) \((\d+)\)\]"
COUNT_GROW_RE = re.compile(GROW_RE % "count tables")
ENC_GROW_RE = re.compile(GROW_RE % "encoder cache")


def _run(code: str, env: dict):
    e = dict(os.environ)
    e.update(env)
    r = subprocess.run([sys.executable, "-c", textwrap.dedent(code)], cwd=ROOT, env=e, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-5000:]
    return r.stdout, r.stderr


def _growths(err: str, rx):
    """[(tier, old, new, entries)] of every growth note on stderr, one entry per tier that grew."""
    out = []
    for m in rx.findall(err):
        v = [int(x) for x in m]
        for k, tier in enumerate(("short", "medium", "long")):
            old, new, entries = v[3 * k: 3 * k + 3]
            if new > old:
                out.append((tier, old, new, entries))
    return out


# ---- count table ---------------------------------------------------------------------------------------------------------
def export_dict(counter) -> dict:
    """bpe_count_export as {word: count}; every word once, every count positive."""
    blob, offs, counts = counter.export()
    b = blob.cpu().numpy().tobytes()
    o = offs.cpu().numpy()
    c = counts.cpu().numpy()
    words = [b[int(o[i]):int(o[i + 1])] for i in range(len(c))]
    out = dict(zip(words, c.tolist()))
    assert len(out) == len(words), "a word appears %d times in the export" % (len(words) - len(out) + 1)
    assert len(c) == 0 or int(c.min()) > 0, "a zero count in the export"
    assert int(o[len(c)]) == len(b)
    return out


def diff(got: dict, want: dict) -> str:
    """'' when equal, else a short account of the differences (by length)."""
    if got == want:
        return ""
    missing = [k for k in want if k not in got]
    extra = [k for k in got if k not in want]
    wrong = [k for k in want if k in got and got[k] != want[k]]
    show = lambda ks: [(len(k), k[:24], want.get(k), got.get(k)) for k in ks[:5]]       # noqa: E731
    return "missing %d %s, extra %d %s, wrong count %d %s" % (len(missing), show(missing), len(extra), show(extra), len(wrong), show(wrong))


def add_in_shards(counter, data: bytes, n_shards: int, halo: int = 64 << 10):
    """Every shard of data cut as the ranks of sharded training cut it (sharded.plan_shard, with halos), all into ONE counter."""
    from transformer_lm_b200 import sharded
    peek = lambda lo, hi: data[lo:hi]      # noqa: E731
    for r in range(n_shards):
        lo, hi, rlo, rhi = sharded.plan_shard(peek, len(data), r, n_shards, halo)
        st = counter.add(data[rlo:rhi], lo - rlo, hi - rlo, rlo == 0, rhi == len(data))
        assert st is None, (r, st)


def add_all(counter, data: bytes):
    assert counter.add(data, 0, len(data), True, True) is None


def add_sum(*dicts) -> dict:
    out = {}
    for d in dicts:
        for k, v in d.items():
            out[k] = out.get(k, 0) + v
    return out


@pytest.fixture(scope="module")
def tier():
    text, info = tc.tier_corpus(0)
    return text, info, oracle.count_pretokens(text, [])


def _counter():
    from transformer_lm_b200 import sharded
    return sharded.DeviceCounter()


def test_count_export_equals_oracle(tier):
    text, _, want = tier
    c = _counter()
    add_all(c, text)
    got = export_dict(c)
    assert not diff(got, want), diff(got, want)


@pytest.mark.parametrize("n_shards", [3, 16])
def test_count_many_adds_on_one_counter(tier, n_shards):
    """Shards of the text into one counter: growth with entries in every tier between the adds, the long words of every add re-homed
    from the text arena to the pool, and the long words of a later shard matched against those pool copies."""
    text, _, want = tier
    c = _counter()
    add_in_shards(c, text, n_shards)
    got = export_dict(c)
    assert not diff(got, want), diff(got, want)


def _blob(words, counts):
    import torch
    blob = b"".join(words)
    offs = np.zeros(len(words) + 1, dtype=np.int64)
    np.cumsum([len(w) for w in words], out=offs[1:])
    dev = torch.device("cuda")
    return (torch.frombuffer(bytearray(blob), dtype=torch.uint8).to(dev), torch.from_numpy(offs).to(dev),
            torch.tensor(counts, dtype=torch.int64, device=dev))


def test_count_import_adds_exactly(tier):
    text, info, want_a = tier
    rnd = __import__("random").Random(9)
    # text B shares words with A in every tier (a third of A's words) and has its own
    shared = [w for w in info["words"] if rnd.random() < 0.33]
    text_b = tc.render(rnd, shared + tc.distinct_words(rnd, 5000, 5000, 5000, avoid=frozenset(info["words"])), tc.FREQUENT, 50)
    want_b = oracle.count_pretokens(text_b, [])
    assert {min(len(k) // 8, 2) for k in want_b if k in want_a} == {0, 1, 2}        # shared words in every tier
    # (the counters of one context share its table: each is used up before the next one begins; the exports are torch tensors)
    a = _counter()
    add_all(a, text)
    ea = a.export()
    b = _counter()
    add_all(b, text_b)
    eb = b.export()
    # A, B and A again into a fresh counter: 2 A + B
    c = _counter()
    for e in (ea, eb, ea):
        c.import_(*e)
    got = export_dict(c)
    want = add_sum(want_a, want_a, want_b)
    assert not diff(got, want), diff(got, want)
    # a counted text, then the export of another one
    d = _counter()
    add_all(d, text_b)
    d.import_(*ea)
    got = export_dict(d)
    want = add_sum(want_a, want_b)
    assert not diff(got, want), diff(got, want)


@pytest.mark.parametrize("last_len", [15, 16, 17])
def test_count_import_blob_ending_in_a_tier_edge_word(tier, last_len):
    """A blob whose last word ends the blob at 15, 16 or 17 bytes: its key loads read up to 15 bytes past the end of the copy in the
    pool.  Imported twice, after text that holds the same word."""
    rnd = __import__("random").Random(last_len)
    last = tc.ascii_word(rnd, last_len)
    words = [tc.ascii_word(rnd, n) for n in (3, 9, 20, 40)] + [last]
    counts = [5, 6, 7, 8, 9]
    c = _counter()
    add_all(c, last + b" x" + last)
    c.import_(*_blob(words, counts))
    c.import_(*_blob(words, counts))
    got = export_dict(c)
    want = add_sum({last: 2, b" x": 1}, dict(zip(words, counts)), dict(zip(words, counts)))
    assert not diff(got, want), diff(got, want)


def test_count_max_token_len():
    """A pretoken of exactly MAX_TOKEN_LEN bytes is counted once with its bytes intact; one byte more is refused with the library's
    'unsupported' error, through add and through import, instead of being counted wrong."""
    from transformer_lm_b200 import _lib
    rnd = __import__("random").Random(5)
    big = bytearray(b" " + bytes(rnd.choice(b"abcdefghij") for _ in range(1000)) * (MAX_TOKEN_LEN // 1000 + 1))[:MAX_TOKEN_LEN]
    big = bytes(big)
    assert len(big) == MAX_TOKEN_LEN and oracle.pretokenize(b" x" + big[:100000] + b" y") == [0, 2, 100002]
    c = _counter()
    add_all(c, b" x" + big + b" y" + big)
    got = export_dict(c)
    assert got == {b" x": 1, b" y": 1, big: 2}
    with pytest.raises(_lib.BpeError) as e:
        add_all(_counter(), b" x" + big + b"z y")
    assert e.value.code == _lib.ERR_UNSUPPORTED
    # import: exactly MAX_TOKEN_LEN is taken, one byte more is refused
    c = _counter()
    c.import_(*_blob([b" x", big], [3, 4]))
    assert export_dict(c) == {b" x": 3, big: 4}
    with pytest.raises(_lib.BpeError) as e:
        _counter().import_(*_blob([b" x", big + b"z"], [3, 4]))
    assert e.value.code == _lib.ERR_UNSUPPORTED


# ---- count table in a fresh interpreter: small batches, hot table --------------------------------------------------------------
COUNT_CODE = """
    import _bootstrap
    from oracle import oracle
    from tests.helpers import tier_corpus as tc
    from tests.test_gpu_pretoken_tables import _counter, add_all, add_in_shards, diff, export_dict
    text, _ = tc.tier_corpus(0)
    want = oracle.count_pretokens(text, [])
    c = _counter()
    add_all(c, text)
    d = diff(export_dict(c), want)
    assert not d, "one add: " + d
    c = _counter()
    add_in_shards(c, text, 16)
    d = diff(export_dict(c), want)
    assert not d, "16 adds: " + d
    print("count ok", len(want))
"""


@pytest.mark.parametrize("knobs", [{}, {"BPE_COUNT_BATCH_KB": "64"},
                                   {"BPE_COUNT_BATCH_KB": "256", "BPE_COUNT_HOT_TEST": "1", "BPE_COUNT_HOT_AFTER": "20000"}],
                         ids=["default", "batch64k", "hot-table"])
def test_count_growth_and_hot_table_match_oracle(knobs):
    env = dict(knobs, BPE_COUNT_PROFILE="1")
    out, err = _run(COUNT_CODE, env)
    assert "count ok" in out
    g = _growths(err, COUNT_GROW_RE)
    print(knobs, "growths (tier, old, new, entries):", g)
    if not knobs:
        # 16 shards of ~280 KB: every tier grows while it holds the words of the shards before
        for tier in ("short", "medium", "long"):
            assert any(t == tier and entries > 1000 for t, _, _, entries in g), (tier, g)
    elif "BPE_COUNT_HOT_TEST" not in knobs:
        # 64 KB batches: the long table grows from its first 2^14 slots holding > 10 000 words, the medium one with words in it
        assert any(t == "long" and old == 1 << 14 and entries > 10000 for t, old, _, entries in g), g
        assert any(t == "medium" and entries > 1000 for t, _, _, entries in g), g
    else:
        # built after 20 000 pretokens and rebuilt twice (4x, 16x), in each of the two adds: every rebuild flushes the counts first
        assert err.count("[hot table:") >= 4, err[-3000:]


# ---- encoder cache -----------------------------------------------------------------------------------------------------------
# specials in every tier: 3 bytes, <|endoftext|> (13) and a twin that differs from it in the masked tail of the byte compare, 15 and
# 16 bytes, and two of 41 bytes that differ only in the last byte (their bytes live in the key pool)
SPECIALS = ["<|>", "<|endoftext|>", "<|endoftexu|>", "<|" + "a" * 11 + "|>", "<|" + "b" * 12 + "|>",
            "<|" + "c" * 37 + "|>", "<|" + "c" * 37 + "|)"]

ENCODE_CODE = """
    import sys
    import numpy as np
    import _bootstrap
    from oracle import oracle
    from tests.helpers import tier_corpus as tc
    from tests.adapters import get_tokenizer
    from tests.test_gpu_pretoken_tables import SPECIALS
    from models.tokenizer.train import train_bpe_on_bytes
    sp = [s.encode() for s in SPECIALS]
    assert sorted(len(s) for s in sp) == [3, 13, 13, 15, 16, 41, 41]
    t1, t2, train = tc.encoder_texts(1, sp)
    vocab, merges = train_bpe_on_bytes(train, 2000, SPECIALS)
    assert any(len(a + b) >= 6 for a, b in merges)
    tok = get_tokenizer(dict(vocab), list(merges), SPECIALS)
    otok = oracle.OracleTokenizer(dict(vocab), list(merges), SPECIALS)
    p1, p2 = tc.encoder_pretokens(t1, sp), tc.encoder_pretokens(t2, sp)
    assert p1 <= p2
    def step(label, data, want_new):
        print("@@ " + label, file=sys.stderr, flush=True)
        got = tok.encode_to_numpy(data, np.int32)
        want = otok.encode_bytes(data)
        assert len(got) == len(want) and bool((got == want).all()), label + ": ids differ from the oracle"
        new = tok.last_stats["cache_new_unique"]
        assert new == want_new, (label, "new cache entries", new, "expected", want_new)
        print(label, "ok", len(want), new, flush=True)
    # every distinct pretoken of a call that the cache lacks is claimed exactly once; the specials are in the cache from the start
    step("t1 fresh", t1, len(p1))
    step("t1 again", t1, 0)
    step("t2", t2, len(p2 - p1))
    step("t1 third", t1, 0)
    step("t2 again", t2, 0)
    print("@@ batch", file=sys.stderr, flush=True)
    docs = t2.decode("utf-8").split(SPECIALS[1])
    assert len(docs) > 100
    got = tok.encode_batch(docs)
    assert tok.last_stats["cache_new_unique"] == 0, tok.last_stats
    assert got == [otok.encode(d) for d in docs], "encode_batch"
    # the same special listed twice: one entry, the oracle's id
    tok2 = get_tokenizer(dict(vocab), list(merges), SPECIALS + [SPECIALS[5], SPECIALS[1]])
    otok2 = oracle.OracleTokenizer(dict(vocab), list(merges), SPECIALS + [SPECIALS[5], SPECIALS[1]])
    small = t1[:200000]
    assert tok2.encode_to_numpy(small, np.int32).tolist() == otok2.encode_bytes(small).tolist()
    print("@@ end", file=sys.stderr, flush=True)
    print("encode ok")
"""


@pytest.mark.parametrize("knobs", [{}, {"BPE_ENC_BATCH_KB": "64"},
                                   {"BPE_ENC_BATCH_KB": "64", "BPE_ENC_HOT_MIN": "2000", "BPE_ENC_HOT_TEST": "1"}],
                         ids=["default", "batch64k", "hot-table"])
def test_encoder_cache_entries_match_oracle(knobs):
    env = dict(knobs, BPE_ENC_PROFILE="1")
    out, err = _run(ENCODE_CODE, env)
    assert "encode ok" in out, out[-2000:]
    assert "[encoder cache reset:" not in err
    phases = dict(re.findall(r"@@ ([\w ]+)\n(.*?)(?=@@ )", err, re.S))
    g = {p: _growths(s, ENC_GROW_RE) for p, s in phases.items()}
    print(knobs, "growths (tier, old, new, entries):", g)
    if not knobs:
        # t2's bound outgrows the tables t1 left: every tier grows with t1's entries in it (long keys already in the pool)
        for tier in ("short", "medium", "long"):
            assert any(t == tier and entries > 0 for t, _, _, entries in g["t2"]), (tier, g)
        assert any(t == "long" and entries > 5000 for t, _, _, entries in g["t2"]), g
    else:
        # 64 KB batches: growth between the batches of one call; the long table from its first 2^14 slots with > 10 000 entries
        assert any(t == "long" and old == 1 << 14 and entries > 10000 for t, old, _, entries in g["t2"]), g
        assert any(t == "medium" and entries > 1000 for t, _, _, entries in g["t2"]), g
    assert ("[encoder hot table:" in err) == ("BPE_ENC_HOT_TEST" in knobs), err[-3000:]
