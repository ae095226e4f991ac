"""The capacity paths of the merge loop and of the encoder against the oracle: growth of the merge loop's pair table, the slice sort
and record dealing at small thresholds, and eviction of the encoder's pretoken cache.

At their production sizes these paths need far more text than the oracle can follow (the pair table has at least 2^22 slots and
grows when it is half full; the encoder's cache is dropped above 384 M entries).  The library reads the knobs that lower those limits
once per process, so those cases run in a fresh interpreter and prove from the library's stderr notes that the path really ran:
a case that silently stopped growing or evicting fails.  The merge-loop knobs that are read at every call run in-process."""
import json
import os
import random
import re
import subprocess
import sys
import textwrap

import pytest

import _bootstrap  # noqa: F401
from oracle import oracle
from tests.common import FIXTURES_PATH
from tests.test_gpu_train import WORDS, _adjacency_corpus, _fuzz_corpus, _shared_token_corpus

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EOT = "<|endoftext|>"
GROW_RE = re.compile(r"\[pair table: (\d+) -> (\d+) slots at merge (\d+), (\d+) keys\]")
RESET_RE = re.compile(r"\[encoder cache reset: (\d+) entries \+ up to (\d+) new > (\d+), before batch (\d+) of (\d+)\]")


def _run(code: str, env: dict):
    e = dict(os.environ)
    e.update(env)
    r = subprocess.run([sys.executable, "-c", textwrap.dedent(code)], cwd=ROOT, env=e, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-5000:]
    return r.stdout, r.stderr


def _train(data, vocab_size, specials):
    from models.tokenizer.train import train_bpe_on_bytes
    return train_bpe_on_bytes(data, vocab_size, specials, return_stats=True)


# ---- corpora -------------------------------------------------------------------------------------------------------
def _random_words_corpus(n_unique=6000, n_words=40000):
    rnd = random.Random(77)
    words = ["".join(rnd.choice("abcdefghijklmnopqrstuvwxyz") for _ in range(rnd.randint(2, 9))) for _ in range(n_unique)]
    return " ".join(rnd.choice(words) for _ in range(n_words)).encode()


def _tail_corpus():
    """The fuzz corpus with 400 random words added to its alphabet: 5 708 distinct pairs in all (the 31 words alone give 742, too
    few to fill half of the smallest table), every one of them merged before the table runs empty at merge 5 708, the last ones
    with count 0."""
    rnd = random.Random(5)
    extra = ["".join(rnd.choice("abcdefghijklmnopqrstuvwxyz") for _ in range(rnd.randint(3, 8))) for _ in range(400)]
    return _fuzz_corpus(31, 3000, WORDS + extra)


def _owt(mb):
    from transformer_lm_b200.synth import synth_host
    return synth_host("owt", 4321, mb << 20).tobytes()


# name -> (corpus, vocab size, specials).  Measured on a B200: the first four start at 8 192 .. 16 384 slots and grow once or
# twice; the large random-word corpus (52 K distinct words) starts at 65 536 slots and grows to 2^20 (> 128 K keys).
CORPORA = {
    "random_words": (_random_words_corpus, 2500, []),
    "corpus_en": (lambda: (FIXTURES_PATH / "corpus.en").read_bytes(), 3000, [EOT]),
    "fuzz_tail": (_tail_corpus, 6000, []),                                   # until the pair table runs empty
    "shared_tokens": (lambda: _shared_token_corpus(3, n_words=20000), 256 + 1500, []),   # steps of up to 15 merges sharing tokens
    "random_words_large": (lambda: _random_words_corpus(60000, 400000), 20000, []),
}
# (corpus, per-call knobs).  The last run repeats the second: the same inputs must give the same statistics.
GROWTH_RUNS = [
    ("random_words", {}),
    ("corpus_en", {}),
    ("fuzz_tail", {}),
    ("shared_tokens", {}),
    ("random_words", {"BPE_MERGE_BATCH": "1"}),
    ("random_words_large", {"BPE_MERGE_G": "2"}),
    ("corpus_en", {}),
]
STAT_KEYS = ("n_pairs_final", "log_records", "duplicate_tokens", "sum_live_pairs", "merge_steps", "n_pairs_initial")


def run_growth_cases():
    """(In the fresh interpreter.)  Every run of GROWTH_RUNS against the oracle; one JSON line per run on stdout, a marker line
    before every run on stderr (the library's growth notes of a run follow its marker)."""
    want = {}
    for i, (name, knobs) in enumerate(GROWTH_RUNS):
        make, vocab_size, specials = CORPORA[name]
        data = make()
        if name not in want:
            want[name] = oracle.train_bpe_on_bytes(data, vocab_size, specials)
        print("@@ run %d" % i, file=sys.stderr, flush=True)
        os.environ.update(knobs)
        res = {"run": i}
        try:
            vocab, merges, st = _train(data, vocab_size, specials)
            wv, wm = want[name]
            res["merges_equal"] = merges == wm
            res["vocab_equal"] = vocab == wv
            res["n_merges"] = len(merges)
            res["first_diff"] = next((k for k, (x, y) in enumerate(zip(merges, wm)) if x != y), min(len(merges), len(wm)))
            res.update({k: st[k] for k in STAT_KEYS})
        except Exception as e:                   # noqa: BLE001  (reported, and failed, by the test)
            res["error"] = "%s: %s" % (type(e).__name__, e)
        for k in knobs:
            del os.environ[k]
        print(json.dumps(res), flush=True)
    print("@@ end", file=sys.stderr, flush=True)


GROWTH_CODE = """
    import _bootstrap
    from tests.test_gpu_capacity import run_growth_cases
    run_growth_cases()
"""


@pytest.fixture(scope="module")
def growth():
    """Runs GROWTH_RUNS with a 4 096-slot pair table: [(result, [(old_cap, new_cap, at_merge, keys), ...]) per run]."""
    out, err = _run(GROWTH_CODE, {"BPE_MERGE_PCAP_MIN": "4096", "BPE_MERGE_VERBOSE": "1"})
    results = [json.loads(l) for l in out.splitlines() if l.startswith("{")]
    assert len(results) == len(GROWTH_RUNS), out[-2000:] + err[-3000:]
    parts = re.split(r"@@ run \d+\n", err.split("@@ end")[0])[1:]
    assert len(parts) == len(GROWTH_RUNS), err[-3000:]
    growths = [[tuple(int(x) for x in m) for m in GROW_RE.findall(p)] for p in parts]
    for (name, knobs), r, g in zip(GROWTH_RUNS, results, growths):      # (shown by -s / on failure)
        print(name, knobs, "growths (new size, merge, keys):", [x[1:] for x in g], {k: r.get(k) for k in ("n_merges", "n_pairs_final", "merge_steps")})
    return list(zip(results, growths))


def test_pair_table_growth_matches_oracle(growth):
    for (name, knobs), (r, g) in zip(GROWTH_RUNS, growth):
        label = "%s %s" % (name, knobs)
        assert "error" not in r, (label, r)
        assert r["merges_equal"] and r["vocab_equal"], (label, "first differing merge", r["first_diff"])
        assert r["duplicate_tokens"] == 0, label
        # the path under test really ran: a case that stops growing has stopped testing anything
        assert len(g) >= 1, (label, "the pair table never grew")
        for k, (old, new, at, keys) in enumerate(g):
            assert new == 4 * old and old >= 4096 and at < r["n_merges"] and keys <= r["n_pairs_final"], (label, g)
            assert k == 0 or (old == g[k - 1][1] and at >= g[k - 1][2]), (label, g)
    assert max(len(g) for _, g in growth) >= 2, [len(g) for _, g in growth]
    # the shared-token corpus runs steps of many merges, the BATCH=1 run one merge per step
    by_run = {i: r for i, (r, _) in enumerate(growth)}
    assert by_run[3]["merge_steps"] < by_run[3]["n_merges"] * 3 // 4               # (measured: 1 043 steps for 1 500 merges)
    assert by_run[4]["merge_steps"] == by_run[4]["n_merges"]
    assert by_run[2]["n_merges"] < CORPORA["fuzz_tail"][1] - 256                  # the pair table ran empty
    # a grid of two CTAs: after a growth to 2^20 slots (16 384 blocks) the first step lists more dirty blocks than a CTA's list
    # holds (2 048) and owns more blocks than its shared-memory cache of block maxima (4 096)
    g2 = growth[5][1]
    assert any(new >= (1 << 20) for _, new, _, _ in g2), g2


def test_pair_table_statistics_do_not_depend_on_its_size(growth, monkeypatch):
    """n_pairs_final (distinct keys ever created), log_records and duplicate_tokens of the grown small table equal those of the
    default table, which never grows on these inputs.  merge_steps and sum_live_pairs depend on how merges are batched into
    steps, which the block layout of the table decides: they are compared only between identical runs."""
    assert growth[1][0]["sum_live_pairs"] == growth[6][0]["sum_live_pairs"]
    assert growth[1][0]["merge_steps"] == growth[6][0]["merge_steps"]
    done = {}
    for (name, knobs), (r, _) in zip(GROWTH_RUNS, growth):
        make, vocab_size, specials = CORPORA[name]
        for k, v in knobs.items():
            monkeypatch.setenv(k, v)
        key = (name, tuple(sorted(knobs.items())))
        if key not in done:
            done[key] = _train(make(), vocab_size, specials)[2]
        st = done[key]
        for k in knobs:
            monkeypatch.delenv(k)
        for k in ("n_pairs_final", "log_records", "duplicate_tokens", "n_pairs_initial"):
            assert r[k] == st[k], (name, knobs, k, r[k], st[k])
        assert st["duplicate_tokens"] == 0
    # two identical runs at the default size
    make, vocab_size, specials = CORPORA["corpus_en"]
    again = _train(make(), vocab_size, specials)[2]
    first = done[("corpus_en", ())]
    assert (again["sum_live_pairs"], again["merge_steps"]) == (first["sum_live_pairs"], first["merge_steps"])


# ---- slice sort and record dealing (read at every call) ------------------------------------------------------------
@pytest.mark.parametrize("knobs", [{"BPE_MERGE_SORTMIN": "64"}, {"BPE_MERGE_SORTMIN": "512"}, {"BPE_MERGE_MINREC": "32"},
                                   {"BPE_MERGE_SORTMIN": "64", "BPE_MERGE_SORTPOOL": "20000"}],
                         ids=["sortmin64", "sortmin512", "minrec32", "sortmin64-pool-runs-out"])
def test_slice_sort_and_dealing_knobs_match_oracle(monkeypatch, knobs):
    """SORTMIN=64 / 512 sorts small slices into 16..64 buckets (the default sorts only slices of >= 65 536 records); MINREC=32 deals
    whole warps of records.  The default pool of bucket offsets does not run out on these inputs (SORTMIN=64 on the 12 MB corpus
    uses 43 958 of its 526 459 entries for 38 slices); a pool of 20 000 entries does: on a B200 it held 10 of those 38 slices,
    and the later ones stayed unsorted."""
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    cases = [(_owt(12), 600, [EOT]), ((FIXTURES_PATH / "corpus.en").read_bytes(), 1500, [EOT])]
    cases += [(_adjacency_corpus(seed, n_pairs=6 + seed % 7), 256 + 60, []) for seed in range(4)]
    for i, (data, vocab_size, specials) in enumerate(cases):
        want = oracle.train_bpe_on_bytes(data, vocab_size, specials)
        vocab, merges, st = _train(data, vocab_size, specials)
        assert merges == want[1] and vocab == want[0], (knobs, i)


# ---- eviction of the encoder's pretoken cache ----------------------------------------------------------------------
ENCODE_CODE = """
    import sys
    import numpy as np
    import _bootstrap
    from oracle import oracle
    from transformer_lm_b200.synth import synth_host
    from models.tokenizer.train import train_bpe_on_bytes
    from tests.adapters import get_tokenizer
    EOT, PAD = "<|endoftext|>", "<|pad|>"                      # PAD is not in the vocab: it gets the next id (SURVEY A-12)
    def mark(s):
        print("@@ " + s, file=sys.stderr, flush=True)
    vocab, merges = train_bpe_on_bytes(synth_host("owt", 4321, 32 << 20), 3000, [EOT])
    # one more merge whose product is not in the vocab: a pretoken " \\x01\\x02" raises KeyError(b"\\x01\\x02")
    merges = list(merges) + [(b"\\x01", b"\\x02")]
    tok = get_tokenizer(dict(vocab), list(merges), [EOT, PAD])
    otok = oracle.OracleTokenizer(dict(vocab), list(merges), [EOT, PAD])
    text = synth_host("owt", 4322, 6 << 20).tobytes()
    text = text[: text.rfind(EOT.encode())]
    docs = text.split(EOT.encode())
    text = EOT.encode().join(d + PAD.encode() if i % 7 == 3 else d for i, d in enumerate(docs))
    want = otok.encode_bytes(text)
    mark("call 1")
    got = tok.encode_to_numpy(text, np.int32)
    assert len(got) == len(want) and bool((got == want).all()), "int32"
    mark("call 2")                                             # the same tokenizer: its cache is full from call 1
    got16 = tok.encode_to_numpy(text, np.uint16)
    assert len(got16) == len(want) and bool((got16 == want).all()), "uint16"
    mark("batch")
    dtexts = text.decode("utf-8").split(EOT)
    gotb = tok.encode_batch(dtexts)
    assert gotb == [otok.encode(d) for d in dtexts], "encode_batch"
    mark("keyerror")
    bad = text + b" \\x01\\x02 tail"
    try:
        tok.encode_to_numpy(bad, np.int32)
        raise SystemExit("no KeyError")
    except KeyError as e:
        try:
            otok.encode_bytes(bad)
            raise SystemExit("the oracle raised no KeyError")
        except KeyError as e2:
            assert e.args == e2.args == (b"\\x01\\x02",), (e.args, e2.args)
    mark("after")
    assert bool((tok.encode_to_numpy(text, np.int32) == want).all()), "after the KeyError"
    mark("end")
    print("encode ok", len(want), len(dtexts))
"""


@pytest.mark.parametrize("limit,hot", [("200000", False), ("200000", True), ("20000", False)],
                         ids=["evict", "evict-hot-table", "batch-over-limit"])
def test_encoder_cache_eviction_matches_oracle(limit, hot):
    """512 KB batches hold ~115 000 pretokens, ~42 000 of them distinct.  Limit 200 000: the cache is dropped every few batches,
    within a call and at the start of the next one.  Limit 20 000: every batch alone holds more than the limit, so the cache is
    dropped before every batch but the first of a fresh tokenizer (it holds only the specials then) and grows past the limit."""
    env = {"BPE_ENC_BATCH_KB": "512", "BPE_ENC_CACHE_MAX": limit, "BPE_ENC_PROFILE": "1"}
    env.update({"BPE_ENC_HOT_MIN": "50000", "BPE_ENC_HOT_TEST": "1"} if hot else {"BPE_ENC_HOT_MIN": str(1 << 40)})
    out, err = _run(ENCODE_CODE, env)
    assert "encode ok" in out
    phases = dict(re.findall(r"@@ (\w+(?: \d)?)\n(.*?)(?=@@ )", err, re.S))
    resets = {p: [tuple(int(x) for x in m) for m in RESET_RE.findall(s)] for p, s in phases.items()}
    print({p: len(v) for p, v in resets.items()})
    for p in ("call 1", "call 2", "batch", "keyerror"):
        assert len(resets[p]) >= 2, (p, resets[p], err[-3000:])
        for entries, bound, lim, b, n in resets[p]:
            assert lim == int(limit) and entries + bound > lim and entries > 2 and 0 <= b < n
    # across calls: the cache left by call 1 is dropped before the first batch of call 2.  (The KeyError's pretoken is at the end
    # of the text, in the last batch: after every eviction of its call.)
    assert resets["call 2"][0][3] == 0
    if limit == "20000":
        # a fresh tokenizer's cache holds only the specials: no reset before batch 0, one before every later batch, and the cache
        # grows past the limit in every batch
        n = resets["call 1"][0][4]
        assert [x[3] for x in resets["call 1"]] == list(range(1, n))
        assert all(entries > int(limit) for entries, *_ in resets["call 1"])
    else:
        assert resets["call 1"][0][3] > 1                    # several batches are cached before the first eviction
        assert len(resets["call 1"]) < resets["call 1"][0][4] - 1
    hot_lines = [m.start() for m in re.finditer(r"\[encoder hot table:", err)]
    reset_lines = [m.start() for m in re.finditer(r"\[encoder cache reset:", err)]
    if hot:
        # built, dropped by an eviction, and built again after it
        assert hot_lines and hot_lines[0] < reset_lines[0] and any(h > reset_lines[0] for h in hot_lines), err[-3000:]
    else:
        assert not hot_lines
