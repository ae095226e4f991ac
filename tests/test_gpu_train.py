"""GPU parity of BPE training (bpe_train through the reference-compatible adapter) against the reference's
golden snapshot, golden vectors generated from the reference, and the CPU oracle on seeded corpora."""
import random
import time

import pytest

import _bootstrap  # noqa: F401
from oracle import oracle
from tests.adapters import run_train_bpe
from tests.common import FIXTURES_PATH, load_golden, load_reference_train_snapshot

pytestmark = pytest.mark.gpu


def _train_bytes(data, vocab_size, specials, **kw):
    from models.tokenizer.train import train_bpe_on_bytes
    return train_bpe_on_bytes(data, vocab_size, specials, **kw)


def test_train_bpe_reference_snapshot():
    """The reference's golden test (tests/test_train_bpe.py:28-65): corpus.en, vocab 500."""
    vocab, merges = run_train_bpe(FIXTURES_PATH / "corpus.en", 500, ["<|endoftext|>"])
    ref_vocab, ref_merges = load_reference_train_snapshot()
    assert merges == ref_merges
    assert set(vocab.keys()) == set(ref_vocab.keys())
    assert set(vocab.values()) == set(ref_vocab.values())


def test_train_bpe_speed():
    """tests/test_train_bpe.py:9-25 of the reference: < 1.5 s (CUDA context already created by earlier tests
    or not -- the budget includes it)."""
    t0 = time.time()
    run_train_bpe(FIXTURES_PATH / "corpus.en", 500, ["<|endoftext|>"])
    assert time.time() - t0 < 1.5


def _golden_input(case):
    src = case["source"]
    if src.startswith("fixture:"):
        return (FIXTURES_PATH / src.split(":", 1)[1]).read_bytes()
    return bytes.fromhex(case["input_hex"])


@pytest.mark.parametrize("name", sorted(load_golden("train_golden.json").keys()))
def test_train_golden(name):
    case = load_golden("train_golden.json")[name]
    data = _golden_input(case)
    if "error" in case:
        with pytest.raises(UnicodeDecodeError):
            _train_bytes(data, case["vocab_size"], case["special_tokens"])
        return
    vocab, merges = _train_bytes(data, case["vocab_size"], case["special_tokens"])
    assert [[a.hex(), b.hex()] for a, b in merges] == case["merges"]
    assert {str(k): v.hex() for k, v in vocab.items()} == case["vocab"]


def _fuzz_corpus(seed, n_words, alphabet_words):
    r = random.Random(seed)
    out = []
    for _ in range(n_words):
        out.append(r.choice(alphabet_words))
        out.append(r.choice([" ", " ", " ", "\n", "  ", ", ", ". ", ""]))
    return "".join(out).encode("utf-8")


WORDS = ["the", "there", "then", "other", "a", "an", "and", "band", "hand", "it's", "don't", "we'll", "naïve", "日本", "日本語",
         "🙃", "🙃🙃", "1", "12", "123", "2024", "x_y", "--", "----", "http://a.b/c", "aaaa", "aaa", "aa", "abab", "ababab", "Zürich"]


@pytest.mark.parametrize("seed,n_words,vocab_size", [(1, 50, 400), (2, 500, 600), (3, 5000, 900), (4, 20000, 1500), (5, 12, 2000)])
def test_train_differential_vs_oracle(seed, n_words, vocab_size):
    data = _fuzz_corpus(seed, n_words, WORDS)
    want = oracle.train_bpe_on_bytes(data, vocab_size, ["<|endoftext|>"])
    got = _train_bytes(data, vocab_size, ["<|endoftext|>"])
    assert got[1] == want[1]
    assert got[0] == want[0]


def test_train_corpus_vocab_3000_vs_oracle():
    data = (FIXTURES_PATH / "corpus.en").read_bytes()
    want = oracle.train_bpe_on_bytes(data, 3000, ["<|endoftext|>"])
    got = _train_bytes(data, 3000, ["<|endoftext|>"])
    assert got[1] == want[1]
    assert got[0] == want[0]


def test_train_is_deterministic():
    data = _fuzz_corpus(7, 8000, WORDS)
    a = _train_bytes(data, 1200, [])
    b = _train_bytes(data, 1200, [])
    assert a == b


def test_train_long_pretokens_and_crlf():
    data = (b"x" * 5000 + b" " + b"ab" * 3000 + b"\r\n" + b"x" * 5000 + b"\r" + b"ab" * 3000 + b" 0123456789abcdef 0123456789abcdef ") * 3
    want = oracle.train_bpe_on_bytes(data, 400, [])
    got = _train_bytes(data, 400, [])
    assert got == want


def test_train_stats_are_reported():
    data = (FIXTURES_PATH / "corpus.en").read_bytes()
    vocab, merges, stats = _train_bytes(data, 500, ["<|endoftext|>"], return_stats=True)
    assert stats["n_bytes"] == len(data.replace(b"\r\n", b"\n"))
    assert stats["n_pretokens"] == len(oracle.pretokenize(data))
    assert len(merges) == 243 and stats["duplicate_tokens"] == 0


# ---- sharded counting through the C ABI (bpe_count_*): the per-GPU half of multi-GPU training ----------------
def _sharded_train_one_gpu(data, n_shards, vocab_size, specials, halo=64 << 10):
    """Emulates n_shards ranks on one GPU: every shard is counted into a fresh table and exported; all tables are
    then imported into one and the merge loop runs on the sum."""
    import numpy as np
    import torch
    from transformer_lm_b200 import sharded
    peek = lambda lo, hi: data[lo:hi]      # noqa: E731
    tables = []
    for r in range(n_shards):
        h = halo
        while True:
            c = sharded.DeviceCounter()
            lo, hi, rlo, rhi = sharded.plan_shard(peek, len(data), r, n_shards, h)
            st = c.add(data[rlo:rhi], lo - rlo, hi - rlo, rlo == 0, rhi == len(data))
            if st is not None and st[0] == "halo":
                h *= 16
                continue
            assert st is None, st
            break
        blob, offs, counts = c.export()
        tables.append((blob.clone(), offs.clone(), counts.clone(), c.pair_table(specials)))
    c = sharded.DeviceCounter()
    for blob, offs, counts, _ in tables:
        c.import_(blob, offs, counts)
    total_pairs = sum(t[3] for t in tables)
    assert bool((c.pair_table(specials) == total_pairs).all())      # linearity of the byte-pair table
    return c.finish(vocab_size, specials)


@pytest.mark.parametrize("n_shards", [2, 3, 8])
def test_sharded_count_then_merge_equals_single_shot(n_shards):
    data = (FIXTURES_PATH / "corpus.en").read_bytes()
    want = _train_bytes(data, 700, ["<|endoftext|>"])
    got = _sharded_train_one_gpu(data, n_shards, 700, ["<|endoftext|>"])
    assert got[1] == want[1] and got[0] == want[0]


def test_sharded_count_small_halo_and_unicode():
    data = _fuzz_corpus(21, 30000, WORDS + ["x" * 200, " " * 100, "\n\n\n"])
    want = oracle.train_bpe_on_bytes(data, 800, [])
    got = _sharded_train_one_gpu(data, 5, 800, [], halo=32)
    assert got[1] == want[1] and got[0] == want[0]


def test_shard_reports_only_owned_utf8_errors_and_refuses_cr():
    from transformer_lm_b200 import sharded
    data = b"hello world, this is a shard of text " * 10
    bad = bytearray(data)
    bad[5] = 0xFF                                   # in the left halo
    c = sharded.DeviceCounter()
    assert c.add(bytes(bad), 64, 300, False, False) is None
    c = sharded.DeviceCounter()
    bad[100] = 0xFF
    assert c.add(bytes(bad), 64, 300, False, False) == ("utf8", 100)
    c = sharded.DeviceCounter()
    assert c.add(data[:200] + b"\r\n" + data[200:], 64, 300, False, False) == ("newline", 0)
    c = sharded.DeviceCounter()
    long_tail = b"x" * 90 + b" " + b"a" * 309                           # " aaa..." starts at 90 (owned) and never ends
    assert c.add(long_tail, 64, 300, False, False) == ("halo", 0)
    c = sharded.DeviceCounter()
    assert c.add(b"a" * 400, 64, 300, False, False) is None             # its only pretoken starts at 0: not owned
    c = sharded.DeviceCounter()
    assert c.add(long_tail, 0, 400, True, True) is None


# ---- several merges per grid step (csrc/merge.cuh): the batches must be exactly the reference's sequence ----------------
def _adjacency_corpus(seed, n_words=400, n_pairs=10):
    """Words glued from letter pairs with distinct, well separated frequencies: the top pairs share no token, so a step
    takes several of them, and their occurrences sit next to each other in every order (abcd, cdab, ababcd, ...)."""
    rnd = random.Random(seed)
    letters = "abcdefghijklmnopqrstuvwxyz"[: 2 * n_pairs]
    pairs = [letters[2 * i: 2 * i + 2] for i in range(n_pairs)]
    weights = [2.0 ** -(i / 2) for i in range(n_pairs)]
    out = []
    for _ in range(n_words):
        pieces = []
        for _ in range(rnd.randint(1, 6)):
            pieces.append(rnd.choices(pairs, weights)[0] if rnd.random() < 0.85 else rnd.choice(letters))
        out.extend(["".join(pieces)] * rnd.randint(1, 40))
    rnd.shuffle(out)
    return " ".join(out).encode()


@pytest.mark.parametrize("grid", [None, "3", "17", "148"])
def test_multi_merge_steps_match_oracle_on_adjacent_sites(monkeypatch, grid):
    if grid:
        monkeypatch.setenv("BPE_MERGE_G", grid)
    batched = 0
    for seed in range(12):
        data = _adjacency_corpus(seed, n_pairs=6 + seed % 7)
        want = oracle.train_bpe_on_bytes(data, 256 + 60, [])
        vocab, merges, st = _train_bytes(data, 256 + 60, [], return_stats=True)
        assert merges == want[1] and vocab == want[0], seed
        batched += st["merge_steps"] < len(merges)
    assert batched >= 6                                   # the multi-merge path really ran


def _shared_token_corpus(seed, n_words=500):
    """Words over a small alphabet with skewed letter frequencies: the top pairs SHARE tokens ((a,b), (a,c), (c,b), ...), sit next
    to each other in every order and overlap (aba, abab, aab): what the relaxed batching rule admits into one step."""
    rnd = random.Random(seed)
    alpha = "abcdefg"[: 4 + seed % 4]
    weights = [1.0 / (k + 1) for k in range(len(alpha))]
    out = []
    for _ in range(n_words):
        w = "".join(rnd.choices(alpha, weights, k=rnd.randint(2, 9)))
        out.extend([w] * rnd.randint(1, 30 + 13 * (seed % 5)))
    rnd.shuffle(out)
    return " ".join(out).encode()


@pytest.mark.parametrize("grid", [None, "5", "148"])
def test_multi_merge_steps_with_shared_tokens_match_oracle(monkeypatch, grid):
    if grid:
        monkeypatch.setenv("BPE_MERGE_G", grid)
    batched = 0
    for seed in range(24):
        data = _shared_token_corpus(seed)
        want = oracle.train_bpe_on_bytes(data, 256 + 80, [])
        vocab, merges, st = _train_bytes(data, 256 + 80, [], return_stats=True)
        assert merges == want[1] and vocab == want[0], seed
        batched += st["merge_steps"] < len(merges)
    assert batched >= 8


@pytest.mark.parametrize("batch", ["1", "2", "5"])
def test_merges_do_not_depend_on_the_batch_limit(monkeypatch, batch):
    from transformer_lm_b200.synth import synth_host
    data = synth_host("owt", 4321, 48 << 20)
    vocab, merges, st = _train_bytes(data, 3000, ["<|endoftext|>"], return_stats=True)
    assert st["merge_steps"] < len(merges) // 2           # default: up to 8 merges per step
    monkeypatch.setenv("BPE_MERGE_BATCH", batch)
    v2, m2, st2 = _train_bytes(data, 3000, ["<|endoftext|>"], return_stats=True)
    assert m2 == merges and v2 == vocab
    if batch == "1":
        assert st2["merge_steps"] == len(merges)
    # deep into the tie-heavy tail and the zero-count exhaustion phase, against the oracle
    small = (FIXTURES_PATH / "corpus.en").read_bytes()
    assert _train_bytes(small, 1500, ["<|endoftext|>"]) == oracle.train_bpe_on_bytes(small, 1500, ["<|endoftext|>"])
    tiny = b"aaaa abab aaaa"
    assert _train_bytes(tiny, 300, []) == oracle.train_bpe_on_bytes(tiny, 300, [])
    fz = _fuzz_corpus(31, 3000, WORDS)
    assert _train_bytes(fz, 5000, []) == oracle.train_bpe_on_bytes(fz, 5000, [])


# ---- big host inputs: chunked, double-buffered upload (bpe_train) must equal the one-piece device path -----------------
def test_pipelined_host_training_equals_one_piece():
    import numpy as np
    import torch
    from transformer_lm_b200.synth import synth_host
    n = 600 << 20
    host = synth_host("owt", 4321, n)
    got = _train_bytes(host, 1500, ["<|endoftext|>"])                       # host path: 3 chunks with halos
    dev = torch.from_numpy(host).cuda()
    want = _train_bytes(None, 1500, ["<|endoftext|>"], device_ptr=dev.data_ptr(), n_bytes=n)
    assert got[1] == want[1] and got[0] == want[0]
    # a carriage return anywhere sends the whole input down the one-piece path (newline translation shifts offsets)
    host2 = host[: 200 << 20].copy()
    host2[150 << 20] = 0x0D
    dev2 = torch.from_numpy(host2).cuda()
    assert _train_bytes(host2, 600, []) == _train_bytes(None, 600, [], device_ptr=dev2.data_ptr(), n_bytes=host2.size)
    # invalid UTF-8 in a later chunk: same exception and offset as CPython
    host3 = host[: 400 << 20].copy()
    host3[(300 << 20) + 12345] = 0xFF
    with pytest.raises(UnicodeDecodeError) as ei:
        _train_bytes(host3, 600, [])
    try:
        host3.tobytes().decode("utf-8")
    except UnicodeDecodeError as e:
        assert ei.value.start == e.start


def test_streamed_file_ingest_equals_in_memory(tmp_path, monkeypatch):
    """train_bpe(path) on a big file reads it in chunks on a few threads while the GPU counts the previous chunk."""
    import transformer_lm_b200.train as T
    from transformer_lm_b200.synth import synth_host
    monkeypatch.setattr(T, "_STREAM_MIN", 64 << 20)
    monkeypatch.setattr(T, "_STREAM_CHUNK", 48 << 20)
    n = 200 << 20
    host = synth_host("owt", 4321, n)
    path = tmp_path / "corpus.txt"
    host.tofile(path)
    got = run_train_bpe(path, 1200, ["<|endoftext|>"])
    want = _train_bytes(host, 1200, ["<|endoftext|>"])
    assert got[1] == want[1] and got[0] == want[0]
    # the same path (four chunks with halos, reader threads, pinned staging) against the ORACLE on a file it finishes
    monkeypatch.setattr(T, "_STREAM_MIN", 16 << 20)
    monkeypatch.setattr(T, "_STREAM_CHUNK", 12 << 20)
    small = synth_host("owt", 4321, 44 << 20)
    small.tofile(path)
    got = run_train_bpe(path, 800, ["<|endoftext|>"])
    want = oracle.train_bpe_on_bytes(small.tobytes(), 800, ["<|endoftext|>"])
    assert got[1] == want[1] and got[0] == want[0]
    # O_DIRECT reads (block-aligned ranges around the chunks; buffered where the file system refuses the flag): same result
    got = T.train_bpe(path, 800, ["<|endoftext|>"], direct_io=True)
    assert got[1] == want[1] and got[0] == want[0]
    # carriage return -> one-piece path; invalid UTF-8 -> UnicodeDecodeError
    host2 = host[: 100 << 20].copy()
    host2[(70 << 20) + 5] = 0x0D
    host2.tofile(path)
    assert run_train_bpe(path, 500, []) == _train_bytes(host2, 500, [])
    host2[(70 << 20) + 5] = 0xFF
    host2.tofile(path)
    with pytest.raises(UnicodeDecodeError):
        run_train_bpe(path, 500, [])


def test_finish_checks_the_expected_pair_table():
    # multi-GPU linearity check: the all-reduced per-rank pair tables are compared with the table the merge phase builds
    import torch
    from transformer_lm_b200 import sharded
    data = (FIXTURES_PATH / "corpus.en").read_bytes()
    c = sharded.DeviceCounter()
    assert c.add(data, 0, len(data), True, True) is None
    good = c.pair_table(["<|endoftext|>"])
    c.expect_pair_table(good)
    vocab, merges = c.finish(500, ["<|endoftext|>"])
    assert (vocab, merges) == oracle.train_bpe_on_bytes(data, 500, ["<|endoftext|>"])
    c = sharded.DeviceCounter()
    assert c.add(data, 0, len(data), True, True) is None
    bad = good.clone()
    bad[ord("t") * 256 + ord("h")] += 1
    c.expect_pair_table(bad)
    with pytest.raises(RuntimeError):
        c.finish(500, ["<|endoftext|>"])


def test_live_view_of_the_merge_loop():
    """bpe_train_set_live: the kernel stores every merge into page-locked host memory as it is made (the host builds its Python
    objects beside the loop); the buffer must be page-locked, and what appears there is the result."""
    import ctypes as C
    import numpy as np
    from transformer_lm_b200 import _lib
    ctx = _lib.default_context(0)
    L = _lib.lib()
    plain = np.zeros(64, dtype=np.int32)
    assert L.bpe_train_set_live(ctx.handle, _lib.ptr(plain), 32) == _lib.ERR_ARG      # pageable memory is refused
    n_merges = 300
    live = _lib.PinnedBuffer(n_merges * 8)
    live.array[:] = 0xFF
    ctx.check(L.bpe_train_set_live(ctx.handle, _lib.ptr(live.array), n_merges))
    data = np.frombuffer((FIXTURES_PATH / "corpus.en").read_bytes(), dtype=np.uint8)
    pairs = np.zeros((n_merges, 2), dtype=np.int32)
    n_done = C.c_int(0)
    sp_blob, sp_offs = _lib.pack_blobs([])
    ctx.check(L.bpe_train(ctx.handle, _lib.ptr(data), data.size, _lib.ptr(sp_blob), _lib.ptr(sp_offs), 0, n_merges, _lib.ptr(pairs), C.byref(n_done), None))
    ctx.check(L.bpe_train_set_live(ctx.handle, None, 0))
    assert n_done.value == n_merges
    assert np.array_equal(live.array.view(np.int32).reshape(n_merges, 2), pairs)
    live.free()
