"""train_bpe(..., split_special_tokens=True) without a GPU: the split oracle (tests/helpers/split_train_oracle.c) against a
pure-Python restatement of the spec, the C ABI symbols, and the host cut logic of the streamed ingest and of the multi-rank
path, with a checker-backed counter standing in for the device."""
import os
import random
import re
import socket

import numpy as np
import pytest
import regex

import _bootstrap  # noqa: F401
from oracle import oracle
from tests.common import FIXTURES_PATH
from tests.helpers import split_train_oracle as sto
from tests.helpers.fake_counter import OracleCounter

GPT2 = regex.compile(r"""'(?:[sdmt]|ll|ve|re)| ?\p{L}+| ?\p{N}+| ?[^\s\p{L}\p{N}]+|\s+(?!\S)|\s+""")
EOT = "<|endoftext|>"


def restated_counts(data: bytes, specials) -> dict:
    """The spec in plain Python: strict decode, universal newlines, re.split on the escaped alternation sorted longest first,
    the GPT-2 pattern on every piece, occurrences counted nowhere."""
    text = data.decode("utf-8").replace("\r\n", "\n").replace("\r", "\n")
    pieces = [text]
    sp = [s for s in specials if s]
    if sp:
        pieces = re.split("|".join(re.escape(s) for s in sorted(sp, key=len, reverse=True)), text)
    out: dict = {}
    for piece in pieces:
        for m in GPT2.finditer(piece):
            w = m.group().encode("utf-8")
            out[w] = out.get(w, 0) + 1
    return out


SPECIAL_SETS = [
    [EOT], ["aa"], ["ab", "bc"], ["<|", EOT], ["x\ry"], ["never-occurs-here"], [EOT, "<pad>", "ab"], ["a", "aa", "aaa"],
    ["é", "🙃"], [" ", "  "], [], ["\n\n"],
]
PARTS = ["a", "aa", "aaa", "b", "ab", "bc", "abc", " ", "  ", "\n", "\r\n", "\r", "x\ry", "<|", "|>", EOT, "endoftext", "é",
         "🙃", "the", " the", "don't", "'s", "12", ".", "<pad>", "\t", "  \n"]


def _fuzz_text(r: random.Random, specials) -> bytes:
    parts = PARTS + specials * 3
    n = r.randint(0, 40)
    s = "".join(r.choice(parts) for _ in range(n))
    if specials and r.random() < 0.3:
        s = r.choice(specials) + s                 # at the start
    if specials and r.random() < 0.3:
        s = s + r.choice(specials) * r.randint(1, 3)   # at the end, back to back
    return s.encode("utf-8")


def test_split_oracle_counts_equal_the_restated_spec_on_fuzzed_texts():
    r = random.Random(1234)
    n = 0
    for sp in SPECIAL_SETS:
        for _ in range(60):
            data = _fuzz_text(r, sp)
            assert sto.count_words(data, sp) == restated_counts(data, sp), (data, sp)
            n += 1
    runs = b"a" * 37 + b" " + b"a" * 2 + b"\n" + b"a" * 5                 # ['aa'] on runs of a
    assert sto.count_words(runs, ["aa"]) == restated_counts(runs, ["aa"])
    assert n >= 500


def test_split_oracle_on_the_fixtures_and_crlf():
    for name in ("corpus.en", "tinystories_sample.txt"):
        data = (FIXTURES_PATH / name).read_bytes()
        want = restated_counts(data, [EOT])
        assert sto.count_words(data, [EOT]) == want
        assert sto.count_words(data.replace(b"\n", b"\r\n"), [EOT]) == want
        # no special occurs: the split mode trains as the default mode
        if EOT.encode() not in data:
            assert sto.count_words(data, [EOT]) == oracle.count_pretokens(data, [EOT])


def test_split_oracle_training_invariants():
    data = (FIXTURES_PATH / "tinystories_sample.txt").read_bytes()
    assert EOT.encode() in data
    vocab, merges = sto.train_bpe_on_bytes(data, 1000, [EOT])
    learned = list(vocab.values())[1 + 256:]
    assert learned and not any(EOT.encode() in t or t in (b"<|", b"|>") for t in learned)
    dv, dm = oracle.train_bpe_on_bytes(data, 1000, [EOT])
    assert any(b"<|" in t or b"|>" in t for t in list(dv.values())[257:])   # the default mode spends tokens on the separator
    # no occurrence in the text: identical to the default mode, also past the zero-count tail
    plain = data.replace(EOT.encode(), b"\n")
    assert sto.train_bpe_on_bytes(plain[:3000], 2000, [EOT]) == oracle.train_bpe_on_bytes(plain[:3000], 2000, [EOT])
    with pytest.raises(UnicodeDecodeError):
        sto.train_bpe_on_bytes(b"ab\xffcd", 300, [EOT])


def test_split_oracle_merge_loop_is_the_oracles():
    """Without a special-token occurrence both modes count the same words, so the split oracle's copy of the merge loop must give
    orc_train_bpe's result exactly: fixtures, fuzzed texts, CRLF input, specials that never occur, zero-count tails."""
    r = random.Random(99)
    texts = [(FIXTURES_PATH / "corpus.en").read_bytes().replace(EOT.encode(), b""),
             (FIXTURES_PATH / "tinystories_sample.txt").read_bytes().replace(EOT.encode(), b"\r\n")]
    texts += [b"".join(_fuzz_text(r, []) for _ in range(200)).replace(EOT.encode(), b"").replace(b"<pad>", b"") for _ in range(4)]
    for data in texts:
        for specials, vocab_size in (([], 300), ([EOT], 1000), (["never-occurs-here", "<pad>"], 5000)):
            assert sto.train_bpe_on_bytes(data, vocab_size, specials) == oracle.train_bpe_on_bytes(data, vocab_size, specials)


def test_new_train_entry_points_are_declared_bound_and_exported():
    import ctypes
    from transformer_lm_b200 import _build, _lib
    header = (FIXTURES_PATH.parent.parent / "include" / "bpe_sm100.h").read_text()
    dll = ctypes.CDLL(str(_build.build()))
    for name in ("bpe_train_ex", "bpe_train_dev_ex", "bpe_count_add_shard_ex", "bpe_count_add_shard_dev_ex"):
        assert re.search(r"\b%s\s*\(" % name, header) and name in _lib.EXPORTS and hasattr(dll, name)
    assert re.search(r"#define BPE_TRAIN_SPLIT_SPECIALS 1\b", header) and _lib.TRAIN_SPLIT_SPECIALS == 1


# ---- host cut logic -------------------------------------------------------------------------------------------------------
class SplitCounter(OracleCounter):
    """OracleCounter that also follows bpe_count_add_shard_ex: with split_specials the shard is one whole text, split on them."""
    adds_split = 0

    def __init__(self, ctx=None):
        super().__init__()

    def add(self, data, own_begin, own_end, at_file_start, at_file_end, device_ptr=None, n_bytes=None, split_specials=None):
        if split_specials is None:
            return super().add(data, own_begin, own_end, at_file_start, at_file_end)
        data = bytes(data)
        assert (own_begin, own_end) == (0, len(data))
        SplitCounter.adds_split += 1
        self.adds += 1
        bad = oracle.utf8_validate(data)
        if bad >= 0:
            return ("utf8", bad)
        if b"\r" in data:
            return ("newline", 0)
        for w, c in sto.count_words(data, split_specials).items():
            self.table[w] = self.table.get(w, 0) + c
        return None

    def finish(self, vocab_size, special_tokens, return_stats=False):
        return dict(self.table)


class AlignedBuffer:
    def __init__(self, nbytes):
        self.nbytes = int(nbytes)
        self.array = np.zeros(self.nbytes, dtype=np.uint8)

    def free(self):
        self.array = None


@pytest.fixture()
def small_chunks(monkeypatch):
    from transformer_lm_b200 import sharded, train
    train.release_buffers()
    monkeypatch.setattr(train._lib, "PinnedBuffer", AlignedBuffer)
    monkeypatch.setattr(sharded, "DeviceCounter", SplitCounter)
    monkeypatch.setattr(train, "_STREAM_CHUNK", 4096)
    monkeypatch.setattr(train, "_READ_THREADS", 3)
    SplitCounter.adds_split = 0
    yield train
    train.release_buffers()


def _dense_chains(r: random.Random, n: int) -> bytes:
    """Stretches of overlapping candidates (aaaa..., ababab..., <|<|<|endoftext|>) between ordinary text."""
    body = (FIXTURES_PATH / "tinystories_sample.txt").read_bytes().replace(b"\r", b"")
    out = bytearray()
    while len(out) < n:
        k = r.randrange(len(body) - 600)
        out += body[k: k + r.randint(50, 600)]
        out += r.choice([b"a" * r.randint(1, 900), b"ab" * r.randint(1, 500), b"bc" * 300 + b"abc" * 200, b"<|" * 400 + EOT.encode(),
                         (EOT.encode() * 3) + b"  ", b"x\ry".replace(b"\r", b"")])
    return bytes(out)


@pytest.mark.parametrize("specials", [[EOT], ["aa"], ["ab", "bc"], ["<|", EOT]])
def test_streamed_split_table_equals_the_whole_text_count(tmp_path, small_chunks, specials):
    train = small_chunks
    data = _dense_chains(random.Random(7), 60000)
    path = tmp_path / "c.txt"
    path.write_bytes(data)
    table = train._train_bpe_streamed(path, len(data), 1000, specials, split_special_tokens=True)
    assert table == sto.count_words(data, specials)
    assert SplitCounter.adds_split >= 5                      # really cut into chunks
    assert not any(s.encode() in w for w in table for s in specials)


def test_streamed_split_grows_a_chunk_without_exact_cut_and_falls_back_on_cr(tmp_path, small_chunks):
    train = small_chunks
    # after 20 000 bytes there is no exact cut at all: one run of a's (every position inside a chain of 'aa' candidates)
    data = _dense_chains(random.Random(3), 20000) + b"a" * 30000
    path = tmp_path / "c.txt"
    path.write_bytes(data)
    assert train._train_bpe_streamed(path, len(data), 1000, ["aa"], split_special_tokens=True) == sto.count_words(data, ["aa"])
    assert SplitCounter.adds_split <= 20000 // 4096 + 2      # the rest stayed one chunk
    path.write_bytes(data[:30000] + b"\r\n" + data[30000:])
    assert train._train_bpe_streamed(path, len(data) + 2, 1000, ["aa"], split_special_tokens=True) is None
    bad = bytearray(data)
    bad[25000] = 0xFF
    path.write_bytes(bytes(bad))
    with pytest.raises(UnicodeDecodeError) as e:
        train._train_bpe_streamed(path, len(bad), 1000, ["aa"], split_special_tokens=True)
    assert e.value.object[e.value.start] == 0xFF


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, scenarios, q):
    import torch.distributed as dist
    from transformer_lm_b200 import sharded
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        for name, data, specials in scenarios:
            counter = SplitCounter()
            try:
                out = sharded.sharded_count(counter, sharded.FileShards(lambda lo, hi: data[lo:hi], len(data)), specials, None, True,
                                            split_special_tokens=True)
                q.put((name, rank, out, dict(counter.table)))
            except UnicodeDecodeError as e:
                q.put((name, rank, "utf8", e.object[e.start]))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_split_tables_equal_the_whole_text_count(world):
    import torch.multiprocessing as mp
    r = random.Random(world)
    dense = _dense_chains(r, 30000)
    scenarios = [
        ("eot", dense, [EOT]), ("aa", dense, ["aa"]), ("abbc", dense, ["ab", "bc"]), ("chain", dense, ["<|", EOT]),
        ("no-cut", b"a" * 5000 + b" b" + b"a" * 5000, ["aa"]),                 # one exact cut only: later ranks idle
        ("cr", dense[:9000] + b"\r" + dense[9000:], [EOT]),
        ("utf8", dense[:20000] + b"\xff" + dense[20000:], [EOT]),
    ]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(k, world, port, scenarios, q)) for k in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=240) for _ in range(world * len(scenarios))]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    by = {}
    for name, rank, out, table in res:
        by.setdefault(name, []).append((out, table))
    for name, data, specials in scenarios:
        outs = by[name]
        if name == "cr":
            assert all(o == "newline" for o, _ in outs)
        elif name == "utf8":
            assert all(o == "utf8" and t == 0xFF for o, t in outs)
        else:
            want = sto.count_words(data, specials)
            assert all(o == "ok" and t == want for o, t in outs), name
