"""GPU: train_bpe(..., split_special_tokens=True) against the split oracle (tests/helpers/split_train_oracle.c), on every path
train_bpe can take: one piece (bpe_train_dev_ex), pipelined chunks (bpe_train_ex), the streamed file ingest
(bpe_count_add_shard_ex) and, with two GPUs, distributed=True."""
import os
import pathlib
import random
import subprocess
import sys

import numpy as np
import pytest

import _bootstrap  # noqa: F401
from oracle import oracle
from tests.common import FIXTURES_PATH
from tests.helpers import split_train_oracle as sto

pytestmark = pytest.mark.gpu
EOT = "<|endoftext|>"
ROOT = pathlib.Path(__file__).resolve().parent.parent


def _train(data, vocab_size, specials, **kw):
    from transformer_lm_b200.train import train_bpe_on_bytes
    return train_bpe_on_bytes(data, vocab_size, specials, split_special_tokens=True, **kw)


def _learned(vocab, specials):
    return list(vocab.values())[len(oracle._ref_vocab(specials)):]


def _no_special_inside(vocab, specials):
    return not any(s.encode() in t for t in _learned(vocab, specials) for s in specials if s)


@pytest.mark.parametrize("name,vocab_size", [("corpus.en", 500), ("corpus.en", 3000), ("tinystories_sample.txt", 1000),
                                             ("tinystories_sample.txt", 6000)])
def test_fixtures_equal_the_split_oracle(name, vocab_size):
    from transformer_lm_b200.tokenizer import Tokenizer
    from transformer_lm_b200.train import train_bpe
    path = FIXTURES_PATH / name
    want = sto.train_bpe(path, vocab_size, [EOT])
    got = train_bpe(path, vocab_size, [EOT], split_special_tokens=True)
    assert got[1] == want[1] and got[0] == want[0]
    assert _no_special_inside(got[0], [EOT])
    tok = Tokenizer.train_from_file(str(path), vocab_size, [EOT], split_special_tokens=True)
    assert tok.merges == want[1]
    data = path.read_bytes()
    assert _train(data.replace(b"\n", b"\r\n"), vocab_size, [EOT]) == want      # newlines are translated before the split


def test_stats_count_ordinary_pretokens_only():
    data = (FIXTURES_PATH / "tinystories_sample.txt").read_bytes()
    _, _, st = _train(data, 400, [EOT], return_stats=True)
    assert st["n_pretokens"] == sum(sto.count_words(data, [EOT]).values())


SPECIAL_SETS = [[EOT], ["aa"], ["ab", "bc"], ["<|", EOT], ["x\ry"], ["never-occurs"], [EOT, "<pad>", "ab"], ["a", "aa", "aaa"],
                ["é", "🙃"], ["\n\n"]]
WORDS = ["the", "there", "a", "aa", "aaa", "ab", "abc", "bc", "b", "<|", "|>", EOT, "endoftext", "<pad>", "naïve", "日本", "🙃", "12",
         "don't", "x\ry", "é"]


def _fuzz_corpus(seed, specials, n_words=20000):
    r = random.Random(seed)
    out = []
    for _ in range(n_words):
        out.append(r.choice(WORDS + specials * 2))
        out.append(r.choice([" ", " ", " ", "\n", "  ", ", ", ". ", "", "\r\n", "\n\n"]))
    return "".join(out).encode("utf-8")


@pytest.mark.parametrize("k", range(len(SPECIAL_SETS)))
def test_fuzz_corpora_equal_the_split_oracle(k):
    sp = SPECIAL_SETS[k]
    data = _fuzz_corpus(100 + k, sp)
    for vocab_size in (300 + 40 * k, 4000):                                  # 4000 reaches the zero-count tail
        want = sto.train_bpe_on_bytes(data, vocab_size, sp)
        got = _train(data, vocab_size, sp)
        assert got[1] == want[1] and got[0] == want[0], (sp, vocab_size)
        assert _no_special_inside(got[0], [s for s in sp if "\r" not in s])
    # the order of the caller's list does not matter (longest first is the rule)
    assert _train(data, 500, sp[::-1])[1] == sto.train_bpe_on_bytes(data, 500, sp)[1]


def test_without_occurrences_the_split_mode_is_the_default_mode():
    from transformer_lm_b200.train import train_bpe_on_bytes
    data = (FIXTURES_PATH / "corpus.en").read_bytes().replace(EOT.encode(), b"")
    for vocab_size in (500, 5000):
        assert _train(data, vocab_size, [EOT]) == train_bpe_on_bytes(data, vocab_size, [EOT])


def test_invalid_utf8_raises_as_in_the_default_mode():
    from transformer_lm_b200.train import train_bpe_on_bytes
    data = bytearray(_fuzz_corpus(5, [EOT], 3000))
    data[7777] = 0xFF
    with pytest.raises(UnicodeDecodeError) as want:
        train_bpe_on_bytes(bytes(data), 400, [EOT])
    with pytest.raises(UnicodeDecodeError) as got:
        _train(bytes(data), 400, [EOT])
    assert (got.value.start, got.value.reason) == (want.value.start, want.value.reason)


def test_unknown_flag_bits_are_rejected():
    import ctypes as C
    from transformer_lm_b200 import _lib
    ctx = _lib.default_context()
    L = _lib.lib()
    arr = np.frombuffer(b"hello world", dtype=np.uint8)
    sb, so = _lib.pack_blobs([EOT.encode()])
    pairs = np.zeros((4, 2), dtype=np.int32)
    n_done = C.c_int(0)
    rc = L.bpe_train_ex(ctx.handle, _lib.ptr(arr), arr.size, _lib.ptr(sb), _lib.ptr(so), 1, 4, _lib.ptr(pairs), C.byref(n_done), None, 2)
    assert rc == _lib.ERR_ARG
    assert L.bpe_count_begin(ctx.handle) == 0
    assert L.bpe_count_add_shard_ex(ctx.handle, _lib.ptr(arr), arr.size, 0, arr.size, 1, 1, _lib.ptr(sb), _lib.ptr(so), 1, 4) == _lib.ERR_ARG
    # split mode counts a shard whole
    assert L.bpe_count_add_shard_ex(ctx.handle, _lib.ptr(arr), arr.size, 1, arr.size, 1, 1, _lib.ptr(sb), _lib.ptr(so), 1, 1) == _lib.ERR_ARG


def test_a_rank_table_holds_no_special():
    from transformer_lm_b200.sharded import DeviceCounter
    data = (FIXTURES_PATH / "tinystories_sample.txt").read_bytes()
    c = DeviceCounter()
    assert c.add(data, 0, len(data), True, True, split_specials=[EOT]) is None
    blob, offs, counts = c.export()
    raw, o = blob.cpu().numpy().tobytes(), offs.cpu().tolist()
    table = {raw[o[i]:o[i + 1]]: int(x) for i, x in enumerate(counts.cpu().tolist())}
    assert table == sto.count_words(data, [EOT])
    assert not any(EOT.encode() in w for w in table)


@pytest.mark.parametrize("shape", ["tinystories", "owt"])
def test_every_path_agrees_on_a_large_corpus(shape, tmp_path, monkeypatch):
    import torch
    from transformer_lm_b200 import train
    from transformer_lm_b200.synth import synth_host
    n = 400 << 20                                  # > 1.5 pipeline chunks: bpe_train_ex cuts at least once
    data = synth_host(shape, 77, n)
    assert EOT.encode() in data[: 1 << 20].tobytes()
    vocab_size = 3000
    dev = torch.from_numpy(data).cuda()
    one = _train(None, vocab_size, [EOT], device_ptr=dev.data_ptr(), n_bytes=n)          # bpe_train_dev_ex: one piece
    del dev
    piped = _train(data, vocab_size, [EOT])                                              # bpe_train_ex: pipelined
    assert piped == one
    path = tmp_path / "big.txt"
    data.tofile(path)
    monkeypatch.setattr(train, "_STREAM_MIN", 256 << 20)
    monkeypatch.setattr(train, "_STREAM_CHUNK", 64 << 20)
    streamed = train._train_bpe_streamed(path, n, vocab_size, [EOT], split_special_tokens=True)
    assert streamed == one
    assert _no_special_inside(one[0], [EOT])
    default = train.train_bpe_on_bytes(data, vocab_size, [EOT])
    assert default != one                                                                # documents are separated by <|endoftext|>
    train.release_buffers()


def test_distributed_split_training_nccl(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, PYTHONPATH=str(ROOT))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29541", str(ROOT / "tests" / "helpers" / "nccl_split_train_worker.py"), str(tmp_path)]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    for rank in range(2):
        assert (tmp_path / ("ok.%d" % rank)).exists()
