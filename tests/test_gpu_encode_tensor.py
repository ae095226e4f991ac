"""GPU: encode straight into CUDA tensors (Tokenizer.encode_to_tensor / encode_batch_to_tensor, bpe_encode_opts.out_device) and padded
batches collated on the device (Tokenizer.encode_batch_padded, bpe_pad_rows_dev).  The expected values are the host-output calls
(encode_to_numpy, encode_batch_to_numpy and their offsets forms, themselves checked against the oracle elsewhere) and, for padding, a
numpy restatement of the spec in include/bpe_sm100.h."""
import ctypes as C

import numpy as np
import pytest
import torch

import _bootstrap  # noqa: F401
from tests.common import FIXTURES_PATH
from tests.test_gpu_encode_batch import _document_lists, _keyerror_tok, _pair
from transformer_lm_b200 import _lib
from transformer_lm_b200.synth import synth_host

pytestmark = pytest.mark.gpu

EOT = "<|endoftext|>"
EOT_ID = 50256
DROPS = [(0.0, 0), (0.1, 3), (1.0, 0)]
UNITS = [None, "byte", "char"]


@pytest.fixture(scope="module", params=["gpt2", "gpt2_plain", "corpus1000"])
def toks(request):
    return _pair(request.param)


@pytest.fixture(scope="module")
def gpt2():
    return _pair("gpt2")[0]


def _np(t):
    assert t.is_cuda
    return t.cpu().numpy()


def _host_batch(tok, docs, drop, unit):
    """(ids, id offsets, spans or None) of the host-output batch calls."""
    if unit is None:
        ids, offs = tok.encode_batch_to_numpy(docs, np.int32, dropout=drop[0], seed=drop[1])
        return ids, offs, None
    ids, spans, offs = tok.encode_batch_offsets_to_numpy(docs, np.int32, unit=unit, dropout=drop[0], seed=drop[1])
    return ids, offs, spans


def _check_ragged(tok, docs, drop, unit):
    want_ids, want_offs, want_spans = _host_batch(tok, docs, drop, unit)
    got = tok.encode_batch_to_tensor(docs, dropout=drop[0], seed=drop[1], offsets=unit)
    assert len(got) == (2 if unit is None else 3)
    assert got[0].dtype == torch.int32 and got[1].dtype == torch.int64 and got[0].dim() == 1
    assert np.array_equal(_np(got[0]), want_ids) and np.array_equal(_np(got[1]), want_offs)
    if unit is not None:
        assert got[2].dtype == torch.int64 and tuple(got[2].shape) == (want_ids.size, 2)
        assert np.array_equal(_np(got[2]), want_spans)


def test_ragged_parity_on_document_lists(toks):
    tok, _ = toks
    for docs in _document_lists():
        for drop in DROPS:
            for unit in UNITS:
                _check_ragged(tok, docs, drop, unit)


def test_one_document_parity_on_fixtures(toks):
    tok, _ = toks
    for name in ["corpus.en", "german.txt", "address.txt", "tinystories_sample.txt"]:
        data = (FIXTURES_PATH / name).read_bytes()
        for drop in DROPS:
            want = tok.encode_to_numpy(data, np.int32, dropout=drop[0], seed=drop[1])
            got = tok.encode_to_tensor(data, dropout=drop[0], seed=drop[1])
            assert got.dtype == torch.int32 and got.device == torch.device("cuda", tok._tok_ctx.device)
            assert np.array_equal(_np(got), want)
            for unit in ("byte", "char"):
                w_ids, w_spans = tok.encode_offsets_to_numpy(data, np.int32, unit=unit, dropout=drop[0], seed=drop[1])
                g_ids, g_spans = tok.encode_to_tensor(data, dropout=drop[0], seed=drop[1], offsets=unit)
                assert np.array_equal(_np(g_ids), w_ids) and np.array_equal(_np(g_spans), w_spans)
    assert tok.encode_to_tensor(b"").numel() == 0
    ids, spans = tok.encode_to_tensor(b"", offsets="char")
    assert ids.numel() == 0 and tuple(spans.shape) == (0, 2)


def test_results_are_compact(gpt2):
    docs = ["hello world", "a"]
    ids, offs = gpt2.encode_batch_to_tensor(docs)
    assert ids.untyped_storage().nbytes() == ids.numel() * 4       # a copy of the used prefix, not a view of the scratch
    ids, spans = gpt2.encode_to_tensor(b"hello world", offsets="byte")
    assert spans.untyped_storage().nbytes() == spans.numel() * 8


def test_multi_chunk(gpt2, monkeypatch):
    # The pipeline cuts texts of 96 MiB and more into chunks (BPE_ENCODE_CHUNK_MB, read per call): chunk k's ids and spans land at
    # its running offset in the caller's tensors, and the character count carries from chunk to chunk.
    monkeypatch.setenv("BPE_ENCODE_CHUNK_MB", "8")
    text = synth_host("tinystories", 1234, 112 << 20).tobytes().decode("utf-8", errors="ignore")
    docs = text.split(EOT)
    big = " ".join(["once", "upon", "a", "time", "Lily", "saw", "3", "dog.", "中文"][i % 9] for i in range(3_000_000))
    docs.insert(len(docs) // 2, big)                        # one document longer than a chunk
    for drop, unit in [((0.0, 0), None), ((0.0, 0), "char"), ((0.1, 3), "byte")]:
        _check_ragged(gpt2, docs, drop, unit)
    data = text.encode("utf-8")
    for drop, unit in [((0.0, 0), "char"), ((0.1, 3), None)]:
        if unit is None:
            assert np.array_equal(_np(gpt2.encode_to_tensor(data, dropout=drop[0], seed=drop[1])),
                                  gpt2.encode_to_numpy(data, np.int32, dropout=drop[0], seed=drop[1]))
        else:
            g_ids, g_spans = gpt2.encode_to_tensor(data, dropout=drop[0], seed=drop[1], offsets=unit)
            w_ids, w_spans = gpt2.encode_offsets_to_numpy(data, np.int32, unit=unit, dropout=drop[0], seed=drop[1])
            assert np.array_equal(_np(g_ids), w_ids) and np.array_equal(_np(g_spans), w_spans)


# ---- padding ---------------------------------------------------------------------------------------------------------------------
def pad_reference(ids, offs, spans, row_len, pad_id, padding_side, truncation_side):
    """The spec of bpe_pad_rows_dev / encode_batch_padded in numpy: for row r, k = min(m, row_len) tokens are kept -- the first k (the
    last k with left truncation) -- at columns [0, k) (right padding) or [row_len - k, row_len) (left padding); the rest is pad_id, a
    mask of False and the span (0, 0)."""
    n_rows = len(offs) - 1
    out = np.full((n_rows, row_len), pad_id, dtype=np.int64)
    mask = np.zeros((n_rows, row_len), dtype=bool)
    sp = np.zeros((n_rows, row_len, 2), dtype=np.int64)
    for r in range(n_rows):
        lo, hi = int(offs[r]), int(offs[r + 1])
        k = min(hi - lo, row_len)
        src = slice(hi - k, hi) if truncation_side == "left" else slice(lo, lo + k)
        dst = slice(row_len - k, row_len) if padding_side == "left" else slice(0, k)
        out[r, dst] = ids[src]
        mask[r, dst] = True
        if spans is not None:
            sp[r, dst] = spans[src]
    return out, mask, sp


PAD_DOCS = ["Once upon a time there was a little dog.", "", "hi there", "A story" + EOT + "and another one" + EOT, EOT + EOT,
            "The quick brown fox jumps over the lazy dog. " * 6, "naïve café 中文 \U0001F643", "  \n\n x", "ok then"]


@pytest.mark.parametrize("pad_id", [EOT_ID, -1])
def test_padding_against_the_spec(gpt2, pad_id):
    tok = gpt2
    ids, spans, offs = tok.encode_batch_offsets_to_numpy(PAD_DOCS, np.int32, unit="char")
    lens = np.diff(offs)
    nz = lens[lens > 0]
    assert nz.min() >= 2
    lengths = [None, int(nz.min()) - 1, int(nz.min() + nz.max()) // 2, int(nz.max()) + 5]   # none / below / between / above
    for pad_to in ("longest", "max_length"):
        for max_length in lengths:
            if pad_to == "max_length" and max_length is None:
                continue
            row_len = max_length if pad_to == "max_length" else min(int(lens.max()), max_length or 1 << 62)
            for ps in ("left", "right"):
                for ts in ("left", "right"):
                    kw = dict(pad_id=pad_id, max_length=max_length, pad_to=pad_to, padding_side=ps, truncation_side=ts)
                    w_ids, w_mask, w_sp = pad_reference(ids, offs, spans, row_len, pad_id, ps, ts)
                    r = tok.encode_batch_padded(PAD_DOCS, offsets="char", **kw)
                    assert set(r) == {"input_ids", "attention_mask", "offsets"}
                    assert r["input_ids"].dtype == torch.int64 and r["attention_mask"].dtype == torch.bool
                    assert tuple(r["offsets"].shape) == (len(PAD_DOCS), row_len, 2), kw
                    assert np.array_equal(_np(r["input_ids"]), w_ids), kw
                    assert np.array_equal(_np(r["attention_mask"]), w_mask), kw
                    assert np.array_equal(_np(r["offsets"]), w_sp), kw
                    r = tok.encode_batch_padded(PAD_DOCS, **kw)
                    assert set(r) == {"input_ids", "attention_mask"}
                    assert np.array_equal(_np(r["input_ids"]), w_ids) and np.array_equal(_np(r["attention_mask"]), w_mask), kw


def test_padding_edge_cases(gpt2):
    tok = gpt2
    r = tok.encode_batch_padded([], pad_id=0)
    assert tuple(r["input_ids"].shape) == (0, 0) and tuple(r["attention_mask"].shape) == (0, 0)
    r = tok.encode_batch_padded([], pad_id=0, max_length=7, pad_to="max_length", offsets="byte")
    assert tuple(r["input_ids"].shape) == (0, 7) and tuple(r["offsets"].shape) == (0, 7, 2)
    r = tok.encode_batch_padded(["", ""], pad_id=5)
    assert tuple(r["input_ids"].shape) == (2, 0)
    r = tok.encode_batch_padded(["", ""], pad_id=5, max_length=3, pad_to="max_length", offsets="char")
    assert _np(r["input_ids"]).tolist() == [[5] * 3] * 2 and not _np(r["attention_mask"]).any() and not _np(r["offsets"]).any()
    one = "Lily saw a dog."
    want = tok.encode(one)
    r = tok.encode_batch_padded([one], pad_id=-1)
    assert _np(r["input_ids"]).tolist() == [want] and _np(r["attention_mask"]).all()
    r = tok.encode_batch_padded([one], pad_id=-1, max_length=3, truncation_side="left", offsets="byte")
    assert _np(r["input_ids"]).tolist() == [want[-3:]]
    spans = _np(r["offsets"])[0]
    assert spans[-1, 1] == len(one.encode()) and spans[0, 0] > 0          # still relative to the document


def test_padding_with_dropout(gpt2):
    docs = PAD_DOCS * 3
    ids, offs = gpt2.encode_batch_to_numpy(docs, np.int32, dropout=0.2, seed=9)
    r = gpt2.encode_batch_padded(docs, pad_id=-1, max_length=12, dropout=0.2, seed=9)
    w_ids, w_mask, _ = pad_reference(ids, offs, None, 12, -1, "right", "right")
    assert np.array_equal(_np(r["input_ids"]), w_ids) and np.array_equal(_np(r["attention_mask"]), w_mask)


# ---- streams ---------------------------------------------------------------------------------------------------------------------
def _stream_check(tok, docs):
    """Runs on torch's current stream: queued work there (a spin, then a fill of memory the allocator hands out again) must come
    before the library's writes, and torch ops queued after the call see them."""
    want_ids, want_offs = tok.encode_batch_to_numpy(docs, np.int32)
    w_pad, w_mask, _ = pad_reference(want_ids, want_offs, None, 32, -1, "left", "right")
    junk = torch.empty(len(docs) * 32 * 8, dtype=torch.int64, device="cuda")
    torch.cuda._sleep(50_000_000)
    junk.fill_(7)
    del junk
    r = tok.encode_batch_padded(docs, pad_id=-1, max_length=32, pad_to="max_length", padding_side="left")
    ids, offs = tok.encode_batch_to_tensor(docs)
    pad_sum = torch.where(r["attention_mask"], r["input_ids"], torch.zeros_like(r["input_ids"])).sum()
    ids_sum = ids.to(torch.int64).sum()
    return (pad_sum, ids_sum, r, ids, offs), (int(w_pad[w_mask].sum()), int(want_ids.astype(np.int64).sum()), w_pad, want_ids, want_offs)


def test_side_stream_and_default_stream(gpt2):
    docs = (FIXTURES_PATH / "tinystories_sample.txt").read_text(encoding="utf-8").split(EOT)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        got, want = _stream_check(gpt2, docs)
    s.synchronize()
    for g, w in ((got, want), _stream_check(gpt2, docs)):           # again on the default stream
        torch.cuda.synchronize()
        assert int(g[0]) == w[0] and int(g[1]) == w[1]
        assert np.array_equal(_np(g[2]["input_ids"]), w[2])
        assert np.array_equal(_np(g[3]), w[3]) and np.array_equal(_np(g[4]), w[4])
    ids, offs = gpt2.encode_batch_to_numpy(docs, np.int32)               # the context is back on its own stream
    assert np.array_equal(ids, want[3]) and np.array_equal(offs, want[4])


# ---- errors ----------------------------------------------------------------------------------------------------------------------
def _same_error(fn, want_fn):
    with pytest.raises(Exception) as want:
        want_fn()
    with pytest.raises(type(want.value)) as got:
        fn()
    assert got.value.args == want.value.args


def test_errors_are_those_of_the_host_calls(gpt2):
    ktok, _ = _keyerror_tok()
    cases = [(ktok, ["xyz"] * 50 + ["q abc"] + ["zz"] * 10 + ["zab"] + ["x"] * 5),
             (ktok, ["ok", "zab", "ok", "bad \ud800"]),
             (ktok, ["ok", "bad \ud800", "zab"]),
             (ktok, [b"ok", b"zab", b"\xff", b"q"]),
             (gpt2, [b"ok ", b"abc\xe4\xb8", b"\xad rest"]),
             (gpt2, ["fine", "bad \udc00 surrogate"])]
    for tok, docs in cases:
        host = lambda: tok.encode_batch_to_numpy(docs, np.int32)    # noqa: E731
        _same_error(lambda: tok.encode_batch_to_tensor(docs), host)
        _same_error(lambda: tok.encode_batch_to_tensor(docs, offsets="char"), host)
        _same_error(lambda: tok.encode_batch_padded(docs, pad_id=0, max_length=4), host)
    _same_error(lambda: ktok.encode_to_tensor(b"q abc"), lambda: ktok.encode_to_numpy(b"q abc"))
    _same_error(lambda: gpt2.encode_to_tensor(b"ab\xffc", offsets="byte"), lambda: gpt2.encode_to_numpy(b"ab\xffc"))
    ids, _ = gpt2.encode_batch_to_tensor(["still works"])                # nothing is left behind by a failed call
    assert _np(ids).tolist() == gpt2.encode("still works")


# ---- C ABI rejections ------------------------------------------------------------------------------------------------------------
def test_c_abi_rejections(gpt2):
    L = _lib.lib()
    h = gpt2._device_tok()
    ctx = gpt2._tok_ctx
    dev = torch.device("cuda", ctx.device)
    blob = np.frombuffer(b"hello world, hello tensors", dtype=np.uint8)
    n_out = C.c_uint64(0)

    def encode(out, cap, offs_out=None):
        opts = _lib.EncodeOpts(out_device=1)
        if offs_out is not None:
            opts.with_offsets, opts.offset_unit, opts.offs_out = 1, _lib.OFF_BYTES, offs_out
        return L.bpe_encode_ex(h, _lib.ptr(blob), blob.size, C.byref(opts), _lib.DTYPE_I32, out, cap, C.byref(n_out), None)

    def rejected(rc):
        return rc == _lib.ERR_ARG and L.bpe_launch_count() == launches

    pinned = _lib.PinnedBuffer(blob.size * 4)                               # page-locked host memory: not device memory
    pinned.array[:] = 0xAB
    out = torch.empty(blob.size, dtype=torch.int32, device=dev)
    spans = torch.empty((blob.size + 1, 2), dtype=torch.int64, device=dev)
    launches = L.bpe_launch_count()
    assert rejected(encode(C.c_void_p(pinned.array.ctypes.data), blob.size))
    assert (pinned.array == 0xAB).all()
    assert rejected(encode(C.c_void_p(out.data_ptr()), blob.size, spans.data_ptr() + 8))
    assert rejected(encode(C.c_void_p(out.data_ptr()), blob.size, pinned.array.ctypes.data))
    assert encode(C.c_void_p(out.data_ptr()), blob.size, spans.data_ptr()) == 0        # the same call with good pointers
    torch.cuda.synchronize()
    w_ids, w_spans = gpt2.encode_offsets_to_numpy(blob, np.int32, unit="byte")
    assert n_out.value == w_ids.size and np.array_equal(_np(out[: n_out.value]), w_ids)
    assert np.array_equal(_np(spans[: n_out.value]), w_spans)
    assert encode(None, 0) == 0 and n_out.value == w_ids.size                        # size query

    ids = torch.from_numpy(w_ids).to(dev)
    sp = torch.from_numpy(w_spans).to(dev)
    n = w_ids.size
    rows, row_len = 2, 4
    x = torch.empty((rows, row_len), dtype=torch.int64, device=dev)
    m = torch.empty((rows, row_len), dtype=torch.uint8, device=dev)
    y = torch.empty((rows, row_len, 2), dtype=torch.int64, device=dev)

    def pad(offs, flags=0, spans_in=None, spans_out=None, mask=m.data_ptr(), ids_out=x.data_ptr()):
        o = np.array(offs, dtype=np.uint64)
        return L.bpe_pad_rows_dev(ctx.handle, C.c_void_p(ids.data_ptr()), n, _lib.ptr(o), len(offs) - 1,
                                  None if spans_in is None else C.c_void_p(spans_in), row_len, -1, flags, C.c_void_p(ids_out),
                                  None if mask is None else C.c_void_p(mask), None if spans_out is None else C.c_void_p(spans_out))

    launches = L.bpe_launch_count()
    assert rejected(pad([0, 3, 2]))
    assert L.bpe_last_error_detail(ctx.handle) == 1
    assert rejected(pad([0, 2, n + 1]))
    assert L.bpe_last_error_detail(ctx.handle) == 1
    assert rejected(pad([0, 2, n], flags=4))
    assert rejected(pad([0, 2, n], spans_in=sp.data_ptr()))
    assert rejected(pad([0, 2, n], spans_out=y.data_ptr()))
    assert rejected(pad([0, 2, n], spans_in=sp.data_ptr() + 8, spans_out=y.data_ptr()))
    assert rejected(pad([0, 2, n], spans_in=sp.data_ptr(), spans_out=y.data_ptr() + 8))
    assert rejected(pad([0, 2, n], ids_out=pinned.array.ctypes.data))
    assert rejected(pad([0, 2, n], mask=pinned.array.ctypes.data))
    assert (pinned.array == 0xAB).all()
    assert pad([0, 2, n], mask=None) == 0                                            # no mask: accepted
    torch.cuda.synchronize()
    w, _, _ = pad_reference(w_ids, [0, 2, n], None, row_len, -1, "right", "right")
    assert np.array_equal(_np(x), w)
    assert pad([0, 2, n], flags=_lib.PAD_LEFT | _lib.TRUNC_LEFT, spans_in=sp.data_ptr(), spans_out=y.data_ptr()) == 0
    torch.cuda.synchronize()
    w, wm, ws = pad_reference(w_ids, [0, 2, n], w_spans, row_len, -1, "left", "left")
    assert np.array_equal(_np(x), w) and np.array_equal(_np(m).astype(bool), wm) and np.array_equal(_np(y), ws)
    pinned.free()
