"""GPU: encode into CUDA tensors (encode_batch_to_tensor, encode_batch_padded, bpe_pad_rows_dev) against the host-output calls followed
by an upload, the path a training loop on this library took before.

usage: python tools/time_encode_tensor.py OUT.json [bytes=1.1e9] [reps=5]

GPT-2 fixture tokenizer (with <|endoftext|>), synthetic TinyStories text (seed 1234) of `bytes`, split on <|endoftext|>.  Every time is
a host clock around calls that end with torch.cuda.synchronize(), so both results are on the GPU when the clock stops; each is the
median (and range) of `reps` runs after one warm-up, the compared calls alternated.
  (a) ragged: encode_batch_to_tensor(docs) against torch.from_numpy(encode_batch_to_numpy(docs)).cuda() (ids and id offsets), and the
      same with char offsets (encode_batch_offsets_to_numpy; the spans uploaded too).  The results are compared.
  (b) padded: 256 documents at max_length=1024, pad_to="max_length": encode_batch_padded against encode_batch_to_numpy + numpy padding
      + upload of the ids and the mask.  50 consecutive 256-document slices per run.
  (c) the pad kernel at 16384 rows x 1024 columns, ids only and with spans: the device time of k_pad_rows (torch.profiler, 20
      launches) and the bytes it moves over that time; and the whole bpe_pad_rows_dev call on torch's stream (CUDA events over 50
      calls, the upload of the row offsets included).
The card's name and power limit are read in the same run and stored with the numbers."""
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import _bootstrap  # noqa: E402,F401
from tests.adapters import get_tokenizer  # noqa: E402
from tests.common import load_gpt2_fixture  # noqa: E402
from transformer_lm_b200 import _lib  # noqa: E402
from transformer_lm_b200.synth import SEED_TINY_TRAIN, synth_host  # noqa: E402

EOT = "<|endoftext|>"
EOT_ID = 50256


def timed(fns, reps, tok=None):
    """fns: name -> call; one warm-up each, then `reps` rounds with the calls alternated.  Wall ms per call: median, min, max; with
    `tok`, also the median of the encode pipeline's own time (last_stats ms_total: chunks uploaded, encoded, outputs written)."""
    runs = {k: [] for k in fns}
    pipe = {k: [] for k in fns}
    for fn in fns.values():
        fn()
        torch.cuda.synchronize()
    for _ in range(reps):
        for k, fn in fns.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            runs[k].append((time.perf_counter() - t0) * 1e3)
            if tok is not None:
                pipe[k].append(tok.last_stats["ms_total"])
    res = {k: {"ms_median": statistics.median(v), "ms_min": min(v), "ms_max": max(v), "runs": v} for k, v in runs.items()}
    if tok is not None:
        for k, v in pipe.items():
            res[k]["pipeline_ms_total_median"] = statistics.median(v)
    return res


def host_padded(tok, docs, row_len, pad_id):
    """What a caller did before encode_batch_padded: host ids, numpy padding (right side, first tokens kept), upload."""
    ids, offs = tok.encode_batch_to_numpy(docs, np.int32)
    lens = np.minimum(np.diff(offs), row_len)
    col = np.arange(row_len)
    mask = col[None, :] < lens[:, None]
    src = offs[:-1, None] + col[None, :]
    out = np.where(mask, ids[np.minimum(src, max(ids.size - 1, 0))] if ids.size else pad_id, pad_id).astype(np.int64)
    return {"input_ids": torch.from_numpy(out).cuda(), "attention_mask": torch.from_numpy(mask).cuda()}


def pad_kernel(tok, n_rows, row_len, with_spans, launches=50):
    """Device time of k_pad_rows (torch.profiler) and of whole bpe_pad_rows_dev calls (CUDA events around `launches` back-to-back calls
    on torch's stream), and the bytes the kernel moves."""
    from torch.profiler import ProfilerActivity, profile
    ctx = tok._tok_ctx
    dev = torch.device("cuda", ctx.device)
    rng = np.random.default_rng(0)
    lens = rng.integers(0, 2 * row_len, n_rows)              # half the rows longer than row_len, half shorter
    offs = np.zeros(n_rows + 1, dtype=np.uint64)
    np.cumsum(lens, out=offs[1:])
    n = int(offs[-1])
    ids = torch.randint(0, 50257, (n,), dtype=torch.int32, device=dev)
    spans = torch.randint(0, 1 << 30, (n, 2), dtype=torch.int64, device=dev) if with_spans else None
    x = torch.empty((n_rows, row_len), dtype=torch.int64, device=dev)
    m = torch.empty((n_rows, row_len), dtype=torch.bool, device=dev)
    y = torch.empty((n_rows, row_len, 2), dtype=torch.int64, device=dev) if with_spans else None
    L = _lib.lib()

    def launch():
        ctx.check(L.bpe_pad_rows_dev(ctx.handle, C.c_void_p(ids.data_ptr()), n, _lib.ptr(offs), n_rows,
                                     C.c_void_p(spans.data_ptr()) if with_spans else None, row_len, -1, 0,
                                     C.c_void_p(x.data_ptr()), C.c_void_p(m.data_ptr()), C.c_void_p(y.data_ptr()) if with_spans else None))
    with ctx.lock:
        ctx.use_stream(torch.cuda.current_stream(dev).cuda_stream)
        try:
            launch()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(launches):
                launch()
            b.record()
            b.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(20):
                    launch()
                torch.cuda.synchronize()
        finally:
            ctx.use_stream(None)
    ms_call = a.elapsed_time(b) / launches
    ms = sum(e.device_time_total for e in prof.events() if e.device_type.name == "CUDA" and "k_pad_rows" in e.name) / 1e3 / 20
    kept = int(np.minimum(lens, row_len).sum())
    elems = n_rows * row_len
    nbytes = elems * (8 + 1) + kept * 4 + (n_rows + 1) * 8 + ((elems + kept) * 16 if with_spans else 0)
    return {"rows": n_rows, "row_len": row_len, "spans": with_spans, "kept_tokens": kept, "ms_kernel": ms, "bytes": nbytes,
            "GB_per_s": nbytes / ms / 1e6, "ms_per_call": ms_call}


def main():
    out_path = sys.argv[1]
    n = int(float(sys.argv[2])) if len(sys.argv) > 2 else int(1.1e9)
    reps = int(sys.argv[3]) if len(sys.argv) > 3 else 5
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    vocab, merges = load_gpt2_fixture()
    tok = get_tokenizer(dict(vocab), list(merges), [EOT])
    data = synth_host("tinystories", SEED_TINY_TRAIN, n)
    docs = bytes(data).decode("utf-8", errors="ignore").split(EOT)
    del data
    res = {"gpu": gpu, "tokenizer": "GPT-2 fixture + <|endoftext|>", "text": "synthetic TinyStories, seed %d" % SEED_TINY_TRAIN,
           "bytes": n, "n_docs": len(docs), "reps": reps}

    # (a) ragged batch, ids only and with char offsets
    a = tok.encode_batch_to_tensor(docs)
    w = [torch.from_numpy(v).cuda() for v in tok.encode_batch_to_numpy(docs, np.int32)]
    assert all(torch.equal(g, v) for g, v in zip(a, w))
    a = tok.encode_batch_to_tensor(docs, offsets="char")
    ids, spans, offs = tok.encode_batch_offsets_to_numpy(docs, np.int32, unit="char")
    assert torch.equal(a[0], torch.from_numpy(ids).cuda()) and torch.equal(a[1], torch.from_numpy(offs).cuda())
    assert torch.equal(a[2], torch.from_numpy(spans).cuda())
    res["n_tokens"] = int(ids.size)
    del a, w, ids, spans, offs
    res["ragged"] = timed({
        "to_tensor": lambda: tok.encode_batch_to_tensor(docs),
        "numpy_then_upload": lambda: [torch.from_numpy(v).cuda() for v in tok.encode_batch_to_numpy(docs, np.int32)],
        "to_tensor_char_offsets": lambda: tok.encode_batch_to_tensor(docs, offsets="char"),
        "numpy_then_upload_char_offsets": lambda: [torch.from_numpy(v).cuda() for v in
                                                   tok.encode_batch_offsets_to_numpy(docs, np.int32, unit="char")],
    }, reps, tok)
    r = res["ragged"]
    r["speedup_ids"] = r["numpy_then_upload"]["ms_median"] / r["to_tensor"]["ms_median"]
    r["speedup_char_offsets"] = r["numpy_then_upload_char_offsets"]["ms_median"] / r["to_tensor_char_offsets"]["ms_median"]
    r["char_offsets_over_ids_to_tensor"] = r["to_tensor_char_offsets"]["ms_median"] / r["to_tensor"]["ms_median"]
    print(json.dumps(r, indent=1), flush=True)

    # (b) training-step-sized padded batches
    B, T, K = 256, 1024, 50
    batches = [docs[i * B:(i + 1) * B] for i in range(K)]
    for bd in batches[:3]:
        g = tok.encode_batch_padded(bd, pad_id=EOT_ID, max_length=T, pad_to="max_length")
        h = host_padded(tok, bd, T, EOT_ID)
        assert torch.equal(g["input_ids"], h["input_ids"]) and torch.equal(g["attention_mask"], h["attention_mask"])
    res["padded"] = timed({
        "encode_batch_padded": lambda: [tok.encode_batch_padded(bd, pad_id=EOT_ID, max_length=T, pad_to="max_length") for bd in batches],
        "numpy_pad_then_upload": lambda: [host_padded(tok, bd, T, EOT_ID) for bd in batches],
    }, reps)
    p = res["padded"]
    p["batch"], p["max_length"], p["batches_per_run"] = B, T, K
    for k in ("encode_batch_padded", "numpy_pad_then_upload"):
        p[k]["ms_per_batch"] = p[k]["ms_median"] / K
    p["speedup"] = p["numpy_pad_then_upload"]["ms_median"] / p["encode_batch_padded"]["ms_median"]
    print(json.dumps(p, indent=1), flush=True)

    # (c) the pad kernel alone
    res["pad_kernel"] = [pad_kernel(tok, 16384, 1024, False), pad_kernel(tok, 16384, 1024, True)]
    print(json.dumps(res["pad_kernel"], indent=1), flush=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
