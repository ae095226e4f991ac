"""GPU: token offsets (bpe_encode_ex with offsets) against the ids-only encode on the same bytes.

usage: python tools/time_encode_offsets.py OUT.json [bytes=1.1e9] [reps=3]

GPT-2 fixture tokenizer (with <|endoftext|>), synthetic TinyStories (seed 1234) and OWT (seed 4322) shapes of `bytes` each.  For each shape:
bpe_encode and the encode with offsets in bytes and in characters, alternated, each the median (and the range) of `reps` runs after one warm-up,
timed from host memory to the host arrays (bpe_encode_stats ms_total; the spans' download is part of it).  The device time of the offsets
stage: one profiled run per unit (torch.profiler, CUDA kernels), the kernels only the stage launches plus the extra scans it adds over an
ids-only run; and the device time of all kernels and copies of each call (the spans' download is most of the difference).  Then the TinyStories text split on <|endoftext|> through the batch encode without and with offsets.  For comparison, the
same spans derived on the host with numpy from the ids (cumsum of the vocabulary lengths, and a cumulative lead-byte count for
characters).  The card's name and power limit are read in the same run and stored with the numbers."""
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import _bootstrap  # noqa: E402,F401
from tests.adapters import get_tokenizer  # noqa: E402
from tests.common import load_gpt2_fixture  # noqa: E402
from transformer_lm_b200.synth import SEED_OWT_ENCODE, SEED_TINY_TRAIN, synth_host  # noqa: E402

EOT = "<|endoftext|>"
STAGE_KERNELS = ("k_enc_lead_bits", "k_enc_off_count", "k_enc_offsets", "k_enc_lead_span", "k_enc_drop_starts")


def timed(fns, tok, reps):
    """fns: name -> call; one warm-up each, then `reps` rounds with the calls alternated.  ms_total per call: median, min, max."""
    runs = {k: [] for k in fns}
    for k, fn in fns.items():
        fn()
    for _ in range(reps):
        for k, fn in fns.items():
            fn()
            runs[k].append(tok.last_stats["ms_total"])
    return {k: {"ms_total_median": statistics.median(v), "ms_total_min": min(v), "ms_total_max": max(v), "runs": v} for k, v in runs.items()}


def kernel_ms(fn):
    """Device time of one call by kernel or copy name (torch.profiler CUDA events)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.events():
        if e.device_type.name == "CUDA":
            out[e.name] = out.get(e.name, 0.0) + e.device_time_total / 1e3
    return out


def stage_ms(tok, plain, with_offs):
    a, b = kernel_ms(plain), kernel_ms(with_offs)
    own = sum(v for k, v in b.items() if any(s in k for s in STAGE_KERNELS))
    scans = sum(v for k, v in b.items() if "k_scan" in k) - sum(v for k, v in a.items() if "k_scan" in k)
    return {"ms_stage_kernels": own, "ms_extra_scans": scans, "ms_stage": own + scans,
            "ms_device_kernels_and_copies_ids_only": sum(a.values()),
            "ms_device_kernels_and_copies_offsets": sum(b.values())}


def host_spans(tok, data, ids, unit):
    """The byte / character spans of the ids on the host (numpy): what a caller without this feature computes."""
    t0 = time.perf_counter()
    lens = tok._vlen[ids]
    ends = np.cumsum(lens)
    spans = np.stack([ends - lens, ends], axis=1)
    if unit == "char":
        lead = (np.frombuffer(data, dtype=np.uint8) & 0xC0) != 0x80
        before = np.zeros(len(data) + 1, dtype=np.int64)
        np.cumsum(lead, out=before[1:])
        spans = np.stack([before[spans[:, 0] + 1] - 1, before[spans[:, 1]]], axis=1)
    return spans, (time.perf_counter() - t0) * 1e3


def main():
    out_path = sys.argv[1]
    n = int(float(sys.argv[2])) if len(sys.argv) > 2 else int(1.1e9)
    reps = int(sys.argv[3]) if len(sys.argv) > 3 else 3
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    vocab, merges = load_gpt2_fixture()
    tok = get_tokenizer(dict(vocab), list(merges), [EOT])
    # vocabulary lengths for host_spans (the GPT-2 vocabulary holds <|endoftext|>: its id's bytes are the special's)
    tok._vlen = np.zeros(max(k for k in tok.vocab if isinstance(k, int)) + 1, dtype=np.int64)
    for k, v in tok.vocab.items():
        if isinstance(k, int):
            tok._vlen[k] = len(v)
    res = {"gpu": gpu, "tokenizer": "GPT-2 fixture + <|endoftext|>", "bytes": n, "reps": reps, "shapes": {}}
    for shape, seed in (("tinystories", SEED_TINY_TRAIN), ("owt", SEED_OWT_ENCODE)):
        data = synth_host(shape, seed, n)
        data = np.frombuffer(bytes(data).decode("utf-8", errors="ignore").encode(), dtype=np.uint8)
        r = timed({"encode": lambda: tok.encode_to_numpy(data, np.int32),
                   "offsets_byte": lambda: tok.encode_offsets_to_numpy(data, np.int32, unit="byte"),
                   "offsets_char": lambda: tok.encode_offsets_to_numpy(data, np.int32, unit="char")}, tok, reps)
        for unit in ("byte", "char"):
            r["offsets_" + unit]["ms_total_vs_encode"] = r["offsets_" + unit]["ms_total_median"] / r["encode"]["ms_total_median"]
            r["offsets_" + unit].update(stage_ms(tok, lambda: tok.encode_to_numpy(data, np.int32),
                                                 lambda: tok.encode_offsets_to_numpy(data, np.int32, unit=unit)))
            ids, spans = tok.encode_offsets_to_numpy(data, np.int32, unit=unit)
            hs, ms = host_spans(tok, bytes(data), ids, unit)
            r["offsets_" + unit]["numpy_host_ms"] = ms
            r["offsets_" + unit]["numpy_host_equal"] = bool(np.array_equal(hs, spans))
            r["offsets_" + unit]["n_tokens"] = int(ids.size)
            del ids, spans, hs
        if shape == "tinystories":
            docs = bytes(data).decode("utf-8").split(EOT)
            r["n_docs"] = len(docs)
            r.update(timed({"encode_batch": lambda: tok.encode_batch_to_numpy(docs, np.int32),
                            "encode_batch_offsets_char": lambda: tok.encode_batch_offsets_to_numpy(docs, np.int32, unit="char")}, tok, reps))
            r["encode_batch_offsets_char"]["ms_total_vs_encode_batch"] = (r["encode_batch_offsets_char"]["ms_total_median"] /
                                                                          r["encode_batch"]["ms_total_median"])
            del docs
        res["shapes"][shape] = r
        del data
        print(json.dumps(r, indent=1), flush=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
