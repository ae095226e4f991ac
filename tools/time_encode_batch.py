"""GPU: batched encode against the joined text and against a loop of Tokenizer.encode.

usage: python tools/time_encode_batch.py OUT.json [bytes=1.1e9] [loop_docs=100000] [reps=3]

Input: the TinyStories-shape synthetic corpus (seed 1234) split on <|endoftext|> into documents, GPT-2 fixture tokenizer.
Reports, each the median of `reps` runs after one warm-up run:
  (a) stats.ms_total (device timeline) of bpe_encode_batch on all documents against bpe_encode on the same bytes joined;
  (b) wall time of encode_batch_to_numpy and of encode_batch from the list[str];
  (c) wall time of [tok.encode(d) for d in docs] over the first `loop_docs` documents, and encode_batch on the same documents.
The card's name and power limit are read in the same run and stored with the numbers."""
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
from transformer_lm_b200.synth import synth_host  # noqa: E402

EOT = "<|endoftext|>"


def timed(fn, reps):
    fn()
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        r = fn()
        out.append(time.perf_counter() - t0)
    return statistics.median(out), r


def main():
    out_path = sys.argv[1]
    n = int(float(sys.argv[2])) if len(sys.argv) > 2 else int(1.1e9)
    loop_docs = int(sys.argv[3]) if len(sys.argv) > 3 else 100_000
    reps = int(sys.argv[4]) if len(sys.argv) > 4 else 3
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    vocab, merges = load_gpt2_fixture()
    tok = get_tokenizer(dict(vocab), list(merges), [EOT])
    text = synth_host("tinystories", 1234, n).tobytes().decode("utf-8", errors="ignore")
    docs = text.split(EOT)
    del text
    res = {"gpu": gpu, "corpus": "synthetic TinyStories shape, seed 1234", "bytes": n, "n_docs": len(docs), "reps": reps}

    # (a) device time: batch against the joined bytes
    blob = "".join(docs).encode("utf-8")
    res["doc_bytes"] = len(blob)
    ms = []
    for _ in range(reps + 1):
        ids_b, offs = tok.encode_batch_to_numpy(docs, np.uint16)
        ms.append(tok.last_stats["ms_total"])
    res["a_batch_ms_total"] = statistics.median(ms[1:])
    ms = []
    for _ in range(reps + 1):
        ids_j = tok.encode_to_numpy(blob, np.uint16)
        ms.append(tok.last_stats["ms_total"])
    res["a_joined_ms_total"] = statistics.median(ms[1:])
    res["a_ratio"] = res["a_batch_ms_total"] / res["a_joined_ms_total"]
    res["ids_batch"], res["ids_joined"] = int(ids_b.size), int(ids_j.size)
    del blob, ids_j

    # (b) end to end from the list[str]
    res["b_encode_batch_to_numpy_s"], _ = timed(lambda: tok.encode_batch_to_numpy(docs, np.int32), reps)
    res["b_encode_batch_s"], _ = timed(lambda: tok.encode_batch(docs), reps)

    # (c) the loop over the first loop_docs documents, measured, and the batch on the same documents
    sub = docs[:loop_docs]
    res["c_docs"], res["c_doc_bytes"] = len(sub), sum(len(d.encode("utf-8")) for d in sub)
    t_loop, want = timed(lambda: [tok.encode(d) for d in sub], 1)
    t_batch, got = timed(lambda: tok.encode_batch(sub), reps)
    assert got == want, "encode_batch differs from the encode loop"
    res["c_encode_loop_s"], res["c_encode_batch_s"] = t_loop, t_batch
    res["c_speedup"] = t_loop / t_batch
    res["c_loop_us_per_doc"] = t_loop / len(sub) * 1e6
    print(json.dumps(res, indent=1))
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
