"""GPU: BPE-dropout encode (bpe_encode_ex with dropout > 0) against the deterministic encode on the same bytes.

usage: python tools/time_encode_dropout.py OUT.json [bytes=1.1e9] [reps=2]

GPT-2 fixture tokenizer (with <|endoftext|>), synthetic TinyStories (seed 1234) and OWT (seed 4322) shapes of `bytes` each.  For each
shape: bpe_encode, and dropout at p = 0.1 and p = 0.5, every one the median of `reps` runs after one warm-up run, with the device time
per stage from bpe_encode_stats (ms_pretok, ms_lookup, ms_bpe -- the dropout stage is part of it --, ms_emit, ms_total).  Then the
TinyStories text split on <|endoftext|> through the batch encode without and with dropout at p = 0.1.  For context, the CPU
oracle (one core) on a 16 MB slice of each shape.  The card's name and power limit are read in the same run and stored with the numbers."""
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import _bootstrap  # noqa: E402,F401
from tests.helpers.dropout_oracle import DropoutOracle  # noqa: E402
from tests.adapters import get_tokenizer  # noqa: E402
from tests.common import load_gpt2_fixture  # noqa: E402
from transformer_lm_b200.synth import SEED_OWT_ENCODE, SEED_TINY_TRAIN, synth_host  # noqa: E402

EOT = "<|endoftext|>"
STAGES = ("ms_pretok", "ms_lookup", "ms_bpe", "ms_emit", "ms_total")


def stage_times(fn, tok, reps):
    fn()
    runs = []
    for _ in range(reps):
        r = fn()
        runs.append(dict(tok.last_stats))
    out = {k: statistics.median(s[k] for s in runs) for k in STAGES}
    out["n_tokens"] = int(runs[0]["n_tokens"])
    out["GB_per_s"] = runs[0]["n_bytes"] / out["ms_total"] / 1e6
    return out, r


def main():
    out_path = sys.argv[1]
    n = int(float(sys.argv[2])) if len(sys.argv) > 2 else int(1.1e9)
    reps = int(sys.argv[3]) if len(sys.argv) > 3 else 2
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    vocab, merges = load_gpt2_fixture()
    tok = get_tokenizer(dict(vocab), list(merges), [EOT])
    otok = DropoutOracle(dict(vocab), list(merges), [EOT])
    res = {"gpu": gpu, "tokenizer": "GPT-2 fixture + <|endoftext|>", "bytes": n, "reps": reps, "shapes": {}}
    for shape, seed in (("tinystories", SEED_TINY_TRAIN), ("owt", SEED_OWT_ENCODE)):
        data = synth_host(shape, seed, n)
        r = {}
        r["encode"], base = stage_times(lambda: tok.encode_to_numpy(data, np.uint16), tok, reps)
        for p in (0.1, 0.5):
            r["dropout_%g" % p], ids = stage_times(lambda: tok.encode_to_numpy(data, np.uint16, dropout=p, seed=1), tok, reps)
            r["dropout_%g" % p]["tokens_vs_encode"] = ids.size / base.size
            r["dropout_%g" % p]["ms_total_vs_encode"] = r["dropout_%g" % p]["ms_total"] / r["encode"]["ms_total"]
        sl = bytes(data[: 16 << 20]).decode("utf-8", errors="ignore").encode()
        for p in (0.0, 0.1):
            t0 = time.perf_counter()
            otok.encode_bytes(sl, dropout=p, seed=1)
            r["oracle_cpu_16MB_p%g_MB_per_s" % p] = len(sl) / (time.perf_counter() - t0) / 1e6
        if shape == "tinystories":
            docs = bytes(data).decode("utf-8", errors="ignore").split(EOT)
            r["n_docs"] = len(docs)
            r["encode_batch"], _ = stage_times(lambda: tok.encode_batch_to_numpy(docs, np.uint16), tok, reps)
            r["encode_batch_dropout_0.1"], _ = stage_times(lambda: tok.encode_batch_to_numpy(docs, np.uint16, dropout=0.1, seed=1), tok, reps)
            del docs
        res["shapes"][shape] = r
        del data
        print(json.dumps(r, indent=1), flush=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
