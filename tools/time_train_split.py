"""GPU: device time per stage of train_bpe with and without split_special_tokens on the synthetic corpora, and how many learned
tokens hold a piece of the document separator in each mode.
usage: python tools/time_train_split.py [out.json] [reps]   (2 GiB TinyStories shape / vocab 10 000, 11 GB OWT shape / vocab 32 000)"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import _bootstrap  # noqa: F401,E402
import torch  # noqa: E402
from transformer_lm_b200 import _lib  # noqa: E402
from transformer_lm_b200.synth import SEED_OWT_TRAIN, SEED_TINY_TRAIN, synth_device  # noqa: E402
from transformer_lm_b200.train import train_bpe_on_bytes  # noqa: E402

EOT = "<|endoftext|>"
CASES = [("tinystories", SEED_TINY_TRAIN, 2 << 30, 10000), ("owt", SEED_OWT_TRAIN, 11 * 10**9 // 4096 * 4096, 32000)]
PIECES = [b"<|", b"endoftext", b"|>"]


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else None
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    ctx = _lib.default_context(0)
    p = torch.cuda.get_device_properties(0)
    res = {"device": p.name, "cases": []}
    try:
        import subprocess
        res["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                            capture_output=True, text=True).stdout.strip()
    except OSError:
        pass
    for shape, seed, n, vocab in CASES:
        t = torch.empty(n, dtype=torch.uint8, device="cuda")
        synth_device(shape, seed, n, t.data_ptr(), ctx=ctx)
        torch.cuda.synchronize()
        runs = {False: [], True: []}
        learned = {}
        for _ in range(reps):                    # the two modes alternate: same box, same moment
            for split in (False, True):
                v, m, st = train_bpe_on_bytes(None, vocab, [EOT], ctx=ctx, return_stats=True, device_ptr=t.data_ptr(), n_bytes=n,
                                              split_special_tokens=split)
                runs[split].append(st)
                toks = list(v.values())[257:]
                learned[split] = {pc.decode(): sum(pc in x for x in toks) for pc in PIECES}
        del t
        torch.cuda.empty_cache()
        case = {"shape": shape, "bytes": n, "vocab": vocab}
        for split in (False, True):
            key = "split" if split else "default"
            sts = runs[split]
            case[key] = {k: round(sorted(s[k] for s in sts)[len(sts) // 2], 2) for k in sts[0] if k.startswith("ms_")}
            case[key].update({k: sts[0][k] for k in ("n_pretokens", "n_unique", "merge_steps")})
            case[key]["learned_tokens_containing"] = learned[split]
        print(json.dumps(case))
        res["cases"].append(case)
    if out:
        with open(out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
