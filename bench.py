#!/usr/bin/env python3
"""Benchmark of the byte-level BPE hot path on B200 (contract and definitions: DESIGN.md, "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload train|train-tiny|encode] [--bytes B] [--vocab V] [--dump-outputs DIR]
    torchrun --nproc-per-node N bench.py --gpus N ...       # one rank per GPU, NCCL
    python bench.py --impl reference ...                    # the reference's own CPU path on a bounded sample

Default workload: BPE training on the 11 GB synthetic OWT-shaped corpus, vocab 32000, special token
<|endoftext|> (BASELINE.json configs[3]; the shape of perf/bpe/owt.py:4-8 in the reference).  One "step" is one
complete train_bpe over the corpus (pretokenise, count, exchange when N > 1, 31 743 merges).
  value  = corpus MB per second of a whole training run, text already resident in HBM, CUDA-event time
  e2e    = the same through the public API with the text in pinned HOST memory (H2D inside the timed region)
The line also carries
  "encode"      bulk encode of the 10 GB OWT-shaped text with the vocab just trained (BASELINE.json configs[4]);
  "train_tiny"  BPE training on the 2 GiB TinyStories-shaped corpus, vocab 10000 (BASELINE.json configs[2]);
  "same_slice"  the SAME bytes and vocab the CPU arms run (the reference arm's sample and a 64 MiB slice for the C
                port): GPU time, the CPU time measured in this run, and whether the outputs are identical;
  digests       merges_sha / ids_checksum, identical at every N (at N > 1 rank 0 also runs the unsharded path on the
                whole input and asserts equality).
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import pathlib
import subprocess
import sys
import tempfile
import threading
import time

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

SPECIALS = ["<|endoftext|>"]
L2_BYTES = 126 << 20
BLOCK = 4096

WORKLOADS = {
    # name: (shape, seed, default bytes, default vocab, description)
    "train": ("owt", 4321, 11e9, 32000, "BPE train, 11 GB synthetic OWT-shape corpus, vocab 32000, special <|endoftext|>"),
    "train-tiny": ("tinystories", 1234, 2 * 2**30, 10000, "BPE train, 2 GiB synthetic TinyStories-shape corpus, vocab 10000, special <|endoftext|>"),
    "encode": ("owt", 4322, 10e9, 32000, "bulk encode to uint16, 10 GB synthetic OWT-shape text, 32K vocab trained on the OWT-shape train corpus"),
}
# The two slices both arms run on identical bytes (prefixes of the workload's corpus: same generator and seed):
#   "ref":  what `--impl reference` times per step with the reference's own Python train_bpe (or the C port when
#           baseline/_ref is absent) -- a few MiB, because the Python reference needs seconds per MiB;
#   "port": a 64 MiB slice for the C port of the reference (oracle/bpe_oracle.c), about 10 s of one core.
SLICE_REF_BYTES, SLICE_PORT_BYTES, SLICE_VOCAB = 2 << 20, 64 << 20, 1000
ENC_SLICE_REF_BYTES, ENC_SLICE_PORT_BYTES = 1 << 20, 32 << 20


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="train", choices=list(WORKLOADS))
    ap.add_argument("--bytes", type=float, default=None, help="corpus size in bytes (default: the BASELINE config)")
    ap.add_argument("--encode-bytes", type=float, default=None, help="size of the encode text (default 10e9)")
    ap.add_argument("--vocab-train-bytes", type=float, default=1e9, help="--workload encode: slice of the train corpus the vocab is trained on")
    ap.add_argument("--vocab", type=int, default=None)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-encode", action="store_true", help="train workloads: skip the secondary encode measurement")
    ap.add_argument("--no-tiny", action="store_true", help="skip the TinyStories-shape training sub-measurement")
    ap.add_argument("--no-files", action="store_true", help="skip the file-level legs (train_bpe(path), encode_file) at N = 1")
    ap.add_argument("--no-slices", action="store_true", help="skip the same-slice legs")
    ap.add_argument("--no-unsharded-check", action="store_true", help="N > 1: do not re-run the unsharded path on rank 0")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float32 / float64): the trained vocab and merges, and "
                         "a fixed, seeded sample of the encoded ids (at N > 1 drawn from rank 0's shard, the start of the text)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    return args


def merges_sha(merges) -> str:
    h = hashlib.sha256()
    for a, b in merges:
        h.update(len(a).to_bytes(4, "little")); h.update(a); h.update(len(b).to_bytes(4, "little")); h.update(b)
    return h.hexdigest()[:16]


class ClockSampler:
    """Samples SM clocks and throttle reasons with nvidia-smi while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_gbs():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured copy bandwidth (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel: str, config: dict):
    """DRAM bytes (read + written) `kernel` moves per bench step, from the committed ncu capture of this configuration
    (profiles/r2_traffic.json: bytes of one launch x the launches a step makes), or None."""
    try:
        tj = json.loads((ROOT / "profiles" / "r2_traffic.json").read_text())
        kernel = kernel.split("<")[0]
        for e in tj["captures"]:
            if e["kernel"] == kernel and all(k in e["config"] and e["config"][k] == v for k, v in config.items()):
                return e["dram_bytes_per_step"], "%s; %d launch(es) per step" % (e["source"], e["launches_per_step"])
    except Exception:
        pass
    return None, None


def ncu_traffic_sum(kernels, config: dict):
    """Sum of ncu_traffic over several kernels (every captured instance of each, e.g. both k_enc_bpe_short shapes); None unless the
    first kernel of the list (the stage's dominant one) has a capture of this configuration."""
    try:
        tj = json.loads((ROOT / "profiles" / "r2_traffic.json").read_text())
        hit = [e for e in tj["captures"] if e["kernel"] in kernels and all(k in e["config"] and e["config"][k] == v for k, v in config.items())]
        if not any(e["kernel"] == kernels[0] for e in hit):
            return None, None
        names = sorted({e["kernel"] for e in hit})
        return sum(e["dram_bytes_per_step"] for e in hit), "sum over %s; %s" % (", ".join(names), "; ".join(sorted({e["source"] for e in hit})))
    except Exception:
        return None, None


# --dump-outputs: the arrays are a pure function of the bench arguments (seeded corpora, fixed sample seed), so two builds
# run with the same arguments can be compared file by file.
DUMP_LIMIT_BYTES = 64 << 20
DUMP_SAMPLE_IDS, DUMP_SAMPLE_SEED = 1 << 20, 20240601


def train_output_arrays(np, vocab, merges) -> dict:
    """train_bpe's (vocab, merges) as arrays: the ids of the vocab, the bytes of its entries in id order back to back with the
    offset of each entry's first byte, and every merge as the vocab ids of its two parts."""
    ids = sorted(vocab)
    toks = [vocab[i] for i in ids]
    offsets = np.zeros(len(toks) + 1, dtype=np.float64)
    np.cumsum([len(t) for t in toks], out=offsets[1:])
    inv = {t: i for i, t in vocab.items()}
    return {"train_vocab_ids": np.array(ids, dtype=np.float64),
            "train_vocab_bytes": np.frombuffer(b"".join(toks), dtype=np.uint8).astype(np.float32),
            "train_vocab_offsets": offsets,
            "train_merges": np.array([[inv[a], inv[b]] for a, b in merges], dtype=np.float64).reshape(-1, 2)}


def encode_output_arrays(np, torch, ids, n_ids: int) -> dict:
    """A fixed, seeded sample of the n_ids token ids in the device tensor ids (uint16): their positions, their values, and n_ids."""
    if n_ids <= DUMP_SAMPLE_IDS:
        pos = np.arange(n_ids, dtype=np.int64)
    else:
        pos = np.sort(np.random.default_rng(DUMP_SAMPLE_SEED).choice(n_ids, size=DUMP_SAMPLE_IDS, replace=False))
    vals = ids[:n_ids].view(torch.int16)[torch.from_numpy(pos).to(ids.device)].to(torch.int32) & 0xFFFF
    return {"encode_ids_sample_positions": pos.astype(np.float64), "encode_ids_sample": vals.cpu().numpy().astype(np.float32),
            "encode_n_ids": np.array([n_ids], dtype=np.float64)}


def write_outputs(np, out_dir: str, arrays: dict) -> None:
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ----------------------------------------------------------------------------------------------
# CPU arms: the reference's own Python implementation (baseline/_ref, installed from /root/reference in the build
# container, see DESIGN.md section 7) and its C port (oracle/bpe_oracle.c).  Host cores only; these functions never
# load the product's CUDA library (the input comes from oracle/libsynth_host.so).
# ----------------------------------------------------------------------------------------------
REF_DIR = ROOT / "baseline" / "_ref"
_REF_RUNNER = r'''
import json, logging, sys, time
sys.path.insert(0, sys.argv[1])
import models.tokenizer.train as T            # the unmodified reference, models/tokenizer/train.py
import models.tokenizer.tokenizer as K        # models/tokenizer/tokenizer.py
logging.disable(logging.CRITICAL)
T.tqdm = lambda x, *a, **k: x                 # (only silences the progress bar)
job = json.loads(sys.argv[2])
out = {}
if job["what"] == "train":
    import regex as re
    pat = re.compile(r"""'(?:[sdmt]|ll|ve|re)| ?\p{L}+| ?\p{N}+| ?[^\s\p{L}\p{N}]+|\s+(?!\S)|\s+""", re.UNICODE)
    t0 = time.perf_counter()
    freqs = T.extract_subword_frequencies(job["path"], set(job["specials"]), pat)      # train.py:16-28, timed on its own
    out["pretok_s"] = time.perf_counter() - t0
    out["unique_pretokens"] = len(freqs)
    del freqs
    times = []
    for i in range(job["warmup"] + job["steps"]):
        t0 = time.perf_counter()
        vocab, merges = T.train_bpe(job["path"], job["vocab"], job["specials"])        # train.py:142-231
        if i >= job["warmup"]:
            times.append(time.perf_counter() - t0)
    out["times"] = times
    out["merges"] = [[a.hex(), b.hex()] for a, b in merges]
    out["vocab_len"] = len(vocab)
else:
    vocab = {int(k): bytes.fromhex(v) for k, v in job["tok_vocab"].items()}
    merges = [(bytes.fromhex(a), bytes.fromhex(b)) for a, b in job["tok_merges"]]
    tok = K.Tokenizer(vocab, merges, job["specials"])
    text = open(job["path"], "rb").read().decode("utf-8")
    times = []
    for i in range(job["warmup"] + job["steps"]):
        t0 = time.perf_counter()
        ids = tok.encode(text)                                                         # tokenizer.py:111-138
        if i >= job["warmup"]:
            times.append(time.perf_counter() - t0)
    out["times"] = times
    import hashlib, array
    out["n_ids"] = len(ids)
    out["ids_sha"] = hashlib.sha256(array.array("q", ids).tobytes()).hexdigest()[:16]
print("REFJSON" + json.dumps(out))
'''


def reference_available() -> bool:
    return (REF_DIR / "models" / "tokenizer" / "train.py").exists()


def _run_reference_python(job: dict) -> dict:
    """Runs the reference's Python code in a fresh interpreter whose import path starts at baseline/_ref (its package is
    called `models`, like this repo's shim package: it must not be imported into this process)."""
    r = subprocess.run([sys.executable, "-c", _REF_RUNNER, str(REF_DIR), json.dumps(job)], capture_output=True, text=True, cwd=tempfile.gettempdir())
    for line in r.stdout.splitlines():
        if line.startswith("REFJSON"):
            return json.loads(line[7:])
    raise RuntimeError("reference run failed: " + r.stderr[-2000:])


def _slice_file(shape: str, seed: int, n_bytes: int) -> str:
    from oracle import synth
    d = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    path = os.path.join(d, "bpe_bench_%s_%d_%d.txt" % (shape, seed, n_bytes))
    if not os.path.exists(path) or os.path.getsize(path) != n_bytes:
        synth.synth_host(shape, seed, n_bytes).tofile(path)
    return path


def cpu_train_port(shape, seed, n_bytes, vocab):
    import _bootstrap  # noqa: F401
    from oracle import oracle, synth
    data = synth.synth_host(shape, seed, n_bytes).tobytes()
    t0 = time.perf_counter()
    vocab_d, merges = oracle.train_bpe_on_bytes(data, vocab, SPECIALS)
    return time.perf_counter() - t0, vocab_d, merges


def cpu_train_reference(shape, seed, n_bytes, vocab, steps=1, warmup=0):
    """The reference's Python train_bpe on the slice; returns (mean seconds, merges, detail)."""
    out = _run_reference_python({"what": "train", "path": _slice_file(shape, seed, n_bytes), "vocab": vocab, "specials": SPECIALS,
                                 "steps": steps, "warmup": warmup})
    merges = [(bytes.fromhex(a), bytes.fromhex(b)) for a, b in out["merges"]]
    return sum(out["times"]) / len(out["times"]), merges, out


def cpu_encode_port(tok_vocab, tok_merges, shape, seed, n_bytes):
    import _bootstrap  # noqa: F401
    from oracle import oracle, synth
    tok = oracle.OracleTokenizer(dict(tok_vocab), list(tok_merges), SPECIALS)
    data = synth.synth_host(shape, seed, n_bytes).tobytes()
    t0 = time.perf_counter()
    ids = tok.encode_bytes(data)
    return time.perf_counter() - t0, ids


def cpu_encode_reference(tok_vocab, tok_merges, shape, seed, n_bytes, steps=1, warmup=0):
    out = _run_reference_python({"what": "encode", "path": _slice_file(shape, seed, n_bytes), "specials": SPECIALS, "steps": steps, "warmup": warmup,
                                 "tok_vocab": {str(k): v.hex() for k, v in tok_vocab.items()}, "tok_merges": [[a.hex(), b.hex()] for a, b in tok_merges]})
    return sum(out["times"]) / len(out["times"]), out


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores.  It is single-threaded
    (SURVEY 2.1: no threads, no processes), so one core is all it can use.  Every step is a bounded sample of the workload: the
    first SLICE_REF_BYTES of the same corpus (same generator and seed) at vocab SLICE_VOCAB -- the b200 arm times exactly these
    bytes and this vocab too ("same_slice" on its line) and compares the merges.  The full configuration is out of reach of the
    CPU path (SURVEY 6); the line carries a LABELLED lower-bound extrapolation from the measured pretokenisation rate."""
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    shape, seed, nbytes, vocab, desc = WORKLOADS[args.workload]
    have_ref = reference_available()
    line_extra = {}
    if args.workload == "encode":
        # tokenizer of the slice: the C port's training result on the "ref" training slice (the b200 arm trains the same bytes on
        # the GPU and obtains the identical vocab, so both arms encode the same text with the same tokenizer)
        _, tv, tm = cpu_train_port("owt", 4321, SLICE_REF_BYTES, SLICE_VOCAB)
        if have_ref:
            n = ENC_SLICE_REF_BYTES
            sec, det = cpu_encode_reference(tv, tm, shape, seed, n, steps=args.steps, warmup=args.warmup)
            kind, what = "reference", "the reference's Python Tokenizer.encode (baseline/_ref/models/tokenizer/tokenizer.py:111-138)"
            sha_info = {"n_ids": det["n_ids"], "ids_sha": det["ids_sha"]}
        else:
            n = ENC_SLICE_PORT_BYTES
            times = []
            for i in range(args.warmup + args.steps):
                dt, ids = cpu_encode_port(tv, tm, shape, seed, n)
                if i >= args.warmup:
                    times.append(dt)
            sec = sum(times) / len(times)
            kind, what = "port", "oracle/bpe_oracle.c, the C port of Tokenizer.encode"
            sha_info = {"n_ids": int(ids.size), "ids_sha": hashlib.sha256(ids.astype("<i8").tobytes()).hexdigest()[:16]}
        metric = "bpe_encode_MBps"
        sample = "%s on the first %.1f MiB of the encode text (same generator and seed) with the vocab-%d tokenizer trained on the first %d MiB of the train corpus" % (
            what, n / 2**20, SLICE_VOCAB, SLICE_REF_BYTES >> 20)
        line_extra["same_slice"] = [dict(name="ref", text_bytes=n, seconds=round(sec, 4), MBps=round(n / 1e6 / sec, 4), kind=kind, **sha_info)]
    else:
        slice_vocab = args.vocab or SLICE_VOCAB
        same = []
        if have_ref:
            n = SLICE_REF_BYTES
            sec, merges, det = cpu_train_reference(shape, seed, n, slice_vocab, steps=args.steps, warmup=args.warmup)
            kind, what = "reference", "the reference's Python train_bpe (baseline/_ref/models/tokenizer/train.py:142-231)"
            pretok_rate = n / 1e6 / det["pretok_s"]
            same.append(dict(name="ref", corpus_bytes=n, vocab_size=slice_vocab, seconds=round(sec, 3), MBps=round(n / 1e6 / sec, 4), kind=kind,
                             merges_sha=merges_sha(merges), pretokenise_MBps=round(pretok_rate, 3)))
            # the C port on the bigger slice, once (not a timed step): the second point of comparison with the b200 arm
            psec, _, pm = cpu_train_port(shape, seed, SLICE_PORT_BYTES, slice_vocab)
            same.append(dict(name="port", corpus_bytes=SLICE_PORT_BYTES, vocab_size=slice_vocab, seconds=round(psec, 3),
                             MBps=round(SLICE_PORT_BYTES / 1e6 / psec, 4), kind="port", merges_sha=merges_sha(pm)))
            line_extra["extrapolation"] = {
                "labelled": "EXTRAPOLATION, not a measurement", "full_config_lower_bound_s": round(nbytes / 1e6 / pretok_rate, 1),
                "method": "full corpus bytes / the pretokenise+count rate of extract_subword_frequencies measured on the slice (%.2f MB/s); the merge loop "
                          "(O(live pairs) per merge, %d merges at the full vocab) comes on top" % (pretok_rate, (args.vocab or vocab) - 257)}
        else:
            n = SLICE_PORT_BYTES
            times = []
            for i in range(args.warmup + args.steps):
                dt, _, merges = cpu_train_port(shape, seed, n, slice_vocab)
                if i >= args.warmup:
                    times.append(dt)
            sec = sum(times) / len(times)
            kind, what = "port", "oracle/bpe_oracle.c, the C port of train_bpe (baseline/_ref is absent)"
            same.append(dict(name="port", corpus_bytes=n, vocab_size=slice_vocab, seconds=round(sec, 3), MBps=round(n / 1e6 / sec, 4), kind=kind,
                             merges_sha=merges_sha(merges)))
        metric = "bpe_train_MBps"
        sample = "%s on the first %d MiB of the corpus (same generator and seed) at vocab %d (%d merges)" % (what, n >> 20, slice_vocab, len(merges))
        line_extra["same_slice"] = same
    value = n / 1e6 / sec
    line = {
        "impl": "reference", "metric": metric, "value": round(value, 4), "unit": "MB/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(sec * 1e3, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": desc, "sample_bytes": n, "sample_vocab": SLICE_VOCAB if args.workload != "encode" else None,
                   "note": "a step of this arm is the bounded sample, not the full workload: compare with the b200 arm's same_slice, not with its headline"},
        "cpu_baseline": {"value": round(value, 4), "unit": "MB/s", "cores": 1, "kind": kind, "sample": sample, "host_cores_available": os.cpu_count()},
        "e2e": {"value": round(value, 4), "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    line.update(line_extra)
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------------------------
class DeviceShards:
    """Shard source for sharded_count over text this rank already holds in HBM (synthetic corpus blocks
    [b0 - left halo, b1 + right halo) of the global corpus) or in pinned host memory (data=...)."""

    def __init__(self, ptr, n_bytes, own_begin, own_end, at_start, at_end, base, data=None):
        self.d = dict(data=data, device_ptr=ptr, n_bytes=n_bytes, own_begin=own_begin, own_end=own_end, at_start=at_start, at_end=at_end, base=base)

    def load(self, rank, world, halo_right):
        return self.d

    def raise_decode_error(self, offset):
        raise UnicodeDecodeError("utf-8", b"", 0, 1, "synthetic corpus invalid at byte %d" % offset)


def make_shard(torch, ctx, shape, seed, total_bytes, rank, world, halo_blocks=64):
    from transformer_lm_b200.synth import synth_device
    nb = total_bytes // BLOCK
    b0, b1 = nb * rank // world, nb * (rank + 1) // world
    r0, r1 = max(0, b0 - 1), min(nb, b1 + halo_blocks)
    n = (r1 - r0) * BLOCK
    t = torch.empty(max(n, 1), dtype=torch.uint8, device="cuda")
    synth_device(shape, seed, n, t.data_ptr(), ctx=ctx, first_block=r0)
    torch.cuda.synchronize()
    return t, dict(n=n, own_begin=(b0 - r0) * BLOCK, own_end=(b1 - r0) * BLOCK, at_start=r0 == 0, at_end=r1 == nb, base=r0 * BLOCK)


def ids_checksum(torch, ids, n, first_index: int) -> int:
    """Position-weighted 64-bit checksum of ids[0:n] whose first token has global index first_index: additive over shards, so
    the sum over ranks at any N equals the checksum of the unsharded encode."""
    total = 0
    step = 1 << 27
    for lo in range(0, n, step):
        hi = min(n, lo + step)
        k = torch.arange(first_index + lo + 1, first_index + hi + 1, dtype=torch.int64, device=ids.device)
        w = (k * -7046029254386353131) ^ (k >> 7)          # (int64 arithmetic wraps: the weights are a fixed function of the index)
        total += int(((ids[lo:hi].to(torch.int64) + 1) * w).sum().item())
    return total & 0xFFFFFFFFFFFFFFFF


def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import _bootstrap  # noqa: F401
    from transformer_lm_b200 import _lib, sharded
    from transformer_lm_b200.synth import synth_device
    from transformer_lm_b200.tokenizer import Tokenizer
    from transformer_lm_b200.train import train_bpe_on_bytes

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local_rank)
    # one process per GPU: sit on the GPU's NUMA node before any page-locked buffer is allocated (best effort; reported on the line)
    numa = _lib.bind_to_gpu_numa_node(local_rank) if world > 1 and not os.environ.get("BPE_NO_NUMA_BIND") else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = _lib.Context(local_rank)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.use_stream(stream.cuda_stream)                           # library work, NCCL and the timing events share one stream
    L = _lib.lib()
    dev = torch.device("cuda", local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, steps):
        """K steps bracketed by barrier + synchronize, CUDA events on the stream everything runs on; max over ranks."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        out = []
        for _ in range(steps):
            out.append(fn())
        e1.record()
        barrier()
        wall = time.perf_counter() - t0
        return max_over_ranks(e0.elapsed_time(e1)) / steps, max_over_ranks(wall * 1e3) / steps, out

    peak, peak_src = measured_peak_gbs()

    # ------------------------------------------------------------------------------------------
    def measure_train(shape, seed, nbytes, vocab_size, steps, warmup, with_e2e, unsharded_check):
        """One training workload at `world` ranks: device-resident steps, e2e steps, digests.  Returns (dict, last result)."""
        text, meta = make_shard(torch, ctx, shape, seed, nbytes, rank, world)

        def train_step():
            if world == 1:
                return train_bpe_on_bytes(None, vocab_size, SPECIALS, ctx=ctx, return_stats=True, device_ptr=text.data_ptr(), n_bytes=meta["n"])
            counter = sharded.DeviceCounter(ctx)
            src = DeviceShards(text.data_ptr(), meta["n"], meta["own_begin"], meta["own_end"], meta["at_start"], meta["at_end"], meta["base"])
            t_a = time.perf_counter()
            out = sharded.sharded_count(counter, src, SPECIALS, None, True)
            assert out == "ok"
            torch.cuda.synchronize()
            t_b = time.perf_counter()
            v, m, st = counter.finish(vocab_size, SPECIALS, return_stats=True)
            st["ms_count_exchange_wall"] = (t_b - t_a) * 1e3
            if sharded.LAST_TIMES:
                st["exchange_profile_ms"] = {k: round(v, 2) for k, v in sharded.LAST_TIMES.items()}
            return v, m, st

        res = None
        for _ in range(warmup):
            res = train_step()
        launches0 = L.bpe_launch_count()
        sampler = ClockSampler(local_rank).start()
        ms_dev, ms_wall, outs = timed(train_step, steps)
        clocks = sampler.stop()
        launches = L.bpe_launch_count() - launches0
        res = outs[-1]
        merges = res[1]
        sha = merges_sha(merges)
        if world > 1:
            d = int(sha, 16) >> 4
            lo, hi = torch.tensor([d], device=dev), torch.tensor([d], device=dev)
            dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            assert int(lo) == int(hi), "ranks disagree on the merge list"
        stats = [o[2] for o in outs]

        def avg(key):
            vals = [s[key] for s in stats if key in s]
            return sum(vals) / len(vals) if vals else 0.0

        st = stats[-1]
        stages = {k: round(avg(k), 3) for k in ("ms_h2d", "ms_pretok", "ms_count", "ms_build", "ms_merge", "ms_total", "ms_count_exchange_wall")
                  if any(k in s for s in stats)}
        if "exchange_profile_ms" in st:
            stages["exchange_profile_ms"] = st["exchange_profile_ms"]
        local_bytes = meta["own_end"] - meta["own_begin"]
        out = {
            "ms_per_step": round(ms_dev, 3), "wall_ms_per_step": round(ms_wall, 3), "value": round(nbytes / 1e6 / (ms_dev / 1e3), 2),
            "merges": len(merges), "merges_sha": sha, "merge_steps": int(st["merge_steps"]),
            "stages_ms": stages, "gpu_launches": int(launches), "clocks": clocks, "local_bytes": int(local_bytes),
            "counts": {k: st[k] for k in ("n_pretokens", "n_unique", "n_symbols", "n_pairs_initial", "n_pairs_final", "log_records", "sum_live_pairs")},
            "_avg": {k: avg(k) for k in ("ms_pretok", "ms_count", "ms_build", "ms_merge")},
        }
        # ---- N > 1: the unsharded path on the whole corpus, on rank 0, must give the same merges ----
        if world > 1 and unsharded_check:
            ok = 1
            if rank == 0:
                full = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
                synth_device(shape, seed, nbytes, full.data_ptr(), ctx=ctx)
                _, m1 = train_bpe_on_bytes(None, vocab_size, SPECIALS, ctx=ctx, device_ptr=full.data_ptr(), n_bytes=nbytes)
                ok = int(m1 == merges)
                out["unsharded_merges_sha"] = merges_sha(m1)
                del full
            t = torch.tensor([ok], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            assert int(t) == 1, "sharded merges differ from the 1-GPU merges on the same corpus"
            out["unsharded_check"] = "rank 0 re-ran the 1-GPU path on the whole corpus: identical merges"
        # ---- end to end: text in pinned host memory, H2D inside the timed region, merges read back ----
        if with_e2e:
            n_loc = meta["n"]
            host = _lib.PinnedBuffer(n_loc)
            torch.from_numpy(host.array).copy_(text[:n_loc])
            torch.cuda.synchronize()

            def e2e_step():
                if world == 1:
                    return train_bpe_on_bytes(host.array, vocab_size, SPECIALS, ctx=ctx, return_stats=True)
                counter = sharded.DeviceCounter(ctx)
                src = DeviceShards(None, n_loc, meta["own_begin"], meta["own_end"], meta["at_start"], meta["at_end"], meta["base"], data=host.array)
                assert sharded.sharded_count(counter, src, SPECIALS, None, True) == "ok"
                return counter.finish(vocab_size, SPECIALS, return_stats=True)

            e2e_step()
            _, ms_wall2, outs2 = timed(e2e_step, steps)
            assert outs2[-1][1] == merges
            out["e2e"] = {"value": round(nbytes / 1e6 / (ms_wall2 / 1e3), 2), "unit": "MB/s", "h2d_bytes_per_step": int(n_loc),
                          "d2h_bytes_per_step": 8 * len(merges), "ms_per_step": round(ms_wall2, 3),
                          "api": "train_bpe_on_bytes(pinned host buffer) -> bpe_train (C ABI); wall clock, includes building the python vocab/merges"}
            host.free()
        del text
        torch.cuda.empty_cache()
        return out, res

    def parallelism(world_):
        return "1 GPU" if world_ == 1 else ("%d ranks: byte-range shards + halo, NCCL exchange of the count tables, pair-table all-reduce check, "
                                            "replicated merge loop" % world_)

    primary = args.workload
    is_train = primary != "encode"
    shape, seed, nbytes, vocab_size, desc = WORKLOADS[primary]
    vocab_size = args.vocab or vocab_size
    line = {}
    train_res = None
    dumps = {}

    # ======================= training =======================
    if is_train:
        nbytes = int(args.bytes or nbytes) // BLOCK * BLOCK
        m, train_res = measure_train(shape, seed, nbytes, vocab_size, args.steps, args.warmup, not args.no_e2e, not args.no_unsharded_check)
        if args.dump_outputs:
            dumps.update(train_output_arrays(np, train_res[0], train_res[1]))
        avg = m.pop("_avg")
        merge_ms, pretok_ms, count_ms = avg["ms_merge"], avg["ms_pretok"], avg["ms_count"]
        local_bytes = m["local_bytes"]
        cfg_key = {"corpus_bytes": nbytes, "vocab_size": vocab_size, "shape": shape, "seed": seed, "n_gpus": world}

        def hbm_kernel(name, alg_bytes, ms, note):
            tr, src = ncu_traffic(name, cfg_key)
            gbs = alg_bytes / 1e9 / (ms / 1e3) if ms else None
            return {"bound": "hbm", "algorithmic_bytes": alg_bytes, "ms": round(ms, 3), "achieved": round(gbs, 1) if gbs else None, "peak": peak, "unit": "GB/s",
                    "frac": round(gbs / peak, 4) if gbs else None, "traffic": tr, "traffic_source": src, "note": note}

        tr_merge, tr_src = ncu_traffic("k_merge_loop", cfg_key)
        dram_gbs = tr_merge / 1e9 / (merge_ms / 1e3) if tr_merge and merge_ms else None
        roofline = {
            # The dominant kernel is LATENCY-bound, not HBM-bound: sequential grid steps of two grid barriers and ~10 dependent memory
            # round trips each over tables that mostly sit in L2.  Its numbers to drive are us per merge / per step; `achieved` is the
            # DRAM traffic ncu measured for this launch divided by its duration (null without a committed capture of this configuration).
            "bound": "latency", "kernel": "k_merge_loop (one persistent cooperative launch, %d merges in %d grid steps)" % (m["merges"], m["merge_steps"]),
            "achieved": round(dram_gbs, 1) if dram_gbs else None, "peak": peak, "unit": "GB/s", "frac": round(dram_gbs / peak, 4) if dram_gbs else None,
            "traffic": tr_merge, "traffic_source": tr_src, "peak_source": peak_src,
            "ms": round(merge_ms, 3), "share_of_step": round(merge_ms / m["ms_per_step"], 4) if m["ms_per_step"] else None,
            "us_per_merge": round(1e3 * merge_ms / max(m["merges"], 1), 3), "us_per_grid_step": round(1e3 * merge_ms / max(m["merge_steps"], 1), 3),
            "merges_per_grid_step": round(m["merges"] / max(m["merge_steps"], 1), 2), "grid_barrier_floor_us": 1.2,
            "hbm_kernels": {
                "k_pretok_flags": hbm_kernel("k_pretok_flags", local_bytes * 1.125, pretok_ms, "N text bytes read + N/8 flag bytes written; stage time"),
                "count stage (k_count_pretokens)": hbm_kernel("k_count_pretokens", local_bytes * 1.125, count_ms,
                                                             "N text bytes + N/8 flag bytes read once (table traffic is overhead, SURVEY 8d); stage time incl. table growth and the hot-table builds"),
            },
        }
        line = {
            "metric": "bpe_train_MBps", "value": m["value"], "unit": "MB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": m["ms_per_step"], "wall_ms_per_step": m["wall_ms_per_step"], "train_wall_s": round(m["wall_ms_per_step"] / 1e3, 4),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": desc if not args.bytes else desc + " [--bytes %d]" % nbytes, "corpus_bytes": nbytes, "vocab_size": vocab_size,
                       "merges": m["merges"], "shape": shape, "seed": seed,
                       "l2_policy": "per-rank input (%.2f GB) larger than L2 (126 MB)" % (local_bytes / 1e9) if local_bytes > L2_BYTES else "input smaller than L2",
                       "unicode_tables": L.bpe_unicode_table_source().decode(), "parallelism": parallelism(world)},
            "merges_sha": m["merges_sha"], "stages_ms": m["stages_ms"], "counts": m["counts"],
            "roofline": roofline, "gpu_launches": m["gpu_launches"], "clocks": m["clocks"],
        }
        for k in ("unsharded_check", "unsharded_merges_sha", "e2e"):
            if k in m:
                line[k] = m[k]
        if world > 1:
            # strong scaling with a replicated tail: build + merge loop run on every rank (DESIGN.md section 6), only pretokenise + count shard
            try:
                rep = float(m["stages_ms"]["ms_build"]) + float(m["stages_ms"]["ms_merge"])
                line["scaling_note"] = {"replicated_ms": round(rep, 3), "sharded_ms": round(float(m["ms_per_step"]) - rep, 3),
                                        "amdahl": "build + merge loop (replicated_ms) run replicated: the step cannot go below them at any N, so the speed-up "
                                                  "over the 1-GPU step T1 is bounded by T1 / (replicated_ms + (T1 - replicated_ms) / N)"}
            except Exception:
                pass

        # ---- BASELINE.json configs[2]: TinyStories shape, 2 GiB, vocab 10000 ----
        if primary == "train" and not args.no_tiny and not args.bytes:
            t_shape, t_seed, t_bytes, t_vocab, t_desc = WORKLOADS["train-tiny"]
            tm, _ = measure_train(t_shape, t_seed, int(t_bytes) // BLOCK * BLOCK, t_vocab, args.steps, max(1, min(args.warmup, 3)),
                                  not args.no_e2e, not args.no_unsharded_check)
            tavg = tm.pop("_avg")
            tm.update({"metric": "bpe_train_MBps", "unit": "MB/s", "config": {"workload": t_desc, "corpus_bytes": int(t_bytes), "vocab_size": t_vocab,
                                                                                 "shape": t_shape, "seed": t_seed, "parallelism": parallelism(world)},
                       "us_per_merge": round(1e3 * tavg["ms_merge"] / max(tm["merges"], 1), 3),
                       "us_per_grid_step": round(1e3 * tavg["ms_merge"] / max(tm["merge_steps"], 1), 3)})
            line["train_tiny"] = tm

    # ======================= encoding =======================
    if (not is_train) or not args.no_encode:
        e_shape, e_seed, e_bytes, _, e_desc = WORKLOADS["encode"]
        e_bytes = int(args.encode_bytes or (args.bytes if not is_train and args.bytes else e_bytes)) // BLOCK * BLOCK
        if train_res is None:
            vt_bytes = int(args.vocab_train_bytes) // BLOCK * BLOCK
            tt = torch.empty(vt_bytes, dtype=torch.uint8, device="cuda")
            synth_device("owt", 4321, vt_bytes, tt.data_ptr(), ctx=ctx)
            train_res = train_bpe_on_bytes(None, vocab_size, SPECIALS, ctx=ctx, return_stats=True, device_ptr=tt.data_ptr(), n_bytes=vt_bytes)
            del tt
            vocab_src = "trained on the first %.2f GB of the OWT-shape train corpus" % (vt_bytes / 1e9)
        else:
            vocab_src = "the vocab trained above"
        tok = Tokenizer(dict(train_res[0]), list(train_res[1]), SPECIALS, ctx=ctx)
        h = tok._device_tok()
        etext, emeta = make_shard(torch, ctx, e_shape, e_seed, e_bytes, rank, world, halo_blocks=256)
        # shards are cut at exact boundaries (the product's rule, sharded_encode.first_exact_cut: the start of a special-token
        # occurrence -- Tokenizer.segment splits there first, tokenizer.py:63-66 -- else a lone space between ASCII non-spaces)
        from transformer_lm_b200.sharded_encode import first_exact_cut
        sp_bytes = [s.encode() for s in SPECIALS]

        def peek_dev(a, b):
            return etext[a:b].cpu().numpy().tobytes()

        lo = emeta["own_begin"] if rank == 0 else first_exact_cut(peek_dev, emeta["n"], sp_bytes, emeta["own_begin"])
        hi = emeta["own_end"] if rank == world - 1 else first_exact_cut(peek_dev, emeta["n"], sp_bytes, emeta["own_end"])
        n_loc = hi - lo
        out = torch.empty(max(n_loc, 1), dtype=torch.uint16, device="cuda")
        src_ptr = etext.data_ptr() + lo
        enc_stats = []

        def encode_step():
            # every step does the whole job: the pretoken -> ids cache is dropped first, so all BPE merges are recomputed
            ctx.check(L.bpe_tok_cache_reset(h))
            n_out, stt = C.c_uint64(0), _lib.EncodeStats()
            ctx.check(L.bpe_encode_dev(h, C.c_void_p(src_ptr), n_loc, _lib.DTYPE_U16, C.c_void_p(out.data_ptr()), out.numel(), C.byref(n_out), C.byref(stt)))
            enc_stats.append(stt.as_dict())
            return n_out.value

        for _ in range(max(args.warmup, 1)):
            encode_step()
        enc_stats.clear()
        l0 = L.bpe_launch_count()
        sampler = ClockSampler(local_rank).start()
        ems_dev, ems_wall, n_tok = timed(encode_step, args.steps)
        eclocks = sampler.stop()
        e_launches = L.bpe_launch_count() - l0
        tokens_local = n_tok[-1]
        if args.dump_outputs and rank == 0:
            dumps.update(encode_output_arrays(np, torch, out, tokens_local))
        tok_total, bytes_total, first_index = tokens_local, n_loc, 0
        if world > 1:
            t = torch.tensor([tokens_local, n_loc], dtype=torch.int64, device=dev)
            allt = torch.empty(world * 2, dtype=torch.int64, device=dev)
            dist.all_gather_into_tensor(allt, t)
            allt = allt.view(world, 2).cpu()
            tok_total, bytes_total = int(allt[:, 0].sum()), int(allt[:, 1].sum())
            first_index = int(allt[:rank, 0].sum())
            assert bytes_total == e_bytes, (bytes_total, e_bytes)
        csum = ids_checksum(torch, out, tokens_local, first_index)
        if world > 1:
            parts = torch.tensor([csum & 0xFFFFFFFF, csum >> 32], dtype=torch.int64, device=dev)
            dist.all_reduce(parts)
            csum = (int(parts[0]) + (int(parts[1]) << 32)) & 0xFFFFFFFFFFFFFFFF

        def eavg(key):
            return sum(s[key] for s in enc_stats) / len(enc_stats)

        alg = n_loc + 2.0 * tokens_local                       # text read once + one uint16 per token (SURVEY 8d)
        dom = max(("ms_pretok", "ms_lookup", "ms_bpe", "ms_emit"), key=eavg)
        ecfg_key = {"text_bytes": e_bytes, "n_gpus": world}
        stage_alg = {"ms_pretok": n_loc * 1.125, "ms_lookup": float(n_loc), "ms_bpe": None, "ms_emit": 2.0 * tokens_local}
        stage_kernels = {"ms_pretok": ["k_pretok_flags", "k_special_candidates", "k_special_resolve", "k_popc_words16"],
                         "ms_lookup": ["k_enc_lookup"], "ms_emit": ["k_enc_scan_emit"]}
        tr_all, tr_all_src = ncu_traffic_sum(["k_enc_lookup", "k_pretok_flags", "k_special_candidates", "k_special_resolve", "k_popc_words16",
                                              "k_enc_bpe_short", "k_enc_bpe", "k_enc_scan_emit"], ecfg_key)
        hbm_stages = {}
        for k, kern in (("ms_pretok", "k_pretok_flags<1> + special-token passes"), ("ms_lookup", "k_enc_lookup"), ("ms_emit", "k_enc_scan_emit")):
            ms_k = eavg(k)
            tr, src = ncu_traffic_sum(stage_kernels[k], ecfg_key)
            gbs = stage_alg[k] / 1e9 / (ms_k / 1e3) if ms_k else None
            hbm_stages[kern] = {"algorithmic_bytes": stage_alg[k], "ms": round(ms_k, 3), "achieved": round(gbs, 1) if gbs else None,
                                "frac": round(gbs / peak, 4) if gbs else None, "traffic": tr, "traffic_source": src}
        enc = {
            "metric": "bpe_encode_MBps", "value": round(e_bytes / 1e6 / (ems_dev / 1e3), 2), "unit": "MB/s", "ms_per_step": round(ems_dev, 3),
            "config": {"workload": e_desc if e_bytes == 10e9 else e_desc + " [%d bytes]" % e_bytes, "text_bytes": e_bytes, "vocab": vocab_src,
                       "tokens": tok_total, "bytes_per_token": round(e_bytes / max(tok_total, 1), 3), "cache": "pretoken cache reset at the start of every step",
                       "parallelism": "1 GPU" if world == 1 else "%d ranks, shards cut at <|endoftext|>, no data collective" % world},
            "ids_checksum": "%016x" % csum,
            "stages_ms": {k: round(eavg(k), 3) for k in ("ms_h2d", "ms_pretok", "ms_lookup", "ms_bpe", "ms_emit", "ms_total")},
            "new_unique_pretokens": int(eavg("cache_new_unique")), "pretokens": int(eavg("n_pretokens")),
            "roofline": {"bound": "hbm", "kernel": "whole encode pipeline (flags, lookup, bpe, fused scan+emit); slowest stage: " + dom,
                         "achieved": round(alg / 1e9 / (ems_dev / 1e3), 1), "peak": peak, "unit": "GB/s",
                         "frac": round(alg / 1e9 / (ems_dev / 1e3) / peak, 4), "traffic": tr_all, "traffic_source": tr_all_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg, "algorithmic_bytes_definition": "N text bytes read once + 2 B per token written",
                         "stages": hbm_stages},
            "gpu_launches": int(e_launches), "clocks": eclocks,
        }
        # ---- N > 1: rank 0 encodes the WHOLE text on one GPU; token count and checksum must match the sharded run ----
        if world > 1 and not args.no_unsharded_check:
            ok = 1
            if rank == 0:
                del out
                full = torch.empty(e_bytes, dtype=torch.uint8, device="cuda")
                synth_device(e_shape, e_seed, e_bytes, full.data_ptr(), ctx=ctx)
                fout = torch.empty(e_bytes // 2, dtype=torch.uint16, device="cuda")
                ctx.check(L.bpe_tok_cache_reset(h))
                n_out = C.c_uint64(0)
                ctx.check(L.bpe_encode_dev(h, C.c_void_p(full.data_ptr()), e_bytes, _lib.DTYPE_U16, C.c_void_p(fout.data_ptr()), fout.numel(), C.byref(n_out), None))
                c1 = ids_checksum(torch, fout, n_out.value, 0)
                ok = int(n_out.value == tok_total and c1 == csum)
                enc["unsharded_ids_checksum"] = "%016x" % c1
                del full, fout
                out = torch.empty(max(n_loc, 1), dtype=torch.uint16, device="cuda")
            t = torch.tensor([ok], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            assert int(t) == 1, "sharded encode differs from the 1-GPU encode of the same text"
            enc["unsharded_check"] = "rank 0 re-encoded the whole text on one GPU: identical token count and checksum"
        if not args.no_e2e:
            hbuf = _lib.PinnedBuffer(n_loc)
            torch.from_numpy(hbuf.array).copy_(etext[lo:hi])
            hout = _lib.PinnedBuffer(2 * (tokens_local + 1024))
            torch.cuda.synchronize()
            out_view = hout.array.view(np.uint16)

            def e2e_encode():
                ctx.check(L.bpe_tok_cache_reset(h))
                n_out = C.c_uint64(0)
                ctx.check(L.bpe_encode(h, _lib.ptr(hbuf.array), n_loc, _lib.DTYPE_U16, _lib.ptr(out_view), out_view.size, C.byref(n_out), None))
                return n_out.value

            e2e_encode()
            _, ems2, n2 = timed(e2e_encode, args.steps)
            assert n2[-1] == tokens_local
            enc["e2e"] = {"value": round(e_bytes / 1e6 / (ems2 / 1e3), 2), "unit": "MB/s", "h2d_bytes_per_step": int(n_loc),
                          "d2h_bytes_per_step": int(2 * tokens_local), "ms_per_step": round(ems2, 3),
                          "per_gpu_pcie_GBps": round((n_loc + 2 * tokens_local) / 1e9 / (ems2 / 1e3), 2),
                          "api": "bpe_encode (C ABI) with pinned host text in, pinned host uint16 ids out; wall clock"}
            hbuf.free(); hout.free()
        del etext
        if is_train:
            line["encode"] = enc
        else:
            line = {"metric": enc["metric"], "value": enc["value"], "unit": "MB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                    "ms_per_step": enc["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8",
                    "data": "synthetic", "config": enc["config"], "ids_checksum": enc["ids_checksum"], "stages_ms": enc["stages_ms"],
                    "roofline": enc["roofline"], "gpu_launches": enc["gpu_launches"], "clocks": enc["clocks"]}
            for k in ("e2e", "unsharded_check"):
                if k in enc:
                    line[k] = enc[k]

    # ======================= file-level legs (N = 1): train_bpe(path) and encode_file(path -> .bin), SURVEY 8f rows 1-2 =======================
    if world == 1 and is_train and not args.no_files and not args.bytes:
        import shutil
        import tempfile
        from transformer_lm_b200.train import train_bpe as train_bpe_path
        from transformer_lm_b200.encode_file import encode_file
        from transformer_lm_b200.tokenizer import Tokenizer
        f_shape, f_seed, f_bytes, f_vocab, _ = WORKLOADS["train-tiny"]
        f_bytes = int(f_bytes) // BLOCK * BLOCK
        d = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > 3 * f_bytes else tempfile.gettempdir()
        fdir = tempfile.mkdtemp(prefix="bpe_bench_", dir=d)
        try:
            src = os.path.join(fdir, "corpus.txt")
            t = torch.empty(f_bytes, dtype=torch.uint8, device="cuda")
            synth_device(f_shape, f_seed, f_bytes, t.data_ptr(), ctx=ctx)
            t.cpu().numpy().tofile(src)
            del t
            walls = []
            for _ in range(1 + args.steps):      # (first run: page cache and buffer pools warm up)
                t0 = time.time()
                f_vocab_d, f_merges = train_bpe_path(src, f_vocab, SPECIALS, ctx=ctx)
                walls.append(time.time() - t0)
            f_sha = merges_sha(f_merges)
            tok_f = Tokenizer(f_vocab_d, f_merges, SPECIALS, ctx=ctx)
            dst = os.path.join(fdir, "tokens.bin")
            ewalls = []
            for _ in range(args.steps):
                ctx.check(L.bpe_tok_cache_reset(tok_f._device_tok()))
                t0 = time.time()
                n_tok_f = encode_file(tok_f, src, dst, np.uint16)
                ewalls.append(time.time() - t0)
            assert os.path.getsize(dst) == 2 * n_tok_f
            tiny_sha = line.get("train_tiny", {}).get("merges_sha")
            line["files"] = {
                "note": "the reference's file-level entry points on a %.2f GB TinyStories-shape file in %s (page cache warm): wall clock, "
                        "includes reading the file, H2D, kernels, D2H and writing the .bin" % (f_bytes / 1e9, d),
                "train_bpe(path)": {"wall_s": round(min(walls[1:]), 4), "MBps": round(f_bytes / 1e6 / min(walls[1:]), 1), "merges_sha": f_sha,
                                    "same_merges_as_device_resident_run": (f_sha == tiny_sha) if tiny_sha else None,
                                    "api": "transformer_lm_b200.train.train_bpe(path, 10000, ['<|endoftext|>']) (streamed ingest: reader threads -> page-locked buffers -> bpe_count_add_shard)"},
                "encode_file(path -> .bin)": {"wall_s": round(min(ewalls), 4), "MBps": round(f_bytes / 1e6 / min(ewalls), 1), "tokens": int(n_tok_f),
                                               "api": "transformer_lm_b200.encode_file.encode_file(tokenizer, path, out.bin, uint16) (reader thread -> bpe_encode -> writer thread)"},
            }
        except Exception as e:                   # (no room in the scratch directory, ...: the leg is informative, the headline stands)
            line["files"] = {"error": "%s: %s" % (type(e).__name__, e)}
        finally:
            shutil.rmtree(fdir, ignore_errors=True)

    # ======================= same bytes, same vocab as the CPU arms (N = 1) =======================
    if world == 1 and not args.no_slices:
        s_shape, s_seed = (shape, seed) if is_train else ("owt", 4321)
        slices = []
        slice_results = {}
        for name, n_s in (("ref", SLICE_REF_BYTES), ("port", SLICE_PORT_BYTES)):
            t = torch.empty(n_s, dtype=torch.uint8, device="cuda")
            synth_device(s_shape, s_seed, n_s, t.data_ptr(), ctx=ctx)
            host = _lib.PinnedBuffer(n_s)
            torch.from_numpy(host.array).copy_(t)
            torch.cuda.synchronize()

            def dev_step():
                return train_bpe_on_bytes(None, SLICE_VOCAB, SPECIALS, ctx=ctx, device_ptr=t.data_ptr(), n_bytes=n_s)

            def host_step():
                return train_bpe_on_bytes(host.array, SLICE_VOCAB, SPECIALS, ctx=ctx)

            dev_step(); host_step()
            ms_d, _, o = timed(dev_step, args.steps)
            _, ms_h, o2 = timed(host_step, args.steps)
            assert o[-1][1] == o2[-1][1]
            slice_results[name] = o[-1]
            slices.append({"name": name, "corpus_bytes": n_s, "vocab_size": SLICE_VOCAB, "shape": s_shape, "seed": s_seed,
                           "gpu_ms": round(ms_d, 3), "gpu_MBps": round(n_s / 1e6 / (ms_d / 1e3), 2),
                           "gpu_e2e_ms": round(ms_h, 3), "gpu_e2e_MBps": round(n_s / 1e6 / (ms_h / 1e3), 2), "merges_sha": merges_sha(o[-1][1])})
            host.free()
            del t
        line["same_slice"] = slices
        # the encode slice: the encode text's prefix with the vocab of the "ref" training slice (what the reference arm encodes)
        sv, sm = slice_results["ref"]
        stok = Tokenizer(dict(sv), list(sm), SPECIALS, ctx=ctx)
        enc_slices = []
        for name, n_s in (("ref", ENC_SLICE_REF_BYTES), ("port", ENC_SLICE_PORT_BYTES)):
            from oracle import synth as osynth                   # (host generator of the CPU arms: identical bytes, tests/test_synth.py)
            data = osynth.synth_host("owt", 4322, n_s)
            stok.encode_to_numpy(data, np.uint16)
            dt = 1e9
            for _ in range(args.steps):                          # best of the warm calls (the first ones may still grow the cache tables)
                t0 = time.perf_counter()
                ids = stok.encode_to_numpy(data, np.uint16)
                dt = min(dt, time.perf_counter() - t0)
            enc_slices.append({"name": name, "text_bytes": n_s, "gpu_e2e_ms": round(dt * 1e3, 3), "gpu_e2e_MBps": round(n_s / 1e6 / dt, 2), "n_ids": int(ids.size),
                               "ids_sha": hashlib.sha256(ids.astype("<i8").tobytes()).hexdigest()[:16],
                               "tokenizer": "vocab %d trained on the first %d MiB of the train corpus" % (SLICE_VOCAB, SLICE_REF_BYTES >> 20),
                               "cache": "warm pretoken cache (best of %d calls after a first one)" % args.steps})
        line["same_slice_encode"] = enc_slices

        # ======================= CPU baseline: the CPU arms on those slices, timed in this run (rank 0, N = 1) =======================
        if not args.no_cpu_baseline:
            cores = os.cpu_count()
            by_name = {s["name"]: s for s in slices}
            psec, _, pm = cpu_train_port(s_shape, s_seed, SLICE_PORT_BYTES, SLICE_VOCAB)
            by_name["port"].update({"cpu_seconds": round(psec, 3), "cpu_MBps": round(SLICE_PORT_BYTES / 1e6 / psec, 4), "cpu_kind": "port",
                                    "outputs_identical": pm == slice_results["port"][1],
                                    "ratio_device_resident": round(psec * 1e3 / by_name["port"]["gpu_ms"], 1), "ratio_e2e": round(psec * 1e3 / by_name["port"]["gpu_e2e_ms"], 1)})
            assert by_name["port"]["outputs_identical"], "GPU merges differ from the C port on the 64 MiB slice"
            if reference_available():
                rsec, rm, det = cpu_train_reference(s_shape, s_seed, SLICE_REF_BYTES, SLICE_VOCAB)
                by_name["ref"].update({"cpu_seconds": round(rsec, 3), "cpu_MBps": round(SLICE_REF_BYTES / 1e6 / rsec, 4), "cpu_kind": "reference (python)",
                                       "outputs_identical": rm == slice_results["ref"][1], "reference_pretokenise_MBps": round(SLICE_REF_BYTES / 1e6 / det["pretok_s"], 3),
                                       "ratio_device_resident": round(rsec * 1e3 / by_name["ref"]["gpu_ms"], 1), "ratio_e2e": round(rsec * 1e3 / by_name["ref"]["gpu_e2e_ms"], 1)})
                assert by_name["ref"]["outputs_identical"], "GPU merges differ from the Python reference on the slice"
                kind, val, sample = "reference", SLICE_REF_BYTES / 1e6 / rsec, (
                    "the reference's Python train_bpe (baseline/_ref, 1 thread: it has no other) on the first %d MiB of the corpus at vocab %d: %.1f s; "
                    "the GPU on the same bytes and vocab: %.1f ms, identical merges" % (SLICE_REF_BYTES >> 20, SLICE_VOCAB, rsec, by_name["ref"]["gpu_ms"]))
            else:
                kind, val, sample = "port", SLICE_PORT_BYTES / 1e6 / psec, (
                    "oracle/bpe_oracle.c (C port of the reference's train_bpe, 1 thread like the reference) on the first %d MiB of the corpus at vocab %d: "
                    "%.1f s; the GPU on the same bytes and vocab: %.1f ms, identical merges" % (SLICE_PORT_BYTES >> 20, SLICE_VOCAB, psec, by_name["port"]["gpu_ms"]))
            cpu_b = {"value": round(val, 4), "unit": "MB/s", "cores": 1, "kind": kind, "sample": sample, "host_cores_available": cores}
            # encode slices on the CPU
            eby = {s["name"]: s for s in enc_slices}
            esec, eids = cpu_encode_port(sv, sm, "owt", 4322, ENC_SLICE_PORT_BYTES)
            esha = hashlib.sha256(eids.astype("<i8").tobytes()).hexdigest()[:16]
            eby["port"].update({"cpu_seconds": round(esec, 3), "cpu_MBps": round(ENC_SLICE_PORT_BYTES / 1e6 / esec, 4), "cpu_kind": "port", "outputs_identical": esha == eby["port"]["ids_sha"]})
            assert eby["port"]["outputs_identical"], "GPU ids differ from the C port on the encode slice"
            enc_cpu = {"value": eby["port"]["cpu_MBps"], "unit": "MB/s", "cores": 1, "kind": "port",
                       "sample": "oracle/bpe_oracle.c Tokenizer.encode port on the first %d MiB of the encode text, vocab-%d tokenizer: %.1f s" % (ENC_SLICE_PORT_BYTES >> 20, SLICE_VOCAB, esec),
                       "host_cores_available": cores}
            if reference_available():
                rsec, det = cpu_encode_reference(sv, sm, "owt", 4322, ENC_SLICE_REF_BYTES)
                eby["ref"].update({"cpu_seconds": round(rsec, 3), "cpu_MBps": round(ENC_SLICE_REF_BYTES / 1e6 / rsec, 4), "cpu_kind": "reference (python)",
                                   "outputs_identical": det["ids_sha"] == eby["ref"]["ids_sha"] and det["n_ids"] == eby["ref"]["n_ids"]})
                assert eby["ref"]["outputs_identical"], "GPU ids differ from the Python reference on the encode slice"
                enc_cpu = {"value": eby["ref"]["cpu_MBps"], "unit": "MB/s", "cores": 1, "kind": "reference",
                           "sample": "the reference's Python Tokenizer.encode (baseline/_ref) on the first %d MiB of the encode text, vocab-%d tokenizer: %.1f s, identical ids" % (
                               ENC_SLICE_REF_BYTES >> 20, SLICE_VOCAB, rsec), "host_cores_available": cores}
            if is_train:
                line["cpu_baseline"] = cpu_b
                if "encode" in line:
                    line["encode"]["cpu_baseline"] = enc_cpu
            else:
                line["cpu_baseline"] = enc_cpu
    if numa is not None:
        # every rank's binding result, gathered on rank 0 (host-side objects: one small all_gather_object)
        allnuma = [None] * world
        dist.all_gather_object(allnuma, numa)
        line["numa_binding"] = {"note": "each rank binds itself to the CPUs of its GPU's NUMA node before allocating page-locked buffers (best effort)",
                                "ranks": allnuma}
    if args.dump_outputs and rank == 0:
        write_outputs(np, args.dump_outputs, dumps)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
