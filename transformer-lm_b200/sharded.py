"""Multi-GPU BPE training: one process per GPU, corpus sharded by byte range, one exchange step, replicated merge loop.

The reference is single-process (models/tokenizer/train.py:142-231); SURVEY 8(e) derives the sharding:
  * pretoken starts are a local function of <= 4 code points of left and <= 2 of right context, so a rank that
    reads its byte range plus a small halo finds exactly the pretokens that START in its range;
  * extract_subword_frequencies (train.py:16-28) is a sum over occurrences, so per-rank (word, count) tables add;
  * the merge loop (train.py:183-228) depends only on the multiset {(word, count)} (SURVEY A-8), so every rank
    runs it on the merged table and obtains the identical result (checked with a digest all-reduce).
The exchange is an all-gather of the per-rank tables (NCCL over NVLink when the tensors live on the GPU) plus an
all-reduce of the dense 256x256 byte-pair table used as a linearity check.

`sharded_count` holds the host logic (cuts, halos, error agreement, exchange) and talks to the device through a
small counter interface, so the same code runs under `gloo` on CPU tensors in the tests (with a checker-backed
counter there) and under `nccl` on CUDA tensors in the product (`DeviceCounter`, C ABI).
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
from typing import List

import numpy as np

from . import _lib
from .vocab import Vocab

HALO_LEFT = 64                  # >= 4 code points of left context
HALO_RIGHT = 64 << 10           # first guess; grown when a pretoken runs past it
NO_ERROR = (1 << 62)


# ---- byte-range planning -----------------------------------------------------------------------------
def _is_continuation(b: int) -> bool:
    return (b & 0xC0) == 0x80


def align_cut(peek, pos: int, size: int) -> int:
    """Largest position <= pos that does not split a UTF-8 sequence (at most 3 bytes back).
    `peek(lo, hi)` returns the file bytes [lo, hi)."""
    if pos <= 0 or pos >= size:
        return max(0, min(pos, size))
    window = peek(max(0, pos - 3), pos + 1)
    k = len(window) - 1                          # index of byte `pos`
    back = 0
    while back < 3 and k - back >= 0 and _is_continuation(window[k - back]):
        back += 1
    return pos - back


def plan_shard(peek, size: int, rank: int, world: int, halo_right: int = HALO_RIGHT):
    """(lo, hi, read_lo, read_hi): rank owns the pretokens starting in [lo, hi) and reads [read_lo, read_hi)."""
    lo = align_cut(peek, size * rank // world, size)
    hi = size if rank == world - 1 else align_cut(peek, size * (rank + 1) // world, size)
    read_lo = align_cut(peek, max(0, lo - HALO_LEFT), size)
    read_hi = align_cut(peek, min(size, hi + halo_right), size)
    return lo, hi, read_lo, read_hi


# ---- device counter (the product) -----------------------------------------------------------------------
class DeviceCounter:
    """Per-rank pretoken count table on the GPU (bpe_count_* in include/bpe_sm100.h)."""

    def __init__(self, ctx=None):
        import torch
        self.ctx = ctx or _lib.default_context()
        self.L = _lib.lib()
        self.torch = torch
        self.device = torch.device("cuda", self.ctx.device)
        self.ctx.check(self.L.bpe_count_begin(self.ctx.handle))
        self._expected_pairs = None

    # returns None, or ("utf8", offset within data) / ("halo", 0) / ("newline", 0).  split_specials (split_special_tokens): the
    # special tokens; data is then one whole text cut at exact boundaries (bpe_count_add_shard_ex)
    def add(self, data, own_begin: int, own_end: int, at_file_start: bool, at_file_end: bool, device_ptr: int | None = None,
            n_bytes: int | None = None, split_specials: List[str] | None = None):
        if split_specials is not None:
            sp_blob, sp_offs = _lib.pack_blobs([s.encode("utf-8") for s in split_specials])
            sp = (_lib.ptr(sp_blob), _lib.ptr(sp_offs), len(split_specials), _lib.TRAIN_SPLIT_SPECIALS)
            if device_ptr is not None:
                rc = self.L.bpe_count_add_shard_dev_ex(self.ctx.handle, C.c_void_p(device_ptr), int(n_bytes), own_begin, own_end,
                                                       int(at_file_start), int(at_file_end), *sp)
            else:
                arr = _lib.as_u8(data)
                rc = self.L.bpe_count_add_shard_ex(self.ctx.handle, _lib.ptr(arr) if arr.size else None, arr.size, own_begin, own_end,
                                                   int(at_file_start), int(at_file_end), *sp)
        elif device_ptr is not None:
            rc = self.L.bpe_count_add_shard_dev(self.ctx.handle, C.c_void_p(device_ptr), int(n_bytes), own_begin, own_end,
                                                int(at_file_start), int(at_file_end))
        else:
            arr = _lib.as_u8(data)
            rc = self.L.bpe_count_add_shard(self.ctx.handle, _lib.ptr(arr) if arr.size else None, arr.size, own_begin, own_end,
                                            int(at_file_start), int(at_file_end))
        if rc == _lib.ERR_UTF8:
            return ("utf8", int(self.L.bpe_last_error_detail(self.ctx.handle)))
        if rc == _lib.ERR_HALO:
            return ("halo", 0)
        if rc == _lib.ERR_NEWLINE:
            return ("newline", 0)
        self.ctx.check(rc)
        return None

    def restart(self):
        self.ctx.check(self.L.bpe_count_begin(self.ctx.handle))

    def export(self):
        torch = self.torch
        nw, nb = C.c_uint64(0), C.c_uint64(0)
        self.ctx.check(self.L.bpe_count_export_size(self.ctx.handle, C.byref(nw), C.byref(nb)))
        blob = torch.empty(max(nb.value, 1), dtype=torch.uint8, device=self.device)
        offs = torch.zeros(nw.value + 1, dtype=torch.int64, device=self.device)
        counts = torch.empty(max(nw.value, 1), dtype=torch.int64, device=self.device)
        torch.cuda.synchronize(self.device)
        self.ctx.check(self.L.bpe_count_export_dev(self.ctx.handle, C.c_void_p(blob.data_ptr()), C.c_void_p(offs.data_ptr()),
                                                   C.c_void_p(counts.data_ptr())))
        return blob[: nb.value], offs, counts[: nw.value]

    def import_(self, blob, offs, counts):
        n_words = counts.numel()
        if n_words == 0:
            return
        self.torch.cuda.synchronize(self.device)   # the collective that produced these tensors ran on torch's stream
        self.ctx.check(self.L.bpe_count_import_dev(self.ctx.handle, C.c_void_p(blob.data_ptr()), C.c_void_p(offs.data_ptr()),
                                                   C.c_void_p(counts.data_ptr()), n_words, blob.numel()))

    def pair_table(self, special_tokens: List[str]):
        sp_blob, sp_offs = _lib.pack_blobs([s.encode("utf-8") for s in special_tokens])
        dense = np.zeros(65536, dtype=np.int64)
        self.ctx.check(self.L.bpe_count_pair_table(self.ctx.handle, _lib.ptr(sp_blob), _lib.ptr(sp_offs), len(special_tokens), _lib.ptr(dense)))
        return self.torch.from_numpy(dense).to(self.device)

    def expect_pair_table(self, dense):
        """Remember the all-reduced per-rank pair table; finish() compares it with the merged one."""
        self._expected_pairs = dense

    def finish(self, vocab_size: int, special_tokens: List[str], return_stats: bool = False):
        """Merge loop over the merged table (bpe_train_from_counts): train.py:165-228."""
        vocab = Vocab(special_tokens=list(special_tokens))
        n_merges = max(vocab_size - len(vocab), 0)
        sp_blob, sp_offs = _lib.pack_blobs([s.encode("utf-8") for s in special_tokens])
        pairs = np.zeros((max(n_merges, 1), 2), dtype=np.int32)
        n_done = C.c_int(0)
        stats = _lib.TrainStats()
        from .train import LiveMerges
        live = LiveMerges(self.ctx, vocab, n_merges)
        rc = -1
        try:
            rc = self.L.bpe_train_from_counts(self.ctx.handle, _lib.ptr(sp_blob), _lib.ptr(sp_offs), len(special_tokens), n_merges,
                                              _lib.ptr(pairs), C.byref(n_done), C.byref(stats))
        finally:
            out = live.finish(pairs, n_done.value if rc == _lib.BPE_OK else 0)
        self.ctx.check(rc)
        if stats.duplicate_tokens:
            raise AssertionError("invariant violated: a merge with a positive count produced the bytes of an earlier token (SURVEY A-6)")   # see train.py
        if self._expected_pairs is not None:
            # linearity check of the sharded count: the all-reduced per-rank byte-pair tables must equal the table of the
            # merged counts, which the merge phase has just built
            merged = np.zeros(65536, dtype=np.int64)
            self.ctx.check(self.L.bpe_last_pair_table(self.ctx.handle, _lib.ptr(merged)))
            expected, self._expected_pairs = self._expected_pairs, None
            if not np.array_equal(expected.cpu().numpy(), merged):
                raise RuntimeError("pair-count all-reduce does not match the merged word table")
        return out + (stats.as_dict(),) if return_stats else out


# ---- collectives ----------------------------------------------------------------------------------------
def _dist():
    import torch.distributed as dist
    return dist


def _all_reduce_scalar(value: int, op: str, device, group=None) -> int:
    import torch
    dist = _dist()
    t = torch.tensor([value], dtype=torch.int64, device=device)
    dist.all_reduce(t, op={"min": dist.ReduceOp.MIN, "max": dist.ReduceOp.MAX, "sum": dist.ReduceOp.SUM}[op], group=group)
    return int(t.item())


LAST_TIMES: dict = {}                           # BPE_SHARD_PROFILE=1: wall ms of the phases of the last sharded_count (synchronising)


def _tick(name, t0):
    import os
    import time
    if os.environ.get("BPE_SHARD_PROFILE") != "1":
        return t0
    import torch
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    LAST_TIMES[name] = LAST_TIMES.get(name, 0.0) + (t1 - t0) * 1e3
    return t1


def exchange_tables(counter, group=None):
    """All-gather every rank's (blob, offs, counts) table and import the other ranks' into `counter`.
    Returns the number of bytes this rank received."""
    import torch
    dist = _dist()
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    import time
    t0 = time.perf_counter()
    blob, offs, counts = counter.export()
    t0 = _tick("export", t0)
    dev = counter.device
    meta = torch.tensor([counts.numel(), blob.numel()], dtype=torch.int64, device=dev)
    metas = torch.empty(world * 2, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(metas, meta, group=group)
    metas = metas.view(world, 2).cpu()
    max_w, max_b = int(metas[:, 0].max()), int(metas[:, 1].max())
    pb = torch.zeros(max(max_b, 1), dtype=torch.uint8, device=dev); pb[: blob.numel()] = blob
    po = torch.zeros(max_w + 1, dtype=torch.int64, device=dev); po[: offs.numel()] = offs
    pc = torch.zeros(max(max_w, 1), dtype=torch.int64, device=dev); pc[: counts.numel()] = counts
    gb = torch.empty(world * pb.numel(), dtype=torch.uint8, device=dev)
    go = torch.empty(world * po.numel(), dtype=torch.int64, device=dev)
    gc = torch.empty(world * pc.numel(), dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(gb, pb, group=group)
    dist.all_gather_into_tensor(go, po, group=group)
    dist.all_gather_into_tensor(gc, pc, group=group)
    t0 = _tick("all_gather", t0)
    received = 0
    for r in range(world):
        if r == rank:
            continue
        nw, nb = int(metas[r, 0]), int(metas[r, 1])
        if nw == 0:
            continue
        counter.import_(gb[r * pb.numel(): r * pb.numel() + nb], go[r * po.numel(): r * po.numel() + nw + 1],
                        gc[r * pc.numel(): r * pc.numel() + nw])
        received += nb + 16 * nw
    _tick("import", t0)
    return received


def _raise_decode_error(peek, size: int, offset: int):
    lo, hi = max(0, offset - 8), min(size, offset + 8)
    window = bytes(peek(lo, hi))
    try:
        window[offset - lo:].decode("utf-8")
    except UnicodeDecodeError as e:
        raise UnicodeDecodeError("utf-8", window, offset - lo + e.start, min(len(window), offset - lo + e.end), e.reason) from None
    raise UnicodeDecodeError("utf-8", window, offset - lo, offset - lo + 1, "invalid start byte")


class FileShards:
    """Shard source over a file (or any byte source `peek(lo, hi)` of `size` bytes): rank r owns [size*r/W, size*(r+1)/W)
    moved back to a code-point boundary and reads a halo on both sides."""

    def __init__(self, peek, size: int):
        self.peek, self.size = peek, size

    def load(self, rank: int, world: int, halo_right: int):
        lo, hi, read_lo, read_hi = plan_shard(self.peek, self.size, rank, world, halo_right)
        return dict(data=self.peek(read_lo, read_hi), device_ptr=None, n_bytes=read_hi - read_lo, own_begin=lo - read_lo, own_end=hi - read_lo,
                    at_start=read_lo == 0, at_end=read_hi == self.size, base=read_lo)

    def raise_decode_error(self, offset: int):
        _raise_decode_error(self.peek, self.size, offset)

    def load_exact(self, rank: int, world: int, special_tokens: List[str]):
        """split_special_tokens: rank r's range between exact cuts (sharded_encode.shard_cuts: every rank computes the same list),
        read without a halo and counted as one whole text."""
        from .sharded_encode import shard_cuts
        cuts = shard_cuts(self.peek, self.size, [s.encode("utf-8") for s in special_tokens], world)
        lo, hi = cuts[rank], cuts[rank + 1]
        return dict(data=self.peek(lo, hi), device_ptr=None, n_bytes=hi - lo, own_begin=0, own_end=hi - lo, at_start=True, at_end=True,
                    base=lo)


def sharded_count(counter, shards, special_tokens: List[str], group=None, verify: bool = True, split_special_tokens: bool = False):
    """Count the pretokens of the corpus behind `shards` across the ranks of `group` into `counter` (every rank ends
    with the merged table).  Returns "ok", or "newline" when some shard contains a carriage return (the caller
    then takes the unsharded path: universal-newline translation shifts byte offsets).  split_special_tokens: the ranges are
    cut at exact boundaries and split on the specials (FileShards.load_exact, DeviceCounter.add)."""
    dist = _dist()
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    import time
    LAST_TIMES.clear()
    t0 = time.perf_counter()
    halo = HALO_RIGHT
    while True:
        if split_special_tokens:
            sh = shards.load_exact(rank, world, special_tokens)
            status = None
            if sh["n_bytes"]:                      # (a rank past the last exact cut has nothing to count)
                status = counter.add(sh["data"], 0, sh["n_bytes"], True, True, device_ptr=sh["device_ptr"], n_bytes=sh["n_bytes"],
                                     split_specials=list(special_tokens))
            break
        sh = shards.load(rank, world, halo)
        status = counter.add(sh["data"], sh["own_begin"], sh["own_end"], sh["at_start"], sh["at_end"], device_ptr=sh["device_ptr"],
                             n_bytes=sh["n_bytes"])
        if status is not None and status[0] == "halo" and not sh["at_end"]:
            counter.restart()
            halo *= 16
            continue
        break
    err = NO_ERROR
    if status is not None and status[0] == "utf8":
        err = sh["base"] + status[1]
    first_err = _all_reduce_scalar(err, "min", counter.device, group)
    if first_err != NO_ERROR:
        shards.raise_decode_error(first_err)                   # same exception on every rank (train.py:22)
    any_cr = _all_reduce_scalar(1 if (status is not None and status[0] == "newline") else 0, "max", counter.device, group)
    if any_cr:
        return "newline"
    if status is not None:
        raise _lib.BpeError(_lib.ERR_HALO, "a pretoken runs past the end of the corpus")
    t0 = _tick("count", t0)
    local_pairs = counter.pair_table(special_tokens) if verify else None
    t0 = _tick("pair_table_local", t0)
    exchange_tables(counter, group)
    t0 = time.perf_counter()
    if verify:
        # linearity check: the per-rank byte-pair tables must sum to the table of the merged counts
        dist.all_reduce(local_pairs, op=dist.ReduceOp.SUM, group=group)
        if hasattr(counter, "expect_pair_table"):
            counter.expect_pair_table(local_pairs)         # compared in finish(), against the table the merge phase builds anyway
        else:
            merged = counter.pair_table(special_tokens)
            if not bool((local_pairs == merged).all()):
                raise RuntimeError("pair-count all-reduce does not match the merged word table")
        _tick("verify", t0)
    return "ok"


def _file_peek(path):
    f = open(path, "rb", buffering=0)

    def peek(lo, hi):
        f.seek(lo)
        out = bytearray(hi - lo)
        mv, got = memoryview(out), 0
        while got < hi - lo:
            k = f.readinto(mv[got:])
            if not k:
                break
            got += k
        return out[:got]
    return peek, f


def merges_digest(merges) -> int:
    h = hashlib.sha256()
    for a, b in merges:
        h.update(len(a).to_bytes(4, "little")); h.update(a); h.update(len(b).to_bytes(4, "little")); h.update(b)
    return int.from_bytes(h.digest()[:7], "little")


def train_bpe_sharded(input_path, vocab_size: int, special_tokens: List[str] = [], *, group=None, ctx=None, verify: bool = True,
                      return_stats: bool = False, split_special_tokens: bool = False):
    """train_bpe over the ranks of an initialised torch.distributed group (one process per GPU).  Every rank
    returns the same (vocab, merges) as the single-GPU train_bpe / the reference (with split_special_tokens, as train_bpe's)."""
    dist = _dist()
    size = os.path.getsize(input_path)
    peek, f = _file_peek(input_path)
    try:
        counter = DeviceCounter(ctx)
        outcome = sharded_count(counter, FileShards(peek, size), special_tokens, group, verify, split_special_tokens)
        if outcome == "newline":
            from .train import train_bpe
            return train_bpe(input_path, vocab_size, special_tokens, ctx=ctx, return_stats=return_stats,
                             split_special_tokens=split_special_tokens)
        res = counter.finish(vocab_size, special_tokens, return_stats=return_stats)
    finally:
        f.close()
    d = merges_digest(res[1])
    lo = _all_reduce_scalar(d, "min", counter.device, group)
    hi = _all_reduce_scalar(d, "max", counter.device, group)
    if lo != hi:
        raise RuntimeError("ranks disagree on the merge list")
    return res
