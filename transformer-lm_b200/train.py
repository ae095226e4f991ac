"""BPE training host: mirrors models/tokenizer/train.py:142-231 of the reference.

train_bpe(input_path, vocab_size, special_tokens) -> (vocab: dict[int, bytes], merges: list[tuple[bytes, bytes]])

The file is read as raw bytes; strict UTF-8 validation, universal-newline translation, GPT-2
pretokenisation, pretoken counting and the whole merge loop run on the GPU (bpe_train in
include/bpe_sm100.h).  The host only rebuilds the Python objects from the symbol-id merge list.
"""
from __future__ import annotations

import ctypes as C
import logging
import os
import threading
import time
from typing import List

import numpy as np

from . import _lib
from .vocab import Vocab

logger = logging.getLogger(__name__)

_PINNED_READ_THRESHOLD = 64 << 20


def _read_file(input_path):
    """Raw bytes of the file as a uint8 array (page-locked for big files so the H2D copy runs at PCIe speed)."""
    size = os.path.getsize(input_path)           # FileNotFoundError like open() in the reference
    if size >= _PINNED_READ_THRESHOLD:
        buf = _lib.PinnedBuffer(size)
        with open(input_path, "rb", buffering=0) as f:
            mv = memoryview(buf.array)
            got = 0
            while got < size:
                k = f.readinto(mv[got:])
                if not k:
                    break
                got += k
        return buf.array[:got], buf
    with open(input_path, "rb") as f:
        data = f.read()
    return np.frombuffer(data, dtype=np.uint8), data


class MergeBuilder:
    """Symbol-id merge list of the device -> (vocab dict, merges list) of the reference (train.py:190-191, 228), fed in order and in
    pieces: tokens are byte strings, `Vocab.add_token` skips a byte string that is already present (vocab.py:28-34)."""

    def __init__(self, vocab: Vocab):
        self.vocab = vocab
        self.sym = [bytes([i]) for i in range(256)]      # symbol id -> bytes: 0..255 the bytes, 256 + k the product of merge k
        self.merges: list = []

    def feed(self, chunk: np.ndarray) -> None:
        """The next merges: int32 array [m, 2] of symbol ids."""
        if not len(chunk):
            return
        ia, ib = chunk[:, 0].tolist(), chunk[:, 1].tolist()
        sym, append = self.sym, self.sym.append
        n0 = len(sym)
        for x, y in zip(ia, ib):                 # the one loop that cannot be avoided: token j is built from earlier tokens
            append(sym[x] + sym[y])
        get = sym.__getitem__
        self.merges.extend(zip(map(get, ia), map(get, ib)))
        new = sym[n0:]
        idx_to_token, present = self.vocab.idx_to_token, self.vocab._present     # (Vocab.add_token inlined: tens of thousands of calls)
        fresh = set(new)
        if len(fresh) == len(new) and present.isdisjoint(fresh):       # the usual case: no byte string twice (A-5 / A-6 never triggered)
            base = len(idx_to_token)
            idx_to_token.update(zip(range(base, base + len(new)), new))
            present |= fresh
        else:
            for t in new:
                if t not in present:
                    present.add(t)
                    idx_to_token[len(idx_to_token)] = t

    @property
    def n_fed(self) -> int:
        return len(self.merges)

    def result(self):
        return self.vocab.get_idx_to_token(), self.merges


_LIVE_BUFFERS: dict = {}         # context id -> page-locked buffer of the live merge view


class LiveMerges:
    """Follows the merge loop from the host (bpe_train_set_live): while the GPU makes merges, a thread feeds the pairs that have
    appeared so far to a MergeBuilder, so that the reference's Python objects (32 000 byte strings, tuples and dict entries: ~9 ms after
    an 11 GB / vocab-32 000 run) are nearly complete when the loop ends.  ctypes releases the GIL during the training call, so the
    thread runs beside it."""

    def __init__(self, ctx, vocab: Vocab, n_merges: int):
        self.ctx, self.n = ctx, int(n_merges)
        self.builder = MergeBuilder(vocab)
        self.active = False
        if self.n <= 0 or os.environ.get("BPE_LIVE_MERGES", "1") in ("", "0"):
            return
        # (the buffer is kept between calls: page-locking and unlocking cost milliseconds each when the process holds GBs of pinned memory)
        buf = _LIVE_BUFFERS.get(id(ctx))
        if buf is None or buf.nbytes < self.n * 8:
            if buf is not None:
                buf.free()
            buf = _LIVE_BUFFERS[id(ctx)] = _lib.PinnedBuffer(max(self.n * 8, 1 << 20))
        self._pairs = buf
        self._pairs.array[: self.n * 8] = 0xFF       # -1, -1: "not made yet" (the kernel stores a pair with one 8-byte write)
        self.pairs = self._pairs.array[: self.n * 8].view(np.int32).reshape(self.n, 2)
        ctx.check(_lib.lib().bpe_train_set_live(ctx.handle, _lib.ptr(self._pairs.array), self.n))
        self.active = True
        self._stop = threading.Event()
        self._thread = threading.Thread(target=self._follow, daemon=True)
        self._thread.start()

    def _follow(self) -> None:
        first = self.pairs[:, 0]
        nap = float(os.environ.get("BPE_LIVE_POLL_MS", "1.0")) / 1e3     # (the loop makes ~230 merges per millisecond at 11 GB)
        while not self._stop.is_set():
            k = self.builder.n_fed
            if k < self.n and first[k] >= 0:
                blk = first[k: k + 4096] < 0             # the complete entries in front (they may land out of order)
                m = int(np.argmax(blk)) if blk.any() else blk.size
                if m < 64 and k + m < self.n:            # (a handful: wait for more, the per-piece overhead is what we are hiding)
                    self._stop.wait(nap)
                    continue
                self.builder.feed(self.pairs[k: k + m].copy())
            else:
                self._stop.wait(nap if k else 4 * nap)   # (nothing yet: the text is still being uploaded and counted)

    def finish(self, pairs: np.ndarray, n_done: int):
        """Stop following and complete the objects from the authoritative `pairs`; returns (vocab dict, merges list)."""
        if self.active:
            self._stop.set()
            self._thread.join()
            _lib.lib().bpe_train_set_live(self.ctx.handle, None, 0)
            k = self.builder.n_fed
            ok = k <= n_done and (k == 0 or np.array_equal(self.pairs[:k], pairs[:k]))
            self.active = False
            if not ok:
                raise RuntimeError("the live view of the merge loop disagrees with its result")
        self.builder.feed(pairs[self.builder.n_fed:n_done])
        return self.builder.result()


def merges_to_python(vocab: Vocab, pairs: np.ndarray, n_done: int):
    """Symbol-id merge list of the device -> (vocab dict, merges list) of the reference (see MergeBuilder)."""
    b = MergeBuilder(vocab)
    b.feed(pairs[:n_done])
    return b.result()


def train_bpe_on_bytes(data, vocab_size: int, special_tokens: List[str] = [], *, ctx=None, return_stats: bool = False,
                       device_ptr: int | None = None, n_bytes: int | None = None, split_special_tokens: bool = False):
    """train_bpe on an in-memory byte buffer (bytes / numpy uint8) or, with device_ptr, on text already in HBM.
    split_special_tokens: see train_bpe."""
    ctx = ctx or _lib.default_context()
    L = _lib.lib()
    vocab = Vocab(special_tokens=list(special_tokens))
    n_merges = max(vocab_size - len(vocab), 0)                    # range(vocab_size - len(vocab)), train.py:183
    sp_blob, sp_offs = _lib.pack_blobs([s.encode("utf-8") for s in special_tokens])
    pairs = np.zeros((max(n_merges, 1), 2), dtype=np.int32)
    n_done = C.c_int(0)
    stats = _lib.TrainStats()
    live = LiveMerges(ctx, vocab, n_merges)
    rc = -1
    try:
        rc = _call_train(L, ctx, data, device_ptr, n_bytes, sp_blob, sp_offs, special_tokens, n_merges, pairs, n_done, stats,
                         _lib.TRAIN_SPLIT_SPECIALS if split_special_tokens else 0)
    finally:
        res = live.finish(pairs, n_done.value if rc == _lib.BPE_OK else 0)
    arr = None if device_ptr is not None else _lib.as_u8(data)
    if rc == _lib.ERR_UTF8 and arr is not None:
        bytes(arr).decode("utf-8")                                # raises the reference's UnicodeDecodeError
        raise AssertionError("device flagged invalid UTF-8 at %d but CPython accepts the data" % L.bpe_last_error_detail(ctx.handle))
    ctx.check(rc)
    if stats.duplicate_tokens:
        # SURVEY A-6: the reference identifies a token by its bytes, the device by its merge index.  The two differ only if a merge
        # with a positive count produces bytes an earlier merge produced -- which cannot happen (DESIGN.md section 8 has the
        # argument), so a non-zero counter means the device result is wrong, not that a rare input was met.
        raise AssertionError("invariant violated: a merge with a positive count produced the bytes of an earlier token (SURVEY A-6)")
    out = (*res,)
    return out + (stats.as_dict(),) if return_stats else out


def _call_train(L, ctx, data, device_ptr, n_bytes, sp_blob, sp_offs, special_tokens, n_merges, pairs, n_done, stats, flags=0):
    ex = (flags,) if flags else ()
    if device_ptr is not None:
        fn = L.bpe_train_dev_ex if flags else L.bpe_train_dev
        rc = fn(ctx.handle, C.c_void_p(device_ptr), int(n_bytes), _lib.ptr(sp_blob), _lib.ptr(sp_offs),
                len(special_tokens), n_merges, _lib.ptr(pairs), C.byref(n_done), C.byref(stats), *ex)
    else:
        arr = _lib.as_u8(data)
        fn = L.bpe_train_ex if flags else L.bpe_train
        rc = fn(ctx.handle, _lib.ptr(arr) if arr.size else None, arr.size, _lib.ptr(sp_blob), _lib.ptr(sp_offs),
                len(special_tokens), n_merges, _lib.ptr(pairs), C.byref(n_done), C.byref(stats), *ex)
    return rc


_STREAM_MIN = 512 << 20          # files at least this big are streamed: read, upload and counting overlap
_STREAM_CHUNK = 256 << 20
_STREAM_HALO_LEFT = 64
_STREAM_HALO_RIGHT = 64 << 10
_READ_THREADS = int(os.environ.get("BPE_READ_THREADS", "8"))      # (2 -> 0.22 s, 4 -> 0.14 s, 8 -> 0.11 s for a 2 GiB file in tmpfs)
_PIN_CACHE: list = []            # page-locked chunk buffers of the streamed ingest, kept between calls (pinning costs ~0.3 s per GB)


def release_buffers() -> None:
    """Free the page-locked buffers train_bpe keeps between calls."""
    while _PIN_CACHE:
        _PIN_CACHE.pop().free()
    for b in _LIVE_BUFFERS.values():
        b.free()
    _LIVE_BUFFERS.clear()


_DIRECT_ALIGN = 4096             # O_DIRECT: file offsets, lengths and buffer addresses in multiples of the logical block size


def _pread_into(fd: int, view: memoryview, offset: int, size: int | None = None) -> None:
    """Fill `view` from file offset `offset`.  With `size` (the file size; O_DIRECT reads) the view may extend past the end of the
    file: the read stops there."""
    got = 0
    want = len(view) if size is None else min(len(view), size - offset)
    while got < want:
        k = os.preadv(fd, [view[got:]], offset + got)
        if k <= 0:
            raise OSError("short read at offset %d" % (offset + got))
        got += k


def _open_for_read(path, direct: bool):
    """(fd, direct): the file opened O_RDONLY, with O_DIRECT when asked for and the file system takes it (page cache bypassed: the
    ingest path reads every byte once; SURVEY 8f row 2).  tmpfs and some network file systems refuse O_DIRECT: buffered then."""
    if direct and hasattr(os, "O_DIRECT"):
        try:
            return os.open(os.fspath(path), os.O_RDONLY | os.O_DIRECT), True
        except OSError:
            logger.info("O_DIRECT not supported for %s: buffered reads", path)
    return os.open(os.fspath(path), os.O_RDONLY), False


def _train_bpe_streamed(input_path, size: int, vocab_size: int, special_tokens: List[str], ctx=None, return_stats: bool = False,
                        direct_io: bool | None = None, split_special_tokens: bool = False):
    """Ingest path for big files (SURVEY 8f row 2): the file is read in 256 MB chunks, each with a small halo, by a few
    threads into page-locked buffers while the GPU pretokenises and counts the previous chunk (bpe_count_add_shard --
    the same shard contract as the multi-GPU path); then the merge loop runs on the counts.  Returns None when the file
    needs the one-piece path (a carriage return: universal newlines shift offsets; or a pretoken longer than the halo).
    split_special_tokens: the chunks are cut only at exact boundaries (sharded_encode.first_exact_cut) and each is counted whole,
    with no halo: special-token resolution at a cut can depend on context further left than any fixed halo.  Where no exact
    boundary follows a nominal cut the chunk grows to the next one."""
    import concurrent.futures as cf
    from .sharded import DeviceCounter, align_cut, _raise_decode_error
    from .sharded_encode import first_exact_cut
    if direct_io is None:
        direct_io = os.environ.get("BPE_IO_DIRECT", "0") not in ("", "0")
    fd, direct = _open_for_read(input_path, direct_io)
    fd_peek = os.open(os.fspath(input_path), os.O_RDONLY) if direct else fd      # (small unaligned reads: cut search, error context)
    bufs = []
    pool = None
    pending: dict = {}
    try:
        def peek(lo, hi):
            return os.pread(fd_peek, hi - lo, lo)
        split = list(special_tokens) if split_special_tokens else None
        specials_b = [s.encode("utf-8") for s in special_tokens]
        cuts = [0]
        p = _STREAM_CHUNK
        while p + _STREAM_CHUNK // 2 < size:
            if split is None:
                cuts.append(align_cut(peek, p, size))
            else:
                try:
                    c = first_exact_cut(peek, size, specials_b, max(p, cuts[-1] + 1))
                except RuntimeError:
                    break                                # no exact boundary from here on: the rest is one chunk
                if c >= size:
                    break
                cuts.append(c)
                p = max(p, c)
            p += _STREAM_CHUNK
        cuts.append(size)
        ranges = []
        for k in range(len(cuts) - 1):
            lo, hi = cuts[k], cuts[k + 1]
            if split is None:
                rlo = align_cut(peek, max(0, lo - _STREAM_HALO_LEFT), size)
                rhi = align_cut(peek, min(size, hi + _STREAM_HALO_RIGHT), size)
            else:
                rlo, rhi = lo, hi
            ranges.append((lo, hi, rlo, rhi))
        # with O_DIRECT a chunk is read as the block-aligned range around it (the page-locked buffers are page aligned); `skew` =
        # where the chunk starts inside its buffer
        A = _DIRECT_ALIGN if direct else 1
        cap = max(-(-r[3] // A) * A - r[2] // A * A for r in ranges)
        want_bufs = min(3, len(ranges))
        while _PIN_CACHE and (_PIN_CACHE[0].nbytes < cap or len(_PIN_CACHE) > want_bufs):
            _PIN_CACHE.pop(0).free()
        while len(_PIN_CACHE) < want_bufs:
            _PIN_CACHE.append(_lib.PinnedBuffer(cap))
        bufs = list(_PIN_CACHE)
        pool = cf.ThreadPoolExecutor(max_workers=_READ_THREADS)

        def submit(k):
            lo, hi, rlo, rhi = ranges[k]
            alo, ahi = rlo // A * A, -(-rhi // A) * A
            mv = memoryview(bufs[k % len(bufs)].array)[: ahi - alo]
            step = -(-(-(-(ahi - alo) // _READ_THREADS)) // A) * A
            return [pool.submit(_pread_into, fd, mv[o: min(o + step, ahi - alo)], alo + o, size if direct else None) for o in range(0, ahi - alo, step)]

        counter = DeviceCounter(ctx)
        pending = {k: submit(k) for k in range(min(len(bufs) - 1, len(ranges)))}
        for k, (lo, hi, rlo, rhi) in enumerate(ranges):
            nxt = k + len(bufs) - 1
            if nxt < len(ranges) and nxt not in pending:
                pending[nxt] = submit(nxt)       # its buffer was consumed by chunk nxt - len(bufs), already counted
            for fut in pending.pop(k):
                fut.result()
            skew = rlo - rlo // A * A
            status = counter.add(bufs[k % len(bufs)].array[skew: skew + rhi - rlo], lo - rlo, hi - rlo, rlo == 0, rhi == size,
                                 **({} if split is None else {"split_specials": split}))
            if status is not None:
                if status[0] == "utf8":
                    _raise_decode_error(peek, size, rlo + status[1])      # what open(path, encoding="utf-8").read() raises
                return None
        return counter.finish(vocab_size, special_tokens, return_stats=return_stats)
    finally:
        # reader threads may still be writing into the page-locked buffers (an error or an early return above): wait for every
        # submitted read before the buffers are freed
        for futs in pending.values():
            for fut in futs:
                try:
                    fut.result()
                except Exception:
                    pass
        if pool is not None:
            pool.shutdown(wait=True)
        os.close(fd)
        if fd_peek != fd:
            os.close(fd_peek)


def train_bpe(input_path, vocab_size: int, special_tokens: List[str] = [], *, distributed: bool = False,
              split_special_tokens: bool = False, **kwargs):
    """Drop-in for models/tokenizer/train.py:142 train_bpe.  Extra keyword arguments are ours (the reference's
    adapter never passes any): ctx=, return_stats=, direct_io= (files of >= 512 MB are streamed; True or BPE_IO_DIRECT=1 reads them
    with O_DIRECT), and distributed=True to shard the file over the ranks of the initialised torch.distributed group (one process
    per GPU; see sharded.py).
    split_special_tokens=True splits the text on the special tokens before counting, as the tokenizer does before encoding: no
    pretoken, pair or merge crosses an occurrence and the occurrences are not counted (BPE_TRAIN_SPLIT_SPECIALS in
    include/bpe_sm100.h).  The default (False) counts the text whole, exactly as the reference does."""
    if distributed:
        from .sharded import train_bpe_sharded
        return train_bpe_sharded(input_path, vocab_size, special_tokens, split_special_tokens=split_special_tokens, **kwargs)
    t0 = time.time()
    size = os.path.getsize(input_path)           # FileNotFoundError like open() in the reference
    kwargs = dict(kwargs)
    want_stats = kwargs.pop("return_stats", False)
    direct_io = kwargs.pop("direct_io", None)
    res = None
    if size >= _STREAM_MIN:
        res = _train_bpe_streamed(input_path, size, vocab_size, special_tokens, return_stats=True, direct_io=direct_io,
                                  split_special_tokens=split_special_tokens, **kwargs)
    if res is None:
        arr, _keep = _read_file(input_path)
        res = train_bpe_on_bytes(arr, vocab_size, special_tokens, return_stats=True, split_special_tokens=split_special_tokens, **kwargs)
    _log_stages(res[2], time.time() - t0)
    return res if want_stats else res[:2]


def _log_stages(st: dict, wall_s: float) -> None:
    """The reference's five stage lines (models/tokenizer/train.py:148-229), so CPU and GPU logs line up.  The stages ran
    on the device: the times are their CUDA-event durations (the words and the pair table are built in one pass)."""
    logger.info("Creating vocab")
    logger.info("Took %s seconds to create vocab", 0.0)
    logger.info("Extracting subword frequencies")
    logger.info("Took %s seconds to extract subword frequencies", round((st["ms_h2d"] + st["ms_pretok"] + st["ms_count"]) / 1e3, 4))
    logger.info("Encoding subwords")
    logger.info("Took %s seconds to encode subwords", round(st["ms_build"] / 1e3, 4))
    logger.info("Calculating byte pair frequencies")
    logger.info("Took %s seconds to calculate byte pair frequencies", 0.0)
    logger.info("Merging subwords")
    logger.info("Took %s seconds to merge subwords", round(st["ms_merge"] / 1e3, 4))
    logger.info("train_bpe on the GPU: %d bytes, %d pretokens (%d unique), %d merge steps; %.3f s wall including the file read",
                st["n_bytes"], st["n_pretokens"], st["n_unique"], st["merge_steps"], wall_s)
