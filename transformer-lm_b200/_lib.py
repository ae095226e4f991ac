"""ctypes binding of libbpe_sm100.so (C ABI declared in include/bpe_sm100.h).

Fails loudly when the library cannot be built/loaded or no sm_100 GPU is present: the product has no
CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

from . import _build

BPE_OK = 0
(ERR_ARG, ERR_CUDA, ERR_OOM, ERR_UTF8, ERR_KEY, ERR_CAPACITY, ERR_TOO_SMALL, ERR_UNSUPPORTED, ERR_NO_DEVICE, ERR_HALO,
 ERR_NEWLINE) = range(-1, -12, -1)
DTYPE_U16, DTYPE_I32 = 0, 1
TRAIN_SPLIT_SPECIALS = 1
OFF_BYTES, OFF_CHARS = 0, 1
SYNTH_TINYSTORIES, SYNTH_OWT = 0, 1


class BpeError(RuntimeError):
    def __init__(self, code: int, message: str, detail: int = 0):
        super().__init__("libbpe_sm100 error %d: %s" % (code, message))
        self.code = code
        self.detail = detail


class TrainStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("n_bytes", "n_pretokens", "n_unique", "n_symbols", "n_pairs_initial",
                                          "n_pairs_final", "log_records", "duplicate_tokens", "sum_live_pairs", "merge_steps")] + \
               [(n, C.c_float) for n in ("ms_h2d", "ms_validate", "ms_pretok", "ms_count", "ms_build", "ms_merge", "ms_total")]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class EncodeStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("n_bytes", "n_pretokens", "n_tokens", "cache_new_unique")] + \
               [(n, C.c_float) for n in ("ms_h2d", "ms_pretok", "ms_lookup", "ms_bpe", "ms_emit", "ms_d2h", "ms_total")]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class EncodeOpts(C.Structure):
    """bpe_encode_opts: documents, BPE-dropout and token offsets of bpe_encode_ex (all zero: bpe_encode)."""
    _fields_ = [("doc_offs", C.c_void_p), ("n_docs", C.c_uint64), ("id_offs_out", C.c_void_p), ("dropout", C.c_double),
                ("seed", C.c_uint64), ("with_offsets", C.c_int), ("offset_unit", C.c_int), ("offs_out", C.c_void_p)]


_lib = None
_lock = threading.Lock()

# every symbol include/bpe_sm100.h declares (tests check the .so exports all of them)
EXPORTS = [
    "bpe_version", "bpe_unicode_table_source", "bpe_ctx_create", "bpe_ctx_destroy", "bpe_last_error",
    "bpe_last_error_detail", "bpe_device_sync", "bpe_utf8_validate", "bpe_pretokenize", "bpe_train", "bpe_train_dev",
    "bpe_train_ex", "bpe_train_dev_ex", "bpe_count_begin", "bpe_count_add_shard", "bpe_count_add_shard_dev",
    "bpe_count_add_shard_ex", "bpe_count_add_shard_dev_ex", "bpe_count_export_size", "bpe_count_export",
    "bpe_count_export_dev", "bpe_count_import", "bpe_count_import_dev", "bpe_count_pair_table",
    "bpe_train_from_counts", "bpe_last_pair_table", "bpe_train_set_live", "bpe_tok_create", "bpe_tok_destroy", "bpe_encode", "bpe_encode_ex",
    "bpe_encode_dev", "bpe_tok_key_error", "bpe_tok_saw_cr",
    "bpe_tok_cache_reset", "bpe_decode", "bpe_decode_batch", "bpe_batch_windows_dev", "bpe_synth_dev", "bpe_synth_host", "bpe_synth_dev_at", "bpe_synth_host_at", "bpe_ctx_set_stream", "bpe_host_alloc", "bpe_host_free", "bpe_launch_count",
]


def lib():
    global _lib
    with _lock:
        if _lib is None:
            path = os.environ.get("BPE_LIB_PATH") or _build.build()   # (BPE_LIB_PATH: A/B runs of two builds in one process tree)
            L = C.CDLL(str(path))
            vp, u64p = C.c_void_p, C.POINTER(C.c_uint64)
            L.bpe_version.restype = C.c_int
            L.bpe_unicode_table_source.restype = C.c_char_p
            L.bpe_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
            L.bpe_ctx_destroy.argtypes = [vp]
            L.bpe_ctx_destroy.restype = None
            L.bpe_last_error.argtypes = [vp]
            L.bpe_last_error.restype = C.c_char_p
            L.bpe_last_error_detail.argtypes = [vp]
            L.bpe_last_error_detail.restype = C.c_int64
            L.bpe_device_sync.argtypes = [vp]
            L.bpe_utf8_validate.argtypes = [vp, vp, C.c_uint64]
            L.bpe_pretokenize.argtypes = [vp, vp, C.c_uint64, vp, vp, C.c_int, vp, C.c_uint64, u64p]
            L.bpe_train.argtypes = [vp, vp, C.c_uint64, vp, vp, C.c_int, C.c_int, vp, C.POINTER(C.c_int), C.POINTER(TrainStats)]
            L.bpe_train_dev.argtypes = L.bpe_train.argtypes
            L.bpe_train_ex.argtypes = L.bpe_train.argtypes + [C.c_int]
            L.bpe_train_dev_ex.argtypes = L.bpe_train_ex.argtypes
            L.bpe_count_begin.argtypes = [vp]
            L.bpe_count_add_shard.argtypes = [vp, vp, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, C.c_int]
            L.bpe_count_add_shard_dev.argtypes = L.bpe_count_add_shard.argtypes
            L.bpe_count_add_shard_ex.argtypes = L.bpe_count_add_shard.argtypes + [vp, vp, C.c_int, C.c_int]
            L.bpe_count_add_shard_dev_ex.argtypes = L.bpe_count_add_shard_ex.argtypes
            L.bpe_count_export_dev.argtypes = [vp, vp, vp, vp]
            L.bpe_count_import_dev.argtypes = [vp, vp, vp, vp, C.c_uint64, C.c_uint64]
            L.bpe_count_pair_table.argtypes = [vp, vp, vp, C.c_int, vp]
            L.bpe_count_export_size.argtypes = [vp, u64p, u64p]
            L.bpe_count_export.argtypes = [vp, vp, vp, vp]
            L.bpe_count_import.argtypes = [vp, vp, vp, vp, C.c_uint64]
            L.bpe_train_from_counts.argtypes = [vp, vp, vp, C.c_int, C.c_int, vp, C.POINTER(C.c_int), C.POINTER(TrainStats)]
            L.bpe_tok_create.argtypes = [vp, vp, vp, C.c_int, vp, vp, vp, C.c_int, vp, vp, vp, C.c_int64, vp, vp, vp, C.c_int,
                                         C.POINTER(vp)]
            L.bpe_tok_destroy.argtypes = [vp]
            L.bpe_tok_destroy.restype = None
            L.bpe_encode.argtypes = [vp, vp, C.c_uint64, C.c_int, vp, C.c_uint64, u64p, C.POINTER(EncodeStats)]
            L.bpe_encode_dev.argtypes = L.bpe_encode.argtypes
            L.bpe_encode_ex.argtypes = [vp, vp, C.c_uint64, C.POINTER(EncodeOpts), C.c_int, vp, C.c_uint64, u64p, C.POINTER(EncodeStats)]
            L.bpe_tok_key_error.argtypes = [vp, vp, C.c_uint64, u64p]
            L.bpe_tok_cache_reset.argtypes = [vp]
            L.bpe_tok_saw_cr.argtypes = [vp]
            L.bpe_decode.argtypes = [vp, vp, C.c_uint64, vp, C.c_uint64, u64p]
            L.bpe_last_pair_table.argtypes = [vp, vp]
            L.bpe_train_set_live.argtypes = [vp, vp, C.c_int]
            L.bpe_decode_batch.argtypes = [vp, vp, C.c_uint64, vp, C.c_uint64, vp, C.c_uint64, u64p, vp]
            L.bpe_batch_windows_dev.argtypes = [vp, vp, C.c_int, C.c_uint64, vp, C.c_uint32, C.c_uint32, vp, vp]
            L.bpe_synth_dev.argtypes = [vp, C.c_int, C.c_uint64, vp, C.c_uint64]
            L.bpe_synth_host.argtypes = [C.c_int, C.c_uint64, vp, C.c_uint64]
            L.bpe_synth_dev_at.argtypes = [vp, C.c_int, C.c_uint64, C.c_uint64, vp, C.c_uint64]
            L.bpe_synth_host_at.argtypes = [C.c_int, C.c_uint64, C.c_uint64, vp, C.c_uint64]
            L.bpe_ctx_set_stream.argtypes = [vp, vp]
            L.bpe_host_alloc.argtypes = [C.c_size_t]
            L.bpe_host_alloc.restype = vp
            L.bpe_host_free.argtypes = [vp]
            L.bpe_host_free.restype = None
            L.bpe_launch_count.restype = C.c_ulonglong
            _lib = L
    return _lib


def ptr(a):
    """void* of a numpy array / None."""
    if a is None:
        return None
    return a.ctypes.data_as(C.c_void_p)


def as_u8(data) -> np.ndarray:
    """Zero-copy uint8 view of bytes / bytearray / memoryview / numpy array."""
    if isinstance(data, np.ndarray):
        a = data.view(np.uint8).reshape(-1)
    else:
        a = np.frombuffer(data, dtype=np.uint8)
    return a


def pack_blobs(items: list[bytes]):
    """(blob u8[], offs u32[n+1]) for a list of byte strings (never zero-length arrays)."""
    offs = np.zeros(len(items) + 1, dtype=np.uint32)
    if items:
        np.cumsum([len(b) for b in items], out=offs[1:])
    blob = np.frombuffer(b"".join(items) or b"\0", dtype=np.uint8)
    return blob, offs


def pack_blobs64(items: list[bytes]):
    """(blob u8[], offs u64[n+1]) for a list of byte strings."""
    offs = np.zeros(len(items) + 1, dtype=np.uint64)
    if items:
        np.cumsum(np.fromiter((len(b) for b in items), dtype=np.uint64, count=len(items)), out=offs[1:])
    blob = np.frombuffer(b"".join(items) or b"\0", dtype=np.uint8)
    return blob, offs


class Context:
    """One bpe_ctx (device, stream, workspaces).  A process-wide default lives in `default_context()`."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        rc = lib().bpe_ctx_create(device, C.byref(self._h))
        if rc == ERR_NO_DEVICE:
            raise BpeError(rc, "no usable sm_100 (B200) device %d -- this library has no CPU fallback" % device)
        if rc != BPE_OK:
            raise BpeError(rc, "bpe_ctx_create failed")
        self.device = device
        # the C ABI allows one in-flight call per context (include/bpe_sm100.h): host code that may call from two
        # threads (Tokenizer.encode_iterable's look-ahead worker) serialises on this lock
        self.lock = threading.RLock()

    @property
    def handle(self):
        return self._h

    def check(self, rc: int):
        if rc != BPE_OK:
            msg = lib().bpe_last_error(self._h)
            raise BpeError(rc, msg.decode("utf-8", "replace") if msg else "", lib().bpe_last_error_detail(self._h))

    def use_stream(self, cuda_stream: int | None):
        """Enqueue all library work on this CUDA stream (e.g. torch.cuda.current_stream().cuda_stream)."""
        self.check(lib().bpe_ctx_set_stream(self._h, C.c_void_p(cuda_stream) if cuda_stream else None))

    def close(self):
        if self._h:
            lib().bpe_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx: dict[int, Context] = {}


def default_context(device: int | None = None) -> Context:
    import os
    if device is None:
        device = int(os.environ.get("BPE_DEVICE", os.environ.get("LOCAL_RANK", "0")))
    ctx = _default_ctx.get(device)
    if ctx is None:
        ctx = _default_ctx[device] = Context(device)
    return ctx


class PinnedBuffer:
    """Page-locked host memory exposed as a numpy uint8 array (H2D copies from it run at PCIe speed)."""

    def __init__(self, nbytes: int):
        self.nbytes = int(nbytes)
        self._p = lib().bpe_host_alloc(max(self.nbytes, 1))
        if not self._p:
            raise MemoryError("cudaMallocHost(%d) failed" % nbytes)
        self.array = np.ctypeslib.as_array((C.c_uint8 * max(self.nbytes, 1)).from_address(self._p))[: self.nbytes]

    def free(self):
        if self._p:
            self.array = None
            lib().bpe_host_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def bind_to_gpu_numa_node(device: int = 0) -> dict:
    """Best effort: run this process (and so allocate its page-locked buffers, first touch) on the CPUs of the NUMA node the GPU hangs
    off.  With one process per GPU and all of them on node 0, the host ends of the PCIe copies of eight ranks share one memory
    controller / root complex (round 1: 54 GB/s per GPU at N = 1, 18.7 at N = 8).  Returns what was found and done; never raises."""
    info = {"device": device, "bound": False}
    try:
        import torch
        bus = torch.cuda.get_device_properties(device).pci_bus_id
        dom = getattr(torch.cuda.get_device_properties(device), "pci_domain_id", 0)
        dev_id = getattr(torch.cuda.get_device_properties(device), "pci_device_id", 0)
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bus, dev_id)
        node = int(open(path).read().strip())
        info["numa_node"] = node
        if node < 0:
            return info
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        info["allowed_cpus"] = len(allowed)
        target = cpus & allowed
        info["node_cpus_allowed"] = len(target)
        if target and target != allowed:
            os.sched_setaffinity(0, target)
            info["bound"] = True
        elif target == allowed:
            info["bound"] = True                     # already there
    except Exception as e:                           # no sysfs, no permission, ...: leave the process where it is
        info["error"] = "%s: %s" % (type(e).__name__, e)
    return info
