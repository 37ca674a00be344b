"""ctypes binding of the product library starrocks_b200/libsr_gpu.so (C-ABI: include/sr_gpu_ops.h).

Used by tests/, bench.py and __graft_entry__.py.  There is no CPU fallback: if the library is
missing or no CUDA device is visible, every entry point raises.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from . import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SR_GPU_LIB") or os.path.join(_HERE, "libsr_gpu.so")   # SR_GPU_LIB: an experimental build
_LIB = None

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-shared",
              "-Xcompiler", "-fPIC", "-cudart", "static"]


def _source_files():
    csrc = os.path.join(_HERE, "csrc")
    return sorted(os.path.join(csrc, f) for f in os.listdir(csrc)) + [os.path.join(_HERE, "..", "include", "sr_gpu_ops.h")]


def _source_hash():
    """content hash of everything the library is compiled from: survives copies of the tree (file times do not -- a fresh
    checkout / the snapshot sent to a GPU box would otherwise look stale and every process would recompile on import)"""
    import hashlib
    h = hashlib.sha256()
    for f in _source_files():
        h.update(os.path.basename(f).encode())
        with open(f, "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS + os.environ.get("SR_NVCC_EXTRA", "").split()).encode())
    return h.hexdigest()


def build(verbose=False):
    """compile libsr_gpu.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).  Safe against concurrent callers
    (the ranks of a torchrun job): one process compiles under a file lock into a temporary name and renames it into place."""
    import fcntl
    src = os.path.join(_HERE, "csrc", "sr_gpu.cu")
    extra = os.environ.get("SR_NVCC_EXTRA", "").split()   # e.g. -DSR_GATHER_AGG_MIN_BLOCKS=4 for timing experiments
    want = _source_hash()
    with open(LIB_PATH + ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not verbose and os.path.exists(LIB_PATH) and _recorded_hash() == want:
                return LIB_PATH                     # another process built it while this one waited for the lock
            tmp = LIB_PATH + ".tmp.%d" % os.getpid()
            cmd = ["nvcc"] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", tmp, src]
            subprocess.check_call(cmd)
            os.replace(tmp, LIB_PATH)
            with open(LIB_PATH + ".srchash", "w") as fh:
                fh.write(want)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB_PATH


def _recorded_hash():
    try:
        with open(LIB_PATH + ".srchash") as fh:
            return fh.read().strip()
    except OSError:
        return None


def _needs_build():
    if not os.path.exists(LIB_PATH):
        return True
    if os.environ.get("SR_GPU_LIB"):
        return False
    return _recorded_hash() != _source_hash()


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    if _needs_build():
        build()
    L = C.CDLL(LIB_PATH)
    i32, i64, u32, vp = C.c_int32, C.c_int64, C.c_uint32, C.c_void_p
    sig = {
        "sr_abi_version": (i32, []),
        "sr_type_width": (i32, [i32]),
        "sr_ctx_create": (vp, [i32, vp]),
        "sr_ctx_destroy": (None, [vp]),
        "sr_ctx_sync": (i32, [vp]),
        "sr_last_error": (C.c_char_p, [vp]),
        "sr_last_error_code": (i32, [vp]),
        "sr_ctx_kernel_launches": (i64, [vp]),
        "sr_ctx_device_bytes": (i64, [vp]),
        "sr_ctx_stream": (vp, [vp]),
        "sr_scan_create": (vp, [vp, vp]),
        "sr_scan_destroy": (None, [vp]),
        "sr_scan_filter": (i32, [vp, vp, vp]),
        "sr_scan_evaluate": (i32, [vp, vp, vp, i32]),
        "sr_join_create": (vp, [vp, vp]),
        "sr_join_destroy": (None, [vp]),
        "sr_join_append_build": (i32, [vp, vp]),
        "sr_join_build_finish": (i32, [vp]),
        "sr_join_is_build_done": (i32, [vp]),
        "sr_join_get_info": (i32, [vp, vp]),
        "sr_join_copy_table": (i32, [vp, vp, vp]),
        "sr_join_probe": (i32, [vp, i32, vp, vp]),
        "sr_join_probe_remain": (i32, [vp, vp]),
        "sr_join_probe_indexes": (i32, [vp, i32, vp, vp]),
        "sr_join_key_hash": (i32, [vp, vp, i32, i64, u32, vp, i32]),
        "sr_join_build_runtime_filter": (vp, [vp, i32, i32, i32]),
        "sr_rf_create": (vp, [vp, i32, i64, i32]),
        "sr_rf_insert": (i32, [vp, vp, i32, i32]),
        "sr_rf_destroy": (None, [vp]),
        "sr_rf_get_info": (i32, [vp, vp]),
        "sr_rf_copy_directory": (i32, [vp, vp, i64, i32]),
        "sr_rf_merge_directory": (i32, [vp, vp, i64, i32, vp]),
        "sr_rf_evaluate": (i32, [vp, vp, i32, vp, i32, i32]),
        "sr_scan_add_runtime_filter": (i32, [vp, vp, i32]),
        "sr_scan_get_rf_stats": (i32, [vp, i32, vp]),
        "sr_scan_set_rf_adaptive": (i32, [vp, i32]),
        "sr_rf_copy_in_values": (i32, [vp, vp, i32]),
        "sr_rf_merge_in_values": (i32, [vp, vp, i32]),
        "sr_agg_create": (vp, [vp, vp]),
        "sr_agg_destroy": (None, [vp]),
        "sr_agg_push": (i32, [vp, vp]),
        "sr_agg_sink_finish": (i32, [vp]),
        "sr_agg_num_groups": (i64, [vp]),
        "sr_agg_pull": (i32, [vp, i64, i32, vp]),
        "sr_agg_merge": (i32, [vp, vp]),
        "sr_agg_two_phase_descs": (i32, [vp, vp, vp]),
        "sr_agg_convert_to_states": (i32, [vp, vp, vp]),
        "sr_agg_push_selective": (i32, [vp, vp, vp]),
        "sr_agg_current_groups": (i64, [vp]),
        "sr_agg_dense_state": (i32, [vp, vp, i32, vp]),
        "sr_agg_reset": (i32, [vp]),
        "sr_fragment_reset": (i32, [vp]),
        "sr_fragment_get_plan": (i32, [vp, vp]),
        "sr_fragment_last_pass_ms": (i32, [vp, vp]),
        "sr_fragment_create": (vp, [vp, vp]),
        "sr_fragment_destroy": (None, [vp]),
        "sr_fragment_push": (i32, [vp, vp]),
        "sr_fragment_agg": (vp, [vp]),
        "sr_fragment_rows_passed": (i64, [vp]),
        "sr_xchg_create": (vp, [vp, vp]),
        "sr_xchg_destroy": (None, [vp]),
        "sr_xchg_partition": (i32, [vp, vp, vp, vp]),
        "sr_xchg_hash": (i32, [vp, vp, vp, vp, i32]),
        "sr_gather": (i32, [vp, vp, i32, vp, i64, vp, i32]),
        "sr_memcpy": (i32, [vp, vp, vp, i64, i32]),
        "sr_abi_sizeof": (i32, [i32]),
        "sr_bandwidth_probe": (i32, [vp, vp, i64, vp]),
        "sr_flush_l2": (i32, [vp]),
        "sr_chunk_serialized_size": (i64, [vp, i64, i64]),
        "sr_chunk_serialize": (i32, [vp, vp, i64, i64, vp, i64, i32, vp]),
        "sr_serde_create": (vp, [vp]),
        "sr_serde_destroy": (None, [vp]),
        "sr_chunk_deserialize": (i32, [vp, vp, i64, i32, vp, vp]),
        "sr_host_alloc": (i32, [vp, i64, vp]),
        "sr_host_free": (i32, [vp, vp]),
        "sr_event_create": (vp, [vp]),
        "sr_event_destroy": (None, [vp]),
        "sr_event_record": (i32, [vp]),
        "sr_event_query": (i32, [vp]),
        "sr_event_sync": (i32, [vp]),
        "sr_page_decoder_create": (vp, [vp]),
        "sr_page_decoder_destroy": (None, [vp]),
        "sr_pages_decode": (i32, [vp, i32, i32, vp, i32, i32, vp, i64, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    if L.sr_abi_version() != abi.SR_ABI_VERSION:
        raise RuntimeError("libsr_gpu.so ABI version mismatch")
    _LIB = L
    return L


EXPORTED_SYMBOLS = [
    "sr_abi_version", "sr_type_width", "sr_ctx_create", "sr_ctx_destroy", "sr_ctx_sync", "sr_last_error", "sr_last_error_code",
    "sr_ctx_kernel_launches", "sr_ctx_device_bytes", "sr_ctx_stream", "sr_scan_create", "sr_scan_destroy",
    "sr_scan_filter", "sr_scan_evaluate", "sr_join_create", "sr_join_destroy", "sr_join_append_build",
    "sr_join_build_finish", "sr_join_is_build_done", "sr_join_get_info", "sr_join_copy_table", "sr_join_probe", "sr_join_probe_remain",
    "sr_join_probe_indexes", "sr_join_key_hash", "sr_agg_create", "sr_agg_destroy", "sr_agg_push",
    "sr_agg_sink_finish", "sr_agg_num_groups", "sr_agg_pull", "sr_agg_merge", "sr_agg_two_phase_descs", "sr_agg_convert_to_states", "sr_agg_push_selective", "sr_agg_current_groups", "sr_agg_dense_state", "sr_agg_reset", "sr_fragment_reset", "sr_fragment_get_plan", "sr_fragment_last_pass_ms",
    "sr_fragment_create",
    "sr_fragment_destroy", "sr_fragment_push", "sr_fragment_agg", "sr_fragment_rows_passed", "sr_xchg_create",
    "sr_join_build_runtime_filter", "sr_rf_create", "sr_rf_insert", "sr_rf_destroy", "sr_rf_get_info", "sr_rf_copy_directory",
    "sr_rf_merge_directory", "sr_rf_evaluate", "sr_scan_add_runtime_filter", "sr_scan_get_rf_stats", "sr_scan_set_rf_adaptive", "sr_rf_copy_in_values", "sr_rf_merge_in_values",
    "sr_xchg_destroy", "sr_xchg_partition", "sr_xchg_hash", "sr_gather", "sr_memcpy", "sr_abi_sizeof", "sr_bandwidth_probe", "sr_flush_l2",
    "sr_chunk_serialized_size", "sr_chunk_serialize", "sr_serde_create", "sr_serde_destroy", "sr_chunk_deserialize",
    "sr_host_alloc", "sr_host_free", "sr_event_create", "sr_event_destroy", "sr_event_record", "sr_event_query", "sr_event_sync",
    "sr_page_decoder_create", "sr_page_decoder_destroy", "sr_pages_decode",
]


class GpuError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"sr_gpu error {code}: {msg}")
        self.code = code


class Context:
    def __init__(self, device=0, stream=None):
        self.h = lib().sr_ctx_create(device, stream)
        if not self.h:
            raise GpuError(abi.SR_ERR_NO_DEVICE, lib().sr_last_error(None).decode())
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            lib().sr_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        # handles created on this context must be destroyed first; tests call close() explicitly
        pass

    def check(self, rc):
        if rc is not None and rc < 0:
            raise GpuError(rc, lib().sr_last_error(self.h).decode())
        return rc

    def sync(self):
        self.check(lib().sr_ctx_sync(self.h))

    @property
    def launches(self):
        return lib().sr_ctx_kernel_launches(self.h)

    @property
    def device_bytes(self):
        return lib().sr_ctx_device_bytes(self.h)

    @property
    def stream(self):
        return lib().sr_ctx_stream(self.h)

    def flush_l2(self):
        self.check(lib().sr_flush_l2(self.h))

    def bandwidth_probe(self, dev_ptr, nbytes):
        out = C.c_uint64(0)
        self.check(lib().sr_bandwidth_probe(self.h, dev_ptr, nbytes, C.byref(out)))
        return out.value

    def join_key_hash(self, keys, log_buckets):
        """host numpy int32/int64 keys -> uint32 buckets (K5)"""
        out = np.zeros(len(keys), dtype=np.uint32)
        typ = abi.NUMPY_TYPE[keys.dtype]
        self.check(lib().sr_join_key_hash(self.h, keys.ctypes.data, typ, len(keys), log_buckets, out.ctypes.data,
                                          abi.MEM_HOST))
        return out


def _copy_dev_to_host(ctx, ptr, nbytes):
    """D2H copy of a raw device pointer through the library's own plumbing call."""
    buf = np.empty(nbytes, dtype=np.uint8)
    if nbytes:
        ctx.check(lib().sr_memcpy(ctx.h, buf.ctypes.data, ptr, nbytes, 1))
    return buf


def chunk_out_to_host(ctx, out):
    """sr_chunk_out -> list of (slot, type, data ndarray, nulls ndarray|None).  Device buffers are copied."""
    ctx.sync()
    res = []
    n = out.num_rows
    for k in range(out.num_cols):
        c = out.cols[k]
        w = abi.TYPE_WIDTH[c.type]
        dt = abi.TYPE_NUMPY.get(c.type)
        if out.mem == abi.MEM_DEVICE:
            raw = _copy_dev_to_host(ctx, c.data, n * w) if n else np.empty(0, dtype=np.uint8)
            nul = (_copy_dev_to_host(ctx, c.nulls, n) if n else np.empty(0, dtype=np.uint8)) if c.nulls else None
        else:
            raw = np.ctypeslib.as_array(C.cast(c.data, C.POINTER(C.c_uint8)), shape=(n * w,)).copy() if n else \
                np.empty(0, dtype=np.uint8)
            nul = np.ctypeslib.as_array(C.cast(c.nulls, C.POINTER(C.c_uint8)), shape=(n,)).copy() \
                if (c.nulls and n) else (np.empty(0, dtype=np.uint8) if c.nulls else None)
        data = raw.view(dt) if dt is not None else raw.view(np.dtype((np.void, 16)))
        res.append((c.slot_id, c.type, data, nul))
    return res


class Scan:
    def __init__(self, ctx, scan_desc):
        self.ctx = ctx
        self.desc = scan_desc
        self.h = lib().sr_scan_create(ctx.h, scan_desc.ref())
        if not self.h:
            ctx.check(lib().sr_last_error_code(ctx.h) or -1)

    def close(self):
        if self.h:
            lib().sr_scan_destroy(self.h)
            self.h = None

    def evaluate(self, chunk):
        sel = np.zeros(chunk.num_rows, dtype=np.uint8)
        self.ctx.check(lib().sr_scan_evaluate(self.h, chunk.ref(), sel.ctypes.data, abi.MEM_HOST))
        return sel

    def filter(self, chunk):
        out = abi.sr_chunk_out()
        self.ctx.check(lib().sr_scan_filter(self.h, chunk.ref(), C.byref(out)))
        return out

    def rf_stats(self, index):
        st = abi.sr_scan_rf_stats()
        self.ctx.check(lib().sr_scan_get_rf_stats(self.h, index, C.byref(st)))
        return st

    def set_rf_adaptive(self, on):
        self.ctx.check(lib().sr_scan_set_rf_adaptive(self.h, 1 if on else 0))

    def add_runtime_filter(self, rf, probe_slot):
        self.ctx.check(lib().sr_scan_add_runtime_filter(self.h, rf.h, probe_slot))
        self._rfs = getattr(self, "_rfs", []) + [rf]  # the filter must outlive the scan


class RuntimeFilter:
    """sr_rf: min/max + SimdBlockFilter-compatible bloom filter (include/sr_gpu_ops.h)"""

    def __init__(self, ctx, key_type=None, expected_rows=0, with_bloom=True, handle=None):
        self.ctx = ctx
        self.h = handle if handle is not None else lib().sr_rf_create(ctx.h, key_type, expected_rows, 1 if with_bloom else 0)
        if not self.h:
            ctx.check(lib().sr_last_error_code(ctx.h) or -1)

    @classmethod
    def from_join(cls, join, key_index=0, with_bloom=True, insert_nulls=False):
        h = lib().sr_join_build_runtime_filter(join.h, key_index, 1 if with_bloom else 0, 1 if insert_nulls else 0)
        return cls(join.ctx, handle=h)

    def close(self):
        if self.h:
            lib().sr_rf_destroy(self.h)
            self.h = None

    def insert(self, chunk, slot, insert_nulls=False):
        self.ctx.check(lib().sr_rf_insert(self.h, chunk.ref(), slot, 1 if insert_nulls else 0))

    def info(self):
        inf = abi.sr_rf_info()
        self.ctx.check(lib().sr_rf_get_info(self.h, C.byref(inf)))
        return inf

    def directory(self):
        logb = self.info().log_num_buckets
        out = np.zeros((8 << logb) if logb else 0, dtype=np.uint32)
        self.ctx.check(lib().sr_rf_copy_directory(self.h, out.ctypes.data, out.nbytes, abi.MEM_HOST))
        return out

    def in_values(self):
        """sorted distinct keys of the IN part (int64 array), or None when the filter has none"""
        out = np.zeros(abi.RF_IN_FILTER_ROW_LIMIT, dtype=np.int64)
        n = lib().sr_rf_copy_in_values(self.h, out.ctypes.data, len(out))
        if n == -1:
            return None
        if n < 0:
            self.ctx.check(n)
        return out[:n].copy()

    def merge_in_values(self, values):
        """values: int64 array of the other filter's IN part, or None when it has none"""
        if values is None:
            self.ctx.check(lib().sr_rf_merge_in_values(self.h, None, -1))
        else:
            v = np.ascontiguousarray(values, dtype=np.int64)
            self.ctx.check(lib().sr_rf_merge_in_values(self.h, v.ctypes.data if v.size else None, len(v)))

    def merge(self, directory, info):
        """directory: uint32 array (host) of the other filter, info: its sr_rf_info"""
        d = np.ascontiguousarray(directory, dtype=np.uint32)
        self.ctx.check(lib().sr_rf_merge_directory(self.h, d.ctypes.data if d.size else None, d.nbytes, abi.MEM_HOST, C.byref(info)))

    def evaluate(self, chunk, slot, selection=None):
        sel = np.zeros(chunk.num_rows, dtype=np.uint8) if selection is None else np.ascontiguousarray(selection, dtype=np.uint8).copy()
        self.ctx.check(lib().sr_rf_evaluate(self.h, chunk.ref(), slot, sel.ctypes.data, abi.MEM_HOST, 0 if selection is None else 1))
        return sel


class Join:
    def __init__(self, ctx, desc):
        self.ctx = ctx
        self.desc = desc
        self.h = lib().sr_join_create(ctx.h, C.byref(desc))
        if not self.h:
            ctx.check(lib().sr_last_error_code(ctx.h) or -1)

    def close(self):
        if self.h:
            lib().sr_join_destroy(self.h)
            self.h = None

    def append_build(self, chunk):
        self.ctx.check(lib().sr_join_append_build(self.h, chunk.ref()))

    def build_finish(self):
        self.ctx.check(lib().sr_join_build_finish(self.h))

    def info(self):
        inf = abi.sr_join_info()
        self.ctx.check(lib().sr_join_get_info(self.h, C.byref(inf)))
        return inf

    def copy_table(self):
        inf = self.info()
        first = np.zeros(max(inf.bucket_size, 1), dtype=np.uint32)
        nxt = np.zeros(inf.build_rows + 1, dtype=np.uint32)
        self.ctx.check(lib().sr_join_copy_table(self.h, first.ctypes.data, nxt.ctypes.data))
        return first[:inf.bucket_size], nxt

    def probe(self, chunk, prober_id=0):
        out = abi.sr_chunk_out()
        self.ctx.check(lib().sr_join_probe(self.h, prober_id, chunk.ref(), C.byref(out)))
        return out

    def probe_remain(self):
        """POST_PROBE rows of a RIGHT / FULL join (device chunk owned by the join)"""
        out = abi.sr_chunk_out()
        self.ctx.check(lib().sr_join_probe_remain(self.h, C.byref(out)))
        return out

    def probe_indexes(self, n, prober_id=0):
        pi, bi = C.c_void_p(), C.c_void_p()
        self.ctx.check(lib().sr_join_probe_indexes(self.h, prober_id, C.byref(pi), C.byref(bi)))
        self.ctx.sync()
        if n == 0:
            return np.empty(0, dtype=np.uint32), np.empty(0, dtype=np.uint32)
        return (_copy_dev_to_host(self.ctx, pi.value, 4 * n).view(np.uint32),
                _copy_dev_to_host(self.ctx, bi.value, 4 * n).view(np.uint32))


class Agg:
    def __init__(self, ctx, desc=None, handle=None):
        self.ctx = ctx
        self.desc = desc
        self.owned = handle is None
        self.h = handle if handle is not None else lib().sr_agg_create(ctx.h, C.byref(desc))
        if not self.h:
            ctx.check(lib().sr_last_error_code(ctx.h) or -1)

    def close(self):
        if self.h and self.owned:
            lib().sr_agg_destroy(self.h)
        self.h = None

    def push(self, chunk):
        self.ctx.check(lib().sr_agg_push(self.h, chunk.ref()))

    def finish(self):
        self.ctx.check(lib().sr_agg_sink_finish(self.h))

    def merge(self, other):
        self.ctx.check(lib().sr_agg_merge(self.h, other.h))

    def reset(self):
        self.ctx.check(lib().sr_agg_reset(self.h))

    def current_groups(self):
        return self.ctx.check(lib().sr_agg_current_groups(self.h))

    def convert_to_states(self, chunk):
        """pass-through leg of the streaming aggregate: rows -> intermediate rows (device chunk owned by the handle)"""
        out = abi.sr_chunk_out()
        self.ctx.check(lib().sr_agg_convert_to_states(self.h, chunk.ref(), C.byref(out)))
        return out

    def push_selective(self, chunk):
        """SELECTIVE_PREAGG: aggregate the rows whose group exists, return the others as intermediate rows (sr_chunk_out)"""
        out = abi.sr_chunk_out()
        self.ctx.check(lib().sr_agg_push_selective(self.h, chunk.ref(), C.byref(out)))
        return out

    def dense_state(self):
        """[(device_ptr, count, elem_type, reduce)] -- the element-wise mergeable arrays of a dense table"""
        n_max = 1 + 3 * abi.SR_MAX_AGG_FNS
        arr = (abi.sr_agg_state_array * n_max)()
        n = C.c_int32(0)
        self.ctx.check(lib().sr_agg_dense_state(self.h, arr, n_max, C.byref(n)))
        return [(arr[k].data, arr[k].count, arr[k].elem_type, arr[k].reduce) for k in range(n.value)]

    @property
    def num_groups(self):
        return self.ctx.check(lib().sr_agg_num_groups(self.h))

    def pull(self, max_rows=1 << 62, mem=abi.MEM_HOST):
        out = abi.sr_chunk_out()
        self.ctx.check(lib().sr_agg_pull(self.h, max_rows, mem, C.byref(out)))
        return out

    def result(self):
        """finish + pull everything to the host -> list of (slot, type, data, nulls)"""
        self.finish()
        out = self.pull()
        return chunk_out_to_host(self.ctx, out)


def two_phase_descs(desc):
    """sr_agg_two_phase_descs: (first-phase desc, merge-phase desc) of a single-phase aggregate desc"""
    p1, p2 = abi.sr_agg_desc(), abi.sr_agg_desc()
    rc = lib().sr_agg_two_phase_descs(C.byref(desc), C.byref(p1), C.byref(p2))
    if rc != 0:
        raise GpuError(rc, "sr_agg_two_phase_descs: the aggregate cannot be split into two phases (128-bit states or too many functions)")
    return p1, p2


def chunk_out_as_view(out):
    """device sr_chunk_out -> abi.Chunk-like object usable as the input of another operator (no copy)"""
    class _View:
        pass
    v = _View()
    v.view = abi.sr_chunk_view(C.cast(out.cols, C.POINTER(abi.sr_col_view)), out.num_cols, out.mem, out.num_rows)
    v.num_rows = out.num_rows
    v._keep = out
    v.ref = lambda: C.byref(v.view)
    return v


class Fragment:
    def __init__(self, ctx, scan_desc, joins, agg_desc, mode=0):
        """joins: list of (Join, probe_key_slot, [payload build slots]); mode: 0 auto, 1 fused cascade,
        2 selection-vector passes"""
        self.ctx = ctx
        self._keep = (scan_desc, joins, agg_desc)
        d = abi.sr_fragment_desc()
        d.scan = scan_desc.desc
        d.num_joins = len(joins)
        d.mode_hint = mode
        for k, (j, slot, payload) in enumerate(joins):
            d.joins[k].join = j.h
            d.joins[k].probe_key_slot = slot
            d.joins[k].num_payload = len(payload)
            for q, s in enumerate(payload):
                d.joins[k].payload_build_slots[q] = s
        d.agg = agg_desc
        self.desc = d
        self.h = lib().sr_fragment_create(ctx.h, C.byref(d))
        if not self.h:
            ctx.check(lib().sr_last_error_code(ctx.h) or -1)
        self.agg = Agg(ctx, agg_desc, handle=lib().sr_fragment_agg(self.h))

    def close(self):
        if self.h:
            lib().sr_fragment_destroy(self.h)
            self.h = None

    def push(self, chunk):
        self.ctx.check(lib().sr_fragment_push(self.h, chunk.ref()))

    def reset(self):
        self.ctx.check(lib().sr_fragment_reset(self.h))

    def last_pass_ms(self):
        """device ms of the (stream, gather-join, final) passes of the last push; None in fused-cascade mode"""
        ms = (C.c_float * 3)()
        rc = lib().sr_fragment_last_pass_ms(self.h, ms)
        if rc == abi.SR_ERR_STATE:
            return None
        self.ctx.check(rc)
        return [float(x) for x in ms]

    def plan(self):
        p = abi.sr_fragment_plan()
        self.ctx.check(lib().sr_fragment_get_plan(self.h, C.byref(p)))
        nj = p.num_joins
        return {"order": list(p.order[:nj]), "bitmap_in_smem": list(p.bitmap_in_smem[:nj]),
                "pass_rate": [round(x, 4) for x in p.pass_rate[:nj]], "smem_bytes": p.smem_bytes, "grid": p.grid,
                "block": p.block, "agg_in_smem": bool(p.agg_in_smem),
                "mode": {1: "fused-cascade", 2: "selection-vector-passes"}.get(p.mode, p.mode),
                "num_stream_joins": p.num_stream_joins, "num_gather_passes": p.num_gather_passes,
                "pred_rate": round(p.pred_rate, 4)}

    @property
    def rows_passed(self):
        return self.ctx.check(lib().sr_fragment_rows_passed(self.h))


def chunk_serialize(ctx, chunk, row_begin=0, row_end=None):
    """ChunkPB.data bytes of rows [row_begin, row_end) of `chunk` (host or device columns) -> (uint8 ndarray, sr_chunk_pb_meta)"""
    row_end = chunk.num_rows if row_end is None else row_end
    n = ctx.check(lib().sr_chunk_serialized_size(chunk.ref(), row_begin, row_end))
    buf = np.zeros(n, dtype=np.uint8)
    meta = abi.sr_chunk_pb_meta()
    ctx.check(lib().sr_chunk_serialize(ctx.h, chunk.ref(), row_begin, row_end, buf.ctypes.data, n, abi.MEM_HOST, C.byref(meta)))
    return buf, meta


class PageDecoder:
    """sr_page_decoder: frame-of-reference / plain data pages -> a device column"""

    def __init__(self, ctx):
        self.ctx = ctx
        self.h = lib().sr_page_decoder_create(ctx.h)

    def close(self):
        if self.h:
            lib().sr_page_decoder_destroy(self.h)
            self.h = None

    def decode(self, encoding, typ, pages, out_ptr, out_capacity, mem=abi.MEM_HOST):
        """pages: list of uint8 numpy arrays (host) or (pointer, size) pairs; out_ptr: device pointer.  -> rows"""
        views = (abi.sr_page_view * max(1, len(pages)))()
        keep = []
        for k, pg in enumerate(pages):
            if isinstance(pg, tuple):
                views[k].data, views[k].size = pg
            else:
                a = np.ascontiguousarray(pg, dtype=np.uint8)
                keep.append(a)
                views[k].data, views[k].size = (a.ctypes.data if a.size else None), a.size
        rows = C.c_int64(0)
        self.ctx.check(lib().sr_pages_decode(self.h, encoding, typ, views, len(pages), mem, out_ptr, out_capacity, C.byref(rows)))
        return rows.value


class Serde:
    """sr_serde: owner of the device columns a ChunkPB.data payload deserialises into"""

    def __init__(self, ctx):
        self.ctx = ctx
        self.h = lib().sr_serde_create(ctx.h)

    def close(self):
        if self.h:
            lib().sr_serde_destroy(self.h)
            self.h = None

    def deserialize(self, payload, meta):
        out = abi.sr_chunk_out()
        payload = np.ascontiguousarray(payload, dtype=np.uint8)
        self.ctx.check(lib().sr_chunk_deserialize(self.h, payload.ctypes.data, payload.nbytes, abi.MEM_HOST, C.byref(meta), C.byref(out)))
        return out


class Xchg:
    def __init__(self, ctx, part_desc):
        self.ctx = ctx
        self.desc = part_desc
        self.h = lib().sr_xchg_create(ctx.h, C.byref(part_desc))
        if not self.h:
            ctx.check(lib().sr_last_error_code(ctx.h) or -1)

    def close(self):
        if self.h:
            lib().sr_xchg_destroy(self.h)
            self.h = None

    def hash(self, chunk):
        n = chunk.num_rows
        hv = np.zeros(n, dtype=np.uint32)
        ch = np.zeros(n, dtype=np.uint32)
        self.ctx.check(lib().sr_xchg_hash(self.h, chunk.ref(), hv.ctypes.data, ch.ctypes.data, abi.MEM_HOST))
        return hv, ch

    def partition(self, chunk):
        out = abi.sr_chunk_out()
        offs = np.zeros(self.desc.num_channels + 1, dtype=np.int64)
        self.ctx.check(lib().sr_xchg_partition(self.h, chunk.ref(), C.byref(out), offs.ctypes.data))
        return out, offs
