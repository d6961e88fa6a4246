"""ctypes binding of liblambdipy_b200.so (C ABI: include/lambdipy_b200.h).

The library is CUDA-only: there is no CPU implementation behind it, and nothing here falls back
to one.  `load()` raises if the shared object is missing (build it with
`python -m lambdipy_b200.build`); `Context()` raises `NoDeviceError` without a B200.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LAMBDIPY_B200_LIB") or os.path.join(_HERE, "liblambdipy_b200.so")  # (override: diagnostic builds)

# return codes / status / flags (mirror include/lambdipy_b200.h)
LB2_OK, LB2_E_CUDA, LB2_E_ARG, LB2_E_CAPACITY, LB2_E_IO, LB2_E_NODEVICE, LB2_E_STATE = 0, -1, -2, -3, -4, -5, -6
ST_OK, ST_NOT_ELF, ST_NOT_ELF64LE, ST_BAD_TYPE, ST_NO_SECTIONS, ST_XINDEX = 0, 1, 2, 3, 4, 5
ST_UNSUPPORTED_LAYOUT, ST_BAD_NOTES, ST_PLANNER_LIMIT, ST_MALFORMED = 6, 7, 8, -1
F_NO_MERGE_NOTES = 1
TREE_FALLBACK_HOST_STRIP, TREE_TOLERATE_NON_ELF, TREE_DRY_RUN, TREE_CLEANUP = 0x100, 0x200, 0x400, 0x800

EXPORTS = [
    "lb2_ctx_create", "lb2_ctx_destroy", "lb2_last_error", "lb2_version", "lb2_sm_count",
    "lb2_dev_alloc", "lb2_dev_free", "lb2_pinned_alloc", "lb2_pinned_free",
    "lb2_memcpy_h2d", "lb2_memcpy_d2h", "lb2_memset_d",
    "lb2_strip_device_async", "lb2_batch_results", "lb2_strip_host", "lb2_strip_tree",
    "lb2_plan_device", "lb2_corpus_fill", "lb2_corpus_scatter",
    "lb2_strip_device_chunked", "lb2_tree_prepare", "lb2_strip_tree_ex", "lb2_tree_cleanup",
    "lb2_deflate_device", "lb2_gzip_segments",
]


class Stats(C.Structure):
    _fields_ = [
        ("n_files", C.c_uint32), ("n_ok", C.c_uint32), ("n_unsupported", C.c_uint32), ("overflow", C.c_uint32),
        ("in_bytes", C.c_uint64), ("out_bytes", C.c_uint64), ("copy_bytes", C.c_uint64), ("header_bytes", C.c_uint64),
        ("n_tiles", C.c_uint64), ("out_bytes_needed", C.c_uint64),
        ("plan_ms", C.c_float), ("compact_ms", C.c_float), ("h2d_ms", C.c_float), ("d2h_ms", C.c_float),
        ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class TreeStats(C.Structure):
    _fields_ = [
        ("n_selected", C.c_uint32), ("n_gpu", C.c_uint32), ("n_fallback", C.c_uint32), ("n_skipped", C.c_uint32),
        ("n_failed", C.c_uint32), ("n_removed", C.c_uint32),
        ("in_bytes", C.c_uint64), ("out_bytes", C.c_uint64),
        ("walk_read_s", C.c_double), ("gpu_s", C.c_double), ("write_s", C.c_double), ("fallback_s", C.c_double),
        ("read_cpu_s", C.c_double), ("write_cpu_s", C.c_double), ("dma_wait_s", C.c_double), ("io_threads", C.c_uint32), ("n_batches", C.c_uint32),
        ("batch", Stats),
    ]

    def as_dict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_ if k != "batch"}
        d["batch"] = self.batch.as_dict()
        return d


class GzipStats(C.Structure):
    _fields_ = [
        ("in_bytes", C.c_uint64), ("out_bytes", C.c_uint64), ("kernel_ms", C.c_float),
        ("read_s", C.c_double), ("upload_s", C.c_double), ("download_s", C.c_double), ("write_s", C.c_double),
        ("setup_s", C.c_double), ("n_chunks", C.c_uint64), ("n_windows", C.c_uint32), ("io_threads", C.c_uint32),
        ("phase_cycles", C.c_uint64 * 6),
    ]
    PHASES = ("hash_sort", "scatter", "match", "parse", "huffman_header", "emit")

    def as_dict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_ if k != "phase_cycles"}
        d["phase_cycles"] = dict(zip(self.PHASES, list(self.phase_cycles)))
        return d


class GzSegment(C.Structure):
    _fields_ = [("data", C.c_void_p), ("path", C.c_char_p), ("len", C.c_uint64)]


class FillRegion(C.Structure):
    _fields_ = [("offset", C.c_uint64), ("len", C.c_uint64)]


class NativeError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("lambdipy_b200: rc=%d: %s" % (code, msg))
        self.code = code


class NoDeviceError(NativeError):
    pass


_lib = None


def load():
    """dlopen the in-tree CUDA library; raise (never fall back) when it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("%s is missing: run `python -m lambdipy_b200.build` (needs nvcc); "
                          "there is no CPU fallback for the strip path" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp, u64p, i32p = C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_int32)
    lib.lb2_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
    lib.lb2_ctx_create.restype = C.c_int
    lib.lb2_ctx_destroy.argtypes = [vp]
    lib.lb2_ctx_destroy.restype = None
    lib.lb2_last_error.argtypes = [vp]
    lib.lb2_last_error.restype = C.c_char_p
    lib.lb2_version.restype = C.c_char_p
    lib.lb2_sm_count.argtypes = [vp]
    lib.lb2_sm_count.restype = C.c_int
    lib.lb2_dev_alloc.argtypes = [vp, C.c_uint64]
    lib.lb2_dev_alloc.restype = vp
    lib.lb2_dev_free.argtypes = [vp, vp]
    lib.lb2_dev_free.restype = None
    lib.lb2_pinned_alloc.argtypes = [vp, C.c_uint64]
    lib.lb2_pinned_alloc.restype = vp
    lib.lb2_pinned_free.argtypes = [vp, vp]
    lib.lb2_pinned_free.restype = None
    lib.lb2_memcpy_h2d.argtypes = [vp, vp, vp, C.c_uint64]
    lib.lb2_memcpy_h2d.restype = C.c_int
    lib.lb2_memcpy_d2h.argtypes = [vp, vp, vp, C.c_uint64]
    lib.lb2_memcpy_d2h.restype = C.c_int
    lib.lb2_memset_d.argtypes = [vp, vp, C.c_int, C.c_uint64]
    lib.lb2_memset_d.restype = C.c_int
    lib.lb2_strip_device_async.argtypes = [vp, vp, u64p, u64p, C.c_uint32, vp, C.c_uint64, C.c_uint32, vp]
    lib.lb2_strip_device_async.restype = C.c_int
    lib.lb2_batch_results.argtypes = [vp, u64p, u64p, i32p, C.POINTER(Stats)]
    lib.lb2_batch_results.restype = C.c_int
    lib.lb2_strip_host.argtypes = [vp, vp, u64p, u64p, C.c_uint32, vp, C.c_uint64, u64p, u64p, i32p, C.c_uint32,
                                   C.POINTER(Stats)]
    lib.lb2_strip_host.restype = C.c_int
    lib.lb2_strip_tree.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_uint32, C.POINTER(TreeStats)]
    lib.lb2_strip_tree.restype = C.c_int
    lib.lb2_plan_device.argtypes = [vp, vp, u64p, u64p, C.c_uint32, C.c_uint32, u64p, i32p, C.POINTER(Stats)]
    lib.lb2_plan_device.restype = C.c_int
    lib.lb2_corpus_fill.argtypes = [vp, vp, C.POINTER(FillRegion), C.c_uint32, C.c_uint64, vp]
    lib.lb2_corpus_fill.restype = C.c_int
    lib.lb2_corpus_scatter.argtypes = [vp, vp, vp, C.c_uint64, u64p, u64p, u64p, C.c_uint32]
    lib.lb2_corpus_scatter.restype = C.c_int
    lib.lb2_strip_device_chunked.argtypes = [vp, vp, u64p, u64p, C.c_uint32, vp, C.c_uint64, C.c_uint64, C.c_uint32, vp,
                                             vp, vp, u64p, i32p, C.POINTER(Stats)]
    lib.lb2_strip_device_chunked.restype = C.c_int
    lib.lb2_strip_tree_ex.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_uint32, C.c_char_p, C.POINTER(TreeStats)]
    lib.lb2_strip_tree_ex.restype = C.c_int
    lib.lb2_tree_cleanup.argtypes = [C.c_char_p, C.c_char_p, C.POINTER(C.c_uint32)]
    lib.lb2_tree_cleanup.restype = C.c_int
    lib.lb2_tree_prepare.argtypes = [vp, C.c_uint64]
    lib.lb2_tree_prepare.restype = C.c_int
    lib.lb2_deflate_device.argtypes = [vp, vp, C.c_uint64, C.c_uint32, C.c_uint32, vp, C.c_uint64, u64p,
                                       C.POINTER(C.c_uint32), C.POINTER(GzipStats), vp]
    lib.lb2_deflate_device.restype = C.c_int
    lib.lb2_gzip_segments.argtypes = [vp, C.POINTER(GzSegment), C.c_uint32, C.c_char_p, C.c_char_p, C.c_uint32,
                                      C.POINTER(GzipStats)]
    lib.lb2_gzip_segments.restype = C.c_int
    _lib = lib
    return lib


# consumer callback of lb2_strip_device_chunked (include/lambdipy_b200.h: lb2_chunk_fn)
CHUNK_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.POINTER(C.c_uint64),
                       C.POINTER(C.c_uint64), C.POINTER(C.c_int32), C.POINTER(Stats))


class Context:
    """One CUDA device + the library's workspaces.  Not thread-safe (one per thread and device)."""

    def __init__(self, device=0):
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.lb2_ctx_create(int(device), C.byref(h))
        if rc != LB2_OK:
            msg = (self.lib.lb2_last_error(None) or b"").decode()
            raise (NoDeviceError if rc == LB2_E_NODEVICE else NativeError)(rc, msg)
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.lb2_ctx_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc):
        if rc != LB2_OK:
            raise NativeError(rc, (self.lib.lb2_last_error(self.h) or b"").decode())

    @property
    def sm_count(self):
        return self.lib.lb2_sm_count(self.h)

    # -- raw memory helpers -------------------------------------------------------------------
    def dev_alloc(self, n):
        p = self.lib.lb2_dev_alloc(self.h, n)
        if not p:
            raise NativeError(LB2_E_CUDA, (self.lib.lb2_last_error(self.h) or b"").decode())
        return p

    def dev_free(self, p):
        self.lib.lb2_dev_free(self.h, p)

    def pinned_alloc(self, n):
        p = self.lib.lb2_pinned_alloc(self.h, n)
        if not p:
            raise NativeError(LB2_E_CUDA, (self.lib.lb2_last_error(self.h) or b"").decode())
        return p

    def pinned_free(self, p):
        self.lib.lb2_pinned_free(self.h, p)

    def h2d(self, d, h, n):
        self.check(self.lib.lb2_memcpy_h2d(self.h, d, h, n))

    def d2h(self, h, d, n):
        self.check(self.lib.lb2_memcpy_d2h(self.h, h, d, n))
