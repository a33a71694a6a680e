"""ctypes binding of ``librecometrics_b200.so`` (the C-ABI declared in ``include/recometrics_b200.h``).

This is the only door from Python into the product's native code.  It fails loudly when the library
is missing or when no CUDA device is usable: there is no CPU fallback anywhere in the package.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# RMB200_LIB: developer override, loads another build of the same library (e.g. to time two builds side by side)
LIB_PATH = os.environ.get("RMB200_LIB") or os.path.join(_HERE, "librecometrics_b200.so")

OK, ERR_BAD_ARG, ERR_NO_DEVICE, ERR_CUDA, ERR_OOM, ERR_INTERRUPTED, ERR_UNSUPPORTED, ERR_RUNTIME = range(8)
MAX_K = 384     # largest k_metrics of the selection kernels; above it the call takes the full-order path

# order of the ten outputs in the C signature (src/recometrics_signatures.hpp:56-65 of the reference)
METRIC_ORDER = ("p", "tp", "r", "ap", "tap", "ndcg", "hit", "rr", "roc", "pr")
TOPK_METRICS = METRIC_ORDER[:8]

EXPORTS = (
    "rmb200_calc_metrics_f32", "rmb200_calc_metrics_f64",
    "rmb200_calc_metrics_ex_f32", "rmb200_calc_metrics_ex_f64",
    "rmb200_calc_metrics_exposure_f32", "rmb200_calc_metrics_exposure_f64", "rmb200_exposure_stats", "rmb200_sizeof_exposure",
    "rmb200_calc_metrics_beyond_f32", "rmb200_calc_metrics_beyond_f64", "rmb200_sizeof_beyond", "rmb200_item_popularity",
    "rmb200_calc_metrics_serendipity_f32", "rmb200_calc_metrics_serendipity_f64", "rmb200_sizeof_serendipity",
    "rmb200_device_count", "rmb200_version", "rmb200_last_error",
    "rmb200_request_interrupt", "rmb200_measure_fma_peak", "rmb200_release_workspace",
    "rmb200_sizeof_extra", "rmb200_sizeof_timing",
    "rmb200_split_selected_users_f32", "rmb200_split_selected_users_f64",
    "rmb200_split_separate_users_f32", "rmb200_split_separate_users_f64",
    "rmb200_split_joined_users_f32", "rmb200_split_joined_users_f64",
    "rmb200_split_plan", "rmb200_split_free", "rmb200_sizeof_split",
)


class Timing(ctypes.Structure):
    _fields_ = [
        ("total_ms", ctypes.c_double), ("h2d_ms", ctypes.c_double), ("prep_ms", ctypes.c_double),
        ("score_select_ms", ctypes.c_double), ("metrics_ms", ctypes.c_double), ("d2h_ms", ctypes.c_double),
        ("kernel_launches", ctypes.c_int64), ("h2d_bytes", ctypes.c_int64), ("d2h_bytes", ctypes.c_int64),
        ("scoring_path", ctypes.c_int64), ("filter_fallback_batches", ctypes.c_int64),
        ("dominant_kernel_ms", ctypes.c_double), ("filter_retry_rows", ctypes.c_int64),
        ("filter_fallback_users", ctypes.c_int64), ("filter_err_ratio_max", ctypes.c_double),
        ("noise_handback_users", ctypes.c_int64), ("devices_used", ctypes.c_int64),
    ]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


class Extra(ctypes.Structure):
    _fields_ = [
        ("struct_size", ctypes.c_int32), ("device", ctypes.c_int32),
        ("user_begin", ctypes.c_int32), ("user_end", ctypes.c_int32),
        ("inputs_on_device", ctypes.c_int32), ("strict_min_pos_test", ctypes.c_int32),
        ("topk_items", ctypes.c_void_p), ("topk_scores", ctypes.c_void_p),
        ("pos_rank", ctypes.c_void_p), ("status", ctypes.c_void_p),
        ("timing", ctypes.POINTER(Timing)),
        ("scoring_path", ctypes.c_int32), ("skip_row_copy", ctypes.c_int32),
        ("metric_means", ctypes.c_void_p), ("metric_counts", ctypes.c_void_p),
        ("has_nan_bits", ctypes.c_int32), ("filter_stats", ctypes.c_int32), ("nan_bits", ctypes.c_uint64),
        ("devices", ctypes.POINTER(ctypes.c_int32)), ("n_devices", ctypes.c_int32), ("reserved0", ctypes.c_int32),
    ]


class Exposure(ctypes.Structure):
    """rmb200_exposure_t (include/recometrics_b200.h): item exposure of a call's ranked lists."""
    _fields_ = [
        ("struct_size", ctypes.c_int32), ("reserved0", ctypes.c_int32), ("item_counts", ctypes.c_void_p),
        ("users", ctypes.c_int64), ("entries", ctypes.c_int64), ("items_covered", ctypes.c_int64),
        ("coverage", ctypes.c_double), ("gini", ctypes.c_double), ("entropy_bits", ctypes.c_double),
    ]

    def catalogue(self):
        """The statistics as the front-ends return them (``EvalResult.catalogue``)."""
        return {"Coverage@K": float(self.coverage), "Gini@K": float(self.gini), "Entropy@K": float(self.entropy_bits),
                "users": int(self.users), "entries": int(self.entries), "items_covered": int(self.items_covered)}


def make_exposure(item_counts=None):
    """rmb200_exposure_t asking for the exposure of a call; `item_counts`: int64 numpy array [n], device address or None."""
    e = Exposure()
    e.struct_size = ctypes.sizeof(Exposure)
    e.item_counts = _vp(item_counts)
    return e


# order of the three beyond-accuracy rows in rmb200_beyond_t (and of its means / counts) and their result keys
BEYOND_KEYS = (("novelty", "Novelty@K"), ("avg_popularity", "AvgPop@K"), ("ild", "ILD@K"))


class Beyond(ctypes.Structure):
    """rmb200_beyond_t (include/recometrics_b200.h): Novelty / AvgPop / ILD rows of a call's ranked lists."""
    _fields_ = [
        ("struct_size", ctypes.c_int32), ("reserved0", ctypes.c_int32),
        ("item_popularity", ctypes.c_void_p), ("popularity_users", ctypes.c_int64),
        ("novelty", ctypes.c_void_p), ("avg_popularity", ctypes.c_void_p), ("ild", ctypes.c_void_p),
        ("means", ctypes.c_void_p), ("counts", ctypes.c_void_p),
    ]


def make_beyond(rows, item_popularity=None, popularity_users=0, means=None, counts=None):
    """rmb200_beyond_t; `rows` maps "novelty" / "avg_popularity" / "ild" -> array, device address or None; the other
    arguments are int64 [n] counts, U, and the optional [3 * W] means / counts (arrays or device addresses)."""
    b = Beyond()
    b.struct_size = ctypes.sizeof(Beyond)
    b.item_popularity = _vp(item_popularity)
    b.popularity_users = int(popularity_users)
    for name, _ in BEYOND_KEYS:
        setattr(b, name, _vp(rows.get(name)))
    b.means = _vp(means)
    b.counts = _vp(counts)
    return b


# order of the two history rows in rmb200_serendipity_t (and of its means / counts) and their result keys
SERENDIPITY_KEYS = (("unexpectedness", "Unexpectedness@K"), ("serendipity", "Serendipity@K"))


class Serendipity(ctypes.Structure):
    """rmb200_serendipity_t (include/recometrics_b200.h): Unexpectedness / Serendipity rows of a call's ranked lists."""
    _fields_ = [
        ("struct_size", ctypes.c_int32), ("reserved0", ctypes.c_int32),
        ("unexpectedness", ctypes.c_void_p), ("serendipity", ctypes.c_void_p),
        ("means", ctypes.c_void_p), ("counts", ctypes.c_void_p),
    ]


def make_serendipity(rows, means=None, counts=None):
    """rmb200_serendipity_t; `rows` maps "unexpectedness" / "serendipity" -> array, device address or None; `means` /
    `counts` are the optional [2 * W] tables (arrays or device addresses)."""
    s = Serendipity()
    s.struct_size = ctypes.sizeof(Serendipity)
    for name, _ in SERENDIPITY_KEYS:
        setattr(s, name, _vp(rows.get(name)))
    s.means = _vp(means)
    s.counts = _vp(counts)
    return s


class Csr(ctypes.Structure):
    _fields_ = [("rows", ctypes.c_int32), ("cols", ctypes.c_int32), ("nnz", ctypes.c_int64),
                ("indptr", ctypes.c_void_p), ("indices", ctypes.c_void_p), ("values", ctypes.c_void_p)]


class Split(ctypes.Structure):
    """rmb200_split_t (include/recometrics_b200.h)."""
    _fields_ = [
        ("train", Csr), ("test", Csr), ("rem", Csr),
        ("users_test", ctypes.c_void_p), ("n_users_test", ctypes.c_int32), ("value_bytes", ctypes.c_int32),
        ("rows_sorted_on_device", ctypes.c_int32), ("device", ctypes.c_int32),
        ("total_ms", ctypes.c_double), ("plan_ms", ctypes.c_double), ("h2d_ms", ctypes.c_double),
        ("kernel_ms", ctypes.c_double), ("d2h_ms", ctypes.c_double),
        ("kernel_launches", ctypes.c_int64), ("h2d_bytes", ctypes.c_int64), ("d2h_bytes", ctypes.c_int64),
        ("owner", ctypes.c_void_p),
    ]
    TIMING = ("total_ms", "plan_ms", "h2d_ms", "kernel_ms", "d2h_ms", "kernel_launches", "h2d_bytes", "d2h_bytes",
              "rows_sorted_on_device", "device")


class NativeLibraryError(RuntimeError):
    pass


_lib = None


def load():
    """Load the shared library (once).  Raises NativeLibraryError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryError(
            "recometrics_b200: %s is missing -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C recometrics_b200/csrc`.  There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name in EXPORTS:
        if not hasattr(lib, name):
            raise NativeLibraryError("recometrics_b200: %s does not export %s" % (LIB_PATH, name))
    lib.rmb200_device_count.restype = ctypes.c_int
    lib.rmb200_version.restype = ctypes.c_int
    lib.rmb200_sizeof_extra.restype = ctypes.c_int
    lib.rmb200_sizeof_timing.restype = ctypes.c_int
    lib.rmb200_sizeof_split.restype = ctypes.c_int
    lib.rmb200_sizeof_exposure.restype = ctypes.c_int
    lib.rmb200_sizeof_beyond.restype = ctypes.c_int
    lib.rmb200_sizeof_serendipity.restype = ctypes.c_int
    if (lib.rmb200_sizeof_extra() != ctypes.sizeof(Extra) or lib.rmb200_sizeof_timing() != ctypes.sizeof(Timing)
            or lib.rmb200_sizeof_split() != ctypes.sizeof(Split) or lib.rmb200_sizeof_exposure() != ctypes.sizeof(Exposure)
            or lib.rmb200_sizeof_beyond() != ctypes.sizeof(Beyond) or lib.rmb200_sizeof_serendipity() != ctypes.sizeof(Serendipity)):
        raise NativeLibraryError("recometrics_b200: %s was built from a different include/recometrics_b200.h (struct sizes differ); rebuild it" % LIB_PATH)
    lib.rmb200_last_error.restype = ctypes.c_char_p
    lib.rmb200_request_interrupt.restype = None
    lib.rmb200_release_workspace.restype = None
    lib.rmb200_measure_fma_peak.restype = ctypes.c_double
    lib.rmb200_measure_fma_peak.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_double)]
    for name in EXPORTS[:7]:
        getattr(lib, name).restype = ctypes.c_int
    lib.rmb200_exposure_stats.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.POINTER(Exposure)]
    for name in ("rmb200_calc_metrics_beyond_f32", "rmb200_calc_metrics_beyond_f64", "rmb200_item_popularity",
                 "rmb200_calc_metrics_serendipity_f32", "rmb200_calc_metrics_serendipity_f64"):
        getattr(lib, name).restype = ctypes.c_int
    lib.rmb200_item_popularity.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                           ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p]
    for name in EXPORTS:
        if name.startswith("rmb200_split_") and name != "rmb200_split_free":
            getattr(lib, name).restype = ctypes.c_int
    lib.rmb200_split_free.restype = None
    lib.rmb200_split_free.argtypes = [ctypes.POINTER(Split)]
    _lib = lib
    return lib


def device_count():
    return int(load().rmb200_device_count())


def release_workspace():
    """Give the device scratch cached between calls back to the driver."""
    load().rmb200_release_workspace()


def last_error():
    return load().rmb200_last_error().decode("utf-8", "replace")


def measure_fma_peak(device=-1, dtype=np.float32):
    ms = ctypes.c_double(0)
    v = load().rmb200_measure_fma_peak(int(device), 4 if np.dtype(dtype) == np.float32 else 8, ctypes.byref(ms))
    if v < 0:
        raise RuntimeError("rmb200_measure_fma_peak failed: " + last_error())
    return float(v), float(ms.value)


def raise_for_status(rc):
    """Map rmb200_status to the exceptions the reference's Cython layer would surface
    (``except +`` in recometrics/wrapper.pyx:62,145: bad_alloc -> MemoryError, runtime_error -> RuntimeError)."""
    if rc == OK:
        return
    msg = last_error()
    if rc == ERR_BAD_ARG:
        raise ValueError(msg)
    if rc == ERR_OOM:
        raise MemoryError(msg)
    if rc == ERR_INTERRUPTED:
        raise RuntimeError("Error: procedure was interrupted.")
    if rc == ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    if rc == ERR_NO_DEVICE:
        raise RuntimeError("recometrics_b200 needs a CUDA device (no CPU fallback): " + msg)
    if rc == ERR_RUNTIME:          # the reference's own std::runtime_error, message included (Cython `except +` -> RuntimeError)
        raise RuntimeError(msg)
    raise RuntimeError("recometrics_b200 CUDA failure: " + msg)


def _vp(x):
    """void* from a numpy array (host), an int (device address) or None."""
    if x is None:
        return ctypes.c_void_p(None)
    if isinstance(x, (int, np.integer)):
        return ctypes.c_void_p(int(x))
    if x.size == 0:
        return ctypes.c_void_p(None)
    return ctypes.c_void_p(x.ctypes.data)


def calc_metrics(dtype, A, lda, B, ldb, m, n, k, trp, tri, tep, tei, tev, k_metrics, cumulative,
                 break_ties_with_noise, outs, consider_cold_start, min_items_pool, min_pos_test,
                 nthreads=1, seed=1, item_biases=None, extra=None, exposure=None, beyond=None, serendipity=None):
    """Thin call into rmb200_calc_metrics_ex_{f32,f64} (rmb200_calc_metrics_exposure_{f32,f64} with an `exposure` struct,
    rmb200_calc_metrics_beyond_{f32,f64} with a `beyond` struct, rmb200_calc_metrics_serendipity_{f32,f64} with a
    `serendipity` struct).  Array arguments are numpy arrays (host memory), raw integer addresses (device memory, with
    extra.inputs_on_device=1) or None.  `outs` maps metric name -> array/address/None in METRIC_ORDER.  Returns the status
    code."""
    lib = load()
    if serendipity is not None:
        kind = "serendipity"
    else:
        kind = "ex" if exposure is None and beyond is None else ("exposure" if beyond is None else "beyond")
    fn = getattr(lib, "rmb200_calc_metrics_%s_%s" % (kind, "f32" if np.dtype(dtype) == np.float32 else "f64"))
    args = [
        _vp(A), ctypes.c_size_t(int(lda)), _vp(B), ctypes.c_size_t(int(ldb)),
        ctypes.c_int32(int(m)), ctypes.c_int32(int(n)), ctypes.c_int32(int(k)),
        _vp(trp), _vp(tri), _vp(tep), _vp(tei), _vp(tev),
        ctypes.c_int32(int(k_metrics)), ctypes.c_int(int(bool(cumulative))), ctypes.c_int(int(bool(break_ties_with_noise))),
    ]
    args += [_vp(outs.get(q)) for q in METRIC_ORDER]
    args += [
        ctypes.c_int(int(bool(consider_cold_start))), ctypes.c_int32(int(min_items_pool)), ctypes.c_int32(int(min_pos_test)),
        ctypes.c_int32(int(nthreads)), ctypes.c_uint64(int(seed)),
        _vp(item_biases), ctypes.byref(extra) if extra is not None else ctypes.c_void_p(None),
    ]
    if kind != "ex":
        args.append(ctypes.byref(exposure) if exposure is not None else ctypes.c_void_p(None))
    if kind in ("beyond", "serendipity"):
        args.append(ctypes.byref(beyond) if beyond is not None else ctypes.c_void_p(None))
    if serendipity is not None:
        args.append(ctypes.byref(serendipity))
    return int(fn(*args))


def item_popularity(indptr, indices, row_begin, row_end, n, counts, device=-1, inputs_on_device=False):
    """rmb200_item_popularity: counts[j] = entries of item j in CSR rows [row_begin, row_end), counted on the GPU.  The arrays
    are numpy arrays (host) or device addresses (inputs_on_device).  Raises on failure."""
    rc = load().rmb200_item_popularity(_vp(indptr), _vp(indices), int(row_begin), int(row_end), int(n), int(device),
                                       int(bool(inputs_on_device)), _vp(counts))
    raise_for_status(rc)


def exposure_stats(counts, users=0):
    """rmb200_exposure_stats (host only, no GPU): the catalogue statistics of int64 item counts [n], as
    ``Exposure.catalogue()`` returns them; `users` is passed through (the counts do not tell it)."""
    counts = np.ascontiguousarray(counts, dtype=np.int64)
    e = make_exposure()
    raise_for_status(load().rmb200_exposure_stats(_vp(counts), ctypes.c_int32(int(counts.size)), ctypes.byref(e)))
    e.users = int(users)
    return e.catalogue()


def make_extra(device=-1, user_begin=0, user_end=0, inputs_on_device=False, strict_min_pos_test=False,
               topk_items=None, topk_scores=None, pos_rank=None, status=None, timing=None, scoring_path=0,
               metric_means=None, metric_counts=None, skip_row_copy=False, nan_bits=None, filter_stats=False, devices=None):
    ex = Extra()
    ex.struct_size = ctypes.sizeof(Extra)
    ex.device = int(device)
    ex.user_begin = int(user_begin)
    ex.user_end = int(user_end)
    ex.inputs_on_device = int(bool(inputs_on_device))
    ex.strict_min_pos_test = int(bool(strict_min_pos_test))
    ex.scoring_path = {"auto": 0, "fma": 1, "tensor": 2, "full": 3}.get(scoring_path, scoring_path)
    ex.topk_items = _vp(topk_items)
    ex.topk_scores = _vp(topk_scores)
    ex.pos_rank = _vp(pos_rank)
    ex.status = _vp(status)
    ex.metric_means = _vp(metric_means)
    ex.metric_counts = _vp(metric_counts)
    ex.skip_row_copy = int(bool(skip_row_copy))
    ex.has_nan_bits = int(nan_bits is not None)
    ex.nan_bits = int(nan_bits or 0)
    ex.filter_stats = int(bool(filter_stats))
    if devices is not None and len(devices) > 0:
        arr = (ctypes.c_int32 * len(devices))(*[int(d) for d in devices])
        ex._devices_keepalive = arr            # (the struct only holds the pointer)
        ex.devices = ctypes.cast(arr, ctypes.POINTER(ctypes.c_int32))
        ex.n_devices = len(devices)
    if timing is not None:
        ex.timing = ctypes.pointer(timing)
    return ex


class _SplitOwner:
    """Keeps one rmb200_split_t alive while numpy arrays look at its library-owned arrays; releases it afterwards."""

    def __init__(self, lib, out):
        self.lib, self.out = lib, out

    def __del__(self):
        try:
            self.lib.rmb200_split_free(ctypes.byref(self.out))
        except Exception:       # interpreter shutdown
            pass


def _view(owner, addr, count, dtype):
    """numpy array over `count` elements at host address `addr` without a copy; the array (through its base) keeps `owner` alive."""
    if not count:
        return np.empty(0, dtype=dtype)
    buf = (ctypes.c_uint8 * (int(count) * np.dtype(dtype).itemsize)).from_address(addr)
    buf._rmb200_owner = owner
    return np.frombuffer(buf, dtype=dtype)


def _view_csr(owner, c, dtype):
    if not c.indptr:
        return None
    return (_view(owner, c.indptr, c.rows + 1, np.int32), _view(owner, c.indices, c.nnz, np.int32), _view(owner, c.values, c.nnz, dtype),
            (int(c.rows), int(c.cols)))


def split(kind, indptr, indices, data, m, n, n_users_test=0, test_fraction=0.3, consider_cold_start=False,
          min_items_pool=2, min_pos_test=1, seed=1, device=-1):
    """rmb200_split_{selected,separate,joined}_users_f32/_f64.  kind: "all" | "separated" | "joined".
    Returns {"train", "test", "rem": (indptr, indices, data, shape) or None, "users_test": int32 array or None, "timing": dict};
    the arrays are views of the library's own result arrays (no copy), released with the last of them."""
    lib = load()
    dtype = np.dtype(data.dtype)
    assert dtype in (np.float32, np.float64) and indptr.dtype == np.int32 and indices.dtype == np.int32
    sfx = "f32" if dtype == np.float32 else "f64"
    # the reference's float entry points take the fraction as a float (src/recometrics_signatures.hpp:127, :174, :217)
    frac = ctypes.c_double(float(np.float32(test_fraction)) if dtype == np.float32 else float(test_fraction))
    out = Split()
    common = (_vp(indptr), _vp(indices), _vp(data), ctypes.c_int32(m), ctypes.c_int32(n))
    if kind == "all":
        rc = getattr(lib, "rmb200_split_selected_users_" + sfx)(*common, frac, ctypes.c_uint64(seed), ctypes.c_int32(device), ctypes.byref(out))
    else:
        fn = getattr(lib, ("rmb200_split_separate_users_" if kind == "separated" else "rmb200_split_joined_users_") + sfx)
        rc = fn(*common, ctypes.c_int32(n_users_test), frac, ctypes.c_int(int(consider_cold_start)), ctypes.c_int32(min_items_pool),
                ctypes.c_int32(min_pos_test), ctypes.c_uint64(seed), ctypes.c_int32(device), ctypes.byref(out))
    owner = _SplitOwner(lib, out)          # (releases the arrays when the last view goes away -- or right here if the call failed)
    raise_for_status(rc)
    return {"train": _view_csr(owner, out.train, dtype), "test": _view_csr(owner, out.test, dtype), "rem": _view_csr(owner, out.rem, dtype),
            "users_test": _view(owner, out.users_test, out.n_users_test, np.int32) if out.users_test else None,
            "timing": {k: getattr(out, k) for k in Split.TIMING}}


def split_plan(indptr, m, n, sample_users, n_users_test=0, test_fraction=0.3, consider_cold_start=False, min_items_pool=2,
               min_pos_test=1, seed=1):
    """rmb200_split_plan: the host half of a split (needs no GPU).  Returns (users_test or None, held bytes)."""
    lib = load()
    indptr = np.ascontiguousarray(indptr, dtype=np.int32)
    users = np.zeros(max(m, 1), dtype=np.int32)
    held = np.zeros(max(int(indptr[m]), 1), dtype=np.uint8)
    nu, ne = ctypes.c_int32(0), ctypes.c_int64(0)
    rc = lib.rmb200_split_plan(_vp(indptr), ctypes.c_int32(m), ctypes.c_int32(n), ctypes.c_int32(int(sample_users)),
                               ctypes.c_int32(n_users_test), ctypes.c_double(test_fraction), ctypes.c_int(int(consider_cold_start)),
                               ctypes.c_int32(min_items_pool), ctypes.c_int32(min_pos_test), ctypes.c_uint64(seed),
                               _vp(users), ctypes.byref(nu), _vp(held), ctypes.byref(ne))
    raise_for_status(rc)
    return (users[: nu.value].copy() if sample_users else None), held[: ne.value].copy()
