"""Device-resident front-end: the same evaluation with the factors (and optionally the CSR matrices) already
in the GPU's memory -- SURVEY 8(f)-1: "device-array inputs (``__cuda_array_interface__`` / torch)".

``calc_reco_metrics`` (frontend.py) mirrors the reference's call: numpy in, numpy out, every byte crosses
PCIe on every call (1.5 GB for the 1M x 1M configuration).  A model that was trained on the GPU has its
factors there already; ``calc_reco_metrics_device`` takes them where they are:

* ``A``, ``B``, ``item_biases``: anything exposing ``__cuda_array_interface__`` (torch CUDA tensors, CuPy arrays),
  float32 or float64, row-major (a row stride larger than the row is fine: reference ``_as_row_major``,
  /root/reference/recometrics/__init__.py:11-16);
* ``X_train``, ``X_test``: scipy sparse matrices (canonicalised like the reference does, :553-558, and uploaded:
  a few hundred MB at most) or :class:`DeviceCSR` objects that stay resident between calls;
* the per-user metric rows come back as torch CUDA tensors (``result.metrics``); nothing is copied to the host
  unless the caller does it.

The call goes through the same C-ABI entry point (``rmb200_calc_metrics_ex_*`` with ``inputs_on_device=1``); torch is
used for device allocations only.  Argument meaning, defaults, validation messages and NaN rules are those of
``calc_reco_metrics_ex``.
"""
from dataclasses import dataclass

import numpy as np
from scipy.sparse import issparse

from .frontend import (_canonical_csr, _check_bias_items, _check_csr_kind, _check_factor_shapes, _check_train_shape,
                       _counts, _evaluate, _metric_flags, _popularity, item_popularity as _item_popularity)

__all__ = ["DeviceCSR", "calc_reco_metrics_device"]


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("recometrics_b200 needs a CUDA device (no CPU fallback)")
    return torch


class _Dev2D:
    """Pointer, shape, dtype and leading dimension (in elements) of a device matrix or vector."""

    def __init__(self, x, name, ndim):
        cai = getattr(x, "__cuda_array_interface__", None)
        if cai is None:
            raise TypeError("'%s' must expose __cuda_array_interface__ (a torch CUDA tensor, a CuPy array, ...)." % name)
        self.obj = x                      # keeps the memory alive for the duration of the call
        self.shape = tuple(int(v) for v in cai["shape"])
        self.dtype = np.dtype(cai["typestr"])
        self.ptr = int(cai["data"][0])
        if self.dtype not in (np.dtype(np.float32), np.dtype(np.float64)):
            raise TypeError("'%s' must be float32 or float64." % name)
        if len(self.shape) != ndim:
            raise ValueError("'%s' must be a %d-dimensional array." % (name, ndim))
        strides = cai.get("strides")
        item = self.dtype.itemsize
        if ndim == 2:
            if strides is None:
                self.ld = self.shape[1]
            else:
                s0, s1 = int(strides[0]), int(strides[1])
                if (s1 != item and self.shape[1] > 1) or s0 % item or s0 < self.shape[1] * item:
                    raise ValueError("'%s' must be row-major (unit column stride); make it contiguous first." % name)
                self.ld = s0 // item
        else:
            if strides is not None and self.shape[0] > 1 and int(strides[0]) != item:
                raise ValueError("'%s' must be contiguous." % name)
            self.ld = 1
        dev = getattr(getattr(x, "device", None), "index", None)
        if dev is None:
            dev = getattr(getattr(x, "device", None), "id", None)      # CuPy
        self.device = None if dev is None else int(dev)


@dataclass
class DeviceCSR:
    """A CSR matrix resident on one CUDA device: int32 ``indptr`` [rows+1] and sorted ``indices`` [nnz] (torch tensors),
    ``data`` [nnz] (float32/float64 torch tensor; may be None for X_train, whose values are never read)."""
    indptr: object
    indices: object
    data: object
    shape: tuple

    @classmethod
    def from_scipy(cls, X, device=0, dtype=None, with_data=True):
        """Canonicalise like the reference front-end (sorted indices, int32 index arrays) and upload."""
        torch = _torch()
        X, indptr, indices = _canonical_csr(X)
        dev = torch.device("cuda", int(device))
        data = None
        if with_data:
            data = torch.from_numpy(np.ascontiguousarray(X.data, dtype=dtype or X.data.dtype)).to(dev)
        return cls(torch.from_numpy(indptr).to(dev), torch.from_numpy(indices).to(dev), data, tuple(int(v) for v in X.shape))


def calc_reco_metrics_device(
        X_train, X_test, A, B, k=5, item_biases=None,
        precision=True, trunc_precision=False, recall=False, average_precision=True,
        trunc_average_precision=False, ndcg=True, hit=False, rr=False, roc_auc=False, pr_auc=False,
        all_metrics=False, break_ties_with_noise=True, min_pos_test=1, min_items_pool=2,
        consider_cold_start=True, cumulative=False, seed=1,
        user_range=None, strict_min_pos_test=False, return_topk=False, return_status=False, scoring_path="auto",
        return_means=False, means_only=False, return_exposure=False,
        novelty=False, avg_popularity=False, diversity=False, item_popularity=None, unexpectedness=False, serendipity=False):
    """``calc_reco_metrics_ex`` for inputs that live on the GPU (see the module docstring).  Returns an
    :class:`EvalResult` whose ``metrics`` / ``status`` / ``topk_*`` / ``exposure`` entries are torch CUDA tensors on the
    device of ``A`` (``means`` / ``counts`` / ``catalogue`` are small and come back as Python numbers / numpy vectors).
    ``item_popularity`` (for ``novelty`` / ``avg_popularity``) may be a numpy array or a torch tensor; without it the counts
    of ``X_train``'s first m rows are taken on the device."""
    torch = _torch()
    if A is None or B is None:
        raise ValueError("'A' and 'B' must be passed (device-resident factor matrices).")
    dA, dB = _Dev2D(A, "A", 2), _Dev2D(B, "B", 2)
    if dA.dtype != dB.dtype:
        raise TypeError("'A' and 'B' must have the same dtype on the device (the host front-end would promote to float64).")
    dtype = dA.dtype.type
    tdt = torch.float32 if dtype == np.float32 else torch.float64
    device = dA.device if dA.device is not None else torch.cuda.current_device()
    if dB.device is not None and dB.device != device:
        raise ValueError("'A' and 'B' must be on the same device.")
    dev = torch.device("cuda", device)

    flags = _metric_flags(all_metrics, precision, trunc_precision, recall, average_precision, trunc_average_precision, ndcg,
                          hit, rr, roc_auc, pr_auc)

    _check_csr_kind(X_test, "X_test")
    if issparse(X_test):
        X_test = DeviceCSR.from_scipy(X_test, device, dtype)
    m, n = X_test.shape
    if X_train is None:
        X_train = DeviceCSR(torch.zeros(m + 1, dtype=torch.int32, device=dev), torch.zeros(0, dtype=torch.int32, device=dev), None, (m, n))
        consider_cold_start = True
    _check_csr_kind(X_train, "X_train")
    if issparse(X_train):
        X_train = DeviceCSR.from_scipy(X_train, device, dtype, with_data=False)
    _check_train_shape(X_train.shape, m, n)
    _check_factor_shapes(dA.shape, dB.shape, m, n)
    seed, k, min_pos_test, min_items_pool = _counts(seed, k, min_pos_test, min_items_pool, n)
    for name, X in (("X_train", X_train), ("X_test", X_test)):
        for part in ("indptr", "indices"):
            t = getattr(X, part)
            if t.dtype != torch.int32 or not t.is_cuda or t.device.index != device or not t.is_contiguous():
                raise TypeError("%s.%s must be a contiguous int32 tensor on cuda:%d." % (name, part, device))
    tev = X_test.data
    if tev is not None and (tev.dtype != tdt or not tev.is_contiguous()):
        tev = tev.to(tdt).contiguous()
    if tev is None and flags["ndcg"]:
        raise ValueError("'X_test' needs its values for NDCG.")

    bias_ptr, bias_keep = None, None
    if item_biases is not None:
        if isinstance(item_biases, np.ndarray):
            bias_keep = torch.from_numpy(np.ascontiguousarray(item_biases.reshape(-1), dtype=dtype)).to(dev)
        else:
            db = _Dev2D(item_biases, "item_biases", 1)
            if db.dtype != dA.dtype:
                raise TypeError("'item_biases' must have the dtype of the factors.")
            bias_keep = item_biases
        _check_bias_items(int(bias_keep.shape[0]), n)
        bias_ptr = int(bias_keep.__cuda_array_interface__["data"][0])

    # the addresses stay valid while X_train, X_test, tev and bias_keep live: until this function returns
    prep = dict(A=dA.ptr, lda=dA.ld, B=dB.ptr, ldb=dB.ld, dtype=dtype, m=m, n=n, p=dA.shape[1],
                trp=X_train.indptr.data_ptr(), tri=X_train.indices.data_ptr() if X_train.indices.numel() else None,
                tep=X_test.indptr.data_ptr(), tei=X_test.indices.data_ptr(), tev=None if tev is None else tev.data_ptr(),
                k=k, item_biases=bias_ptr, min_pos_test=min_pos_test, min_items_pool=min_items_pool,
                consider_cold_start=bool(consider_cold_start), nthreads=1, seed=seed, flags=flags)
    tdts = {np.float32: torch.float32, np.float64: torch.float64, np.int32: torch.int32, np.int64: torch.int64}

    def popularity():
        return _item_popularity(X_train, m=m) if item_popularity is None else _popularity(item_popularity, n, m, dev)
    return _evaluate(lambda size, dt, fill: torch.empty(size, dtype=tdts[dt], device=dev) if fill is None
                     else torch.full((size,), fill, dtype=tdts[dt], device=dev), lambda t: t.data_ptr(), prep, popularity,
                     cumulative, break_ties_with_noise, user_range, return_topk, return_status, return_means, means_only,
                     return_exposure, dict(novelty=novelty, avg_popularity=avg_popularity, ild=diversity,
                     unexpectedness=unexpectedness, serendipity=serendipity), to_numpy=lambda t: t.cpu().numpy(),
                     # the library runs on its own stream: the caller's pending writes and the fills above must have landed
                     sync=lambda: torch.cuda.synchronize(dev),
                     device=device, inputs_on_device=True, strict_min_pos_test=strict_min_pos_test, scoring_path=scoring_path)
