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
from warnings import warn

import numpy as np
from scipy.sparse import issparse

from . import _capi
from .frontend import EvalResult, _ResultRows, _canonical_csr, _popularity_array, item_popularity as _item_popularity

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
        novelty=False, avg_popularity=False, diversity=False, item_popularity=None):
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

    flags = dict(p=precision, tp=trunc_precision, r=recall, ap=average_precision, tap=trunc_average_precision,
                 ndcg=ndcg, hit=hit, rr=rr, roc=roc_auc, pr=pr_auc)
    flags = {q: bool(v) or bool(all_metrics) for q, v in flags.items()}
    if not (flags["p"] or flags["ap"] or flags["ndcg"] or flags["hit"] or flags["rr"] or flags["roc"]):
        raise ValueError("Must pass at least one metric to calculate.")
    cumulative = bool(cumulative)

    if issparse(X_test):
        X_test = DeviceCSR.from_scipy(X_test, device, dtype)
    if not isinstance(X_test, DeviceCSR):
        raise TypeError("'X_test' must be a sparse matrix or a DeviceCSR.")
    m, n = X_test.shape
    if X_train is None:
        X_train = DeviceCSR(torch.zeros(m + 1, dtype=torch.int32, device=dev), torch.zeros(0, dtype=torch.int32, device=dev), None, (m, n))
        consider_cold_start = True
    elif issparse(X_train):
        X_train = DeviceCSR.from_scipy(X_train, device, dtype, with_data=False)
    if not isinstance(X_train, DeviceCSR):
        raise TypeError("'X_train' must be a sparse matrix or a DeviceCSR.")
    if X_train.shape[1] != n:
        raise ValueError("'X_train' and 'X_test' should have the same number of columns.")
    if X_train.shape[0] < m:
        raise ValueError("'X_train' and 'X_test' should have the same number of rows.")
    if dA.shape[1] != dB.shape[1]:
        raise ValueError("'A' and 'B' must have the same number of columns.")
    if 0 in (dA.shape[0], dA.shape[1], m, n):
        raise ValueError("Input matrices cannot be empty.")
    if dA.shape[0] < m:
        raise ValueError("Number of users in 'A' and 'X_test' does not match.")
    if dB.shape[0] < n:
        raise ValueError("Number of items in 'B' and 'X_test' does not match.")
    if dA.shape[0] > m:
        warn("'A' has more users than 'X_test'.")
    if dB.shape[0] > n:
        warn("'B' has more items than 'X_test'.")
    seed, k, min_pos_test, min_items_pool = int(seed), int(k), int(min_pos_test), int(min_items_pool)
    if seed < 1 or k < 1 or min_pos_test < 1 or min_items_pool < 1:
        raise ValueError("'seed', 'k', 'min_pos_test' and 'min_items_pool' must be >= 1.")
    if k > n:
        raise ValueError("'k' should be smaller than the number of items.")
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
        nb = int(bias_keep.shape[0])
        if nb < n:
            raise ValueError("Number of items in 'item_biases' must match with 'X_test'.")
        bias_ptr = int(bias_keep.__cuda_array_interface__["data"][0])

    K = k
    bflags = dict(novelty=bool(novelty), avg_popularity=bool(avg_popularity), ild=bool(diversity))
    tdts = {np.float32: torch.float32, np.float64: torch.float64, np.int64: torch.int64}
    res = _ResultRows(lambda size, dt, fill: torch.empty(size, dtype=tdts[dt], device=dev) if fill is None
                      else torch.full((size,), fill, dtype=tdts[dt], device=dev),
                      dtype, m, K, cumulative, flags, bflags, user_range, bool(return_means) or bool(means_only))
    timing = _capi.Timing()
    status = torch.zeros(m, dtype=torch.int32, device=dev) if return_status else None
    topk_items = torch.full((m * K,), -1, dtype=torch.int32, device=dev) if return_topk else None
    topk_scores = torch.full((m * K,), float("nan"), dtype=tdt, device=dev) if return_topk else None
    ub, ue = (0, 0) if user_range is None else (int(user_range[0]), int(user_range[1]))
    if user_range is not None and ub == ue:
        ub, ue = 0, -1          # an EMPTY block; 0,0 would mean "all users" in the C-ABI
    ptr = lambda t: None if t is None else t.data_ptr()
    extra = _capi.make_extra(device=device, user_begin=ub, user_end=ue, inputs_on_device=True,
                             strict_min_pos_test=strict_min_pos_test, topk_items=ptr(topk_items), topk_scores=ptr(topk_scores),
                             status=ptr(status), timing=timing, scoring_path=scoring_path, metric_means=ptr(res.means),
                             metric_counts=ptr(res.counts), skip_row_copy=bool(means_only))
    item_counts = torch.zeros(n, dtype=torch.int64, device=dev) if return_exposure else None
    expo = _capi.make_exposure(ptr(item_counts)) if return_exposure else None
    bey = None
    if res.brows:
        pop = None
        if bflags["novelty"] or bflags["avg_popularity"]:
            if item_popularity is None:
                pop = _item_popularity(X_train, m=m)
            elif isinstance(item_popularity, torch.Tensor):
                if item_popularity.dim() != 1 or item_popularity.shape[0] != n:
                    raise ValueError("'item_popularity' must be a 1-d array with one count per item (%d)." % n)
                if item_popularity.dtype.is_floating_point or item_popularity.dtype.is_complex or item_popularity.dtype == torch.bool:
                    raise TypeError("'item_popularity' must hold integer counts.")
                pop = item_popularity.to(device=dev, dtype=torch.int64).contiguous()
                if n and bool(((pop < 0) | (pop > m)).any()):
                    raise ValueError("'item_popularity' counts must lie in [0, %d] (the number of users)." % m)
            else:
                pop = torch.from_numpy(_popularity_array(item_popularity, n, m)).to(dev)
        bey = _capi.make_beyond({name: t.data_ptr() for name, t in res.brows.items()}, ptr(pop), m, ptr(res.bmeans), ptr(res.bcounts))
    torch.cuda.synchronize(dev)            # the library runs on its own stream: the caller's pending writes must have landed
    rc = _capi.calc_metrics(dtype, dA.ptr, dA.ld, dB.ptr, dB.ld, m, n, dA.shape[1],
                            ptr(X_train.indptr), ptr(X_train.indices) if X_train.indices.numel() else None,
                            ptr(X_test.indptr), ptr(X_test.indices), ptr(tev), K, cumulative, bool(break_ties_with_noise),
                            {q: t.data_ptr() for q, t in res.outs.items()}, bool(consider_cold_start), min_items_pool,
                            min_pos_test, 1, seed, bias_ptr, extra, exposure=expo, beyond=bey)
    _capi.raise_for_status(rc)

    metrics, mean_d, count_d = res.unpack(means_only, lambda t: t.cpu().numpy())
    return EvalResult(metrics=metrics, timing=timing.as_dict(), status=status, means=mean_d, counts=count_d,
                      topk_items=None if topk_items is None else topk_items.view(m, K),
                      topk_scores=None if topk_scores is None else topk_scores.view(m, K),
                      exposure=item_counts, catalogue=None if expo is None else expo.catalogue())
