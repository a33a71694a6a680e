"""Host-side mirror of the reference's Python front-end for the evaluation path.

``calc_reco_metrics`` keeps the call surface of ``recometrics.calc_reco_metrics``
(/root/reference/recometrics/__init__.py:44-628): same argument names and defaults, same
validation errors, same float32/float64 rule (:469), same output packaging (:590-628) -- so a user
of the reference can switch the import and nothing else.  What changes is below the surface:

* the call goes to ``librecometrics_b200.so`` (sm_100a CUDA) through the C-ABI instead of the
  Cython/OpenMP extension;
* ``item_biases`` travel as their own vector and are added inside the scoring kernel, instead of
  being folded into copies of A and B (reference :548-551);
* ``nthreads`` is accepted and ignored (the parallelism is the GPU's);
* extras the reference cannot return (top-K ids, ranks of held-out items, per-call timing) are
  available through ``calc_reco_metrics_ex``.

There is no CPU fallback: without the built library or without a CUDA device the call raises.
"""
import ctypes
import re
from collections import namedtuple
from dataclasses import dataclass
from warnings import warn

import numpy as np
from scipy.sparse import csr_array, issparse

from . import _capi

__all__ = ["calc_reco_metrics", "calc_reco_metrics_ex", "EvalResult", "item_popularity"]

# reference dict keys, in the order the reference inserts them (__init__.py:591-610)
_KEYS = (("p", "P@K"), ("tp", "TP@K"), ("r", "R@K"), ("ap", "AP@K"), ("tap", "TAP@K"),
         ("ndcg", "NDCG@K"), ("hit", "Hit@K"), ("rr", "RR@K"), ("roc", "ROC_AUC"), ("pr", "PR_AUC"))


@dataclass
class EvalResult:
    metrics: dict            # reference-style dict: "P@K" -> array, ..., "K" -> k
    timing: dict             # rmb200_timing_t of the call
    status: np.ndarray = None
    topk_items: np.ndarray = None
    topk_scores: np.ndarray = None
    pos_rank: np.ndarray = None
    means: dict = None       # return_means: reference-style keys -> mean over the evaluated users (NaN rows left out)
    counts: dict = None      # ... -> how many users entered each mean
    exposure: np.ndarray = None   # return_exposure: int64 [n], how many evaluated users have item j in their ranked top-K list
    catalogue: dict = None   # ... and its statistics: "Coverage@K", "Gini@K", "Entropy@K", "users", "entries", "items_covered"


def _rows_c_layout(X):
    """Row-major view + leading dimension in elements (reference _as_row_major, :11-16)."""
    if X.flags["C_CONTIGUOUS"]:
        return X, X.shape[1]
    if X.strides[1] != X.dtype.itemsize or X.strides[0] % X.dtype.itemsize or X.strides[0] < X.shape[1] * X.dtype.itemsize:
        return np.ascontiguousarray(X), X.shape[1]
    return X, X.strides[0] // X.dtype.itemsize


def _canonical_csr(X):
    """CSR with sorted indices and int32 index arrays (reference :553-558)."""
    if not issparse(X):
        X = csr_array(X)
    elif X.format != "csr":
        X = X.tocsr()
    if not X.has_sorted_indices:
        X = X.copy()
        X.sort_indices()
    indptr = X.indptr if X.indptr.dtype == np.int32 else X.indptr.astype(np.int32)
    indices = X.indices if X.indices.dtype == np.int32 else X.indices.astype(np.int32)
    return X, np.ascontiguousarray(indptr), np.ascontiguousarray(indices)


def _popularity(item_popularity, n, m, device=None):
    """A caller's item popularity for Novelty@K / AvgPop@K: integer counts, one per item, each in [0, m]; int64 numpy --
    or, with a torch ``device`` (the device front-end, which also takes a torch tensor), an int64 tensor on it."""
    if device is not None:
        import torch
    p = item_popularity
    if device is not None and isinstance(p, torch.Tensor):
        integer = not (p.dtype.is_floating_point or p.dtype.is_complex or p.dtype == torch.bool)
    else:
        p = np.asarray(p)
        integer = p.dtype.kind in "iu"
    if p.ndim != 1 or p.shape[0] != n:
        raise ValueError("'item_popularity' must be a 1-d array with one count per item (%d)." % n)
    if not integer:
        raise TypeError("'item_popularity' must hold integer counts.")
    if isinstance(p, np.ndarray):
        p = np.ascontiguousarray(p, dtype=np.int64)
    if device is not None:
        p = torch.as_tensor(p).to(device=device, dtype=torch.int64).contiguous()
    if bool(((p < 0) | (p > m)).any()):
        raise ValueError("'item_popularity' counts must lie in [0, %d] (the number of users)." % m)
    return p


def _popularity_rows(rows, m, user_range):
    """Rows [begin, end) of an item_popularity count: user_range, else the first m rows (default: all)."""
    b, e = (0, rows if m is None else int(m)) if user_range is None else (int(user_range[0]), int(user_range[1]))
    if not (0 <= b <= e <= rows):
        raise ValueError("rows to count must lie within [0, %d] (the rows of 'X_train')." % rows)
    return b, e


def item_popularity(X_train, m=None, user_range=None, device=-1):
    """How many users have each item in their ``X_train`` row -- the column count of rows ``[0, m)`` (default: every row) or
    of rows ``user_range=(begin, end)`` -- counted on the GPU.  This is the popularity of ``novelty`` / ``avg_popularity``
    (with ``U = m``); the evaluation calls compute it when they are not given one, so a caller who evaluates several models
    against one split computes it once and passes it as ``item_popularity``.  ``X_train``: a scipy sparse matrix (returns a
    numpy int64 ``[n]``; ``device``: the CUDA ordinal, -1 = default) or a :class:`DeviceCSR` (returns a torch int64 ``[n]``
    on its device)."""
    from .device import DeviceCSR
    _check_csr_kind(X_train, "X_train")
    if isinstance(X_train, DeviceCSR):
        import torch
        rows, n = int(X_train.shape[0]), int(X_train.shape[1])
        b, e = _popularity_rows(rows, m, user_range)
        dev = X_train.indptr.device
        counts = torch.zeros(n, dtype=torch.int64, device=dev)
        torch.cuda.synchronize(dev)            # the library runs on its own stream: the caller's pending writes must have landed
        _capi.item_popularity(X_train.indptr.data_ptr(), X_train.indices.data_ptr() if X_train.indices.numel() else None,
                              b, e, n, counts.data_ptr(), device=dev.index, inputs_on_device=True)
        return counts
    X_train, indptr, indices = _canonical_csr(X_train)
    b, e = _popularity_rows(X_train.shape[0], m, user_range)
    counts = np.zeros(X_train.shape[1], dtype=np.int64)
    _capi.item_popularity(indptr, indices, b, e, X_train.shape[1], counts, device=device)
    return counts


# A family of per-user rows: its (name, result key) pairs in the order of its C struct and of its means / counts table, how
# many of them are W wide when cumulative, the requested rows by name, and the table (None: not requested)
_Family = namedtuple("_Family", "keys wide_slots rows means counts")


class _ResultRows:
    """The per-user rows of one call -- the requested metrics, Novelty / AvgPop / ILD and Unexpectedness / Serendipity rows,
    NaN outside ``user_range`` -- and their means / counts tables, allocated with ``alloc(size, dtype, fill)`` (numpy or
    torch; ``fill=None``: left uninitialised).  ``flags`` maps every row name to whether it is requested.  The families are
    the ten metrics (arguments of the C call, means in rmb200_extra_t), rmb200_beyond_t's and rmb200_serendipity_t's rows.  A
    table is ``[slot][W]``, ``W = K`` when ``cumulative`` else 1, over its family's rows, and exists when one of them does."""

    def __init__(self, alloc, dtype, m, K, cumulative, flags, user_range, return_means):
        self.m, self.K, self.W, self.cumulative = m, K, (K if cumulative else 1), cumulative
        fill = None if user_range is None else np.nan
        self.families = []
        for keys, wide_slots in ((_KEYS, 8), (_capi.BEYOND_KEYS, 3), (_capi.SERENDIPITY_KEYS, 2)):
            rows = {name: alloc(m * (self.W if i < wide_slots else 1), dtype, fill) for i, (name, _) in enumerate(keys) if flags[name]}
            on, cells = return_means and bool(rows), len(keys) * self.W
            self.families.append(_Family(keys, wide_slots, rows, alloc(cells, np.float64, np.nan) if on else None,
                                         alloc(cells, np.int64, 0) if on else None))

    def unpack(self, means_only, to_numpy=lambda x: x):
        """``metrics`` (W wide rows as ``(m, K)``, ``"K"`` last), ``means`` and ``counts`` of the call's EvalResult;
        ``to_numpy`` brings a means / counts table to the host."""
        metrics, W = {}, self.W
        mean_d, count_d = ({}, {}) if self.families[0].means is not None else (None, None)
        for f in self.families:
            means, counts = (None, None) if f.means is None else (to_numpy(f.means), to_numpy(f.counts))
            for i, (name, key) in enumerate(f.keys):
                if name not in f.rows:
                    continue
                wide = self.cumulative and i < f.wide_slots
                if not means_only:
                    metrics[key] = f.rows[name].reshape(self.m, self.K) if wide else f.rows[name]
                if means is not None:
                    mean_d[key] = means[i * W:(i + 1) * W].copy() if wide else float(means[i * W])
                    count_d[key] = counts[i * W:(i + 1) * W].copy() if wide else int(counts[i * W])
        metrics["K"] = self.K
        return metrics, mean_d, count_d


# Argument checks that both front-ends make, each front-end in its own order (the reference's for the host one).
def _metric_flags(all_metrics, *switches):
    """The ten metric switches, in METRIC_ORDER, as flags (``all_metrics`` sets them all)."""
    flags = {q: bool(v) or bool(all_metrics) for q, v in zip(_capi.METRIC_ORDER, switches, strict=True)}
    # the reference's guard ignores recall / trunc_* / pr_auc (quirk Q7, :499-500) -- kept as is
    if not (flags["p"] or flags["ap"] or flags["ndcg"] or flags["hit"] or flags["rr"] or flags["roc"]):
        raise ValueError("Must pass at least one metric to calculate.")
    return flags


def _check_factor_shapes(a_shape, b_shape, m, n):
    """A [users, p] and B [items, p] against X_test [m, n]; the rows past m / n are not read."""
    if a_shape[1] != b_shape[1]:
        raise ValueError("'A' and 'B' must have the same number of columns.")
    if 0 in (a_shape[0], a_shape[1], m, n):
        raise ValueError("Input matrices cannot be empty.")
    if a_shape[0] < m:
        raise ValueError("Number of users in 'A' and 'X_test' does not match.")
    if b_shape[0] < n:
        raise ValueError("Number of items in 'B' and 'X_test' does not match.")
    if a_shape[0] > m:
        warn("'A' has more users than 'X_test'.")
    if b_shape[0] > n:
        warn("'B' has more items than 'X_test'.")


def _check_csr_kind(X, name):
    from .device import DeviceCSR
    if not (issparse(X) or isinstance(X, DeviceCSR)):
        raise TypeError("'%s' must be a sparse matrix or a DeviceCSR." % name)


def _check_train_shape(train_shape, m, n):
    if train_shape[1] != n:
        raise ValueError("'X_train' and 'X_test' should have the same number of columns.")
    if train_shape[0] < m:
        raise ValueError("'X_train' and 'X_test' should have the same number of rows.")


def _counts(seed, k, min_pos_test, min_items_pool, n):
    """The call's integer arguments as ints: each at least 1, ``k`` at most the ``n`` items."""
    seed, k, min_pos_test, min_items_pool = int(seed), int(k), int(min_pos_test), int(min_items_pool)
    if seed < 1 or k < 1 or min_pos_test < 1 or min_items_pool < 1:
        raise ValueError("'seed', 'k', 'min_pos_test' and 'min_items_pool' must be >= 1.")
    if k > n:
        raise ValueError("'k' should be smaller than the number of items.")
    return seed, k, min_pos_test, min_items_pool


def _check_bias_items(items, n):
    if items < n:
        raise ValueError("Number of items in 'item_biases' must match with 'X_test'.")


def _validate_and_prepare(X_train, X_test, A, B, k, item_biases, min_pos_test, min_items_pool, consider_cold_start,
                          nthreads, seed, *metric_switches):
    """The host front-end's checks and conversions (``metric_switches``: as :func:`_metric_flags` takes them)."""
    if (A is None) != (B is None):
        raise ValueError("'A' and 'B' must either be passed together or passed as 'None' together.")
    if item_biases is not None and hasattr(item_biases, "to_numpy"):
        item_biases = item_biases.to_numpy()
    if A is None:
        # non-personalised model: score = item bias (reference :429-436)
        if item_biases is None:
            raise ValueError("Must pass item biases if not passing factors.")
        A = np.ones((X_test.shape[0], 1), dtype=np.float64)
        B = np.ascontiguousarray(item_biases, dtype=np.float64).reshape((-1, 1))
        item_biases = None

    if not isinstance(A, np.ndarray) or not isinstance(B, np.ndarray):
        raise TypeError("'A' and 'B' must be numpy arrays.")
    if not issparse(X_test):
        raise TypeError("'X_test' must be a sparse matrix.")
    imax = np.iinfo(np.int32).max
    if X_test.shape[0] >= imax:
        raise ValueError("Number of test user is larger than maximum supported.")
    if X_test.shape[1] >= imax:
        raise ValueError("Number of items is larger than maximum supported.")
    if not X_test.data.shape[0]:
        raise ValueError("'X_test' is empty.")
    if A.ndim != 2:
        raise ValueError("'A' must be a 2-dimensional array.")
    if B.ndim != 2:
        raise ValueError("'B' must be a 2-dimensional array.")
    _check_factor_shapes(A.shape, B.shape, X_test.shape[0], X_test.shape[1])
    A, B = A[:X_test.shape[0], :], B[:X_test.shape[1], :]

    # float32 only if both factor matrices are float32 (reference :469)
    dtype = np.float32 if (A.dtype == np.float32 and B.dtype == np.float32) else np.float64

    if X_train is None:
        X_train = csr_array(X_test.shape, dtype=dtype)
        consider_cold_start = True
    if not issparse(X_train):
        raise TypeError("'X_train' must be a sparse matrix.")
    _check_train_shape(X_train.shape, X_test.shape[0], X_test.shape[1])
    if X_train.shape[0] > X_test.shape[0]:
        warn("'X_train' mas more rows than 'X_test'.")

    flags = _metric_flags(*metric_switches)

    if isinstance(seed, np.random.RandomState):
        seed = int(seed.randint(imax))
    elif isinstance(seed, np.random.Generator):
        seed = int(seed.integers(imax))
    nthreads = 1 if nthreads is None else int(nthreads)
    seed, k, min_pos_test, min_items_pool = _counts(seed, k, min_pos_test, min_items_pool, X_test.shape[1])

    if item_biases is not None:
        if not isinstance(item_biases, np.ndarray):
            raise TypeError("'item_biases' must be a numpy array.")
        if item_biases.ndim > 2:
            raise ValueError("'item_biases' should be a 1-d array.")
        item_biases = item_biases.reshape(-1)
        if not item_biases.shape[0]:
            raise ValueError("'item_biases' is empty.")
        _check_bias_items(item_biases.shape[0], X_test.shape[1])
        if item_biases.shape[0] > X_test.shape[1]:
            warn("'item_biases' has more items than 'X_test'.")
            item_biases = item_biases[:X_test.shape[1]]
        item_biases = np.ascontiguousarray(item_biases, dtype=dtype)

    X_train, trp, tri = _canonical_csr(X_train)
    X_test, tep, tei = _canonical_csr(X_test)
    tev = np.ascontiguousarray(X_test.data, dtype=dtype)
    A = A if A.dtype == dtype else A.astype(dtype)
    B = B if B.dtype == dtype else B.astype(dtype)
    A, lda = _rows_c_layout(A)
    B, ldb = _rows_c_layout(B)
    return dict(A=A, lda=lda, B=B, ldb=ldb, dtype=dtype, m=X_test.shape[0], n=X_test.shape[1], p=A.shape[1],
                trp=trp, tri=tri, tep=tep, tei=tei, tev=tev, k=k, item_biases=item_biases,
                min_pos_test=min_pos_test, min_items_pool=min_items_pool,
                consider_cold_start=bool(consider_cold_start), nthreads=nthreads, seed=seed, flags=flags)


def _evaluate(alloc, addr, prep, popularity, cumulative, break_ties_with_noise, user_range, return_topk, return_status,
              return_means, means_only, return_exposure, list_rows, return_ranks=False, to_numpy=lambda x: x,
              sync=lambda: None, **extra):
    """The evaluation call both front-ends end in, on the inputs ``prep`` they validated (``_validate_and_prepare``'s keys:
    host arrays or device addresses, as ``_capi.calc_metrics`` takes them).  The result rows and the asked-for extras are
    allocated with ``alloc(size, dtype, fill)`` (see :class:`_ResultRows`) and handed to the library as ``addr(array)``;
    ``list_rows`` switches the beyond-accuracy and history rows by name; ``popularity()`` gives the item popularity when
    Novelty / AvgPop is asked for, ``sync()`` runs right before the call, ``to_numpy`` brings a means / counts table to the
    host and ``extra`` goes to ``_capi.make_extra``."""
    dtype, m, n, K, cumulative = prep["dtype"], prep["m"], prep["n"], prep["k"], bool(cumulative)
    ptr = lambda x: None if x is None else addr(x)
    flags = {**prep["flags"], **{name: bool(on) for name, on in list_rows.items()}}
    res = _ResultRows(alloc, dtype, m, K, cumulative, flags, user_range, bool(return_means) or bool(means_only))
    metric, beyond, history = res.families
    timing = _capi.Timing()
    status = alloc(m, np.int32, 0) if return_status else None
    topk_items = alloc(m * K, np.int32, -1) if return_topk else None
    topk_scores = alloc(m * K, dtype, np.nan) if return_topk else None
    pos_rank = alloc(max(int(prep["tep"][-1]), 1), np.int64, 0) if return_ranks else None
    ub, ue = (0, 0) if user_range is None else (int(user_range[0]), int(user_range[1]))
    if user_range is not None and ub == ue:
        ub, ue = 0, -1          # an EMPTY block (a rank with no users); 0,0 would mean "all users" in the C-ABI
    ex = _capi.make_extra(user_begin=ub, user_end=ue, topk_items=ptr(topk_items), topk_scores=ptr(topk_scores),
                          pos_rank=ptr(pos_rank), status=ptr(status), timing=timing, metric_means=ptr(metric.means),
                          metric_counts=ptr(metric.counts), skip_row_copy=bool(means_only), **extra)
    item_counts = alloc(n, np.int64, 0) if return_exposure else None
    expo = _capi.make_exposure(ptr(item_counts)) if return_exposure else None
    addrs = [{name: addr(r) for name, r in f.rows.items()} for f in res.families]
    pop = popularity() if "novelty" in beyond.rows or "avg_popularity" in beyond.rows else None
    bey = _capi.make_beyond(addrs[1], ptr(pop), m, ptr(beyond.means), ptr(beyond.counts)) if beyond.rows else None
    ser = _capi.make_serendipity(addrs[2], ptr(history.means), ptr(history.counts)) if history.rows else None
    sync()
    rc = _capi.calc_metrics(dtype, prep["A"], prep["lda"], prep["B"], prep["ldb"], m, n, prep["p"],
                            prep["trp"], prep["tri"], prep["tep"], prep["tei"], prep["tev"], K, cumulative,
                            bool(break_ties_with_noise), addrs[0], prep["consider_cold_start"],
                            prep["min_items_pool"], prep["min_pos_test"], prep["nthreads"], prep["seed"], prep["item_biases"],
                            ex, exposure=expo, beyond=bey, serendipity=ser)
    _capi.raise_for_status(rc)

    metrics, mean_d, count_d = res.unpack(means_only, to_numpy)
    return EvalResult(metrics=metrics, timing=timing.as_dict(), status=status, means=mean_d, counts=count_d,
                      topk_items=None if topk_items is None else topk_items.reshape(m, K),
                      topk_scores=None if topk_scores is None else topk_scores.reshape(m, K),
                      pos_rank=None if pos_rank is None else pos_rank[: int(prep["tep"][-1])],
                      exposure=item_counts, catalogue=None if expo is None else expo.catalogue())


def calc_reco_metrics_ex(
        X_train, X_test, A, B, k=5, item_biases=None,
        precision=True, trunc_precision=False, recall=False, average_precision=True,
        trunc_average_precision=False, ndcg=True, hit=False, rr=False, roc_auc=False, pr_auc=False,
        all_metrics=False, break_ties_with_noise=True, min_pos_test=1, min_items_pool=2,
        consider_cold_start=True, cumulative=False, nthreads=-1, seed=1,
        device=-1, user_range=None, strict_min_pos_test=False,
        return_topk=False, return_ranks=False, return_status=False, scoring_path="auto",
        return_means=False, means_only=False, filter_stats=False, nan_bits=None, devices=None, return_exposure=False,
        novelty=False, avg_popularity=False, diversity=False, item_popularity=None, unexpectedness=False, serendipity=False):
    """Same evaluation as :func:`calc_reco_metrics`, returning an :class:`EvalResult` with the
    reference-style dict plus timing and the optional extras (top-K ids/scores, held-out ranks,
    per-user status).  ``user_range=(begin, end)`` evaluates only those rows (the sharding unit);
    rows outside it are left as NaN in the returned arrays.  ``scoring_path``: "auto" | "fma" (every score on
    the FP32/FP64 FMA pipe) | "tensor" (fp16 tensor-core candidate filter + exact FMA re-scoring of the
    survivors: identical top-K and scores, top-K metrics only).  ``return_means``: also reduce every requested
    metric to its mean over the evaluated users on the device (``numpy.nanmean`` of the per-user output; ``(k,)`` vectors
    when ``cumulative``) -- ``result.means`` / ``result.counts``; with ``means_only`` the per-user rows are not copied
    back at all (``result.metrics`` then only holds ``"K"``).  ``devices``: list of CUDA ordinals to spread the users of
    this one call over (one host thread per GPU inside the native call).  ``nan_bits``: bit pattern written wherever a
    metric is undefined (R's ``NA_REAL``) instead of a plain NaN.  ``filter_stats``: fill ``timing["filter_err_ratio_max"]``.
    ``return_exposure``: count, on the device, how many evaluated users have each item in their ranked top-K list
    (``result.exposure``, int64 ``[n]``: ``numpy.bincount`` of the defined ``topk_items``) and derive the catalogue's coverage,
    Gini index and entropy from the counts (``result.catalogue``); the lists themselves stay on the device.
    ``novelty`` / ``avg_popularity`` / ``diversity``: per-user Novelty@K, AvgPop@K and ILD@K (intra-list diversity: the mean
    pairwise cosine distance of the listed items' rows of ``B``) of the ranked lists, computed on the device -- rows
    ``result.metrics["Novelty@K"]``, ``["AvgPop@K"]``, ``["ILD@K"]`` (``(m,)``, ``(m, k)`` when ``cumulative``) and, with
    ``return_means``, their means and counts under the same keys; NaN for users without a list.  ``item_popularity``: int64
    ``[n]`` counts of how many of the m users have each item in ``X_train`` (see :func:`item_popularity`, which computes it
    when it is not given).  ``unexpectedness`` / ``serendipity``: per-user Unexpectedness@K and Serendipity@K of the ranked
    lists against each user's ``X_train`` row, computed on the device -- with ``sim_r`` the mean cosine similarity of the
    r-th listed item's row of ``B`` to the rows of the user's training items, Unexpectedness@K is the mean of ``1 - sim_r``
    over the list and Serendipity@K the mean of ``rel_r * (1 - sim_r)``, ``rel_r = 1`` when the item is in the user's
    ``X_test`` row (Microsoft Recommenders' ``user_serendipity`` with held-out relevance); rows
    ``result.metrics["Unexpectedness@K"]`` and ``["Serendipity@K"]``, shaped and reduced like the rows above; NaN for users
    without a list or without a training item (cold-start users, and every user when ``X_train`` is None).  ``all_metrics``
    does not turn these on."""
    prep = _validate_and_prepare(X_train, X_test, A, B, k, item_biases, min_pos_test, min_items_pool, consider_cold_start,
                                 nthreads, seed, all_metrics, precision, trunc_precision, recall, average_precision,
                                 trunc_average_precision, ndcg, hit, rr, roc_auc, pr_auc)

    def popularity():
        if item_popularity is not None:
            return _popularity(item_popularity, prep["n"], prep["m"])
        pop = np.zeros(prep["n"], dtype=np.int64)
        _capi.item_popularity(prep["trp"], prep["tri"], 0, prep["m"], prep["n"], pop,
                              device=device if device >= 0 else (devices[0] if devices else -1))
        return pop
    return _evaluate(lambda size, dt, fill: np.empty(size, dt) if fill is None else np.full(size, fill, dt), lambda x: x,
                     prep, popularity, cumulative, break_ties_with_noise, user_range, return_topk, return_status,
                     return_means, means_only, return_exposure, dict(novelty=novelty, avg_popularity=avg_popularity,
                     ild=diversity, unexpectedness=unexpectedness, serendipity=serendipity), return_ranks=return_ranks,
                     device=device, strict_min_pos_test=strict_min_pos_test, scoring_path=scoring_path,
                     filter_stats=filter_stats, nan_bits=nan_bits, devices=devices)


def calc_reco_metrics(
        X_train, X_test, A, B, k=5, item_biases=None, as_df=True,
        precision=True, trunc_precision=False, recall=False, average_precision=True,
        trunc_average_precision=False, ndcg=True, hit=False, rr=False, roc_auc=False, pr_auc=False,
        all_metrics=False, rename_k=True, break_ties_with_noise=True, min_pos_test=1, min_items_pool=2,
        consider_cold_start=True, cumulative=False, nthreads=-1, seed=1):
    """Drop-in for ``recometrics.calc_reco_metrics`` (reference __init__.py:44-628), computed on a B200.

    Returns what the reference returns: a ``pandas.DataFrame`` (``as_df=True``; columns ``P@5`` ... or
    ``P@1..P@k`` blocks when ``cumulative``) or a dict keyed ``"P@K"``, ..., ``"ROC_AUC"``, ``"PR_AUC"``,
    ``"K"`` (``as_df=False``).  Rows of users that cannot be evaluated are NaN (reference rules,
    src/recometrics.hpp:193-209)."""
    res = calc_reco_metrics_ex(
        X_train, X_test, A, B, k=k, item_biases=item_biases,
        precision=precision, trunc_precision=trunc_precision, recall=recall, average_precision=average_precision,
        trunc_average_precision=trunc_average_precision, ndcg=ndcg, hit=hit, rr=rr, roc_auc=roc_auc, pr_auc=pr_auc,
        all_metrics=all_metrics, break_ties_with_noise=break_ties_with_noise, min_pos_test=min_pos_test,
        min_items_pool=min_items_pool, consider_cold_start=consider_cold_start, cumulative=cumulative,
        nthreads=nthreads, seed=seed)
    out = res.metrics
    if not as_df:
        return out
    import pandas as pd
    K = out.pop("K")
    if not cumulative:
        df = pd.DataFrame(out)
        if rename_k:
            df.columns = [re.sub(r"@K$", "@" + str(K), c) for c in df.columns]
        return df
    blocks = []
    for name, v in out.items():
        if name.endswith("@K"):
            cols = [name[:-1] + str(i + 1) for i in range(v.shape[1])]
            blocks.append(pd.DataFrame(v, columns=cols))
        else:
            blocks.append(pd.DataFrame({name: v}))
    return pd.concat(blocks, axis=1)
