"""GPU: per-user Novelty@K, AvgPop@K and ILD@K of the ranked top-K lists (novelty / avg_popularity / diversity).  The reference
is numpy in float64 on the same call's own topk_items (return_topk=True), with ILD from an explicit L x L Gram matrix of the
normalised rows of B, not from the running-sum formula the kernel uses.  Checked on every scoring path and every way a list
can be decided, cumulative calls, bit-identity over shards, front-ends and devices, the popularity counter, closed-form
cases, the means, and that the accuracy outputs do not change."""
import struct

import numpy as np
import pytest
from scipy.sparse import csr_array

from golden_io import load_case
from tools import synth

pytestmark = pytest.mark.gpu

TOPK4 = dict(precision=True, recall=True, average_precision=True, ndcg=True)
BEYOND = dict(novelty=True, avg_popularity=True, diversity=True)
KEYS = ("Novelty@K", "AvgPop@K", "ILD@K")


def _reference(ids, B, pop, U, cumulative):
    """float64 rows from the listed ids (-1 = no list): Novelty, AvgPop, ILD; (m,) or (m, K)."""
    m, K = ids.shape
    Bd = np.asarray(B, dtype=np.float64)
    nrm = np.linalg.norm(Bd, axis=1, keepdims=True)
    Un = np.divide(Bd, nrm, out=np.zeros_like(Bd), where=nrm > 0)
    si = -np.log2((np.asarray(pop, dtype=np.float64) + 1.0) / (U + 1.0))
    out = {key: np.full((m, K), np.nan) for key in KEYS}
    for u in range(m):
        L = int((ids[u] >= 0).sum())
        if L == 0:
            continue
        it = ids[u, :L]
        i = np.arange(1, L + 1, dtype=np.float64)
        out["Novelty@K"][u, :L] = np.cumsum(si[it]) / i
        out["AvgPop@K"][u, :L] = np.cumsum(np.asarray(pop, dtype=np.float64)[it]) / i
        G = Un[it] @ Un[it].T
        P = np.cumsum(np.tril(G, -1).sum(axis=1))        # sum of the pairs among the first i items
        with np.errstate(invalid="ignore", divide="ignore"):
            out["ILD@K"][u, :L] = 1.0 - 2.0 * P / (i * (i - 1))
        out["ILD@K"][u, 0] = np.nan
    if not cumulative:
        out = {key: v[:, -1] for key, v in out.items()}
    return out


def _assert_rows(res, B, pop, U, cumulative=False, rows=slice(None)):
    ids = np.asarray(res.topk_items)[rows]
    ref = _reference(ids, B, pop, U, cumulative)
    f64 = res.metrics[KEYS[0]].dtype == np.float64
    undefined = ids[:, 0] < 0
    for key in KEYS:
        got = np.asarray(res.metrics[key])[rows].astype(np.float64)
        want = ref[key]
        nan_want = np.isnan(want)
        if not cumulative:
            assert np.array_equal(np.isnan(got), undefined | (key == "ILD@K" and ids.shape[1] == 1)), key
        assert np.array_equal(np.isnan(got), nan_want), key
        if f64:
            np.testing.assert_allclose(got[~nan_want], want[~nan_want], rtol=1e-12, atol=1e-12, err_msg=key)
        elif key == "ILD@K":
            np.testing.assert_allclose(got[~nan_want], want[~nan_want], rtol=0, atol=1e-6, err_msg=key)
        else:
            np.testing.assert_allclose(got[~nan_want], want[~nan_want], rtol=1e-6, atol=0, err_msg=key)
    return int((~undefined).sum())


def _pop(X_train, m):
    X = csr_array(X_train)[:m]
    return np.bincount(X.indices, minlength=X.shape[1]).astype(np.int64)


def _run(rb, d, k, **kw):
    kw = {**TOPK4, "break_ties_with_noise": False, **BEYOND, **kw}
    return rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], k=k, item_biases=d.get("item_biases"),
                                   return_topk=True, return_status=True, **kw)


def _same(a, b):
    """Equal bytes (NaN payloads included)."""
    a, b = np.ascontiguousarray(np.atleast_1d(np.asarray(a))), np.ascontiguousarray(np.atleast_1d(np.asarray(b)))
    return a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


# (k, scoring_path, noise, extra flags, expected timing["scoring_path"]): tensor filter (with and without the noise); FMA tiles;
# K = 300, which only the FMA tiles take; full order for K = 400 and for K = 300 with the noise; ROC/PR-AUC rank counting
PATHS = [(10, "auto", False, {}, 2), (10, "auto", True, {}, 2), (10, "fma", False, {}, 1), (300, "auto", False, {}, 1),
         (400, "auto", False, {}, 3), (300, "auto", True, {}, 3), (10, "auto", False, dict(roc_auc=True, pr_auc=True), 1)]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("k,path,noise,flags,expect", PATHS)
def test_rows_equal_the_reference(rb, dtype, k, path, noise, flags, expect):
    d = synth.make(2, m=1200, n=3000, p=16)
    d["A"], d["B"], d["item_biases"] = d["A"].astype(dtype), d["B"].astype(dtype), d["item_biases"].astype(dtype)
    res = _run(rb, d, k, scoring_path=path, break_ties_with_noise=noise, **flags)
    assert res.timing["scoring_path"] == expect
    assert res.metrics["ILD@K"].dtype == dtype
    assert _assert_rows(res, d["B"], _pop(d["X_train"], 1200), 1200) > 400


def test_rank_counting_with_the_noise_hand_back(rb):
    c = load_case("g_noise_ties_f64")
    res = rb.calc_reco_metrics_ex(c["X_train"], c["X_test"], c["A"], c["B"], k=c["k"], all_metrics=True, seed=3,
                                  break_ties_with_noise=True, return_topk=True, **BEYOND)
    assert res.timing["noise_handback_users"] > 0
    m = c["X_test"].shape[0]
    _assert_rows(res, c["B"], _pop(c["X_train"], m), m)


def test_ineligible_and_nan_users(rb):
    d = synth.make(1, m=1200, n=1500, p=16)
    Xtr = d["X_train"].tolil()
    Xtr[:100] = 0
    Xtr = csr_array(Xtr.tocsr())
    Xtr.eliminate_zeros()
    A = d["A"].copy()
    A[200:260] = 0
    res = rb.calc_reco_metrics_ex(Xtr, d["X_test"], A, d["B"], k=10, **TOPK4, **BEYOND, break_ties_with_noise=False,
                                  consider_cold_start=False, min_pos_test=3, strict_min_pos_test=True, return_topk=True,
                                  return_status=True)
    assert (res.status[:100] == 1).all() and (res.status[200:260] == 3).any()
    users = _assert_rows(res, d["B"], _pop(Xtr, 1200), 1200)
    assert users == int((res.status == 0).sum())


def test_filter_fallback_users(rb):
    d = synth.make(4, m=4000, n=20000, p=32)
    A = d["A"].copy()
    A[np.arange(5, 4000, 211)] *= np.float32(1e-36)
    A[np.arange(9, 4000, 307)] *= np.float32(1e33)
    B = d["B"].copy()
    B[:, 0] = np.random.default_rng(2).integers(0, 3, 20000).astype(np.float32)
    A[np.arange(13, 4000, 401), 1:] = 0
    d["A"], d["B"] = A, B
    res = _run(rb, d, 20, scoring_path="tensor")
    assert res.timing["filter_fallback_users"] > 0
    _assert_rows(res, B, _pop(d["X_train"], 4000), 4000)


def test_forced_retry_pass(rb, monkeypatch):
    d = synth.make(4, m=300, n=70000)
    monkeypatch.setenv("RMB200_SAMPLE_RANK", "1")
    res = _run(rb, d, 100, scoring_path="tensor")
    assert res.timing["filter_retry_rows"] > 0
    _assert_rows(res, d["B"], _pop(d["X_train"], 300), 300)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("path", ["auto", "fma"])
def test_cumulative(rb, dtype, path):
    d = synth.make(1, m=800, n=1200, p=16)
    d["A"], d["B"] = d["A"].astype(dtype), d["B"].astype(dtype)
    cum = _run(rb, d, 15, cumulative=True, scoring_path=path)
    one = _run(rb, d, 15, scoring_path=path)
    _assert_rows(cum, d["B"], _pop(d["X_train"], 800), 800, cumulative=True)
    for key in KEYS:
        assert cum.metrics[key].shape == (800, 15)
        assert _same(cum.metrics[key][:, -1], one.metrics[key]), key
    assert np.isnan(cum.metrics["ILD@K"][:, 0]).all()


def test_shards_device_front_end_and_devices_are_bit_identical(rb):
    import torch
    d = synth.make(2, m=2500, n=4000, p=32)
    full = _run(rb, d, 20)
    halves = [_run(rb, d, 20, user_range=r) for r in ((0, 1100), (1100, 2500))]
    for key in KEYS:
        assert _same(np.concatenate([halves[0].metrics[key][:1100], halves[1].metrics[key][1100:]]), full.metrics[key]), key
    dev = torch.device("cuda", 0)
    A, B, b = (torch.from_numpy(x).to(dev) for x in (d["A"], d["B"], d["item_biases"]))
    r = rb.calc_reco_metrics_device(d["X_train"], d["X_test"], A, B, k=20, item_biases=b, **TOPK4, **BEYOND,
                                    break_ties_with_noise=False)
    for key in KEYS:
        assert r.metrics[key].is_cuda and _same(r.metrics[key].cpu().numpy(), full.metrics[key]), key
    if rb.device_count() >= 2:
        two = _run(rb, d, 20, devices=[0, 1])
        assert two.timing["devices_used"] == 2
        for key in KEYS:
            assert _same(two.metrics[key], full.metrics[key]), key


def test_two_devices_with_means(rb):
    if rb.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    d = synth.make(3, m=3001, n=9000, p=48)
    one = _run(rb, d, 20, return_means=True)
    two = _run(rb, d, 20, return_means=True, devices=[0, 1])
    for key in KEYS:
        assert _same(one.metrics[key], two.metrics[key]), key
        assert one.counts[key] == two.counts[key]
        assert two.means[key] == pytest.approx(one.means[key], rel=1e-12)


def test_item_popularity_is_the_bincount(rb):
    import torch
    d = synth.make(2, m=2000, n=3000, p=16)
    want = _pop(d["X_train"], 2000)
    assert np.array_equal(rb.item_popularity(d["X_train"]), want)
    assert np.array_equal(rb.item_popularity(d["X_train"], m=700), _pop(d["X_train"], 700))
    part = rb.item_popularity(d["X_train"], user_range=(700, 2000))
    assert np.array_equal(part + rb.item_popularity(d["X_train"], m=700), want)
    dev_csr = rb.DeviceCSR.from_scipy(d["X_train"], 0, with_data=False)
    got = rb.item_popularity(dev_csr)
    assert got.is_cuda and got.dtype == torch.int64 and np.array_equal(got.cpu().numpy(), want)
    # explicit counts give the very same rows, on both front-ends
    a = _run(rb, d, 10)
    b = _run(rb, d, 10, item_popularity=want)
    for key in KEYS:
        assert _same(a.metrics[key], b.metrics[key]), key
    A, B, bias = (torch.from_numpy(x).to("cuda:0") for x in (d["A"], d["B"], d["item_biases"]))
    for pop in (None, want, got):
        r = rb.calc_reco_metrics_device(d["X_train"], d["X_test"], A, B, k=10, item_biases=bias, **TOPK4, **BEYOND,
                                        break_ties_with_noise=False, item_popularity=pop)
        for key in KEYS:
            assert _same(r.metrics[key].cpu().numpy(), a.metrics[key]), key


def test_skewed_popularity_counter(rb):
    """Half the entries on one item: the grouped atomics still count exactly."""
    rng = np.random.default_rng(5)
    m, n = 20000, 50000
    nnz = rng.integers(0, 40, m)
    indptr = np.r_[0, np.cumsum(nnz)].astype(np.int32)
    rows = []
    for u in range(m):
        r = rng.choice(n - 1, nnz[u], replace=False) + 1
        if rng.random() < 0.5 and nnz[u]:
            r[0] = 0
        rows.append(np.sort(r))
    X = csr_array((np.ones(indptr[-1], np.float32), np.concatenate(rows).astype(np.int32), indptr), shape=(m, n))
    assert np.array_equal(rb.item_popularity(X), np.bincount(X.indices, minlength=n))


def test_closed_form_cases(rb):
    """Orthogonal rows: ILD 1.  Identical rows: ILD 0.  z zero rows among L identical ones: 1 - C(L - z, 2) / C(L, 2)."""
    rng = np.random.default_rng(3)
    m, n, K = 300, 64, 8
    A = rng.standard_normal((m, n)).astype(np.float64) * 1e-3
    bias = np.arange(n, dtype=np.float64)[::-1].copy()             # the list: items 0..K-1, in that order
    te = csr_array((np.ones(m), rng.integers(0, n, m), np.arange(m + 1)), shape=(m, n))
    kw = dict(k=K, item_biases=bias, **TOPK4, **BEYOND, break_ties_with_noise=False, return_topk=True)
    eye = np.eye(n) * rng.uniform(0.5, 2.0, (n, 1))
    r = rb.calc_reco_metrics_ex(None, te, A, eye, **kw)
    assert (r.topk_items == np.arange(K)).all()
    assert (r.metrics["ILD@K"] == 1.0).all()
    same = np.tile(rng.standard_normal((1, n)), (n, 1)) * rng.uniform(0.5, 2.0, (n, 1))
    r = rb.calc_reco_metrics_ex(None, te, A, same, **kw)
    np.testing.assert_allclose(r.metrics["ILD@K"], 0.0, atol=1e-12)
    z = 3
    same[[1, 4, 6]] = 0.0
    r = rb.calc_reco_metrics_ex(None, te, A, same, **kw)
    assert (r.topk_items == np.arange(K)).all()
    np.testing.assert_allclose(r.metrics["ILD@K"], 1.0 - (K - z) * (K - z - 1) / (K * (K - 1)), atol=1e-12)
    # no training data: every popularity is 0, Novelty log2(m + 1), AvgPop 0
    assert np.allclose(r.metrics["Novelty@K"], np.log2(m + 1), rtol=1e-14) and (r.metrics["AvgPop@K"] == 0).all()


@pytest.mark.parametrize("cumulative", [False, True])
def test_means_counts_and_means_only(rb, cumulative):
    d = synth.make(2, m=3000, n=5000, p=16)
    A = d["A"].copy()
    A[100:400] = 0                                                     # NaN users
    d["A"] = A
    res = _run(rb, d, 10, return_means=True, cumulative=cumulative)
    only = _run(rb, d, 10, means_only=True, cumulative=cumulative)
    for key in KEYS:
        rows = res.metrics[key].astype(np.float64)
        want = np.nanmean(rows, axis=0) if cumulative else float(np.nanmean(rows))
        cnt = (~np.isnan(rows)).sum(axis=0)
        np.testing.assert_allclose(res.means[key], want, rtol=1e-12, atol=1e-12, equal_nan=True)
        assert np.array_equal(res.counts[key], cnt)
        assert key not in only.metrics
        assert _same(np.asarray(only.means[key]), np.asarray(res.means[key])) and np.array_equal(only.counts[key], res.counts[key])


def test_nan_bits(rb):
    d = synth.make(1, m=600, n=900, p=8)
    A = d["A"].astype(np.float64)
    A[:25] = 0
    na_real = struct.unpack("<Q", struct.pack("<II", 1954, 0x7FF00000))[0]
    r0 = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], A, d["B"].astype(np.float64), k=5, **BEYOND, break_ties_with_noise=False)
    r1 = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], A, d["B"].astype(np.float64), k=5, **BEYOND, break_ties_with_noise=False,
                                 nan_bits=na_real)
    for key in KEYS:
        v, w = r0.metrics[key], r1.metrics[key]
        nan = np.isnan(v)
        assert nan[:25].all() and np.array_equal(nan, np.isnan(w)) and np.array_equal(v[~nan], w[~nan])
        assert (w[nan].view(np.uint64) == na_real).all(), key


def test_determinism(rb):
    d = synth.make(4, m=3000, n=70000, p=32)
    a, b = _run(rb, d, 100), _run(rb, d, 100)
    for key in KEYS:
        assert _same(a.metrics[key], b.metrics[key]), key


@pytest.mark.parametrize("path", ["auto", "fma"])
def test_accuracy_outputs_do_not_change(rb, path):
    d = synth.make(2, m=1500, n=3000, p=16)
    kw = dict(k=10, item_biases=d["item_biases"], all_metrics=True, break_ties_with_noise=False, scoring_path=path, return_topk=True,
              return_ranks=True, return_status=True, return_exposure=True, return_means=True)
    a = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], **kw)
    b = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], **kw, **BEYOND)
    for key, v in a.metrics.items():
        if key != "K":
            assert _same(v, b.metrics[key]), key
            assert _same(np.asarray(a.means[key]), np.asarray(b.means[key])), key
    for f in ("topk_items", "topk_scores", "pos_rank", "status", "exposure"):
        assert _same(getattr(a, f), getattr(b, f)), f
    assert a.catalogue == b.catalogue


def test_bad_popularity_on_the_device(rb):
    import torch
    d = synth.make(1, m=300, n=500, p=8)
    dev = torch.device("cuda", 0)
    A, B = torch.from_numpy(d["A"]).to(dev), torch.from_numpy(d["B"]).to(dev)
    from recometrics_b200 import _capi
    from recometrics_b200.frontend import _canonical_csr
    _, trp, tri = _canonical_csr(d["X_train"])
    Xte, tep, tei = _canonical_csr(d["X_test"])
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    bufs = [t(x) for x in (trp, tri, tep, tei, Xte.data.astype(np.float32))]
    pop = t(np.full(500, 301, dtype=np.int64))                         # above U = 300
    out = torch.empty(300, dtype=torch.float32, device=dev)
    bey = _capi.make_beyond({"novelty": out.data_ptr()}, pop.data_ptr(), 300)
    ex = _capi.make_extra(device=0, inputs_on_device=True)
    rc = _capi.calc_metrics(np.float32, A.data_ptr(), 8, B.data_ptr(), 8, 300, 500, 8, *[b.data_ptr() for b in bufs], 5, False, False,
                            {"p": torch.empty(300, device=dev).data_ptr()}, True, 2, 1, extra=ex, beyond=bey)
    assert rc == _capi.ERR_BAD_ARG and "outside" in _capi.last_error()
