"""GPU: per-user Unexpectedness@K and Serendipity@K of the ranked top-K lists against each user's training history
(unexpectedness / serendipity).  The reference is numpy in float64 on the same call's own topk_items (return_topk=True), the
X_train / X_test rows and the normalised rows of B, with the similarities from an explicit L x T_u matrix, not from the
history centroid the kernel uses.  Checked on every scoring path and every way a list can be decided, cold-start and
ineligible users, cumulative calls, bit-identity over shards, front-ends and devices, closed-form cases, the means, and
that no other output changes."""
import struct

import numpy as np
import pytest
from scipy.sparse import csr_array

from golden_io import load_case
from tools import synth

pytestmark = pytest.mark.gpu

TOPK4 = dict(precision=True, recall=True, average_precision=True, ndcg=True)
SER = dict(unexpectedness=True, serendipity=True)
KEYS = ("Unexpectedness@K", "Serendipity@K")


def _reference(ids, B, X_train, X_test, cumulative):
    """float64 rows from the listed ids (-1 = no list): Unexpectedness, Serendipity; (m,) or (m, K)."""
    m, K = ids.shape
    Bd = np.asarray(B, dtype=np.float64)
    nrm = np.linalg.norm(Bd, axis=1, keepdims=True)
    Un = np.divide(Bd, nrm, out=np.zeros_like(Bd), where=nrm > 0)
    Xtr, Xte = csr_array(X_train), csr_array(X_test)
    out = {key: np.full((m, K), np.nan) for key in KEYS}
    for u in range(m):
        L = int((ids[u] >= 0).sum())
        hist = Xtr.indices[Xtr.indptr[u]:Xtr.indptr[u + 1]]
        if L == 0 or hist.size == 0:
            continue
        it = ids[u, :L]
        S = Un[it] @ Un[hist].T                         # L x T_u cosine similarities
        dist = 1.0 - S.mean(axis=1)
        rel = np.isin(it, Xte.indices[Xte.indptr[u]:Xte.indptr[u + 1]])
        i = np.arange(1, L + 1, dtype=np.float64)
        out["Unexpectedness@K"][u, :L] = np.cumsum(dist) / i
        out["Serendipity@K"][u, :L] = np.cumsum(np.where(rel, dist, 0.0)) / i
    if not cumulative:
        out = {key: v[:, -1] for key, v in out.items()}
    return out


def _assert_rows(res, B, X_train, X_test, cumulative=False):
    """The rows against the reference; returns how many users are defined."""
    ids = np.asarray(res.topk_items)
    ref = _reference(ids, B, X_train, X_test, cumulative)
    f64 = res.metrics[KEYS[0]].dtype == np.float64
    ntrain = np.diff(csr_array(X_train).indptr)[: ids.shape[0]]
    undefined = (ids[:, 0] < 0) | (ntrain == 0)
    for key in KEYS:
        got = np.asarray(res.metrics[key]).astype(np.float64)
        want = ref[key]
        nan_want = np.isnan(want)
        if not cumulative:
            assert np.array_equal(np.isnan(got), undefined), key
        assert np.array_equal(np.isnan(got), nan_want), key
        if f64:
            np.testing.assert_allclose(got[~nan_want], want[~nan_want], rtol=1e-12, atol=1e-12, err_msg=key)
        else:
            np.testing.assert_allclose(got[~nan_want], want[~nan_want], rtol=0, atol=1e-6, err_msg=key)
    return int((~undefined).sum())


def _run(rb, d, k, **kw):
    kw = {**TOPK4, "break_ties_with_noise": False, **SER, **kw}
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
    assert res.metrics["Serendipity@K"].dtype == dtype
    assert _assert_rows(res, d["B"], d["X_train"], d["X_test"]) > 400
    assert np.nanmax(res.metrics["Serendipity@K"]) > 0          # some listed items are held out


def test_rank_counting_with_the_noise_hand_back(rb):
    c = load_case("g_noise_ties_f64")
    res = rb.calc_reco_metrics_ex(c["X_train"], c["X_test"], c["A"], c["B"], k=c["k"], all_metrics=True, seed=3,
                                  break_ties_with_noise=True, return_topk=True, **SER)
    assert res.timing["noise_handback_users"] > 0
    _assert_rows(res, c["B"], c["X_train"], c["X_test"])


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
    _assert_rows(res, B, d["X_train"], d["X_test"])


def test_forced_retry_pass(rb, monkeypatch):
    d = synth.make(4, m=300, n=70000)
    monkeypatch.setenv("RMB200_SAMPLE_RANK", "1")
    res = _run(rb, d, 100, scoring_path="tensor")
    assert res.timing["filter_retry_rows"] > 0
    _assert_rows(res, d["B"], d["X_train"], d["X_test"])


def _without_history(X, rows):
    X = X.tolil()
    X[rows] = 0
    X = csr_array(X.tocsr())
    X.eliminate_zeros()
    return X


def test_ineligible_nan_and_cold_start_users(rb):
    d = synth.make(1, m=1200, n=1500, p=16)
    Xtr = _without_history(d["X_train"], slice(0, 100))
    A = d["A"].copy()
    A[200:260] = 0
    kw = dict(k=10, **TOPK4, **SER, break_ties_with_noise=False, min_pos_test=3, strict_min_pos_test=True, return_topk=True,
              return_status=True)
    # without cold-start users: no list for the first 100 users (status 1) and NaN rows for the zero-factor ones (status 3)
    res = rb.calc_reco_metrics_ex(Xtr, d["X_test"], A, d["B"], consider_cold_start=False, **kw)
    assert (res.status[:100] == 1).all() and (res.status[200:260] == 3).any()
    users = _assert_rows(res, d["B"], Xtr, d["X_test"])
    assert users == int((res.status == 0).sum())
    # with them: the first 100 users have a list, but no history -- NaN rows
    res = rb.calc_reco_metrics_ex(Xtr, d["X_test"], A, d["B"], consider_cold_start=True, **kw)
    cold = (res.status[:100] == 0) & (res.topk_items[:100, 0] >= 0)
    assert cold.sum() > 50
    for key in KEYS:
        assert np.isnan(res.metrics[key][:100]).all(), key
    assert users == _assert_rows(res, d["B"], Xtr, d["X_test"])


def test_no_training_data(rb):
    import torch
    d = synth.make(1, m=500, n=800, p=8)
    r = rb.calc_reco_metrics_ex(None, d["X_test"], d["A"], d["B"], k=5, **TOPK4, **SER, break_ties_with_noise=False,
                                return_topk=True, return_means=True)
    assert (r.topk_items[:, 0] >= 0).sum() > 400
    dev = torch.device("cuda", 0)
    A, B = torch.from_numpy(d["A"]).to(dev), torch.from_numpy(d["B"]).to(dev)
    rd = rb.calc_reco_metrics_device(None, d["X_test"], A, B, k=5, **TOPK4, **SER, break_ties_with_noise=False)
    for key in KEYS:
        assert np.isnan(r.metrics[key]).all(), key
        assert np.isnan(r.means[key]) and r.counts[key] == 0, key
        assert torch.isnan(rd.metrics[key]).all(), key


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("path", ["auto", "fma"])
def test_cumulative(rb, dtype, path):
    d = synth.make(1, m=800, n=1200, p=16)
    d["A"], d["B"] = d["A"].astype(dtype), d["B"].astype(dtype)
    cum = _run(rb, d, 40, cumulative=True, scoring_path=path)
    one = _run(rb, d, 40, scoring_path=path)
    _assert_rows(cum, d["B"], d["X_train"], d["X_test"], cumulative=True)
    for key in KEYS:
        assert cum.metrics[key].shape == (800, 40)
        assert _same(cum.metrics[key][:, -1], one.metrics[key]), key


def test_shards_device_front_end_and_devices_are_bit_identical(rb):
    import torch
    d = synth.make(2, m=2500, n=4000, p=32)
    full = _run(rb, d, 20)
    halves = [_run(rb, d, 20, user_range=r) for r in ((0, 1100), (1100, 2500))]
    for key in KEYS:
        assert _same(np.concatenate([halves[0].metrics[key][:1100], halves[1].metrics[key][1100:]]), full.metrics[key]), key
    dev = torch.device("cuda", 0)
    A, B, b = (torch.from_numpy(x).to(dev) for x in (d["A"], d["B"], d["item_biases"]))
    kw = dict(k=20, item_biases=b, **TOPK4, **SER, break_ties_with_noise=False)
    r = rb.calc_reco_metrics_device(d["X_train"], d["X_test"], A, B, **kw)
    # device-resident CSR, one shard: the history rows are read at the shard's offset
    Xtr = rb.DeviceCSR.from_scipy(d["X_train"], 0, with_data=False)
    Xte = rb.DeviceCSR.from_scipy(d["X_test"], 0)
    part = rb.calc_reco_metrics_device(Xtr, Xte, A, B, user_range=(1100, 2500), **kw)
    for key in KEYS:
        assert r.metrics[key].is_cuda and _same(r.metrics[key].cpu().numpy(), full.metrics[key]), key
        assert _same(part.metrics[key][1100:].cpu().numpy(), full.metrics[key][1100:]), key
        assert torch.isnan(part.metrics[key][:1100]).all(), key
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


def _closed_form_case(rng, m=300, n=64, K=8):
    """The list of every user is items 0..K-1 (item biases decide it), the history lies in items 40..63 and the held-out
    items in 0..39."""
    A = rng.standard_normal((m, n)) * 1e-3
    bias = np.arange(n, dtype=np.float64)[::-1].copy()
    nh = rng.integers(1, 6, m)
    tr_idx = np.concatenate([np.sort(rng.choice(np.arange(40, n), c, replace=False)) for c in nh])
    tr = csr_array((np.ones(tr_idx.size), tr_idx, np.r_[0, np.cumsum(nh)]), shape=(m, n))
    nt = rng.integers(1, 4, m)
    te_idx = np.concatenate([np.sort(rng.choice(40, c, replace=False)) for c in nt])
    te = csr_array((np.ones(te_idx.size), te_idx, np.r_[0, np.cumsum(nt)]), shape=(m, n))
    kw = dict(k=K, item_biases=bias, **TOPK4, **SER, hit=True, break_ties_with_noise=False, return_topk=True)
    return A, tr, te, kw


def test_closed_form_cases(rb):
    """One-hot rows: a list orthogonal to the history gives Unexpectedness 1 and Serendipity = P@K.  Parallel rows: 0.  A
    history of zero rows: c = 0, so again 1 and P@K."""
    rng = np.random.default_rng(3)
    A, tr, te, kw = _closed_form_case(rng)
    K, n = kw["k"], A.shape[1]
    eye = np.eye(n) * rng.uniform(0.5, 2.0, (n, 1))
    r = rb.calc_reco_metrics_ex(tr, te, A, eye, **kw)
    assert (r.topk_items == np.arange(K)).all()
    assert (r.metrics["Unexpectedness@K"] == 1.0).all()
    assert _same(r.metrics["Serendipity@K"], r.metrics["P@K"]) and (r.metrics["Hit@K"] > 0).sum() > 50
    same = np.tile(rng.standard_normal((1, n)), (n, 1)) * rng.uniform(0.5, 2.0, (n, 1))
    r = rb.calc_reco_metrics_ex(tr, te, A, same, **kw)
    assert (r.topk_items == np.arange(K)).all()
    for key in KEYS:
        np.testing.assert_allclose(r.metrics[key], 0.0, atol=1e-12, err_msg=key)
    zero_hist = rng.standard_normal((n, n))
    zero_hist[40:] = 0.0
    r = rb.calc_reco_metrics_ex(tr, te, A, zero_hist, **kw)
    assert (r.topk_items == np.arange(K)).all()
    assert (r.metrics["Unexpectedness@K"] == 1.0).all()
    assert _same(r.metrics["Serendipity@K"], r.metrics["P@K"])


def test_unsupported_factor_count(rb):
    rng = np.random.default_rng(1)
    _, tr, te, kw = _closed_form_case(rng, m=50)
    for dtype, p in ((np.float32, 1025), (np.float64, 513)):
        A, B = rng.standard_normal((50, p)).astype(dtype), rng.standard_normal((64, p)).astype(dtype)
        for one in ("unexpectedness", "serendipity"):
            with pytest.raises(NotImplementedError, match="k <= 1024"):
                rb.calc_reco_metrics_ex(tr, te, A, B, **{**kw, **SER, one: False})
        r = rb.calc_reco_metrics_ex(tr, te, A[:, :-1], B[:, :-1], **kw)
        assert np.isfinite(r.metrics["Unexpectedness@K"]).all()


@pytest.mark.parametrize("cumulative", [False, True])
def test_means_counts_and_means_only(rb, cumulative):
    d = synth.make(2, m=3000, n=5000, p=16)
    A = d["A"].copy()
    A[100:400] = 0                                                     # NaN users
    d["A"] = A
    d["X_train"] = _without_history(d["X_train"], slice(500, 600))    # cold-start users: a list, NaN rows
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
    Xtr = _without_history(d["X_train"], slice(25, 40))
    na_real = struct.unpack("<Q", struct.pack("<II", 1954, 0x7FF00000))[0]
    kw = dict(k=5, **SER, break_ties_with_noise=False)
    r0 = rb.calc_reco_metrics_ex(Xtr, d["X_test"], A, d["B"].astype(np.float64), **kw)
    r1 = rb.calc_reco_metrics_ex(Xtr, d["X_test"], A, d["B"].astype(np.float64), **kw, nan_bits=na_real)
    for key in KEYS:
        v, w = r0.metrics[key], r1.metrics[key]
        nan = np.isnan(v)
        assert nan[:40].all() and np.array_equal(nan, np.isnan(w)) and np.array_equal(v[~nan], w[~nan])
        assert (w[nan].view(np.uint64) == na_real).all(), key


def test_determinism(rb):
    d = synth.make(4, m=3000, n=70000, p=32)
    a, b = _run(rb, d, 100), _run(rb, d, 100)
    for key in KEYS:
        assert _same(a.metrics[key], b.metrics[key]), key


@pytest.mark.parametrize("path", ["auto", "fma"])
def test_other_outputs_do_not_change(rb, path):
    d = synth.make(2, m=1500, n=3000, p=16)
    kw = dict(k=10, item_biases=d["item_biases"], all_metrics=True, break_ties_with_noise=False, scoring_path=path, return_topk=True,
              return_ranks=True, return_status=True, return_exposure=True, return_means=True,
              novelty=True, avg_popularity=True, diversity=True)
    a = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], **kw)
    b = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], **kw, **SER)
    assert set(b.metrics) == set(a.metrics) | set(KEYS)
    for key, v in a.metrics.items():
        if key != "K":
            assert _same(v, b.metrics[key]), key
            assert _same(np.asarray(a.means[key]), np.asarray(b.means[key])), key
            assert np.array_equal(a.counts[key], b.counts[key]), key
    for f in ("topk_items", "topk_scores", "pos_rank", "status", "exposure"):
        assert _same(getattr(a, f), getattr(b, f)), f
    assert a.catalogue == b.catalogue
