"""GPU: item exposure of the ranked top-K lists (return_exposure).  The central identity, on every scoring path and every way
a list can be decided: the counts equal numpy.bincount of the call's own defined topk_items, the counted users are its
status-0 rows, and the statistics are rmb200_exposure_stats of the counts.  Plus sharding (user_range, means_only, the device
front-end, two GPUs), a contention fixture with closed-form statistics, both catalogue sizes and determinism."""
import numpy as np
import pytest
from scipy.sparse import csr_array

from golden_io import load_case
from tools import synth

pytestmark = pytest.mark.gpu

TOPK4 = dict(precision=True, recall=True, average_precision=True, ndcg=True)


def _check(res, n, rows=slice(None)):
    """exposure == bincount(topk_items) of the same call; users == its status-0 rows; statistics from the counts."""
    from recometrics_b200 import _capi
    ids = np.asarray(res.topk_items)[rows]
    want = np.bincount(ids[ids >= 0], minlength=n)
    got = np.asarray(res.exposure)
    assert got.dtype == np.int64 and got.shape == (n,)
    assert np.array_equal(got, want)
    users = int((np.asarray(res.status)[rows] == 0).sum())
    assert res.catalogue["users"] == users
    assert res.catalogue["entries"] == int(want.sum())
    stats = _capi.exposure_stats(got, users=users)
    assert _same_stats(res.catalogue, stats)
    return users


def _same_stats(a, b):
    """Equal statistics, bit for bit (NaN equal to NaN)."""
    return a.keys() == b.keys() and all(np.array_equal(np.float64(a[k]), np.float64(b[k]), equal_nan=True) for k in a)


def _run(rb, d, k, **kw):
    kw = {**TOPK4, "break_ties_with_noise": False, **kw}
    return rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], k=k, item_biases=d.get("item_biases"),
                                   return_topk=True, return_status=True, return_exposure=True, **kw)


# (k, scoring_path, noise, expected timing["scoring_path"]): tensor filter; FMA tiles; K = 300 without the noise, which only
# the FMA tiles take; full order for K = 400 and for K = 300 with the noise
PATHS = [(10, "auto", False, 2), (10, "auto", True, 2), (10, "fma", False, 1), (300, "auto", False, 1),
         (400, "auto", False, 3), (300, "auto", True, 3)]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("k,path,noise,expect", PATHS)
def test_counts_are_the_bincount_of_the_lists(rb, dtype, k, path, noise, expect):
    d = synth.make(2, m=1500, n=3000, p=16)
    d["A"], d["B"], d["item_biases"] = d["A"].astype(dtype), d["B"].astype(dtype), d["item_biases"].astype(dtype)
    res = _run(rb, d, k, scoring_path=path, break_ties_with_noise=noise)
    assert res.timing["scoring_path"] == expect
    assert _check(res, 3000) > 500


def test_without_exposure_nothing_changes(rb):
    """The same call without return_exposure: identical rows and lists, and exactly the two kinds of kernels fewer
    (one count per user batch, one widening)."""
    d = synth.make(2, m=1500, n=3000, p=16)
    a = _run(rb, d, 10)
    b = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], k=10, item_biases=d["item_biases"], **TOPK4,
                                break_ties_with_noise=False, return_topk=True, return_status=True)
    assert b.exposure is None and b.catalogue is None
    assert np.array_equal(a.topk_items, b.topk_items) and np.array_equal(a.status, b.status)
    for key, v in b.metrics.items():
        if key != "K":
            assert np.array_equal(v, a.metrics[key], equal_nan=True), key
    assert a.timing["kernel_launches"] == b.timing["kernel_launches"] + 2


def test_rank_counting_with_the_noise_hand_back(rb):
    """ROC/PR-AUC with the tie-breaking noise on inputs full of exact ties: users for whom the noise decides a rank are re-ranked
    on the full-order path after the FMA tiles counted; their final lists are what is counted."""
    c = load_case("g_noise_ties_f64")
    res = rb.calc_reco_metrics_ex(c["X_train"], c["X_test"], c["A"], c["B"], k=c["k"], all_metrics=True, seed=3,
                                  break_ties_with_noise=True, return_topk=True, return_status=True, return_exposure=True)
    assert res.timing["noise_handback_users"] > 0
    _check(res, c["B"].shape[0])


@pytest.mark.parametrize("path", ["auto", "fma"])
def test_cumulative(rb, path):
    d = synth.make(1, m=800, n=1200, p=16)
    res = _run(rb, d, 15, cumulative=True, scoring_path=path)
    _check(res, 1200)


def test_ineligible_and_nan_users_add_nothing(rb):
    """Cold-start users (no training items, consider_cold_start=False), users below min_pos_test and users whose scores all tie
    (zero factors, no biases) have no list: status 1 / 3, all -1 rows, nothing counted."""
    d = synth.make(1, m=1200, n=1500, p=16)
    Xtr = d["X_train"].tolil()
    Xtr[:100] = 0
    Xtr = csr_array(Xtr.tocsr())
    Xtr.eliminate_zeros()
    A = d["A"].copy()
    A[200:260] = 0
    res = rb.calc_reco_metrics_ex(Xtr, d["X_test"], A, d["B"], k=10, **TOPK4, break_ties_with_noise=False, consider_cold_start=False,
                                  min_pos_test=3, strict_min_pos_test=True, return_topk=True, return_status=True, return_exposure=True)
    st = res.status
    assert (st[:100] == 1).all() and np.isin(st[200:260], (1, 3)).all() and (st[200:260] == 3).any()
    users = _check(res, 1500)
    assert users == int((st == 0).sum()) and res.catalogue["entries"] == 10 * users


def test_filter_fallback_users(rb):
    """Heavy-tailed input: users whose factors cannot be scaled into fp16 or whose scores nearly tie leave the tensor path
    per user; their re-ranked lists are counted."""
    d = synth.make(4, m=5000, n=20000, p=32)
    A = d["A"].copy()
    A[np.arange(5, 5000, 211)] *= np.float32(1e-36)
    A[np.arange(9, 5000, 307)] *= np.float32(1e33)
    B = d["B"].copy()
    B[:, 0] = np.random.default_rng(2).integers(0, 3, 20000).astype(np.float32)
    A[np.arange(13, 5000, 401), 1:] = 0
    d["A"], d["B"] = A, B
    res = _run(rb, d, 20, scoring_path="tensor")
    assert res.timing["filter_fallback_users"] > 0
    _check(res, 20000)


def test_forced_retry_pass(rb, monkeypatch):
    d = synth.make(4, m=300, n=70000)
    monkeypatch.setenv("RMB200_SAMPLE_RANK", "1")
    res = _run(rb, d, 100, scoring_path="tensor")
    assert res.timing["filter_retry_rows"] > 0
    _check(res, 70000)


def test_user_range_shards_add_up(rb):
    """Per-shard counts add up to the whole call's; the statistics of the sum are the whole call's, bit for bit."""
    from recometrics_b200 import _capi
    d = synth.make(1, m=2000, n=1500, p=16)
    full = _run(rb, d, 10)
    _check(full, 1500)
    parts = [_run(rb, d, 10, user_range=r) for r in ((0, 700), (700, 700), (700, 2000))]
    for p, r in zip(parts, ((0, 700), (700, 700), (700, 2000))):
        _check(p, 1500, rows=slice(*r))
    total = sum(p.exposure for p in parts)
    assert np.array_equal(total, full.exposure)
    assert parts[1].catalogue["users"] == 0 and parts[1].exposure.sum() == 0 and np.isnan(parts[1].catalogue["Gini@K"])
    users = sum(p.catalogue["users"] for p in parts)
    assert _same_stats(_capi.exposure_stats(total, users=users), full.catalogue)


def test_means_only(rb):
    d = synth.make(2, m=3000, n=5000, p=16)
    full = _run(rb, d, 10)
    only = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], k=10, item_biases=d["item_biases"], **TOPK4,
                                   break_ties_with_noise=False, means_only=True, return_exposure=True)
    assert list(only.metrics) == ["K"]
    assert np.array_equal(only.exposure, full.exposure) and _same_stats(only.catalogue, full.catalogue)
    # through the C-ABI, a call asking for nothing but the exposure computes the lists as well
    from recometrics_b200 import _capi
    from recometrics_b200.frontend import _canonical_csr
    _, trp, tri = _canonical_csr(d["X_train"])
    Xte, tep, tei = _canonical_csr(d["X_test"])
    counts = np.full(5000, -7, dtype=np.int64)
    expo = _capi.make_exposure(counts)
    rc = _capi.calc_metrics(np.float32, d["A"], 16, d["B"], 16, 3000, 5000, 16, trp, tri, tep, tei, Xte.data.astype(np.float32), 10,
                            False, False, {}, True, 2, 1, item_biases=d["item_biases"], exposure=expo)
    _capi.raise_for_status(rc)
    assert np.array_equal(counts, full.exposure) and _same_stats(expo.catalogue(), full.catalogue)


def test_device_front_end_equals_host_front_end(rb):
    import torch
    d = synth.make(2, m=2500, n=4000, p=32)
    host = _run(rb, d, 20)
    dev = torch.device("cuda", 0)
    A, B, b = (torch.from_numpy(x).to(dev) for x in (d["A"], d["B"], d["item_biases"]))
    for means_only in (False, True):
        r = rb.calc_reco_metrics_device(d["X_train"], d["X_test"], A, B, k=20, item_biases=b, **TOPK4, break_ties_with_noise=False,
                                        return_exposure=True, means_only=means_only)
        assert r.exposure.is_cuda and r.exposure.dtype == torch.int64
        assert np.array_equal(r.exposure.cpu().numpy(), host.exposure)
        assert _same_stats(r.catalogue, host.catalogue)


def test_two_devices_equal_one_device(rb):
    if rb.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    d = synth.make(3, m=3001, n=9000, p=48)
    one = _run(rb, d, 20, all_metrics=True)
    two = _run(rb, d, 20, all_metrics=True, devices=[0, 1])
    assert two.timing["devices_used"] == 2
    assert np.array_equal(one.exposure, two.exposure) and _same_stats(one.catalogue, two.catalogue)
    _check(two, 9000)


@pytest.mark.parametrize("n", [3706, 1 << 20])
def test_contention_every_user_lists_the_same_items(rb, n):
    """Item biases dominate the scores: every user's list is the same K items, so every increment of a rank goes to one
    address.  Counts are the users at exactly those items; coverage K/n, Gini (n - K)/n, entropy log2 K."""
    m, K = 4000 if n < 100000 else 600, 10
    rng = np.random.default_rng(8)
    A = (1e-6 * rng.standard_normal((m, 8))).astype(np.float32)
    B = rng.standard_normal((n, 8)).astype(np.float32)
    bias = rng.permutation(n).astype(np.float32)                   # distinct, far apart: the top K are the K largest
    te = csr_array((np.ones(m, dtype=np.float32), rng.integers(0, n, m), np.arange(m + 1)), shape=(m, n))
    res = rb.calc_reco_metrics_ex(None, te, A, B, k=K, item_biases=bias, **TOPK4, break_ties_with_noise=False,
                                  return_topk=True, return_status=True, return_exposure=True)
    assert (res.status == 0).all()
    top = np.argsort(bias)[-K:]
    want = np.zeros(n, dtype=np.int64)
    want[top] = m
    assert np.array_equal(res.exposure, want)
    cat = res.catalogue
    assert cat["users"] == m and cat["entries"] == m * K and cat["items_covered"] == K
    assert cat["Coverage@K"] == K / n
    assert cat["Gini@K"] == pytest.approx((n - K) / n, rel=1e-15)
    assert cat["Entropy@K"] == pytest.approx(np.log2(K), rel=1e-15)
    _check(res, n)


@pytest.mark.parametrize("n", [3706, 1 << 20])
def test_catalogue_sizes(rb, n):
    d = synth.make(4, m=4000 if n < 100000 else 400, n=n, p=32)
    res = _run(rb, d, 50)
    _check(res, n)


def test_determinism(rb):
    d = synth.make(4, m=3000, n=70000, p=32)
    a, b = _run(rb, d, 100), _run(rb, d, 100)
    assert np.array_equal(a.exposure, b.exposure)
    assert _same_stats(a.catalogue, b.catalogue)
