"""CPU: the oracle's rules for non-finite scores and gains, pinned against hand-computed answers (the GPU tests of
test_gpu_nonfinite.py take the oracle as the spec).  One user row scores item j with B[j, 0] (A = [[1]]), so every score is
exactly the value written into B:

  * NaN candidate score                  -> NaN row (status 3), noise on or off, with or without ROC-AUC
  * noise off, partial path              -> only cs[0] and cs[K-1] are checked: -inf below the top K is harmless
  * noise off, ROC-AUC (full order)      -> cs[0] and the last candidate: -inf anywhere is fatal
  * noise on                             -> any +-inf candidate is fatal
  * non-finite scores of train items     -> no effect
  * gains: +inf or NaN anywhere -> NDCG NaN; -inf -> NaN exactly when fewer than L = min(K, npos) finite gains remain"""
import numpy as np
import pytest
from scipy.sparse import csr_array

N = 40
K = 5
TEST_ITEMS = (0, 2, 7, 30)        # held-out items; ranks 1, 3 and 8 of the clean order, and 31
INF, NAN = np.inf, np.nan


def _clean():
    return np.linspace(10.0, 1.0, N)                    # item j ranked j + 1: strictly decreasing scores


def _case(scores, train=(), gains=None, test=TEST_ITEMS):
    test = np.asarray(sorted(test), dtype=np.int32)
    g = np.ones(test.size) if gains is None else np.asarray(gains, dtype=np.float64)
    tr = np.asarray(sorted(train), dtype=np.int32)
    Xte = csr_array((g, test, np.array([0, test.size], dtype=np.int32)), shape=(1, N))
    Xtr = csr_array((np.ones(tr.size), tr, np.array([0, tr.size], dtype=np.int32)), shape=(1, N))
    return np.ones((1, 1)), np.asarray(scores, dtype=np.float64).reshape(N, 1), Xtr, Xte


def _run(oracle_mod, case, dtype, metrics=("p", "ndcg"), noise=False, k=K):
    A, B, Xtr, Xte = case
    return oracle_mod.oracle_calc(A, B, Xtr, Xte, k, metrics=metrics, extras=True, break_ties_with_noise=noise, seed=3,
                                  dtype=dtype)


DTYPES = [np.float32, np.float64]
MODES = [(False, ("p", "ndcg")), (False, ("p", "ndcg", "roc", "pr")), (True, ("p", "ndcg")), (True, ("p", "ndcg", "roc", "pr"))]


@pytest.mark.parametrize("dtype", DTYPES)
def test_clean_row_hand_computed(oracle_mod, dtype):
    r = _run(oracle_mod, _case(_clean()), dtype, metrics=("p", "ndcg", "roc"))
    assert r["status"][0] == 0
    assert r["p"][0] == dtype(2 / 5)
    idcg = sum(1 / np.log2(i + 2) for i in range(4))
    np.testing.assert_allclose(r["ndcg"][0], (1 / np.log2(2) + 1 / np.log2(4)) / idcg, rtol=1e-6)
    # ranks 1, 3, 8, 31 among 40 candidates: ROC = 1 - (sum(ranks) - 10) / (4 * 36)
    np.testing.assert_allclose(r["roc"][0], 1 - (1 + 3 + 8 + 31 - 10) / (4 * 36), rtol=1e-6)


@pytest.mark.parametrize("dtype", DTYPES)
def test_noise_off_partial_path_minus_inf_outside_the_top_k(oracle_mod, dtype):
    clean = _run(oracle_mod, _case(_clean()), dtype)
    for j in (K, 20, N - 1):                            # ranks K + 1, 21, 40: below the top K
        s = _clean()
        s[j] = -INF
        r = _run(oracle_mod, _case(s), dtype)
        assert r["status"][0] == 0, j
        assert r["p"][0] == clean["p"][0] and r["ndcg"][0] == clean["ndcg"][0], j
        assert list(r["topk_items"][0]) == [0, 1, 2, 3, 4]


@pytest.mark.parametrize("dtype", DTYPES)
def test_noise_off_partial_path_minus_inf_at_rank_k(oracle_mod, dtype):
    s = _clean()
    s[K - 1:] = -INF                                    # the K-th best score is -inf
    r = _run(oracle_mod, _case(s), dtype)
    assert r["status"][0] == 3 and np.isnan(r["p"][0]) and np.isnan(r["ndcg"][0])
    assert (r["topk_items"][0] == -1).all()


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("noise,metrics", MODES)
def test_plus_inf_at_the_top(oracle_mod, dtype, noise, metrics):
    s = _clean()
    s[13] = INF
    r = _run(oracle_mod, _case(s), dtype, metrics=metrics, noise=noise)
    assert r["status"][0] == 3 and all(np.isnan(r[q][0]) for q in metrics)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("j", [1, 20, N - 1])
def test_noise_off_roc_minus_inf_anywhere(oracle_mod, dtype, j):
    s = _clean()
    s[j] = -INF
    r = _run(oracle_mod, _case(s), dtype, metrics=("p", "ndcg", "roc"))
    # ROC-AUC needs the full order, whose smallest score is checked: -inf anywhere is a NaN row
    assert r["status"][0] == 3 and np.isnan(r["roc"][0]) and np.isnan(r["p"][0])


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("metrics", [("p", "ndcg"), ("p", "ndcg", "roc", "pr"), ("p", "ndcg", "pr")])
@pytest.mark.parametrize("value,j", [(INF, 20), (-INF, 20), (-INF, N - 1), (INF, 0)])
def test_noise_on_any_infinite_candidate(oracle_mod, dtype, metrics, value, j):
    s = _clean()
    s[j] = value
    r = _run(oracle_mod, _case(s), dtype, metrics=metrics, noise=True)
    assert r["status"][0] == 3 and all(np.isnan(r[q][0]) for q in metrics)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("noise,metrics", MODES)
@pytest.mark.parametrize("j", [0, K - 1, 20, N - 1])
def test_nan_anywhere(oracle_mod, dtype, noise, metrics, j):
    s = _clean()
    s[j] = NAN
    r = _run(oracle_mod, _case(s), dtype, metrics=metrics, noise=noise)
    assert r["status"][0] == 3 and all(np.isnan(r[q][0]) for q in metrics)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("noise,metrics", MODES)
def test_non_finite_train_items_change_nothing(oracle_mod, dtype, noise, metrics):
    train = (1, 5, 12, 25)
    clean = _run(oracle_mod, _case(_clean(), train=train), dtype, metrics=metrics, noise=noise)
    s = _clean()
    s[1], s[5], s[12], s[25] = NAN, INF, -INF, NAN
    r = _run(oracle_mod, _case(s, train=train), dtype, metrics=metrics, noise=noise)
    assert r["status"][0] == 0 == clean["status"][0]
    assert np.array_equal(r["topk_items"], clean["topk_items"])
    for q in metrics:
        assert r[q][0] == clean[q][0], q


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("cumulative", [False, True])
def test_gains(oracle_mod, dtype, cumulative):
    """NDCG with K = 5 and 4 held-out items (L = 4).  The gains sit on items 0, 2, 7, 30 (ranks 1, 3, 8, 31)."""
    def ndcg(gains):
        r = oracle_mod.oracle_calc(*_case(_clean(), gains=gains), K, metrics=("p", "ndcg"), extras=True, cumulative=cumulative,
                                   dtype=dtype)
        assert r["status"][0] == 0 and np.isfinite(r["p"]).all()        # gains never touch the row's status
        return np.atleast_1d(r["ndcg"][0])

    def want(gains):                                                    # hand-computed, finite gains only
        g = np.asarray(gains, dtype=np.float64)
        dcg = g[0] / np.log2(2) + g[1] / np.log2(4)
        ideal = np.sort(g)[::-1]
        return dcg / sum(ideal[i] / np.log2(i + 2) for i in range(4))

    assert np.isfinite(ndcg([1, 2, 3, 4])).all()
    np.testing.assert_allclose(ndcg([1, 2, 3, 4])[-1], want([1, 2, 3, 4]), rtol=1e-6)
    assert np.isnan(ndcg([1, INF, 3, 4])).all()                         # +inf: NaN
    assert np.isnan(ndcg([1, 2, 3, -INF])).all()                        # L = 4 but 3 finite gains: NaN
    assert np.isnan(ndcg([-INF, -INF, -INF, -INF])).all()
    for pos in range(4):                                                # NaN anywhere (quirk Q9): NaN
        g = [1.0, 2.0, 3.0, 4.0]
        g[pos] = NAN
        assert np.isnan(ndcg(g)).all(), pos
    # K = 2 (L = 2): two -inf gains leave exactly L finite ones, three leave fewer
    r = oracle_mod.oracle_calc(*_case(_clean(), gains=[4, -INF, -INF, 3]), 2, metrics=("ndcg",), extras=True, dtype=dtype)
    np.testing.assert_allclose(r["ndcg"][0], (4 / np.log2(2)) / (4 / np.log2(2) + 3 / np.log2(3)), rtol=1e-6)
    r = oracle_mod.oracle_calc(*_case(_clean(), gains=[4, -INF, -INF, -INF]), 2, metrics=("ndcg",), extras=True, dtype=dtype)
    assert np.isnan(r["ndcg"][0])
    r = oracle_mod.oracle_calc(*_case(_clean(), gains=[4, NAN, 2, 3]), 2, metrics=("ndcg",), extras=True, dtype=dtype)
    assert np.isnan(r["ndcg"][0])                                       # a NaN beyond L counts too


@pytest.mark.parametrize("dtype", DTYPES)
def test_noise_on_cases_match_the_compiled_reference(oracle_mod, dtype):
    """With the noise on the reference checks every candidate before sorting, so its answer is defined: compare."""
    if not oracle_mod.have_ref():
        pytest.skip("the compiled reference (oracle/_ref) is not built here")
    metrics = ("p", "ndcg", "roc", "pr")
    cases = []
    for j, v in ((20, -INF), (N - 1, -INF), (13, INF), (4, NAN), (30, NAN)):
        s = _clean()
        s[j] = v
        cases.append(_case(s))
    cases.append(_case(_clean()))
    for case in cases:
        A, B, Xtr, Xte = case
        ref = oracle_mod.ref_calc(A, B, Xtr, Xte, K, metrics=metrics, break_ties_with_noise=True, seed=3, dtype=dtype)
        orc = _run(oracle_mod, case, dtype, metrics=metrics, noise=True)
        for q in metrics:
            np.testing.assert_allclose(np.asarray(orc[q], np.float64), np.asarray(ref[q], np.float64), rtol=0, atol=1e-6,
                                       equal_nan=True, err_msg=q)
