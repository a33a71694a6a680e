"""GPU: non-finite and overflowing scores on every scoring path, against the oracle's NaN-row rules (DESIGN.md, "Non-finite
scores").  Inputs are synth.make data with one defect injected into a few percent of the users or items:

  N1  NaN rows of B, some of them in train rows (those users rank normally)
  N2  +-inf elements of B: +inf, -inf and NaN scores (inf * 0 on an exact zero of A, inf - inf)
  N3  item_biases -inf on ~1 % of the items ("banned"), +inf on one item, NaN on one item
  N4  NaN / +inf / -inf elements of A
  N5  finite float32 factors whose scores overflow: +inf at the top for some users, -inf far below the top K for others
  N6  X_test gains +inf, -inf (below and at the L = min(K, npos) threshold) and NaN

Each input goes through the tensor-core filter (and its hand-backs to the FMA tiles at n = 20 000 and to the full-order path
at n >= 32 768), the FMA tiles and the full-order path, noise off and on, with and without ROC/PR-AUC.  Checked: status and
the NaN pattern of every metric exactly as the oracle's; ids, scores and metrics by the north-star rule for users whose
candidate scores are all finite; and bit-identical results across paths where the paths promise them."""
import numpy as np
import pytest

import parity_utils as pu
from test_gpu_beyond import _assert_rows, _pop
from test_gpu_exposure import _check as _check_exposure
from tools import synth

pytestmark = pytest.mark.gpu

SEED = 7
TOPK = ("p", "r", "ap", "ndcg", "hit", "rr")
AUC = TOPK + ("roc", "pr")
PR_ONLY = ("p", "ap", "ndcg", "pr")


# ---------------------------------------------------------------------------------------------------------- inputs
def _base(n, m=300, p=32, dtype=np.float32, bias=False, cfg=1):
    d = synth.make(cfg, m=m, n=n, p=p)
    d["A"], d["B"] = d["A"].astype(dtype), d["B"].astype(dtype)
    d["item_biases"] = (0.5 * np.random.default_rng(5).standard_normal(n)).astype(dtype) if bias else None
    return d


def _train_items(d, u):
    X = d["X_train"]
    return X.indices[X.indptr[u]:X.indptr[u + 1]]


def n1_nan_rows(n, dtype=np.float32):
    """NaN in 3 rows of B, all three in the train rows of a few users: those users rank normally, everyone else is NaN."""
    d = _base(n, dtype=dtype)
    X = d["X_train"]
    cnt = np.bincount(X.indices, minlength=n)
    items = np.argsort(-cnt, kind="stable")[:3]            # the most popular items: many users have one or two of them
    has = np.zeros(X.shape[0], dtype=np.int64)
    for it in items:
        has += np.asarray((X[:, [int(it)]] != 0).todense()).ravel()
    d["B"][items] = np.nan
    d["spare"] = np.nonzero(has == 3)[0]
    return d


def n2_inf_elements(n, dtype=np.float32):
    """+-inf elements in 3 rows of B: B[r0, 0] = +inf, B[r1, 1] = -inf, B[r2, 2] = +inf with B[r2, 3] = -inf.  The signs of A
    make all three scores -inf for most users (harmless below the top K with the noise off); 2 % of the users score +inf on
    r0 (at the top), 2 % score inf - inf = NaN on r2, and 2 % have A[u, 1] = 0 exactly: -inf * 0 = NaN on r1."""
    d = _base(n, dtype=dtype)
    A = d["A"]
    rng = np.random.default_rng(21)
    r0, r1, r2 = rng.choice(n, 3, replace=False)
    d["B"][r0, 0], d["B"][r1, 1], d["B"][r2, 2], d["B"][r2, 3] = np.inf, -np.inf, np.inf, -np.inf
    A[:, 0], A[:, 1], A[:, 2], A[:, 3] = -np.abs(A[:, 0]), np.abs(A[:, 1]), -np.abs(A[:, 2]), np.abs(A[:, 3])
    top, diff, zero = np.split(rng.choice(A.shape[0], 3 * max(1, A.shape[0] // 50), replace=False), 3)
    A[top, 0] = -A[top, 0]
    A[diff, 2] = -A[diff, 2]
    A[zero, 1] = 0
    return d


def n3_bias(n, kind, dtype=np.float32):
    d = _base(n, dtype=dtype, bias=True)
    rng = np.random.default_rng(31)
    if kind == "banned":
        d["item_biases"][rng.choice(n, max(1, n // 100), replace=False)] = -np.inf
    else:
        d["item_biases"][int(rng.integers(n))] = np.inf if kind == "+inf" else np.nan
    return d


def n4_user_rows(n, dtype=np.float32):
    """NaN, +inf and -inf in one element each of 3 % of the users' rows of A."""
    d = _base(n, dtype=dtype)
    m, p = d["A"].shape
    rng = np.random.default_rng(41)
    users = rng.choice(m, 3 * max(1, m // 100), replace=False).reshape(3, -1)
    for val, us in zip((np.nan, np.inf, -np.inf), users):
        d["A"][us, rng.integers(p, size=us.shape[0])] = val
    return d


def n5_overflow(n, dtype=np.float32, scale=1e22):
    """Finite factors whose scores leave the range, through the last factor c alone.  A block of users (3 %) has
    A[u, c] = +scale * (1 + |a|), a block (3 %) -scale * (1 + |a|), every other user A[u, c] = 0; a set of items (2 %) has
    B[j, c] = scale * (1 + |b|).  A scaled user and a scaled item meet in one product >= scale**2, >= 100x beyond the range
    whatever the order of summation: the first block scores +inf at the top, the second -inf far below the top K.  Every
    other score is a sum of unscaled terms, or one scaled term plus unscaled ones: finite, and without cancellation."""
    d = _base(n, dtype=dtype)
    A, B = d["A"].astype(np.float64), d["B"].astype(np.float64)
    m = A.shape[0]
    rng = np.random.default_rng(51)
    up, down = np.split(rng.choice(m, 2 * max(1, (3 * m) // 100), replace=False), 2)
    items = rng.choice(n, max(1, n // 50), replace=False)
    A[:, -1] = 0
    A[up, -1] = scale * (1 + np.abs(rng.standard_normal(up.size)))
    A[down, -1] = -scale * (1 + np.abs(rng.standard_normal(down.size)))
    B[items, -1] = scale * (1 + np.abs(rng.standard_normal(items.size)))
    d["A"], d["B"] = A.astype(dtype), B.astype(dtype)
    assert np.isfinite(d["A"]).all() and np.isfinite(d["B"]).all()
    d["up"], d["down"] = up, down
    return d


def n5_narrow(n, dtype=np.float32):
    """Float32 overflow with a narrow spread of norms, which the fp16 filter can rank without handing anyone back.  B is scaled
    by 1e18; a contiguous block of items (2 %, whole 32-item chunks) gets B[j, c] = 4e21 * (1 + |b| / 10) in the last factor c.
    Two blocks of users (3 % each) get A[u] = 5e17 * a with A[u, c] = +1e19 or -1e19.  Such a user and such an item meet in
    one product >= 4e40, >= 100x beyond the range whatever the order of summation: +inf at the top for the first block,
    -inf far below the top K for the second.  The user's other scores stay below ||a|| ||b|| < 1.7e38: finite.  The norms
    involved lie within a factor of ~1000 of each other (||a|| ~ 1e19, ||b|| ~ 6e18 and ~4e21)."""
    d = _base(n, dtype=dtype)
    A, B = d["A"].astype(np.float64), d["B"].astype(np.float64)
    m = A.shape[0]
    rng = np.random.default_rng(52)
    B *= 1e18
    nb = 32 * max(1, n // 1600)
    items = np.arange(n // 2 // 32 * 32, n // 2 // 32 * 32 + nb)
    B[items, -1] = 4e21 * (1 + 0.1 * np.abs(rng.standard_normal(nb)))
    up, down = np.split(rng.choice(m, 2 * max(1, (3 * m) // 100), replace=False), 2)
    for users, sign in ((up, 1.0), (down, -1.0)):
        A[users] *= 5e17
        A[users, -1] = sign * 1e19
    d["A"], d["B"] = A.astype(dtype), B.astype(dtype)
    assert np.isfinite(d["A"]).all() and np.isfinite(d["B"]).all()
    d["up"], d["down"] = up, down
    return d


def n6_gains(n, K, dtype=np.float32):
    """X_test values: +inf (one user in 30), NaN (one in 30), -inf below the L threshold, and -inf on all but L - 1 values
    (one short of it), on users with enough held-out items."""
    d = _base(n, dtype=dtype)
    X = d["X_test"].copy()
    X.data = X.data.astype(dtype)
    npos = np.diff(X.indptr)
    rng = np.random.default_rng(61)
    for u in range(X.shape[0]):
        lo, hi = X.indptr[u], X.indptr[u + 1]
        if hi == lo:
            continue
        L = min(K, int(npos[u]))
        r = u % 30
        if r == 0:
            X.data[lo + rng.integers(hi - lo)] = np.inf
        elif r == 1:
            X.data[lo + rng.integers(hi - lo)] = np.nan
        elif r == 2 and npos[u] > L:
            X.data[lo:lo + (npos[u] - L)] = -np.inf          # exactly L finite gains remain: defined
        elif r == 3 and npos[u] >= L and L > 1:
            X.data[lo:lo + (npos[u] - L + 1)] = -np.inf      # L - 1 finite gains remain: NaN
    d["X_test"] = X
    return d


# ---------------------------------------------------------------------------------------------------------- checks
def _vs_oracle(res, orc, d, metrics, K, cumulative, label, pre=None):
    """status and every metric's NaN pattern exactly; ids, scores, ranks and metrics by the north-star rule (parity_utils:
    near ties are measured against the user's finite scores, so users with -inf candidates below the top K are compared
    too; N5's float32 overflow is invisible to the float64 scores there, and its users are held to status and NaN pattern)."""
    bad = np.nonzero(res.status != orc["status"])[0]
    assert bad.size == 0, f"{label}: status differs for users {bad[:10]}: {res.status[bad][:10]} vs oracle {orc['status'][bad][:10]}"
    for q in metrics:
        g, o = np.asarray(res.metrics[pu.KEY[q]]), np.asarray(orc[q])
        diff = np.nonzero((np.isnan(g) != np.isnan(o)).reshape(g.shape[0], -1).any(axis=1))[0]
        assert diff.size == 0, f"{label}: NaN pattern of {q} differs for users {diff[:10]}: {g[diff][:3]} vs oracle {o[diff][:3]}"
    assert (res.topk_items[res.status != 0] == -1).all(), label
    with np.errstate(invalid="ignore", over="ignore"):
        pu.compare(res, orc, d, metrics, K, cumulative=cumulative, max_amb_frac=1.0, label=label, pre=pre)


def _same(a, b, what):
    assert np.array_equal(a.status, b.status), what + ": status"
    assert np.array_equal(a.topk_items, b.topk_items), what + ": top-K ids"
    assert np.array_equal(a.topk_scores, b.topk_scores, equal_nan=True), what + ": top-K scores"
    if a.pos_rank is not None and b.pos_rank is not None:
        assert np.array_equal(a.pos_rank, b.pos_rank), what + ": ranks"
    for key, v in a.metrics.items():
        if key != "K":
            assert np.array_equal(v, b.metrics[key], equal_nan=True), what + ": " + key


def _run_all(rb, oracle_mod, d, K, metrics, noise, paths, cumulative=False, label=""):
    """Every path of `paths` against the oracle, then the cross-path identities; returns {path: EvalResult}."""
    dtype = d["A"].dtype.type
    orc = pu.run_oracle(oracle_mod, d, metrics, K, cumulative=cumulative, break_ties_with_noise=noise, seed=SEED)
    with np.errstate(invalid="ignore", over="ignore"):
        pre = pu.near_ties(d, K)                               # (once for all paths)
    out = {}
    for path in paths:
        res = pu.run_product(rb, d, metrics, K, cumulative=cumulative, break_ties_with_noise=noise, seed=SEED, scoring_path=path)
        _vs_oracle(res, orc, d, metrics, K, cumulative, f"{label} {path} K={K} noise={noise} {np.dtype(dtype).name} {metrics}", pre)
        out[path] = res
    if noise and "auto" in out and "full" in out:
        _same(out["auto"], out["full"], label + " auto vs full (noise)")
    if not noise and "fma" in out and "full" in out:
        _same(out["fma"], out["full"], label + " fma vs full")
    if not noise and "tensor" in out and "fma" in out:
        _same(out["tensor"], out["fma"], label + " tensor vs fma")
    out["oracle"] = orc
    return out


def _matrix(rb, oracle_mod, d, label):
    """The call matrix of one input: top-K only on every path (noise off and on), ROC/PR-AUC, PR-AUC alone (noise off and on),
    K = 100 / 300 / 500.  From 32 768 items on, where the filter hands users back to the full-order path instead of the FMA
    tiles, only the calls that take the filter.  Returns the results of the top-K calls at K = 10."""
    large = d["B"].shape[0] >= 32768
    top_off = _run_all(rb, oracle_mod, d, 10, TOPK, False, ("auto", "full") if large else ("auto", "tensor", "fma", "full"), label=label)
    top_on = _run_all(rb, oracle_mod, d, 10, TOPK, True, ("auto", "full") if large else ("auto", "tensor", "full"), label=label)
    assert top_off["auto"].timing["scoring_path"] == 2 and top_on["auto"].timing["scoring_path"] == 2
    assert top_off["full"].timing["scoring_path"] == 3
    auc_on = _run_all(rb, oracle_mod, d, 10, AUC, True, ("auto", "full"), label=label)
    assert auc_on["auto"].timing["scoring_path"] == 2          # tensor top-K after the FMA tiles counted the ranks
    _run_all(rb, oracle_mod, d, 10, PR_ONLY, True, ("auto", "full"), label=label)
    if large:
        return top_off, top_on
    assert top_off["fma"].timing["scoring_path"] == 1
    _run_all(rb, oracle_mod, d, 10, AUC, False, ("auto", "full"), label=label)
    pr_off = _run_all(rb, oracle_mod, d, 10, PR_ONLY, False, ("auto", "fma", "full"), label=label)
    assert pr_off["auto"].timing["scoring_path"] == 1          # rank counting without the noise: the FMA tiles
    _run_all(rb, oracle_mod, d, 100, TOPK, False, ("tensor", "fma", "full"), label=label)
    _run_all(rb, oracle_mod, d, 300, TOPK, False, ("auto", "full"), label=label)
    k300 = _run_all(rb, oracle_mod, d, 300, TOPK, True, ("auto", "full"), label=label)
    assert k300["auto"].timing["scoring_path"] == 3
    _run_all(rb, oracle_mod, d, 500, AUC, True, ("auto",), label=label)
    return top_off, top_on


def _status_counts(res):
    return {int(s): int((res.status == s).sum()) for s in np.unique(res.status)}


# ---------------------------------------------------------------------------------------------------------- tests
@pytest.mark.parametrize("n", [20000, 40000])
def test_n1_nan_item_rows(rb, oracle_mod, n):
    d = n1_nan_rows(n)
    assert d["spare"].size > 0
    off, on = _matrix(rb, oracle_mod, d, f"N1 n={n}")
    for res in (off["auto"], on["auto"]):
        assert (res.status[d["spare"]] == 0).any()                       # train-row NaN items change nothing
        assert _status_counts(res).get(3, 0) > d["A"].shape[0] // 2
        assert res.timing["filter_fallback_users"] > 0                    # non-finite max ||b||: every user is handed back


def test_n1_float64_and_beyond_accuracy(rb, oracle_mod):
    d = n1_nan_rows(20000, dtype=np.float64)
    _run_all(rb, oracle_mod, d, 10, TOPK, True, ("auto", "full"), label="N1 f64")
    _run_all(rb, oracle_mod, d, 10, AUC, False, ("auto", "full"), label="N1 f64")
    _beyond(rb, d, noise=False)
    _beyond(rb, d, noise=True)


@pytest.mark.parametrize("n", [20000, 40000])
def test_n2_inf_item_elements(rb, oracle_mod, n):
    d = n2_inf_elements(n)
    off, on = _matrix(rb, oracle_mod, d, f"N2 n={n}")
    assert off["auto"].timing["filter_fallback_users"] > 0
    # noise off: only the +inf and NaN users are NaN rows; noise on: every user (each one has an infinite candidate)
    assert 0 < _status_counts(off["auto"]).get(3, 0) < d["A"].shape[0] // 5
    assert (on["auto"].status == 3).all()


@pytest.mark.parametrize("kind", ["banned", "+inf", "nan"])
@pytest.mark.parametrize("n", [20000, 40000])
def test_n3_item_biases(rb, oracle_mod, kind, n):
    d = n3_bias(n, kind)
    off, on = _matrix(rb, oracle_mod, d, f"N3 {kind} n={n}")
    assert off["auto"].timing["filter_fallback_users"] > 0
    if kind == "banned":
        # noise off: a banned item below the top K is harmless; noise on (the reference's default): every row is NaN
        assert (off["auto"].status == 0).sum() > d["A"].shape[0] // 2
        assert (on["auto"].status[off["auto"].status == 0] == 3).all()


def test_n3_banned_float64_cumulative_and_beyond_accuracy(rb, oracle_mod):
    d = n3_bias(20000, "banned", dtype=np.float64)
    _run_all(rb, oracle_mod, d, 10, TOPK, True, ("auto", "full"), label="N3 f64")
    _run_all(rb, oracle_mod, d, 10, TOPK, False, ("auto", "fma", "full"), cumulative=True, label="N3 f64 cumulative")
    _beyond(rb, d, noise=False)


@pytest.mark.parametrize("n", [20000, 40000, 70000])
def test_n4_user_rows(rb, oracle_mod, n):
    d = n4_user_rows(n, dtype=np.float32)
    if n == 70000:                                                         # sampled threshold guess (pass 0) of the filter
        d = dict(d, A=d["A"][:200], X_train=d["X_train"][:200], X_test=d["X_test"][:200])
        off = _run_all(rb, oracle_mod, d, 10, TOPK, False, ("auto", "fma"), label="N4 n=70000")
        on = _run_all(rb, oracle_mod, d, 10, TOPK, True, ("auto", "full"), label="N4 n=70000")
        _run_all(rb, oracle_mod, d, 10, PR_ONLY, True, ("auto", "full"), label="N4 n=70000")
    else:
        off, on = _matrix(rb, oracle_mod, d, f"N4 n={n}")
    bad = ~np.isfinite(d["A"]).all(axis=1)
    assert (on["auto"].status[bad] != 0).all() and (off["auto"].status[bad] != 0).all()
    assert (off["auto"].status[~bad] == 0).sum() > 0.9 * (~bad).sum()
    assert off["auto"].timing["filter_fallback_users"] > 0                # unscalable user norms: handed back


def test_n4_float64(rb, oracle_mod):
    d = n4_user_rows(20000, dtype=np.float64)
    _run_all(rb, oracle_mod, d, 10, TOPK, True, ("auto", "full"), label="N4 f64")
    _run_all(rb, oracle_mod, d, 100, TOPK, False, ("tensor", "fma", "full"), label="N4 f64")


@pytest.mark.parametrize("n", [20000, 40000])
def test_n5_float32_overflow(rb, oracle_mod, n):
    d = n5_overflow(n)
    off, on = _matrix(rb, oracle_mod, d, f"N5 n={n}")
    orc_off, orc_on = off["oracle"], on["oracle"]
    # a spread of norms wide enough to overflow is too wide for the fp16 image: the overflowing users are handed back
    assert off["auto"].timing["filter_fallback_users"] >= d["up"].size + d["down"].size
    assert (orc_off["status"][d["up"]] == 3).all() and (orc_on["status"][d["up"]] == 3).all()      # +inf at the top
    assert (orc_off["status"][d["down"]] == 0).all() and (orc_on["status"][d["down"]] == 3).all()  # -inf below the top K


def test_n5_float32_overflow_narrow_spread(rb, oracle_mod):
    """Overflow the filter could rank itself: the users whose ||a|| * max ||b|| reaches the float range are handed back (flag
    8), so that a -inf below the top K is seen by the full-order path under the noise, with and without PR-AUC."""
    d = n5_narrow(20000)
    off, on = _matrix(rb, oracle_mod, d, "N5 narrow")
    orc_off, orc_on = off["oracle"], on["oracle"]
    assert (orc_off["status"][d["up"]] == 3).all() and (orc_on["status"][d["up"]] == 3).all()
    assert (orc_off["status"][d["down"]] == 0).all() and (orc_on["status"][d["down"]] == 3).all()
    others = np.setdiff1d(np.arange(d["A"].shape[0]), np.concatenate([d["up"], d["down"]]))
    assert (orc_off["status"][others] == 0).mean() > 0.9
    for res in (off["auto"], on["auto"]):
        assert res.timing["filter_fallback_users"] >= d["up"].size + d["down"].size     # the overflowing users at least


def test_n5_float64_overflow(rb, oracle_mod):
    d = n5_overflow(20000, dtype=np.float64, scale=1e160)
    off = _run_all(rb, oracle_mod, d, 10, TOPK, False, ("auto", "fma", "full"), label="N5 f64")
    on = _run_all(rb, oracle_mod, d, 10, TOPK, True, ("auto", "full"), label="N5 f64")
    _run_all(rb, oracle_mod, d, 10, AUC, True, ("auto", "full"), label="N5 f64")
    assert (off["oracle"]["status"][d["down"]] == 0).all() and (on["oracle"]["status"][d["down"]] == 3).all()


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n", [20000, 70000])
def test_n6_gains(rb, oracle_mod, dtype, n):
    for K in (10, 100):
        d = n6_gains(n, K, dtype=dtype)
        if n == 70000:
            d = dict(d, A=d["A"][:200], X_train=d["X_train"][:200], X_test=d["X_test"][:200])
        r = _run_all(rb, oracle_mod, d, K, TOPK, False, ("auto", "fma"), label=f"N6 K={K}")
        _run_all(rb, oracle_mod, d, K, TOPK, True, ("auto", "full"), label=f"N6 K={K}")
        _run_all(rb, oracle_mod, d, K, ("ndcg",), False, ("auto", "full"), cumulative=True, label=f"N6 K={K} cumulative")
        nd = r["auto"].metrics["NDCG@K"]
        assert np.isnan(nd[r["auto"].status == 0]).any() and np.isfinite(nd).any()


def _beyond(rb, d, noise):
    """Exposure and beyond-accuracy rows: NaN-row users count nothing and get NaN rows."""
    res = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], k=10, item_biases=d.get("item_biases"),
                                  precision=True, ndcg=True, break_ties_with_noise=noise, seed=SEED, return_topk=True,
                                  return_status=True, return_exposure=True, novelty=True, avg_popularity=True, diversity=True)
    m, n = d["A"].shape[0], d["B"].shape[0]
    users = _check_exposure(res, n)
    assert users == int((res.status == 0).sum())
    for key in ("Novelty@K", "AvgPop@K", "ILD@K"):
        assert np.isnan(res.metrics[key][res.status != 0]).all(), key
    if users:
        Bf = np.where(np.isfinite(d["B"]), d["B"], 0)                     # rows of listed items are finite
        assert _assert_rows(res, Bf, _pop(d["X_train"], m), m) == users
