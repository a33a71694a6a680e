"""Shared helpers for the parity tests: run product + oracle on the same inputs and compare with the
north-star's rule:

  * float metrics within 1e-6 (same NaN pattern),
  * top-K item ids, hit counts and held-out ranks bit-exact,
  * EXCEPT for users flagged by a float64 re-scoring as near-tied: two candidate scores within a
    relative gap of 1e-6 at a place where their order matters (SURVEY 8(c)).  "Relative" is taken
    against the user's score scale S_u = max_j |score(u,j)| over the candidates: the rounding error
    of a p-term dot product does not shrink when the sum happens to land near zero, so a gap
    relative to the two scores themselves would be meaningless mid-ranking.  Those users are
    compared as sets / with a rank band, and their number is reported and bounded.
"""
import numpy as np

from tools import synth

REL_GAP = 1e-6     # the north-star's stated relative gap
METRIC_TOL = 1e-6  # the north-star's tolerance on float metrics

KEY = {"p": "P@K", "tp": "TP@K", "r": "R@K", "ap": "AP@K", "tap": "TAP@K", "ndcg": "NDCG@K",
       "hit": "Hit@K", "rr": "RR@K", "roc": "ROC_AUC", "pr": "PR_AUC"}


def scores_f64(A, B, bias=None):
    S = A.astype(np.float64) @ B.astype(np.float64).T
    if bias is not None:
        S += bias.astype(np.float64)[None, :]
    return S


def ambiguity(S64, X_train, X_test, K):
    """Per-user flags from float64 scores.
    topk_amb[u]: two neighbours inside ranks [1, K+1] of the candidate order are within REL_GAP.
    rank_amb[u]: some held-out item has another candidate within REL_GAP of its score.
    band[e]    : for every held-out entry, number of OTHER candidates inside its gap band."""
    m, n = S64.shape
    topk_amb = np.zeros(m, dtype=bool)
    rank_amb = np.zeros(m, dtype=bool)
    band = np.zeros(X_test.indptr[-1], dtype=np.int64)
    for u in range(m):
        s = S64[u].copy()
        tr = X_train.indices[X_train.indptr[u]:X_train.indptr[u + 1]]
        te = X_test.indices[X_test.indptr[u]:X_test.indptr[u + 1]]
        cand = n - tr.shape[0]
        if cand < 2 or np.isnan(np.delete(s, tr)).any():
            continue                                  # (a NaN candidate score: NaN row)
        s[tr] = np.nan                                # train items sort after every candidate, -inf ones included
        order = np.argsort(-s, kind="stable")[:cand]
        so = s[order]
        fin = so[np.isfinite(so)]
        if fin.size == 0:
            continue
        S_u = max(abs(fin[0]), abs(fin[-1]))          # the user's score scale (over its finite scores)
        top = so[: min(K + 1, cand)]
        gaps = np.abs(np.diff(top))
        topk_amb[u] = bool(np.any(gaps <= REL_GAP * S_u))
        if te.shape[0]:
            asc = so[::-1]
            tol = REL_GAP * S_u
            for q, item in enumerate(te):
                v = s[item]
                lo = np.searchsorted(asc, v - tol, side="left")
                hi = np.searchsorted(asc, v + tol, side="right")
                band[X_test.indptr[u] + q] = hi - lo - 1
            rank_amb[u] = bool(np.any(band[X_test.indptr[u]:X_test.indptr[u + 1]] > 0))
    return topk_amb, rank_amb, band


def nan_equal_close(a, b, tol):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    both_nan = np.isnan(a) & np.isnan(b)
    with np.errstate(invalid="ignore"):
        close = np.abs(a - b) <= tol
    return both_nan | (close & ~np.isnan(a) & ~np.isnan(b))


def run_product(rb, data, metrics, k, cumulative=False, dtype=None, separate_bias=True, extras=True, **kw):
    flags = dict(precision="p" in metrics, trunc_precision="tp" in metrics, recall="r" in metrics,
                 average_precision="ap" in metrics, trunc_average_precision="tap" in metrics,
                 ndcg="ndcg" in metrics, hit="hit" in metrics, rr="rr" in metrics,
                 roc_auc="roc" in metrics, pr_auc="pr" in metrics)
    A, B, bias = data["A"], data["B"], data.get("item_biases")
    if dtype is not None:
        A, B = A.astype(dtype), B.astype(dtype)
        bias = None if bias is None else bias.astype(dtype)
    if bias is not None and not separate_bias:
        A, B = synth.fold_biases(A, B, bias)
        bias = None
    noise = bool(kw.pop("break_ties_with_noise", False))
    return rb.calc_reco_metrics_ex(
        data["X_train"], data["X_test"], A, B, k=k, item_biases=bias, cumulative=cumulative,
        break_ties_with_noise=noise, return_topk=extras, return_ranks=extras and ("roc" in metrics or "pr" in metrics),
        return_status=extras, **flags, **kw)


def run_oracle(oracle, data, metrics, k, cumulative=False, dtype=None, **kw):
    A, B, bias = data["A"], data["B"], data.get("item_biases")
    dt = A.dtype.type if dtype is None else dtype
    A, B = synth.fold_biases(A.astype(dt), B.astype(dt), None if bias is None else bias.astype(dt))
    return oracle.oracle_calc(A, B, data["X_train"], data["X_test"], k, metrics=metrics, cumulative=cumulative,
                              nthreads=8, fix_quirks=True, extras=True, dtype=dt, **kw)


def near_ties(data, k):
    """The float64 scores and ambiguity() of `data` at `k`: what compare() needs from the inputs alone, to be reused by
    several compare() calls on the same inputs (pre=)."""
    S64 = scores_f64(data["A"], data["B"], data.get("item_biases"))
    return (S64,) + ambiguity(S64, data["X_train"], data["X_test"], k)


def compare(res, orc, data, metrics, k, cumulative=False, check_ranks=True, max_amb_frac=0.25, label="", pre=None):
    """Assert parity between a product EvalResult and the oracle's dict.  Returns a report dict.
    pre: near_ties(data, k), when the caller compares several results on the same inputs."""
    A, B, bias = data["A"], data["B"], data.get("item_biases")
    X_train, X_test = data["X_train"], data["X_test"]
    m = X_test.shape[0]
    S64, topk_amb, rank_amb, band = near_ties(data, k) if pre is None else pre
    # exact ties inside the oracle's own float scores (reference order unspecified there too)
    tie = orc["tie_flags"]
    topk_amb = topk_amb | ((tie & 1) != 0)
    rank_amb = rank_amb | ((tie & 2) != 0)

    rep = dict(label=label, users=m, topk_ambiguous=int(topk_amb.sum()), rank_ambiguous=int(rank_amb.sum()))

    # ---- status (NaN-row decisions): exact, apart from the score-validity rule on near-tied users
    st_bad = (res.status != orc["status"]) & ~topk_amb
    assert not st_bad.any(), f"{label}: status differs for users {np.nonzero(st_bad)[0][:10]}"

    # ---- top-K ids: exact; near-tied users must at least agree as sets up to the tied items
    ids_g, ids_o = res.topk_items, orc["topk_items"]
    row_equal = (ids_g == ids_o).all(axis=1)
    bad = ~row_equal & ~topk_amb
    assert not bad.any(), (f"{label}: top-K ids differ for non-ambiguous users {np.nonzero(bad)[0][:10]}: "
                           f"{ids_g[bad][:2]} vs {ids_o[bad][:2]}")
    rep["topk_rows_differing"] = int((~row_equal).sum())
    for u in np.nonzero(~row_equal)[0]:
        # near-tied user: whatever differs must sit inside a near-tie of the float64 scores
        go, oo = ids_g[u], ids_o[u]
        if (go < 0).any() or (oo < 0).any():
            continue   # NaN-row decision differed on a near-tie (status check above covers non-ambiguous)
        pos = go != oo
        sa, sb = S64[u][go[pos]], S64[u][oo[pos]]
        lim = 4 * REL_GAP * np.maximum(1.0, np.maximum(np.abs(sa), np.abs(sb)))
        assert np.all(np.abs(sa - sb) <= lim), \
            f"{label}: user {u}: top-K order differs where float64 scores are NOT near-tied: {go[pos]} vs {oo[pos]}"

    # ---- top-K scores: GPU fp accumulation order differs from the CPU's SIMD order -> tolerance
    sg, so = res.topk_scores, orc["topk_scores"]
    eps = 2e-5 if sg.dtype == np.float32 else 1e-12
    scale = np.maximum(1.0, np.where(np.isfinite(S64), np.abs(S64), 0).max(axis=1, keepdims=True))
    ok = nan_equal_close(sg / scale, so / scale, eps) | ~row_equal[:, None]
    assert ok.all(), f"{label}: top-K scores differ beyond accumulation-order tolerance"

    # ---- float metrics within 1e-6 with the same NaN pattern.  Users on a near-tie: top-K metrics are
    #      exempt (their ids are checked above to differ only at the near-tied positions); ROC/PR-AUC get
    #      the tolerance that their rank bands allow (a rank moving by d changes ROC by d/(npos*nneg)).
    user_of = np.repeat(np.arange(m), np.diff(X_test.indptr))
    npos_u = np.diff(X_test.indptr).astype(np.float64)
    cand_u = (X_test.shape[1] - np.diff(X_train.indptr)).astype(np.float64)
    tot_band = np.zeros(m, dtype=np.float64)
    np.add.at(tot_band, user_of, band)
    tot_band += 2.0 * ((tie & 2) != 0)
    with np.errstate(divide="ignore", invalid="ignore"):
        roc_tol = METRIC_TOL + 2.0 * tot_band / np.maximum(npos_u * (cand_u - npos_u), 1.0)
    pr_tol = np.full(m, METRIC_TOL)
    if orc.get("pos_rank") is not None and ("pr" in metrics):
        ro = orc["pos_rank"].astype(np.float64)
        for u in np.nonzero(rank_amb)[0]:
            r = np.sort(ro[X_test.indptr[u]:X_test.indptr[u + 1]])
            if r.size == 0 or r[0] <= 0:
                continue
            h = np.arange(1, r.size + 1, dtype=np.float64)
            lo_rank = np.maximum(r - 2 * tot_band[u], h)
            pr_tol[u] += 2.0 * float(np.sum(h / lo_rank - h / r)) / r.size
    worst = 0.0
    for q in metrics:
        g, o = res.metrics[KEY[q]], orc[q]
        if q == "roc":
            okm = nan_equal_close(g, o, roc_tol)
            amb = np.zeros(m, dtype=bool)
        elif q == "pr":
            okm = nan_equal_close(g, o, pr_tol)
            amb = np.zeros(m, dtype=bool)
        else:
            okm = nan_equal_close(g, o, METRIC_TOL)
            amb = topk_amb
        if okm.ndim == 2:
            okm = okm.all(axis=1)
        badm = ~okm & ~amb
        assert not badm.any(), (f"{label}: metric {q} differs for non-ambiguous users {np.nonzero(badm)[0][:10]}: "
                                f"{np.asarray(g)[badm][:3]} vs {np.asarray(o)[badm][:3]}")
        with np.errstate(invalid="ignore"):
            d = np.abs(np.asarray(g, dtype=np.float64) - np.asarray(o, dtype=np.float64))
        if d.ndim == 2:
            d = np.nanmax(np.where(np.isnan(d), 0, d), axis=1)
        excl = (rank_amb if q in ("roc", "pr") else topk_amb) | np.isnan(d)
        rep["max_abs_diff_" + q] = float(np.where(np.isnan(d), 0, d).max()) if d.size else 0.0
        d = np.where(excl, 0, d)
        worst = max(worst, float(d.max()) if d.size else 0.0)
        rep["mismatch_" + q] = int((~nan_equal_close(g, o, METRIC_TOL).reshape(m, -1).all(axis=1)).sum())
    rep["max_metric_abs_diff_nonambiguous"] = worst

    # ---- hit counts (integers) recovered from P@K: exact for non-ambiguous users
    if "p" in metrics and not cumulative:
        hg = np.rint(np.nan_to_num(res.metrics["P@K"].astype(np.float64)) * k)
        ho = np.rint(np.nan_to_num(orc["p"].astype(np.float64)) * k)
        assert ((hg == ho) | topk_amb).all(), f"{label}: hit counts differ"

    # ---- ranks of held-out items: exact, or within the band of near-tied candidates
    if check_ranks and res.pos_rank is not None and ("roc" in metrics or "pr" in metrics):
        rg, ro = res.pos_rank, orc["pos_rank"]
        slack = band.copy()
        slack[((tie & 2) != 0)[user_of]] += 2
        # a near-tie between two other candidates cannot move this entry, but near-ties of
        # held-out items among themselves shift each other: allow the user's total band
        slack = np.where(band > 0, tot_band[user_of].astype(np.int64) + slack, slack)
        badr = np.abs(rg - ro) > slack
        assert not badr.any(), (f"{label}: held-out ranks differ beyond the near-tie band for entries "
                                f"{np.nonzero(badr)[0][:10]}: {rg[badr][:5]} vs {ro[badr][:5]} slack {slack[badr][:5]}")
        rep["rank_entries_differing"] = int((rg != ro).sum())

    frac = rep["topk_ambiguous"] / max(m, 1)
    assert frac <= max_amb_frac, f"{label}: {frac:.3f} of users ambiguous -- test data too degenerate to prove parity"
    return rep
