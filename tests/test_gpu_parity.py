"""GPU: parity of the CUDA path (called through the C-ABI) with the oracle, on the BASELINE
configurations at sizes the oracle finishes in seconds, on the committed golden vectors of the
unmodified reference, and on the edge cases the reference's own tests cover.

Rule (north star): integer outputs and top-K ids exact except inside a stated 1e-6 relative score gap
(float64 re-scoring decides, parity_utils.ambiguity); float metrics within 1e-6, NaN pattern equal."""
import json
import os

import numpy as np
import pytest
from scipy.sparse import csr_array

import parity_utils as pu
from golden_io import case_names, load_case
from tools import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True, params=["auto", "fma"])
def scoring_path(request, monkeypatch):
    """Every parity case runs twice: with the library's automatic choice (tensor-core filter + exact
    re-scoring wherever only top-K metrics are requested) and with every score on the FMA pipe."""
    if request.param == "auto":
        monkeypatch.delenv("RMB200_PATH", raising=False)
    else:
        monkeypatch.setenv("RMB200_PATH", request.param)
    return request.param

REPORT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out", "parity_report.jsonl")


def _log(rep):
    os.makedirs(os.path.dirname(REPORT), exist_ok=True)
    with open(REPORT, "a") as f:
        f.write(json.dumps(rep) + "\n")


def _check(rb, oracle_mod, data, metrics, k, cumulative=False, label="", product_kw=None, oracle_kw=None, **cmp_kw):
    res = pu.run_product(rb, data, metrics, k, cumulative=cumulative, **(product_kw or {}))
    orc = pu.run_oracle(oracle_mod, data, metrics, k, cumulative=cumulative, **(oracle_kw or {}))
    rep = pu.compare(res, orc, data, metrics, k, cumulative=cumulative, label=label, **cmp_kw)
    rep["timing"] = res.timing
    _log(rep)
    return res, orc, rep


# ---------------------------------------------------------------- BASELINE configurations
def test_cfg1_full_all_metrics(rb, oracle_mod):
    """configs[0]: 6,040 x 3,706, p=32, f32, K=10, all ten metrics -- at full size."""
    d = synth.make(1)
    _check(rb, oracle_mod, d, synth.ALL10, 10, label="cfg1 full")


def test_cfg1_full_cumulative(rb, oracle_mod):
    d = synth.make(1)
    _check(rb, oracle_mod, d, ("p", "tp", "r", "ap", "tap", "ndcg", "hit", "rr"), 10, cumulative=True, label="cfg1 full cumulative")


def test_cfg2_shape_item_biases(rb, oracle_mod):
    """configs[1] shape: p=64 + item_biases, K=10, P/R/AP/NDCG.  Biases go in as a separate vector
    (fused add) on the product side, folded into the factors on the oracle side (reference way)."""
    d = synth.make(2, m=4000, n=6000)
    _check(rb, oracle_mod, d, ("p", "r", "ap", "ndcg"), 10, label="cfg2 4000x6000 separate bias")
    # and through the plain drop-in signature (bias folded by the caller: p' = 65, not a multiple of 16)
    _check(rb, oracle_mod, d, ("p", "r", "ap", "ndcg"), 10, label="cfg2 4000x6000 folded bias",
           product_kw=dict(separate_bias=False))


def test_cfg3_shape_auc(rb, oracle_mod):
    """configs[2] shape: p=128, K=20, P/R/AP/NDCG + ROC-AUC + PR-AUC (full-rank counting)."""
    d = synth.make(3, m=1500, n=20000)
    _check(rb, oracle_mod, d, ("p", "r", "ap", "ndcg", "roc", "pr"), 20, label="cfg3 1500x20000")


def test_cfg4_shape_k100(rb, oracle_mod):
    """configs[3] shape: p=128, K=100, P/R/AP/NDCG."""
    d = synth.make(4, m=1200, n=40000)
    _check(rb, oracle_mod, d, ("p", "r", "ap", "ndcg"), 100, label="cfg4 1200x40000")


def test_cfg5_shape_f64_cumulative(rb, oracle_mod):
    """configs[4] shape: float64, p=64, cumulative K=1..50 AP/NDCG, min_pos_test=2 (clamped like the
    reference, quirk Q1), 2% cold-start users."""
    d = synth.make(5, m=2500, n=12000)
    _check(rb, oracle_mod, d, ("ap", "ndcg"), 50, cumulative=True, label="cfg5 2500x12000 f64",
           product_kw=dict(min_pos_test=2), oracle_kw=dict(min_pos_test=2))


def test_f64_all_metrics_with_auc(rb, oracle_mod):
    d = synth.make(1, m=1500, n=2500)
    d["A"] = d["A"].astype(np.float64)
    d["B"] = d["B"].astype(np.float64)
    res, orc, rep = _check(rb, oracle_mod, d, synth.ALL10, 10, label="f64 all metrics 1500x2500")
    # in float64 the accumulation-order differences are ~1e-15: everything is in fact identical
    assert rep["topk_rows_differing"] == 0


# ---------------------------------------------------------------- BASELINE catalogue sizes (full n, a block of the users)
def test_full_catalogue_cfg4_1m_items(rb, oracle_mod):
    """configs[3] at its full catalogue (1,000,000 items, p=128, K=100): a block of users against the oracle, and the
    tensor-core path (sampled guess, 7813 item tiles per CTA) against the FMA path bit for bit on a larger block."""
    d = synth.make(4, m=96, n=1_000_000)
    _check(rb, oracle_mod, d, ("p", "r", "ap", "ndcg"), 100, label="cfg4 96x1000000 (full catalogue)")
    d = synth.make(4, m=2048, n=1_000_000)
    out = {}
    for path in ("fma", "tensor"):
        out[path] = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], k=100, precision=True, recall=True,
                                            average_precision=True, ndcg=True, break_ties_with_noise=False, return_topk=True,
                                            return_status=True, scoring_path=path)
    a, b = out["fma"], out["tensor"]
    assert b.timing["scoring_path"] == 2 and b.timing["filter_fallback_batches"] == 0
    assert np.array_equal(a.status, b.status)
    assert np.array_equal(a.topk_items, b.topk_items)
    assert np.array_equal(a.topk_scores, b.topk_scores, equal_nan=True)
    for key in ("P@K", "R@K", "AP@K", "NDCG@K"):
        assert np.array_equal(a.metrics[key], b.metrics[key], equal_nan=True), key
    # size-independent properties of the rows: hits are integers within [0, min(K, npos)], ids unique and scores sorted
    npos = np.diff(d["X_test"].indptr)
    ok = b.status == 0
    hits = b.metrics["P@K"][ok].astype(np.float64) * 100
    assert np.all(np.abs(hits - np.rint(hits)) < 1e-4) and np.all(np.rint(hits) <= np.minimum(100, npos[ok]))
    assert np.allclose(np.rint(hits) / npos[ok], b.metrics["R@K"][ok], atol=1e-6)
    ts = b.topk_scores[ok]
    assert np.all(ts[:, :-1] >= ts[:, 1:])
    ti = np.sort(b.topk_items[ok], axis=1)
    assert np.all(ti[:, :-1] != ti[:, 1:])


def test_full_catalogue_cfg3_auc_and_cfg5_f64(rb, oracle_mod):
    """configs[2] (160,112 items, K=20 + ROC/PR-AUC rank counting) and configs[4] (float64, 300,000 items, cumulative
    K=1..50, min_pos_test=2, cold users) at their full catalogue sizes, a block of users each, against the oracle."""
    d = synth.make(3, m=400)
    assert d["B"].shape[0] == 160112
    _check(rb, oracle_mod, d, ("p", "r", "ap", "ndcg", "roc", "pr"), 20, label="cfg3 400x160112 (full catalogue)")
    d = synth.make(5, m=600)
    assert d["B"].shape[0] == 300000 and d["B"].dtype == np.float64
    _check(rb, oracle_mod, d, ("ap", "ndcg"), 50, cumulative=True, label="cfg5 600x300000 f64 (full catalogue)",
           product_kw=dict(min_pos_test=2), oracle_kw=dict(min_pos_test=2))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("cumulative", [False, True])
def test_metric_rows_long_walks_ties_and_negative_gains(rb, oracle_mod, dtype, cumulative):
    """user_metrics_kernel is a warp per user that splits walks and held-out rows into chunks of 32: K = 100 (walk and
    IDCG longer than a chunk), rows with up to a few hundred held-out items, gains with many ties, zeros and negative
    values (hpp:906-913, :938), users whose gains are all <= 0 (NaN, hpp:875-887) -- against the oracle, all eight
    top-K metrics."""
    d = synth.make(1, m=1200, n=3000, p=16)
    rng = np.random.default_rng(7)
    Xte = d["X_test"].copy()
    vals = rng.integers(-2, 6, size=Xte.data.shape[0]).astype(dtype)
    for u in range(0, 1200, 97):                                      # some users: nothing positive
        vals[Xte.indptr[u]:Xte.indptr[u + 1]] = -np.abs(vals[Xte.indptr[u]:Xte.indptr[u + 1]])
    Xte.data = vals
    d["X_test"] = Xte
    d["A"], d["B"] = d["A"].astype(dtype), d["B"].astype(dtype)
    assert np.diff(Xte.indptr).max() > 100
    res, orc, rep = _check(rb, oracle_mod, d, ("p", "tp", "r", "ap", "tap", "ndcg", "hit", "rr"), 100, cumulative=cumulative,
                           label="long walks / ties / negative gains %s cum=%d" % (np.dtype(dtype).name, cumulative))
    nd = res.metrics["NDCG@K"]
    assert np.isnan(nd).any() and np.isfinite(nd).any()


# ---------------------------------------------------------------- golden vectors of the reference
@pytest.mark.parametrize("name", case_names())
def test_golden_vectors(rb, name, scoring_path):
    c = load_case(name)
    res = pu.run_product(rb, c, c["metrics"], c["k"], cumulative=c["cumulative"], extras=True, **c["params"])
    S64 = pu.scores_f64(c["A"], c["B"])
    topk_amb, rank_amb, _ = pu.ambiguity(S64, c["X_train"], c["X_test"], c["k"])
    # exact ties in the scores (hand-made cases): without the tie-breaking noise the reference's order there is libstdc++'s.
    # With it (g_noise_* cases) the per-user mt19937 stream decides, and the tensor path's exact stage reproduces it: the
    # ranked top-K must then match exactly.  The rank counts (ROC/PR-AUC) and the all-FMA path use the scores without
    # noise (DESIGN.md): ties stay set aside there.
    noise_exact = bool(c["params"].get("break_ties_with_noise")) and scoring_path == "auto"
    for u in range(S64.shape[0]):
        s = np.sort(S64[u])
        if np.any(np.diff(s) == 0):
            rank_amb[u] = True
            if not noise_exact:
                topk_amb[u] = True
    if noise_exact:
        assert res.timing["scoring_path"] == 2
    for q in c["metrics"]:
        if q in ("hit", "rr") and not any(x in c["metrics"] for x in ("p", "tp", "r", "ap", "tap", "ndcg")):
            continue   # reference returns uninitialised memory there (quirk Q2)
        if q == "pr" and "roc" not in c["metrics"]:
            continue   # reference walks a partially sorted list there (quirk Q3)
        g, o = res.metrics[pu.KEY[q]], c["ref"][q]
        ok = pu.nan_equal_close(g, o, pu.METRIC_TOL)
        if ok.ndim == 2:
            ok = ok.all(axis=1)
        amb = rank_amb if q in ("roc", "pr") else topk_amb
        assert (ok | amb).all(), f"{name}: {q}: {np.asarray(g)[~ok & ~amb][:4]} vs {np.asarray(o)[~ok & ~amb][:4]}"


# ---------------------------------------------------------------- edge cases
def _tiny(n=10, scores=None, te=(2, 3, 7), vals=(1, 2, 3), tr=(), dtype=np.float64):
    A = np.ones((1, 1), dtype=dtype)
    B = np.asarray(scores, dtype=dtype).reshape(n, 1)
    Xtr = csr_array((np.ones(len(tr)), np.array(tr, dtype=np.int32), np.array([0, len(tr)], dtype=np.int32)), shape=(1, n))
    Xte = csr_array((np.array(vals, dtype=dtype), np.array(te, dtype=np.int32), np.array([0, len(te)], dtype=np.int32)), shape=(1, n))
    return dict(A=A, B=B, X_train=Xtr, X_test=Xte, item_biases=None)


def test_reference_r_tests_invalid_cases(rb):
    """tests/testthat/test-ndcg.R:7-35: constant / NaN / Inf scores give NaN."""
    for scores in ([0.0] * 10, [1.0] * 10, [np.nan] * 10, [np.inf] * 10):
        d = _tiny(scores=scores)
        r = rb.calc_reco_metrics(d["X_train"], d["X_test"], d["A"], d["B"], k=5, precision=False, average_precision=False,
                                 ndcg=True, as_df=False, break_ties_with_noise=False)
        assert np.isnan(r["NDCG@K"][0]), scores
    rng = np.random.default_rng(1)
    s = rng.standard_normal(10)
    s2 = s.copy(); s2[1] = np.nan; s2[3] = np.nan
    s3 = s.copy(); s3[1] = -np.inf; s3[3] = np.inf
    for scores in (s2, s3):
        d = _tiny(scores=scores)
        r = rb.calc_reco_metrics(d["X_train"], d["X_test"], d["A"], d["B"], k=5, precision=False, average_precision=False,
                                 ndcg=True, as_df=False, break_ties_with_noise=False)
        assert np.isnan(r["NDCG@K"][0])


def test_reference_r_tests_auc(rb):
    """tests/testthat/test-auc.R:22-61: perfect ranking -> ROC=PR=1; inverted -> ROC=0; random -> ~0.5."""
    rng = np.random.default_rng(1)
    n, npos = 100, 20
    pos = np.sort(rng.choice(n, npos, replace=False))
    for sign, want in ((1.0, 1.0), (-1.0, 0.0)):
        B = np.full((n, 2), -100.0 * sign)
        B[pos] = 100.0 * sign
        B += rng.standard_normal(B.shape)
        A = np.ones((1, 2))
        Xte = csr_array((np.ones(npos), pos.astype(np.int32), np.array([0, npos], dtype=np.int32)), shape=(1, n))
        r = rb.calc_reco_metrics(None, Xte, A, B, k=10, precision=False, average_precision=False, ndcg=False,
                                 roc_auc=True, pr_auc=True, as_df=False, break_ties_with_noise=False)
        assert r["ROC_AUC"][0] == want
        if want == 1.0:
            assert r["PR_AUC"][0] == 1.0
    m, n, k = 400, 20, 3
    A = rng.standard_normal((m, k)).astype(np.float32)
    B = rng.standard_normal((n, k)).astype(np.float32)
    X = (rng.random((m, n)) < 0.1).astype(np.float32)
    r = rb.calc_reco_metrics(None, csr_array(X), A, B, k=3, precision=False, average_precision=False, ndcg=False,
                             roc_auc=True, as_df=False, break_ties_with_noise=False)
    assert abs(np.nanmean(r["ROC_AUC"]) - 0.5) < 0.03


@pytest.mark.parametrize("k", [1, 2, 31, 32, 33, 64, 128, 129, 200, 384])
def test_k_sweep_selection_boundaries(rb, oracle_mod, k):
    """K across the selection-buffer boundaries (32-lane groups; C=256 up to K=128, C=512 above)."""
    d = synth.make(4, m=300, n=3000, p=24)
    # (top-384 of 3000 items: neighbours are dense, many users sit on a near-tie somewhere in the list;
    #  the comparator then requires the lists to differ ONLY at float64-near-tied positions)
    _check(rb, oracle_mod, d, ("p", "tp", "r", "ap", "tap", "ndcg", "hit", "rr"), k, label=f"k sweep K={k}", max_amb_frac=1.0)


@pytest.mark.parametrize("p", [1, 3, 15, 16, 17, 33, 100])
def test_factor_counts_not_multiple_of_tile(rb, oracle_mod, p):
    d = synth.make(1, m=260, n=700, p=p)
    _check(rb, oracle_mod, d, ("p", "ap", "ndcg", "roc", "pr"), 7, label=f"p={p}", max_amb_frac=0.6 if p < 3 else 0.25)


@pytest.mark.parametrize("m,n", [(1, 130), (127, 128), (129, 127), (257, 1000), (5, 11)])
def test_ragged_shapes(rb, oracle_mod, m, n):
    d = synth.make(1, m=m, n=n, p=8)
    k = min(5, n // 3)
    _check(rb, oracle_mod, d, synth.ALL10, k, label=f"ragged {m}x{n}", max_amb_frac=1.0)


def test_no_train_matrix_and_cold_start_rule(rb, oracle_mod):
    d = synth.make(1, m=500, n=800, p=8)
    # X_train=None => empty train, cold start forced on (reference __init__.py:471-473)
    r = rb.calc_reco_metrics(None, d["X_test"], d["A"], d["B"], k=5, as_df=False, break_ties_with_noise=False)
    empty = csr_array(d["X_test"].shape, dtype=np.float32)
    o = oracle_mod.oracle_calc(d["A"], d["B"], empty, d["X_test"], 5, metrics=("p", "ap", "ndcg"))
    assert pu.nan_equal_close(r["P@K"], o["p"], 1e-6).all()
    # consider_cold_start=False: users without train rows are NaN (hpp:446)
    Xtr = d["X_train"].copy().tolil()
    Xtr[:50] = 0
    Xtr = Xtr.tocsr(); Xtr.eliminate_zeros()
    d2 = dict(d, X_train=csr_array(Xtr))
    _check(rb, oracle_mod, d2, ("p", "ap", "ndcg", "roc"), 5, label="no cold start",
           product_kw=dict(consider_cold_start=False), oracle_kw=dict(consider_cold_start=False))


def test_quirks_eligibility_rules(rb, oracle_mod):
    """SURVEY App. B: Q1 (min_pos_test clamp), Q4 (frozen cumulative NDCG), Q6 (cand == K), only_ndcg,
    min_items_pool -- against the oracle restatement (itself pinned to the reference on the same cases)."""
    c = load_case("g_edge_f64_all")
    for cum in (False, True):
        for k in (5, 7):
            _check(rb, oracle_mod, c, synth.ALL10, k, cumulative=cum, label=f"edge cases k={k} cum={cum}", max_amb_frac=1.0)
    # Q1: min_pos_test > 1 is ignored by default, honoured with strict_min_pos_test
    d = synth.make(1, m=400, n=600, p=8)
    a = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], k=5, min_pos_test=1, break_ties_with_noise=False)
    b = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], k=5, min_pos_test=30, break_ties_with_noise=False)
    c2 = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], k=5, min_pos_test=30, strict_min_pos_test=True,
                                 break_ties_with_noise=False)
    assert pu.nan_equal_close(a.metrics["P@K"], b.metrics["P@K"], 0).all()
    npos = np.diff(d["X_test"].indptr)
    assert np.isnan(c2.metrics["P@K"][npos < 30]).all() and not np.isnan(c2.metrics["P@K"][npos >= 30]).any()


def test_hit_rr_alone_are_computed(rb, oracle_mod):
    """Quirk Q2: the reference leaves Hit@K / RR@K uninitialised when requested alone; here they are
    computed and equal the values of an all-metrics call."""
    d = synth.make(1, m=300, n=500, p=8)
    a = rb.calc_reco_metrics(d["X_train"], d["X_test"], d["A"], d["B"], k=5, precision=False, average_precision=False,
                             ndcg=False, hit=True, rr=True, as_df=False, break_ties_with_noise=False)
    b = rb.calc_reco_metrics(d["X_train"], d["X_test"], d["A"], d["B"], k=5, all_metrics=True, as_df=False,
                             break_ties_with_noise=False)
    assert pu.nan_equal_close(a["Hit@K"], b["Hit@K"], 0).all() and pu.nan_equal_close(a["RR@K"], b["RR@K"], 0).all()


def test_strided_factors_and_dataframe_output(rb, oracle_mod):
    """lda/ldb > k (row-strided views, reference _as_row_major :11-16) and the DataFrame packaging."""
    d = synth.make(1, m=200, n=300, p=8)
    Abig = np.zeros((200, 13), dtype=np.float32); Abig[:, :8] = d["A"]
    Bbig = np.zeros((300, 11), dtype=np.float32); Bbig[:, :8] = d["B"]
    df = rb.calc_reco_metrics(d["X_train"], d["X_test"], Abig[:, :8], Bbig[:, :8], k=5, break_ties_with_noise=False)
    assert list(df.columns) == ["P@5", "AP@5", "NDCG@5"] and df.shape[0] == 200
    o = oracle_mod.oracle_calc(d["A"], d["B"], d["X_train"], d["X_test"], 5, metrics=("p", "ap", "ndcg"))
    assert pu.nan_equal_close(df["P@5"].to_numpy(), o["p"], 1e-6).all()
    dfc = rb.calc_reco_metrics(d["X_train"], d["X_test"], d["A"], d["B"], k=3, cumulative=True, break_ties_with_noise=False)
    assert list(dfc.columns)[:3] == ["P@1", "P@2", "P@3"]


def test_non_personalised_model_biases_only(rb, oracle_mod):
    """A=B=None: score = item bias (reference __init__.py:429-436)."""
    d = synth.make(2, m=300, n=500, p=4)
    bias = d["item_biases"].astype(np.float64)
    r = rb.calc_reco_metrics(d["X_train"], d["X_test"], None, None, k=5, item_biases=bias, as_df=False,
                             break_ties_with_noise=False)
    o = oracle_mod.oracle_calc(np.ones((300, 1)), bias.reshape(-1, 1), d["X_train"], d["X_test"], 5,
                               metrics=("p", "ap", "ndcg"), dtype=np.float64)
    assert pu.nan_equal_close(r["P@K"], o["p"], 1e-6).all() and pu.nan_equal_close(r["NDCG@K"], o["ndcg"], 1e-6).all()


# ---------------------------------------------------------------- sharding / residency
def test_user_range_shards_equal_full_call(rb):
    """The multi-GPU unit: evaluating [0,h) and [h,m) separately writes the same rows as one call."""
    d = synth.make(3, m=900, n=3000, p=32)
    kw = dict(k=20, all_metrics=True, break_ties_with_noise=False, return_topk=True, return_ranks=True)
    full = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], **kw)
    h = 389
    lo = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], user_range=(0, h), **kw)
    hi = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], user_range=(h, 900), **kw)
    for key, v in full.metrics.items():
        if key == "K":
            continue
        assert pu.nan_equal_close(v[:h], lo.metrics[key][:h], 0).all(), key
        assert pu.nan_equal_close(v[h:], hi.metrics[key][h:], 0).all(), key
        assert np.isnan(lo.metrics[key][h:]).all()
    assert (full.topk_items[:h] == lo.topk_items[:h]).all() and (full.topk_items[h:] == hi.topk_items[h:]).all()
    split = d["X_test"].indptr[h]
    assert (full.pos_rank[:split] == lo.pos_rank[:split]).all() and (full.pos_rank[split:] == hi.pos_rank[split:]).all()


def test_small_batches_equal_single_batch(rb, monkeypatch):
    """User batches are an implementation detail: forcing 128-user batches changes nothing."""
    d = synth.make(1, m=700, n=900, p=16)
    kw = dict(k=10, all_metrics=True, break_ties_with_noise=False)
    a = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], **kw)
    monkeypatch.setenv("RMB200_BATCH_USERS", "128")
    b = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], **kw)
    for key, v in a.metrics.items():
        if key != "K":
            assert pu.nan_equal_close(v, b.metrics[key], 0).all(), key
    assert b.timing["kernel_launches"] > a.timing["kernel_launches"]


def test_device_resident_call_equals_host_call(rb):
    """inputs_on_device=1 (HBM-resident inputs and outputs, what bench.py's `value` times) gives
    bit-identical results to the host-pointer call."""
    import torch
    from recometrics_b200 import _capi
    d = synth.make(2, m=1000, n=2000)
    A, B, bias = d["A"], d["B"], d["item_biases"]
    Xtr, Xte = d["X_train"], d["X_test"]
    host = rb.calc_reco_metrics_ex(Xtr, Xte, A, B, k=10, item_biases=bias, recall=True, break_ties_with_noise=False)
    dev = torch.device("cuda", 0)
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    tA, tB, tb = t(A), t(B), t(bias)
    trp, tri, tep, tei, tev = t(Xtr.indptr), t(Xtr.indices), t(Xte.indptr), t(Xte.indices), t(Xte.data.astype(np.float32))
    m, n, p = A.shape[0], B.shape[0], A.shape[1]
    outs = {q: torch.empty(m, dtype=torch.float32, device=dev) for q in ("p", "r", "ap", "ndcg")}
    ex = _capi.make_extra(device=0, inputs_on_device=True)
    rc = _capi.calc_metrics(np.float32, tA.data_ptr(), p, tB.data_ptr(), p, m, n, p, trp.data_ptr(), tri.data_ptr(),
                            tep.data_ptr(), tei.data_ptr(), tev.data_ptr(), 10, False, False,
                            {q: v.data_ptr() for q, v in outs.items()}, True, 2, 1, item_biases=tb.data_ptr(), extra=ex)
    _capi.raise_for_status(rc)
    torch.cuda.synchronize()
    for q, key in (("p", "P@K"), ("r", "R@K"), ("ap", "AP@K"), ("ndcg", "NDCG@K")):
        assert pu.nan_equal_close(outs[q].cpu().numpy(), host.metrics[key], 0).all(), q


def test_device_front_end_torch_tensors(rb, oracle_mod):
    """calc_reco_metrics_device: factors as torch CUDA tensors (one of them a row-strided view), CSR matrices either
    scipy (uploaded) or DeviceCSR (resident); rows come back as CUDA tensors and equal the host front-end's bit for bit."""
    import torch
    dev = torch.device("cuda", 0)
    for cfg_id, m, n, k, cum, dtype in ((2, 700, 5000, 10, False, np.float32), (5, 500, 4000, 20, True, np.float64)):
        d = synth.make(cfg_id, m=m, n=n)
        A, B = d["A"].astype(dtype), d["B"].astype(dtype)
        kw = dict(k=k, precision=True, recall=True, average_precision=True, ndcg=True, hit=True, cumulative=cum,
                  break_ties_with_noise=False, return_topk=True, return_status=True, return_means=True)
        host = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], A, B, item_biases=d["item_biases"], **kw)
        tA = torch.from_numpy(A).to(dev)
        wide = torch.zeros(n, A.shape[1] + 5, dtype=tA.dtype, device=dev)
        wide[:, :A.shape[1]] = torch.from_numpy(B).to(dev)
        tB = wide[:, :A.shape[1]]                                       # row stride p + 5
        tb = None if d["item_biases"] is None else torch.from_numpy(d["item_biases"].astype(dtype)).to(dev)
        Xtr = rb.DeviceCSR.from_scipy(d["X_train"], 0, dtype, with_data=False)
        Xte = rb.DeviceCSR.from_scipy(d["X_test"], 0, dtype)
        for xtr, xte in ((d["X_train"], d["X_test"]), (Xtr, Xte)):
            r = rb.calc_reco_metrics_device(xtr, xte, tA, tB, item_biases=tb, **kw)
            assert r.timing["h2d_bytes"] == 0 and r.timing["d2h_bytes"] == 0
            assert np.array_equal(host.status, r.status.cpu().numpy())
            assert np.array_equal(host.topk_items, r.topk_items.cpu().numpy())
            for key, v in host.metrics.items():
                if key == "K":
                    continue
                assert r.metrics[key].is_cuda and tuple(r.metrics[key].shape) == v.shape
                assert np.array_equal(v, r.metrics[key].cpu().numpy(), equal_nan=True), key
                assert np.array_equal(np.asarray(host.means[key]), np.asarray(r.means[key]), equal_nan=True), key
    with pytest.raises(TypeError):
        rb.calc_reco_metrics_device(d["X_train"], d["X_test"], A, B, k=5)        # numpy factors: use calc_reco_metrics


def test_cpp_shim_computes_on_the_gpu(rb, tmp_path):
    """The C++ drop-in layer (include/recometrics_b200_shim.hpp: the reference's calc_metrics_float / _double / template
    names) built with g++ and linked against the library: on a GPU box the calls compute (known answers checked inside
    tests/shim/shim_dropin.cpp) instead of throwing."""
    import test_capi_host
    assert rb.device_count() > 0
    test_capi_host.test_cpp_shim_is_a_drop_in_for_the_reference_declarations(tmp_path)


def test_pageable_upload_pipeline_equals_plain_copies(rb, monkeypatch):
    """Host inputs in ordinary (pageable) numpy memory go up through copy threads and pinned bounce buffers once they are
    large (runtime.cu upload_rows); forced on for every array here -- pitched factor matrices, the contiguous CSR arrays,
    several user batches (two alternating staging buffers on the prefetch stream) -- the results must be those of the
    plain cudaMemcpy path, bit for bit."""
    d = synth.make(3, m=5000, n=6000, p=40)
    Abig = np.zeros((5000, 47), dtype=np.float32)
    Abig[:, :40] = d["A"]
    A = Abig[:, :40]                                                    # row pitch 47 floats
    kw = dict(k=20, all_metrics=True, break_ties_with_noise=False, return_topk=True, return_ranks=True)
    monkeypatch.setenv("RMB200_BATCH_USERS", "1024")
    monkeypatch.setenv("RMB200_UPLOAD_THREADS", "0")
    plain = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], A, d["B"], **kw)
    monkeypatch.setenv("RMB200_UPLOAD_THREADS", "3")
    monkeypatch.setenv("RMB200_UPLOAD_MIN_BYTES", "1")
    piped = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], A, d["B"], **kw)
    for key, v in plain.metrics.items():
        if key != "K":
            assert np.array_equal(v, piped.metrics[key], equal_nan=True), key
    assert np.array_equal(plain.topk_items, piped.topk_items) and np.array_equal(plain.pos_rank, piped.pos_rank)
    assert plain.timing["h2d_bytes"] == piped.timing["h2d_bytes"]


def test_reference_cython_wrapper_computes_on_the_gpu(rb, tmp_path):
    """The reference's unmodified Cython wrapper built against the library (oracle/build_ref_cython.py; the compiled module
    travels in oracle/_ref/cy_b200): its cpp_funs.calc_reco_metrics returns, on the GPU, the rows of this package's own
    front-end bit for bit."""
    import test_capi_host
    stdout, path = test_capi_host.run_reference_cython_wrapper(tmp_path)
    assert "HAS 1" in stdout and "COMPUTED" in stdout, stdout
    rows = np.load(path)
    d = synth.make(1, m=300, n=500, p=8)
    r = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], k=5, precision=True, average_precision=True, ndcg=True,
                                break_ties_with_noise=False)
    for i, key in enumerate(("P@K", "AP@K", "NDCG@K")):
        assert np.array_equal(rows[i], r.metrics[key], equal_nan=True), key


_SIGINT_PROBE = r"""
import os, signal, sys, threading, time
sys.path.insert(0, sys.argv[1])
import numpy as np
import recometrics_b200 as rb
from tools import synth
d = synth.make(3, m=200000, n=60000)
rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], k=20, roc_auc=True, break_ties_with_noise=False,
                        user_range=(0, 2000))                                   # warm-up (library load, workspace)
def fire():
    time.sleep(1.0)
    os.kill(os.getpid(), signal.SIGINT)
t0 = time.time()
threading.Thread(target=fire, daemon=True).start()
calls = 0
try:
    for i in range(200):                                                         # ~0.3 s per call: a minute if nothing stops it
        rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], k=20, roc_auc=True, break_ties_with_noise=False)
        calls += 1
    print("COMPLETED", calls)
except (KeyboardInterrupt, RuntimeError) as e:
    print("INTERRUPTED", type(e).__name__, str(e)[:60].replace("\n", " "), "after %.2f s and %d calls" % (time.time() - t0, calls))
# the handler was put back: the library is usable afterwards and a later Ctrl-C would reach Python again
assert signal.getsignal(signal.SIGINT) is signal.default_int_handler
r = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], k=20, roc_auc=True, break_ties_with_noise=False,
                            user_range=(0, 2000))
print("AFTER", int(np.isfinite(r.metrics["ROC_AUC"][:2000]).sum() > 0))
"""


def test_sigint_stops_the_call_between_user_batches():
    """Ctrl-C (reference: SignalSwitcher, src/recometrics.hpp:114-174 -- drain the loop, restore the handler, re-raise, throw):
    a SIGINT sent while calls are running ends them within a batch or two with KeyboardInterrupt / "procedure was
    interrupted", the previous handler is back in place, and the library keeps working.  The probe process inherits
    RMB200_PATH from the scoring_path fixture: it runs once with the library's choice and once with RMB200_PATH=fma."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    run = subprocess.run([sys.executable, "-c", _SIGINT_PROBE, root], capture_output=True, text=True, timeout=600)
    assert run.returncode == 0, run.stdout + run.stderr
    line = [ln for ln in run.stdout.splitlines() if ln.startswith("INTERRUPTED")]
    assert line, run.stdout + run.stderr
    secs = float(line[0].split("after ")[1].split(" s")[0])
    assert 0.9 <= secs < 6.0, line[0]
    assert "AFTER 1" in run.stdout, run.stdout + run.stderr


def test_unsupported_requests_fail_loudly(rb):
    """k_metrics beyond the selection kernels' buffers is computed (full-order path, tests/test_gpu_full_order.py) unless
    the caller insists on a selection path."""
    d = synth.make(1, m=100, n=900, p=8)
    df = rb.calc_reco_metrics(d["X_train"], d["X_test"], d["A"], d["B"], k=500, break_ties_with_noise=False)
    assert df.shape[0] == 100
    with pytest.raises(NotImplementedError):
        rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], k=500, break_ties_with_noise=False, scoring_path="tensor")


def test_tensor_filter_path_equals_fma_path_bit_for_bit(rb):
    """The tensor-core path only decides which scores get looked at: ranked ids and scores must be the FMA path's."""
    for cfg_id, m, n, k, dtype in ((4, 700, 30000, 100, np.float32), (2, 900, 9000, 10, np.float32), (5, 600, 8000, 50, np.float64)):
        d = synth.make(cfg_id, m=m, n=n)
        A, B = d["A"].astype(dtype), d["B"].astype(dtype)
        out = {}
        for path in ("fma", "tensor"):
            r = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], A, B, k=k, item_biases=d["item_biases"], precision=True,
                                        average_precision=True, ndcg=True, break_ties_with_noise=False, return_topk=True,
                                        return_status=True, scoring_path=path)
            assert r.timing["scoring_path"] == (1 if path == "fma" else 2)
            out[path] = r
        a, b = out["fma"], out["tensor"]
        assert np.array_equal(a.status, b.status)
        assert np.array_equal(a.topk_items, b.topk_items)
        assert np.array_equal(a.topk_scores, b.topk_scores, equal_nan=True)
        for key in ("P@K", "AP@K", "NDCG@K"):
            assert np.array_equal(a.metrics[key], b.metrics[key], equal_nan=True)


def test_tensor_path_refuses_rank_counting(rb):
    d = synth.make(1, m=200, n=500)
    with pytest.raises(NotImplementedError):
        rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], k=5, roc_auc=True, break_ties_with_noise=False,
                                scoring_path="tensor")


def test_sampled_threshold_guess_and_retry_pass(rb, monkeypatch):
    """Catalogues of >= 64K items start the filter's thresholds from a sampled guess (filter_select.cuh pass 0) and
    verify it; a deliberately hopeless guess (the best item of the sample) sends rows through the retry pass.
    Either way the ranked ids and scores are the FMA path's, bit for bit."""
    d = synth.make(4, m=300, n=70000)
    kw = dict(k=100, precision=True, recall=True, average_precision=True, ndcg=True, break_ties_with_noise=False,
              return_topk=True, return_status=True)
    monkeypatch.delenv("RMB200_SAMPLE_RANK", raising=False)
    ref = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], scoring_path="fma", **kw)
    for rank, d64 in ((None, False), ("1", False), ("1", True)):
        if rank is None:
            monkeypatch.delenv("RMB200_SAMPLE_RANK", raising=False)
        else:
            monkeypatch.setenv("RMB200_SAMPLE_RANK", rank)
        A, B = (d["A"].astype(np.float64), d["B"].astype(np.float64)) if d64 else (d["A"], d["B"])
        want = ref if not d64 else rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], A, B, scoring_path="fma", **kw)
        r = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], A, B, scoring_path="tensor", **kw)
        assert r.timing["scoring_path"] == 2 and r.timing["filter_fallback_batches"] == 0
        if rank == "1":
            assert r.timing["filter_retry_rows"] > 0
        assert np.array_equal(want.status, r.status)
        assert np.array_equal(want.topk_items, r.topk_items)
        assert np.array_equal(want.topk_scores, r.topk_scores, equal_nan=True)
        for key in ("P@K", "R@K", "AP@K", "NDCG@K"):
            assert np.array_equal(want.metrics[key], r.metrics[key], equal_nan=True), key


@pytest.mark.parametrize("cumulative", [False, True])
def test_metric_means_on_device(rb, cumulative):
    """Extension (SURVEY 8f-2): per-metric means over users, reduced on the device, equal numpy.nanmean of the rows;
    means_only leaves the per-user rows on the device."""
    d = synth.make(1, m=1500, n=1200, p=16)
    kw = dict(k=7, all_metrics=True, break_ties_with_noise=False, cumulative=cumulative)
    r = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], return_means=True, **kw)
    assert set(r.means) == {k for k in r.metrics if k != "K"}
    for key, rows in r.metrics.items():
        if key == "K":
            continue
        rows = np.asarray(rows, dtype=np.float64)
        want_cnt = (~np.isnan(rows)).sum(axis=0)
        assert np.array_equal(np.asarray(r.counts[key]), want_cnt), key
        with np.errstate(invalid="ignore"):
            want = np.nansum(rows, axis=0) / want_cnt
        assert np.allclose(np.asarray(r.means[key]), want, rtol=1e-12, atol=0, equal_nan=True), key
    only = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], means_only=True, user_range=(100, 1400), **kw)
    assert list(only.metrics) == ["K"]
    sub = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], user_range=(100, 1400), **kw)
    for key, rows in sub.metrics.items():
        if key == "K":
            continue
        rows = np.asarray(rows, dtype=np.float64)[100:1400]
        with np.errstate(invalid="ignore"):
            want = np.nansum(rows, axis=0) / (~np.isnan(rows)).sum(axis=0)
        assert np.allclose(np.asarray(only.means[key]), want, rtol=1e-12, atol=0, equal_nan=True), key
    assert only.timing["d2h_bytes"] < sub.timing["d2h_bytes"] / 10


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_tie_breaking_noise_default_call(rb, oracle_mod, dtype):
    """break_ties_with_noise=True is the reference's default: same call through the oracle (which restates the per-user
    mt19937 noise, pinned against the compiled reference) -- top-K metrics of a default call, and all ten metrics."""
    d = synth.make(1, m=800, n=1500, p=16)
    A, B = d["A"].astype(dtype), d["B"].astype(dtype)
    df = rb.calc_reco_metrics(d["X_train"], d["X_test"], A, B, k=10, seed=123)          # every default, DataFrame out
    o = oracle_mod.oracle_calc(A, B, d["X_train"], d["X_test"], 10, metrics=("p", "ap", "ndcg"), nthreads=4, dtype=dtype,
                               break_ties_with_noise=True, seed=123, extras=True)
    S64 = pu.scores_f64(A, B)
    topk_amb, rank_amb, _ = pu.ambiguity(S64, d["X_train"], d["X_test"], 10)
    for q, col in (("p", "P@10"), ("ap", "AP@10"), ("ndcg", "NDCG@10")):
        ok = pu.nan_equal_close(df[col].to_numpy(), o[q], pu.METRIC_TOL)
        assert (ok | topk_amb).all(), q
    res = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], A, B, k=10, all_metrics=True, seed=5, return_status=True)
    o = oracle_mod.oracle_calc(A, B, d["X_train"], d["X_test"], 10, metrics=synth.ALL10, nthreads=4, dtype=dtype,
                               break_ties_with_noise=True, seed=5, extras=True)
    assert np.array_equal(res.status[~topk_amb], o["status"][~topk_amb])
    for q in synth.ALL10:
        ok = pu.nan_equal_close(res.metrics[pu.KEY[q]], o[q], pu.METRIC_TOL)
        amb = rank_amb if q in ("roc", "pr") else topk_amb
        assert (ok | amb).all(), q
