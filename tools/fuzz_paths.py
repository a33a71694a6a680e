"""Randomised differential test of the three scoring paths (GPU): random shapes, metric sets and flags; the FMA tiles, the
tensor-core filter (where it applies) and the full-order path must return identical status, ranked top-K ids / scores, held-out
ranks and metric rows (break_ties_with_noise off: all three rank equal scores by item id).  With the noise on, the automatic
path (filter + noise-reach hand-back) must equal the full-order path.  One case in ten carries NaN / inf factors or biases,
or factors whose scores overflow, in a few rows.  Usage: python tools/fuzz_paths.py [seconds] [seed]"""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import recometrics_b200 as rb          # noqa: E402
from tools import synth                # noqa: E402

budget = float(sys.argv[1]) if len(sys.argv) > 1 else 120.0
rng = np.random.default_rng(int(sys.argv[2]) if len(sys.argv) > 2 else 1)
FLAGS = ("precision", "trunc_precision", "recall", "average_precision", "trunc_average_precision", "ndcg", "hit", "rr", "roc_auc", "pr_auc")


def same(a, b, what):
    assert np.array_equal(a.status, b.status), what + ": status"
    assert np.array_equal(a.topk_items, b.topk_items), what + ": top-K ids"
    assert np.array_equal(a.topk_scores, b.topk_scores, equal_nan=True), what + ": top-K scores"
    if a.pos_rank is not None and b.pos_rank is not None:
        assert np.array_equal(a.pos_rank, b.pos_rank), what + ": ranks"
    for key, v in a.metrics.items():
        if key != "K":
            assert np.array_equal(v, b.metrics[key], equal_nan=True), what + ": " + key


t0, cases = time.time(), 0
while time.time() - t0 < budget:
    m = int(rng.integers(1, 2500))
    n = int(rng.choice([int(rng.integers(40, 600)), int(rng.integers(600, 9000)), int(rng.integers(33000, 70000))], p=[0.3, 0.5, 0.2]))
    p = int(rng.integers(1, 100))
    K = int(min(n - 1, rng.choice([1, 3, 10, 33, 100, 257, 390, 700])))
    dtype = np.float32 if rng.random() < 0.6 else np.float64
    d = synth.make(int(rng.integers(1, 6)), m=m, n=n, p=p)
    A, B = d["A"].astype(dtype), d["B"].astype(dtype)
    if rng.random() < 0.3:                       # integer-valued factors: exact ties everywhere
        A, B = np.rint(A), np.rint(B)
    if rng.random() < 0.2:
        A[rng.random(m) < 0.1] = 0               # users unseen in training
    bias = (0.5 * rng.standard_normal(n)).astype(dtype) if rng.random() < 0.3 else None
    bad = 0
    if rng.random() < 0.1:                       # non-finite or overflowing scores (tests/test_gpu_nonfinite.py N1-N5), a few rows
        bad = int(rng.integers(1, 6))
        items, users = rng.random(n) < 0.01, rng.random(m) < 0.03
        if bad == 1:
            B[items] = np.nan
        elif bad == 2:
            B[items, int(rng.integers(p))] = rng.choice([np.inf, -np.inf])
        elif bad == 3:
            bias = np.zeros(n, dtype=dtype) if bias is None else bias
            bias[items] = rng.choice([-np.inf, np.inf, np.nan], p=[0.8, 0.1, 0.1])
        elif bad == 4:
            A[users, int(rng.integers(p))] = rng.choice([np.nan, np.inf, -np.inf])
        elif dtype == np.float64:                # one product of a scaled user and a scaled item leaves the range
            A[users, -1] = 1e160 * rng.choice([-1.0, 1.0], int(users.sum()))
            B[items, -1] = 1e160
        else:                                    # ... with norms within ~1000x of each other (B * 1e18, ||a|| ~ 1e19, items ~4e21),
            B *= 1e18                            # which the filter could rank: every other score stays below ||a|| ||b|| < 1.7e38
            A[users] *= 5e17 / np.maximum(1.0, np.abs(A[users]).max(axis=1, keepdims=True))
            A[users, -1] = 1e19 * rng.choice([-1.0, 1.0], int(users.sum()))
            B[items, -1] = 4e21
    flags = {f: bool(rng.random() < 0.4) for f in FLAGS}
    if not any(flags[f] for f in ("precision", "average_precision", "ndcg")):      # (the reference's "at least one metric" guard, quirk Q7)
        flags["precision"] = True
    cumulative = bool(rng.random() < 0.3)
    noise = bool(rng.random() < 0.3)
    kw = dict(k=K, item_biases=bias, cumulative=cumulative, break_ties_with_noise=noise, seed=int(rng.integers(1, 1000)),
              return_topk=True, return_status=True, return_ranks=flags["roc_auc"] or flags["pr_auc"],
              min_pos_test=int(rng.integers(1, 3)), consider_cold_start=bool(rng.random() < 0.8), **flags)
    what = "m=%d n=%d p=%d K=%d %s cum=%d noise=%d bias=%d nonfinite=N%d flags=%s" % (
        m, n, p, K, np.dtype(dtype).name, cumulative, noise, bias is not None, bad, [f for f in FLAGS if flags[f]])
    try:
        full = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], A, B, scoring_path="full", **kw)
        auto = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], A, B, scoring_path="auto", **kw)
        same(full, auto, what + " [full vs auto, path %d]" % auto.timing["scoring_path"])
        if not noise and K <= 384:
            fma = rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], A, B, scoring_path="fma", **kw)
            same(full, fma, what + " [full vs fma]")
    except AssertionError as e:
        print("FUZZ MISMATCH:", e)
        sys.exit(1)
    cases += 1
print("fuzz_paths: %d random cases, all paths identical (%.0f s)" % (cases, time.time() - t0))
