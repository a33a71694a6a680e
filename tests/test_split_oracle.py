"""CPU: the splitter oracle (oracle/split_oracle.c) pinned against the committed golden outputs of the UNMODIFIED reference
(tests/golden/split_*.npz, made by tests/golden/make_golden_split.py) and, where oracle/_ref exists, against the reference
itself on fresh random inputs; and the HOST half of the product's splitters (rmb200_split_plan: the replay of the
reference's mt19937 stream, include/recometrics_b200.h) against the oracle -- the part of a split that needs no GPU."""
import hashlib
import os

import numpy as np
import pytest

from tools import split_cases

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def check_against_golden(name, flat):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    seen = set()
    for key in g.files:
        if key.startswith("len_"):
            continue
        if key.startswith("sha256_"):
            k = key[len("sha256_"):]
            assert flat[k].size == int(g["len_" + k][0]), f"{name}: {k} length"
            digest = np.frombuffer(hashlib.sha256(np.ascontiguousarray(flat[k]).tobytes()).digest(), dtype=np.uint8)
            assert np.array_equal(digest, g[key]), f"{name}: {k} differs from the reference (sha-256)"
        else:
            k = key
            assert flat[k].dtype == g[k].dtype and np.array_equal(flat[k], g[k]), f"{name}: {k} differs from the reference"
        seen.add(k)
    assert seen == set(flat), f"{name}: outputs {sorted(set(flat) ^ seen)} present on one side only"


@pytest.mark.parametrize("name", sorted(split_cases.CASES))
def test_oracle_matches_golden(oracle_mod, name):
    mk, kw = split_cases.CASES[name]
    p, i, v = split_cases.make_csr(**mk)
    check_against_golden(name, split_cases.flatten(oracle_mod.oracle_split(p, i, v, mk["m"], mk["n"], **kw)))


@pytest.mark.parametrize("name", sorted(split_cases.REFUSALS))
def test_oracle_refuses_what_the_reference_refuses(oracle_mod, name):
    mk, kw, message = split_cases.REFUSALS[name]
    p, i, v = split_cases.make_csr(**mk)
    with pytest.raises(RuntimeError, match=message):
        oracle_mod.oracle_split(p, i, v, mk["m"], mk["n"], **kw)
    if oracle_mod.have_ref():
        with pytest.raises(RuntimeError, match=message):
            oracle_mod.ref_split(p, i, v, mk["m"], mk["n"], **kw)


def test_oracle_satisfies_the_invariants_of_the_reference_r_tests(oracle_mod):
    """tests/testthat/test-split.R:7-93 of the reference, on the oracle: X_train + X_test == X[users_test, ], shapes, a fixed
    number of users, the error when no user can meet the criteria."""
    import scipy.sparse as sp

    def rsparse(m, n, density, seed):
        X = sp.random(m, n, density=density, format="csr", random_state=seed, dtype=np.float64)
        X.data = np.round(X.data * 10 + 1)
        X.sort_indices()
        return sp.csr_array(X)

    def mat(parts, n):
        p, i, v = parts
        return sp.csr_array((v, i, p), shape=(len(p) - 1, n))

    for n in (10000, 3):
        X = rsparse(1000, n, 0.01, 123)
        o = oracle_mod.oracle_split(X.indptr, X.indices, X.data, 1000, n, split_type="all", test_fraction=0.3)
        assert abs((mat(o["train"], n) + mat(o["test"], n)) - X).sum() == 0
    X = rsparse(1000, 10000, 0.01, 123)
    o = oracle_mod.oracle_split(X.indptr, X.indices, X.data, 1000, 10000, split_type="separated", n_users_test=100, test_fraction=0.3)
    ut = o["users_test"]
    assert len(ut) == 100 and abs((mat(o["train"], 10000) + mat(o["test"], 10000)) - X[ut, :]).sum() == 0
    assert mat(o["rem"], 10000).shape[0] == 900
    o = oracle_mod.oracle_split(X.indptr, X.indices, X.data, 1000, 10000, split_type="joined", n_users_test=100, test_fraction=0.3)
    tr, te = mat(o["train"], 10000), mat(o["test"], 10000)
    assert tr.shape[0] == 1000 and te.shape[0] == 100
    assert abs((tr[:100, :] + te) - X[o["users_test"], :]).sum() == 0
    X = rsparse(10, 9, 0.5, 123)
    o = oracle_mod.oracle_split(X.indptr, X.indices, X.data, 10, 9, split_type="separated", n_users_test=2, test_fraction=0.3)
    assert len(o["users_test"]) == 2 and len(o["rem"][0]) - 1 == 8
    X = rsparse(1000, 3, 0.01, 1)
    with pytest.raises(RuntimeError, match="No users satisfy criteria"):
        oracle_mod.oracle_split(X.indptr, X.indices, X.data, 1000, 3, split_type="separated", n_users_test=100, test_fraction=0.3, min_pos_test=2)


def _random_case(rs):
    m, n = int(rs.randint(2, 300)), int(rs.randint(3, 2000))
    dtype = np.float32 if rs.rand() < 0.5 else np.float64
    p, i, v = split_cases.make_csr(m, n, int(rs.randint(1 << 30)), mean_len=float(rs.choice([2.0, 8.0, 40.0])), dtype=dtype,
                                   unsorted=bool(rs.rand() < 0.3), empty_frac=float(rs.choice([0.0, 0.1, 0.5])))
    kw = dict(split_type=str(rs.choice(["all", "separated", "joined"])), n_users_test=int(rs.randint(0, m + 1)),
              test_fraction=float(rs.choice([0.1, 0.25, 0.3, 0.5, 0.7, 0.9])), consider_cold_start=bool(rs.rand() < 0.5),
              min_items_pool=int(rs.randint(0, 4)), min_pos_test=int(rs.randint(0, 3)), seed=int(rs.randint(0, 1 << 31)))
    return m, n, p, i, v, kw


def test_oracle_equals_the_compiled_reference_on_random_inputs(oracle_mod):
    if not oracle_mod.have_ref():
        pytest.skip("oracle/_ref not built here (the golden fixtures above carry the reference's outputs)")
    rs = np.random.RandomState(5)
    done = 0
    for _ in range(250):
        m, n, p, i, v, kw = _random_case(rs)
        try:
            r, er = oracle_mod.ref_split(p, i, v, m, n, **kw), None
        except RuntimeError as e:
            r, er = None, str(e)
        try:
            o, eo = oracle_mod.oracle_split(p, i, v, m, n, **kw), None
        except RuntimeError as e:
            o, eo = None, str(e)
        assert er == eo, (kw, er, eo)
        if r is None:
            continue
        fr, fo = split_cases.flatten(r), split_cases.flatten(o)
        assert set(fr) == set(fo)
        for k in fr:
            assert fr[k].shape == fo[k].shape and np.array_equal(fr[k], fo[k]), (kw, k)
        done += 1
    assert done > 150


# ---- the product's host half (no GPU) ----
def _held_from_oracle(o, p, i, m, kind):
    """One byte per entry of the split rows, from the oracle's matrices: an entry is held out iff its item is in the row's
    test part (item ids are unique inside a row in these inputs)."""
    rows = np.arange(m) if kind == "all" else o["users_test"]
    tep, tei = o["test"][0], o["test"][1]
    held = []
    for r, u in enumerate(rows):
        items = i[p[u]:p[u + 1]]
        held.append(np.isin(items, tei[tep[r]:tep[r + 1]]).astype(np.uint8))
    return np.concatenate(held) if held else np.zeros(0, np.uint8)


@pytest.mark.parametrize("name", sorted(split_cases.CASES))
def test_host_plan_of_the_product_matches_the_oracle(rb, oracle_mod, name):
    from recometrics_b200 import _capi
    mk, kw = split_cases.CASES[name]
    kw = dict(kw)
    p, i, v = split_cases.make_csr(**mk)
    kind = kw.pop("split_type")
    o = oracle_mod.oracle_split(p, i, v, mk["m"], mk["n"], split_type=kind, **kw)
    frac = float(np.float32(kw["test_fraction"])) if v.dtype == np.float32 else kw["test_fraction"]
    users, held = _capi.split_plan(p, mk["m"], mk["n"], kind != "all", **dict(kw, test_fraction=frac))
    if kind != "all":
        assert np.array_equal(users, o["users_test"])
    assert np.array_equal(held, _held_from_oracle(o, p, i, mk["m"], kind)), name


def test_host_plan_on_random_inputs(rb, oracle_mod):
    from recometrics_b200 import _capi
    rs = np.random.RandomState(6)
    done = 0
    for _ in range(150):
        m, n, p, i, v, kw = _random_case(rs)
        kind = kw.pop("split_type")
        frac = float(np.float32(kw["test_fraction"])) if v.dtype == np.float32 else kw["test_fraction"]
        try:
            o, eo = oracle_mod.oracle_split(p, i, v, m, n, split_type=kind, **kw), None
        except RuntimeError as e:
            o, eo = None, str(e)
        try:
            (users, held), ep = _capi.split_plan(p, m, n, kind != "all", **dict(kw, test_fraction=frac)), None
        except RuntimeError as e:
            ep = str(e)
        assert eo == ep, (kw, eo, ep)
        if o is None:
            continue
        if kind != "all":
            assert np.array_equal(users, o["users_test"])
        assert np.array_equal(held, _held_from_oracle(o, p, i, m, kind))
        done += 1
    assert done > 80


@pytest.mark.parametrize("knobs", [dict(RMB200_SPLIT_THREADS="0"), dict(RMB200_SPLIT_THREADS="3"),
                                   dict(RMB200_SPLIT_THREADS="2", RMB200_SPLIT_SCOUT_FAULT="0"),
                                   dict(RMB200_SPLIT_THREADS="3", RMB200_SPLIT_SCOUT_FAULT="3")])
def test_host_plan_threaded_replay(rb, oracle_mod, monkeypatch, knobs):
    """The replay of the random stream on several threads (recometrics_b200/csrc/split.cu, struct Replay): a scout runs ahead
    counting the draws every std::shuffle will take, workers redo the chunks for real and publish them only if their generator
    ends where the scout said.  Forced here on small inputs (chunks of 150 entries), with the scout made to MISCOUNT in one
    chunk as well: the result must not change -- the disagreement is noticed and the rest replayed sequentially."""
    from recometrics_b200 import _capi
    monkeypatch.setenv("RMB200_SPLIT_CHUNK", "150")
    for k, val in knobs.items():
        monkeypatch.setenv(k, val)
    for name in ("split_all_f64", "split_all_long_rows_f32", "split_separated_f32_strict", "split_joined_f64"):
        mk, kw = split_cases.CASES[name]
        kw = dict(kw)
        p, i, v = split_cases.make_csr(**mk)
        kind = kw.pop("split_type")
        o = oracle_mod.oracle_split(p, i, v, mk["m"], mk["n"], split_type=kind, **kw)
        frac = float(np.float32(kw["test_fraction"])) if v.dtype == np.float32 else kw["test_fraction"]
        users, held = _capi.split_plan(p, mk["m"], mk["n"], kind != "all", **dict(kw, test_fraction=frac))
        assert np.array_equal(held, _held_from_oracle(o, p, i, mk["m"], kind)), (name, knobs)


def test_host_plan_threaded_replay_randomised(rb, monkeypatch):
    """A few hundred calls with random worker counts, random injected miscounts and seeds beyond 32 bits, on rows that reach
    the shuffle's second regime (65,536 entries and more): always the bytes of the sequential replay."""
    from recometrics_b200 import _capi
    rs = np.random.RandomState(11)
    p, i, v = split_cases.make_csr(m=1500, n=70001, seed=31, mean_len=12.0, heavy_rows=(66000, 65535, 2, 3, 4, 5))
    for seed in (9, 2 ** 32 + 5, 2 ** 63 + 12345):
        monkeypatch.setenv("RMB200_SPLIT_THREADS", "0")
        monkeypatch.delenv("RMB200_SPLIT_SCOUT_FAULT", raising=False)
        _, ref = _capi.split_plan(p, 1500, 70001, False, test_fraction=0.35, seed=seed)
        monkeypatch.setenv("RMB200_SPLIT_CHUNK", "9000")
        for _ in range(60):
            monkeypatch.setenv("RMB200_SPLIT_THREADS", str(rs.randint(1, 7)))
            fault = int(rs.randint(-1, 20))
            if fault >= 0:
                monkeypatch.setenv("RMB200_SPLIT_SCOUT_FAULT", str(fault))
            else:
                monkeypatch.delenv("RMB200_SPLIT_SCOUT_FAULT", raising=False)
            _, held = _capi.split_plan(p, 1500, 70001, False, test_fraction=0.35, seed=seed)
            assert np.array_equal(held, ref), (seed, fault)


@pytest.mark.parametrize("name", sorted(split_cases.REFUSALS))
def test_host_plan_refuses_with_the_reference_message(rb, name):
    from recometrics_b200 import _capi
    mk, kw, message = split_cases.REFUSALS[name]
    kw = dict(kw)
    kw.pop("split_type")
    p, _, _ = split_cases.make_csr(**mk)
    with pytest.raises(RuntimeError, match=message):
        _capi.split_plan(p, mk["m"], mk["n"], True, **kw)


# ---- the Python front: the reference's checks, in its order, before anything native (recometrics/__init__.py:764-822) ----
def test_front_end_argument_checks(rb):
    import scipy.sparse as sp
    X = sp.random(30, 20, density=0.3, format="csr", random_state=1)
    with pytest.raises(ValueError, match="'min_pos_test' must be smaller"):
        rb.split_reco_train_test(X, min_pos_test=20)
    with pytest.raises(ValueError, match="'min_items_pool' must be smaller"):
        rb.split_reco_train_test(X, min_items_pool=20)
    with pytest.raises(ValueError, match="less than 2 rows"):
        rb.split_reco_train_test(X[:1], split_type="joined")
    with pytest.raises(ValueError, match="no non-zero entries"):
        rb.split_reco_train_test(sp.csr_array((30, 20), dtype=np.float64), split_type="all")
    for bad in (dict(items_test_fraction=0.0), dict(items_test_fraction=1.0), dict(users_test_fraction=1.5), dict(seed=-1),
                dict(split_type="some"), dict(max_test_users=-3)):
        with pytest.raises(AssertionError):
            rb.split_reco_train_test(X, **bad)
    with pytest.warns(UserWarning, match="implies <1"), pytest.raises(RuntimeError):   # (RuntimeError: no GPU here / fine on a GPU box)
        rb.split_reco_train_test(X, users_test_fraction=0.001)
        raise RuntimeError("reached the native call")
