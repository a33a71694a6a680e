"""GPU: the train/test splitters (rmb200_split_*, recometrics_b200/csrc/split.cu) against the oracle (oracle/split_oracle.c,
pinned to the reference by tests/test_split_oracle.py) and against the committed outputs of the reference itself
(tests/golden/split_*.npz): every index pointer, item id, value and selected user must be identical.  Also the invariants
the reference's own tests check (tests/testthat/test-split.R:7-93) through the Python drop-in, and, at a size the oracle
still finishes in seconds, properties that do not need an oracle at all."""
import numpy as np
import pytest
import scipy.sparse as sp

from test_split_oracle import check_against_golden
from tools import split_cases

pytestmark = pytest.mark.gpu


def _product(rb, p, i, v, m, n, **kw):
    from recometrics_b200 import _capi
    kw = dict(kw)
    return _capi.split(kw.pop("split_type"), p, i, v, m, n, **kw)


@pytest.mark.parametrize("name", sorted(split_cases.CASES))
def test_split_equals_reference_golden_and_oracle(rb, oracle_mod, name):
    mk, kw = split_cases.CASES[name]
    p, i, v = split_cases.make_csr(**mk)
    res = _product(rb, p, i, v, mk["m"], mk["n"], **kw)
    flat = split_cases.flatten(res)
    check_against_golden(name, flat)
    o = split_cases.flatten(oracle_mod.oracle_split(p, i, v, mk["m"], mk["n"], **kw))
    assert set(o) == set(flat)
    for k in o:
        assert np.array_equal(o[k], flat[k]), f"{name}: {k}"
    t = res["timing"]
    assert t["kernel_launches"] >= 4 and t["h2d_bytes"] > 0 and t["d2h_bytes"] > 0
    assert t["rows_sorted_on_device"] == (1 if mk.get("unsorted") else 0)


@pytest.mark.parametrize("knobs", [dict(RMB200_SPLIT_THREADS="0"), dict(RMB200_SPLIT_THREADS="3"),
                                   dict(RMB200_SPLIT_THREADS="3", RMB200_SPLIT_SCOUT_FAULT="2")])
def test_split_in_many_chunks_and_with_a_threaded_replay(rb, monkeypatch, knobs):
    """Chunks of 150 entries: the device thread works through dozens of chunks behind the replay (which runs sequentially, on
    several threads, and on several threads with its scout made to miscount once) -- same golden outputs."""
    monkeypatch.setenv("RMB200_SPLIT_CHUNK", "150")
    for k, val in knobs.items():
        monkeypatch.setenv(k, val)
    for name in ("split_all_f64", "split_all_unsorted_f64", "split_separated_f64", "split_joined_unsorted_f32", "split_all_long_rows_f32"):
        mk, kw = split_cases.CASES[name]
        p, i, v = split_cases.make_csr(**mk)
        check_against_golden(name, split_cases.flatten(_product(rb, p, i, v, mk["m"], mk["n"], **kw)))


def test_split_through_the_pageable_copy_pipelines(rb, oracle_mod, monkeypatch):
    """X goes up and the untouched users' rows come down through the library's copy pipelines for pageable memory (several
    copy threads + pinned bounce buffers, recometrics_b200/csrc/runtime.cu upload_rows / download_bytes) once a block reaches
    32 MB.  Forced here on small blocks (RMB200_UPLOAD_MIN_BYTES=1), and run on blocks of several bounce buffers each
    (2 M entries: 8 MB per index array and per lane buffer), against the oracle."""
    monkeypatch.setenv("RMB200_UPLOAD_MIN_BYTES", "1")
    for name in ("split_separated_f64", "split_joined_f64", "split_all_f32_half"):
        mk, kw = split_cases.CASES[name]
        p, i, v = split_cases.make_csr(**mk)
        check_against_golden(name, split_cases.flatten(_product(rb, p, i, v, mk["m"], mk["n"], **kw)))
    m, n = 60000, 30000
    rs = np.random.RandomState(8)
    lens = np.minimum(n - 2, (rs.pareto(1.4, m) * 40 + 1).astype(np.int64))
    indptr = np.zeros(m + 1, np.int32)
    indptr[1:] = np.cumsum(lens)
    nnz = int(indptr[-1])
    row_of = np.repeat(np.arange(m), lens)
    step = np.maximum(1, (n - 1) // np.maximum(lens[row_of], 1))
    indices = ((np.arange(nnz) - indptr[row_of]) * step + rs.randint(0, 1 << 30, size=m)[row_of] % step).astype(np.int32)
    data = ((np.arange(nnz) % 89) + 1).astype(np.float64)
    assert nnz > 5_000_000
    for kind in ("separated", "joined"):
        kw = dict(split_type=kind, n_users_test=3000, test_fraction=0.3, consider_cold_start=False, min_items_pool=2, min_pos_test=1, seed=6)
        got = split_cases.flatten(_product(rb, indptr, indices, data, m, n, **kw))
        want = split_cases.flatten(oracle_mod.oracle_split(indptr, indices, data, m, n, **kw))
        assert set(got) == set(want)
        for k in want:
            assert np.array_equal(got[k], want[k]), (kind, k)


@pytest.mark.parametrize("name", sorted(split_cases.REFUSALS))
def test_split_refuses_with_the_reference_message(rb, name):
    mk, kw, message = split_cases.REFUSALS[name]
    p, i, v = split_cases.make_csr(**mk)
    with pytest.raises(RuntimeError, match=message):
        _product(rb, p, i, v, mk["m"], mk["n"], **kw)


def test_random_splits_against_the_oracle(rb, oracle_mod):
    from test_split_oracle import _random_case
    rs = np.random.RandomState(77)
    done = 0
    for _ in range(120):
        m, n, p, i, v, kw = _random_case(rs)
        try:
            o, eo = oracle_mod.oracle_split(p, i, v, m, n, **kw), None
        except RuntimeError as e:
            o, eo = None, str(e)
        try:
            r, er = _product(rb, p, i, v, m, n, **kw), None
        except RuntimeError as e:
            r, er = None, str(e)
        assert eo == er, (kw, eo, er)
        if o is None:
            continue
        fo, fr = split_cases.flatten(o), split_cases.flatten(r)
        assert set(fo) == set(fr), kw
        for k in fo:
            assert fo[k].dtype == fr[k].dtype and np.array_equal(fo[k], fr[k]), (kw, k)
        done += 1
    assert done > 60


def _rsparse(m, n, density, seed, dtype=np.float64):
    X = sp.random(m, n, density=density, format="csr", random_state=seed, dtype=np.float64)
    X.data = np.round(X.data * 10 + 1).astype(dtype)
    return sp.csr_array(X)


def test_reference_r_tests_split_all(rb):
    """tests/testthat/test-split.R:7-33."""
    for n in (10000, 3):
        X = _rsparse(1000, n, 0.01, 123)
        X_train, X_test = rb.split_reco_train_test(X, split_type="all", users_test_fraction=0.2)
        assert abs((X_train + X_test) - X).sum() == 0
        assert X_train.shape == X_test.shape == X.shape


def test_reference_r_tests_split_separated_and_joined(rb):
    """tests/testthat/test-split.R:35-71."""
    X = _rsparse(1000, 10000, 0.01, 123)
    X_rem, X_train, X_test, users_test = rb.split_reco_train_test(X, split_type="separated", users_test_fraction=0.1)
    assert abs((X_train + X_test) - X[users_test, :]).sum() == 0
    assert X_train.shape == X_test.shape == (100, 10000)
    assert X_rem.shape == (900, 10000)
    assert abs(X_rem - X[np.setdiff1d(np.arange(1000), users_test), :]).sum() == 0
    assert np.all(np.diff(users_test) > 0)

    X_train, X_test, users_test = rb.split_reco_train_test(X, split_type="joined", users_test_fraction=0.1)
    assert abs((X_train[:100, :] + X_test) - X[users_test, :]).sum() == 0
    assert X_train.shape == X.shape and X_test.shape == (100, 10000)
    assert abs(X_train[100:, :] - X[np.setdiff1d(np.arange(1000), users_test), :]).sum() == 0


def test_reference_r_tests_fixed_number_of_users_and_error(rb):
    """tests/testthat/test-split.R:73-93."""
    X = _rsparse(10, 9, 0.5, 123)
    X_rem, X_train, X_test, users_test = rb.split_reco_train_test(X, users_test_fraction=None, max_test_users=2)
    assert len(users_test) == 2 and X_test.shape[0] == 2 and X_train.shape[0] == 2 and X_rem.shape[0] == 8
    X = _rsparse(1000, 3, 0.01, 1)
    with pytest.raises(RuntimeError, match="No users satisfy criteria"):
        rb.split_reco_train_test(X, min_pos_test=2)


def test_float32_values_and_other_input_types(rb, oracle_mod):
    """float32 data stays float32 (recometrics/__init__.py:811-812), anything else becomes float64; COO / dense inputs are
    converted to CSR first (__init__.py:34-41)."""
    X = _rsparse(300, 200, 0.05, 5, dtype=np.float32)
    tr, te = rb.split_reco_train_test(X, split_type="all", items_test_fraction=0.25, seed=3)
    assert tr.dtype == np.float32 and te.dtype == np.float32
    o = oracle_mod.oracle_split(X.indptr, X.indices, X.data, 300, 200, split_type="all", test_fraction=0.25, seed=3)
    assert np.array_equal(te.indptr, o["test"][0]) and np.array_equal(te.indices, o["test"][1]) and np.array_equal(te.data, o["test"][2])
    Xi = sp.csr_array((np.arange(1, X.nnz + 1, dtype=np.int64), X.indices, X.indptr), shape=X.shape)
    tr2, te2 = rb.split_reco_train_test(Xi.tocoo(), split_type="all", items_test_fraction=0.25, seed=3)
    assert tr2.dtype == np.float64 and np.array_equal(te2.indices, te.indices)
    tr3, te3 = rb.split_reco_train_test(Xi.toarray(), split_type="all", items_test_fraction=0.25, seed=3)
    assert abs(tr3 - tr2).sum() == 0 and abs(te3 - te2).sum() == 0


def test_empty_matrix_of_the_c_abi(rb):
    """split_data_selected_users returns without touching its outputs for m = 0 (src/recometrics.hpp:1033)."""
    from recometrics_b200 import _capi
    r = _capi.split("all", np.zeros(1, np.int32), np.zeros(0, np.int32), np.zeros(0, np.float64), 0, 5)
    assert r["train"] is None and r["test"] is None and r["rem"] is None


def test_large_split_properties_and_oracle(rb, oracle_mod):
    """150,000 users x 40,000 items, ~4.6 M entries with a few very long rows: per-row held-out counts are round(count *
    fraction) (hpp:1038), each half of a row is ascending, train + test is X row for row -- and the whole result equals the
    oracle's."""
    m, n = 150000, 40000
    rs = np.random.RandomState(3)
    lens = np.minimum(n - 1, (rs.pareto(1.3, m) * 12 + 1).astype(np.int64))
    lens[:3] = (39000, 20000, 1)
    lens[rs.rand(m) < 0.02] = 0
    indptr = np.zeros(m + 1, np.int32)
    indptr[1:] = np.cumsum(lens)
    nnz = int(indptr[-1])
    # unique ascending items per row: a random start and strictly positive steps that fit the catalogue
    indices = np.empty(nnz, np.int32)
    row_of = np.repeat(np.arange(m), lens)
    pos = np.arange(nnz) - indptr[row_of]
    step = np.maximum(1, (n - 1) // np.maximum(lens[row_of], 1))
    indices[:] = (pos * step + rs.randint(0, 1 << 30, size=m)[row_of] % step).astype(np.int32)
    data = ((np.arange(nnz) % 97) + 1).astype(np.float32)
    from recometrics_b200 import _capi
    frac = 0.3
    r = _capi.split("all", indptr, indices, data, m, n, test_fraction=frac, seed=42)
    trp, tri, trv, _ = r["train"]
    tep, tei, tev, _ = r["test"]
    want = np.round(lens * float(np.float32(frac))).astype(np.int64)
    assert np.array_equal(np.diff(tep), want) and np.array_equal(np.diff(trp), lens - want)
    X = sp.csr_array((data, indices, indptr), shape=(m, n))
    Xtr = sp.csr_array((trv, tri, trp), shape=(m, n))
    Xte = sp.csr_array((tev, tei, tep), shape=(m, n))
    for ptr, idx in ((trp, tri), (tep, tei)):            # each half of every row ascending (hpp:1064-1066, :1075-1077)
        same_row = np.diff(np.repeat(np.arange(m), np.diff(ptr))) == 0
        assert np.all(np.diff(idx)[same_row] > 0)
    assert abs((Xtr + Xte) - X).sum() == 0
    o = oracle_mod.oracle_split(indptr, indices, data, m, n, split_type="all", test_fraction=frac, seed=42)
    assert np.array_equal(o["test"][1], tei) and np.array_equal(o["test"][2], tev)
    assert np.array_equal(o["train"][1], tri) and np.array_equal(o["train"][2], trv)
    t = r["timing"]
    print("large split: total %.1f ms (plan %.1f, h2d %.1f, kernels %.2f, d2h %.1f), %d launches" % (
        t["total_ms"], t["plan_ms"], t["h2d_ms"], t["kernel_ms"], t["d2h_ms"], t["kernel_launches"]))


def test_reference_python_package_splits_on_the_library(rb, oracle_mod, tmp_path):
    """The reference's own Python package (recometrics/__init__.py + its unmodified Cython wrapper, built against
    include/recometrics_b200_shim.hpp by oracle/build_ref_cython.py -- no reference C++ compiled in) calling
    split_reco_train_test: every native call lands in librecometrics_b200.so and the result is the oracle's."""
    import glob
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cy = glob.glob(os.path.join(root, "oracle", "_ref", "cy_b200", "cpp_funs*.so"))
    if not cy:
        pytest.skip("oracle/_ref/cy_b200 was not built (no /root/reference in the build container)")
    probe = (
        "import sys; sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[2])\n"
        "import numpy as np, cpp_funs\n"
        "from scipy.sparse import csr_array\n"
        "from tools import split_cases\n"
        "p, i, v = split_cases.make_csr(m=500, n=350, seed=16)\n"
        "X = csr_array((v, i, p), shape=(500, 350))\n"
        "rem, tr, te, ut = cpp_funs.split_csr_separated_users(X, 60, 0.3, False, 2, 1, True, 1)\n"
        "np.savez(sys.argv[3], rem_p=rem.indptr, rem_i=rem.indices, rem_v=rem.data, train_p=tr.indptr, train_i=tr.indices, train_v=tr.data,\n"
        "         test_p=te.indptr, test_i=te.indices, test_v=te.data, users_test=ut)\n"
        "print('SPLIT', len(ut))\n")
    out = str(tmp_path / "cy_split.npz")
    run = subprocess.run([sys.executable, "-c", probe, os.path.dirname(cy[0]), root, out], capture_output=True, text=True, timeout=300)
    assert run.returncode == 0 and "SPLIT 60" in run.stdout, run.stdout + run.stderr
    check_against_golden("split_separated_f64", dict(np.load(out)))
