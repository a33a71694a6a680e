"""GPU: the C-ABI's telescoping entry points and which means / counts tables a call writes.

* ``rmb200_calc_metrics_exposure_*(..., NULL)``, ``_beyond_*(..., NULL, NULL)`` and ``_serendipity_*(..., NULL, NULL,
  NULL)`` are exactly the ``_ex`` call (the header's promise); the front-ends only ever call the entry point their arguments
  select, so these are reached here by sending the ``_ex`` call to each of them.
* A family's means table is written only together with one of its rows: a beyond-accuracy or history table passed without
  its rows is left untouched, on one device and on several.  The metric table is written whenever it is given, NaN with a
  count of 0 when no metric row is requested."""
import numpy as np
import pytest

from tools import synth

pytestmark = pytest.mark.gpu

SENTINEL_MEAN, SENTINEL_COUNT = 7.25, -3


def _same(a, b):
    """Equal bytes (NaN payloads included); None only equals None."""
    if a is None or b is None:
        return a is None and b is None
    a, b = np.ascontiguousarray(np.atleast_1d(np.asarray(a))), np.ascontiguousarray(np.atleast_1d(np.asarray(b)))
    return a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


class _ToEntryPoint:
    """The loaded library with its ``rmb200_calc_metrics_ex_*`` calls sent to ``rmb200_calc_metrics_<kind>_*`` with NULL for
    each of its ``nulls`` trailing struct arguments."""

    def __init__(self, lib, kind, nulls):
        self.lib, self.kind, self.nulls = lib, kind, nulls

    def __getattr__(self, name):
        if name.startswith("rmb200_calc_metrics_ex_"):
            fn = getattr(self.lib, name.replace("_ex_", "_%s_" % self.kind))
            return lambda *args: fn(*args, *([None] * self.nulls))
        return getattr(self.lib, name)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_null_structs_are_the_ex_call(rb, monkeypatch, dtype):
    from recometrics_b200 import _capi
    d = synth.make(1, m=2000, n=3000, p=24)
    A, B = d["A"].astype(dtype), d["B"].astype(dtype)

    def run():
        return rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], A, B, k=10, all_metrics=True, break_ties_with_noise=False,
                                       return_topk=True, return_status=True, return_ranks=True, return_means=True)
    want = run()
    lib = _capi.load()
    for kind, nulls in (("exposure", 1), ("beyond", 2), ("serendipity", 3)):
        monkeypatch.setattr(_capi, "load", lambda: _ToEntryPoint(lib, kind, nulls))
        got = run()
        monkeypatch.undo()
        assert got.metrics.keys() == want.metrics.keys(), kind
        for key in want.metrics:
            assert _same(got.metrics[key], want.metrics[key]), (kind, key)
        for field in ("status", "topk_items", "topk_scores", "pos_rank"):
            assert _same(getattr(got, field), getattr(want, field)), (kind, field)
        assert got.means.keys() == want.means.keys() and got.counts == want.counts, kind
        assert all(_same(got.means[key], want.means[key]) for key in want.means), kind
        assert got.timing["scoring_path"] == want.timing["scoring_path"], kind


def _call(devices=None, metric_rows=True, beyond=None, serendipity=None):
    """One float32 call from host arrays with top-K items; returns (rc, topk_items, metric means, metric counts)."""
    from recometrics_b200 import _capi
    d = synth.make(1, m=3000, n=4000, p=16)
    Xtr, Xte = d["X_train"], d["X_test"]
    m, n, K = 3000, 4000, 10
    topk = np.full(m * K, -7, dtype=np.int32)
    means, counts = np.full(10, SENTINEL_MEAN), np.full(10, SENTINEL_COUNT, dtype=np.int64)
    outs = {"p": np.empty(m, dtype=np.float32), "ndcg": np.empty(m, dtype=np.float32)} if metric_rows else {}
    ex = _capi.make_extra(topk_items=topk, metric_means=means, metric_counts=counts, devices=devices)
    rc = _capi.calc_metrics(np.float32, d["A"], 16, d["B"], 16, m, n, 16, Xtr.indptr, Xtr.indices, Xte.indptr, Xte.indices,
                            Xte.data.astype(np.float32), K, False, False, outs, True, 2, 1, extra=ex,
                            beyond=beyond, serendipity=serendipity)
    return rc, topk, means, counts


def _family_tables_without_rows(devices):
    from recometrics_b200 import _capi
    tables = {}
    for name, make in (("beyond", lambda mn, ct: _capi.make_beyond({}, None, 0, mn, ct)),
                       ("serendipity", lambda mn, ct: _capi.make_serendipity({}, mn, ct))):
        slots = 3 if name == "beyond" else 2
        mn, ct = np.full(slots, SENTINEL_MEAN), np.full(slots, SENTINEL_COUNT, dtype=np.int64)
        rc, topk, means, counts = _call(devices, **{name: make(mn, ct)})
        assert rc == _capi.OK, _capi.last_error()
        assert (topk >= 0).any() and np.isfinite(means[[0, 5]]).all() and (counts[[0, 5]] > 0).all()
        assert (mn == SENTINEL_MEAN).all() and (ct == SENTINEL_COUNT).all(), (name, mn, ct)
        tables[name] = means
    # the metric table without a metric row: written, NaN with a count of 0
    rc, topk, means, counts = _call(devices, metric_rows=False)
    assert rc == _capi.OK, _capi.last_error()
    assert (topk >= 0).any() and np.isnan(means).all() and (counts == 0).all()
    return tables


def test_family_means_without_rows_one_device(rb):
    _family_tables_without_rows(None)


def test_family_means_without_rows_two_devices(rb):
    if rb.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    one = _family_tables_without_rows(None)
    two = _family_tables_without_rows([0, 1])
    for name in one:
        np.testing.assert_allclose(two[name], one[name], rtol=1e-12)
