"""GPU: the argument checks of calc_reco_metrics_device -- every error and warning with its full text, which of several
faults is reported first, and the places where it knowingly checks less than calc_reco_metrics_ex does."""
import re
import warnings

import numpy as np
import pytest
from scipy.sparse import csr_array, vstack

from tools import synth

pytestmark = pytest.mark.gpu


def _exact(msg):
    return "^%s$" % re.escape(msg)


@pytest.fixture(scope="module")
def case(rb):
    import torch
    dev = torch.device("cuda", 0)
    d = synth.make(1, m=30, n=50, p=4, k=3)
    tA, tB = torch.from_numpy(d["A"]).to(dev), torch.from_numpy(d["B"]).to(dev)

    def call(**kw):
        return rb.calc_reco_metrics_device(**{**dict(X_train=d["X_train"], X_test=d["X_test"], A=tA, B=tB, k=3,
                                                     break_ties_with_noise=False), **kw})
    # a bad item_popularity is checked after every other argument: a call with one stops there, before the library runs
    short_pop = dict(novelty=True, item_popularity=torch.zeros(49, dtype=torch.int64, device=dev))
    return d, tA, tB, dev, call, short_pop


NO_METRIC = dict(precision=False, average_precision=False, ndcg=False, recall=True)
POP_LEN = "'item_popularity' must be a 1-d array with one count per item (50)."
POP_RANGE = "'item_popularity' counts must lie in [0, 30] (the number of users)."


def test_device_front_end_errors(rb, case):
    import torch
    d, tA, tB, dev, call, _ = case
    Xtr, Xte = d["X_train"], d["X_test"]
    other = torch.float64 if tA.dtype == torch.float32 else torch.float32
    Xte_dev = rb.DeviceCSR.from_scipy(Xte, 0, d["A"].dtype)
    counts_rule = "'seed', 'k', 'min_pos_test' and 'min_items_pool' must be >= 1."
    nb_rule = "Number of items in 'item_biases' must match with 'X_test'."
    for kw, exc, msg in (
            (dict(B=None), ValueError, "'A' and 'B' must be passed (device-resident factor matrices)."),
            (dict(A=d["A"]), TypeError, "'A' must expose __cuda_array_interface__ (a torch CUDA tensor, a CuPy array, ...)."),
            (dict(A=tA.int()), TypeError, "'A' must be float32 or float64."),
            (dict(B=tB[:, 0]), ValueError, "'B' must be a 2-dimensional array."),
            (dict(A=tA.t()), ValueError, "'A' must be row-major (unit column stride); make it contiguous first."),
            (dict(A=tA.to(other)), TypeError,
             "'A' and 'B' must have the same dtype on the device (the host front-end would promote to float64)."),
            (NO_METRIC, ValueError, "Must pass at least one metric to calculate."),
            (dict(X_test=Xte.toarray()), TypeError, "'X_test' must be a sparse matrix or a DeviceCSR."),
            (dict(X_train=Xtr.toarray()), TypeError, "'X_train' must be a sparse matrix or a DeviceCSR."),
            (dict(X_train=Xtr[:, :49]), ValueError, "'X_train' and 'X_test' should have the same number of columns."),
            (dict(X_train=Xtr[:29]), ValueError, "'X_train' and 'X_test' should have the same number of rows."),
            (dict(B=tB[:, :3]), ValueError, "'A' and 'B' must have the same number of columns."),
            (dict(A=tA[:, :0], B=tB[:, :0]), ValueError, "Input matrices cannot be empty."),
            (dict(A=tA[:10]), ValueError, "Number of users in 'A' and 'X_test' does not match."),
            (dict(B=tB[:10]), ValueError, "Number of items in 'B' and 'X_test' does not match."),
            (dict(seed=0), ValueError, counts_rule),
            (dict(k=0), ValueError, counts_rule),
            (dict(min_pos_test=0), ValueError, counts_rule),
            (dict(min_items_pool=0), ValueError, counts_rule),
            (dict(k=51), ValueError, "'k' should be smaller than the number of items."),
            (dict(X_test=rb.DeviceCSR(Xte_dev.indptr.long(), Xte_dev.indices, Xte_dev.data, Xte_dev.shape)), TypeError,
             "X_test.indptr must be a contiguous int32 tensor on cuda:0."),
            (dict(X_test=rb.DeviceCSR(Xte_dev.indptr, Xte_dev.indices, None, Xte_dev.shape)), ValueError,
             "'X_test' needs its values for NDCG."),
            (dict(item_biases=torch.ones(100, dtype=tA.dtype, device=dev)[::2]), ValueError, "'item_biases' must be contiguous."),
            (dict(item_biases=torch.ones(50, dtype=other, device=dev)), TypeError, "'item_biases' must have the dtype of the factors."),
            (dict(item_biases=torch.ones(10, dtype=tA.dtype, device=dev)), ValueError, nb_rule),
            (dict(item_biases=np.ones(10, dtype=d["A"].dtype)), ValueError, nb_rule),
            (dict(novelty=True, item_popularity=torch.zeros(49, dtype=torch.int64, device=dev)), ValueError, POP_LEN),
            (dict(avg_popularity=True, item_popularity=torch.zeros((50, 1), dtype=torch.int64, device=dev)), ValueError, POP_LEN),
            (dict(novelty=True, item_popularity=torch.zeros(50, device=dev)), TypeError, "'item_popularity' must hold integer counts."),
            (dict(novelty=True, item_popularity=torch.zeros(50, dtype=torch.bool)), TypeError, "'item_popularity' must hold integer counts."),
            (dict(novelty=True, item_popularity=torch.full((50,), 31, dtype=torch.int64, device=dev)), ValueError, POP_RANGE),
            (dict(avg_popularity=True, item_popularity=torch.full((50,), -1, dtype=torch.int32)), ValueError, POP_RANGE),
            (dict(novelty=True, item_popularity=np.zeros(49, dtype=np.int64)), ValueError, POP_LEN),
            (dict(novelty=True, item_popularity=np.zeros(50)), TypeError, "'item_popularity' must hold integer counts."),
            (dict(novelty=True, item_popularity=np.full(50, 31, dtype=np.int64)), ValueError, POP_RANGE),
            # several faults: the metric guard comes first here (the host front-end reports the column count first)
            (dict(B=tB[:, :3], **NO_METRIC), ValueError, "Must pass at least one metric to calculate.")):
        with pytest.raises(exc, match=_exact(msg)):
            call(**kw)
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError, match=_exact("'A' and 'B' must be on the same device.")):
            call(B=tB.to("cuda:1"))


def test_device_front_end_warnings(case):
    import torch
    d, tA, tB, dev, call, short_pop = case
    for kw, msg in ((dict(A=torch.cat([tA, tA[:1]])), "'A' has more users than 'X_test'."),
                    (dict(B=torch.cat([tB, tB[:1]])), "'B' has more items than 'X_test'.")):
        with pytest.warns(UserWarning, match=_exact(msg)), pytest.raises(ValueError, match=_exact(POP_LEN)):
            call(**kw, **short_pop)


def test_device_front_end_checks_less_than_the_host_one(case):
    """Not a wish but a record: the device front-end does not warn of extra X_train rows or item_biases entries, does not
    check the shape of numpy item_biases beyond their length, lets an empty X_test through, takes integer seeds only and
    has none of return_ranks / devices / nan_bits / filter_stats / nthreads."""
    import torch
    d, tA, tB, dev, call, short_pop = case
    dt = d["A"].dtype
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        for kw in (dict(X_train=vstack([d["X_train"], d["X_train"][:1]]).tocsr()),
                   dict(item_biases=torch.ones(51, dtype=tA.dtype, device=dev)),
                   dict(item_biases=np.ones(51, dtype=dt)),
                   dict(item_biases=np.ones((50, 1, 1), dtype=dt)),
                   dict(X_test=csr_array(d["X_test"].shape, dtype=dt))):
            with pytest.raises(ValueError, match=_exact(POP_LEN)):
                call(**kw, **short_pop)
    with pytest.raises(ValueError, match=_exact("Number of items in 'item_biases' must match with 'X_test'.")):
        call(item_biases=np.ones(0, dtype=dt))
    with pytest.raises(TypeError):
        call(seed=np.random.RandomState(1))
    for name, value in (("return_ranks", True), ("devices", [0]), ("nan_bits", 0), ("filter_stats", True), ("nthreads", 1)):
        with pytest.raises(TypeError, match="unexpected keyword argument '%s'" % name):
            call(**{name: value})
