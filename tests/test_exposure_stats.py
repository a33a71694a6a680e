"""CPU: the catalogue statistics of item exposure (rmb200_exposure_stats, the host function every call uses) against an
independent restatement, their exact values, the 128-bit Gini numerator, the C struct mirror, the new entry point without a
GPU, and the sum of per-rank counts over gloo (recometrics_b200.dist.reduce_exposure)."""
import ctypes
import os
import socket
import sys

import numpy as np
import pytest
import scipy.stats

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _restated(c):
    """Sorted-order Gini over all n items (RecBole's GiniIndex), scipy's entropy, coverage."""
    c = np.asarray(c, dtype=np.float64)
    n, S = c.size, c.sum()
    cs = np.sort(c)
    i = np.arange(1, n + 1, dtype=np.float64)
    gini = float(((2 * i - n - 1) * cs).sum() / (n * S))
    return {"Coverage@K": float((c > 0).sum()) / n, "Gini@K": gini, "Entropy@K": float(scipy.stats.entropy(c, base=2)),
            "entries": int(np.asarray(c, dtype=np.int64).sum()), "items_covered": int((c > 0).sum())}


@pytest.mark.parametrize("seed", range(6))
def test_stats_equal_an_independent_restatement(rb, seed):
    from recometrics_b200 import _capi
    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 50000))
    c = np.minimum(rng.zipf(1.3 + 0.2 * seed, size=n), 10 ** 6).astype(np.int64) - 1     # heavy tail, many zeros
    c[rng.random(n) < 0.5] = 0
    c[0] += 1                                                             # (at least one entry)
    got = _capi.exposure_stats(c, users=17)
    want = _restated(c)
    assert got["users"] == 17
    assert got["entries"] == want["entries"] and got["items_covered"] == want["items_covered"]
    assert got["Coverage@K"] == want["Coverage@K"]
    for key in ("Gini@K", "Entropy@K"):
        assert got[key] == pytest.approx(want[key], rel=1e-12, abs=1e-14), key


def test_exact_values(rb):
    from recometrics_b200 import _capi
    n = 1000
    u = _capi.exposure_stats(np.full(n, 7, dtype=np.int64))
    assert u["Gini@K"] == 0.0 and u["Coverage@K"] == 1.0 and u["Entropy@K"] == pytest.approx(np.log2(n), rel=1e-15)
    one = np.zeros(n, dtype=np.int64)
    one[123] = 99
    o = _capi.exposure_stats(one)
    assert o["Gini@K"] == (n - 1) / n and o["Entropy@K"] == 0.0 and o["items_covered"] == 1 and o["Coverage@K"] == 1 / n
    z = _capi.exposure_stats(np.zeros(n, dtype=np.int64))
    assert z["Coverage@K"] == 0.0 and np.isnan(z["Gini@K"]) and np.isnan(z["Entropy@K"]) and z["entries"] == 0


def test_gini_numerator_beyond_int64(rb):
    """Counts near 2^31 on 1M items: sum_i (2i - n - 1) c_(i) is ~1e21, past int64 -- the 128-bit path, and the sort branch
    (the largest count is far above the counts-of-counts table's bound)."""
    from recometrics_b200 import _capi
    rng = np.random.default_rng(3)
    n = 1 << 20
    c = (2 ** 31 - 1 - rng.integers(0, 2 ** 20, size=n)).astype(np.int64)
    c[rng.random(n) < 0.3] = 0
    got = _capi.exposure_stats(c)
    cs = np.sort(c)
    num = sum(int(2 * i - n - 1) * int(v) for i, v in zip(range(1, n + 1), cs.tolist()))     # Python integers: exact
    assert abs(num) > 2 ** 63
    assert got["Gini@K"] == num / (n * int(c.sum()))
    assert got["entries"] == int(c.sum())
    assert got["Entropy@K"] == pytest.approx(scipy.stats.entropy(c.astype(np.float64), base=2), rel=1e-12)


def test_bad_counts_are_refused(rb):
    from recometrics_b200 import _capi
    with pytest.raises(ValueError):
        _capi.exposure_stats(np.array([3, -1, 2], dtype=np.int64))
    with pytest.raises(ValueError):
        _capi.exposure_stats(np.zeros(0, dtype=np.int64))
    with pytest.raises(ValueError):
        _capi.exposure_stats(np.array([2 ** 62, 2 ** 62], dtype=np.int64))     # total beyond int64
    e = _capi.make_exposure()
    e.struct_size = 8
    c = np.ones(4, dtype=np.int64)
    assert _capi.load().rmb200_exposure_stats(_capi._vp(c), 4, ctypes.byref(e)) == _capi.ERR_BAD_ARG


def test_exposure_struct_layout_matches_header(rb):
    from recometrics_b200 import _capi
    E = _capi.Exposure
    assert ctypes.sizeof(E) == 64 and _capi.load().rmb200_sizeof_exposure() == 64
    assert (E.struct_size.offset, E.item_counts.offset, E.users.offset, E.entries.offset, E.items_covered.offset) == (0, 8, 16, 24, 32)
    assert (E.coverage.offset, E.gini.offset, E.entropy_bits.offset) == (40, 48, 56)


def test_exposure_entry_without_a_device(rb):
    """The new entry point checks the struct size first (RMB200_ERR_BAD_ARG), then fails for want of a GPU; _ex is unaffected."""
    from recometrics_b200 import _capi
    if _capi.device_count() > 0:
        pytest.skip("a CUDA device is present")
    from tools import synth
    d = synth.make(1, m=40, n=60, p=4, k=3)
    A, B, Xtr, Xte = d["A"], d["B"], d["X_train"], d["X_test"]
    args = (np.float32, A, 4, B, 4, 40, 60, 4, Xtr.indptr, Xtr.indices, Xte.indptr, Xte.indices, Xte.data.astype(np.float32), 3,
            False, False, {"p": np.empty(40, dtype=np.float32)}, True, 2, 1)
    bad = _capi.make_exposure()
    bad.struct_size = 16
    assert _capi.calc_metrics(*args, exposure=bad) == _capi.ERR_BAD_ARG
    assert "rmb200_exposure_t" in _capi.last_error()
    assert _capi.calc_metrics(*args, exposure=_capi.make_exposure(np.zeros(60, dtype=np.int64))) == _capi.ERR_NO_DEVICE
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        rb.calc_reco_metrics_ex(Xtr, Xte, A, B, k=3, break_ties_with_noise=False, return_exposure=True)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _reduce_worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist
    from recometrics_b200 import _capi
    from recometrics_b200.dist import reduce_exposure
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        n = 5000
        per_rank = [np.random.default_rng(40 + r).poisson(0.7, size=n).astype(np.int64) for r in range(world)]
        got = reduce_exposure(per_rank[rank], dst=0, local_users=100 + rank)
        if rank == 0:
            total = per_rank[0] + per_rank[1]
            counts, cat = got
            ok = np.array_equal(counts, total) and cat == _capi.exposure_stats(total, users=201)
            q.put("ok" if ok else "mismatch")
        else:
            q.put("ok" if got is None else "rank 1 got a result")
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_reduce_exposure_world2_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_reduce_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=240) for _ in procs]
    for p in procs:
        p.join(60)
    assert res == ["ok", "ok"], res
