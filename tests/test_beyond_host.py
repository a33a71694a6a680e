"""CPU: the beyond-accuracy interface without a GPU -- the rmb200_beyond_t mirror, the argument checks the new entry points
make before they look for a device, the Python checks of item_popularity, and dist.reduce_popularity over gloo."""
import ctypes
import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_struct_mirror(rb):
    from recometrics_b200 import _capi
    Bt = _capi.Beyond
    assert ctypes.sizeof(Bt) == 64 and _capi.load().rmb200_sizeof_beyond() == 64
    assert (Bt.struct_size.offset, Bt.item_popularity.offset, Bt.popularity_users.offset) == (0, 8, 16)
    assert (Bt.novelty.offset, Bt.avg_popularity.offset, Bt.ild.offset, Bt.means.offset, Bt.counts.offset) == (24, 32, 40, 48, 56)


def _args():
    from recometrics_b200 import _capi
    from tools import synth
    d = synth.make(1, m=40, n=60, p=4, k=3)
    Xtr, Xte = d["X_train"], d["X_test"]
    return (np.float32, d["A"], 4, d["B"], 4, 40, 60, 4, Xtr.indptr, Xtr.indices, Xte.indptr, Xte.indices,
            Xte.data.astype(np.float32), 3, False, False, {"p": np.empty(40, dtype=np.float32)}, True, 2, 1), _capi


def test_entry_checks_before_the_device(rb):
    """struct_size, missing popularity, popularity_users < 1 and out-of-range host counts are RMB200_ERR_BAD_ARG whether or
    not a GPU is present; a valid request then fails for want of a device."""
    args, _capi = _args()
    rows = {"novelty": np.empty(40, dtype=np.float32)}
    pop = np.zeros(60, dtype=np.int64)
    bad = _capi.make_beyond(rows, pop, 40)
    bad.struct_size = 16
    assert _capi.calc_metrics(*args, beyond=bad) == _capi.ERR_BAD_ARG and "rmb200_beyond_t" in _capi.last_error()
    assert _capi.calc_metrics(*args, beyond=_capi.make_beyond(rows, None, 40)) == _capi.ERR_BAD_ARG
    assert "item_popularity" in _capi.last_error()
    assert _capi.calc_metrics(*args, beyond=_capi.make_beyond({"avg_popularity": rows["novelty"]}, pop, 0)) == _capi.ERR_BAD_ARG
    for v in (-1, 41):
        p = pop.copy()
        p[7] = v
        assert _capi.calc_metrics(*args, beyond=_capi.make_beyond(rows, p, 40)) == _capi.ERR_BAD_ARG
        assert "outside" in _capi.last_error()
    # ILD alone needs no popularity
    if _capi.device_count() == 0:
        assert _capi.calc_metrics(*args, beyond=_capi.make_beyond({"ild": np.empty(40, dtype=np.float32)})) == _capi.ERR_NO_DEVICE
        assert _capi.calc_metrics(*args, beyond=_capi.make_beyond(rows, pop, 40)) == _capi.ERR_NO_DEVICE
        counts = np.zeros(60, dtype=np.int64)
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            _capi.item_popularity(args[8], args[9], 0, 40, 60, counts)
    with pytest.raises(ValueError):
        _capi.item_popularity(args[8], args[9], 5, 2, 60, np.zeros(60, dtype=np.int64))


def test_python_checks_of_item_popularity(rb):
    from tools import synth
    d = synth.make(1, m=40, n=60, p=4, k=3)
    kw = dict(k=3, break_ties_with_noise=False, novelty=True)
    call = lambda pop: rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], item_popularity=pop, **kw)
    with pytest.raises(ValueError, match="one count per item"):
        call(np.zeros(59, dtype=np.int64))
    with pytest.raises(ValueError, match="one count per item"):
        call(np.zeros((60, 1), dtype=np.int64))
    with pytest.raises(TypeError, match="integer"):
        call(np.zeros(60, dtype=np.float64))
    with pytest.raises(ValueError, match=r"\[0, 40\]"):
        call(np.full(60, 41, dtype=np.int64))
    with pytest.raises(ValueError, match=r"\[0, 40\]"):
        call(np.full(60, -1, dtype=np.int32))
    with pytest.raises(ValueError):
        rb.item_popularity(d["X_train"], user_range=(10, 5))
    with pytest.raises(TypeError):
        rb.item_popularity(np.zeros((4, 4)))


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
    from recometrics_b200.dist import reduce_popularity
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        n = 5000
        per_rank = [np.random.default_rng(70 + r).poisson(3.0, size=n).astype(np.int64) for r in range(world)]
        got = reduce_popularity(per_rank[rank])
        ok = got.dtype == np.int64 and np.array_equal(got, per_rank[0] + per_rank[1])
        q.put("ok" if ok else "mismatch on rank %d" % rank)
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_reduce_popularity_world2_gloo():
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
