"""CPU: the unexpectedness / serendipity interface without a GPU -- the rmb200_serendipity_t mirror and the checks the new
entry points make before they look for a device."""
import ctypes

import numpy as np


def test_struct_mirror(rb):
    from recometrics_b200 import _capi
    S = _capi.Serendipity
    assert ctypes.sizeof(S) == 40 and _capi.load().rmb200_sizeof_serendipity() == 40
    assert (S.struct_size.offset, S.reserved0.offset, S.unexpectedness.offset, S.serendipity.offset) == (0, 4, 8, 16)
    assert (S.means.offset, S.counts.offset) == (24, 32)
    s = _capi.make_serendipity({"serendipity": 0x1000}, means=0x2000)
    assert (s.struct_size, s.unexpectedness, s.serendipity, s.means, s.counts) == (40, None, 0x1000, 0x2000, None)


def _args():
    from recometrics_b200 import _capi
    from tools import synth
    d = synth.make(1, m=40, n=60, p=4, k=3)
    Xtr, Xte = d["X_train"], d["X_test"]
    return (np.float32, d["A"], 4, d["B"], 4, 40, 60, 4, Xtr.indptr, Xtr.indices, Xte.indptr, Xte.indices,
            Xte.data.astype(np.float32), 3, False, False, {"p": np.empty(40, dtype=np.float32)}, True, 2, 1), _capi


def test_entry_checks_before_the_device(rb):
    """A wrong struct_size is RMB200_ERR_BAD_ARG whether or not a GPU is present, also next to a beyond struct; without a
    device a valid request fails for want of one."""
    args, _capi = _args()
    rows = {"unexpectedness": np.empty(40, dtype=np.float32), "serendipity": np.empty(40, dtype=np.float32)}
    for size in (16, 48):
        bad = _capi.make_serendipity(rows)
        bad.struct_size = size
        assert _capi.calc_metrics(*args, serendipity=bad) == _capi.ERR_BAD_ARG
        assert "rmb200_serendipity_t" in _capi.last_error()
        ild = _capi.make_beyond({"ild": np.empty(40, dtype=np.float32)})
        assert _capi.calc_metrics(*args, beyond=ild, serendipity=bad) == _capi.ERR_BAD_ARG
        assert "rmb200_serendipity_t" in _capi.last_error()
    if _capi.device_count() == 0:
        for one in ({"unexpectedness": rows["unexpectedness"]}, {"serendipity": rows["serendipity"]}, rows):
            assert _capi.calc_metrics(*args, serendipity=_capi.make_serendipity(one)) == _capi.ERR_NO_DEVICE
        means, counts = np.empty(2), np.empty(2, dtype=np.int64)
        s = _capi.make_serendipity(rows, means, counts)
        assert _capi.calc_metrics(*args, exposure=_capi.make_exposure(), serendipity=s) == _capi.ERR_NO_DEVICE
