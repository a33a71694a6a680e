"""CPU: the C-ABI library loads, exports every symbol include/*.h declares, and refuses to compute
without a device (no CPU fallback).  No compute calls are made here."""
import ctypes
import glob
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    names = []
    for h in glob.glob(os.path.join(ROOT, "include", "*.h")):
        txt = open(h).read()
        names += re.findall(r"RMB200_API\s+[\w\s\*]+?\b(rmb200_\w+)\s*\(", txt)
    return sorted(set(names))


def test_header_declares_the_boundary():
    names = _declared_symbols()
    for want in ("rmb200_calc_metrics_f32", "rmb200_calc_metrics_f64", "rmb200_calc_metrics_ex_f32",
                 "rmb200_calc_metrics_ex_f64", "rmb200_last_error", "rmb200_device_count",
                 "rmb200_split_selected_users_f32", "rmb200_split_selected_users_f64", "rmb200_split_separate_users_f32",
                 "rmb200_split_separate_users_f64", "rmb200_split_joined_users_f32", "rmb200_split_joined_users_f64",
                 "rmb200_split_free"):
        assert want in names


def test_library_exports_every_declared_symbol(rb):
    from recometrics_b200 import _capi
    lib = ctypes.CDLL(_capi.LIB_PATH)
    for name in _declared_symbols():
        assert hasattr(lib, name), name
    assert set(_declared_symbols()) == set(_capi.EXPORTS)
    assert lib.rmb200_version() == 100


def test_extra_struct_layout_matches_header(rb):
    """ctypes mirror of rmb200_extra_t / rmb200_timing_t has the C layout (LP64)."""
    from recometrics_b200 import _capi
    assert ctypes.sizeof(_capi.Timing) == 6 * 8 + 11 * 8
    assert ctypes.sizeof(_capi.Extra) == 6 * 4 + 5 * 8 + 2 * 4 + 2 * 8 + 2 * 4 + 8 + 8 + 2 * 4
    assert _capi.Extra.nan_bits.offset == 96 and _capi.Extra.devices.offset == 104
    assert _capi.Extra.topk_items.offset == 24
    assert _capi.Extra.scoring_path.offset == 64
    assert _capi.Extra.metric_means.offset == 72
    lib = _capi.load()          # the sizes the library itself was compiled with
    assert lib.rmb200_sizeof_extra() == ctypes.sizeof(_capi.Extra)
    assert lib.rmb200_sizeof_timing() == ctypes.sizeof(_capi.Timing)


def test_split_struct_layout_matches_header(rb):
    """ctypes mirror of rmb200_csr_t / rmb200_split_t (LP64)."""
    from recometrics_b200 import _capi
    assert ctypes.sizeof(_capi.Csr) == 2 * 4 + 8 + 3 * 8
    assert ctypes.sizeof(_capi.Split) == 3 * 40 + 8 + 4 * 4 + 5 * 8 + 3 * 8 + 8
    assert _capi.Split.users_test.offset == 120 and _capi.Split.total_ms.offset == 144 and _capi.Split.owner.offset == 208
    assert _capi.load().rmb200_sizeof_split() == ctypes.sizeof(_capi.Split)


def test_no_device_means_no_split_either(rb):
    """The splitters need the GPU for every matrix they return: without one the call fails (RMB200_ERR_NO_DEVICE) after the
    reference's own argument checks -- which still answer first, with the reference's messages."""
    from recometrics_b200 import _capi
    if _capi.device_count() > 0:
        pytest.skip("a CUDA device is present")
    from tools import split_cases
    p, i, v = split_cases.make_csr(m=50, n=80, seed=21)
    for kind in ("all", "separated", "joined"):
        with pytest.raises(RuntimeError, match="no CPU"):
            _capi.split(kind, p, i, v, 50, 80, n_users_test=5)
    with pytest.raises(RuntimeError, match="Target number of test users is larger"):
        _capi.split("separated", p, i, v, 50, 80, n_users_test=51)


def test_no_device_means_error_not_fallback(rb):
    """On a machine without a GPU every compute entry fails loudly (the product has no CPU path)."""
    from recometrics_b200 import _capi
    if _capi.device_count() > 0:
        pytest.skip("a CUDA device is present")
    from tools import synth
    d = synth.make(1, m=40, n=60, p=4, k=3)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        rb.calc_reco_metrics(d["X_train"], d["X_test"], d["A"], d["B"], k=3, break_ties_with_noise=False)


def test_no_device_multi_gpu_call_fails_the_same_way(rb, monkeypatch):
    """A device list (or RMB200_DEVICES) does not open a CPU path either."""
    from recometrics_b200 import _capi
    if _capi.device_count() > 0:
        pytest.skip("a CUDA device is present")
    from tools import synth
    d = synth.make(1, m=40, n=60, p=4, k=3)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        rb.calc_reco_metrics_ex(d["X_train"], d["X_test"], d["A"], d["B"], k=3, break_ties_with_noise=False, devices=[0, 1])
    monkeypatch.setenv("RMB200_DEVICES", "0,1")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        rb.calc_reco_metrics(d["X_train"], d["X_test"], d["A"], d["B"], k=3, break_ties_with_noise=False)
    monkeypatch.setenv("RMB200_DEVICES", "zero")
    with pytest.raises(ValueError, match="RMB200_DEVICES"):
        rb.calc_reco_metrics(d["X_train"], d["X_test"], d["A"], d["B"], k=3, break_ties_with_noise=False)


def test_product_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under recometrics_b200/ may reference it."""
    for path in glob.glob(os.path.join(ROOT, "recometrics_b200", "**", "*"), recursive=True):
        if os.path.isfile(path) and path.endswith((".py", ".cu", ".cuh", ".h", ".hpp")):
            txt = open(path, errors="replace").read()
            assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, re.M), path
            assert "librmoracle" not in txt and "librecometrics_ref" not in txt, path


def _exact(msg):
    return "^%s$" % re.escape(msg)


def test_frontend_validation_mirrors_reference(rb):
    """Argument errors and warnings are raised on the host before anything touches the GPU, each with its full text, and of
    several faults the first in the reference's order is reported (reference: recometrics/__init__.py:426-467, :499-500,
    :531-532; then the checks of item_popularity)."""
    from scipy.sparse import coo_array, csr_array, vstack
    from tools import synth
    d = synth.make(1, m=30, n=50, p=4, k=3)
    Xtr, Xte, A, B = d["X_train"], d["X_test"], d["A"], d["B"]
    imax = np.iinfo(np.int32).max

    def call(**kw):
        return rb.calc_reco_metrics_ex(**{**dict(X_train=Xtr, X_test=Xte, A=A, B=B, k=3, break_ties_with_noise=False), **kw})

    no_metric = dict(precision=False, average_precision=False, ndcg=False, recall=True)
    counts_rule = "'seed', 'k', 'min_pos_test' and 'min_items_pool' must be >= 1."
    pop_len = "'item_popularity' must be a 1-d array with one count per item (50)."
    pop_range = "'item_popularity' counts must lie in [0, 30] (the number of users)."
    for kw, exc, msg in (
            (dict(B=None), ValueError, "'A' and 'B' must either be passed together or passed as 'None' together."),
            (dict(A=None, B=None), ValueError, "Must pass item biases if not passing factors."),
            (dict(A=A.tolist()), TypeError, "'A' and 'B' must be numpy arrays."),
            (dict(X_test=Xte.toarray()), TypeError, "'X_test' must be a sparse matrix."),
            (dict(X_test=coo_array((imax, 50))), ValueError, "Number of test user is larger than maximum supported."),
            (dict(X_test=coo_array((30, imax))), ValueError, "Number of items is larger than maximum supported."),
            (dict(X_test=csr_array(Xte.shape, dtype=np.float32)), ValueError, "'X_test' is empty."),
            (dict(A=A[:, 0]), ValueError, "'A' must be a 2-dimensional array."),
            (dict(B=B[:, 0]), ValueError, "'B' must be a 2-dimensional array."),
            (dict(B=B[:, :3]), ValueError, "'A' and 'B' must have the same number of columns."),
            (dict(A=A[:, :0], B=B[:, :0]), ValueError, "Input matrices cannot be empty."),
            (dict(A=A[:10]), ValueError, "Number of users in 'A' and 'X_test' does not match."),
            (dict(B=B[:10]), ValueError, "Number of items in 'B' and 'X_test' does not match."),
            (dict(X_train=Xtr.toarray()), TypeError, "'X_train' must be a sparse matrix."),
            (dict(X_train=Xtr[:, :49]), ValueError, "'X_train' and 'X_test' should have the same number of columns."),
            (dict(X_train=Xtr[:29]), ValueError, "'X_train' and 'X_test' should have the same number of rows."),
            (no_metric, ValueError, "Must pass at least one metric to calculate."),
            (dict(seed=0), ValueError, counts_rule),
            (dict(k=0), ValueError, counts_rule),
            (dict(min_pos_test=0), ValueError, counts_rule),
            (dict(min_items_pool=0), ValueError, counts_rule),
            (dict(k=51), ValueError, "'k' should be smaller than the number of items."),
            (dict(item_biases=[0.0] * 50), TypeError, "'item_biases' must be a numpy array."),
            (dict(item_biases=np.ones((50, 1, 1), dtype=np.float32)), ValueError, "'item_biases' should be a 1-d array."),
            (dict(item_biases=np.ones(0, dtype=np.float32)), ValueError, "'item_biases' is empty."),
            (dict(item_biases=np.ones(10, dtype=np.float32)), ValueError, "Number of items in 'item_biases' must match with 'X_test'."),
            (dict(novelty=True, item_popularity=np.zeros(49, dtype=np.int64)), ValueError, pop_len),
            (dict(avg_popularity=True, item_popularity=np.zeros((50, 1), dtype=np.int64)), ValueError, pop_len),
            (dict(novelty=True, item_popularity=np.zeros(50)), TypeError, "'item_popularity' must hold integer counts."),
            (dict(novelty=True, item_popularity=np.full(50, 31, dtype=np.int64)), ValueError, pop_range),
            (dict(avg_popularity=True, item_popularity=np.full(50, -1, dtype=np.int32)), ValueError, pop_range),
            # several faults: the column count comes first here (the device front-end reports the metric guard first)
            (dict(B=B[:, :3], **no_metric), ValueError, "'A' and 'B' must have the same number of columns.")):
        with pytest.raises(exc, match=_exact(msg)):
            call(**kw)

    # the warnings: the call goes on past each, up to a bad item_popularity, which is checked after all of them
    for kw, msg in ((dict(A=np.vstack([A, A[:1]])), "'A' has more users than 'X_test'."),
                    (dict(B=np.vstack([B, B[:1]])), "'B' has more items than 'X_test'."),
                    (dict(X_train=vstack([Xtr, Xtr[:1]]).tocsr()), "'X_train' mas more rows than 'X_test'."),
                    (dict(item_biases=np.ones(51, dtype=np.float32)), "'item_biases' has more items than 'X_test'.")):
        with pytest.warns(UserWarning, match=_exact(msg)), pytest.raises(ValueError, match=_exact(pop_len)):
            call(novelty=True, item_popularity=np.zeros(49, dtype=np.int64), **kw)


def test_shard_bounds_partition():
    from recometrics_b200.dist import shard_bounds
    for m in (1, 7, 128, 1000, 1000003):
        for w in (1, 2, 3, 8):
            blocks = [shard_bounds(m, w, r) for r in range(w)]
            assert blocks[0][0] == 0 and blocks[-1][1] == m
            assert all(blocks[i][1] == blocks[i + 1][0] for i in range(w - 1))
            sizes = [e - b for b, e in blocks]
            assert max(sizes) - min(sizes) <= 1


def test_device_front_end_needs_a_gpu():
    """calc_reco_metrics_device has no CPU path either: without a CUDA device it raises before touching anything."""
    import numpy as np
    import pytest
    import torch
    import recometrics_b200 as rb
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(RuntimeError, match="CUDA device"):
        rb.calc_reco_metrics_device(None, None, np.zeros((2, 2)), np.zeros((2, 2)))


def test_cpp_shim_is_a_drop_in_for_the_reference_declarations(tmp_path):
    """include/recometrics_b200_shim.hpp defines calc_metrics_float / _double / get_has_openmp with the parameter lists of the
    reference's src/recometrics_signatures.hpp:46-98 (included first when the reference is mounted: a mismatch makes the
    address-of expressions in tests/shim/shim_dropin.cpp ambiguous) and the template Rwrapper.cpp instantiates; linked against
    the C-ABI library the calls throw std::runtime_error when there is no CUDA device instead of computing on the CPU."""
    import os
    import shutil
    import subprocess
    import recometrics_b200 as rb
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
    if cxx is None:
        import pytest
        pytest.skip("no g++")
    libdir = os.path.dirname(rb.native_library_path())
    exe = str(tmp_path / "shim_dropin")
    cmd = [cxx, "-std=c++11", "-O1", "-Wall", "-I", os.path.join(root, "include")]
    ref_src = "/root/reference/src"
    if os.path.exists(os.path.join(ref_src, "recometrics_signatures.hpp")):
        cmd += ["-DHAVE_REFERENCE_HEADER", "-I", ref_src]
    tail = [os.path.join(root, "tests", "shim", "shim_dropin.cpp"), "-L", libdir, "-lrecometrics_b200", "-Wl,-rpath," + libdir]
    # as the Python build would use it, and as an R build would (undefined metrics written as NA_REAL, hpp:75-80)
    for tag, extra in (("py", []), ("r", ["-DRMB200_SHIM_NAN_BITS=0x7FF00000000007A2ull"])):
        subprocess.run(cmd + extra + tail + ["-o", exe + tag], check=True, capture_output=True, text=True)
        run = subprocess.run([exe + tag], capture_output=True, text=True, timeout=120)
        assert run.returncode == 0, run.stdout + run.stderr
        if rb.device_count() == 0:
            assert "threw runtime_error" in run.stdout
        elif tag == "r":
            assert "na_bits=ok" in run.stdout, run.stdout


_CY_PROBE = r"""
import sys, numpy as np
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[2])
import cpp_funs                                   # the reference's wrapper.pyx, unmodified, linked against librecometrics_b200.so
from tools import synth
d = synth.make(1, m=300, n=500, p=8)
print("HAS", int(cpp_funs._get_has_openmp()))
try:
    out = cpp_funs.calc_reco_metrics(d["A"], 8, d["B"], 8, d["X_train"], d["X_test"], k_metrics=5, precision=True, ndcg=True,
                                     average_precision=True, break_ties_with_noise=False)
    np.save(sys.argv[3], np.stack([out[0], out[3], out[5]]))
    print("COMPUTED")
except RuntimeError as e:
    print("RuntimeError:", e)
"""


def run_reference_cython_wrapper(tmp_path):
    """(shared with the GPU suite) Runs the reference's own Cython entry point, cpp_funs.calc_reco_metrics, from the build
    of oracle/build_ref_cython.py in a fresh interpreter.  Returns (stdout, path of the saved P@K / AP@K / NDCG@K rows)."""
    import glob
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cy_dir = os.path.join(root, "oracle", "_ref", "cy_b200")
    if not glob.glob(os.path.join(cy_dir, "cpp_funs*.so")):
        if os.path.isdir("/root/reference/recometrics"):
            subprocess.run([sys.executable, os.path.join(root, "oracle", "build_ref_cython.py")], check=True, capture_output=True)
        else:
            import pytest
            pytest.skip("oracle/_ref/cy_b200 was not built (no /root/reference in the build container)")
    out = str(tmp_path / "cy_rows.npy")
    run = subprocess.run([sys.executable, "-c", _CY_PROBE, cy_dir, root, out], capture_output=True, text=True, timeout=300)
    assert run.returncode == 0, run.stdout + run.stderr
    return run.stdout, out


def test_reference_cython_wrapper_binds_the_library(rb, tmp_path):
    """The north-star's boundary, literally: the reference's existing Cython wrapper (recometrics/wrapper.pyx, cythonized and
    compiled unmodified by oracle/build_ref_cython.py) calling the C-ABI through include/recometrics_b200_shim.hpp.  Without
    a CUDA device its metric entry point raises RuntimeError (Cython's `except +` on the shim's exception) -- it does not
    compute on the CPU."""
    stdout, _ = run_reference_cython_wrapper(tmp_path)
    if rb.device_count() == 0:
        assert "HAS 0" in stdout and "RuntimeError:" in stdout and "no CUDA device" in stdout, stdout
    else:
        assert "COMPUTED" in stdout, stdout


def test_reference_python_package_runs_on_the_library(rb, tmp_path):
    """One level further up: the reference's own Python package (recometrics/__init__.py, symlinked -- not copied -- next to the
    cpp_funs module built by oracle/build_ref_cython.py) imports and validates as usual, and its calc_reco_metrics reaches
    librecometrics_b200.so: on a box without a GPU the call ends in the library's RuntimeError, after the reference's own
    argument handling (bias folding, CSR canonicalisation, dtype rule) has run.  Needs /root/reference (build container only)."""
    import glob
    import os
    import subprocess
    import sys
    import pytest
    ref_init = "/root/reference/recometrics/__init__.py"
    if not os.path.exists(ref_init):
        pytest.skip("no /root/reference here")
    run_reference_cython_wrapper(tmp_path)                       # makes sure oracle/_ref/cy_b200 is built
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    so = glob.glob(os.path.join(root, "oracle", "_ref", "cy_b200", "cpp_funs*.so"))[0]
    pkg = tmp_path / "site" / "recometrics"
    pkg.mkdir(parents=True)
    os.symlink(ref_init, pkg / "__init__.py")
    os.symlink(so, pkg / os.path.basename(so))
    probe = (
        "import sys; sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[2])\n"
        "import numpy as np, recometrics\n"
        "from tools import synth\n"
        "d = synth.make(2, m=200, n=400, p=8)\n"
        "assert recometrics.cpp_funs.__file__.startswith(sys.argv[1])\n"
        "try:\n"
        "    df = recometrics.calc_reco_metrics(d['X_train'], d['X_test'], d['A'], d['B'], k=5, item_biases=d['item_biases'],\n"
        "                                       break_ties_with_noise=False, nthreads=1)\n"
        "    print('COMPUTED', list(df.columns))\n"
        "except RuntimeError as e:\n"
        "    print('RuntimeError:', e)\n")
    env = dict(os.environ)                                       # ($ORIGIN in the module's rpath follows the symlink's directory)
    env["LD_LIBRARY_PATH"] = os.path.dirname(rb.native_library_path()) + os.pathsep + env.get("LD_LIBRARY_PATH", "")
    run = subprocess.run([sys.executable, "-c", probe, str(tmp_path / "site"), root], capture_output=True, text=True, timeout=300, env=env)
    assert run.returncode == 0, run.stdout + run.stderr
    if rb.device_count() == 0:
        assert "RuntimeError:" in run.stdout and "no CUDA device" in run.stdout, run.stdout + run.stderr
    else:
        assert "COMPUTED ['P@5', 'AP@5', 'NDCG@5']" in run.stdout, run.stdout + run.stderr
