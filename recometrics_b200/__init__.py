"""recometrics_b200 -- B200-native (sm_100a) per-user evaluation path of david-cortes/recometrics.

Public surface: :func:`calc_reco_metrics` (drop-in for ``recometrics.calc_reco_metrics``),
:func:`calc_reco_metrics_ex` (same call, plus timing / top-K ids / held-out ranks / beyond-accuracy metrics, with
:func:`item_popularity` for the popularity they use) and
:func:`calc_reco_metrics_device` (factors and, optionally, the CSR matrices already resident on the GPU:
``__cuda_array_interface__`` in, torch CUDA tensors out); and, for the step before the evaluation,
:func:`split_reco_train_test` (drop-in for ``recometrics.split_reco_train_test``).
The native library is ``recometrics_b200/librecometrics_b200.so`` (C-ABI in
``include/recometrics_b200.h``); it is loaded lazily on the first call and there is no CPU fallback.
"""
from . import _capi
from .device import DeviceCSR, calc_reco_metrics_device
from .frontend import EvalResult, calc_reco_metrics, calc_reco_metrics_ex, item_popularity
from .splitting import split_reco_train_test

__all__ = ["calc_reco_metrics", "calc_reco_metrics_ex", "calc_reco_metrics_device", "DeviceCSR", "EvalResult", "split_reco_train_test", "device_count",
           "native_library_path", "item_popularity"]
__version__ = "0.1.0"


def device_count():
    """Number of CUDA devices the native library can use (0 -> every compute call raises)."""
    return _capi.device_count()


def native_library_path():
    return _capi.LIB_PATH
