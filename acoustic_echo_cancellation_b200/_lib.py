"""ctypes binding of ``libaec_b200.so`` (the C ABI declared in ``include/aec_b200.h``).

The shared library is built in-tree by ``make -C acoustic_echo_cancellation_b200/csrc``
(or ``__graft_entry__.build()``).  There is no CPU fallback: if the library is missing
or a call fails, the error is raised to the caller.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# AEC_B200_LIB lets developer tooling A/B a differently built library; default is the in-tree build
LIB_PATH = os.environ.get("AEC_B200_LIB") or os.path.join(_HERE, "libaec_b200.so")

ALGO_NLMS = 0
ALGO_KALMAN = 1
ALGO_PBFDAF = 2
ALGO_PBFKF = 3


class AecCfg(C.Structure):
    """Mirror of ``struct aec_cfg`` (include/aec_b200.h)."""

    _fields_ = [
        ("frame", C.c_int32),
        ("partitions", C.c_int32),
        ("algo", C.c_int32),
        ("mu", C.c_float),
        ("delta", C.c_float),
        ("kalman_a", C.c_float),
        ("kalman_lambda", C.c_float),
        ("kalman_c0", C.c_float),
        ("kalman_eps", C.c_float),
        ("erle_skip_hops", C.c_int32),
        ("variant", C.c_int32),
        ("stagger_ns", C.c_int32),
        ("pb_lambda", C.c_float),
        ("reserved", C.c_int32 * 3),
    ]


class AecDelayCfg(C.Structure):
    """Mirror of ``struct aec_delay_cfg`` (include/aec_b200.h)."""

    _fields_ = [("max_delay", C.c_int32), ("margin", C.c_int32), ("min_peak", C.c_float), ("reserved", C.c_int32 * 5)]


class AecError(RuntimeError):
    def __init__(self, code: int, what: str):
        self.code = code
        super().__init__(what)


class WavInfo(C.Structure):
    """Mirror of ``struct aec_wav_info``."""

    _fields_ = [("rate", C.c_int32), ("channels", C.c_int32), ("bits", C.c_int32), ("format", C.c_int32),
                ("frames", C.c_int64), ("data_offset", C.c_int64)]


class Stage2Weights(C.Structure):
    """Mirror of ``struct aec_stage2_weights`` (device pointers to Little_net's state_dict tensors)."""

    _fields_ = [(n, C.c_void_p) for n in ("gru_w_ih", "gru_w_hh", "gru_b_ih", "gru_b_hh", "lin1_w", "lin1_b",
                                           "lin2_w", "lin2_b")]


# every symbol include/aec_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
_I64 = C.c_int64
_I32 = C.c_int32
SIGNATURES = {
    "aec_version": (C.c_int, []),
    "aec_strerror": (C.c_char_p, [C.c_int]),
    "aec_last_cuda_error": (C.c_char_p, []),
    "aec_init": (C.c_int, []),
    "aec_cfg_default": (C.c_int, [C.POINTER(AecCfg), _I32]),
    "aec_num_frames": (_I64, [_I64, _I32]),
    "aec_out_samples": (_I64, [_I64, _I32]),
    "aec_stage1_run": (C.c_int, [_P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _I64, C.POINTER(AecCfg), _P]),
    "aec_stage1_run_features": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _I64, C.POINTER(AecCfg), _P]),
    "aec_host_ctx_create": (C.c_int, [C.POINTER(_P), _I64, _I64]),
    "aec_host_ctx_create_ex": (C.c_int, [C.POINTER(_P), _I64, _I64, _I32, _I32]),
    "aec_host_ctx_destroy": (C.c_int, [_P]),
    "aec_host_ctx_set_deferred": (C.c_int, [_P, _I32]),
    "aec_host_ctx_wait": (C.c_int, [_P]),
    "aec_stage1_run_host": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _I64, C.POINTER(AecCfg)]),
    "aec_stage1_run_host_pcm16": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _I64, C.POINTER(AecCfg)]),
    "aec_stage1_run_host_ex": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _I64, C.POINTER(AecCfg),
                                         C.POINTER(AecDelayCfg), _P, _P]),
    "aec_stage1_run_host_pcm16_ex": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _I64, C.POINTER(AecCfg),
                                               C.POINTER(AecDelayCfg), _P, _P]),
    "aec_delay_cfg_default": (C.c_int, [C.POINTER(AecDelayCfg)]),
    "aec_delay_estimate": (C.c_int, [_P, _P, _P, _I64, _I64, _I64, C.POINTER(AecDelayCfg), _P, _P, _P, _P, _P]),
    "aec_delay_align": (C.c_int, [_P, _P, _P, _I64, _I64, _I64, _I64, _P]),
    "aec_host_alloc": (C.c_int, [C.POINTER(_P), _I64]),
    "aec_host_alloc_ex": (C.c_int, [C.POINTER(_P), _I64, _I32]),
    "aec_host_free": (C.c_int, [_P]),
    "aec_host_is_pinned": (C.c_int, [_P]),
    "aec_wav_probe": (C.c_int, [C.c_char_p, C.POINTER(WavInfo)]),
    "aec_wav_probe_batch": (C.c_int, [C.POINTER(C.c_char_p), _I64, C.POINTER(WavInfo), _I32]),
    "aec_wav_read_pcm16_batch": (C.c_int, [C.POINTER(C.c_char_p), _I64, _P, _I64, _I64, _P, _I32, _I32]),
    "aec_ex_write_batch": (C.c_int, [C.POINTER(C.c_char_p), _I64, _I32, C.POINTER(C.c_char_p), C.POINTER(_P), _P, _P, _I32]),
    "aec_stft": (C.c_int, [_P, _P, _I64, _I64, _I64, _I32, _P]),
    "aec_istft": (C.c_int, [_P, _P, _I64, _I64, _I64, _I32, _P]),
    "aec_features": (C.c_int, [_P, _P, _P, _P, _I64, _I64, _I64, _I32, _I32, C.c_float, C.c_float, _P]),
    "aec_features_dev": (C.c_int, [_P, _P, _P, _P, _I64, _I64, _I64, _I32, _I32, _P, _P, _P]),
    "aec_batch_shift_workspace_bytes": (_I64, []),
    "aec_batch_shift": (C.c_int, [_P, _I64, _I64, _I64, _P, _P, _I64, _P]),
    "aec_stage2_synth_dev": (C.c_int, [_P, _P, _P, _P, _I64, _I64, _I64, _I64, _I32, _I32, _P, _P]),
    "aec_stage2_mask": (C.c_int, [_P, C.POINTER(Stage2Weights), _P, _I64, _I64, _I32, _P]),
    "aec_stage2_synth": (C.c_int, [_P, _P, _P, _P, _I64, _I64, _I64, _I64, _I32, _I32, C.c_float, _P]),
    "aec_bench_fp32_peak": (C.c_int, [C.c_int, C.POINTER(C.c_double), _P]),
    "aec_launch_count": (_I64, [C.c_int]),
}

_lib = None


def load() -> C.CDLL:
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `make -C {os.path.join(_HERE, 'csrc')} -j8` "
            "(or __graft_entry__.build()).  acoustic_echo_cancellation_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc == 0:
        return
    lib = load()
    msg = lib.aec_strerror(rc).decode()
    if rc == -3:
        msg += ": " + lib.aec_last_cuda_error().decode()
    raise AecError(rc, f"{what} failed ({rc}): {msg}")


def default_cfg(frame: int = 512, **overrides) -> AecCfg:
    cfg = AecCfg()
    check(load().aec_cfg_default(C.byref(cfg), frame), "aec_cfg_default")
    for k, v in overrides.items():
        if not hasattr(cfg, k):
            raise TypeError(f"aec_cfg has no field {k!r}")
        setattr(cfg, k, v)
    return cfg
