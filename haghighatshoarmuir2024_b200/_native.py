"""ctypes binding of libmicloc_b200.so (the C-ABI declared in include/micloc_b200.h).

The product path has NO CPU fallback: if the CUDA library is missing or a call
fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
# MICLOC_B200_LIB points the loader at an instrumented build of the same library (tools/role_timing.py)
LIB_PATH = os.environ.get("MICLOC_B200_LIB") or os.path.join(CSRC, "libmicloc_b200.so")

F32, I16, I32 = 0, 1, 2
ERR_SHAPE, ERR_CONFIG, ERR_CUDA, ERR_UNSUPPORTED, ERR_OVERFLOW = -1, -2, -3, -4, -5

_dp = C.POINTER(C.c_double)
_vp = C.c_void_p
_i64 = C.c_int64
_i32 = C.c_int32


class SnnConfig(C.Structure):
    _fields_ = [
        ("num_mic", _i32), ("kernel_len", _i32), ("stht_kernel", _dp),
        ("n_sections", _i32), ("sos", _dp),
        ("robust_width", _i32), ("bipolar", _i32),
        ("neuron_decay", C.c_double), ("neuron_scale", C.c_double), ("neuron_len", _i32),
        ("num_doa", _i32), ("bf_mat", _dp),
    ]


class XyloConfig(C.Structure):
    _fields_ = [
        ("num_mic", _i32), ("kernel_len", _i32), ("stht_kernel", _dp),
        ("num_bands", _i32), ("n_sections", _i32), ("sos", _dp),
        ("n_ba", _i32), ("ba_b", _dp), ("ba_a", _dp),
        ("robust_width", _i32), ("bipolar", _i32),
        ("num_hidden", _i32), ("num_doa", _i32),
        ("w_in", C.POINTER(C.c_int8)), ("w_rec", C.POINTER(C.c_int8)),
        ("threshold", C.POINTER(C.c_int16)), ("dash_syn", C.POINTER(C.c_int8)),
        ("dash_mem", C.POINTER(C.c_int8)), ("bias", C.POINTER(C.c_int16)),
        ("weight_shift_in", _i32), ("weight_shift_rec", _i32), ("max_spikes", _i32),
    ]


class SynthConfig(C.Structure):
    _fields_ = [
        ("num_mic", _i32), ("r_vec", _dp), ("theta_vec", _dp), ("fs", C.c_double), ("speed", C.c_double),
        ("clip_len", _i64), ("n_targets", _i32), ("mode", _i32), ("source_kind", _i32), ("sine_freq", C.c_double),
    ]


class DesignTemplate(C.Structure):
    _fields_ = [
        ("num_mic", _i32), ("r_vec", _dp), ("theta_vec", _dp), ("speed", C.c_double),
        ("T", _i64), ("time_dev", _vp), ("sig_dev", _vp),
    ]


# every symbol include/micloc_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "micloc_snn_create": (C.c_int, [C.POINTER(SnnConfig), C.c_int, C.POINTER(_vp)]),
    "micloc_snn_destroy": (C.c_int, [_vp]),
    "micloc_snn_set_bf": (C.c_int, [_vp, _dp, _i32]),
    "micloc_snn_run": (C.c_int, [_vp, _vp, C.c_int, _i64, _i64, _vp, _vp, _vp, _vp, C.c_int, _vp]),
    "micloc_snn_refine": (C.c_int, [_vp, _vp, C.c_int, _i64, _i64, _vp, _vp, _vp, _vp, C.POINTER(_i64), _vp]),
    "micloc_snn_refined_count": (_i64, [_vp]),
    "micloc_snn_run_taps": (C.c_int, [_vp, _vp, C.c_int, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "micloc_snn_run_host": (C.c_int, [_vp, _vp, C.c_int, _i64, _i64, _vp, _vp, _vp, _vp, C.c_int]),
    "micloc_snn_gram": (C.c_int, [_vp, _vp, C.c_int, _i64, _i64, _i64, _vp, _vp]),
    "micloc_doa_histogram": (C.c_int, [_vp, _i64, _i32, _vp, C.c_int, _vp]),
    "micloc_snn_stream_create": (C.c_int, [_vp, _i64, C.c_double, C.c_double, C.c_double, C.POINTER(_vp)]),
    "micloc_snn_stream_destroy": (C.c_int, [_vp]),
    "micloc_snn_stream_reset": (C.c_int, [_vp, _vp]),
    "micloc_snn_stream_latency": (C.c_int, [_vp]),
    "micloc_snn_stream_push": (C.c_int, [_vp, _vp, C.c_int, _i64, _i32, _vp, _vp, _vp, _vp, _vp, C.POINTER(_i64), _vp]),
    "micloc_snn_stream_flush": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(_i64), C.POINTER(_i32), _vp]),
    "micloc_snn_streams_create": (C.c_int, [_vp, _i32, _i64, C.c_double, C.c_double, C.c_double, C.POINTER(_vp)]),
    "micloc_snn_streams_destroy": (C.c_int, [_vp]),
    "micloc_snn_streams_latency": (C.c_int, [_vp]),
    "micloc_snn_streams_reset": (C.c_int, [_vp, _vp, _i32, _vp]),
    "micloc_snn_streams_push": (C.c_int, [_vp, _vp, C.c_int, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "micloc_snn_streams_flush": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "micloc_snn_mb_streams_create": (C.c_int, [C.POINTER(_vp), _i32, _i32, _dp, _dp, _i32, _i64, C.POINTER(_vp)]),
    "micloc_snn_mb_streams_destroy": (C.c_int, [_vp]),
    "micloc_snn_mb_streams_latency": (C.c_int, [_vp]),
    "micloc_snn_mb_streams_reset": (C.c_int, [_vp, _vp, _i32, _vp]),
    "micloc_snn_mb_streams_push": (C.c_int, [_vp, _vp, C.c_int, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                             _vp]),
    "micloc_snn_mb_streams_flush": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "micloc_envelope":(C.c_int, [_vp, _i64, _i32, C.c_double, C.c_double, C.c_double, _vp, _vp, C.c_int, _vp]),
    "micloc_filterbank": (C.c_int, [_vp, C.c_int, _i64, _i64, _i32, _i32, _i32, _i32, _dp, _vp, _vp, C.c_int, _vp]),
    "micloc_power_fuse": (C.c_int, [_vp, _i32, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int, _vp]),
    "micloc_synth_clips": (C.c_int, [C.POINTER(SynthConfig), _i64, _vp, _vp, _vp, _vp, _vp, C.c_uint64, _vp, _vp,
                                     C.c_float, _vp, C.c_int, _vp]),
    "micloc_rzcc_encode_f64": (C.c_int, [_vp, _i64, _i64, _i32, _i32, _i32, _vp, C.c_int, _vp]),
    "micloc_hilbert_beamform": (C.c_int, [_vp, _vp, C.c_int, _i64, _i64, _dp, _dp, _i32, _vp, _vp, _vp, _vp]),
    "micloc_hilbert_set_bf": (C.c_int, [_vp, _dp, _dp, _i32]),
    "micloc_hilbert_localize": (C.c_int, [_vp, _vp, C.c_int, _i64, _i64, _i64, C.c_int, _vp, _vp, _vp, _vp, _vp]),
    "micloc_design_templates": (C.c_int, [C.POINTER(DesignTemplate), _vp, _i64, _vp, C.c_int, _vp]),
    "micloc_snn_design": (C.c_int, [_vp, C.POINTER(DesignTemplate), _vp, _i64, _vp, _vp, _vp]),
    "micloc_hilbert_design": (C.c_int, [_vp, C.POINTER(DesignTemplate), _vp, _i64, C.c_int, _vp, _vp, _vp]),
    "micloc_design_vectors": (C.c_int, [C.c_int, _vp, _i32, _i64, _vp, _vp, C.c_int, _vp]),
    "micloc_xylo_create": (C.c_int, [C.POINTER(XyloConfig), C.c_int, C.POINTER(_vp)]),
    "micloc_xylo_destroy": (C.c_int, [_vp]),
    "micloc_xylo_run": (C.c_int, [_vp, _vp, C.c_int, _i64, _i64, C.c_int, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp]),
    "micloc_xylo_process": (C.c_int, [_vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _i32, _vp]),
    "micloc_xylo_streams_create": (C.c_int, [_vp, _i32, _i64, C.POINTER(_vp)]),
    "micloc_xylo_streams_destroy": (C.c_int, [_vp]),
    "micloc_xylo_streams_latency": (C.c_int, [_vp]),
    "micloc_xylo_streams_reset": (C.c_int, [_vp, _vp, _i32, _vp]),
    "micloc_xylo_streams_push": (C.c_int, [_vp, _vp, C.c_int, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp]),
    "micloc_xylo_streams_flush": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp]),
    "micloc_hilbert_streams_create": (C.c_int, [C.POINTER(_vp), _i32, _i32, _dp, _dp, _i32, _i64, C.POINTER(_vp)]),
    "micloc_hilbert_streams_destroy": (C.c_int, [_vp]),
    "micloc_hilbert_streams_latency": (C.c_int, [_vp]),
    "micloc_hilbert_streams_reset": (C.c_int, [_vp, _vp, _i32, _vp]),
    "micloc_hilbert_streams_push": (C.c_int, [_vp, _vp, C.c_int, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                              _vp, _vp]),
    "micloc_last_error": (C.c_char_p, []),
    "micloc_version": (C.c_int, []),
    "micloc_launch_count": (_i64, []),
    "micloc_snn_last_kernel_ms": (C.c_int, [_vp, C.POINTER(C.c_float), C.POINTER(_i32)]),
    "micloc_snn_enable_timing": (C.c_int, [_vp, C.c_int]),
    "micloc_snn_debug_counters": (C.c_int, [_vp, C.POINTER(C.c_uint64)]),
    "micloc_snn_debug_cta_times": (C.c_int, [_vp, C.POINTER(C.c_uint64), _i32]),
    "micloc_fp32_peak": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_double)]),
}

_lib = None


class MiclocError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"micloc_b200 error {code}: {msg}")
        self.code = code
        self.msg = msg


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/ for sm_100a with nvcc (csrc/Makefile)."""
    args = ["make", "-j", "6", "-C", CSRC] + (["-B"] if force else [])
    subprocess.run(args, check=True, stdout=None if verbose else subprocess.DEVNULL)
    return LIB_PATH


def lib():
    """Load the CUDA library; there is no fallback when it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). The hot path has no CPU fallback.")
        _lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(_lib, name)
            fn.restype = res
            fn.argtypes = args
    return _lib


def check(rc: int) -> None:
    """Map a negative status to the exception the reference would raise."""
    if rc == 0:
        return
    msg = lib().micloc_last_error().decode("utf-8", "replace")
    if rc == ERR_SHAPE or rc == ERR_CONFIG:
        raise ValueError(msg)
    raise MiclocError(rc, msg)
