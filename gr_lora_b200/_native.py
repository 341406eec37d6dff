"""ctypes view of liblora_b200.so (include/lora_b200.h).  No fallback: if the library cannot be
loaded the import fails loudly."""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build


class Config(C.Structure):
    """struct lora_b200_config (include/lora_b200.h)."""
    _fields_ = [
        ("samp_rate", C.c_float), ("bandwidth", C.c_uint32), ("sf", C.c_uint8), ("implicit", C.c_uint8),
        ("cr", C.c_uint8), ("crc", C.c_uint8), ("reduced_rate", C.c_uint8), ("disable_drift_correction", C.c_uint8),
        ("demod", C.c_uint8), ("reserved0", C.c_uint8), ("n_streams", C.c_uint32), ("device", C.c_int32),
        ("max_items_per_call", C.c_uint32), ("max_frames_per_call", C.c_uint32), ("trace_capacity", C.c_uint32),
    ]


class Step(C.Structure):
    _fields_ = [("state", C.c_int32), ("consumed", C.c_int32), ("bin", C.c_int32), ("fine_sync", C.c_int32),
                ("metric", C.c_float)]


class GatewayConfig(C.Structure):
    """struct lora_b200_gateway_config (include/lora_b200.h)."""
    _fields_ = [
        ("samp_rate", C.c_float), ("center_freq", C.c_float), ("channel_list", C.POINTER(C.c_float)),
        ("n_channels", C.c_uint32), ("bandwidth", C.c_uint32), ("decimation", C.c_uint32), ("sf_mask", C.c_uint32),
        ("reduced_rate_mask", C.c_uint32), ("implicit", C.c_uint8), ("cr", C.c_uint8), ("crc", C.c_uint8), ("demod", C.c_uint8),
        ("conj", C.c_uint8), ("disable_drift_correction", C.c_uint8), ("reserved", C.c_uint8 * 2), ("device", C.c_int32),
        ("max_in_per_call", C.c_uint32), ("max_frames_per_call", C.c_uint32),
    ]


FRAME_CB = C.CFUNCTYPE(None, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint8), C.c_size_t)

OK, EINVAL, ECUDA, ENOMEM, EUNSUPPORTED, EOVERFLOW = 0, -1, -2, -3, -4, -5
DEMOD_GRADIENT, DEMOD_FFT = 0, 1
STATES = ["DETECT", "SYNC", "FIND_SFD", "PAUSE", "DECODE_HEADER", "DECODE_PAYLOAD", "STOP"]

# every symbol include/lora_b200.h declares: name -> (restype, argtypes)
_vp, _u32, _sz, _i = C.c_void_p, C.c_uint32, C.c_size_t, C.c_int
SIGNATURES = {
    "lora_b200_create": (_vp, [C.POINTER(Config)]),
    "lora_b200_destroy": (None, [_vp]),
    "lora_b200_last_error": (C.c_char_p, []),
    "lora_b200_abi_version": (_i, []),
    "lora_b200_samples_per_symbol": (_u32, [_vp]),
    "lora_b200_bins": (_u32, [_vp]),
    "lora_b200_decimation": (_u32, [_vp]),
    "lora_b200_banner": (_i, [_vp, C.c_char_p, _sz]),
    "lora_b200_set_sf": (_i, [_vp, C.c_uint8]),
    "lora_b200_set_samp_rate": (_i, [_vp, C.c_float]),
    "lora_b200_tables_bytes": (_sz, [_vp]),
    "lora_b200_tables_build_host": (_sz, [C.POINTER(Config), _vp, _sz]),
    "lora_b200_tables_device_ptr": (_vp, [_vp]),
    "lora_b200_tables_export": (_i, [_vp, _vp, _sz]),
    "lora_b200_tables_import": (_i, [_vp, _vp, _sz]),
    "lora_b200_tables_commit": (_i, [_vp]),
    "lora_b200_demod_fft_dev": (_i, [_vp, _vp, _sz, _vp, _vp, _vp]),
    "lora_b200_demod_fft_host": (_i, [_vp, _vp, _sz, _vp, _vp]),
    "lora_b200_demod_fft_host_sc16": (_i, [_vp, _vp, C.c_float, _sz, _vp, _vp]),
    "lora_b200_demod_gradient_dev": (_i, [_vp, _vp, _sz, _vp, _vp]),
    "lora_b200_ifreq_dev": (_i, [_vp, _vp, _sz, _u32, _vp, _vp]),
    "lora_b200_tx_symbols_dev": (_i, [_vp, _vp, _vp, _vp, C.c_float, C.c_uint64, _sz, _vp, _vp]),
    "lora_b200_tx_expand_dev": (_i, [_vp, _vp, _u32, _sz, C.c_float, C.c_uint64, _sz, _vp, _vp]),
    "lora_b200_decode_codewords_dev": (_i, [_vp, _vp, _vp, _sz, _vp, _vp, _sz, _vp, _sz, _vp, _vp]),
    "lora_b200_deinterleave_dev": (_i, [_vp, _vp, _u32, _u32, _sz, _vp, _vp]),
    "lora_b200_work": (_i, [_vp, _u32, _vp, _sz, C.POINTER(_sz), FRAME_CB, _vp]),
    "lora_b200_work_batch": (_i, [_vp, _vp, _sz, _sz, _i, C.POINTER(_sz), FRAME_CB, _vp]),
    "lora_b200_work_batch_sc16": (_i, [_vp, _vp, C.c_float, _sz, _sz, _i, C.POINTER(_sz), FRAME_CB, _vp]),
    "lora_b200_work_batch_sc8": (_i, [_vp, _vp, C.c_float, _sz, _sz, _i, C.POINTER(_sz), FRAME_CB, _vp]),
    "lora_b200_frames_last": (_sz, [_vp, C.POINTER(_vp)]),
    "lora_b200_stream_state": (_i, [_vp, _u32]),
    "lora_b200_reset": (_i, [_vp]),
    "lora_b200_set_cfo_estimate": (_i, [_vp, _i]),
    "lora_b200_last_cfo": (_i, [_vp, _u32, C.POINTER(C.c_float), C.POINTER(C.c_uint32)]),
    "lora_b200_stdout_last": (_i, [_vp, _u32, C.c_char_p, _sz]),
    "lora_b200_trace_read": (_i, [_vp, _u32, C.POINTER(Step), _sz, C.POINTER(_sz)]),
    "lora_b200_launch_count": (C.c_uint64, [_vp]),
    "lora_b200_channelizer_create": (_vp, [C.c_float, C.c_float, C.POINTER(C.c_float), _u32, _u32, _u32, C.c_int32]),
    "lora_b200_channelizer_destroy": (None, [_vp]),
    "lora_b200_channelizer_last_error": (C.c_char_p, []),
    "lora_b200_channelizer_ntaps": (_u32, [_vp]),
    "lora_b200_channelizer_taps": (_i, [_vp, C.POINTER(C.c_float), _sz]),
    "lora_b200_channelizer_apply_cfo": (_i, [_vp, _u32, C.c_float]),
    "lora_b200_channelizer_set_conjugate": (_i, [_vp, _i]),
    "lora_b200_channelizer_work_dev": (_i, [_vp, _vp, _sz, _vp, _sz, C.POINTER(_sz), _vp]),
    "lora_b200_channelizer_work_host": (_i, [_vp, _vp, _sz, C.POINTER(_sz)]),
    "lora_b200_channelizer_output": (_vp, [_vp, _u32, C.POINTER(_sz)]),
    "lora_b200_channelizer_read_output": (_i, [_vp, _u32, _vp, _sz]),
    "lora_b200_channelizer_launch_count": (C.c_uint64, [_vp]),
    "lora_b200_gateway_create": (_vp, [C.POINTER(GatewayConfig)]),
    "lora_b200_gateway_destroy": (None, [_vp]),
    "lora_b200_gateway_reset": (_i, [_vp]),
    "lora_b200_gateway_work": (_i, [_vp, _vp, _sz, _i, C.POINTER(_sz)]),
    "lora_b200_gateway_frames_last": (_sz, [_vp, C.POINTER(_vp)]),
    "lora_b200_gateway_position": (_i, [_vp, _u32, _u32, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]),
    "lora_b200_gateway_timing": (_i, [_vp, C.POINTER(C.c_float), _sz]),
}

_lib = None


def lib() -> C.CDLL:
    """Load (building first if the .so is missing or stale and nvcc is present)."""
    global _lib
    if _lib is None:
        try:
            path = _build.build()
        except Exception as exc:  # stale-check failed but an older build may exist
            if not _build.LIB.exists():
                raise ImportError(f"liblora_b200.so is missing and could not be built: {exc}") from exc
            path = _build.LIB
        alt = os.environ.get("LORA_B200_LIB")      # A/B runs of an alternative build of the same sources (tools/k1_ab.py)
        if alt:
            path = alt
        L = C.CDLL(str(path))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)       # AttributeError here = ABI mismatch: fail loudly
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


class LoraB200Error(RuntimeError):
    def __init__(self, code: int, where: str):
        msg = lib().lora_b200_last_error().decode(errors="replace")
        super().__init__(f"{where} failed ({code}): {msg}")
        self.code = code


def check(code: int, where: str) -> int:
    if code < 0:
        raise LoraB200Error(code, where)
    return code
