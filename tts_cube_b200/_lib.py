"""ctypes binding of libcube_vocoder.so (C ABI: include/cube_vocoder.h).

There is deliberately no fallback: if the shared library is missing or cannot be loaded, importing
any compute entry point raises.  The library is built in-tree by ``__graft_entry__.build()``.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcube_vocoder.so")

MAX_UPS, MAX_RBK, MAX_DIL, MAX_FLOWS = 8, 8, 8, 8
ARCH_HIFIGAN, ARCH_PWN_STUDENT, ARCH_WAVERNN, ARCH_UPSAMPLENET = 0, 1, 2, 3
HEADS = {"mol": 0, "gm": 1, "mulaw": 2, "raw": 3}
MATH_FP32_SIMT, MATH_TC_SPLIT16 = 0, 1


class VocConfig(C.Structure):
    """cube_voc_config; ``struct_size`` is filled in by the constructor (the library rejects a mismatch)."""
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("arch", C.c_int32), ("math", C.c_int32), ("num_mels", C.c_int32),
        ("upsample_initial_channel", C.c_int32), ("n_ups", C.c_int32),
        ("upsample_rates", C.c_int32 * MAX_UPS), ("upsample_kernel_sizes", C.c_int32 * MAX_UPS),
        ("resblock_type", C.c_int32), ("n_resblock_kernels", C.c_int32),
        ("resblock_kernel_sizes", C.c_int32 * MAX_RBK), ("n_dilations", C.c_int32 * MAX_RBK),
        ("resblock_dilations", (C.c_int32 * MAX_DIL) * MAX_RBK),
        ("n_flows", C.c_int32), ("flow_blocks", C.c_int32 * MAX_FLOWS),
        ("res_channels", C.c_int32), ("gate_channels", C.c_int32), ("skip_channels", C.c_int32),
        ("kernel_size", C.c_int32), ("front_kernel", C.c_int32),
        ("dilation_base", C.c_int32), ("dilation_cycle", C.c_int32),
        ("n_upsample", C.c_int32), ("upsample_scales", C.c_int32 * 4),
        ("wrnn_layers", C.c_int32), ("wrnn_size", C.c_int32), ("wrnn_upsample", C.c_int32),
        ("wrnn_upsample_low", C.c_int32), ("wrnn_use_lowres", C.c_int32), ("wrnn_head", C.c_int32),
    ]

    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self.struct_size = C.sizeof(VocConfig)


class MelConfig(C.Structure):
    _fields_ = [("struct_size", C.c_uint32),
                ("n_fft", C.c_int32), ("win_size", C.c_int32), ("hop_size", C.c_int32), ("n_mels", C.c_int32),
                ("pad_left", C.c_int32), ("pad_right", C.c_int32), ("log10_out", C.c_int32), ("layout", C.c_int32),
                ("pad_mode", C.c_int32),
                ("mag_eps", C.c_float), ("floor_val", C.c_float), ("pad_value", C.c_float), ("preemph", C.c_float)]

    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self.struct_size = C.sizeof(MelConfig)


class CubeVocError(RuntimeError):
    pass


_lib = None

# name -> (restype, argtypes); every symbol include/cube_vocoder.h declares
_P = C.c_void_p
SYMBOLS = {
    "cube_voc_create": (C.c_int, [C.POINTER(_P), C.POINTER(VocConfig), C.c_int]),
    "cube_voc_load_weight": (C.c_int, [_P, C.c_char_p, _P, C.POINTER(C.c_int64), C.c_int]),
    "cube_voc_finalize": (C.c_int, [_P]),
    "cube_voc_out_len": (C.c_int64, [_P, C.c_int64]),
    "cube_voc_forward": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int, C.c_int64, _P]),
    "cube_voc_forward_host": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int, C.c_int64]),
    "cube_voc_hifigan_support": (C.c_int, [C.POINTER(VocConfig), C.c_int64, C.c_int64, C.POINTER(C.c_int64),
                                           C.POINTER(C.c_int64)]),
    "cube_voc_forward_range": (C.c_int, [_P, _P, _P, C.POINTER(C.c_int64), C.POINTER(C.c_int64), _P, _P, C.c_int,
                                         C.c_int64, _P]),
    "cube_voc_get_cond": (C.c_int, [_P, _P, C.c_int, C.c_int64, _P]),
    "cube_wavernn_out_len": (C.c_int64, [_P, C.c_int64, C.c_int64]),
    "cube_wavernn_forward": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_int64, C.c_int64, _P]),
    "cube_wavernn_max_batch": (C.c_int, [_P]),
    "cube_voc_last_launches": (C.c_int64, [_P]),
    "cube_voc_workspace_bytes": (C.c_int64, [_P]),
    "cube_voc_set_profile": (C.c_int, [_P, C.c_int]),
    "cube_voc_get_profile": (C.c_int, [_P, _P, _P, C.c_int]),
    "cube_voc_destroy": (None, [_P]),
    "cube_voc_last_error": (C.c_char_p, []),
    "cube_voc_build_info": (C.c_char_p, []),
    "cube_mulaw_encode": (C.c_int, [_P, _P, C.c_int64, _P]),
    "cube_mulaw_decode": (C.c_int, [_P, _P, C.c_int64, _P]),
    "cube_raw_encode": (C.c_int, [_P, _P, C.c_int64, _P]),
    "cube_raw_decode": (C.c_int, [_P, _P, C.c_int64, _P]),
    "cube_mol_sample": (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_int, C.c_float, C.c_float, _P]),
    "cube_gaussian_sample": (C.c_int, [_P, _P, _P, C.c_int64, _P]),
    "cube_categorical_sample": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int, _P]),
    "cube_wav_to_int16": (C.c_int, [_P, _P, C.c_int64, _P]),
    "cube_mel_create": (C.c_int, [C.POINTER(_P), C.POINTER(MelConfig), _P, _P, C.c_int]),
    "cube_mel_out_frames": (C.c_int64, [_P, C.c_int64]),
    "cube_mel_forward": (C.c_int, [_P, _P, C.POINTER(C.c_int32), _P, C.c_int, C.c_int64, C.c_int64, _P]),
    "cube_mel_destroy": (None, [_P]),
}


def lib() -> C.CDLL:
    """Load (once) and return the shared library; raise loudly if it is not there."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CubeVocError(
                f"{LIB_PATH} not found - build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  tts_cube_b200 has no CPU or PyTorch fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(l, name)  # AttributeError if the ABI and the header drifted apart
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise CubeVocError(lib().cube_voc_last_error().decode("utf-8", "replace"))


def build_info() -> str:
    return lib().cube_voc_build_info().decode()
