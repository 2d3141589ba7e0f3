"""ctypes binding of libsdrgpu.so (the C ABI declared in include/sdrgpu.h).

The library is the product: if it is missing or no B200 is usable, everything here fails loudly --
there is no CPU fallback and nothing under oracle/ is ever imported from this package.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsdrgpu.so")

HOST, DEVICE = 0, 1
LAYOUT_RESULTS, LAYOUT_CHANNELS = 0, 1
WINDOW_HAMMING, WINDOW_BLACKMAN = 0, 1
DEMOD_NONE, DEMOD_FM, DEMOD_FM_SQUELCH, DEMOD_DQPSK_DECISION, DEMOD_DQPSK_GARDNER = 0, 1, 2, 3, 4
FORMAT_F32, FORMAT_U8, FORMAT_S8, FORMAT_S16LE, FORMAT_AIRSPY_U16LE, FORMAT_AIRSPY_PACKED12 = 0, 1, 2, 3, 4, 5
PRESET_P25_C4FM, PRESET_P25_LSM, PRESET_P25_HDQPSK, PRESET_NBFM, PRESET_DMR = 0, 1, 2, 3, 4
TUNE_FIR_CTAS_PER_SM, TUNE_PFB_CTAS_PER_SM, TUNE_THROTTLE_ALWAYS, TUNE_FIR_TILES_PER_CTA = 0, 1, 2, 3
SYNC_NONE, SYNC_P25_PHASE1, SYNC_P25_PHASE2, SYNC_P25_PHASE2_FRAMED = 0, 1, 2, 3
P2_EVENT_FRAGMENT, P2_EVENT_SYNC_LOSS, P2_EVENT_INVERSION, P2_EVENT_SYNCHRONIZED = 1, 2, 4, 32
(SYNC_EVENT_NONE, SYNC_EVENT_SYNC, SYNC_EVENT_INVERSION_90_CW, SYNC_EVENT_INVERSION_90_CCW, SYNC_EVENT_INVERSION_180,
 SYNC_EVENT_LOST) = range(6)
SQUELCH_ATTACK, SQUELCH_DECAY, SQUELCH_MUTE, SQUELCH_UNMUTE, SQUELCH_CHANGED = 0, 1, 2, 3, 4

OK, ERR_INVALID_ARG, ERR_BAD_STATE, ERR_CUDA, ERR_OVERFLOW, ERR_DESIGN, ERR_NOMEM = range(7)


class FilterDesignException(Exception):
    """Java: io.github.dsheirer.dsp.filter.design.FilterDesignException"""


class IllegalArgumentException(ValueError):
    """Java: IllegalArgumentException"""


class IllegalStateException(RuntimeError):
    """Java: IllegalStateException"""


class CudaError(RuntimeError):
    """CUDA runtime failure / no usable GPU (there is no CPU fallback)."""


class OverflowError_(RuntimeError):
    """More input than the handle was sized for (reference: OVERFLOW state, buffers dropped)."""


class OutputChannel(C.Structure):
    _fields_ = [("bin1", C.c_int), ("bin2", C.c_int), ("frequency_offset_hz", C.c_longlong), ("gain", C.c_double)]


class BankConfig(C.Structure):
    _fields_ = [
        ("n_channels", C.c_int), ("sample_rate", C.c_double), ("decimation", C.c_int),
        ("fir_taps", C.POINTER(C.c_float)), ("n_fir_taps", C.c_int), ("fir_gain", C.c_float),
        ("agc", C.c_int), ("block_size", C.c_int), ("demod", C.c_int),
        ("symbol_rate", C.c_double), ("pll_bandwidth", C.c_double), ("sample_counter_gain", C.c_float),
        ("fm_gain", C.c_float), ("squelch_alpha", C.c_double), ("squelch_threshold_db", C.c_double),
        ("squelch_ramp", C.c_int), ("max_samples_per_call", C.c_int),
    ]


class BankOutput(C.Structure):
    """sdrgpu_bank_output: one bank's outputs of sdrgpu_pipeline_process_routed"""
    _fields_ = [("symbols", C.c_void_p), ("symbol_stride", C.c_int), ("demod", C.c_void_p),
                ("demod_stride_floats", C.c_longlong), ("counts", C.c_void_p)]


_f32p = C.POINTER(C.c_float)
_i32p = C.POINTER(C.c_int)
_u8p = C.POINTER(C.c_uint8)
_vp = C.c_void_p
_vpp = C.POINTER(C.c_void_p)

# name -> (restype, argtypes); every symbol include/sdrgpu.h declares
PROTOTYPES = {
    "sdrgpu_init": (C.c_int, [C.c_int]),
    "sdrgpu_last_error": (C.c_char_p, []),
    "sdrgpu_version": (C.c_char_p, []),
    "sdrgpu_device_count": (C.c_int, [_i32p]),
    "sdrgpu_alloc_pinned": (C.c_int, [_vpp, C.c_size_t]),
    "sdrgpu_free_pinned": (C.c_int, [_vp]),
    "sdrgpu_device_alloc": (C.c_int, [_vpp, C.c_size_t]),
    "sdrgpu_device_free": (C.c_int, [_vp]),
    "sdrgpu_memcpy": (C.c_int, [_vp, _vp, C.c_size_t, C.c_int, C.c_int]),
    "sdrgpu_device_synchronize": (C.c_int, []),
    "sdrgpu_launch_count": (C.c_uint64, []),
    "sdrgpu_set_tuning": (C.c_int, [C.c_int, C.c_int]),
    "sdrgpu_get_tuning": (C.c_int, [C.c_int]),
    "sdrgpu_design_sinc_m2_channelizer": (C.c_int, [C.c_double, C.c_int, C.c_int, _f32p, C.c_int, _i32p]),
    "sdrgpu_design_sinc_m2_synthesizer": (C.c_int, [C.c_double, C.c_double, C.c_int, C.c_int, _f32p, C.c_int, _i32p]),
    "sdrgpu_design_half_band": (C.c_int, [C.c_int, C.c_int, _f32p]),
    "sdrgpu_design_remez_estimate_order": (C.c_int, [C.c_double] * 5),
    "sdrgpu_design_remez_low_pass": (C.c_int, [C.c_double] * 5 + [C.c_int, C.c_int, C.c_int, _f32p, C.c_int, _i32p]),
    "sdrgpu_channel_count_for_rate": (C.c_int, [C.c_double]),
    "sdrgpu_channel_indexes": (C.c_int, [C.c_double, C.c_int, C.c_double, C.c_longlong, C.c_int, _i32p, C.c_int, _i32p]),
    "sdrgpu_center_frequency_for_indexes": (C.c_int, [C.c_double, C.c_int, C.c_double, _i32p, C.c_int,
                                                      C.POINTER(C.c_longlong)]),
    "sdrgpu_chan_create": (C.c_int, [_vpp, _f32p, C.c_int, C.c_int, C.c_int]),
    "sdrgpu_chan_destroy": (C.c_int, [_vp]),
    "sdrgpu_chan_set_stream": (C.c_int, [_vp, _vp]),
    "sdrgpu_chan_sync": (C.c_int, [_vp]),
    "sdrgpu_convert_samples": (C.c_int, [C.c_int, _vp, C.c_int, C.c_int, _vp, C.c_int]),
    "sdrgpu_airspy_create": (C.c_int, [C.POINTER(_vp), C.c_int]),
    "sdrgpu_airspy_destroy": (C.c_int, [_vp]),
    "sdrgpu_airspy_set_sample_packing": (C.c_int, [_vp, C.c_int]),
    "sdrgpu_airspy_convert": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _vp, C.c_int]),
    "sdrgpu_airspy_mismatches": (C.c_int, [_vp, C.POINTER(C.c_int)]),
    "sdrgpu_airspy_repaired": (C.c_int, [_vp, C.POINTER(C.c_int)]),
    "sdrgpu_chan_set_input_format": (C.c_int, [_vp, C.c_int]),
    "sdrgpu_chan_set_sample_rate": (C.c_int, [_vp, C.c_double]),
    "sdrgpu_chan_select": (C.c_int, [_vp, C.POINTER(OutputChannel), C.c_int, _f32p, C.c_int]),
    "sdrgpu_chan_process": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _vp, C.c_longlong, C.c_int, C.c_int, _i32p]),
    "sdrgpu_chan_blocks_for": (C.c_int, [_vp, C.c_int]),
    "sdrgpu_chan_enable_timing": (C.c_int, [_vp, C.c_int]),
    "sdrgpu_chan_last_kernel_ms": (C.c_int, [_vp, _f32p]),
    "sdrgpu_bank_config_preset": (C.c_int, [C.POINTER(BankConfig), C.c_int, C.c_int, C.c_double, _f32p, C.c_int, C.c_int]),
    "sdrgpu_bank_create": (C.c_int, [_vpp, C.POINTER(BankConfig)]),
    "sdrgpu_bank_destroy": (C.c_int, [_vp]),
    "sdrgpu_bank_set_stream": (C.c_int, [_vp, _vp]),
    "sdrgpu_bank_sync": (C.c_int, [_vp]),
    "sdrgpu_bank_process": (C.c_int, [_vp, _vp, C.c_longlong, C.c_int, C.c_int, _vp, C.c_int, _vp, C.c_longlong, _vp,
                                      C.c_int]),
    "sdrgpu_bank_correct_inversion": (C.c_int, [_vp, C.c_int, C.c_double]),
    "sdrgpu_bank_set_sync_detector": (C.c_int, [_vp, C.c_int]),
    "sdrgpu_bank_set_demodulator_lanes": (C.c_int, [_vp, C.c_int]),
    "sdrgpu_bank_set_symbol_tap": (C.c_int, [_vp, C.c_int]),
    "sdrgpu_bank_read_symbol_tap": (C.c_int, [_vp, C.POINTER(C.c_double), C.c_int, _i32p]),
    "sdrgpu_bank_reset_pll": (C.c_int, [_vp, C.c_int]),
    "sdrgpu_bank_get_loop_state": (C.c_int, [_vp, C.c_int, C.POINTER(C.c_double)]),
    "sdrgpu_bank_set_squelch_reporting": (C.c_int, [_vp, C.c_int]),
    "sdrgpu_bank_set_squelch_threshold": (C.c_int, [_vp, C.c_int, C.c_double]),
    "sdrgpu_pack_dibits": (C.c_int, [_u8p, C.c_int, _u8p]),
    "sdrgpu_bank_enable_timing": (C.c_int, [_vp, C.c_int]),
    "sdrgpu_bank_last_kernel_ms": (C.c_int, [_vp, _f32p]),
    "sdrgpu_pipeline_create": (C.c_int, [_vpp, _vp, _vp]),
    "sdrgpu_pipeline_set_chunks": (C.c_int, [_vp, C.c_int]),
    "sdrgpu_pipeline_set_device_chunks": (C.c_int, [_vp, C.c_int]),
    "sdrgpu_pipeline_create_multi": (C.c_int, [_vpp, _vp, C.c_int, _vp]),
    "sdrgpu_pipeline_process_multi": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _vp, C.c_int, _vp, C.c_longlong, _vp, C.c_int]),
    "sdrgpu_pipeline_submit_multi": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, _vp]),
    "sdrgpu_pipeline_wait": (C.c_int, [_vp]),
    "sdrgpu_pipeline_destroy": (C.c_int, [_vp]),
    "sdrgpu_pipeline_process": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _vp, C.c_int, _vp, C.c_longlong, _vp, C.c_int]),
    "sdrgpu_pipeline_create_routed": (C.c_int, [_vpp, _vp, C.c_int, _vp, C.c_int, _i32p]),
    "sdrgpu_pipeline_process_routed": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.POINTER(BankOutput), C.c_int]),
}

_lib = None


def lib():
    """Loads libsdrgpu.so; raises if it has not been built (python -m sdrtrunk_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("libsdrgpu.so is not built: run `python __graft_entry__.py build` "
                              "(or python sdrtrunk_b200/build.py); there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(status):
    if status == OK:
        return
    msg = lib().sdrgpu_last_error().decode("utf-8", "replace")
    if status == ERR_INVALID_ARG:
        raise IllegalArgumentException(msg)
    if status == ERR_BAD_STATE:
        raise IllegalStateException(msg)
    if status == ERR_DESIGN:
        raise FilterDesignException(msg)
    if status == ERR_OVERFLOW:
        raise OverflowError_(msg)
    if status == ERR_NOMEM:
        raise MemoryError(msg)
    raise CudaError(msg)


_initialised = {}


def init(device=0):
    if not _initialised.get(device):
        check(lib().sdrgpu_init(device))
        _initialised[device] = True


def f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def ptr(a):
    """void* of a numpy array (host) or an int device address."""
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    if a is None:
        return None
    return C.c_void_p(int(a))
