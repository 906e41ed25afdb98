"""ctypes binding of ``include/nsf.h`` (``_lib/libnsf.so``).

There is deliberately no fallback: if the CUDA library has not been built, importing this module
raises, and every compute call raises ``NsfError`` when no sm_100 device is usable.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NSF_LIB_PATH") or os.path.join(_HERE, "_lib", "libnsf.so")   # override: experiments only

# status codes / flags (mirror include/nsf.h)
OK, ERR_BAD_ARG, ERR_TOO_SHORT, ERR_CUDA, ERR_WORKSPACE, ERR_NO_DEVICE, ERR_UNSUPPORTED = range(7)
PCM_F32, PCM_I16 = 0, 1
PEAK_NORMALIZE, NO_AUTOCORR, SMOOTH, NO_CMVN, NO_DELTAS, AC_DELTAS, NO_REDUCE = (
    0x001, 0x002, 0x004, 0x008, 0x010, 0x020, 0x040)
NO_MFCC = 0x080
AC_NO_PAD = 0x800
DEBUG_SIMT_DFT = 0x100
DEBUG_FMA_AUTOCORR = 0x200
DEBUG_UNFUSED_MEL = 0x400
COLLECT_FAST, COLLECT_SLOW, COLLECT_BLEND = 0x1, 0x2, 0x4
F32, F64 = 0, 1
TABLE_MEL, TABLE_DCT, TABLE_HANN_SYM, TABLE_HANN_PER = 0, 1, 2, 3
ROWS_INTERP_SLOWER, ROWS_SMOOTH, ROWS_BLEND_STACK = 0, 1, 2
OPT_EDGE_ZERO_THRESHOLD = 0
OPT_RESAMPLE_QUALITY = 1
RESAMPLE_POLY, RESAMPLE_HQ = 0, 1
POST_EDGEFIX, POST_CMVN, POST_DELTAS, POST_REDUCE = 0x1, 0x2, 0x4, 0x8
ENC_U8, ENC_I16, ENC_I24, ENC_I32, ENC_F32, ENC_F64 = range(6)
# nsf_pcm_source: one clip of the WAV conversion calls (raw data-chunk bytes -> mono float32)
PCM_SOURCE = np.dtype([("byte_offset", "<i8"), ("frames", "<i8"), ("encoding", "<i4"), ("channels", "<i4"),
                       ("sample_rate", "<i4"), ("reserved", "<i4")], align=True)
assert PCM_SOURCE.itemsize == 32
STAGE_NAMES = ("peak_normalize", "fold", "stft_gemm", "mel_db", "dct_stats", "cmvn_delta_reduce",
               "autocorr", "post")


class NsfError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"nsf status {status}: {message}")
        self.status = status


class TooShortError(NsfError):
    pass


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(needs nvcc). neurosync_trainer_lite_b200 has no CPU implementation to fall back to.")

lib = C.CDLL(LIB_PATH)

_i32, _i64, _u32 = C.c_int32, C.c_int64, C.c_uint32
_vp, _i64p, _f32p, _f64p, _i32p = (C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_float),
                                   C.POINTER(C.c_double), C.POINTER(C.c_int32))

_SIGS = {
    "nsf_abi_version": (_i32, []),
    "nsf_last_error": (C.c_char_p, []),
    "nsf_device_count": (_i32, []),
    "nsf_frame_length": (_i32, [_i32]),
    "nsf_hop_length": (_i32, [_i32]),
    "nsf_guard_frames": (_i64, [_i64, _i32, _i32]),
    "nsf_hop_frames": (_i64, [_i64, _i32, _i32]),
    "nsf_feature_rows": (_i64, [_i64, _i32, _i32]),
    "nsf_row_offsets": (_i32, [_i32, _i32, _i64p, _i32, _u32, _i64p]),
    "nsf_feature_cols": (_i32, [_vp, _u32]),
    "nsf_collect_rows": (_i64, [_i64, _i64, _u32, _i32]),
    "nsf_plan_create": (_i32, [_i32, _i32, _i32, _i32, _i32, _i32, C.POINTER(_vp)]),
    "nsf_plan_destroy": (None, [_vp]),
    "nsf_plan_table": (_i64, [_vp, _i32, _f32p, _i64]),
    "nsf_plan_info": (_i32, [_vp, _i32p, _i32p, _i32p, _i32p]),
    "nsf_plan_fold_check": (_i32, [_vp, _f32p, _f64p, _f64p]),
    "nsf_ctx_create": (_i32, [_vp, _i32, C.POINTER(_vp)]),
    "nsf_ctx_destroy": (None, [_vp]),
    "nsf_host_alloc": (_i32, [C.POINTER(_vp), _i64]),
    "nsf_host_free": (None, [_vp]),
    "nsf_host_register": (_i32, [_vp, _i64]),
    "nsf_host_unregister": (_i32, [_vp]),
    "nsf_ctx_set_option": (_i32, [_vp, _i32, C.c_double]),
    "nsf_workspace_bytes": (_i64, [_vp, _i64, _i32, _u32]),
    "nsf_extract_batch": (_i32, [_vp, _vp, _vp, _i32, _i64p, _i32, _u32, _vp, _i64, _i64p, _vp, _vp,
                                 _i64]),
    "nsf_extract_host": (_i32, [_vp, _vp, _i32, _i64p, _i32, _u32, _vp, _i64, _vp]),
    "nsf_normalize_host": (_i32, [_vp, _vp, _i32, _i64p, _i32, _vp, _vp]),
    "nsf_collect_batch": (_i32, [_vp, _vp, _i32, _vp, _i32, _i64p, _vp, _i32, _i64p, _i32, _u32, _i32,
                                 _vp, _vp, _i64p]),
    "nsf_collect_host": (_i32, [_vp, _i32, _vp, _i32, _i64p, _vp, _i32, _i64p, _i32, _u32, _i32, _vp,
                                _vp]),
    "nsf_extract_collect_host": (_i32, [_vp, _vp, _i32, _i64p, _i32, _u32, _vp, _i32, _i64p, _u32, _i32, _vp, _vp,
                                        _vp]),
    "nsf_rows_host": (_i32, [_vp, _i32, _i32, _vp, _i64, _vp, _i64, _i32, _i32, _vp]),
    "nsf_post_host": (_i32, [_vp, _vp, _i64, _i32, _u32, _vp]),
    "nsf_chunk_count": (_i64, [_i64, _i32, _i32]),
    "nsf_chunk_gather": (_i32, [_vp, _vp, _vp, _i64, _i32, _i64, _i32, _i32, _vp]),
    "nsf_chunk_blend": (_i32, [_vp, _vp, _vp, _i64, _i32, _i32, _i32, _i32, C.c_float, _vp]),
    "nsf_resample_len": (_i64, [_i64, _i32, _i32]),
    "nsf_resample_design": (_i64, [_i32, _i32, _f64p, _i64, _i32p, _i32p, _i32p, _i32p]),
    "nsf_resample_design_q": (_i64, [_i32, _i32, _i32, _f64p, _i64, _i32p, _i32p, _i32p, _i32p]),
    "nsf_resample_host": (_i32, [_vp, _vp, _i32, _i64, _i32, _i32, _vp, _i64]),
    "nsf_convert_offsets": (_i32, [_vp, _i32, _i32, _i64, _i64p]),
    "nsf_convert_batch": (_i32, [_vp, _vp, _vp, _i64, _vp, _i32, _i32, _vp, _i64p]),
    "nsf_convert_host": (_i32, [_vp, _vp, _i64, _vp, _i32, _i32, _vp]),
    "nsf_window_offsets": (_i32, [_i64p, _i64p, _i32, _i32, _i64p]),
    "nsf_window_gather": (_i32, [_vp, _vp, _vp, _i32, _i64p, _vp, _i32, _i64p, _i32, _i32, _i64p, _i64, _vp, _vp]),
    "nsf_launch_count": (_i64, [_vp]),
    "nsf_set_profiling": (None, [_vp, _i32]),
    "nsf_stage_times_ms": (_i32, [_vp, _f32p, _i32]),
}
for _name, (_res, _args) in _SIGS.items():
    _fn = getattr(lib, _name)   # AttributeError here == header and library out of sync
    _fn.restype = _res
    _fn.argtypes = _args

EXPORTED = tuple(_SIGS)


def last_error():
    msg = lib.nsf_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(status):
    if status == OK:
        return
    cls = TooShortError if status == ERR_TOO_SHORT else NsfError
    raise cls(status, last_error())


def i64_array(values):
    arr = np.ascontiguousarray(values, dtype=np.int64)
    return arr, arr.ctypes.data_as(_i64p)


def ptr(array):
    """void* of a C-contiguous numpy array (the caller keeps the array alive)."""
    if array is None:
        return None
    assert array.flags["C_CONTIGUOUS"]
    return C.c_void_p(array.ctypes.data)


def pcm_sources(sources):
    """C-contiguous ``PCM_SOURCE`` array from an array of that dtype or from (byte_offset, frames, encoding,
    channels, sample_rate) tuples."""
    if isinstance(sources, np.ndarray) and sources.dtype == PCM_SOURCE:
        return np.ascontiguousarray(sources)
    out = np.zeros(len(sources), dtype=PCM_SOURCE)
    for i, s in enumerate(sources):
        out[i] = tuple(s[:5]) + (0,)
    return out


def convert_offsets(sources, target_sr, payload_bytes):
    """Prefix sum of the per-clip output lengths of a conversion (``nsf_convert_offsets``; validates every
    descriptor, needs no GPU)."""
    src = pcm_sources(sources)
    out = np.empty(len(src) + 1, dtype=np.int64)
    check(lib.nsf_convert_offsets(ptr(src), len(src), int(target_sr), int(payload_bytes), out.ctypes.data_as(_i64p)))
    return out


def window_offsets(audio_offsets, facial_offsets, window):
    """Prefix sum of the per-clip training-window counts of a packed dataset (``nsf_window_offsets``; validates the
    geometry the way ``_WindowedClip`` fails, needs no GPU)."""
    a_off, a_p = i64_array(audio_offsets)
    f_off, f_p = i64_array(facial_offsets)
    if len(a_off) != len(f_off) or len(a_off) < 2:
        raise ValueError("audio and facial offsets need the same length, at least 2")
    out = np.empty(len(a_off), dtype=np.int64)
    check(lib.nsf_window_offsets(a_p, f_p, len(a_off) - 1, int(window), out.ctypes.data_as(_i64p)))
    return out
