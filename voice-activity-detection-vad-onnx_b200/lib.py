"""ctypes binding of libvadx.so (the C ABI in include/vadx.h).

There is NO fallback: if the shared library has not been built (``python -c "import
__graft_entry__ as g; g.build()"`` or ``make -C voice-activity-detection-vad-onnx_b200/csrc``)
or no CUDA device is visible, every compute entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvadx.so")

DT_I16, DT_F32, DT_I32 = 0, 1, 2
ACT_NONE, ACT_RELU, ACT_SIGMOID, ACT_SOFTMAX, ACT_RES_FIRST = 0, 1, 2, 3, 16
FLOOR_CLAMP, FLOOR_ADD = 0, 1
PREEMPH_NONE, PREEMPH_ZERO_HISTORY, PREEMPH_KEEP_FIRST = 0, 1, 2

_ERRORS = {-1: ValueError, -2: RuntimeError, -3: RuntimeError, -4: KeyError, -5: MemoryError}


class PostCfg(C.Structure):
    _fields_ = [("smooth_window", C.c_int32), ("threshold", C.c_float), ("min_speech_frame", C.c_int32),
                ("max_speech_frame", C.c_int32), ("min_silence_frame", C.c_int32),
                ("merge_silence_frame", C.c_int32), ("extend_speech_frame", C.c_int32)]


class StreamPostCfg(C.Structure):
    _fields_ = [("smooth_window", C.c_int32), ("threshold", C.c_float), ("pad_start_frame", C.c_int32),
                ("min_speech_frame", C.c_int32), ("max_speech_frame", C.c_int32), ("min_silence_frame", C.c_int32)]


class FsmnServeCfg(C.Structure):
    _fields_ = [("speaking_score", C.c_double), ("silence_score", C.c_double), ("frame_duration", C.c_double),
                ("fusion_threshold", C.c_double), ("min_speech_duration", C.c_double), ("snr_threshold", C.c_float),
                ("noise_init", C.c_float)]


_i64, _i32, _f32, _vp, _sz = C.c_int64, C.c_int, C.c_float, C.c_void_p, C.c_size_t

# name -> (restype, argtypes); must list every symbol include/vadx.h declares (tests check this)
SIGNATURES = {
    "vadx_abi_version": (C.c_int, []),
    "vadx_last_error": (C.c_char_p, []),
    "vadx_device_count": (C.c_int, []),
    "vadx_launch_count": (C.c_uint64, []),
    "vadx_profile_enable": (C.c_int, [_i32]),
    "vadx_profile_collect": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_uint64), _i32]),
    "vadx_profile_collect_kernels": (C.c_int, [_vp, _i32, C.POINTER(C.c_int)]),
    "vadx_prep_audio": (C.c_int, [_vp, _i32, _i64, _i64, _i64, _f32, _i32, _i32, _f32, _i64, _vp, _i64, _vp]),
    "vadx_stft_power_f32": (C.c_int, [_vp, _i64, _i64, _i32, _i32, _i32, _vp, _i32, _i32, _vp, _i64, _vp]),
    "vadx_stft_tc_supported": (C.c_int, [_i32, _i32]),
    "vadx_pack_stft_basis_tc": (C.c_int, [_vp, _i32, _i32, _i32, C.c_double, C.c_double, _vp, _sz, C.POINTER(_sz)]),
    "vadx_stft_power_tc_i16": (C.c_int, [_vp, _i64, _i64, _i64, _i32, _i32, _i32, _vp, _i32, _vp, _i64, _vp]),
    "vadx_pack_stft_dc_tc": (C.c_int, [_vp, _i32, _i32, _i32, C.c_double, C.c_double, _i64, _i32, _i32, _i32, _vp, _sz,
                                       C.POINTER(_sz), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "vadx_stream_mean_i16": (C.c_int, [_vp, _i64, _i64, _i64, _vp, _vp, _vp]),
    "vadx_stft_power_tc_i16_ex": (C.c_int, [_vp, _i64, _i64, _i64, _i32, _i32, _i32, _vp, _i32, _vp, _i64, _i32, _vp, _vp, _vp,
                                            _i32, _i32, _f32, _i32, _vp]),
    "vadx_pack_stft_basis_tc_fmt": (C.c_int, [_vp, _i32, _i32, _i32, C.c_double, C.c_double, _i32, _vp, _sz, C.POINTER(_sz)]),
    "vadx_mel_log_f32": (C.c_int, [_vp, _i64, _i64, _i32, _i32, _vp, _vp, _vp, _i32, _i32, _f32, _vp, _i64, _vp]),
    "vadx_linear_f32": (C.c_int, [_vp, _i64, _vp, _i32, _vp, _vp, _i64, _vp, _i64, _i64, _i32, _i32, _i32, _vp]),
    "vadx_tc_supported": (C.c_int, [_i32, _i32]),
    "vadx_pack_weight_tc": (C.c_int, [_vp, _i32, _i32, _vp, _sz, C.POINTER(_sz)]),
    "vadx_linear_tc_f32": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _i64, _vp, _i64, _i64, _i32, _i32, _i32, _vp]),
    "vadx_fc2_memory_stages_stream_bytes": (C.c_size_t, [_i32, _i32]),
    "vadx_fc2_memory_stages_supported": (C.c_int, [_i32, _i32, _i32, _i32, _i32, _i32, _i32]),
    "vadx_linear_tc_stream_stages_f32": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _i32, _i32, _i32, _vp]),
    "vadx_fc2_memory_stages_f32": (C.c_int, [_vp, _i32, _vp, _vp, _i32, _vp, _i32, _vp, _i32, _vp, _vp, _i64, _i32, _vp]),
    "vadx_depthwise_conv1d_f32": (C.c_int, [_vp, _i64, _vp, _i32, _i32, _i32, _i32, _vp, _i64, _i64, _i32, _i32, _i32, _vp]),
    "vadx_linear_head_tc_f32": (C.c_int, [_vp, _i64, _vp, _vp, _i64, _i32, _i32, _i32, _vp, _f32, _vp, _vp]),
    "vadx_fsmn_memory_f32": (C.c_int, [_vp, _i64, _vp, _i32, _i32, _vp, _i32, _i32, _vp, _i64, _vp, _i64, _i64,
                                       _i32, _i32, _vp, _vp, _vp]),
    "vadx_lfr_cmvn_f32": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _i64, _i64, _i32, _i32, _i32, _i32, _vp]),
    "vadx_softmax_class0_f32": (C.c_int, [_vp, _i64, _i64, _i32, _vp, _vp]),
    "vadx_frame_energy_log10_f32": (C.c_int, [_vp, _i64, _i64, _i64, _i32, _i32, _i32, _i32, _f32, _f32, _vp, _vp]),
    "vadx_fsmn_gate": (C.c_int, [_vp, _vp, _vp, _f32, _f32, _i64, _i32, _vp, _vp, _vp]),
    "vadx_cfb_front_supported": (C.c_int, [_i32, _i32, _i32]),
    "vadx_cfb_front_f32": (C.c_int, [_vp, _i64, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_float, _vp, _vp, _vp]),
    "vadx_layernorm_perm_f32": (C.c_int, [_vp, _i64, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _i32, C.c_float, _vp, _i64, _i32, _vp]),
    "vadx_ceps_cmul_t_f32": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _i32, _vp]),
    "vadx_add_transposed_f32": (C.c_int, [_vp, _i64, _vp, _vp, _i64, _i32, _i32, _vp]),
    "vadx_lstm_recurrence_supported": (C.c_int, [_i32]),
    "vadx_lstm_recurrence_f32": (C.c_int, [_vp, _i64, _i64, _i64, _vp, _i64, _i64, _i64, _vp, _i64, _i32, _i32, _i32, _i32, _vp]),
    "vadx_affine_f32": (C.c_int, [_vp, C.c_float, C.c_float, _vp, _i64, _vp]),
    "vadx_reflect_windows_f32": (C.c_int, [_vp, _i64, _i64, _i32, _i64, _i32, _i32, _vp, _vp]),
    "vadx_silero_lstm_windows_f32": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _vp, C.c_float, _vp, _i64, _i32, _i32, _vp]),
    "vadx_stft_mag_compact_f32": (C.c_int, [_vp, _i64, _i64, _i32, _i32, _i32, _vp, _vp]),
    "vadx_gather_windows_i16": (C.c_int, [_vp, _i64, _i64, _i32, _i64, _i64, _vp, _vp]),
    "vadx_fsmn_gate_hysteresis_windows": (C.c_int, [_vp, _vp, _i64, _i32, _i32, C.c_float, C.c_float, _i32, C.c_double, C.c_double,
                                                    _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, C.c_float, _vp]),
    "vadx_lookahead_hysteresis": (C.c_int, [_vp, _i32, _i64, _i64, _i32, _i32, C.c_double, C.c_double, _i32, _vp, _vp,
                                            _vp, _i64, _vp, _vp, _f32, _vp]),
    "vadx_runs_to_segments": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _vp, _i32, _vp]),
    "vadx_reflect_window_f32": (C.c_int, [_vp, _i64, _i64, _i32, _i32, _vp, _vp]),
    "vadx_sqrt_inplace_f32": (C.c_int, [_vp, _i64, _vp]),
    "vadx_lstm_cell_f32": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp]),
    "vadx_silero_timestamps": (C.c_int, [_vp, _i64, _vp, _vp, _i64, C.c_double, C.c_double, C.c_double, C.c_double,
                                         C.c_double, C.c_double, _i32, _i32, _vp, _vp, _i32, _vp]),
    "vadx_stft_complex_f32": (C.c_int, [_vp, _i64, _i64, _i32, _i32, _i32, _vp, _i32, _i32, _vp, _i64, _vp]),
    "vadx_permute4_f32": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _i64, _i32, _i32, _i32, _i32, _vp]),
    "vadx_layernorm_f32": (C.c_int, [_vp, _i64, _i32, _vp, _vp, _f32, _vp, _vp]),
    "vadx_lstm_seq_f32": (C.c_int, [_vp, _i64, _i64, _i64, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _i64, _i32, _i32,
                                    _i32, _i32, _i32, _vp]),
    "vadx_ew2_f32": (C.c_int, [_i32, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _i64, _i32, _f32, _vp]),
    "vadx_ceps_cmul_f32": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _vp]),
    "vadx_im2col_f3_f32": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _vp]),
    "vadx_alpha_x4_f32": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _i32, _f32, _f32, _f32, _vp, _f32, _vp, _vp, _vp]),
    "vadx_alpha_x4_const_f32": (C.c_int, [_vp, _vp, _vp, _i32, _i64, _i32, _i32, _i32, _f32, _f32, _f32, _vp, _f32, _vp, _vp,
                                          _vp]),
    "vadx_istft_ola_f32": (C.c_int, [_vp, _i64, _i64, _i32, _i32, _i32, _vp, _i32, _vp, _i64, _vp]),
    "vadx_postprocess_frames": (C.c_int, [_vp, _i64, _vp, _i64, _i32, C.POINTER(PostCfg), _vp, _vp, _vp, _i32, _vp]),
    "vadx_resample_out_len": (C.c_int64, [_i64, C.c_double]),
    "vadx_resample_linear_f32": (C.c_int, [_vp, _i64, _i64, _i64, C.c_double, _vp, _i64, _i64, _vp]),
    "vadx_ingest_out_frames": (C.c_int64, [_i64, _i32, _i32]),
    "vadx_ingest_pcm16": (C.c_int, [_vp, _i64, _vp, _i64, _i64, _i32, _i32, _i32, _vp, _i64, _vp, _vp]),
    "vadx_stream_post_state_words": (C.c_int, [_i32]),
    "vadx_stream_postprocess": (C.c_int, [_vp, _i64, _vp, _i64, _i32, C.POINTER(StreamPostCfg), _vp, _vp, _vp, _i32, _vp,
                                          _vp]),
    "vadx_stream_serve_zero_tail": (C.c_int, [_vp, _i64, _vp, _i64, _i32, _i32, _vp]),
    "vadx_stream_serve_step": (C.c_int, [_vp, _i64, _i32, _vp, _vp, _i64, _i32, _i32, _i32, C.POINTER(StreamPostCfg), _vp,
                                         _vp, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _sz, C.POINTER(_sz), _vp]),
    "vadx_silero_serve_load": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _vp]),
    "vadx_silero_serve_step": (C.c_int, [_vp, _i64, _vp, _vp, _i64, _i32, C.c_double, C.c_double, _vp, _vp, _vp, _vp, _vp,
                                         _vp, _vp, _vp, _vp, _vp, _sz, C.POINTER(_sz), _vp]),
    "vadx_fsmn_serve_state_words": (C.c_int, [_i32]),
    "vadx_fsmn_serve_load": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _i32, _i32, _f32, _vp, _vp, _vp]),
    "vadx_fsmn_serve_step": (C.c_int, [_vp, _i64, _vp, _i32, _vp, _vp, _i64, _i32, _i32, _i32, C.POINTER(FsmnServeCfg), _vp,
                                       _vp, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _sz, C.POINTER(_sz), _vp]),
    "vadx_marblenet_serve_state_words": (C.c_int, [C.POINTER(PostCfg)]),
    "vadx_marblenet_serve_step": (C.c_int, [_vp, _i64, _i32, _vp, _vp, _i64, _i32, C.POINTER(PostCfg), _f32, _vp, _vp,
                                            _vp, _vp, _vp, _vp, _vp, _sz, C.POINTER(_sz), _vp]),
    "vadx_create": (C.c_int, [C.c_char_p, C.POINTER(C.c_int32), _i32, C.POINTER(_vp)]),
    "vadx_destroy": (None, [_vp]),
    "vadx_set_tensor": (C.c_int, [_vp, C.c_char_p, _vp, _i32, C.POINTER(_i64), _i32]),
    "vadx_set_scalar": (C.c_int, [_vp, C.c_char_p, C.c_double]),
    "vadx_workspace_bytes": (C.c_int, [_vp, _i64, _i64, C.POINTER(_sz)]),
    "vadx_output_frames": (C.c_int, [_vp, _i64, C.POINTER(C.c_int32)]),
    "vadx_forward": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), _i64, _i64, _vp, _sz, _vp]),
}

_lib = None


def load() -> C.CDLL:
    """Load libvadx.so and bind every signature.  Raises (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(vadx has no CPU or PyTorch fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.vadx_abi_version() != 1:
        raise RuntimeError(f"libvadx ABI {lib.vadx_abi_version()} != 1; rebuild the library")
    _lib = lib
    return lib


STAGES = ("prep", "stft", "mel", "linear", "memory", "head", "postproc")


def profile_enable(on: bool) -> None:
    check(load().vadx_profile_enable(1 if on else 0))


def profile_collect() -> dict:
    """-> {stage: (milliseconds, calls)} accumulated since the last collect (synchronises)."""
    ms = (C.c_double * len(STAGES))()
    calls = (C.c_uint64 * len(STAGES))()
    check(load().vadx_profile_collect(ms, calls, len(STAGES)))
    return {n: (ms[i], int(calls[i])) for i, n in enumerate(STAGES)}


class _KernelStat(C.Structure):
    _fields_ = [("name", C.c_char_p), ("ms", C.c_double), ("calls", C.c_uint64), ("bytes", C.c_double), ("flops", C.c_double)]


def profile_collect_kernels() -> dict:
    """-> {kernel name: {"ms", "calls", "bytes", "flops"}} accumulated since the last collect (synchronises): the
    algorithmic bytes / flops every entry point reports for its calls, next to their measured device time."""
    n = C.c_int(0)
    check(load().vadx_profile_collect_kernels(None, 0, C.byref(n)))
    if n.value == 0:
        return {}
    buf = (_KernelStat * n.value)()
    check(load().vadx_profile_collect_kernels(C.cast(buf, C.c_void_p), n.value, C.byref(n)))
    return {buf[i].name.decode(): {"ms": buf[i].ms, "calls": int(buf[i].calls), "bytes": buf[i].bytes, "flops": buf[i].flops}
            for i in range(n.value)}


def check(rc: int) -> None:
    if rc == 0:
        return
    msg = load().vadx_last_error().decode("utf-8", "replace")
    raise _ERRORS.get(rc, RuntimeError)(f"libvadx: {msg} (code {rc})")


def require_device() -> None:
    if load().vadx_device_count() < 1:
        raise RuntimeError("libvadx: no CUDA device visible; vadx has no CPU path")


def pack_weight_tc(w):
    """[n_out, n_in] fp32 numpy weight -> uint8 numpy operand image for vadx_linear_tc_f32."""
    import numpy as np
    w = np.ascontiguousarray(w, np.float32)
    n_out, n_in = w.shape
    nbytes = C.c_size_t()
    check(load().vadx_pack_weight_tc(w.ctypes.data, n_out, n_in, None, 0, C.byref(nbytes)))
    img = np.zeros(nbytes.value, np.uint8)
    check(load().vadx_pack_weight_tc(w.ctypes.data, n_out, n_in, img.ctypes.data, img.nbytes, C.byref(nbytes)))
    return img


TC_FMT_BF16, TC_FMT_F16 = 0, 1


def pack_stft_basis_tc(basis, n_bins: int, preemph: float, scale: float, fmt: int = TC_FMT_BF16):
    """[n_taps, ld] fp32 interleaved basis table -> uint8 operand image for vadx_stft_power_tc_i16(_ex)."""
    import numpy as np
    basis = np.ascontiguousarray(basis, np.float32)
    n_taps, ld = basis.shape
    nbytes = C.c_size_t()
    check(load().vadx_pack_stft_basis_tc_fmt(basis.ctypes.data, ld, n_taps, n_bins, preemph, scale, fmt, None, 0,
                                             C.byref(nbytes)))
    img = np.zeros(nbytes.value, np.uint8)
    check(load().vadx_pack_stft_basis_tc_fmt(basis.ctypes.data, ld, n_taps, n_bins, preemph, scale, fmt, img.ctypes.data,
                                             img.nbytes, C.byref(nbytes)))
    return img


def pack_stft_dc_tc(basis, n_bins: int, preemph: float, scale: float, n_samples: int, hop: int, pad_left: int,
                    n_frames: int):
    """DC-response tables for vadx_stft_power_tc_i16_ex -> (float32 array, n_edge_lo, t_edge_hi)"""
    import numpy as np
    basis = np.ascontiguousarray(basis, np.float32)
    n_taps, ld = basis.shape
    n, lo, hi = C.c_size_t(), C.c_int(), C.c_int()
    check(load().vadx_pack_stft_dc_tc(basis.ctypes.data, ld, n_taps, n_bins, preemph, scale, n_samples, hop, pad_left,
                                      n_frames, None, 0, C.byref(n), C.byref(lo), C.byref(hi)))
    tab = np.zeros(n.value, np.float32)
    check(load().vadx_pack_stft_dc_tc(basis.ctypes.data, ld, n_taps, n_bins, preemph, scale, n_samples, hop, pad_left,
                                      n_frames, tab.ctypes.data, tab.size, C.byref(n), C.byref(lo), C.byref(hi)))
    return tab, lo.value, hi.value


def ptr(t) -> int:
    """Device (or host) address of a torch tensor / numpy array, or 0 for None."""
    if t is None:
        return 0
    if hasattr(t, "data_ptr"):
        return t.data_ptr()
    return t.ctypes.data


def stream_ptr(stream=None) -> int:
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return s.cuda_stream
