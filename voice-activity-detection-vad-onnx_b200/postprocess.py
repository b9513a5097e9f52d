"""Post-processing: device state machines (through the C ABI) + the host-side formatting that
turns frame-index segments into the reference's seconds / sample indices / text files.

Reference anchors:
  VadPostprocessor.process / decision_to_segment ... FireRedVAD/Inference_FireRed_ONNX.py:102-305
  MarbleNet copy (frame_shift arg, open tail) ....... NVIDIA_Frame_VAD_Multilingual_MarbleNet/
                                                      Inference_NVIDIA_MarbleNet_VAD_ONNX.py:160-353
  format_time / file writing ........................ FireRedVAD/Inference_FireRed_ONNX.py:593-609,
                                                      FSMN/Inference_FSMN_VAD_ONNX.py:144-153,244-258
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from datetime import timedelta

import numpy as np

from . import lib
# The slot servers' host side lives in serve.py; its public names stay importable from here, where callers found them.
from .serve import (SERVE_END, SERVE_END_OF_STREAM, SERVE_ERR_RANGE, SERVE_ERR_SHORT, SERVE_START,  # noqa: F401
                    FsmnServeTick, FsmnSlotSegmenter, MarbleNetServeTick, MarbleNetSlotSegmenter, ServeTick,
                    ServeTickError, SileroServeTick, SileroSlotSegmenter, StreamSlotSegmenter, load_tick_inputs)


@dataclass(frozen=True)
class FramePostConfig:
    """Defaults = FireRed VAD (FireRedVAD/Inference_FireRed_ONNX.py:40-53)."""
    smooth_window_size: int = 5
    prob_threshold: float = 0.4
    min_speech_frame: int = 20
    max_speech_frame: int = 2000
    min_silence_frame: int = 20
    merge_silence_frame: int = 5
    extend_speech_frame: int = 0
    frame_shift_s: float = 0.01
    frame_length_s: float = 0.025
    tail_adds_frame_length: bool = True   # FireRed: open tail ends at n*shift + length; MarbleNet: n*shift

    def c_struct(self) -> lib.PostCfg:
        return lib.PostCfg(max(1, self.smooth_window_size), float(np.float32(self.prob_threshold)),
                           self.min_speech_frame, self.max_speech_frame, self.min_silence_frame,
                           self.merge_silence_frame, self.extend_speech_frame)


def postprocess_frames(probs, cfg: FramePostConfig, n_frames=None, max_segments: int | None = None, stream=None):
    """probs: CUDA fp32 [S, T] (row stride may exceed T).  n_frames: optional CUDA int32 [S].
    Returns (decisions int8 [S,T], seg_count int32 [S], segments int32 [S,max_segments,2]) on device."""
    import torch
    if not (torch.is_tensor(probs) and probs.is_cuda and probs.dtype == torch.float32 and probs.dim() == 2):
        raise ValueError("postprocess_frames: probs must be a CUDA fp32 tensor [S, T]")
    if probs.stride(1) != 1:
        raise ValueError("postprocess_frames: probs rows must be contiguous")
    S, T = probs.shape
    if max_segments is None:
        max_segments = T // 2 + 1
    dec = torch.empty((S, max(T, 1)), dtype=torch.int8, device=probs.device)
    cnt = torch.empty((S,), dtype=torch.int32, device=probs.device)
    seg = torch.empty((S, max_segments, 2), dtype=torch.int32, device=probs.device)
    if n_frames is not None and not (n_frames.is_cuda and n_frames.dtype == torch.int32 and n_frames.numel() == S):
        raise ValueError("postprocess_frames: n_frames must be a CUDA int32 tensor [S]")
    c = cfg.c_struct()
    lib.check(lib.load().vadx_postprocess_frames(probs.data_ptr(), probs.stride(0) if S > 0 else T, lib.ptr(n_frames),
                                                 S, T, C.byref(c), dec.data_ptr(), cnt.data_ptr(), seg.data_ptr(),
                                                 max_segments, lib.stream_ptr(stream)))
    return dec[:, :T], cnt, seg


def segments_to_seconds(pairs: np.ndarray, n_frames: int, cfg: FramePostConfig, wav_dur: float | None):
    """(start, end_exclusive) frame pairs of ONE stream -> [(start_s, end_s)] with the reference's
    float32 products and round(, 3)  (decision_to_segment, :146-179)."""
    pairs = np.asarray(pairs, np.int64).reshape(-1, 2)
    if pairs.shape[0] == 0 or n_frames == 0:
        return []
    fs, fl = np.float32(cfg.frame_shift_s), np.float32(cfg.frame_length_s)
    seg = np.empty((pairs.shape[0], 2), np.float32)
    seg[:, 0] = pairs[:, 0].astype(np.float32) * fs
    seg[:, 1] = pairs[:, 1].astype(np.float32) * fs
    if pairs[-1, 1] == n_frames:  # last decision is speech: open tail
        end_time = n_frames * fs + fl if cfg.tail_adds_frame_length else n_frames * fs
        if wav_dur is not None and wav_dur < end_time:
            end_time = wav_dur
        seg[-1, 1] = end_time
    return [(round(a, 3), round(b, 3)) for a, b in seg.tolist()]


def take_segments(seg_count, segments, stream_index: int | None = None):
    """Host view of the device post-processors' output with the overflow check every consumer needs: the kernels COUNT
    every segment but only STORE the first max_segments (= segments.shape[1]), so a count above that bound means
    trailing segments were dropped.  seg_count [S], segments [S, max, 2] (CUDA or CPU tensors / numpy arrays).
    Returns (counts ndarray [S], pairs ndarray [S, max, 2]), or the [k, 2] pairs of one stream when stream_index is given."""
    cnt = seg_count.cpu().numpy() if hasattr(seg_count, "cpu") else np.asarray(seg_count)
    seg = segments.cpu().numpy() if hasattr(segments, "cpu") else np.asarray(segments)
    max_segments = seg.shape[1]
    if cnt.size and int(cnt.max()) > max_segments:
        worst = int(cnt.argmax())
        raise RuntimeError(f"stream {worst} produced {int(cnt.max())} segments but only max_segments={max_segments} were stored; "
                           f"pass a larger max_segments")
    if stream_index is None:
        return cnt, seg
    return seg[stream_index, :int(cnt[stream_index])]


def lookahead_hysteresis(values, state, look_backward: int, speaking_score: float, silence_score: float,
                         is_final: bool, noisy_dB=None, snr_threshold: float = 1.0, stream=None):
    """One chunk of the FSMN / DFSMN look-ahead state machine for S streams, on the device.
    values: CUDA uint8 [S,T] flags (FSMN) or fp32 [S,T] probabilities (DFSMN).
    state: HysteresisState (updated in place)."""
    import torch
    mode = 0 if values.dtype == torch.uint8 else 1
    if values.dtype not in (torch.uint8, torch.float32) or values.dim() != 2 or values.stride(1) != 1:
        raise ValueError("lookahead_hysteresis: values must be CUDA uint8/fp32 [S, T] with contiguous rows")
    S, T = values.shape
    lib.check(lib.load().vadx_lookahead_hysteresis(
        values.data_ptr(), mode, values.stride(0), S, T, int(look_backward), float(speaking_score),
        float(silence_score), 1 if is_final else 0, state.silence.data_ptr(), state.n_saved.data_ptr(),
        state.saved.data_ptr(), state.saved.shape[1], lib.ptr(state.noise_avg) if noisy_dB is not None else None,
        lib.ptr(noisy_dB), float(snr_threshold), lib.stream_ptr(stream)))


def fsmn_gate_hysteresis_windows(p_silence, power_dB, state, look_backward: int, speaking_score: float, silence_score: float,
                                 one_minus_speech_threshold: float, speech_2_noise_ratio: float, snr_threshold: float,
                                 keep_trace: bool = False, stream=None):
    """Whole-file twin of (vadx_fsmn_gate + lookahead_hysteresis) x W windows in ONE launch: p_silence / power_dB CUDA fp32
    [S, W, T]; per stream the windows are walked in order because the gate compares against the running background level
    (FSMN/Inference_FSMN_VAD_ONNX.py:177-234).  state: HysteresisState (updated in place).  keep_trace -> (score u8 [S,W,T],
    noisy_dB [S,W], noise_in [S,W])."""
    import torch
    if not (p_silence.is_cuda and p_silence.dtype == torch.float32 and p_silence.dim() == 3 and p_silence.is_contiguous()
            and power_dB.shape == p_silence.shape and power_dB.dtype == torch.float32 and power_dB.is_contiguous()):
        raise ValueError("fsmn_gate_hysteresis_windows: p_silence / power_dB must be contiguous CUDA fp32 [S, W, T]")
    S, Wn, T = p_silence.shape
    score = noisy = noise_in = None
    if keep_trace:
        score = torch.empty((S, Wn, T), dtype=torch.uint8, device=p_silence.device)
        noisy = torch.empty((S, Wn), dtype=torch.float32, device=p_silence.device)
        noise_in = torch.empty((S, Wn), dtype=torch.float32, device=p_silence.device)
    lib.check(lib.load().vadx_fsmn_gate_hysteresis_windows(
        p_silence.data_ptr(), power_dB.data_ptr(), S, Wn, T, float(one_minus_speech_threshold), float(speech_2_noise_ratio),
        int(look_backward), float(speaking_score), float(silence_score), lib.ptr(score), lib.ptr(noisy), lib.ptr(noise_in),
        state.silence.data_ptr(), state.n_saved.data_ptr(), state.saved.data_ptr(), state.saved.shape[1],
        state.noise_avg.data_ptr(), float(snr_threshold), lib.stream_ptr(stream)))
    return score, noisy, noise_in


class HysteresisState:
    """Device-resident per-stream state of the look-ahead machine: current silence flag, number of
    decisions emitted, the decisions themselves (1 = silence) and the running background level."""

    def __init__(self, n_streams: int, capacity: int, device, noise_init: float = 4.0):
        import torch
        self.silence = torch.ones((n_streams,), dtype=torch.uint8, device=device)
        self.n_saved = torch.zeros((n_streams,), dtype=torch.int32, device=device)
        self.saved = torch.zeros((n_streams, capacity), dtype=torch.uint8, device=device)
        self.noise_avg = torch.full((n_streams,), float(np.float32(noise_init)), dtype=torch.float32, device=device)

    def segments(self, max_segments: int | None = None, stream=None):
        """-> (seg_count int32 [S], segments int32 [S, max, 2]) frame pairs (start, end-exclusive)."""
        import torch
        S, cap = self.saved.shape
        max_segments = max_segments or cap // 2 + 1
        cnt = torch.empty((S,), dtype=torch.int32, device=self.saved.device)
        seg = torch.empty((S, max_segments, 2), dtype=torch.int32, device=self.saved.device)
        lib.check(lib.load().vadx_runs_to_segments(self.saved.data_ptr(), cap, self.n_saved.data_ptr(), S,
                                                   cnt.data_ptr(), seg.data_ptr(), max_segments,
                                                   lib.stream_ptr(stream)))
        return cnt, seg


def runs_to_timestamps(pairs, n_flags: int, frame_duration: float):
    """frame pairs of one stream -> [(start_s, end_s)] in Python floats, exactly like vad_to_timestamps
    (FSMN/Inference_FSMN_VAD_ONNX.py:124-141): a run closed by a silence frame i ends at
    i*d + d, a run still open at the end of the stream ends at n*d."""
    out = []
    for a, b in np.asarray(pairs, np.int64).reshape(-1, 2).tolist():
        start = a * frame_duration
        end = b * frame_duration + frame_duration if b < n_flags else n_flags * frame_duration
        out.append((start, end))
    return out


def process_timestamps(timestamps, fusion_threshold: float = 1.0, min_duration: float = 0.5):
    """Drop short segments, then fuse neighbours closer than the threshold -- two passes, like the
    reference (FSMN/Inference_FSMN_VAD_ONNX.py:102-122)."""
    cur = [(a, b) for a, b in timestamps if (b - a) >= min_duration]
    for _ in range(2):
        nxt = []
        for a, b in cur:
            if nxt and (a - nxt[-1][1] <= fusion_threshold):
                nxt[-1] = (nxt[-1][0], b)
            else:
                nxt.append((a, b))
        cur = nxt
    return cur


def format_time(seconds: float) -> str:
    """hh:mm:ss.mmm with truncated milliseconds (FSMN/Inference_FSMN_VAD_ONNX.py:144-153)."""
    td = timedelta(seconds=seconds)
    total = td.total_seconds()
    whole = int(total)
    ms = int((total - whole) * 1000)
    h, rem = divmod(whole, 3600)
    m, s = divmod(rem, 60)
    return f"{h:02}:{m:02}:{s:02}.{ms:03}"


def timestamp_lines(timestamps, sample_rate: int = 16000):
    """-> (lines_seconds, lines_indices) exactly as the reference writes them."""
    sec = [f"{format_time(a)} --> {format_time(b)}\n" for a, b in timestamps]
    idx = [f"{int(a * sample_rate)} --> {int(b * sample_rate)}\n" for a, b in timestamps]
    return sec, idx


def write_timestamp_files(timestamps, path_second: str, path_indices: str, sample_rate: int = 16000):
    sec, idx = timestamp_lines(timestamps, sample_rate)
    with open(path_second, "w", encoding="UTF-8") as f:
        f.writelines(sec)
    with open(path_indices, "w", encoding="UTF-8") as f:
        f.writelines(idx)


class StreamVadPostprocessor:
    """Device twin of the reference's StreamVadPostprocessor (FireRedVAD/Inference_FireRed_ONNX.py:307-490)
    for S streams in lock-step.  Same constructor arguments; `process_batch(probs)` keeps the reference's
    meaning per stream (segments closed in this call, then the still-open segment up to the last frame
    seen) and the state -- ring buffer, counters, open segment -- stays in HBM between calls."""

    def __init__(self, smooth_window_size, speech_threshold, pad_start_frame, min_speech_frame, max_speech_frame,
                 min_silence_frame, n_streams: int = 1, max_segments: int = 256, device=None,
                 frames_per_second: int = 100):
        import torch
        self.cfg = lib.StreamPostCfg(max(1, int(smooth_window_size)), float(np.float32(speech_threshold)),
                                     int(pad_start_frame), int(min_speech_frame), int(max_speech_frame),
                                     int(min_silence_frame))
        self.S, self.max_segments = int(n_streams), int(max_segments)
        self.inv_fps = 1.0 / frames_per_second
        dev = device or torch.device("cuda", torch.cuda.current_device())
        words = lib.load().vadx_stream_post_state_words(self.cfg.smooth_window)
        self.state = torch.zeros((self.S, words), dtype=torch.int32, device=dev)
        self.seg_count = torch.zeros((self.S,), dtype=torch.int32, device=dev)
        self.segments = torch.empty((self.S, self.max_segments, 2), dtype=torch.int32, device=dev)
        self.open = torch.full((self.S, 2), -1, dtype=torch.int32, device=dev)

    def reset(self):
        self.state.zero_()
        self.seg_count.zero_()
        self.open.fill_(-1)

    def feed(self, probs, n_frames=None, stream=None):
        """probs CUDA fp32 [S, T] (this call's frames), n_frames optional CUDA int32 [S].  Asynchronous;
        closed segments accumulate in self.segments / self.seg_count, the open one lands in self.open."""
        import torch
        if not (torch.is_tensor(probs) and probs.is_cuda and probs.dtype == torch.float32 and probs.dim() == 2
                and probs.shape[0] == self.S and probs.stride(1) == 1):
            raise ValueError(f"StreamVadPostprocessor.feed: probs must be CUDA fp32 [{self.S}, T] with contiguous rows")
        if n_frames is not None and not (n_frames.is_cuda and n_frames.dtype == torch.int32 and n_frames.numel() == self.S):
            raise ValueError("StreamVadPostprocessor.feed: n_frames must be a CUDA int32 tensor [S]")
        T = probs.shape[1]
        lib.check(lib.load().vadx_stream_postprocess(probs.data_ptr(), probs.stride(0) if T else 0, lib.ptr(n_frames), self.S,
                                                     T, C.byref(self.cfg), self.state.data_ptr(),
                                                     self.seg_count.data_ptr(), self.segments.data_ptr(),
                                                     self.max_segments, self.open.data_ptr(), lib.stream_ptr(stream)))

    def timestamps(self, first_segment=None):
        """Per stream [(start_s, end_s)]: the closed segments from index first_segment[s] on, then the
        open one.  float64 products frame * (1.0 / fps), as the reference (:352, :465-474)."""
        cnt = self.seg_count.cpu().numpy()
        if int(cnt.max(initial=0)) > self.max_segments:
            raise RuntimeError(f"StreamVadPostprocessor: a stream closed {int(cnt.max())} segments, more than "
                               f"max_segments={self.max_segments}")
        seg = self.segments.cpu().numpy()
        opn = self.open.cpu().numpy()
        out = []
        for s in range(self.S):
            k0 = 0 if first_segment is None else int(first_segment[s])
            ts = [(int(a) * self.inv_fps, int(b) * self.inv_fps) for a, b in seg[s, k0:cnt[s]]]
            if opn[s, 0] >= 0:
                ts.append((int(opn[s, 0]) * self.inv_fps, int(opn[s, 1]) * self.inv_fps))
            out.append(ts)
        return out

    def process_batch(self, raw_probs):
        """The reference's call for ONE stream (numpy or CUDA [T]) or S streams ([S, T]); returns the
        list(s) of (start_s, end_s) this call reports."""
        import torch
        p = raw_probs if torch.is_tensor(raw_probs) else torch.from_numpy(np.ascontiguousarray(raw_probs, np.float32))
        single = p.dim() == 1
        p = p.reshape(1, -1) if single else p
        if p.shape[1] == 0:
            return [] if single else [[] for _ in range(self.S)]
        before = self.seg_count.cpu().numpy().copy()
        self.feed(p.to(self.state.device, torch.float32).contiguous())
        ts = self.timestamps(before)
        return ts[0] if single else ts
