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


SERVE_START, SERVE_END, SERVE_END_OF_STREAM = 0, 1, 2      # event kinds of the slot server (include/vadx.h)
SERVE_ERR_RANGE, SERVE_ERR_SHORT = 1, 2                    # error bits: n_samples out of range, short chunk not last


class ServeTickError(ValueError):
    """A tick in which the device rejected some slots' control words.  Those slots were held (left unchanged); every
    other slot advanced, and its events are in `events` (as host_events / host_seconds would have returned them), so
    a caller that catches this loses no segment.  `error` holds the VADX_SERVE_ERR_* bits."""

    def __init__(self, msg, events, error):
        super().__init__(msg)
        self.events, self.error = events, error


class ServeTick:
    """One tick of the slot server.  Device side: `events` int32 [n_max, 3] (slot, kind, frame) of which the first
    `n_events[0]` rows are this tick's, `error` (int32 [1], VADX_SERVE_ERR_* bits), `probs` fp32 [n_slots, T] and
    `frames` int32 [n_slots] (the frames of `probs` each slot consumed).  probs and frames are valid until the next
    tick; events, n_events and the host read-back until the tick after that."""

    def __init__(self, owner, tick, parity, probs, frames, done):
        self._owner, self._tick, self._i, self._done = owner, tick, parity, done
        self.events, self.n_events, self.error = owner.events[parity], owner.header[parity][0:1], owner.header[parity][1:2]
        self.probs, self.frames = probs, frames

    def host_events(self):
        """-> [(slot, kind, frame)] ordered by slot, then emission order.  Waits for the tick; raises ServeTickError
        (a ValueError carrying the tick's events) if some slot's control words broke the contract on the device."""
        if self._owner.ticks - self._tick > 2:
            raise RuntimeError("ServeTick.host_events: two later ticks have reused this tick's buffers")
        self._done.synchronize()
        n, err = (int(v) for v in self._owner.h_header[self._i])
        events = [tuple(e) for e in self._owner.h_events[self._i][:n].tolist()]
        if err:
            what = [m for b, m in ((SERVE_ERR_RANGE, "n_samples outside [0, chunk_samples]"),
                                   (SERVE_ERR_SHORT, "a short chunk that is not the stream's last")) if err & b]
            raise ServeTickError(f"stream server: rejected slot control words ({'; '.join(what)}); those slots were "
                                 "held, the events of the others are in .events", events, err)
        return events

    def host_seconds(self):
        """-> [(slot, kind, seconds)], seconds = frame * (1 / frames_per_second) as StreamVadPostprocessor.timestamps
        forms.  A ServeTickError carries its events in seconds."""
        inv = self._owner.inv_fps
        try:
            return [(s, k, int(f) * inv) for s, k, f in self.host_events()]
        except ServeTickError as e:
            e.events = [(s, k, int(f) * inv) for s, k, f in e.events]
            raise

    @property
    def d2h_bytes(self) -> int:
        """bytes the device sent to the host for this tick (header + events); read after host_events()"""
        return 8 + 12 * int(self._owner.h_header[self._i][0])


class StreamSlotSegmenter:
    """The segmenter and slot lifecycle of the Stream-VAD slot server (vadx_stream_serve_step) for n_slots slots:
    segmenter state (vadx_stream_post_state_words per slot, the layout StreamVadPostprocessor uses), scratch, and two
    sets of event buffers (device and pinned host) used by alternate ticks.  `step` takes one tick's probabilities
    fp32 [n_slots, n_frames] and control words; with caches it also holds / zeroes them.  Without a model it runs the
    segmenter on given probabilities."""

    def __init__(self, smooth_window_size, speech_threshold, pad_start_frame, min_speech_frame, max_speech_frame,
                 min_silence_frame, n_slots: int, n_frames: int, chunk_samples: int, frame_len: int = 400,
                 frame_hop: int = 160, device=None, frames_per_second: int = 100):
        import torch
        self.cfg = lib.StreamPostCfg(max(1, int(smooth_window_size)), float(np.float32(speech_threshold)),
                                     int(pad_start_frame), int(min_speech_frame), int(max_speech_frame),
                                     int(min_silence_frame))
        self.S, self.T = int(n_slots), int(n_frames)
        self.chunk_samples, self.frame_len, self.frame_hop = int(chunk_samples), int(frame_len), int(frame_hop)
        self.inv_fps = 1.0 / frames_per_second
        dev = device or torch.device("cuda", torch.cuda.current_device())
        L = lib.load()
        need = C.c_size_t()
        lib.check(L.vadx_stream_serve_step(None, self.T, self.T, None, None, self.S, self.chunk_samples, self.frame_len,
                                           self.frame_hop, C.byref(self.cfg), None, None, None, 0, 0, None, None, None,
                                           None, None, None, 0, C.byref(need), None))
        self.scratch = torch.empty((need.value,), dtype=torch.uint8, device=dev)
        self.state = torch.zeros((self.S, L.vadx_stream_post_state_words(self.cfg.smooth_window)), dtype=torch.int32,
                                 device=dev)
        self.frames = torch.zeros((self.S,), dtype=torch.int32, device=dev)
        n_max = self.S * (2 * self.T + 1)
        self.events = [torch.zeros((n_max, 3), dtype=torch.int32, device=dev) for _ in range(2)]
        self.header = [torch.zeros((2,), dtype=torch.int32, device=dev) for _ in range(2)]
        self.h_events = [torch.zeros((n_max, 3), dtype=torch.int32).pin_memory() for _ in range(2)]
        self.h_header = [torch.zeros((2,), dtype=torch.int32).pin_memory() for _ in range(2)]
        self.ticks = 0

    def reset(self):
        """every slot idle (state zeroed); caches are the caller's"""
        self.state.zero_()

    def enqueue(self, probs, n_samples, last, parity: int, caches_in=None, caches_out=None, stream=None):
        """Enqueue vadx_stream_serve_step for one tick (no checks beyond pointers: the server checks shapes once)."""
        c = caches_in
        lib.check(lib.load().vadx_stream_serve_step(
            probs.data_ptr(), probs.stride(0), self.T, n_samples.data_ptr(), last.data_ptr(), self.S, self.chunk_samples,
            self.frame_len, self.frame_hop, C.byref(self.cfg), self.state.data_ptr(), lib.ptr(c), lib.ptr(caches_out),
            c.shape[0] if c is not None else 0, (c.shape[2] * c.shape[3]) if c is not None else 0, self.frames.data_ptr(),
            self.events[parity].data_ptr(), self.header[parity].data_ptr(), self.h_events[parity].data_ptr(),
            self.h_header[parity].data_ptr(), self.scratch.data_ptr(), self.scratch.numel(), None, lib.stream_ptr(stream)))

    def step(self, probs, n_samples, last, caches_in=None, caches_out=None, stream=None) -> ServeTick:
        """One tick on given CUDA tensors: probs fp32 [n_slots, >= n_frames] with contiguous rows, n_samples int32
        [n_slots], last bool / uint8 [n_slots], caches fp32 [R, n_slots, P, Lb] (both or neither, distinct)."""
        import torch
        if not (torch.is_tensor(probs) and probs.is_cuda and probs.dtype == torch.float32 and probs.dim() == 2
                and probs.shape[0] == self.S and probs.shape[1] >= self.T and probs.stride(1) == 1):
            raise ValueError(f"StreamSlotSegmenter.step: probs must be CUDA fp32 [{self.S}, >= {self.T}] with contiguous rows")
        _check_control(n_samples, last, self.S, "StreamSlotSegmenter.step", cuda=True)
        if (caches_in is None) != (caches_out is None):
            raise ValueError("StreamSlotSegmenter.step: caches_in and caches_out go together")
        if caches_in is not None:
            for c in (caches_in, caches_out):
                if not (c.is_cuda and c.dtype == torch.float32 and c.dim() == 4 and c.shape[1] == self.S
                        and c.is_contiguous() and c.shape == caches_in.shape):
                    raise ValueError(f"StreamSlotSegmenter.step: caches must be contiguous CUDA fp32 [R, {self.S}, P, Lb]")
            if caches_in.data_ptr() == caches_out.data_ptr():
                raise ValueError("StreamSlotSegmenter.step: caches_out must be distinct from caches_in")
        i = self.ticks & 1
        self.enqueue(probs, n_samples, last.view(torch.uint8), i, caches_in, caches_out, stream)
        return self.finish(i, probs, stream)

    def finish(self, parity, probs, stream=None) -> ServeTick:
        import torch
        done = torch.cuda.Event()
        done.record(stream)
        t = ServeTick(self, self.ticks, parity, probs, self.frames, done)
        self.ticks += 1
        return t


class SileroServeTick(ServeTick):
    """One tick of the Silero slot server (SileroSlotSegmenter).  As ServeTick, but `events` hold (slot, kind, window),
    `frames` the windows each slot consumed and `probs` is fp32 [n_slots, W] (a view of the forward's [W][n_slots]
    output).  host_samples / host_seconds convert windows to what the reference VADIterator returns."""

    def _value(self, kind, w):
        """the reference's float arithmetic (utils_vad.py:566-585): current_sample = (w + 1) * 512 after window w"""
        o = self._owner
        if kind == SERVE_START:
            return max(0, (w + 1) * o.window - o.speech_pad_samples - o.window)
        if kind == SERVE_END:
            return (w + 1) * o.window + o.speech_pad_samples - o.window
        return w * o.window                          # end of stream: the samples consumed

    def _converted(self, conv):
        try:
            return [(s, k, conv(self._value(k, int(w)))) for s, k, w in self.host_events()]
        except ServeTickError as e:
            e.events = [(s, k, conv(self._value(k, int(w)))) for s, k, w in e.events]
            raise

    def host_samples(self):
        """-> [(slot, kind, sample)] as VADIterator(...)(window) returns them; an end-of-stream event gives the samples
        consumed.  A ServeTickError carries its events in samples."""
        return self._converted(int)

    def host_seconds(self, time_resolution: int = 1):
        """-> [(slot, kind, seconds)] as VADIterator(...)(window, return_seconds=True, time_resolution) returns them"""
        sr = self._owner.sampling_rate
        return self._converted(lambda v: round(v / sr, time_resolution))


class SileroSlotSegmenter:
    """The VADIterator machine and slot lifecycle of the Silero slot server (vadx_silero_serve_step) for n_slots slots
    and W windows per tick: iterator state (3 int32 words per slot), scratch, and two sets of event buffers (device and
    pinned host) used by alternate ticks.  `step` runs it on given probabilities fp32 [W, n_slots], without a model.
    The defaults are the reference VADIterator constructor's."""

    STATE_WORDS = 3
    window = 512
    sampling_rate = 16000

    def __init__(self, threshold: float = 0.5, min_silence_duration_ms: int = 100, speech_pad_ms: int = 30,
                 n_slots: int = 1, windows_per_tick: int = 5, device=None):
        import torch
        self.threshold = float(threshold)
        self.min_silence_samples = self.sampling_rate * min_silence_duration_ms / 1000
        self.speech_pad_samples = self.sampling_rate * speech_pad_ms / 1000
        self.S, self.W = int(n_slots), int(windows_per_tick)
        dev = device or torch.device("cuda", torch.cuda.current_device())
        need = C.c_size_t()
        lib.check(lib.load().vadx_silero_serve_step(None, self.S, None, None, self.S, self.W, self.threshold,
                                                    self.min_silence_samples, None, None, None, None, None, None, None,
                                                    None, None, None, 0, C.byref(need), None))
        self.scratch = torch.empty((need.value,), dtype=torch.uint8, device=dev)
        self.state = torch.zeros((self.S, self.STATE_WORDS), dtype=torch.int32, device=dev)
        self.frames = torch.zeros((self.S,), dtype=torch.int32, device=dev)
        n_max = self.S * (self.W + 1)
        self.events = [torch.zeros((n_max, 3), dtype=torch.int32, device=dev) for _ in range(2)]
        self.header = [torch.zeros((2,), dtype=torch.int32, device=dev) for _ in range(2)]
        self.h_events = [torch.zeros((n_max, 3), dtype=torch.int32).pin_memory() for _ in range(2)]
        self.h_header = [torch.zeros((2,), dtype=torch.int32).pin_memory() for _ in range(2)]
        self.ticks = 0

    def reset(self):
        """every slot idle (state zeroed); the model input and LSTM state are the caller's"""
        self.state.zero_()

    def enqueue(self, probs, n_samples, last, parity: int, x=None, state_in=None, state_out=None, stream=None):
        """Enqueue vadx_silero_serve_step for one tick (no checks beyond pointers: the server checks shapes once)."""
        lib.check(lib.load().vadx_silero_serve_step(
            probs.data_ptr(), probs.stride(0), n_samples.data_ptr(), last.data_ptr(), self.S, self.W, self.threshold,
            self.min_silence_samples, self.state.data_ptr(), lib.ptr(x), lib.ptr(state_in), lib.ptr(state_out),
            self.frames.data_ptr(), self.events[parity].data_ptr(), self.header[parity].data_ptr(),
            self.h_events[parity].data_ptr(), self.h_header[parity].data_ptr(), self.scratch.data_ptr(),
            self.scratch.numel(), None, lib.stream_ptr(stream)))

    def step(self, probs, n_samples, last, stream=None) -> SileroServeTick:
        """One tick on given CUDA tensors: probs fp32 [W, n_slots] with contiguous rows, n_samples int32 [n_slots]
        (in [0, W*512]), last bool / uint8 [n_slots]."""
        import torch
        if not (torch.is_tensor(probs) and probs.is_cuda and probs.dtype == torch.float32 and probs.dim() == 2
                and tuple(probs.shape) == (self.W, self.S) and probs.stride(1) == 1):
            raise ValueError(f"SileroSlotSegmenter.step: probs must be CUDA fp32 [{self.W}, {self.S}] with contiguous rows")
        _check_control(n_samples, last, self.S, "SileroSlotSegmenter.step", cuda=True)
        i = self.ticks & 1
        self.enqueue(probs, n_samples, last.view(torch.uint8), i, stream=stream)
        return self.finish(i, probs, stream)

    def finish(self, parity, probs, stream=None) -> SileroServeTick:
        """probs: the tick's [W, n_slots] probabilities"""
        import torch
        done = torch.cuda.Event()
        done.record(stream)
        t = SileroServeTick(self, self.ticks, parity, probs.t(), self.frames, done)
        self.ticks += 1
        return t


def load_tick_inputs(who, chunk, n_samples, last, dst_chunk, dst_n_samples, dst_last, device):
    """A slot server's step(chunk, n_samples, last): checks the arguments against the static buffers and copies them in
    (non-blocking from pinned host memory).  Host control words are checked here, before anything is copied; control
    words already on the device are checked by the serve kernel.  None for all three leaves the buffers as they are."""
    import torch
    given = [a is not None for a in (chunk, n_samples, last)]
    if any(given) and not all(given):
        raise ValueError(f"{who}: pass chunk, n_samples and last together, or none of them")
    if not all(given):
        return
    S, L = dst_chunk.shape
    if not (torch.is_tensor(chunk) and chunk.dtype == torch.int16 and tuple(chunk.shape) == (S, L)):
        raise ValueError(f"{who}: chunk must be an int16 tensor [{S}, {L}]")
    _check_control(n_samples, last, S, who)
    for a in (chunk, n_samples, last):
        if a.is_cuda and a.device != device:
            raise ValueError(f"{who}: inputs must be on {device} or in host memory")
    if not n_samples.is_cuda:
        n = n_samples.numpy()
        if n.min(initial=0) < 0 or n.max(initial=0) > L:
            raise ValueError(f"{who}: n_samples must be in [0, {L}]")
        if not last.is_cuda:
            short = (n > 0) & (n < L) & (last.view(torch.uint8).numpy() == 0)
            if short.any():
                raise ValueError(f"{who}: slots {np.flatnonzero(short)[:8].tolist()} got a short chunk "
                                 "that is not their stream's last")
    dst_chunk.copy_(chunk, non_blocking=True)
    dst_n_samples.copy_(n_samples, non_blocking=True)
    dst_last.copy_(last.view(torch.uint8), non_blocking=True)


def _check_control(n_samples, last, S, who, cuda=None):
    """dtype / shape of a tick's control arrays; cuda=True requires them on the device"""
    import torch
    if not (torch.is_tensor(n_samples) and n_samples.dtype == torch.int32 and tuple(n_samples.shape) == (S,)
            and n_samples.is_contiguous()):
        raise ValueError(f"{who}: n_samples must be a contiguous int32 tensor [{S}]")
    if not (torch.is_tensor(last) and last.dtype in (torch.bool, torch.uint8) and tuple(last.shape) == (S,)
            and last.is_contiguous()):
        raise ValueError(f"{who}: last must be a contiguous bool or uint8 tensor [{S}]")
    if cuda and not (n_samples.is_cuda and last.is_cuda):
        raise ValueError(f"{who}: n_samples and last must be CUDA tensors")
