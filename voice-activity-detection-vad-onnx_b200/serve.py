"""Host side of the slot servers (firered_vad, silero_vad, fsmn_vad and marblenet_vad.StreamServer): the control words
and their checks, the segmenters with their two parities of event buffers, the tick handles, and the CUDA-graph runner
of a tick body.  The device side is the vadx_*_serve_* entry points of csrc/postproc.cu (include/vadx.h)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import lib

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

    RANGE_TEXT = "n_samples outside [0, chunk_samples]"

    def __init__(self, owner, tick, parity, probs, done):
        self._owner, self._tick, self._i, self._done = owner, tick, parity, done
        self.events, self.n_events, self.error = owner.events[parity], owner.header[parity][0:1], owner.header[parity][1:2]
        self.probs, self.frames = probs, owner.frames

    def host_events(self):
        """-> [(slot, kind, frame)] ordered by slot, then emission order.  Waits for the tick; raises ServeTickError
        (a ValueError carrying the tick's events) if some slot's control words broke the contract on the device."""
        if self._owner.ticks - self._tick > 2:
            raise RuntimeError("ServeTick.host_events: two later ticks have reused this tick's buffers")
        self._done.synchronize()
        n, err = (int(v) for v in self._owner.h_header[self._i])
        events = [tuple(e) for e in self._owner.h_events[self._i][:n].tolist()]
        if err:
            what = [m for b, m in ((SERVE_ERR_RANGE, self.RANGE_TEXT),
                                   (SERVE_ERR_SHORT, "a short chunk that is not the stream's last")) if err & b]
            raise ServeTickError(f"stream server: rejected slot control words ({'; '.join(what)}); those slots were "
                                 "held, the events of the others are in .events", events, err)
        return events

    def _converted(self, fn):
        """host_events() as (slot, kind, fn(kind, value)); a ServeTickError carries its events converted alike"""
        try:
            return [(s, k, fn(k, int(v))) for s, k, v in self.host_events()]
        except ServeTickError as e:
            e.events = [(s, k, fn(k, int(v))) for s, k, v in e.events]
            raise

    def host_seconds(self):
        """-> [(slot, kind, seconds)], seconds = frame * (1 / frames_per_second) as StreamVadPostprocessor.timestamps
        forms.  A ServeTickError carries its events in seconds."""
        inv = self._owner.inv_fps
        return self._converted(lambda k, f: f * inv)

    @property
    def d2h_bytes(self) -> int:
        """bytes the device sent to the host for this tick (header + events); read after host_events()"""
        return 8 + 12 * int(self._owner.h_header[self._i][0])


class _SlotSegmenter:
    """What the slot segmenters share: per-slot `state` (state_words int32), `scratch`, `frames` (what each slot
    consumed this tick), two sets of event buffers (device and pinned host, events_per_slot rows of (slot, kind, value)
    per slot) used by alternate ticks, and the tick count.  A family sets S before calling __init__, builds
    `tick_class` handles and defines enqueue(..., parity, ..., stream=None)."""

    tick_class = ServeTick

    def __init__(self, state_words: int, scratch_bytes: int, events_per_slot: int, device):
        import torch
        dev = device or torch.device("cuda", torch.cuda.current_device())
        self.scratch = torch.empty((scratch_bytes,), dtype=torch.uint8, device=dev)
        self.state = torch.zeros((self.S, state_words), dtype=torch.int32, device=dev)
        self.frames = torch.zeros((self.S,), dtype=torch.int32, device=dev)
        n_max = self.S * events_per_slot
        self.events = [torch.zeros((n_max, 3), dtype=torch.int32, device=dev) for _ in range(2)]
        self.header = [torch.zeros((2,), dtype=torch.int32, device=dev) for _ in range(2)]
        self.h_events = [torch.zeros((n_max, 3), dtype=torch.int32).pin_memory() for _ in range(2)]
        self.h_header = [torch.zeros((2,), dtype=torch.int32).pin_memory() for _ in range(2)]
        self.ticks = 0

    def reset(self):
        """every slot idle (state zeroed); the model's buffers (caches, input rows, LSTM state) are the caller's"""
        self.state.zero_()

    def _outputs(self, parity: int):
        """the arguments every vadx_*_serve_step call ends with, before its stream: frames, the event buffers of this
        parity and their host mirrors, scratch and its size, and no scratch_needed (this is a tick, not a size query)"""
        return (self.frames.data_ptr(), self.events[parity].data_ptr(), self.header[parity].data_ptr(),
                self.h_events[parity].data_ptr(), self.h_header[parity].data_ptr(), self.scratch.data_ptr(),
                self.scratch.numel(), None)

    def _step(self, probs, n_samples, last, stream, *inputs, **extra):
        """step() after the family's input checks: checks the control words, then enqueue(*inputs, n_samples, last,
        parity, **extra) and the tick's handle with `probs` [n_slots, ...]"""
        import torch
        _check_control(n_samples, last, self.S, f"{type(self).__name__}.step", cuda=True)
        i = self.ticks & 1
        self.enqueue(*inputs, n_samples, last.view(torch.uint8), i, stream=stream, **extra)
        return self.finish(i, probs, stream)

    def finish(self, parity, probs, stream=None) -> ServeTick:
        """the handle of the tick just enqueued on `stream` with the event buffers of `parity`; probs [n_slots, ...]"""
        import torch
        done = torch.cuda.Event()
        done.record(stream)
        t = self.tick_class(self, self.ticks, parity, probs, done)
        self.ticks += 1
        return t


class StreamSlotSegmenter(_SlotSegmenter):
    """The segmenter and slot lifecycle of the Stream-VAD slot server (vadx_stream_serve_step) for n_slots slots:
    segmenter state (vadx_stream_post_state_words per slot, the layout StreamVadPostprocessor uses), scratch, and two
    sets of event buffers (device and pinned host) used by alternate ticks.  `step` takes one tick's probabilities
    fp32 [n_slots, n_frames] and control words; with caches it also holds / zeroes them.  Without a model it runs the
    segmenter on given probabilities."""

    def __init__(self, smooth_window_size, speech_threshold, pad_start_frame, min_speech_frame, max_speech_frame,
                 min_silence_frame, n_slots: int, n_frames: int, chunk_samples: int, frame_len: int = 400,
                 frame_hop: int = 160, device=None, frames_per_second: int = 100):
        self.cfg = lib.StreamPostCfg(max(1, int(smooth_window_size)), float(np.float32(speech_threshold)),
                                     int(pad_start_frame), int(min_speech_frame), int(max_speech_frame),
                                     int(min_silence_frame))
        self.S, self.T = int(n_slots), int(n_frames)
        self.chunk_samples, self.frame_len, self.frame_hop = int(chunk_samples), int(frame_len), int(frame_hop)
        self.inv_fps = 1.0 / frames_per_second
        L = lib.load()
        need = C.c_size_t()
        lib.check(L.vadx_stream_serve_step(None, self.T, self.T, None, None, self.S, self.chunk_samples, self.frame_len,
                                           self.frame_hop, C.byref(self.cfg), None, None, None, 0, 0, None, None, None,
                                           None, None, None, 0, C.byref(need), None))
        super().__init__(L.vadx_stream_post_state_words(self.cfg.smooth_window), need.value, 2 * self.T + 1, device)

    def enqueue(self, probs, n_samples, last, parity: int, caches_in=None, caches_out=None, stream=None):
        """Enqueue vadx_stream_serve_step for one tick (no checks beyond pointers: the server checks shapes once)."""
        c = caches_in
        lib.check(lib.load().vadx_stream_serve_step(
            probs.data_ptr(), probs.stride(0), self.T, n_samples.data_ptr(), last.data_ptr(), self.S, self.chunk_samples,
            self.frame_len, self.frame_hop, C.byref(self.cfg), self.state.data_ptr(), lib.ptr(c), lib.ptr(caches_out),
            c.shape[0] if c is not None else 0, (c.shape[2] * c.shape[3]) if c is not None else 0,
            *self._outputs(parity), lib.stream_ptr(stream)))

    def step(self, probs, n_samples, last, caches_in=None, caches_out=None, stream=None) -> ServeTick:
        """One tick on given CUDA tensors: probs fp32 [n_slots, >= n_frames] with contiguous rows, n_samples int32
        [n_slots], last bool / uint8 [n_slots], caches fp32 [R, n_slots, P, Lb] (both or neither, distinct)."""
        import torch
        if not (torch.is_tensor(probs) and probs.is_cuda and probs.dtype == torch.float32 and probs.dim() == 2
                and probs.shape[0] == self.S and probs.shape[1] >= self.T and probs.stride(1) == 1):
            raise ValueError(f"StreamSlotSegmenter.step: probs must be CUDA fp32 [{self.S}, >= {self.T}] with contiguous rows")
        if (caches_in is None) != (caches_out is None):
            raise ValueError("StreamSlotSegmenter.step: caches_in and caches_out go together")
        if caches_in is not None:
            for c in (caches_in, caches_out):
                if not (c.is_cuda and c.dtype == torch.float32 and c.dim() == 4 and c.shape[1] == self.S
                        and c.is_contiguous() and c.shape == caches_in.shape):
                    raise ValueError(f"StreamSlotSegmenter.step: caches must be contiguous CUDA fp32 [R, {self.S}, P, Lb]")
            if caches_in.data_ptr() == caches_out.data_ptr():
                raise ValueError("StreamSlotSegmenter.step: caches_out must be distinct from caches_in")
        return self._step(probs, n_samples, last, stream, probs, caches_in=caches_in, caches_out=caches_out)


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

    def host_samples(self):
        """-> [(slot, kind, sample)] as VADIterator(...)(window) returns them; an end-of-stream event gives the samples
        consumed.  A ServeTickError carries its events in samples."""
        return self._converted(lambda k, w: int(self._value(k, w)))

    def host_seconds(self, time_resolution: int = 1):
        """-> [(slot, kind, seconds)] as VADIterator(...)(window, return_seconds=True, time_resolution) returns them"""
        sr = self._owner.sampling_rate
        return self._converted(lambda k, w: round(self._value(k, w) / sr, time_resolution))


class SileroSlotSegmenter(_SlotSegmenter):
    """The VADIterator machine and slot lifecycle of the Silero slot server (vadx_silero_serve_step) for n_slots slots
    and W windows per tick: iterator state (3 int32 words per slot), scratch, and two sets of event buffers (device and
    pinned host) used by alternate ticks.  `step` runs it on given probabilities fp32 [W, n_slots], without a model.
    The defaults are the reference VADIterator constructor's."""

    STATE_WORDS = 3
    window = 512
    sampling_rate = 16000
    tick_class = SileroServeTick

    def __init__(self, threshold: float = 0.5, min_silence_duration_ms: int = 100, speech_pad_ms: int = 30,
                 n_slots: int = 1, windows_per_tick: int = 5, device=None):
        self.threshold = float(threshold)
        self.min_silence_samples = self.sampling_rate * min_silence_duration_ms / 1000
        self.speech_pad_samples = self.sampling_rate * speech_pad_ms / 1000
        self.S, self.W = int(n_slots), int(windows_per_tick)
        need = C.c_size_t()
        lib.check(lib.load().vadx_silero_serve_step(None, self.S, None, None, self.S, self.W, self.threshold,
                                                    self.min_silence_samples, None, None, None, None, None, None, None,
                                                    None, None, None, 0, C.byref(need), None))
        super().__init__(self.STATE_WORDS, need.value, self.W + 1, device)

    def enqueue(self, probs, n_samples, last, parity: int, x=None, state_in=None, state_out=None, stream=None):
        """Enqueue vadx_silero_serve_step for one tick (no checks beyond pointers: the server checks shapes once)."""
        lib.check(lib.load().vadx_silero_serve_step(
            probs.data_ptr(), probs.stride(0), n_samples.data_ptr(), last.data_ptr(), self.S, self.W, self.threshold,
            self.min_silence_samples, self.state.data_ptr(), lib.ptr(x), lib.ptr(state_in), lib.ptr(state_out),
            *self._outputs(parity), lib.stream_ptr(stream)))

    def step(self, probs, n_samples, last, stream=None) -> SileroServeTick:
        """One tick on given CUDA tensors: probs fp32 [W, n_slots] with contiguous rows, n_samples int32 [n_slots]
        (in [0, W*512]), last bool / uint8 [n_slots]."""
        import torch
        if not (torch.is_tensor(probs) and probs.is_cuda and probs.dtype == torch.float32 and probs.dim() == 2
                and tuple(probs.shape) == (self.W, self.S) and probs.stride(1) == 1):
            raise ValueError(f"SileroSlotSegmenter.step: probs must be CUDA fp32 [{self.W}, {self.S}] with contiguous rows")
        return self._step(probs.t(), n_samples, last, stream, probs)


class FsmnServeTick(ServeTick):
    """One tick of the FSMN slot server (FsmnSlotSegmenter).  As ServeTick, but `events` hold (slot, kind, decision),
    `frames` the decisions each slot made this tick and `probs` is the tick's score flags uint8 [n_slots, T].
    host_seconds / host_indices give the reference's final timestamps (process_timestamps after runs_to_timestamps)."""

    RANGE_TEXT = "n_samples outside [0, full_chunk(received)]"

    def _seconds(self, kind, i):
        """the reference's doubles (FSMN/Inference_FSMN_VAD_ONNX.py:124-141)"""
        d = self._owner.frame_duration
        return i * d + d if kind == SERVE_END else i * d

    def host_seconds(self):
        """-> [(slot, kind, seconds)]: START a*d, END b*d + d, END_OF_STREAM n*d, d = 160 / 16000.  Pairing one stream's
        starts and ends gives its process_timestamps(runs_to_timestamps(...)) list.  A ServeTickError carries its events
        in seconds."""
        return self._converted(self._seconds)

    def host_indices(self):
        """-> [(slot, kind, sample)], int(seconds * 16000) as the reference's indices file writes them"""
        sr = self._owner.sampling_rate
        return self._converted(lambda k, i: int(self._seconds(k, i) * sr))


class FsmnSlotSegmenter(_SlotSegmenter):
    """The look-ahead hysteresis, background level, timestamp machine and slot lifecycle of the FSMN slot server
    (vadx_fsmn_serve_step) for n_slots slots: state (vadx_fsmn_serve_state_words int32 per slot), scratch, and two sets
    of event buffers (device and pinned host) used by alternate ticks.  `step` runs it on given score flags uint8
    [n_slots, T] (0 / 1, as the gate writes them) and noisy_dB fp32 [n_slots], without a model; a slot only consumes
    them on ticks that run a window (see fsmn_vad.StreamServer).  Seconds per decision: 160 / 16000."""

    sampling_rate = 16000
    frame_duration = 160 / 16000
    tick_class = FsmnServeTick

    def __init__(self, n_slots: int, n_frames: int, chunk_len: int, look_backward: int, speaking_score: float = 0.5,
                 silence_score: float = 0.5, snr_threshold: float = 1.0, noise_init: float = 4.0,
                 fusion_threshold: float = 0.3, min_speech_duration: float = 0.2, device=None):
        self.S, self.T, self.L, self.lb = int(n_slots), int(n_frames), int(chunk_len), int(look_backward)
        self.stride = self.L - (self.lb + 1) * 160
        self.cfg = lib.FsmnServeCfg(float(speaking_score), float(silence_score), self.frame_duration,
                                    float(fusion_threshold), float(min_speech_duration), float(snr_threshold),
                                    float(np.float32(noise_init)))
        L = lib.load()
        need = C.c_size_t()
        lib.check(L.vadx_fsmn_serve_step(None, self.T, None, self.T, None, None, self.S, self.L, self.stride, self.lb,
                                         C.byref(self.cfg), None, None, None, 0, 0, None, None, None, None, None, None, 0,
                                         C.byref(need), None))
        super().__init__(L.vadx_fsmn_serve_state_words(self.lb), need.value, 2 * self.T + 2, device)

    def full_chunk(self, received: int) -> int:
        """samples of a full chunk for a stream that has sent `received` samples so far"""
        return min(self.stride, self.L - received) if received < self.L else self.stride

    def enqueue(self, score, noisy_dB, n_samples, last, parity: int, caches_in=None, caches_out=None, stream=None):
        """Enqueue vadx_fsmn_serve_step for one tick (no checks beyond pointers: the server checks shapes once)."""
        c = caches_in
        lib.check(lib.load().vadx_fsmn_serve_step(
            score.data_ptr(), score.stride(0), noisy_dB.data_ptr(), self.T, n_samples.data_ptr(), last.data_ptr(), self.S,
            self.L, self.stride, self.lb, C.byref(self.cfg), self.state.data_ptr(), lib.ptr(c), lib.ptr(caches_out),
            c.shape[0] if c is not None else 0, (c.shape[2] * c.shape[3]) if c is not None else 0,
            *self._outputs(parity), lib.stream_ptr(stream)))

    def step(self, score, noisy_dB, n_samples, last, stream=None) -> FsmnServeTick:
        """One tick on given CUDA tensors: score uint8 [n_slots, >= T] with contiguous rows, noisy_dB fp32 [n_slots],
        n_samples int32 [n_slots], last bool / uint8 [n_slots]."""
        import torch
        if not (torch.is_tensor(score) and score.is_cuda and score.dtype == torch.uint8 and score.dim() == 2
                and score.shape[0] == self.S and score.shape[1] >= self.T and score.stride(1) == 1):
            raise ValueError(f"FsmnSlotSegmenter.step: score must be CUDA uint8 [{self.S}, >= {self.T}] with contiguous rows")
        if not (torch.is_tensor(noisy_dB) and noisy_dB.is_cuda and noisy_dB.dtype == torch.float32
                and tuple(noisy_dB.shape) == (self.S,) and noisy_dB.is_contiguous()):
            raise ValueError(f"FsmnSlotSegmenter.step: noisy_dB must be a contiguous CUDA fp32 tensor [{self.S}]")
        return self._step(score, n_samples, last, stream, score, noisy_dB)


class MarbleNetServeTick(ServeTick):
    """One tick of the MarbleNet slot server (MarbleNetSlotSegmenter).  As ServeTick, but `events` hold (slot, kind,
    value): a frame for START / END, the bit pattern of the reference's float32 end for END_OF_STREAM.  host_seconds /
    host_indices give the reference's timestamps (VadPostprocessor.decision_to_segment)."""

    def _seconds(self, kind, v):
        """round(float32(frame) * float32(frame_shift), 3), or the float32 end of an open last segment"""
        if kind == SERVE_END_OF_STREAM:
            return round(float(np.array(v, np.int32).view(np.float32)), 3)
        return round(float(np.float32(v) * self._owner.fs), 3)

    def host_seconds(self):
        """-> [(slot, kind, seconds)].  Pairing one stream's starts and ends gives its marblenet_vad.run_vad timestamps.
        A ServeTickError carries its events in seconds."""
        return self._converted(self._seconds)

    def host_indices(self):
        """-> [(slot, kind, sample)], int(seconds * 16000) as the reference's indices file writes them"""
        return self._converted(lambda k, v: int(self._seconds(k, v) * 16000))


class MarbleNetSlotSegmenter(_SlotSegmenter):
    """The reference's VadPostprocessor, online, and the slot lifecycle of the MarbleNet slot server
    (vadx_marblenet_serve_step) for n_slots slots of F frames per tick: state (vadx_marblenet_serve_state_words int32 per
    slot), scratch, and two sets of event buffers (device and pinned host) used by alternate ticks.  `step` runs it on
    given probabilities fp32 [n_slots, >= F], without a model; a fed slot consumes all F frames (a short last chunk is
    zero-padded to the window).  `post` is a postprocess.FramePostConfig whose open tail ends at n * frame_shift."""

    tick_class = MarbleNetServeTick

    def __init__(self, post, n_slots: int, n_frames: int, window_samples: int, device=None):
        if post.tail_adds_frame_length:
            raise ValueError("MarbleNetSlotSegmenter: the open tail of MarbleNet's post-processor ends at n * frame_shift "
                             "(post.tail_adds_frame_length must be False)")
        self.cfg = post.c_struct()
        self.fs = np.float32(post.frame_shift_s)
        self.S, self.F, self.L = int(n_slots), int(n_frames), int(window_samples)
        L = lib.load()
        words = L.vadx_marblenet_serve_state_words(C.byref(self.cfg))
        if words < 0:
            lib.check(words)
        need = C.c_size_t()
        lib.check(L.vadx_marblenet_serve_step(None, self.F, self.F, None, None, self.S, self.L, C.byref(self.cfg),
                                              float(self.fs), None, None, None, None, None, None, None, 0, C.byref(need),
                                              None))
        self.events_per_slot = 2 * (self.F + self.delay) + 2
        super().__init__(words, need.value, self.events_per_slot, device)

    @property
    def delay(self) -> int:
        """frames after which a decision before the max-speech split is final (include/vadx.h)"""
        c = self.cfg
        d2 = 0 if c.min_speech_frame <= 0 and c.min_silence_frame <= 0 else max(c.min_speech_frame, 1)
        return d2 + (c.smooth_window if c.smooth_window > 1 else 0) + max(c.merge_silence_frame - 1, 0) + \
            max(c.extend_speech_frame, 0)

    def enqueue(self, probs, n_samples, last, parity: int, stream=None):
        """Enqueue vadx_marblenet_serve_step for one tick (no checks beyond pointers: the server checks shapes once)."""
        lib.check(lib.load().vadx_marblenet_serve_step(
            probs.data_ptr(), probs.stride(0), self.F, n_samples.data_ptr(), last.data_ptr(), self.S, self.L,
            C.byref(self.cfg), float(self.fs), self.state.data_ptr(), *self._outputs(parity), lib.stream_ptr(stream)))

    def step(self, probs, n_samples, last, stream=None) -> MarbleNetServeTick:
        """One tick on given CUDA tensors: probs fp32 [n_slots, >= F] with contiguous rows, n_samples int32 [n_slots]
        (in [0, window_samples]), last bool / uint8 [n_slots]."""
        import torch
        if not (torch.is_tensor(probs) and probs.is_cuda and probs.dtype == torch.float32 and probs.dim() == 2
                and probs.shape[0] == self.S and probs.shape[1] >= self.F and probs.stride(1) == 1):
            raise ValueError(f"MarbleNetSlotSegmenter.step: probs must be CUDA fp32 [{self.S}, >= {self.F}] with "
                             "contiguous rows")
        return self._step(probs, n_samples, last, stream, probs)


def load_tick_inputs(who, chunk, n_samples, last, dst_chunk, dst_n_samples, dst_last, device, check_short: bool = True):
    """A slot server's step(chunk, n_samples, last): checks the arguments against the static buffers and copies them in
    (non-blocking from pinned host memory).  Host control words are checked here, before anything is copied; control
    words already on the device are checked by the serve kernel.  None for all three leaves the buffers as they are.
    check_short=False leaves the short-chunk rule to the device (a server whose full chunk depends on the slot's state)."""
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
        if check_short and not last.is_cuda:
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


class _StreamGraphRunner:
    """Two captured tick bodies, body(0) (caches a -> b) and body(1) (b -> a), over static buffers: a 160 ms step is
    ~30 small launches, so eager execution is bound by host launch cost; replay costs one graph launch."""

    def __init__(self, body):
        self.body = body
        self.graphs = [None, None]

    def step(self, k: int):
        """runs body(k & 1)"""
        import torch
        i = k & 1
        if self.graphs[i] is None:
            self.body(i)                             # this step runs eagerly (constants, workspace) ...
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):                # ... and is recorded (not executed) for the later ones
                self.body(i)
            self.graphs[i] = g
        else:
            self.graphs[i].replay()


class SlotServer:
    """What the four StreamServers share: the device, the static input buffers `chunk` int16 [n_slots, chunk width],
    `n_samples` int32 [n_slots] and `last` uint8 [n_slots], the optional graph runner and step().  A family sets `seg`
    (its segmenter) and defines _tick(i), the tick body on the static buffers with model state parity i (only libvadx
    launches, so it can be captured), and _tick_probs(), the tensor a tick's handle exposes as `probs`."""

    check_short = True          # False: a full chunk depends on the slot's state, so only the device checks short chunks

    def __init__(self, n_slots: int, chunk_width: int, device, graph: bool):
        import torch
        dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.S, self.device = int(n_slots), dev
        self.chunk = torch.zeros((self.S, chunk_width), dtype=torch.int16, device=dev)
        self.n_samples = torch.zeros((self.S,), dtype=torch.int32, device=dev)
        self.last = torch.zeros((self.S,), dtype=torch.uint8, device=dev)
        self._runner = _StreamGraphRunner(self._tick) if graph else None

    def step(self, chunk=None, n_samples=None, last=None) -> ServeTick:
        """Enqueue one tick on the current stream (asynchronous).  chunk int16 [n_slots, chunk width], n_samples int32
        [n_slots], last bool / uint8 [n_slots]: CUDA tensors, or host tensors (pinned for a non-blocking copy); None
        for all three runs the tick on what the static buffers hold.  Returns the tick's handle (seg.tick_class)."""
        import torch
        with torch.cuda.device(self.device):
            load_tick_inputs("StreamServer.step", chunk, n_samples, last, self.chunk, self.n_samples, self.last,
                             self.device, self.check_short)
            i = self.seg.ticks & 1
            if self._runner is not None:
                self._runner.step(i)
            else:
                self._tick(i)
            return self.seg.finish(i, self._tick_probs())
