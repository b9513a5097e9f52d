"""Silero entry point -- the B200 twin of Silero/Inference_Silero_VAD_ONNX.py (:80-120) and of
`get_speech_timestamps` (Silero/modeling_modified/utils_vad.py:247-491).

The reference calls the model once per 32 ms window and pulls every probability to the host with
`.item()` (:359-372).  Here S streams advance together, the LSTM state and the probabilities stay
in HBM, the trigger / release / max-speech machine runs one stream per lane on the device, and the
host only touches the resulting handful of (start, end) pairs (speech padding + rounding, :464-482).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import audio_io, lib, postprocess as PP, weights as W
from .firered_vad import VadResult, _StreamGraphRunner
from .session import SileroSession

use_fp16 = False
ACTIVATE_THRESHOLD = 0.5
FUSION_THRESHOLD = 0.3
MIN_SPEECH_DURATION = 0.25
MAX_SPEECH_DURATION = 20
MIN_SILENCE_DURATION = 250
SAMPLE_RATE = 16000
INT16_SCALE = 0.000030517578      # the reference's literal (Silero/Inference_Silero_VAD_ONNX.py:83)


def raw_segments(probs, n_samples, threshold: float = 0.5, sampling_rate: int = 16000,
                 min_speech_duration_ms: int = 250, max_speech_duration_s: float = float("inf"),
                 min_silence_duration_ms: int = 100, speech_pad_ms: int = 30, neg_threshold: float | None = None,
                 min_silence_at_max_speech: int = 98, use_max_poss_sil_at_max_speech: bool = True,
                 max_segments: int | None = None, stream=None):
    """probs CUDA fp32 [S, n_windows]; n_samples: list/array of audio lengths.
    -> (seg_count int32 [S], segments int64 [S, max, 2]) on the device: the `speeches` list of the
    reference before padding."""
    import torch
    if sampling_rate != 16000:
        raise ValueError("Currently silero VAD models support 8000 and 16000 (or multiply of 16000) sample rates")
    S, n_win = probs.shape
    window = 512
    speech_pad_samples = sampling_rate * speech_pad_ms / 1000
    cfg = dict(
        threshold=float(threshold),
        neg_threshold=float(max(threshold - 0.15, 0.01) if neg_threshold is None else neg_threshold),
        min_speech_samples=sampling_rate * min_speech_duration_ms / 1000,
        max_speech_samples=sampling_rate * max_speech_duration_s - window - 2 * speech_pad_samples,
        min_silence_samples=sampling_rate * min_silence_duration_ms / 1000,
        min_silence_samples_at_max_speech=sampling_rate * min_silence_at_max_speech / 1000)
    n_samples = np.asarray(n_samples, np.int64).reshape(S)
    n_windows = ((n_samples + window - 1) // window).astype(np.int32)
    if (n_windows > n_win).any():
        raise ValueError("raw_segments: fewer probabilities than windows")
    d_ns = torch.from_numpy(n_samples).to(probs.device)
    d_nw = torch.from_numpy(n_windows).to(probs.device)
    max_segments = max_segments or n_win + 1      # a max-speech cut can close a segment in every window
    cnt = torch.empty((S,), dtype=torch.int32, device=probs.device)
    seg = torch.empty((S, max_segments, 2), dtype=torch.int64, device=probs.device)
    lib.check(lib.load().vadx_silero_timestamps(
        probs.data_ptr(), probs.stride(0), d_nw.data_ptr(), d_ns.data_ptr(), S, cfg["threshold"], cfg["neg_threshold"],
        cfg["min_speech_samples"], cfg["max_speech_samples"], cfg["min_silence_samples"],
        cfg["min_silence_samples_at_max_speech"], window, 1 if use_max_poss_sil_at_max_speech else 0, cnt.data_ptr(),
        seg.data_ptr(), max_segments, lib.stream_ptr(stream)))
    return cnt, seg


def pad_and_convert(pairs, audio_length_samples: int, sampling_rate: int = 16000, speech_pad_ms: int = 30,
                    return_seconds: bool = False, time_resolution: int = 1):
    """utils_vad.py:464-482 on one stream's raw pairs -> list of {'start','end'} dicts."""
    speech_pad_samples = sampling_rate * speech_pad_ms / 1000
    speeches = [{"start": int(a), "end": int(b)} for a, b in np.asarray(pairs, np.int64).reshape(-1, 2).tolist()]
    for i, speech in enumerate(speeches):
        if i == 0:
            speech["start"] = int(max(0, speech["start"] - speech_pad_samples))
        if i != len(speeches) - 1:
            silence_duration = speeches[i + 1]["start"] - speech["end"]
            if silence_duration < 2 * speech_pad_samples:
                speech["end"] += int(silence_duration // 2)
                speeches[i + 1]["start"] = int(max(0, speeches[i + 1]["start"] - silence_duration // 2))
            else:
                speech["end"] = int(min(audio_length_samples, speech["end"] + speech_pad_samples))
                speeches[i + 1]["start"] = int(max(0, speeches[i + 1]["start"] - speech_pad_samples))
        else:
            speech["end"] = int(min(audio_length_samples, speech["end"] + speech_pad_samples))
    if return_seconds:
        audio_length_seconds = audio_length_samples / sampling_rate
        for d in speeches:
            d["start"] = max(round(d["start"] / sampling_rate, time_resolution), 0)
            d["end"] = min(round(d["end"] / sampling_rate, time_resolution), audio_length_seconds)
    return speeches


def get_speech_timestamps(audio, model: SileroSession, threshold: float = 0.5, sampling_rate: int = 16000,
                          min_speech_duration_ms: int = 250, max_speech_duration_s: float = float("inf"),
                          min_silence_duration_ms: int = 100, speech_pad_ms: int = 30, return_seconds: bool = False,
                          time_resolution: int = 1, neg_threshold: float | None = None,
                          min_silence_at_max_speech: int = 98, use_max_poss_sil_at_max_speech: bool = True):
    """Same signature and result as the reference function for one 1-D audio tensor/array (float, already
    scaled); a 2-D [S, n] input returns one list per stream."""
    import torch
    a = audio if torch.is_tensor(audio) else torch.as_tensor(np.asarray(audio, np.float32))
    single = a.dim() == 1
    if single:
        a = a.unsqueeze(0)
    if a.dim() != 2:
        raise ValueError("More than one dimension in audio. Are you trying to process audio with 2 channels?")
    step = 1
    if sampling_rate > 16000 and sampling_rate % 16000 == 0:
        step = sampling_rate // 16000
        sampling_rate = 16000
        a = a[:, ::step]
    if sampling_rate != 16000:
        raise ValueError("Currently silero VAD models support 8000 and 16000 (or multiply of 16000) sample rates")
    d = a.to(model._dev, torch.float32).contiguous()
    n = d.shape[1]
    probs = model.speech_probs(d)
    cnt, seg = raw_segments(probs, [n] * d.shape[0], threshold, sampling_rate, min_speech_duration_ms,
                            max_speech_duration_s, min_silence_duration_ms, speech_pad_ms, neg_threshold,
                            min_silence_at_max_speech, use_max_poss_sil_at_max_speech)
    cnt, seg = PP.take_segments(cnt, seg)
    out = []
    for s in range(d.shape[0]):
        sp = pad_and_convert(seg[s, :cnt[s]], n, sampling_rate, speech_pad_ms, return_seconds, time_resolution)
        if not return_seconds and step > 1:
            for x in sp:
                x["start"] *= step
                x["end"] *= step
        out.append(sp)
    return out[0] if single else out


class VADIterator:
    """Online start/end events for one stream, window by window -- the twin of the reference's VADIterator
    (Silero/modeling_modified/utils_vad.py:494-585) with the same constructor, reset_states() and call.
    `model` is anything with the OnnxWrapper surface (`model(x, sr)` -> [[p]], `reset_states()`), normally a
    vadx.SileroSession, whose LSTM state stays on the device between windows."""

    def __init__(self, model, threshold: float = 0.5, sampling_rate: int = 16000, min_silence_duration_ms: int = 100,
                 speech_pad_ms: int = 30):
        if sampling_rate not in (8000, 16000):
            raise ValueError("VADIterator does not support sampling rates other than [8000, 16000]")
        self.model, self.threshold, self.sampling_rate = model, threshold, sampling_rate
        self.min_silence_samples = sampling_rate * min_silence_duration_ms / 1000
        self.speech_pad_samples = sampling_rate * speech_pad_ms / 1000
        self.reset_states()

    def reset_states(self):
        self.model.reset_states()
        self.triggered = False
        self.temp_end = 0          # sample position where the current below-threshold stretch began (0 = none)
        self.current_sample = 0

    def _fmt(self, samples, return_seconds, time_resolution):
        return round(samples / self.sampling_rate, time_resolution) if return_seconds else int(samples)

    def __call__(self, x, return_seconds: bool = False, time_resolution: int = 1):
        import torch
        if not torch.is_tensor(x):
            try:
                x = torch.Tensor(x)
            except Exception:
                raise TypeError("Audio cannot be casted to tensor. Cast it manually")
        n_win = x.shape[-1]
        self.current_sample += n_win
        p = float(self.model(x, self.sampling_rate).item())
        hot = p >= self.threshold
        if hot:
            self.temp_end = 0
            if not self.triggered:
                self.triggered = True
                start = max(0, self.current_sample - self.speech_pad_samples - n_win)
                return {"start": self._fmt(start, return_seconds, time_resolution)}
            return None
        if self.triggered and p < self.threshold - 0.15:
            if not self.temp_end:
                self.temp_end = self.current_sample
            if self.current_sample - self.temp_end >= self.min_silence_samples:
                end = self.temp_end + self.speech_pad_samples - n_win
                self.temp_end, self.triggered = 0, False
                return {"end": self._fmt(end, return_seconds, time_resolution)}
        return None


class StreamServer:
    """Live Silero serving with VADIterator events: n_slots independent stream slots advance one tick of
    windows_per_tick (W) 512-sample windows at a time (W = 5: 160 ms, W = 1: VADIterator's 32 ms cadence).  A stream
    may start in any free slot on any tick.  Per tick and slot the caller gives the chunk (int16 [W*512]), the number of
    valid samples n and a `last` flag:

        n > 0, last 0   feed a full chunk (n == W*512)
        n > 0, last 1   feed the stream's last chunk (may be short), then finalize and free the slot
        n = 0, last 0   hold: LSTM state, context and iterator state are unchanged
        n = 0, last 1   finalize and free the slot without new audio

    A slot consumes ceil(n/512) windows; a short last window is zero-padded to 512, as get_speech_timestamps pads it.
    Samples past n never influence a result.  Each tick is the int16 load, one forward of the session over all slots
    and W windows, the iterator and the event compaction, replayed as one CUDA graph per LSTM-state parity.  Its result
    (PP.SileroServeTick) is a compact list of (slot, kind, window) events: kind 0 = start (the window the iterator
    triggered on), 1 = end (the window the silence began on, VADIterator's temp_end), 2 = the stream ended while
    triggered (the windows consumed; the reference would leave that segment open).  host_samples() / host_seconds()
    give exactly what VADIterator returns.  Windows count from the stream's first window, so a stream may run 2^31
    windows (about 2.2 years).

    The defaults are the reference VADIterator constructor's.  Inputs go through the static buffers `chunk`,
    `n_samples`, `last`: step() copies the arguments it is given into them (non-blocking from pinned host memory), or a
    producer writes them and calls step() with no arguments.  The session stays usable between ticks."""

    def __init__(self, session: SileroSession, n_slots: int, windows_per_tick: int = 5, threshold: float = 0.5,
                 min_silence_duration_ms: int = 100, speech_pad_ms: int = 30, device=None, graph: bool = True):
        import torch
        if not isinstance(session, SileroSession):
            raise ValueError("StreamServer needs a SileroSession")
        c = session.cfg
        if (c.window, c.context, c.hidden) != (512, 64, 128):
            raise ValueError("StreamServer: the session must be the 16 kHz model (512-sample windows, 64-sample "
                             "context, 128 LSTM units)")
        S, W = int(n_slots), int(windows_per_tick)
        if S < 1:
            raise ValueError(f"StreamServer: n_slots must be at least 1, got {n_slots}")
        if W < 1:
            raise ValueError(f"StreamServer: windows_per_tick must be at least 1, got {windows_per_tick}")
        if S * W > SileroSession.MAX_ROWS_PER_CALL:
            raise ValueError(f"StreamServer: n_slots * windows_per_tick must be at most {SileroSession.MAX_ROWS_PER_CALL}, "
                             f"got {S * W}")
        dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.session, self.S, self.W, self.device = session, S, W, dev
        self.chunk_samples = W * c.window
        self.row_stride = c.context + self.chunk_samples
        self.chunk = torch.zeros((S, self.chunk_samples), dtype=torch.int16, device=dev)
        self.n_samples = torch.zeros((S,), dtype=torch.int32, device=dev)
        self.last = torch.zeros((S,), dtype=torch.uint8, device=dev)
        self.x = torch.zeros((S, self.row_stride), dtype=torch.float32, device=dev)     # [context | chunk] per slot
        self.out = torch.zeros((W, S, 1), dtype=torch.float32, device=dev)
        self.state = [torch.zeros((2, S, c.hidden), dtype=torch.float32, device=dev) for _ in range(2)]
        with torch.cuda.device(dev):
            self.seg = PP.SileroSlotSegmenter(threshold, min_silence_duration_ms, speech_pad_ms, S, W, dev)
        self._runner = _StreamGraphRunner(self._tick) if graph else None
        self._k = 0

    def _tick(self, i: int):
        """the tick body on the static buffers; only libvadx launches"""
        lib.check(lib.load().vadx_silero_serve_load(self.chunk.data_ptr(), self.n_samples.data_ptr(), self.S, self.W,
                                                    self.x.data_ptr(), lib.stream_ptr()))
        self.session.forward_windows(self.x, self.out, self.state[i], self.state[1 - i], self.W, self.row_stride)
        self.seg.enqueue(self.out[:, :, 0], self.n_samples, self.last, i, self.x, self.state[i], self.state[1 - i])

    def step(self, chunk=None, n_samples=None, last=None) -> PP.SileroServeTick:
        """Enqueue one tick on the current stream (asynchronous).  chunk int16 [n_slots, W*512], n_samples int32
        [n_slots], last bool / uint8 [n_slots]: CUDA tensors, or host tensors (pinned for a non-blocking copy); None
        for all three runs the tick on what the static buffers hold.  Returns the tick's handle (PP.SileroServeTick)."""
        import torch
        with torch.cuda.device(self.device):
            PP.load_tick_inputs("StreamServer.step", chunk, n_samples, last, self.chunk, self.n_samples, self.last,
                                self.device)
            if self._runner is not None:
                self._runner.step(self._k)
            else:
                self._tick(self._k & 1)
            self._k += 1
            return self.seg.finish((self._k - 1) & 1, self.out[:, :, 0])


def run_vad(audio, model: SileroSession, save_timestamps_second: str | None = None,
            save_timestamps_indices: str | None = None) -> VadResult:
    """One stream, like the reference script: wav path or int16 array in, fused timestamps out."""
    if isinstance(audio, str):
        audio = audio_io.load_wav_int16(audio, SAMPLE_RATE)
    a = np.array(audio, dtype=np.float32) * INT16_SCALE
    sp = get_speech_timestamps(a, model, threshold=ACTIVATE_THRESHOLD, max_speech_duration_s=MAX_SPEECH_DURATION,
                               min_speech_duration_ms=int(MIN_SPEECH_DURATION * 1000),
                               min_silence_duration_ms=MIN_SILENCE_DURATION, return_seconds=True)
    ts = PP.process_timestamps([(d["start"], d["end"]) for d in sp], FUSION_THRESHOLD, MIN_SPEECH_DURATION)
    sec, idx = PP.timestamp_lines(ts, SAMPLE_RATE)
    if save_timestamps_second and save_timestamps_indices:
        PP.write_timestamp_files(ts, save_timestamps_second, save_timestamps_indices, SAMPLE_RATE)
    return VadResult(ts, None, None, sec, idx)


def main(argv=None):
    import argparse
    ap = argparse.ArgumentParser(description="Silero VAD on B200 (random-init weights unless --weights is given)")
    ap.add_argument("audio")
    ap.add_argument("--weights", help=".npz with the v5 16 kHz state dict")
    ap.add_argument("--out-second", default="./timestamps_second.txt")
    ap.add_argument("--out-indices", default="./timestamps_indices.txt")
    a = ap.parse_args(argv)
    cfg = W.SileroConfig()
    w = dict(np.load(a.weights)) if a.weights else W.silero_random_init(cfg, 0)
    r = run_vad(a.audio, SileroSession(w, cfg), a.out_second, a.out_indices)
    print("\nTimestamps in Second:")
    print("".join(r.lines_second), end="")
    print("\nTimestamps in Indices:")
    print("".join(r.lines_indices), end="")


if __name__ == "__main__":
    main()
