"""MarbleNet entry point -- the B200 twin of NVIDIA_Frame_VAD_Multilingual_MarbleNet/
Inference_NVIDIA_MarbleNet_VAD_ONNX.py: raw audio in, speech timestamps out, same two text files.
Config names and defaults follow the reference's module-level constants (:15-30)."""
from __future__ import annotations

import numpy as np

from . import audio_io, lib, postprocess as PP, serve, weights as W
from .firered_vad import VadResult
from .session import MarbleNetSession

IN_SAMPLE_RATE = 16000
OUTPUT_FRAME_LENGTH = 320
OUTPUT_FRAME_SHIFT_S = OUTPUT_FRAME_LENGTH / 16000
SPEAKING_SCORE = 0.5
SMOOTH_WINDOW_SIZE = 3
MIN_SPEECH_FRAME = 10
MAX_SPEECH_FRAME = 1000
MIN_SILENCE_FRAME = 10
MERGE_SILENCE_FRAME = 3
EXTEND_SPEECH_FRAME = 0

POST_DEFAULT = PP.FramePostConfig(SMOOTH_WINDOW_SIZE, SPEAKING_SCORE, MIN_SPEECH_FRAME, MAX_SPEECH_FRAME,
                                  MIN_SILENCE_FRAME, MERGE_SILENCE_FRAME, EXTEND_SPEECH_FRAME, OUTPUT_FRAME_SHIFT_S,
                                  0.025, False)


def normalise_audio(audio: np.ndarray, target_rms: float = 8192.0) -> np.ndarray:
    """Optional loader normalisation (:112-120)."""
    a = audio.astype(np.float32)
    rms = np.sqrt(np.mean(a * a, dtype=np.float32), dtype=np.float32)
    if rms > 0:
        a *= (target_rms / (rms + 1e-7))
        np.clip(a, -32768.0, 32767.0, out=a)
        return a.astype(np.int16)
    return audio


def run_vad_clips(session: MarbleNetSession, clips, post: PP.FramePostConfig = POST_DEFAULT, stream=None):
    """clips: CUDA int16 [S, L] (one window per stream, the dynamic-axis mode of the reference).
    -> (active probs [S, T'-1] view, decisions, seg_count, segments) on the device."""
    scores = session.run_batch(clips, stream=stream)
    n = scores.shape[2] - 1                       # signal_len = T' - 1 (:366-373)
    probs = scores[1, :, :n]
    dec, cnt, seg = PP.postprocess_frames(probs, post, None, stream=stream)
    return probs, dec, cnt, seg


def run_vad_windows(session: MarbleNetSession, windows, post: PP.FramePostConfig = POST_DEFAULT, stream=None):
    """windows: CUDA int16 [S, n_windows, L] -- every stream's recording cut into non-overlapping windows of L samples
    (audio_io.align_non_overlapping; the reference's static-axis mode and its split of recordings longer than one hour,
    :130-147).  All S * n_windows windows go through the network as ONE batch; each window contributes its signal_len
    valid frames, the per-stream concatenation (:358-378) is post-processed on the device.
    -> (probs [S, n_windows * (T'-1)], decisions, seg_count, segments)."""
    S, n_win, L = windows.shape
    scores = session.run_batch(windows.reshape(S * n_win, L), stream=stream)        # [2, S*n_win, T']
    n = scores.shape[2] - 1                                                         # signal_len = T' - 1 (:366-373)
    probs = scores[1, :, :n].reshape(S, n_win * n)
    dec, cnt, seg = PP.postprocess_frames(probs, post, None, stream=stream)
    return probs, dec, cnt, seg


class StreamServer(serve.SlotServer):
    """Live MarbleNet Frame-VAD serving with the reference's timestamps as events: n_slots independent stream slots
    advance one static-axis window of L = window_samples samples per tick, the reference's non-overlapping windows
    (audio_io.align_non_overlapping), of which the first F = session.frames(L) - 1 frames count (signal_len).  At
    L = 16000 a tick is 1 s of 50 frames.  A stream may start in any free slot on any tick.  Per tick and slot the caller
    gives the chunk (int16 [L]), the number of valid samples n and a `last` flag:

        n > 0, last 0   feed a full chunk (n == L)
        n > 0, last 1   feed the stream's last chunk (may be short), then finalize and free the slot
        n = 0, last 0   hold: the slot is unchanged
        n = 0, last 1   finalize and free the slot without new audio

    A short last chunk is zero-padded to L (the reference pads with RMS-matched noise from the unseeded global numpy
    generator), so the offline twin is run_vad(..., input_audio_length=L) with zero noise.  Audio is raw int16:
    normalise_audio is off by default in the reference and is not causal.  Each tick is the tail zeroing, one forward of
    the session over [n_slots][L] and the online VadPostprocessor with the event compaction (vadx_marblenet_serve_step),
    replayed as a CUDA graph.  Its result (serve.MarbleNetServeTick) is a compact list of (slot, kind, value) events, each
    emitted as soon as it is certain: kind 0 = a segment starts at frame a, 1 = it ends before frame b (max-speech cuts
    included), 2 = it was open when the stream ended (the value is the reference's float32 end).  host_seconds() /
    host_indices() give exactly run_vad's timestamps.  Frames count from the stream's first window as int32, so a
    stream may run 2^31 frames.

    `post` is the post-processor's configuration (the reference's module constants by default).  Inputs go through the
    static buffers `chunk`, `n_samples`, `last`: step() copies the arguments it is given into them (non-blocking from
    pinned host memory), or a producer writes them and calls step() with no arguments.  `probs` is the tick's active
    probabilities fp32 [n_slots, F] (a view of the forward's static output).  The session stays usable between ticks."""

    def __init__(self, session: MarbleNetSession, n_slots: int, window_samples: int = 16000,
                 post: PP.FramePostConfig = POST_DEFAULT, device=None, graph: bool = True):
        import torch
        if not isinstance(session, MarbleNetSession):
            raise ValueError("StreamServer needs a MarbleNetSession")
        if session.in_sample_rate != IN_SAMPLE_RATE:
            raise ValueError(f"StreamServer: the session must take {IN_SAMPLE_RATE} Hz audio, not {session.in_sample_rate}")
        S, L = int(n_slots), int(window_samples)
        if S < 1:
            raise ValueError(f"StreamServer: n_slots must be at least 1, got {n_slots}")
        if L < 1:
            raise ValueError(f"StreamServer: window_samples must be at least 1, got {window_samples}")
        T = session.frames(L)
        F = T - 1
        if F < 1:
            raise ValueError(f"StreamServer: a {L}-sample window gives no frame (signal_len = {F})")
        if post.tail_adds_frame_length:
            raise ValueError("StreamServer: MarbleNet's open tail ends at n * frame_shift (post.tail_adds_frame_length "
                             "must be False)")
        self.session, self.L, self.T, self.F, self.post = session, L, T, F, post
        super().__init__(S, L, device, graph)
        self.scores = torch.zeros((2, S, T), dtype=torch.float32, device=self.device)   # the forward's static output
        with torch.cuda.device(self.device):
            self.seg = serve.MarbleNetSlotSegmenter(post, S, F, L, self.device)

    def _tick(self, i: int):
        """the tick body on the static buffers; only libvadx launches (the model keeps no state, so i is unused)"""
        lib.check(lib.load().vadx_stream_serve_zero_tail(self.chunk.data_ptr(), self.L, self.n_samples.data_ptr(), self.S,
                                                         self.L, self.L, lib.stream_ptr()))
        self.session.run_batch(self.chunk, out=self.scores)
        self.seg.enqueue(self._tick_probs(), self.n_samples, self.last, i)

    def _tick_probs(self):
        return self.scores[1, :, :self.F]


def run_vad(audio, session: MarbleNetSession, post: PP.FramePostConfig = POST_DEFAULT, normalize: bool = False,
            save_timestamps_second: str | None = None, save_timestamps_indices: str | None = None,
            input_audio_length: int | None = None, rng=None) -> VadResult:
    """One recording, the reference's behaviour (:121-147, :355-403).  input_audio_length = the export's static audio axis
    (the reference reads it from _inputs_meta[0].shape[-1]); None = the dynamic axis: one window of min(one hour, the
    recording).  Longer recordings are cut into non-overlapping windows, the last one padded with RMS-matched noise (`rng`
    makes the padding reproducible), all windows run as one batch and their valid frames are concatenated."""
    import torch
    if isinstance(audio, str):
        audio = audio_io.load_wav_int16(audio, IN_SAMPLE_RATE)
    audio = np.asarray(audio, np.int16)
    if normalize:
        audio = normalise_audio(audio)
    audio_len = len(audio)
    L = int(input_audio_length) if input_audio_length else min(IN_SAMPLE_RATE * 3600, audio_len)
    if audio_len == L:
        d = torch.from_numpy(audio).cuda().unsqueeze(0)
        probs, dec, cnt, seg = run_vad_clips(session, d, post)
    else:
        windows, _ = audio_io.align_non_overlapping(audio, L, rng)
        probs, dec, cnt, seg = run_vad_windows(session, torch.from_numpy(windows).cuda().unsqueeze(0), post)
    n = probs.shape[1]
    pairs = PP.take_segments(cnt, seg, 0)
    ts = PP.segments_to_seconds(pairs, n, post, audio_len / IN_SAMPLE_RATE)
    sec, idx = PP.timestamp_lines(ts, IN_SAMPLE_RATE)
    if save_timestamps_second and save_timestamps_indices:
        PP.write_timestamp_files(ts, save_timestamps_second, save_timestamps_indices, IN_SAMPLE_RATE)
    return VadResult(ts, probs[0].cpu().numpy(), dec[0, :n].cpu().numpy(), sec, idx)


def main(argv=None):
    import argparse
    ap = argparse.ArgumentParser(description="MarbleNet Frame-VAD on B200 (random-init weights unless --weights is given)")
    ap.add_argument("audio")
    ap.add_argument("--weights", help=".npz with the NeMo state_dict")
    ap.add_argument("--out-second", default="./timestamps_second.txt")
    ap.add_argument("--out-indices", default="./timestamps_indices.txt")
    a = ap.parse_args(argv)
    cfg = W.MarbleNetConfig()
    w = dict(np.load(a.weights)) if a.weights else W.marblenet_random_init(cfg, 0)
    r = run_vad(a.audio, MarbleNetSession(w, cfg), save_timestamps_second=a.out_second,
                save_timestamps_indices=a.out_indices)
    print("\nTimestamps in Second:")
    print("".join(r.lines_second), end="")
    print("\nTimestamps in Indices:")
    print("".join(r.lines_indices), end="")


if __name__ == "__main__":
    main()
