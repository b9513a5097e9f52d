"""FSMN-VAD entry point -- the B200 twin of FSMN/Inference_FSMN_VAD_ONNX.py: raw audio in, speech
timestamps (seconds + sample indices) out, same two text files.

Per chunk the reference calls the graph (:177-187), walks the look-ahead hysteresis in Python
(:188-215) and updates the background level (:217-218).  Here all three run on the device for S
streams in lock-step, the stream state (FSMN caches, silence flag, background level, decisions)
never leaves HBM, and nothing synchronises with the host until the segments are read back.
Config names and defaults follow the reference's module-level constants (:15-24).
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from . import audio_io, lib, postprocess as PP, serve, weights as W
from .session import FsmnSession

SAMPLE_RATE = 16000
ONE_MINUS_SPEECH_THRESHOLD = 1.0
SNR_THRESHOLD = 10.0
BACKGROUND_NOISE_dB_INIT = 30.0
FUSION_THRESHOLD = 0.3
MIN_SPEECH_DURATION = 0.2
SPEAKING_SCORE = 0.5
SILENCE_SCORE = 0.5
LOOK_BACKWARD = 0.3
OUTPUT_FRAME_LENGTH = 160


@dataclass
class FsmnResult:
    timestamps: list
    saved: np.ndarray            # bool per emitted frame, True = silence (the reference's `saved`)
    lines_second: list
    lines_indices: list
    p_silence: list              # per chunk [T] (debug / parity)
    power_dB: list
    noise_avg_in: list


def look_backward_frames(look_backward_s: float) -> int:
    return int(look_backward_s * SAMPLE_RATE // OUTPUT_FRAME_LENGTH)


def run_streams(session: FsmnSession, aligned, stride: int, look_backward_s: float = LOOK_BACKWARD,
                one_minus_speech_threshold: float = ONE_MINUS_SPEECH_THRESHOLD, snr_threshold_db: float = SNR_THRESHOLD,
                noise_init_db: float = BACKGROUND_NOISE_dB_INIT, speaking_score: float = SPEAKING_SCORE,
                silence_score: float = SILENCE_SCORE, keep_trace: bool = False, stream=None, graph: bool = False,
                whole: bool = False):
    """aligned: CUDA int16 [S, n] (already chunk-aligned, see audio_io.align_overlapping).
    -> (HysteresisState, trace) with every decision of every stream on the device.
    whole=True computes ALL windows of the recordings in one pass (FsmnSession.run_windows: two launches-worth of work
    instead of one graph per window; the only sequential part, the running background level, is one small kernel).
    graph=True captures one window (forward + hysteresis + cache hand-over, ~30 kernels) into a CUDA
    graph and replays it per window: the per-window cost drops from ~30 launches to one, which is
    what matters for few streams and short chunks (the reference's 512-sample configuration)."""
    import torch
    if whole:
        return _run_streams_whole(session, aligned, stride, look_backward_s, one_minus_speech_threshold, snr_threshold_db,
                                  noise_init_db, speaking_score, silence_score, keep_trace, stream)
    if graph and not keep_trace:
        return _run_streams_graph(session, aligned, stride, look_backward_s, one_minus_speech_threshold,
                                  snr_threshold_db, noise_init_db, speaking_score, silence_score), []
    S, n = aligned.shape
    L, T = session.chunk_len, session.T
    lb = look_backward_frames(look_backward_s)
    n_windows = (n - L) // stride + 1
    state = PP.HysteresisState(S, n_windows * (T - lb) + lb, aligned.device,
                               noise_init=float(np.float32(noise_init_db + snr_threshold_db) * np.float32(0.1)))
    caches = session.new_caches(S, aligned.device)
    snr = snr_threshold_db * 0.1
    trace = []
    for wdx in range(n_windows):
        s0 = wdx * stride
        chunk = aligned[:, s0:s0 + L].contiguous()
        noise_in = state.noise_avg.clone() if keep_trace else None
        score, caches, noisy, p_sil, power = session.run_batch(chunk, caches, state.noise_avg,
                                                               one_minus_speech_threshold, stream)
        PP.lookahead_hysteresis(score, state, lb, speaking_score, silence_score, is_final=(wdx == n_windows - 1),
                                noisy_dB=noisy, snr_threshold=snr, stream=stream)
        if keep_trace:
            trace.append((score, p_sil, power, noise_in, noisy))
    return state, trace


def _run_streams_whole(session, aligned, stride, look_backward_s, thr, snr_threshold_db, noise_init_db, speaking_score,
                       silence_score, keep_trace, stream):
    S, n = aligned.shape
    L, T = session.chunk_len, session.T
    lb = look_backward_frames(look_backward_s)
    n_windows = (n - L) // stride + 1
    state = PP.HysteresisState(S, n_windows * (T - lb) + lb, aligned.device,
                               noise_init=float(np.float32(noise_init_db + snr_threshold_db) * np.float32(0.1)))
    p_sil, power, _caches = session.run_windows(aligned, stride, session.new_caches(S, aligned.device), stream)
    score, noisy, noise_in = PP.fsmn_gate_hysteresis_windows(p_sil, power, state, lb, speaking_score, silence_score, thr,
                                                             session.cfg.speech_2_noise_ratio, snr_threshold_db * 0.1,
                                                             keep_trace=keep_trace, stream=stream)
    trace = []
    if keep_trace:
        trace = [(score[:, w], p_sil[:, w], power[:, w], noise_in[:, w], noisy[:, w]) for w in range(n_windows)]
    return state, trace


class _GraphRunner:
    """Static buffers + one captured window (forward, hysteresis, cache hand-over) for a fixed
    (streams, chunk length, thresholds) configuration; kept on the session and reused across calls, so
    a steady caller pays the capture once."""

    def __init__(self, session, S, lb, capacity, device, thr, snr, speaking_score, silence_score):
        import torch
        self.session, self.S, self.lb, self.capacity = session, S, lb, capacity
        self.thr, self.snr, self.speaking, self.silence = thr, snr, speaking_score, silence_score
        self.state = PP.HysteresisState(S, capacity, device)
        self.caches = session.new_caches(S, device)
        self.chunk = torch.empty((S, session.chunk_len), dtype=torch.int16, device=device)
        self.graph = None

    def reset(self, noise_init: float):
        s = self.state
        s.silence.fill_(1)
        s.n_saved.zero_()
        s.noise_avg.fill_(float(np.float32(noise_init)))
        for c in self.caches:
            c.zero_()

    def window(self, is_final: bool):
        score, new, noisy, _, _ = self.session.run_batch(self.chunk, self.caches, self.state.noise_avg, self.thr)
        PP.lookahead_hysteresis(score, self.state, self.lb, self.speaking, self.silence, is_final=is_final, noisy_dB=noisy,
                                snr_threshold=self.snr)
        for c, nw in zip(self.caches, new):
            c.copy_(nw)

    def replay(self):
        import torch
        if self.graph is None:
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self.window(False)
            self.graph = g
        self.graph.replay()


def _run_streams_graph(session, aligned, stride, look_backward_s, thr, snr_threshold_db, noise_init_db, speaking_score,
                       silence_score):
    """NOTE: the returned HysteresisState belongs to the cached runner and is overwritten by the next
    graph-mode call on this session with the same configuration; read the segments before that."""
    S, n = aligned.shape
    L, T = session.chunk_len, session.T
    lb = look_backward_frames(look_backward_s)
    n_windows = (n - L) // stride + 1
    need = n_windows * (T - lb) + lb
    runners = session.__dict__.setdefault("_graph_runners", {})
    key = (S, L, lb, float(thr), float(snr_threshold_db), float(speaking_score), float(silence_score), str(aligned.device))
    r = runners.get(key)
    if r is None or r.capacity < need:
        r = _GraphRunner(session, S, lb, max(need, 1 << 15), aligned.device, thr, snr_threshold_db * 0.1, speaking_score,
                         silence_score)
        runners[key] = r
    r.reset(float(np.float32(noise_init_db + snr_threshold_db) * np.float32(0.1)))
    for wdx in range(n_windows):
        r.chunk.copy_(aligned[:, wdx * stride:wdx * stride + L])
        if wdx == n_windows - 1:
            r.window(True)        # the final-window variant flushes the look-ahead buffer: eager
        elif wdx == 0 and r.graph is None:
            r.window(False)       # first ever window eager: uploads constants, warms the allocator
        else:
            r.replay()
    return r.state


class StreamServer(serve.SlotServer):
    """Live FSMN-VAD serving with the reference's final timestamps as events: n_slots independent stream slots advance
    one reference window per tick.  A stream may start in any free slot on any tick.  Windows follow the reference
    (audio_io.align_overlapping): window k covers samples [k*stride, k*stride + L), L = session.chunk_len,
    stride = L - (look_backward_frames + 1) * 160; at the defaults a tick is 11040 samples (690 ms).  Per tick and slot
    the caller gives the chunk (int16 [stride]), the number of valid samples n and a `last` flag:

        n > 0, last 0   feed a full chunk (n == full_chunk(received))
        n > 0, last 1   feed the stream's last chunk (may be short), then finalize and free the slot
        n = 0, last 0   hold: window, caches, level and machine are unchanged
        n = 0, last 1   finalize and free the slot without new audio

    A slot first collects the stream's first L samples: until then a full chunk is min(stride, L - received), and the
    tick that completes them runs the first window; every later fed tick runs one more.  A short last chunk, or a
    stream shorter than L, is zero-padded to its window (the reference pads with unseeded Gaussian noise).  Audio is
    raw int16: the reference's whole-file peak normalisation is not causal, so the offline twin is
    run_vad(..., normalize=False).  Each tick is the window load, one forward of the session over [n_slots][L], the
    look-ahead hysteresis, the level update, the timestamp machine and the event compaction, replayed as one CUDA graph
    per cache parity.  Its result (serve.FsmnServeTick) is a compact list of (slot, kind, decision) events, each emitted as
    soon as it is certain: kind 0 = a segment starts, 1 = it ends (closed by silence decision b), 2 = it was open when
    the stream ended.  host_seconds() / host_indices() give exactly the reference's final timestamps (minimum duration
    and fusion applied).  Decisions count from the stream's first window, so a stream may run 2^31 of them.

    The defaults are the module constants, which are the reference's.  Inputs go through the static buffers `chunk`,
    `n_samples`, `last`: step() copies the arguments it is given into them (non-blocking from pinned host memory), or a
    producer writes them and calls step() with no arguments.  Whether a chunk is full depends on the slot's samples so
    far, so the device checks that rule.  The session stays usable between ticks."""

    check_short = False

    def __init__(self, session: FsmnSession, n_slots: int, look_backward_s: float = LOOK_BACKWARD,
                 one_minus_speech_threshold: float = ONE_MINUS_SPEECH_THRESHOLD, snr_threshold_db: float = SNR_THRESHOLD,
                 noise_init_db: float = BACKGROUND_NOISE_dB_INIT, speaking_score: float = SPEAKING_SCORE,
                 silence_score: float = SILENCE_SCORE, fusion_threshold: float = FUSION_THRESHOLD,
                 min_speech_duration: float = MIN_SPEECH_DURATION, device=None, graph: bool = True):
        import torch
        if not isinstance(session, FsmnSession):
            raise ValueError("StreamServer needs an FsmnSession")
        S, L, T = int(n_slots), session.chunk_len, session.T
        lb = look_backward_frames(look_backward_s)
        stride = L - (lb + 1) * OUTPUT_FRAME_LENGTH
        if S < 1:
            raise ValueError(f"StreamServer: n_slots must be at least 1, got {n_slots}")
        if stride <= 0:
            raise ValueError(f"StreamServer: a {L}-sample window is too short for a look-backward of {lb} frames")
        if L % 8:
            raise ValueError(f"StreamServer: the session's chunk_len {L} must be a multiple of 8")
        self.session, self.L, self.T, self.lb, self.stride = session, L, T, lb, stride
        super().__init__(S, stride, device, graph)
        dev = self.device
        self.thr = float(one_minus_speech_threshold)
        self.noise_init = float(np.float32(noise_init_db + snr_threshold_db) * np.float32(0.1))
        self.window = torch.zeros((S, L), dtype=torch.int16, device=dev)      # the forward's input, one row per slot
        self.noise_avg = torch.zeros((S,), dtype=torch.float32, device=dev)  # the gate's level, written by the load
        self.score = torch.zeros((S, T), dtype=torch.uint8, device=dev)
        self.noisy = torch.zeros((S,), dtype=torch.float32, device=dev)
        self.caches = [torch.zeros((session.cfg.fsmn_layers, S) + session.cache_shape, dtype=torch.float32, device=dev)
                       for _ in range(2)]
        with torch.cuda.device(dev):
            self.seg = serve.FsmnSlotSegmenter(S, T, L, lb, speaking_score, silence_score, snr_threshold_db * 0.1,
                                               self.noise_init, fusion_threshold, min_speech_duration, dev)

    def full_chunk(self, received: int) -> int:
        """samples of a full chunk for a stream that has sent `received` samples so far"""
        return self.seg.full_chunk(received)

    def _tick(self, i: int):
        """the tick body on the static buffers; only libvadx launches"""
        lib.check(lib.load().vadx_fsmn_serve_load(
            self.chunk.data_ptr(), self.n_samples.data_ptr(), self.last.data_ptr(), self.seg.state.data_ptr(), self.S,
            self.L, self.stride, self.lb, self.noise_init, self.window.data_ptr(), self.noise_avg.data_ptr(),
            lib.stream_ptr()))
        self.session.run_batch(self.window, self.caches[i].unbind(0), self.noise_avg, self.thr,
                               out=(self.score, self.noisy, None, None), caches_out=self.caches[1 - i].unbind(0))
        self.seg.enqueue(self.score, self.noisy, self.n_samples, self.last, i, self.caches[i], self.caches[1 - i])

    def _tick_probs(self):
        return self.score


def run_vad(audio, session: FsmnSession, look_backward_s: float = LOOK_BACKWARD, rng=None,
            save_timestamps_second: str | None = None, save_timestamps_indices: str | None = None,
            fusion_threshold: float = FUSION_THRESHOLD, min_speech_duration: float = MIN_SPEECH_DURATION,
            normalize: bool = True, keep_trace: bool = False, graph: bool = False, whole: bool = False) -> FsmnResult:
    """One stream, the reference's behaviour: `audio` is a wav path or an int16/float array.
    whole=True: all windows in one pass (see run_streams); graph=True: one CUDA-graph replay per window."""
    import torch
    if isinstance(audio, str):
        audio = audio_io.load_wav_int16(audio, SAMPLE_RATE)
    a16 = audio_io.normalize_to_int16(np.asarray(audio, np.float32)) if normalize else np.asarray(audio, np.int16)
    lb = look_backward_frames(look_backward_s)
    aligned, stride, _n = audio_io.align_overlapping(a16, session.chunk_len, lb, OUTPUT_FRAME_LENGTH, rng)
    d = torch.from_numpy(aligned).cuda().unsqueeze(0)
    state, trace = run_streams(session, d, stride, look_backward_s, keep_trace=keep_trace, graph=graph, whole=whole)
    cnt, seg = state.segments()
    n_flags = int(state.n_saved[0].item())
    pairs = PP.take_segments(cnt, seg, 0)
    frame_d = OUTPUT_FRAME_LENGTH / SAMPLE_RATE
    ts = PP.process_timestamps(PP.runs_to_timestamps(pairs, n_flags, frame_d), fusion_threshold, min_speech_duration)
    sec, idx = PP.timestamp_lines(ts, SAMPLE_RATE)
    if save_timestamps_second and save_timestamps_indices:
        PP.write_timestamp_files(ts, save_timestamps_second, save_timestamps_indices, SAMPLE_RATE)
    saved = state.saved[0, :n_flags].cpu().numpy().astype(bool)
    return FsmnResult(ts, saved, sec, idx, [t[1][0].cpu().numpy() for t in trace],
                      [t[2][0].cpu().numpy() for t in trace], [float(t[3][0]) for t in trace])


def main(argv=None):
    import argparse
    ap = argparse.ArgumentParser(description="FSMN-VAD on B200 (random-init weights unless --weights is given)")
    ap.add_argument("audio")
    ap.add_argument("--weights", help=".npz with the FunASR encoder state_dict + cmvn_means/cmvn_vars")
    ap.add_argument("--chunk", type=int, default=16000)
    ap.add_argument("--look-backward", type=float, default=LOOK_BACKWARD)
    ap.add_argument("--out-second", default="./timestamps_second.txt")
    ap.add_argument("--out-indices", default="./timestamps_indices.txt")
    a = ap.parse_args(argv)
    cfg = W.FsmnConfig()
    w = dict(np.load(a.weights)) if a.weights else W.fsmn_random_init(cfg, 0)
    sess = FsmnSession(w, cfg, chunk_len=a.chunk)
    r = run_vad(a.audio, sess, a.look_backward, save_timestamps_second=a.out_second,
                save_timestamps_indices=a.out_indices)
    print("\nTimestamps in Second:")
    print("".join(r.lines_second), end="")
    print("\nTimestamps in Indices:")
    print("".join(r.lines_indices), end="")


if __name__ == "__main__":
    main()
