"""FireRedVAD entry point -- the B200 twin of FireRedVAD/Inference_FireRed_ONNX.py: raw audio in, speech
timestamps (seconds + sample indices) out, same two text files.  run_vad = the RUN_VAD section (:523-613),
run_aed = RUN_AED (:620-738, three event tracks), run_stream_vad = RUN_STREAM_VAD (:745-839, 160 ms chunks
with cache carry and the streaming segmenter).

Config names and defaults follow the reference's module-level constants (:26-53).
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from . import audio_io, postprocess as PP, weights as W
from .session import FireRedSession, FireRedStreamSession

IN_SAMPLE_RATE = 16000
INPUT_AUDIO_LENGTH = 16000           # static export axis of the reference graph
SPEAKING_SCORE = 0.4
SMOOTH_WINDOW_SIZE = 5
MIN_SPEECH_FRAME = 20
MAX_SPEECH_FRAME = 2000
MIN_SILENCE_FRAME = 20
MERGE_SILENCE_FRAME = 5
EXTEND_SPEECH_FRAME = 0

# AED (:55-58) and Stream-VAD (:36-37, :60-66) settings
MIN_EVENT_FRAME = 20
MAX_EVENT_FRAME = 2000
SINGING_THRESHOLD = 0.5
MUSIC_THRESHOLD = 0.5
IDX2EVENT = {0: "speech", 1: "singing", 2: "music"}
STREAM_CHUNK_MS = 160
STREAM_CHUNK_SAMPLES = int(IN_SAMPLE_RATE * STREAM_CHUNK_MS / 1000)
WINDOW_LENGTH = 400
HOP_LENGTH = 160
STREAM_VAD_THRESHOLD = 0.4
PAD_START_FRAME = 5
MIN_SPEECH_FRAME_STREAM = 8
MAX_SPEECH_FRAME_STREAM = 2000
MIN_SILENCE_FRAME_STREAM = 20

POST_DEFAULT = PP.FramePostConfig(SMOOTH_WINDOW_SIZE, SPEAKING_SCORE, MIN_SPEECH_FRAME, MAX_SPEECH_FRAME,
                                  MIN_SILENCE_FRAME, MERGE_SILENCE_FRAME, EXTEND_SPEECH_FRAME, 0.01, 0.025, True)


def valid_frame_count(num_samples: int, in_sr: int = IN_SAMPLE_RATE) -> int:
    """FireRedVAD/Inference_FireRed_ONNX.py:84-89"""
    n = int(num_samples * 16000 / in_sr)
    return 0 if n < 400 else 1 + (n - 400) // 160


@dataclass
class VadResult:
    timestamps: list            # [(start_s, end_s)]
    probs: np.ndarray           # kept frame probabilities (valid_frame_count of them)
    decisions: np.ndarray       # int8 per kept frame
    lines_second: list
    lines_indices: list


def run_vad_streams(session: FireRedSession, chunks, lengths, post: PP.FramePostConfig = POST_DEFAULT, stream=None,
                    n_valid=None):
    """Batched core: `chunks` CUDA int16 [S, n_chunks, chunk_len] (already aligned/padded),
    `lengths` the original sample counts per stream.  Everything up to the segment frame pairs
    runs on the device.  Returns (probs [S, n_chunks*T] cuda, decisions, seg_count, segments, n_valid)."""
    import torch
    S, n_chunks, L = chunks.shape
    T = session.frames(L)
    probs = session.run_batch(chunks.reshape(S * n_chunks, L), stream=stream)      # [S*n_chunks, odim, T]
    if session.cfg.odim != 1:
        raise ValueError("run_vad_streams expects the VAD head (odim == 1)")
    probs = probs.reshape(S, n_chunks * T)
    if n_valid is None:   # pass a cached CUDA int32 tensor to keep the call free of host->device copies
        in_sr = getattr(session, "in_sample_rate", IN_SAMPLE_RATE)
        n_valid = torch.tensor([min(valid_frame_count(int(n), in_sr), n_chunks * T) for n in lengths], dtype=torch.int32,
                               device=chunks.device)
    dec, cnt, seg = PP.postprocess_frames(probs, post, n_valid, stream=stream)
    return probs, dec, cnt, seg, n_valid


class HostBatchPipeline:
    """Host-buffer front door for serving: pinned int16 batches in, segment frame pairs back in pinned
    host memory.  The H2D copy of batch i+1 runs on a copy stream while batch i computes (`depth` device
    input buffers, event hand-over), so a steady stream of batches costs max(copy, compute) per batch
    instead of their sum; results (seg_count, segments) are copied back asynchronously.  The copy is
    issued in `copy_chunks` pieces so that the copy engine always has the next piece queued behind the
    running one and a late `consumed` event delays only the first piece.

    gather=True (multi-GPU): after the post-processor the per-rank results are all-gathered on the
    device over NCCL (vadx.distributed.gather_segments, the path's only collective) and rank 0's pinned
    buffers receive the GLOBAL result: seg_count [world*S], segments [world*S, max, 2]; the other ranks read
    nothing back (run returns None there)."""

    def __init__(self, session: FireRedSession, n_streams: int, n_chunks: int, post: PP.FramePostConfig = POST_DEFAULT,
                 device=None, depth: int = 2, copy_chunks: int = 4, gather: bool = False, gather_sizes=None):
        import torch
        import torch.distributed as dist
        self.session, self.post = session, post
        self.S, self.n_chunks, self.L = n_streams, n_chunks, session.chunk_len
        dev = device or torch.device("cuda", torch.cuda.current_device())
        self.T = session.frames(self.L)
        self.max_seg = (n_chunks * self.T) // 2 + 1
        self.depth = max(2, int(depth))
        self.copy_chunks = max(1, min(int(copy_chunks), n_streams))
        self.gather = bool(gather) and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        self.world = dist.get_world_size() if self.gather else 1
        self.gather_sizes = list(gather_sizes) if (self.gather and gather_sizes is not None) else None   # unequal blocks per rank
        self.reads_back = (not self.gather) or dist.get_rank() == 0
        self.d_in = [torch.empty((n_streams, n_chunks, self.L), dtype=torch.int16, device=dev) for _ in range(self.depth)]
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.copied = [torch.cuda.Event() for _ in range(self.depth)]
        self.consumed = [torch.cuda.Event() for _ in range(self.depth)]
        S_out = sum(self.gather_sizes) if self.gather_sizes else n_streams * self.world
        self.h_cnt = [torch.empty((S_out,), dtype=torch.int32).pin_memory() for _ in range(2)]
        self.h_seg = [torch.empty((S_out, self.max_seg, 2), dtype=torch.int32).pin_memory() for _ in range(2)]
        in_sr = getattr(session, "in_sample_rate", IN_SAMPLE_RATE)
        self.n_valid = torch.full((n_streams,), min(valid_frame_count(n_chunks * self.L, in_sr), n_chunks * self.T),
                                  dtype=torch.int32, device=dev)
        self._i = 0            # batches run
        self._queued = 0       # batches whose H2D copy has been enqueued

    @property
    def h2d_bytes(self) -> int:
        return self.S * self.n_chunks * self.L * 2

    @property
    def d2h_bytes(self) -> int:
        return (self.h_cnt[0].numel() * 4 + self.h_seg[0].numel() * 4) if self.reads_back else 0

    def prefetch(self, pinned):
        """enqueue the H2D copy of the NEXT not-yet-queued batch (returns immediately); up to depth - 1 batches
        may be queued ahead of the one being computed"""
        import torch
        if self._queued - self._i >= self.depth:
            raise RuntimeError("HostBatchPipeline.prefetch: every device input buffer already holds a queued batch")
        b = self._queued % self.depth
        src = pinned.view(self.S, self.n_chunks, self.L)
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self.consumed[b])
            step = (self.S + self.copy_chunks - 1) // self.copy_chunks
            for lo in range(0, self.S, step):
                self.d_in[b][lo:lo + step].copy_(src[lo:lo + step], non_blocking=True)
            self.copied[b].record(self.copy_stream)
        self._queued += 1

    def run(self, pinned, next_pinned=None):
        """process one batch; if `next_pinned` is given its copy overlaps this batch's compute.
        Returns the pinned (seg_count, segments) buffers this batch's results are being copied into
        (valid after the current stream is synchronised)."""
        import torch
        if self._queued == self._i:
            self.prefetch(pinned)
        b = self._i % self.depth
        main = torch.cuda.current_stream()
        main.wait_event(self.copied[b])
        self._i += 1
        if next_pinned is not None and self._queued - self._i < self.depth - 1:
            self.prefetch(next_pinned)
        _, _, cnt, seg, _ = run_vad_streams(self.session, self.d_in[b], None, self.post, n_valid=self.n_valid)
        self.consumed[b].record(main)
        if self.gather:
            from . import distributed as D
            cnt, seg = D.gather_segments(cnt, seg, sizes=self.gather_sizes)
            if not self.reads_back:
                return None
        r = (self._i - 1) % 2
        self.h_cnt[r].copy_(cnt, non_blocking=True)
        self.h_seg[r].copy_(seg, non_blocking=True)
        return self.h_cnt[r], self.h_seg[r]


def run_vad(audio, session: FireRedSession, post: PP.FramePostConfig = POST_DEFAULT, rng=None,
            save_timestamps_second: str | None = None, save_timestamps_indices: str | None = None) -> VadResult:
    """One stream, the reference's behaviour: `audio` is a path to a wav file or an int16 array at the session's
    IN_SAMPLE_RATE (FireRedSession(in_sample_rate=...), default 16000): loading, valid_frame_count, the open-tail clamp
    and the sample indices all use that rate, as the reference's module constant does (:84-89, :538, :590, :606)."""
    import torch
    in_sr = getattr(session, "in_sample_rate", IN_SAMPLE_RATE)
    if isinstance(audio, str):
        audio = audio_io.load_wav_int16(audio, in_sr)
    chunk_len = session.chunk_len or min(in_sr * 3600, len(audio))
    chunks, audio_len = audio_io.align_non_overlapping(audio, chunk_len, rng)
    d = torch.from_numpy(chunks).cuda().unsqueeze(0)
    probs, dec, cnt, seg, n_valid = run_vad_streams(session, d, [audio_len], post)
    n = int(n_valid[0].item())
    k = len(PP.take_segments(cnt, seg, 0))
    pairs = seg[0, :k].cpu().numpy()
    ts = PP.segments_to_seconds(pairs, n, post, audio_len / in_sr)
    sec, idx = PP.timestamp_lines(ts, in_sr)
    if save_timestamps_second and save_timestamps_indices:
        PP.write_timestamp_files(ts, save_timestamps_second, save_timestamps_indices, in_sr)
    return VadResult(ts, probs[0, :n].cpu().numpy(), dec[0, :n].cpu().numpy(), sec, idx)


@dataclass
class AedResult:
    event2timestamps: dict      # event -> [(start_s, end_s)]
    event2ratio: dict           # event -> fraction of frames at or above the event threshold, round(, 3)
    probs: np.ndarray           # [3, valid frames]


def run_aed_streams(session: FireRedSession, chunks, lengths, thresholds=None, stream=None):
    """Batched AED core: chunks CUDA int16 [S, n_chunks, L] -> probs [S, odim, n_chunks*T] and, per event,
    (decisions, seg_count, segments) from the device post-processor with that event's threshold."""
    import torch
    S, n_chunks, L = chunks.shape
    T = session.frames(L)
    odim = session.cfg.odim
    thresholds = thresholds or [SPEAKING_SCORE, SINGING_THRESHOLD, MUSIC_THRESHOLD][:odim]
    p = session.run_batch(chunks.reshape(S * n_chunks, L), stream=stream)               # [S*n_chunks, odim, T]
    probs = p.view(S, n_chunks, odim, T).permute(0, 2, 1, 3).reshape(S, odim, n_chunks * T)
    in_sr = getattr(session, "in_sample_rate", IN_SAMPLE_RATE)
    n_valid = torch.tensor([min(valid_frame_count(int(n), in_sr), n_chunks * T) for n in lengths], dtype=torch.int32,
                           device=chunks.device)
    per_event = []
    for e in range(odim):
        post = PP.FramePostConfig(SMOOTH_WINDOW_SIZE, thresholds[e], MIN_EVENT_FRAME, MAX_EVENT_FRAME, MIN_SILENCE_FRAME,
                                  MERGE_SILENCE_FRAME, EXTEND_SPEECH_FRAME, 0.01, 0.025, True)
        per_event.append((post,) + tuple(PP.postprocess_frames(probs[:, e, :], post, n_valid, stream=stream)))
    return probs, per_event, n_valid


def run_aed(audio, session: FireRedSession, rng=None) -> AedResult:
    """One stream, the reference's RUN_AED section (:620-738)."""
    import torch
    in_sr = getattr(session, "in_sample_rate", IN_SAMPLE_RATE)
    if isinstance(audio, str):
        audio = audio_io.load_wav_int16(audio, in_sr)
    chunk_len = session.chunk_len or min(in_sr * 3600, len(audio))
    chunks, audio_len = audio_io.align_non_overlapping(audio, chunk_len, rng)
    d = torch.from_numpy(chunks).cuda().unsqueeze(0)
    probs, per_event, n_valid = run_aed_streams(session, d, [audio_len])
    n = int(n_valid[0].item())
    host = probs[0, :, :n].cpu().numpy()
    ts, ratio = {}, {}
    for e, (post, _dec, cnt, seg) in enumerate(per_event):
        name = IDX2EVENT.get(e, str(e))
        pairs = PP.take_segments(cnt, seg, 0)
        ts[name] = PP.segments_to_seconds(pairs, n, post, audio_len / in_sr)
        ratio[name] = round(float(np.mean(host[e] >= post.prob_threshold)) if n > 0 else 0.0, 3)
    return AedResult(ts, ratio, host)


@dataclass
class StreamVadResult:
    timestamps: list            # [(start_s, end_s)]
    probs: np.ndarray           # frame probabilities (valid_frame_count of them at most)
    caches: object              # final caches (CUDA tensor [R, 1, P, Lb])


def stream_frame_plan(lengths, chunk_samples: int = STREAM_CHUNK_SAMPLES):
    """Frames each stream contributes per call when S streams advance in lock-step (int32 [n_calls, S]).
    Per stream this is what the reference loop produces (:786-811): full chunks give 1 + (c-400)//160
    frames, the last partial chunk its own count (one frame if it had to be zero-padded to 400 samples),
    and the concatenation is cut at valid_frame_count(len)."""
    n = np.asarray([int(v) for v in lengths], np.int64)
    n_calls = int(max(1, ((n + chunk_samples - 1) // chunk_samples).max())) if n.size else 0
    k = np.arange(n_calls, dtype=np.int64)[:, None]
    l = np.clip(n[None, :] - k * chunk_samples, 0, chunk_samples)                       # samples of call k, per stream
    f = np.where(l == 0, 0, np.where(l < WINDOW_LENGTH, 1, 1 + (l - WINDOW_LENGTH) // HOP_LENGTH))
    valid = np.where(n < WINDOW_LENGTH, 0, 1 + (n - WINDOW_LENGTH) // HOP_LENGTH)       # valid_frame_count per stream
    before = np.cumsum(f, axis=0) - f
    return np.clip(np.minimum(f, valid[None, :] - before), 0, None).astype(np.int32)


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


class _LockStep:
    """Static buffers of run_stream_vad_streams(graph=True) for one (streams, chunk) shape."""

    def __init__(self, session, S, chunk_samples, device, post):
        import torch
        self.session, self.post = session, post
        T = session.frames(chunk_samples)
        self.chunk = torch.empty((S, chunk_samples), dtype=torch.int16, device=device)
        self.out = torch.empty((S, 1, T), dtype=torch.float32, device=device)
        self.n_frames = torch.zeros((S,), dtype=torch.int32, device=device)
        self.caches = [session.new_caches(S, device), session.new_caches(S, device)]
        self.runner = _StreamGraphRunner(self._body)

    def _body(self, i: int):
        self.session.run_batch(self.chunk, self.caches[i], out=self.out, caches_out=self.caches[1 - i])
        self.post.feed(self.out[:, 0, :], self.n_frames)

    def step(self, k: int):
        """caches[k & 1] -> caches[1 - (k & 1)]"""
        self.runner.step(k)


def run_stream_vad_streams(session: FireRedStreamSession, audio, lengths, chunk_samples: int = STREAM_CHUNK_SAMPLES,
                           post: PP.StreamVadPostprocessor | None = None, caches=None, stream=None, graph: bool = False):
    """S streams in lock-step: audio CUDA int16 [S, n_calls*chunk_samples] (zero-padded), `lengths` the true
    sample counts.  Per call: model forward with cache hand-over, then the streaming segmenter, all on the
    device.  Returns (probs [S, n_calls*T] cuda, post, caches, plan).
    graph=True replays each step as one CUDA graph (runner cached on the session; its post-processor and caches
    are reset per call and returned -- read them before the next graph-mode call)."""
    import torch
    if graph:
        S, n = audio.shape
        plan = stream_frame_plan(lengths, chunk_samples)
        n_calls = plan.shape[0]
        if n != n_calls * chunk_samples:
            raise ValueError(f"run_stream_vad_streams: audio must be zero-padded to {n_calls * chunk_samples} samples, got {n}")
        runners = session.__dict__.setdefault("_graph_runners", {})
        key = (S, chunk_samples, str(audio.device))
        r = runners.get(key)
        if r is None:
            p = PP.StreamVadPostprocessor(SMOOTH_WINDOW_SIZE, STREAM_VAD_THRESHOLD, PAD_START_FRAME, MIN_SPEECH_FRAME_STREAM,
                                          MAX_SPEECH_FRAME_STREAM, MIN_SILENCE_FRAME_STREAM, n_streams=S, device=audio.device)
            r = runners[key] = _LockStep(session, S, chunk_samples, audio.device, p)
        r.post.reset()
        r.caches[0].zero_()
        T = session.frames(chunk_samples)
        d_plan = torch.from_numpy(plan).to(audio.device)
        probs = torch.empty((S, n_calls, T), dtype=torch.float32, device=audio.device)
        for k in range(n_calls):
            r.chunk.copy_(audio[:, k * chunk_samples:(k + 1) * chunk_samples])
            r.n_frames.copy_(d_plan[k])
            r.step(k)
            probs[:, k, :].copy_(r.out[:, 0, :])
        return probs.reshape(S, n_calls * T), r.post, r.caches[n_calls & 1], plan
    S, n = audio.shape
    plan = stream_frame_plan(lengths, chunk_samples)
    n_calls = plan.shape[0]
    if n != n_calls * chunk_samples:
        raise ValueError(f"run_stream_vad_streams: audio must be zero-padded to {n_calls * chunk_samples} samples, got {n}")
    T = session.frames(chunk_samples)
    post = post or PP.StreamVadPostprocessor(SMOOTH_WINDOW_SIZE, STREAM_VAD_THRESHOLD, PAD_START_FRAME,
                                             MIN_SPEECH_FRAME_STREAM, MAX_SPEECH_FRAME_STREAM,
                                             MIN_SILENCE_FRAME_STREAM, n_streams=S, device=audio.device)
    d_plan = torch.from_numpy(plan).to(audio.device)
    a = caches if caches is not None else session.new_caches(S, audio.device)
    b = torch.empty_like(a)
    probs = torch.empty((S, n_calls, T), dtype=torch.float32, device=audio.device)
    chunk = torch.empty((S, chunk_samples), dtype=torch.int16, device=audio.device)
    out = torch.empty((S, 1, T), dtype=torch.float32, device=audio.device)
    for k in range(n_calls):
        chunk.copy_(audio[:, k * chunk_samples:(k + 1) * chunk_samples])
        session.run_batch(chunk, a, out=out, caches_out=b, stream=stream)
        post.feed(out[:, 0, :], d_plan[k], stream=stream)
        probs[:, k, :].copy_(out[:, 0, :])
        a, b = b, a
    return probs.reshape(S, n_calls * T), post, a, plan


class StreamServer:
    """Live Stream-VAD serving: n_slots independent stream slots advance one tick per chunk of chunk_samples.  A stream
    may start in any free slot on any tick.  Per tick and slot the caller gives the chunk (int16 [chunk_samples]), the
    number of valid samples n and a `last` flag:

        n > 0, last 0   feed a full chunk (n == chunk_samples)
        n > 0, last 1   feed the stream's last chunk (may be short), then finalize and free the slot
        n = 0, last 0   hold: the slot's caches and segmenter state are unchanged (idle slots, streams without audio)
        n = 0, last 1   finalize and free the slot without new audio

    Frames follow the reference loop (stream_frame_plan).  Samples past n never influence a result.  Each tick is one
    model forward over all slots plus three small kernels (tail zeroing, segmenter, event compaction and cache
    lifecycle), replayed as one CUDA graph per cache parity; it costs n_slots, not the number of live streams.  The
    tick's result is a compact list of (slot, kind, frame) events: kind 0 = segment start, 1 = segment end
    (min-silence or max-speech), 2 = end because the stream ended; frame counts from the stream's first frame.
    Pairing a stream's starts and ends gives run_stream_vad(...).timestamps.

    Inputs go through the static buffers `chunk`, `n_samples`, `last`: step() copies the arguments it is given into them
    (non-blocking from pinned host memory), or a producer writes them and calls step() with no arguments."""

    def __init__(self, session: FireRedStreamSession, n_slots: int, chunk_samples: int = STREAM_CHUNK_SAMPLES,
                 smooth_window_size: int = SMOOTH_WINDOW_SIZE, speech_threshold: float = STREAM_VAD_THRESHOLD,
                 pad_start_frame: int = PAD_START_FRAME, min_speech_frame: int = MIN_SPEECH_FRAME_STREAM,
                 max_speech_frame: int = MAX_SPEECH_FRAME_STREAM, min_silence_frame: int = MIN_SILENCE_FRAME_STREAM,
                 frames_per_second: int = 100, device=None, graph: bool = True):
        import torch
        if not isinstance(session, FireRedStreamSession):
            raise ValueError("StreamServer needs a FireRedStreamSession (a streaming FireRed model)")
        if getattr(session, "in_sample_rate", IN_SAMPLE_RATE) != IN_SAMPLE_RATE:
            raise ValueError(f"StreamServer: the session must take {IN_SAMPLE_RATE} Hz audio")
        if not 1 <= int(n_slots) <= FireRedSession.MAX_STREAMS_PER_CALL:
            raise ValueError(f"StreamServer: n_slots must be in [1, {FireRedSession.MAX_STREAMS_PER_CALL}], got {n_slots}")
        if int(chunk_samples) < WINDOW_LENGTH:
            raise ValueError(f"StreamServer: chunk_samples must be at least one frame ({WINDOW_LENGTH}), got {chunk_samples}")
        dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.session, self.S, self.chunk_samples, self.device = session, int(n_slots), int(chunk_samples), dev
        self.T = session.frames(self.chunk_samples)
        self.chunk = torch.zeros((self.S, self.chunk_samples), dtype=torch.int16, device=dev)
        self.n_samples = torch.zeros((self.S,), dtype=torch.int32, device=dev)
        self.last = torch.zeros((self.S,), dtype=torch.uint8, device=dev)
        self.out = torch.zeros((self.S, 1, self.T), dtype=torch.float32, device=dev)
        self.caches = [session.new_caches(self.S, dev), session.new_caches(self.S, dev)]
        with torch.cuda.device(dev):
            self.seg = PP.StreamSlotSegmenter(smooth_window_size, speech_threshold, pad_start_frame, min_speech_frame,
                                              max_speech_frame, min_silence_frame, self.S, self.T, self.chunk_samples,
                                              WINDOW_LENGTH, HOP_LENGTH, dev, frames_per_second)
        self._runner = _StreamGraphRunner(self._tick) if graph else None
        self._k = 0

    def _tick(self, i: int):
        """the tick body on the static buffers, caches[i] -> caches[1 - i]; only libvadx launches"""
        from . import lib
        lib.check(lib.load().vadx_stream_serve_zero_tail(self.chunk.data_ptr(), self.chunk_samples,
                                                         self.n_samples.data_ptr(), self.S, self.chunk_samples,
                                                         WINDOW_LENGTH, lib.stream_ptr()))
        self.session.run_batch(self.chunk, self.caches[i], out=self.out, caches_out=self.caches[1 - i])
        self.seg.enqueue(self.out[:, 0, :], self.n_samples, self.last, i, self.caches[i], self.caches[1 - i])

    def step(self, chunk=None, n_samples=None, last=None) -> PP.ServeTick:
        """Enqueue one tick on the current stream (asynchronous).  chunk int16 [n_slots, chunk_samples], n_samples int32
        [n_slots], last bool / uint8 [n_slots]: CUDA tensors, or host tensors (pinned for a non-blocking copy); None
        for all three runs the tick on what the static buffers hold.  Returns the tick's handle (PP.ServeTick)."""
        import torch
        with torch.cuda.device(self.device):
            PP.load_tick_inputs("StreamServer.step", chunk, n_samples, last, self.chunk, self.n_samples, self.last,
                                self.device)
            if self._runner is not None:
                self._runner.step(self._k)
            else:
                self._tick(self._k & 1)
            self._k += 1
            return self.seg.finish((self._k - 1) & 1, self.out[:, 0, :])


def run_stream_vad(audio, session: FireRedStreamSession, chunk_samples: int = STREAM_CHUNK_SAMPLES) -> StreamVadResult:
    """One stream, the reference's RUN_STREAM_VAD section (:745-839): full chunks in lock-step with
    themselves, the last partial chunk at its own length (zero-padded to one frame if shorter), so the
    final caches equal the reference's too."""
    import torch
    if isinstance(audio, str):
        audio = audio_io.load_wav_int16(audio, IN_SAMPLE_RATE)
    a16 = np.ascontiguousarray(np.asarray(audio, np.int16).reshape(-1))
    n = len(a16)
    dev = torch.device("cuda", torch.cuda.current_device())
    d = torch.from_numpy(a16).to(dev)
    post = PP.StreamVadPostprocessor(SMOOTH_WINDOW_SIZE, STREAM_VAD_THRESHOLD, PAD_START_FRAME, MIN_SPEECH_FRAME_STREAM,
                                     MAX_SPEECH_FRAME_STREAM, MIN_SILENCE_FRAME_STREAM, n_streams=1, device=dev)
    caches = session.new_caches(1, dev)
    left = valid_frame_count(n)
    kept = []
    for pos in range(0, n, chunk_samples):
        chunk = d[pos:pos + chunk_samples]
        if chunk.numel() < WINDOW_LENGTH:
            chunk = torch.nn.functional.pad(chunk, (0, WINDOW_LENGTH - chunk.numel()))
        p, caches = session.run_batch(chunk.reshape(1, -1).contiguous(), caches)
        p = p[:, 0, :min(p.shape[2], left)]
        left -= p.shape[1]
        if p.shape[1]:
            post.feed(p.contiguous())
            kept.append(p[0])
    probs = torch.cat(kept).cpu().numpy() if kept else np.zeros((0,), np.float32)
    return StreamVadResult(post.timestamps()[0], probs, caches)


def main(argv=None):
    import argparse
    ap = argparse.ArgumentParser(description="FireRedVAD on B200 (random-init weights unless --weights is given)")
    ap.add_argument("audio")
    ap.add_argument("--weights", help=".npz with the DetectModel state_dict")
    ap.add_argument("--out-second", default="./timestamps_second.txt")
    ap.add_argument("--out-indices", default="./timestamps_indices.txt")
    a = ap.parse_args(argv)
    cfg = W.FireRedConfig()
    w = dict(np.load(a.weights)) if a.weights else W.firered_random_init(cfg, 0)
    sess = FireRedSession(w, cfg, chunk_len=INPUT_AUDIO_LENGTH)
    r = run_vad(a.audio, sess, save_timestamps_second=a.out_second, save_timestamps_indices=a.out_indices)
    print("\nTimestamps in Second:")
    print("".join(r.lines_second), end="")
    print("\nTimestamps in Indices:")
    print("".join(r.lines_indices), end="")


if __name__ == "__main__":
    main()
