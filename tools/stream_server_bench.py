"""Slot server throughput on one GPU: FireRed Stream-VAD (firered_vad.StreamServer, the default) or, with
--family silero / fsmn / marblenet, that family's StreamServer.

For each slot count, at full occupancy and under churn (about 1 % of slots closing and joining per tick, 10 % held):
  device ms per tick      CUDA events around the tick's graph replay (inputs already in the static buffers)
  host ms per tick        wall clock of step(pinned inputs) + host_events(): pinned H2D, tick, event read-back
  events, D2H bytes       per tick, from the host loop
  realtime streams        n_slots * 160 ms / device ms per tick
  lockstep ms per chunk   run_stream_vad_streams(graph=True) at the same S, alternating with the server in this process
With --family silero, for each slot count and windows per tick (--windows, default 5 and 1) the same rows are
measured, except: realtime streams = n_slots * W * 32 ms / device ms per tick, and instead of the lock-step chunk the
bare forward of the same shape (SileroSession's engine over [n_slots][64 + W*512] rows, W windows, one CUDA graph),
alternating with the server in this process.
With --family fsmn (fsmn_vad.StreamServer), for each slot count and window length (--chunk-lens, default 16000 and
7520, look-backward 0.3 s), the same rows with ticks of one reference window (stride = L - 31 * 160 samples), plus the
bare forward of the same [n_slots][L] shape as one CUDA graph and the lock-step run_streams(graph=True) time per window,
both alternating with the server in this process; realtime streams = n_slots * stride / 16000 / tick.
With --family marblenet (marblenet_vad.StreamServer), for each slot count and window (--window-samples, default 16000
and 32000), the same rows with ticks of one static-axis window and traffic drawn from synth-enveloped chunks, plus the
bare forward (MarbleNetSession.run_batch over the same [n_slots][L] into a static output, one CUDA graph), alternating
with the server in this process; realtime streams = n_slots * L / 16000 / tick.
Prints one JSON line (card name and power limit read in the same run); --out also writes it to a file, --trace writes
the torch.profiler launch list of a few server ticks.

  python tools/stream_server_bench.py --slots 4096,16384 --ticks 100 --out profiles/r03_stream_server.json \
      --trace profiles/r03_launches_stream_server.txt
  python tools/stream_server_bench.py --family silero --slots 4096,16384 --out profiles/r04_silero_server.json \
      --trace profiles/r04_launches_silero_server.txt
  python tools/stream_server_bench.py --family fsmn --slots 4096,16384 --out profiles/r05_fsmn_server.json \
      --trace profiles/r05_launches_fsmn_server.txt
  python tools/stream_server_bench.py --family marblenet --slots 4096,16384 --window-samples 16000,32000 \
      --out profiles/r06_marblenet_server.json --trace profiles/r06_launches_marblenet_server.txt
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (v.strip() for v in q.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:       # the numbers still stand, but without the card they are not comparable
        return {"error": str(e)}


class Traffic:
    """Seeded control words per tick: every slot feeds full chunks; under churn about `churn` of the slots close per
    tick (a short last chunk, or n_samples = 0) and rejoin on the next one, and `hold` of the live ones hold."""

    def __init__(self, S, C, churn, hold, seed, n_pool=4):
        import torch
        rs = np.random.RandomState(seed)
        self.S, self.C = S, C
        audio = rs.randint(-3000, 3000, size=(S, C)).astype(np.int16)
        t = np.arange(C)[None, :]
        audio += (8000 * np.sin(t / rs.uniform(3, 30, size=(S, 1))) * (rs.rand(S, 1) < 0.5)).astype(np.int16)
        self.chunks = [torch.from_numpy(np.roll(audio, 97 * i, axis=0)).pin_memory() for i in range(n_pool)]
        self.ctrl = []
        for _ in range(64):
            n = np.full(S, C, np.int32)
            last = np.zeros(S, np.uint8)
            if churn > 0:
                close = rs.rand(S) < churn
                short = rs.randint(0, C, size=S)
                n[close] = short[close]
                last[close] = 1
                held = (rs.rand(S) < hold) & ~close
                n[held] = 0
            self.ctrl.append((torch.from_numpy(n).pin_memory(), torch.from_numpy(last).pin_memory()))

    def tick(self, k):
        n, last = self.ctrl[k % len(self.ctrl)]
        return self.chunks[k % len(self.chunks)], n, last


def bench_server(server, traffic, ticks, warmup):
    import torch
    for k in range(warmup):
        server.step(*traffic.tick(k)).host_events()
    torch.cuda.synchronize()
    # device time of the tick: inputs copied first, events around the replay only
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(ticks)]
    for k in range(ticks):
        c, n, last = traffic.tick(k)
        server.chunk.copy_(c, non_blocking=True)
        server.n_samples.copy_(n, non_blocking=True)
        server.last.copy_(last, non_blocking=True)
        ev[k][0].record()
        server.step()
        ev[k][1].record()
    torch.cuda.synchronize()
    dev_ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
    # host-inclusive: pinned H2D, tick, read-back of the events
    n_ev, d2h = 0, 0
    t0 = time.perf_counter()
    for k in range(ticks):
        t = server.step(*traffic.tick(k))
        n_ev += len(t.host_events())
        d2h += t.d2h_bytes
    host_ms = (time.perf_counter() - t0) * 1e3 / ticks
    return dev_ms, host_ms, n_ev / ticks, d2h / ticks


def bench_lockstep(session, audio, lengths, reps):
    import torch
    from vadx import firered_vad as FV
    n_calls = audio.shape[1] // FV.STREAM_CHUNK_SAMPLES
    FV.run_stream_vad_streams(session, audio, lengths, graph=True)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        FV.run_stream_vad_streams(session, audio, lengths, graph=True)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / (reps * n_calls)


class SileroForward:
    """the bare forward of a Silero server tick: the session's engine over [S][64 + W*512] rows and W windows, state
    a -> b, captured as one CUDA graph on buffers of its own"""

    def __init__(self, session, S, W):
        import torch
        c = session.cfg
        self.session, self.S, self.W = session, S, W
        self.stride = c.context + W * c.window
        g = torch.Generator(device="cuda").manual_seed(S + W)
        self.x = (torch.rand((S, self.stride), generator=g, device="cuda") - 0.5) * 0.5
        self.out = torch.empty((W, S, 1), dtype=torch.float32, device="cuda")
        self.state = [torch.zeros((2, S, c.hidden), dtype=torch.float32, device="cuda") for _ in range(2)]
        self._run()
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self._run()

    def _run(self):
        self.session.forward_windows(self.x, self.out, self.state[0], self.state[1], self.W, self.stride)

    def time(self, reps):
        import torch
        for _ in range(5):
            self.graph.replay()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            self.graph.replay()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps


def write_trace(path, server, traffic, title):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for k in range(5):
            server.step(*traffic.tick(k)).host_events()
        torch.cuda.synchronize()
    with open(path, "w") as f:
        f.write(f"# {title}\n")
        f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=40))
        names = [e.key for e in prof.key_averages()]
        f.write("\nat:: kernels: %s\n" % ([n for n in names if "at::" in n] or "none"))


def main_silero(a, info):
    import torch
    import vadx
    from vadx import silero_vad as SV, weights as W
    cfg = W.SileroConfig()
    sess = vadx.SileroSession(W.silero_random_init(cfg, 0), cfg)
    rows = []
    for S in [int(v) for v in a.slots.split(",")]:
        for Wt in [int(v) for v in a.windows.split(",")]:
            C = Wt * cfg.window
            fwd = SileroForward(sess, S, Wt)
            for mode, churn, hold in (("full", 0.0, 0.0), ("churn", 0.01, 0.10)):
                traffic = Traffic(S, C, churn, hold, seed=S + Wt + len(mode))
                server = SV.StreamServer(sess, S, windows_per_tick=Wt)
                res = {"dev": [], "host": [], "events": [], "d2h": [], "fwd": []}
                for _ in range(a.rounds):
                    d, h, e, b = bench_server(server, traffic, a.ticks, a.warmup)
                    res["dev"].append(d), res["host"].append(h), res["events"].append(e), res["d2h"].append(b)
                    res["fwd"].append(fwd.time(a.ticks))
                dev = float(np.median(res["dev"]))
                bare = float(np.median(res["fwd"]))
                row = {"n_slots": S, "windows_per_tick": Wt, "traffic": mode, "device_ms_per_tick": round(dev, 4),
                       "device_ms_per_tick_rounds": [round(v, 4) for v in res["dev"]],
                       "host_ms_per_tick": round(float(np.median(res["host"])), 4),
                       "events_per_tick": round(float(np.mean(res["events"])), 2),
                       "d2h_bytes_per_tick": round(float(np.mean(res["d2h"])), 1),
                       "realtime_streams": int(S * Wt * 32.0 / dev),
                       "forward_ms": round(bare, 4), "forward_ms_rounds": [round(v, 4) for v in res["fwd"]],
                       "tick_over_forward": round(dev / bare, 3)}
                rows.append(row)
                print(json.dumps(row), file=sys.stderr)
                if a.trace and len(rows) == 1:
                    write_trace(a.trace, server, traffic, f"silero StreamServer, {S} slots, W = {Wt}, 5 ticks, {info}")
                del server
            del fwd
            torch.cuda.empty_cache()
    return {"what": "silero StreamServer tick vs the bare forward of the same shape", "card": info,
            "ticks": a.ticks, "rounds": a.rounds, "results": rows}


class FsmnTraffic:
    """Seeded control words for the FSMN server, simulated tick by tick because a full chunk depends on the samples a
    slot holds (server.full_chunk): every slot feeds full chunks; under churn about `churn` of the slots close per tick
    (a short last chunk, possibly empty) and a new stream starts there on the next one, and `hold` of the others hold.
    tick() ignores its argument and hands out the next tick, so the control words stay consistent with the device."""

    def __init__(self, S, L, stride, churn, hold, seed, n_ticks, n_pool=2):
        import torch
        rs = np.random.RandomState(seed)
        audio = rs.randint(-3000, 3000, size=(S, stride)).astype(np.int16)
        t = np.arange(stride)[None, :]
        audio += (8000 * np.sin(t / rs.uniform(3, 30, size=(S, 1))) * (rs.rand(S, 1) < 0.5)).astype(np.int16)
        self.chunks = [torch.from_numpy(np.roll(audio, 97 * i, axis=0)).pin_memory() for i in range(n_pool)]
        self.ctrl = []
        rec = np.zeros(S, np.int64)
        for _ in range(n_ticks):
            full = np.where(rec < L, np.minimum(stride, L - rec), stride)
            n = full.astype(np.int32)
            last = np.zeros(S, np.uint8)
            if churn > 0:
                close = rs.rand(S) < churn
                n[close] = (rs.rand(S) * (full + 1)).astype(np.int32)[close]
                last[close] = 1
                n[(rs.rand(S) < hold) & ~close] = 0
            rec += n
            rec[last != 0] = 0
            self.ctrl.append((torch.from_numpy(n).pin_memory(), torch.from_numpy(last).pin_memory()))
        self.k = 0

    def tick(self, _k):
        n, last = self.ctrl[self.k]
        self.k += 1
        return self.chunks[self.k % len(self.chunks)], n, last


class FsmnForward:
    """the bare forward of an FSMN server tick: FsmnSession.run_batch over [S][L] rows into static outputs, caches
    a -> b, captured as one CUDA graph on buffers of its own"""

    def __init__(self, session, S):
        import torch
        L, T = session.chunk_len, session.T
        self.session = session
        g = torch.Generator(device="cuda").manual_seed(S + L)
        self.x = torch.randint(-8000, 8000, (S, L), generator=g, device="cuda", dtype=torch.int16)
        self.noise = torch.full((S,), 4.0, device="cuda")
        self.score = torch.empty((S, T), dtype=torch.uint8, device="cuda")
        self.noisy = torch.empty((S,), dtype=torch.float32, device="cuda")
        self.caches = [torch.zeros((session.cfg.fsmn_layers, S) + session.cache_shape, device="cuda") for _ in range(2)]
        self._run()
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self._run()

    def _run(self):
        self.session.run_batch(self.x, self.caches[0].unbind(0), self.noise, out=(self.score, self.noisy, None, None),
                               caches_out=self.caches[1].unbind(0))

    time = SileroForward.time


def bench_fsmn_lockstep(session, aligned, stride, lb_s, reps):
    """run_streams(graph=True) over recordings of a few windows: ms per window"""
    import torch
    from vadx import fsmn_vad as FSV
    n_windows = (aligned.shape[1] - session.chunk_len) // stride + 1
    FSV.run_streams(session, aligned, stride, lb_s, graph=True)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        FSV.run_streams(session, aligned, stride, lb_s, graph=True)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / (reps * n_windows)


def main_fsmn(a, info):
    import torch
    import vadx
    from vadx import fsmn_vad as FSV, weights as W
    cfg = W.FsmnConfig()
    wts = W.fsmn_random_init(cfg, 0)
    lb_s = FSV.LOOK_BACKWARD
    rows = []
    for L in [int(v) for v in a.chunk_lens.split(",")]:
        sess = vadx.FsmnSession(wts, cfg, chunk_len=L)
        stride = L - (FSV.look_backward_frames(lb_s) + 1) * FSV.OUTPUT_FRAME_LENGTH
        for S in [int(v) for v in a.slots.split(",")]:
            fwd = FsmnForward(sess, S)
            lock = torch.from_numpy(np.random.RandomState(S).randint(-8000, 8000, size=(S, L + 3 * stride))
                                    .astype(np.int16)).cuda()
            for mode, churn, hold in (("full", 0.0, 0.0), ("churn", 0.01, 0.10)):
                n_ticks = a.rounds * (a.warmup + 2 * a.ticks) + (5 if a.trace and not rows else 0)
                traffic = FsmnTraffic(S, L, stride, churn, hold, S + L + len(mode), n_ticks)
                server = FSV.StreamServer(sess, S, look_backward_s=lb_s)
                res = {"dev": [], "host": [], "events": [], "d2h": [], "fwd": [], "lock": []}
                for _ in range(a.rounds):
                    d, h, e, b = bench_server(server, traffic, a.ticks, a.warmup)
                    res["dev"].append(d), res["host"].append(h), res["events"].append(e), res["d2h"].append(b)
                    res["fwd"].append(fwd.time(a.ticks))
                    res["lock"].append(bench_fsmn_lockstep(sess, lock, stride, lb_s, 2))
                dev = float(np.median(res["dev"]))
                bare = float(np.median(res["fwd"]))
                row = {"chunk_len": L, "stride": stride, "n_slots": S, "traffic": mode, "device_ms_per_tick": round(dev, 4),
                       "device_ms_per_tick_rounds": [round(v, 4) for v in res["dev"]],
                       "host_ms_per_tick": round(float(np.median(res["host"])), 4),
                       "events_per_tick": round(float(np.mean(res["events"])), 2),
                       "d2h_bytes_per_tick": round(float(np.mean(res["d2h"])), 1),
                       "realtime_streams": int(S * stride / 16000 / (dev / 1e3)),
                       "forward_ms": round(bare, 4), "forward_ms_rounds": [round(v, 4) for v in res["fwd"]],
                       "tick_over_forward": round(dev / bare, 3),
                       "lockstep_ms_per_window": round(float(np.median(res["lock"])), 4)}
                rows.append(row)
                print(json.dumps(row), file=sys.stderr)
                if a.trace and len(rows) == 1:
                    write_trace(a.trace, server, traffic, f"fsmn StreamServer, L = {L}, {S} slots, 5 ticks, {info}")
                del server, traffic
                torch.cuda.empty_cache()
            del fwd, lock
            torch.cuda.empty_cache()
    return {"what": "fsmn StreamServer tick vs the bare forward of the same shape and the lock-step window", "card": info,
            "look_backward_s": lb_s, "ticks": a.ticks, "rounds": a.rounds, "results": rows}


class MarbleNetTraffic(Traffic):
    """Traffic whose chunks are drawn from a pool of synth-enveloped windows (speech-like bursts and pauses), so that
    segments keep opening and closing after warm-up"""

    def __init__(self, S, C, churn, hold, seed, n_pool=2):
        import torch
        from vadx import synth
        super().__init__(S, C, churn, hold, seed, n_pool=0)
        self.chunks = [torch.from_numpy(synth.synth_streams(S, C, seed=seed + i)).pin_memory() for i in range(n_pool)]


class MarbleNetForward:
    """the bare forward of a MarbleNet server tick: MarbleNetSession.run_batch over [S][L] rows into a static output,
    captured as one CUDA graph on buffers of its own"""

    def __init__(self, session, S, L):
        import torch
        g = torch.Generator(device="cuda").manual_seed(S + L)
        self.session = session
        self.x = torch.randint(-8000, 8000, (S, L), generator=g, device="cuda", dtype=torch.int16)
        self.out = torch.empty((2, S, session.frames(L)), dtype=torch.float32, device="cuda")
        self._run()
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self._run()

    def _run(self):
        self.session.run_batch(self.x, out=self.out)

    time = SileroForward.time


def main_marblenet(a, info):
    import torch
    import vadx
    from vadx import marblenet_vad as MV, weights as W
    cfg = W.MarbleNetConfig()
    sess = vadx.MarbleNetSession(W.marblenet_random_init(cfg, 0), cfg)
    rows = []
    for L in [int(v) for v in a.window_samples.split(",")]:
        for S in [int(v) for v in a.slots.split(",")]:
            fwd = MarbleNetForward(sess, S, L)
            for mode, churn, hold in (("full", 0.0, 0.0), ("churn", 0.01, 0.10)):
                traffic = MarbleNetTraffic(S, L, churn, hold, seed=S + L + len(mode))
                server = MV.StreamServer(sess, S, window_samples=L)
                res = {"dev": [], "host": [], "events": [], "d2h": [], "fwd": []}
                for _ in range(a.rounds):
                    d, h, e, b = bench_server(server, traffic, a.ticks, a.warmup)
                    res["dev"].append(d), res["host"].append(h), res["events"].append(e), res["d2h"].append(b)
                    res["fwd"].append(fwd.time(a.ticks))
                dev = float(np.median(res["dev"]))
                bare = float(np.median(res["fwd"]))
                row = {"window_samples": L, "frames_per_tick": server.F, "n_slots": S, "traffic": mode,
                       "device_ms_per_tick": round(dev, 4), "device_ms_per_tick_rounds": [round(v, 4) for v in res["dev"]],
                       "host_ms_per_tick": round(float(np.median(res["host"])), 4),
                       "events_per_tick": round(float(np.mean(res["events"])), 2),
                       "d2h_bytes_per_tick": round(float(np.mean(res["d2h"])), 1),
                       "realtime_streams": int(S * L / 16000 / (dev / 1e3)),
                       "forward_ms": round(bare, 4), "forward_ms_rounds": [round(v, 4) for v in res["fwd"]],
                       "tick_over_forward": round(dev / bare, 3)}
                rows.append(row)
                print(json.dumps(row), file=sys.stderr)
                if a.trace and len(rows) == 1:
                    write_trace(a.trace, server, traffic, f"marblenet StreamServer, L = {L}, {S} slots, 5 ticks, {info}")
                del server, traffic
                torch.cuda.empty_cache()
            del fwd
            torch.cuda.empty_cache()
    return {"what": "marblenet StreamServer tick vs the bare forward of the same shape", "card": info,
            "ticks": a.ticks, "rounds": a.rounds, "results": rows}


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--family", choices=("firered", "silero", "fsmn", "marblenet"), default="firered")
    ap.add_argument("--chunk-lens", default="16000,7520", help="fsmn: window lengths to measure")
    ap.add_argument("--windows", default="5,1", help="silero: windows per tick to measure")
    ap.add_argument("--window-samples", default="16000,32000", help="marblenet: samples per tick (window) to measure")
    ap.add_argument("--slots", default="4096,16384")
    ap.add_argument("--ticks", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3, help="server / lock-step alternations per configuration")
    ap.add_argument("--out", default=None)
    ap.add_argument("--trace", default=None, help="write the torch.profiler launch list of 5 ticks at the first S here")
    a = ap.parse_args(argv)
    import torch
    import vadx
    from vadx import firered_vad as FV, weights as W
    if not torch.cuda.is_available():
        raise SystemExit("stream_server_bench: needs a CUDA device")
    torch.cuda.set_device(0)
    info = card()
    if a.family in ("silero", "fsmn", "marblenet"):
        out = {"silero": main_silero, "fsmn": main_fsmn, "marblenet": main_marblenet}[a.family](a, info)
        line = json.dumps(out)
        print(line)
        if a.out:
            with open(a.out, "w") as f:
                f.write(line + "\n")
        return
    cfg = W.FireRedConfig(N2=0, S2=0, streaming=True)
    sess = vadx.FireRedStreamSession(W.firered_random_init(cfg, 5), cfg)
    C = FV.STREAM_CHUNK_SAMPLES
    rows = []
    for S in [int(v) for v in a.slots.split(",")]:
        lock_calls = 10
        lock_audio = torch.from_numpy(np.random.RandomState(S).randint(-8000, 8000, size=(S, lock_calls * C))
                                      .astype(np.int16)).cuda()
        lengths = [lock_calls * C] * S
        for mode, churn, hold in (("full", 0.0, 0.0), ("churn", 0.01, 0.10)):
            traffic = Traffic(S, C, churn, hold, seed=S + len(mode))
            server = FV.StreamServer(sess, S)
            res = {"dev": [], "host": [], "events": [], "d2h": [], "lock": []}
            for _ in range(a.rounds):
                d, h, e, b = bench_server(server, traffic, a.ticks, a.warmup)
                res["dev"].append(d), res["host"].append(h), res["events"].append(e), res["d2h"].append(b)
                res["lock"].append(bench_lockstep(sess, lock_audio, lengths, 3))
            dev = float(np.median(res["dev"]))
            lock = float(np.median(res["lock"]))
            row = {"n_slots": S, "traffic": mode, "device_ms_per_tick": round(dev, 4),
                   "device_ms_per_tick_rounds": [round(v, 4) for v in res["dev"]],
                   "host_ms_per_tick": round(float(np.median(res["host"])), 4),
                   "events_per_tick": round(float(np.mean(res["events"])), 2),
                   "d2h_bytes_per_tick": round(float(np.mean(res["d2h"])), 1),
                   "realtime_streams": int(S * 160.0 / dev),
                   "lockstep_ms_per_chunk": round(lock, 4),
                   "lockstep_ms_per_chunk_rounds": [round(v, 4) for v in res["lock"]],
                   "tick_over_lockstep": round(dev / lock, 3)}
            rows.append(row)
            print(json.dumps(row), file=sys.stderr)
            if a.trace and len(rows) == 1:
                write_trace(a.trace, server, traffic, f"StreamServer, {S} slots, 5 ticks, {info}")
            del server
            torch.cuda.empty_cache()
    out = {"what": "firered StreamServer tick vs run_stream_vad_streams(graph=True) chunk", "card": info,
           "chunk_samples": C, "ticks": a.ticks, "rounds": a.rounds, "results": rows}
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
