"""Slot server throughput on one GPU: FireRed Stream-VAD (firered_vad.StreamServer, the default) or, with
--family silero, Silero (silero_vad.StreamServer).

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
Prints one JSON line (card name and power limit read in the same run); --out also writes it to a file, --trace writes
the torch.profiler launch list of a few server ticks.

  python tools/stream_server_bench.py --slots 4096,16384 --ticks 100 --out profiles/r03_stream_server.json \
      --trace profiles/r03_launches_stream_server.txt
  python tools/stream_server_bench.py --family silero --slots 4096,16384 --out profiles/r04_silero_server.json \
      --trace profiles/r04_launches_silero_server.txt
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


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--family", choices=("firered", "silero"), default="firered")
    ap.add_argument("--windows", default="5,1", help="silero: windows per tick to measure")
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
    if a.family == "silero":
        out = main_silero(a, info)
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
