#!/usr/bin/env python
"""bench.py -- RTFx (audio-hours/sec) of the B200 VAD hot path, one JSON line on rank 0.

Workload (BASELINE.json configs[3], the config the 1/2/4/8-GPU metric is quoted on):
FireRedVAD DFSMN, synthetic 16 kHz int16 audio in 16000-sample chunks, 16 chunks per stream.
A "step" is one pass of the hot path (frontend -> DFSMN -> on-device post-processing to
segment frame pairs) over one batch of chunks per GPU.  Streams shard across ranks with no
data-path collective (weak scaling).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--chunks B] [--impl vadx|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

`value`  : device-resident inputs, CUDA-event timed, max over ranks.
`e2e`    : same metric through the public API with pinned HOST buffers, H2D + D2H inside the
           timed region.
`roofline`: dominant stage, timed live with CUDA events on the launching stream (per-stage
           timers inside libvadx), against MEASURED_PEAKS.json.
`cpu_baseline` / `--impl reference`: the oracle port of the reference graph (torch-CPU fp32,
           batch-1 calls like the reference's ORT loop) on the box's host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CHUNK = 16000
CHUNKS_PER_STREAM = 16
METRIC = "RTFx (audio-hours/sec)"
UNIT = "audio-hours/sec"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--chunks", type=int, default=8192, help="16000-sample chunks per GPU per step")
    ap.add_argument("--impl", default="vadx", choices=["vadx", "reference"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-families", action="store_true", help="skip the short RTFx runs of the other model families")
    ap.add_argument("--sustain-seconds", type=float, default=4.0,
                    help="extra device-resident leg of about this many seconds (steady-state clocks / power); 0 = skip")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed device-resident step returned (rank 0's streams) as DIR/<name>.npy, "
                         "float32; inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "vadx":
        ap.error("--dump-outputs applies to --impl vadx")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, probs, dec, cnt, seg, n_valid):
    """One step's results of run_vad_streams as float32 .npy files (every value is exact in float32).  Segment slots
    past a stream's count and decisions past its valid frames were never written by the device and are set to -1 and 0,
    so the files depend only on what was computed.  Above DUMP_LIMIT_BYTES a fixed seeded sample of streams is written,
    the same rows of every array, with their indices in stream_index.npy."""
    import numpy as np
    probs, dec, cnt, seg, n_valid = (t.cpu().numpy().copy() for t in (probs, dec, cnt, seg, n_valid))
    seg[np.arange(seg.shape[1])[None, :] >= np.minimum(cnt, seg.shape[1])[:, None]] = -1
    dec[np.arange(dec.shape[1])[None, :] >= n_valid[:, None]] = 0
    out = {"frame_probs": probs, "decisions": dec, "seg_count": cnt, "segments": seg}
    S = cnt.shape[0]
    per_stream = 4 * (sum(a[0].size for a in out.values()) + 1)
    if S * per_stream > DUMP_LIMIT_BYTES:
        idx = np.sort(np.random.RandomState(0).choice(S, DUMP_LIMIT_BYTES // per_stream, replace=False))
        out = {k: a[idx] for k, a in out.items()}
        out["stream_index"] = idx
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), a.astype(np.float32))


def ncu_traffic_bytes(kernel_substr):
    """DRAM bytes per launch of the named kernel from the committed ncu capture (None when absent)."""
    import re
    p = os.path.join(ROOT, "profiles", "r02_top_kernels_firered.txt")
    if not os.path.exists(p):
        p = os.path.join(ROOT, "profiles", "r01_top_kernels.txt")
    if not os.path.exists(p):
        return None
    vals = []
    for line in open(p):
        if kernel_substr in line.split(";")[0]:
            rd = re.search(r"dram__bytes_read\.sum=([0-9.]+) (\w+)", line)
            wr = re.search(r"dram__bytes_write\.sum=([0-9.]+) (\w+)", line)
            if rd and wr:
                mul = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
                vals.append(float(rd.group(1)) * mul[rd.group(2)] + float(wr.group(1)) * mul[wr.group(2)])
    return sum(vals) / len(vals) if vals else None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons DURING the timed region, through NVML (the same counters
    `nvidia-smi --query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.*` prints, B200_PROFILING.md),
    sampled every 5 ms so that even a 100 ms timed region gets a median."""
    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt, self.max_mhz = index, [], threading.Event(), None
        self.active = threading.Event()

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception:
            return
        while not self._stop_evt.is_set():
            if self.active.is_set():
                try:
                    self.rows.append((float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)),
                                      int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))))
                except Exception:
                    pass
            self._stop_evt.wait(0.005)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=3)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        sm = sorted(r[0] for r in self.rows)
        bits = 0
        for r in self.rows:
            bits |= r[1]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_mhz,
                "reasons": sorted(k for k, v in self.REASONS.items() if bits & v), "samples": len(sm)}


# --------------------------------------------------------------------------------- CPU legs
def cpu_reference_leg(seconds_budget: float, steps: int | None = None, warmup: int = 1):
    """The oracle port of the reference graph on the host cores, batch-1 calls like the reference's
    per-chunk ORT loop (FireRedVAD/Inference_FireRed_ONNX.py:567-572) + its Python post-processing."""
    import numpy as np
    import torch
    import vadx  # noqa: F401  (weights / synth only; no CUDA involved here)
    from vadx import synth, weights as W
    from oracle.firered import FireRedOracle
    from oracle import postproc as OP

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = W.FireRedConfig()
    orc = FireRedOracle(W.firered_random_init(cfg, 0), cfg)
    pool = synth.synth_chunks_fast(256, CHUNK, seed=1234)

    STREAMS_PER_CALL = 4   # 64 chunks per forward call: measured here to be the CPU's best batch size

    def one_call(i0):
        idx = [(i0 * 64 + j) % 256 for j in range(STREAMS_PER_CALL * CHUNKS_PER_STREAM)]
        p = orc.forward(pool[idx]).numpy()[:, 0, :].reshape(STREAMS_PER_CALL, -1)
        out = []
        for s in range(STREAMS_PER_CALL):
            dec = OP.frame_decisions(p[s], 5, 0.4, 20, 2000, 20, 5, 0)
            out.append(OP.segments_from_decisions(dec, 0.01, 0.025, CHUNKS_PER_STREAM * 1.0, True))
        return out

    calls_per_step = 4     # one CPU "step" = 16 streams = 256 chunks = 256 s of audio
    for w in range(max(1, warmup)):
        one_call(w)
    # the reference's literal loop shape (batch-1 ORT calls) for the record
    t0 = time.perf_counter()
    for j in range(16):
        orc.forward(pool[j][None])
    batch1 = 16.0 / (time.perf_counter() - t0) / 3600.0
    per_step = []
    t_end = time.perf_counter() + seconds_budget
    done = 0
    while True:
        t0 = time.perf_counter()
        for c in range(calls_per_step):
            one_call(done * calls_per_step + c)
        per_step.append(time.perf_counter() - t0)
        done += 1
        if steps is not None and done >= steps:
            break
        if steps is None and time.perf_counter() >= t_end:
            break
    n_streams = done * calls_per_step * STREAMS_PER_CALL
    audio_s = n_streams * CHUNKS_PER_STREAM * (CHUNK / 16000.0)
    total = sum(per_step)
    value = audio_s / total / 3600.0
    return {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{n_streams} streams x {CHUNKS_PER_STREAM} chunks of {CHUNK} samples in 64-chunk calls "
                      f"(batch-1 calls like the reference's loop: {batch1:.4f} {UNIT}), torch-CPU fp32 oracle port "
                      f"on {cores} threads + Python post-processing, {total:.1f} s",
            "batch1_value": batch1, "ms_per_step": 1e3 * total / done, "steps": done}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_leg(args.cpu_seconds, steps=args.steps, warmup=args.warmup)
    line = {"metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": r["steps"],
            "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": "FireRedVAD DFSMN, synthetic 16 kHz, 16000-sample chunks (BASELINE configs[3])",
                       "chunks_per_stream": CHUNKS_PER_STREAM, "step": "16 streams (256 chunks) in 64-chunk calls"},
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------- other families
def ncu_family_traffic(family, kernel):
    """DRAM bytes per launch of `kernel` from the committed per-family ncu capture (profiles/r02_top_kernels_<family>.txt)."""
    import re
    p = os.path.join(ROOT, "profiles", f"r02_top_kernels_{family}.txt")
    if not os.path.exists(p):
        return None
    vals = []
    base = kernel.split("(")[0].split("+")[0]
    for line in open(p):
        if base in line.split(";")[0]:
            rd = re.search(r"dram__bytes_read\.sum=([0-9.]+) (\w+)", line)
            wr = re.search(r"dram__bytes_write\.sum=([0-9.]+) (\w+)", line)
            if rd and wr:
                mul = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
                vals.append(float(rd.group(1)) * mul[rd.group(2)] + float(wr.group(1)) * mul[wr.group(2)])
    return sum(vals) / len(vals) if vals else None


def kernel_roofline(family, kernels, pk):
    """roofline block of one family from the library's per-kernel records (lib.profile_collect_kernels): every entry point
    reports its kernel's name and the ALGORITHMIC bytes / flops of each call (include/vadx.h, vadx_kernel_stat), timed by
    CUDA-event pairs on the launching stream.  The dominant kernel (largest share of the step) is the headline; the rest
    is listed by share."""
    kernels = {k: v for k, v in kernels.items() if v["calls"] and v["ms"] > 0}
    if not kernels:
        return None
    total = sum(v["ms"] for v in kernels.values())
    dom = max(kernels, key=lambda k: kernels[k]["ms"])
    d = kernels[dom]
    gbs = d["bytes"] / (d["ms"] * 1e-3) / 1e9
    tf = d["flops"] / (d["ms"] * 1e-3) / 1e12
    # tcgen05 kernels run the fp32 contraction as 3 (dense layers) or 4 (DFT) bf16/fp16 products
    products = 4 if "stft_power_tc" in dom else (3 if "_tc_" in dom or "fc2_memory" in dom else 0)
    frac_hbm = gbs / pk["hbm_gbs"]
    frac_tensor = tf * products / pk["bf16_tflops_sustained"] if products else 0.0
    tensor_bound = frac_tensor > frac_hbm
    roof = {"bound": "tensor" if tensor_bound else "hbm", "kernel": dom,
            "achieved": tf * products if tensor_bound else gbs,
            "peak": pk["bf16_tflops_sustained"] if tensor_bound else pk["hbm_gbs"],
            "unit": "TFLOP/s" if tensor_bound else "GB/s", "frac": frac_tensor if tensor_bound else frac_hbm,
            "traffic": ncu_family_traffic(family, dom), "launches_timed": d["calls"], "avg_launch_ms": d["ms"] / d["calls"],
            "algorithmic_bytes_per_launch": d["bytes"] / d["calls"], "algorithmic_flops_per_launch": d["flops"] / d["calls"],
            "share_of_step": d["ms"] / total, "hbm_gbs": gbs, "fp32_equiv_tflops": tf,
            "peak_source": pk["source"] + " (MEASURED_PEAKS.json: hbm_gbs copy; bf16_tflops_sustained for tensor-bound kernels)"}
    if roof["traffic"] is not None:
        roof["traffic_source"] = f"profiles/r02_top_kernels_{family}.txt (ncu --set full, dram bytes read + written per launch)"
    roof["kernels_by_share"] = [
        {"kernel": k, "share": round(v["ms"] / total, 4), "launches": v["calls"], "avg_launch_ms": round(v["ms"] / v["calls"], 5),
         "hbm_gbs": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1), "frac_hbm": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9 / pk["hbm_gbs"], 4),
         "fp32_equiv_tflops": round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 2)}
        for k, v in sorted(kernels.items(), key=lambda kv: -kv[1]["ms"])[:8]]
    return roof


def family_workloads(dev, only=None):
    """The bench workloads of the other model families (BASELINE configs 0, 1, 2, 4 and the streaming FireRed twin) at the
    SURVEY section 8(d) shapes: name -> dict(step=callable timed as one step, eager=callable with the same kernels launched
    eagerly (for the per-kernel records; None = same as step), audio_s=audio seconds per step per GPU, config=str,
    steps/warm).  Generator: each workload is built when reached and dropped before the next."""
    import numpy as np
    import torch
    import vadx
    from vadx import fsmn_vad, marblenet_vad, postprocess as PP, silero_vad, synth, weights as W

    def want(n):
        return only is None or n in only

    if only is not None and "firered" in only:
        # the headline workload (BASELINE configs[3]) as a family step, for tools/family_step.py (ncu captures)
        from vadx import firered_vad
        cfg = W.FireRedConfig()
        sess = vadx.FireRedSession(W.firered_random_init(cfg, 0), cfg, chunk_len=CHUNK)
        B = 8192
        S = B // CHUNKS_PER_STREAM
        d_audio = torch.from_numpy(synth.synth_chunks_fast(B, CHUNK, seed=1234)).to(dev)
        lengths = [CHUNKS_PER_STREAM * CHUNK] * S
        n_valid = torch.full((S,), min(firered_vad.valid_frame_count(lengths[0]), CHUNKS_PER_STREAM * sess.frames(CHUNK)),
                             dtype=torch.int32, device=dev)
        yield "firered", dict(step=lambda: firered_vad.run_vad_streams(sess, d_audio.view(S, CHUNKS_PER_STREAM, CHUNK), lengths,
                                                                       firered_vad.POST_DEFAULT, n_valid=n_valid),
                              eager=None, audio_s=B * 1.0, steps=10, warm=3, config=f"{B} chunks of {CHUNK} samples")
        del sess, d_audio
    if want("fsmn"):
        # FSMN (config 0 shape, batched): S streams x 4 overlapping 16000-sample windows, state carried on device
        cfg = W.FsmnConfig()
        sess = vadx.FsmnSession(W.fsmn_random_init(cfg, 0), cfg, chunk_len=16000)
        S, stride = 1024, 16000 - 31 * 160
        n = 16000 + 3 * stride
        a = torch.from_numpy(synth.synth_chunks_fast(S, n, seed=11)).to(dev)
        yield "fsmn", dict(step=lambda: fsmn_vad.run_streams(sess, a, stride, whole=True), eager=None, audio_s=S * n / 16000, steps=3,
                           warm=3, config=f"{S} streams/GPU x 4 windows of 16000 samples (stride {stride}), all windows in one forward "
                                          "(whole-file mode), caches + gate + hysteresis on device")
        del sess, a
    if want("marblenet"):
        # MarbleNet (config 2): 60 s clips, the survey's 256 clips per GPU
        cfg = W.MarbleNetConfig()
        sess = vadx.MarbleNetSession(W.marblenet_random_init(cfg, 0), cfg)
        B = 256
        clips = torch.from_numpy(synth.synth_chunks_fast(B, 960000, seed=12)).to(dev)
        yield "marblenet", dict(step=lambda: marblenet_vad.run_vad_clips(sess, clips), eager=None, audio_s=B * 60.0, steps=3, warm=3,
                                config=f"{B} clips/GPU x 60 s, post-processing on device")
        del sess, clips
    if want("silero"):
        # Silero (config 1): 4096 streams, 32 ms windows with LSTM state carry
        cfg = W.SileroConfig()
        sess = vadx.SileroSession(W.silero_random_init(cfg, 0), cfg)
        S, n_win = 4096, 32
        audio = (torch.from_numpy(synth.synth_chunks_fast(S, n_win * 512, seed=13)).to(dev).float() * 0.000030517578)
        lens = [n_win * 512] * S

        def silero_step():
            probs = sess.speech_probs(audio)
            return silero_vad.raw_segments(probs, lens, 0.5, 16000, 250, 20, 250)

        yield "silero", dict(step=silero_step, eager=None, audio_s=S * n_win * 0.032, steps=3, warm=3,
                             config=f"{S} streams/GPU x {n_win} windows of 512 samples, LSTM state + trigger machine on device")
        del sess, audio
    if want("dfsmn_aec"):
        # DFSMN AEC-VAD (config 4): near + far end, 31841-sample chunks; the survey's 1024 pairs per GPU when the workspace
        # (about 80 MB per pair) leaves room, else the largest power of two that does
        from vadx import dfsmn_aec  # noqa: F401
        cfg = W.DfsmnAecConfig()
        sess = vadx.DfsmnAecSession(W.dfsmn_aec_random_init(cfg, 0), cfg, chunk_len=31841)
        free_b, _total = torch.cuda.mem_get_info(dev)
        S = int(os.environ.get("VADX_BENCH_DFSMN_PAIRS", "1024"))     # (the ncu captures run a smaller batch)
        while S > 32 and sess._e.workspace_bytes(S, 31841) > 0.7 * free_b:
            S //= 2
        ws_gb = sess._e.workspace_bytes(S, 31841) / 1e9
        far = torch.from_numpy(synth.synth_chunks_fast(S, 31841, seed=14)).to(dev)
        near = torch.from_numpy(synth.synth_chunks_fast(S, 31841, seed=15)).to(dev)
        state = PP.HysteresisState(S, 100, dev)
        probs = torch.empty((S, sess.T), dtype=torch.float32, device=dev)

        def aec_step():
            sess.run_batch(near, far, out=probs)
            state.n_saved.zero_()
            PP.lookahead_hysteresis(probs, state, 15, 0.5, 0.5, is_final=True)

        yield "dfsmn_aec", dict(step=aec_step, eager=None, audio_s=S * 31841 / 16000, steps=2, warm=2,
                                config=f"{S} near+far stream pairs/GPU x one 31841-sample chunk ({ws_gb:.1f} GB workspace), one "
                                       "vadx_forward of the native dfsmn_aec model (echo estimator on fp32 FFMA kernels, mask-net "
                                       "on tcgen05), hysteresis on device")
        del sess, near, far
    if want("firered_stream"):
        # FireRed Stream-VAD: 4096 streams in lock-step, 160 ms chunks (14 frames) with cache carry + streaming segmenter
        from vadx import firered_vad
        cfg = W.FireRedConfig(N2=0, S2=0, streaming=True)
        sess = vadx.FireRedStreamSession(W.firered_random_init(cfg, 5), cfg)
        S, n_calls = 4096, 25
        a = torch.from_numpy(synth.synth_chunks_fast(S, n_calls * 2560, seed=16)).to(dev)
        lens = [n_calls * 2560] * S
        yield "firered_stream", dict(step=lambda: firered_vad.run_stream_vad_streams(sess, a, lens, graph=True),
                                     eager=lambda: firered_vad.run_stream_vad_streams(sess, a, lens, graph=False),
                                     audio_s=S * n_calls * 0.16, steps=2, warm=2, per_chunk=n_calls,
                                     config=f"{S} streams/GPU x {n_calls} chunks of 2560 samples, caches + streaming segmenter on device, "
                                            "one CUDA-graph replay per chunk")
        del sess, a


def family_rtfx(dev, world, dist):
    """Short device-resident RTFx runs of the other model families (BASELINE configs 0-2, 4), same timing rules (warm-ups,
    CUDA events, max over ranks), each with its own roofline block from the library's per-kernel records.  Reported next
    to the headline, not as it."""
    import numpy as np
    import torch
    import vadx
    from vadx import fsmn_vad, lib, weights as W

    pk = peaks()

    def timed(fn, steps=3, warm=3):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / steps], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    out = {}
    for name, w in family_workloads(dev):
        ms = timed(w["step"], w["steps"], w["warm"])
        r = {"audio_hours_per_sec": world * w["audio_s"] / (ms / 1e3) / 3600, "ms_per_step": ms, "config": w["config"]}
        if "per_chunk" in w:
            r["ms_per_160ms_chunk"] = ms / w["per_chunk"]
        # per-kernel records: a separate, untimed pass with the library's event pairs around every entry point
        lib.profile_enable(True)
        lib.profile_collect_kernels()
        (w["eager"] or w["step"])()
        torch.cuda.synchronize()
        kernels = lib.profile_collect_kernels()
        lib.profile_enable(False)
        lib.profile_collect()
        r["roofline"] = kernel_roofline(name, kernels, pk)
        out[name] = r
        torch.cuda.empty_cache()
    for v in out.values():
        v["rtfx"] = v["audio_hours_per_sec"] * 3600
    # BASELINE configs[0] as the reference runs it: ONE stream, 512-sample chunks, batch 1 (latency-bound; the
    # reference publishes RTF 0.0047 for it on an i3-12300).  Wall clock around the whole entry point.
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "tests", "golden", "vad_sample_16k.npz")
    if os.path.exists(gold):
        import time
        audio = np.load(gold)["audio"].astype(np.int16)
        cfg = W.FsmnConfig()
        sess = vadx.FsmnSession(W.fsmn_random_init(cfg, 0), cfg, chunk_len=512)
        for mode in ("", "_graph", "_whole"):
            kw = {"graph": mode == "_graph", "whole": mode == "_whole"}
            for _ in range(3):
                fsmn_vad.run_vad(audio, sess, 0.0, rng=np.random.RandomState(1), **kw)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(5):
                fsmn_vad.run_vad(audio, sess, 0.0, rng=np.random.RandomState(1), **kw)
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / 5
            out["fsmn_c1_single_stream" + mode] = {
                "rtf": dt / (len(audio) / 16000.0), "rtfx": (len(audio) / 16000.0) / dt, "seconds": dt,
                "config": "vad_sample.wav (5.59 s), one stream, 512-sample chunks, 254 windows, wall clock of run_vad (host "
                          "normalisation, alignment and H2D included)"
                          + {"": ", eager launches per window", "_graph": ", one CUDA-graph replay per window",
                             "_whole": ", ALL windows in one forward + one sequential gate kernel (fsmn_vad.run_vad(whole=True))"}[mode]}
    return out


# --------------------------------------------------------------------------------- GPU arm
def run_vadx(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import vadx
    from vadx import distributed as D, firered_vad, lib, postprocess as PP, synth, weights as W

    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # before any pinned allocation: keep this rank's host buffers on the NUMA node of its GPU (first touch)
    numa = D.bind_to_local_numa_node(local_rank) if not os.environ.get("VADX_BENCH_NO_NUMA_BIND") else {"bound": False, "node_cpus": 0}
    rank, world, dev = D.init("nccl")

    L = lib.load()
    cfg = W.FireRedConfig()
    sess = vadx.FireRedSession(W.firered_random_init(cfg, 0), cfg, chunk_len=CHUNK)
    B = (args.chunks // CHUNKS_PER_STREAM) * CHUNKS_PER_STREAM
    S = B // CHUNKS_PER_STREAM
    T = sess.frames(CHUNK)
    # streams shard across ranks in contiguous blocks (vadx.distributed.shard_streams); the synthetic generator is seeded by
    # the block so that every rank synthesises only its own streams
    my_streams = D.shard_streams(world * S, rank, world)
    assert len(my_streams) == S
    host = synth.synth_chunks_fast(B, CHUNK, seed=1234 + rank)
    pinned = torch.from_numpy(host).pin_memory()
    d_audio = pinned.to(dev)                                   # device-resident copy for `value`
    lengths = [CHUNKS_PER_STREAM * CHUNK] * S
    post = firered_vad.POST_DEFAULT
    stream = torch.cuda.current_stream()

    n_valid = torch.full((S,), min(firered_vad.valid_frame_count(lengths[0]), CHUNKS_PER_STREAM * T),
                         dtype=torch.int32, device=dev)

    def step_device():
        return firered_vad.run_vad_streams(sess, d_audio.view(S, CHUNKS_PER_STREAM, CHUNK), lengths, post,
                                           n_valid=n_valid)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    last = {}

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler.active.set()
        e0.record(stream)
        for i in range(steps):
            if i < steps - 1:
                fn()
            else:
                last["out"] = fn()      # kept from the last step only: no two steps' outputs are alive at once
        e1.record(stream)
        barrier()
        sampler.active.clear()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    W_ = max(3, args.warmup)
    if rank == 0:
        sampler.start()
    # ---- device-resident, with live per-stage timers
    lib.profile_enable(True)
    for _ in range(W_):
        step_device()
    torch.cuda.synchronize()
    lib.profile_collect()                                     # drop warm-up records
    lib.profile_collect_kernels()
    launches0 = L.vadx_launch_count()
    ms_total = timed(step_device, args.steps, 0)
    launches = L.vadx_launch_count() - launches0
    stages = lib.profile_collect()
    kernel_records = lib.profile_collect_kernels()
    lib.profile_enable(False)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last["out"])
    last.clear()
    # ---- the same step back to back for a few seconds: the timed region above is ~0.1 s, this leg shows the step time and
    # the clocks once the part sits at its power / thermal steady state (reported next to `value`, not as it)
    sustained = None
    if args.sustain_seconds > 0:
        n_sus = max(args.steps, int(args.sustain_seconds * 1e3 / max(ms_total / args.steps, 1e-3)))
        sus_sampler = ClockSampler(local_rank)
        if rank == 0:
            sus_sampler.start()
        keep = sampler
        sampler = sus_sampler
        ms_sus = timed(step_device, n_sus, 0)
        sampler = keep
        if rank == 0:
            sus_sampler.stop()
        sustained = {"steps": n_sus, "seconds": ms_sus / 1e3, "ms_per_step": ms_sus / n_sus,
                     "value": world * B * (CHUNK / 16000.0) * n_sus / (ms_sus / 1e3) / 3600.0, "unit": UNIT,
                     "clocks": sus_sampler.summary() if rank == 0 else None}
    # ---- end to end through the public API with host buffers
    # multi-GPU: the final gather of seg_count / segments (the path's only collective) is INSIDE the end-to-end region.
    # The host-fed arm is bound by each GPU's pinned host->device rate, which is NOT the same for all GPUs of the box (PCIe
    # switch sharing: 23 vs 35 GB/s with eight ranks copying, profiles/r02_h2d_ceiling.json), so the SAME total number of
    # streams is split in proportion to the rate each rank measures at start-up, capped by the rate its compute consumes
    # (vadx.distributed.weighted_blocks); the device-resident `value` keeps equal blocks.
    e2e_sizes, h2d_rates = None, None
    S_e2e = S
    if world > 1 and not os.environ.get("VADX_BENCH_EQUAL_E2E_BLOCKS"):
        h2d_rates = D.measure_h2d_rates(dev)
        # what this GPU's compute consumes, from the device-resident timing just taken (3 % headroom for the copy traffic)
        compute_gbs = 0.97 * (B * CHUNK * 2) / (ms_total / args.steps * 1e-3) / 1e9
        e2e_sizes = D.weighted_blocks(world * S, [min(r, compute_gbs) for r in h2d_rates])
        S_e2e = e2e_sizes[rank]
    pipe = firered_vad.HostBatchPipeline(sess, S_e2e, CHUNKS_PER_STREAM, post, dev, gather=world > 1, gather_sizes=e2e_sizes)
    if S_e2e == S:
        host_e2e = host
    else:
        host_e2e = synth.synth_chunks_fast(S_e2e * CHUNKS_PER_STREAM, CHUNK, seed=4321 + rank)
        pinned = torch.from_numpy(host_e2e).pin_memory()
    pinned2 = torch.from_numpy(np.roll(host_e2e, 1, axis=0).copy()).pin_memory()   # batches alternate between two host buffers
    host_batches = [pinned, pinned2]
    e2e_state = {"i": 0, "last": None}

    def step_e2e():
        i = e2e_state["i"]
        e2e_state["i"] = i + 1
        e2e_state["last"] = pipe.run(host_batches[i % 2], host_batches[(i + 1) % 2])

    ms_e2e = timed(step_e2e, args.steps, W_)
    if rank == 0:
        sampler.stop()
    # concurrent pinned-H2D ceiling of this box at this rank count (tools/h2d_microbench.py inlined): the end-to-end arm moves
    # h2d_bytes per rank per step through it, so max(compute, copy at the ceiling) is its floor
    barrier()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(pipe.copy_stream):
        c0.record(pipe.copy_stream)
        for i in range(8):
            pipe.d_in[i % 2].copy_(host_batches[i % 2].view(S_e2e, CHUNKS_PER_STREAM, CHUNK), non_blocking=True)
        c1.record(pipe.copy_stream)
    barrier()
    my_gbs = 8.0 * pipe.h2d_bytes / (c0.elapsed_time(c1) * 1e-3) / 1e9
    h2d_gbs = torch.tensor([my_gbs], device=dev, dtype=torch.float64)
    copy_floor = torch.tensor([1e3 * pipe.h2d_bytes / (my_gbs * 1e9)], device=dev, dtype=torch.float64)   # ms for this rank's block
    h2d_sum = h2d_gbs.clone()
    if world > 1:
        dist.all_reduce(h2d_gbs, op=dist.ReduceOp.MIN)
        dist.all_reduce(h2d_sum, op=dist.ReduceOp.SUM)
        dist.all_reduce(copy_floor, op=dist.ReduceOp.MAX)
    h2d_gbs, h2d_sum, copy_floor = float(h2d_gbs.item()), float(h2d_sum.item()), float(copy_floor.item())
    segs_found = int(e2e_state["last"][0].sum().item()) if e2e_state["last"] is not None else 0
    h2d_bytes, d2h_bytes = pipe.h2d_bytes, pipe.d2h_bytes      # d2h: rank 0 reads the gathered global result back
    h2d_total = torch.tensor([float(h2d_bytes)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(h2d_total, op=dist.ReduceOp.SUM)
    h2d_total = int(h2d_total.item())
    families = None
    if not args.no_families:
        del pipe, d_audio
        torch.cuda.empty_cache()
        families = family_rtfx(dev, world, dist)

    audio_s_per_step = world * B * (CHUNK / 16000.0)
    value = audio_s_per_step * args.steps / (ms_total / 1e3) / 3600.0
    e2e_value = audio_s_per_step * args.steps / (ms_e2e / 1e3) / 3600.0

    if rank == 0:
        pk = peaks()
        rows = B * T
        # algorithmic work per step per GPU (DESIGN.md section 3)
        lin_layers = ([(cfg.idim, cfg.H), (cfg.H, cfg.P)] + [(cfg.P, cfg.H), (cfg.H, cfg.P)] * (cfg.R - 1)
                      + [(cfg.P, cfg.H)] + [(cfg.H, cfg.H)] * (cfg.M - 1))
        if stages.get("mel", (0, 0))[0] == 0:
            # the log-mel contraction runs as a tcgen05 dense layer (bins the filterbank reads -> n_mels) and is
            # timed with the linear stage
            lin_layers = [(cfg.n_fft // 2, cfg.n_mels)] + lin_layers
        # default engine: every block's second dense layer runs inside the fused fc2 + memory kernel (block_stages.cu, timed
        # with the memory stage); detected from the number of dense-layer launches the library timed
        fused = round(stages.get("linear", (0, 0))[1] / max(1, args.steps)) < len(lin_layers)
        mem_bytes = 4.0 * rows * cfg.P * (2 + (cfg.R - 1) * 3)                               # p (+ residual) in, out
        if fused:
            lin_layers = [kn for kn in lin_layers if kn != (cfg.H, cfg.P)]
            mem_bytes = 4.0 * rows * (cfg.R * (cfg.H + cfg.P) + (cfg.R - 1) * cfg.P)         # h stages (+ residual) in, out
        stage_bytes = {"linear": 4.0 * rows * sum(k + n for k, n in lin_layers),           # fp32 rows in + out
                       "memory": mem_bytes,
                       "stft": B * CHUNK * 2.0 + 4.0 * rows * (cfg.n_fft // 2 + 1),        # int16 audio in, power out
                       "mel": 4.0 * rows * ((cfg.n_fft // 2 + 1) + cfg.n_mels),
                       "head": 4.0 * rows * (cfg.H + cfg.odim), "postproc": 5.0 * rows, "prep": 6.0 * B * CHUNK}
        stage_flops = {"linear": 2.0 * rows * sum(k * n for k, n in lin_layers),
                       "stft": 2.0 * rows * cfg.n_fft * 2 * (cfg.n_fft // 2 + 1)}
        total_ms = max(1e-9, sum(x[0] for x in stages.values()))
        dom = max(stages, key=lambda k: stages[k][0])
        dom_ms, dom_calls = stages[dom]
        stage_share = {k: round(v[0] / total_ms, 4) for k, v in stages.items()}
        kernel_names = {"linear": "linear_tc_kernel (tcgen05, bf16 2-term split)",
                        "memory": ("fc2_memory_stages_kernel (tcgen05 transposed product, fp32x2 FIR out of TMEM, bulk-copied operand and residual rings)" if fused
                                   else "fsmn_memory_bulk_kernel (cp.async.bulk ring, fp32x2 FMA)"),
                        "stft": "stft_power_tc_kernel (tcgen05, int16 exact split)", "mel": "mel_log_kernel",
                        "head": "linear_narrow_kernel", "postproc": "postprocess_frames_runs_kernel",
                        "prep": "prep_audio_kernel"}
        # every stage of this path is limited by HBM traffic today (the tensor pipe is <25 % busy in the
        # tcgen05 kernels, see profiles/): report the dominant stage against the measured copy bandwidth,
        # and its tensor-pipe rate next to it when it is a contraction
        per_launch_bytes = stage_bytes[dom] * args.steps / max(1, dom_calls)
        ach = per_launch_bytes / (dom_ms / max(1, dom_calls) * 1e-3) / 1e9
        roof = {"bound": "hbm", "kernel": kernel_names.get(dom, dom), "achieved": ach, "peak": pk["hbm_gbs"],
                "unit": "GB/s", "frac": ach / pk["hbm_gbs"], "traffic": None,
                "peak_source": pk["source"] + " STREAM-style copy (MEASURED_PEAKS.json hbm_gbs)",
                "launches_timed": dom_calls, "avg_launch_ms": dom_ms / max(1, dom_calls),
                "algorithmic_bytes_per_launch": per_launch_bytes}
        roof["traffic"] = ncu_traffic_bytes({"linear": "linear_tc_kernel", "memory": "fc2_memory_stages_kernel" if fused else "fsmn_memory_bulk_kernel",
                                             "stft": "stft_power_tc_kernel", "mel": "mel_log_kernel"}.get(dom, dom))
        if roof["traffic"] is not None:
            roof["traffic_source"] = "profiles/r02_top_kernels_firered.txt (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum, mean over captured launches at this bench size)"
        if dom in stage_flops:
            tf = stage_flops[dom] * args.steps / (dom_ms * 1e-3) / 1e12
            roof["tensor"] = {"achieved_tflops_fp32_equiv": tf, "mma_products_per_fp32_product": 3 if dom == "linear" else 4,
                              "peak_bf16_tflops_sustained": pk["bf16_tflops_sustained"],
                              "frac_of_bf16_peak_incl_split": tf * (3 if dom == "linear" else 4) / pk["bf16_tflops_sustained"]}
        roof["all_stages"] = {k: {"ms_per_step": stages[k][0] / args.steps,
                                  "hbm_gbs": (stage_bytes[k] * args.steps / (stages[k][0] * 1e-3) / 1e9) if stages[k][0] > 0 else None,
                                  "frac": (stage_bytes[k] * args.steps / (stages[k][0] * 1e-3) / 1e9 / pk["hbm_gbs"]) if stages[k][0] > 0 else None}
                              for k in stages}
        kr = kernel_roofline("firered", kernel_records, pk)
        if kr:
            roof["kernels_by_share"] = kr["kernels_by_share"]      # the same step through the library's per-kernel records
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            r = cpu_reference_leg(args.cpu_seconds)
            cpu = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": W_,
                "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": "FireRedVAD DFSMN (R8 H256 P128 N20+20), synthetic 16 kHz int16, 16000-sample "
                                       "chunks, 16 chunks/stream (BASELINE configs[3])",
                           "chunks_per_gpu_per_step": B, "streams_per_gpu_per_step": S, "frames_per_chunk": T,
                           "audio_seconds_per_step": audio_s_per_step,
                           "l2": "inputs (%.0f MB/step/GPU) and activations exceed the 126 MB L2" % (B * CHUNK * 2 / 1e6),
                           "sharding": "streams split across ranks, no data-path collective"},
                "rtfx": value * 3600.0,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_total,
                        "d2h_bytes_per_step": int(d2h_bytes),
                        "api": "vadx.firered_vad.HostBatchPipeline.run(pinned int16 batch): H2D of batch i+1 overlaps compute of batch i"
                               + ("; per-step all_gather of seg_count/segments over NCCL (vadx.distributed.gather_segments), rank 0 reads the global result back" if world > 1 else ""),
                        "numa_bind": numa,
                        "streams_per_rank": e2e_sizes or [S] * world, "h2d_gbs_per_rank_at_startup": h2d_rates,
                        "h2d_ceiling": {"pinned_gbs_per_rank_min": h2d_gbs, "pinned_gbs_aggregate": h2d_sum,
                                        "ranks_copying_concurrently": world,
                                        "copy_floor_ms_per_step": copy_floor,      # slowest rank: its block / its measured rate
                                        "e2e_floor_ms_per_step": max(copy_floor, ms_total / args.steps),
                                        "e2e_frac_of_floor": max(copy_floor, ms_total / args.steps) / (ms_e2e / args.steps)},
                        "ms_per_step": ms_e2e / args.steps, "segments_found_last_step": segs_found},
                "gpu_launches": int(launches),
                "roofline": roof, "stage_ms_per_step": {k: v[0] / args.steps for k, v in stages.items()},
                "stage_share": stage_share,
                "sustained": sustained,
                "cpu_baseline": cpu, "clocks": sampler.summary(), "families": families}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_vadx(args)


if __name__ == "__main__":
    main()
