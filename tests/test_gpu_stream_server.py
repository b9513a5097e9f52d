"""FireRed Stream-VAD slot server (firered_vad.StreamServer, vadx_stream_serve_step): the segmenter against the
reference script's record at kernel level, live churn against the oracle and run_stream_vad, slot reuse, holds,
garbage past n_samples, graph replay, determinism and rejections."""
import os

import numpy as np
import pytest
import torch

import vadx
from vadx import firered_vad as FV, postprocess as PP, synth, weights as W
from oracle import postproc as OP
from oracle.firered import FireRedOracle

pytestmark = pytest.mark.gpu
TOL = 1e-3
BOUND = 3e-4     # the tensor-core stream path's asserted bound (tests/test_gpu_firered_stream.py)
C = FV.STREAM_CHUNK_SAMPLES
POST = (5, 0.4, 5, 8, 2000, 20)


@pytest.fixture(scope="module")
def gold_script(golden_dir):
    return np.load(os.path.join(golden_dir, "firered_script.npz"))


@pytest.fixture(scope="module")
def weights():
    cfg = W.FireRedConfig(N2=0, S2=0, streaming=True)
    return cfg, W.firered_random_init(cfg, 5)


@pytest.fixture(scope="module")
def stream_session(cuda, weights):
    cfg, w = weights
    return vadx.FireRedStreamSession(w, cfg)


def pair(events, inv_fps=0.01):
    """one stream's [(kind, frame)] -> [(start_s, end_s)]"""
    out, start = [], None
    for kind, frame in events:
        if kind == PP.SERVE_START:
            assert start is None, events
            start = frame
        else:
            assert start is not None, events
            out.append((int(start) * inv_fps, int(frame) * inv_fps))
            start = None
    assert start is None, events
    return out


def _pairs(ts):
    return np.array(ts, np.float64).reshape(-1, 2)


# ---------------------------------------------------------------- kernel level, given probabilities
def feed_track(p, prm, T, n_slots=3, slot=1, seed=0, seg=None):
    """one track through slot `slot` of a model-less segmenter (`seg`, or a fresh one) in T-frame ticks, finalized
    with its last tick; the other slots hold, with garbage"""
    rs = np.random.RandomState(seed)
    chunk = 400 + 160 * (T - 1)
    if seg is None:
        seg = PP.StreamSlotSegmenter(*prm, n_slots=n_slots, n_frames=T, chunk_samples=chunk, device="cuda")
    ev = []
    n_ticks = max(1, (len(p) + T - 1) // T)
    for k in range(n_ticks):
        f = min(T, len(p) - k * T)
        probs = rs.uniform(0, 1, size=(n_slots, T)).astype(np.float32)
        probs[slot, :f] = p[k * T:k * T + f]
        n = np.zeros(n_slots, np.int32)
        n[slot] = chunk if f == T else 400 + 160 * (f - 1)
        lst = np.zeros(n_slots, np.uint8)
        lst[slot] = k == n_ticks - 1
        t = seg.step(torch.from_numpy(probs).cuda(), torch.from_numpy(n).cuda(), torch.from_numpy(lst).cuda())
        assert t.frames.cpu().numpy().tolist() == [f if s == slot else 0 for s in range(n_slots)]
        got = t.host_events()
        assert all(s == slot for s, _, _ in got)
        ev += [(kind, frame) for _, kind, frame in got]
    return ev


@pytest.mark.parametrize("i", range(6))
def test_kernel_reference_record(cuda, gold_script, i):
    g = gold_script
    p = g[f"sp{i}_probs"]
    ws, thr, pad, msp, mxs, msi, split = g[f"sp{i}_params"]
    prm = (int(ws), thr, int(pad), int(msp), int(mxs), int(msi))
    for T in sorted({14, int(split) if int(split) else 14}):
        ev = feed_track(p, prm, T, seed=i)
        assert np.array_equal(_pairs(pair(ev)), g[f"sp{i}_whole"]), T
        assert pair(ev) == OP.StreamPost(*prm).feed(p)


def test_kernel_long_lived_slot(cuda):
    """> 1000 segments through one slot in one stream, nothing dropped, then a second stream in the same slot of the
    same segmenter (finalize, then reuse)"""
    rs = np.random.RandomState(11)
    T, S = 200, 4
    runs = rs.randint(25, 60, size=2 * 1100)
    gate = np.concatenate([np.full(r, i % 2 == 0) for i, r in enumerate(runs)])
    p = np.clip(np.where(gate, 0.85, 0.1) + rs.normal(0, 0.05, size=gate.shape), 0, 1).astype(np.float32)
    ref = OP.StreamPost(*POST).feed(p)
    assert len(ref) > 1000
    seg = PP.StreamSlotSegmenter(*POST, n_slots=S, n_frames=T, chunk_samples=400 + 160 * (T - 1), device="cuda")
    ev = feed_track(p, POST, T, n_slots=S, slot=2, seed=1, seg=seg)
    assert pair(ev) == ref
    ev2 = feed_track(p[:5000], POST, T, n_slots=S, slot=2, seed=2, seg=seg)
    assert pair(ev2) == OP.StreamPost(*POST).feed(p[:5000])


def test_kernel_rejection_keeps_other_slots_events(cuda):
    """a tick that rejects one slot's control words still reports every other slot's events on the exception"""
    T, S = 14, 3
    rs = np.random.RandomState(4)
    p = np.clip(np.repeat(rs.rand(40) > 0.5, 14) * 0.8 + rs.normal(0.1, 0.05, 560), 0, 1).astype(np.float32)
    runs = []
    for bad in (False, True):
        seg = PP.StreamSlotSegmenter(*POST, n_slots=S, n_frames=T, chunk_samples=C, device="cuda")
        ev, n_rejected = [], 0
        for k in range(len(p) // T):
            probs = np.zeros((S, T), np.float32)
            probs[0] = p[k * T:(k + 1) * T]
            n = np.array([C, C + 1 if bad and k % 3 == 0 else 0, 0], np.int32)
            t = seg.step(torch.from_numpy(probs).cuda(), torch.from_numpy(n).cuda(), torch.zeros(S, dtype=torch.uint8,
                                                                                               device=cuda))
            try:
                got = t.host_events()
            except PP.ServeTickError as e:
                assert e.error == PP.SERVE_ERR_RANGE
                got, n_rejected = e.events, n_rejected + 1
            ev += got
        runs.append((ev, n_rejected))
    assert runs[1][0] == runs[0][0] and len(runs[0][0]) > 4
    assert runs[0][1] == 0 and runs[1][1] == 14


# ---------------------------------------------------------------- server driver
class Stream:
    def __init__(self, sid, audio):
        self.sid, self.audio, self.pos = sid, audio, 0
        self.frames, self.probs, self.events = [], [], []
        self.done = False


def run_ticks(server, plan, garbage=None):
    """plan: list of ticks, each {slot: (stream, action)} with action 'feed', 'hold' or 'close' (n = 0, last = 1).
    Slots not named hold.  `garbage` (RandomState) fills every sample past n with noise."""
    S, Cs = server.S, server.chunk_samples
    out = []
    for tick in plan:
        chunk = np.zeros((S, Cs), np.int16)
        if garbage is not None:
            chunk = garbage.randint(-32768, 32767, size=(S, Cs)).astype(np.int16)
        n = np.zeros(S, np.int32)
        last = np.zeros(S, np.uint8)
        fed = {}
        for slot, (st, action) in tick.items():
            if action == "feed":
                m = min(Cs, len(st.audio) - st.pos)
                assert m > 0
                chunk[slot, :m] = st.audio[st.pos:st.pos + m]
                n[slot] = m
                st.pos += m
                # a stream that ends on a full chunk may instead be closed by a later tick with n_samples = 0
                last[slot] = st.pos == len(st.audio) and not (getattr(st, "close_after", False) and m == Cs)
                fed[slot] = st
            elif action == "close":
                last[slot] = 1
                fed[slot] = st
        t = server.step(torch.from_numpy(chunk).pin_memory(), torch.from_numpy(n).pin_memory(),
                        torch.from_numpy(last).pin_memory())
        ev = t.host_events()
        slots = [s for s, _, _ in ev]
        assert slots == sorted(slots)
        probs, frames = t.probs.cpu().numpy(), t.frames.cpu().numpy()
        for slot, st in fed.items():
            if n[slot] > 0:
                st.frames.append(int(frames[slot]))
            else:
                assert frames[slot] == 0
            st.probs.append(probs[slot, :frames[slot]].copy())
            if last[slot]:
                st.done = True
        for slot in range(S):
            if slot not in fed:
                assert frames[slot] == 0
        for s, kind, frame in ev:
            assert s in fed, (s, kind, frame)
            fed[s].events.append((kind, frame))
        out.append(ev)
    return out


def churn_plan(streams, S, rs, p_hold=0.1, p_join=0.3):
    """streams join free slots at random ticks, hold at random mid-stream; returns the plan"""
    queue, busy, plan = list(streams), {}, []
    while queue or busy:
        tick = {}
        for slot in range(S):
            if slot not in busy and queue and rs.rand() < p_join:
                busy[slot] = queue.pop(0)
        for slot, st in list(busy.items()):
            fed_so_far = getattr(st, "_planned", 0)
            left = len(st.audio) - fed_so_far
            if fed_so_far > 0 and left > 0 and rs.rand() < p_hold:
                tick[slot] = (st, "hold")
            elif left > 0:
                tick[slot] = (st, "feed")
                st._planned = fed_so_far + min(C, left)
                if st._planned == len(st.audio) and not getattr(st, "close_after", False):
                    del busy[slot]
            else:
                tick[slot] = (st, "close")
                del busy[slot]
        plan.append(tick)
    return plan


def make_streams(rs, n, seed):
    lengths = list(rs.randint(1, 12 * C, size=n))
    lengths[:6] = [1, 300, C * 3 + 250, C * 4, C * 2, 399]      # no frames; short last chunk; exact multiples
    raw = synth.synth_streams(n, max(lengths), seed=seed)
    streams = [Stream(i, raw[i, :lengths[i]].copy()) for i in range(n)]
    for st in streams:
        st.close_after = len(st.audio) % C == 0 and rs.rand() < 0.7    # exact multiples: close with n_samples = 0
    streams[3].close_after = True
    return streams


def oracle_probs(orc, cfg, audio):
    caches = torch.zeros(cfg.R, 1, cfg.P, 19)
    ref = []
    for pos in range(0, len(audio), C):
        ch = audio[pos:pos + C]
        if len(ch) < 400:
            ch = np.pad(ch, (0, 400 - len(ch)))
        p, caches = orc.forward(torch.from_numpy(np.ascontiguousarray(ch)).view(1, 1, -1), caches)
        ref.append(p.numpy()[0, 0])
    return np.concatenate(ref)[:FV.valid_frame_count(len(audio))]


def test_live_churn_against_oracle(stream_session, weights):
    rs = np.random.RandomState(5)
    S = 64
    streams = make_streams(rs, 150, seed=77)
    server = FV.StreamServer(stream_session, S)
    plan = churn_plan(streams, S, rs)
    assert any(a == "hold" for t in plan for _, a in t.values()) and any(a == "close" for t in plan for _, a in t.values())
    run_ticks(server, plan, garbage=np.random.RandomState(9))
    cfg, w = weights
    orc = FireRedOracle(w, cfg)
    worst, n_seg, n_exact = 0.0, 0, 0
    for st in streams:
        assert st.done and st.pos == len(st.audio)
        plan_col = FV.stream_frame_plan([len(st.audio)])[:, 0].tolist()
        assert st.frames == plan_col, st.sid
        mine = np.concatenate(st.probs) if st.probs else np.zeros(0, np.float32)
        ref = oracle_probs(orc, cfg, st.audio)
        assert mine.shape == ref.shape, st.sid
        if len(ref):
            worst = max(worst, float(np.abs(mine - ref).max()))
        got = pair(st.events)
        assert got == OP.StreamPost(*POST).feed(mine), st.sid
        n_seg += len(got)
        if len(ref) == 0:
            assert st.events == []
            continue
        sm = OP.smooth_probs(ref, 5)
        ring = np.array([ref[max(0, t - 4):t + 1].mean() for t in range(len(ref))])
        if min(np.abs(sm - 0.4).min(), np.abs(ring - 0.4).min()) > TOL:
            assert got == FV.run_stream_vad(st.audio, stream_session).timestamps, st.sid
            n_exact += 1
    print(f"churn: {len(streams)} streams, {len(plan)} ticks, max abs err {worst:.2e}, segments {n_seg}, "
          f"{n_exact} streams checked against run_stream_vad")
    assert worst <= BOUND and n_seg > len(streams) // 2 and n_exact > 0


def _one_stream_plan(st, slot, holds=(), close_after=False):
    plan, pos, k = [], 0, 0
    while pos < len(st.audio):
        if k in holds:
            plan.append({slot: (st, "hold")})
        else:
            plan.append({slot: (st, "feed")})
            pos += C
        k += 1
    if close_after:
        plan.append({slot: (st, "close")})
    return plan


def _clone(st):
    c = Stream(st.sid, st.audio)
    c.close_after = getattr(st, "close_after", False)
    return c


def test_reuse_hold_and_garbage(stream_session):
    S, slot = 16, 5
    raw = synth.synth_streams(3, 9 * C, seed=123)
    first, target = Stream(0, raw[0, :6 * C + 1000].copy()), Stream(1, raw[1, :8 * C + 77].copy())
    # the target stream alone in a fresh server
    fresh = FV.StreamServer(stream_session, S)
    a = _clone(target)
    run_ticks(fresh, _one_stream_plan(a, slot))
    assert len(pair(a.events)) > 0
    # ... in a reused slot, with garbage past n_samples and in every held chunk
    reused = FV.StreamServer(stream_session, S)
    run_ticks(reused, _one_stream_plan(first, slot, holds=(2,)), garbage=np.random.RandomState(1))
    b = _clone(target)
    run_ticks(reused, _one_stream_plan(b, slot), garbage=np.random.RandomState(2))
    # ... and with hold ticks inserted mid-stream (and a close without audio)
    c = _clone(target)
    run_ticks(FV.StreamServer(stream_session, S), _one_stream_plan(c, slot, holds=(0, 3, 4, 7)),
              garbage=np.random.RandomState(3))
    for other in (b, c):
        assert other.events == a.events
        assert other.frames == a.frames
        assert np.array_equal(np.concatenate(other.probs), np.concatenate(a.probs))


def test_graph_replay_bit_identical_and_deterministic(stream_session):
    """eager vs graph replay, two graph servers, and a second schedule through the same graph server"""
    S = 32
    eager, g1, g2 = (FV.StreamServer(stream_session, S, graph=g) for g in (False, True, True))
    results = []
    for server in (eager, g1, g1, g2):
        rs = np.random.RandomState(21)
        streams = make_streams(rs, 60, seed=5)
        ev = run_ticks(server, churn_plan(streams, S, rs), garbage=np.random.RandomState(4))
        results.append((ev, [np.concatenate(s.probs) if s.probs else np.zeros(0) for s in streams]))
    base_ev, base_p = results[0]
    assert sum(len(e) for e in base_ev) > 0
    for ev, p in results[1:]:
        assert ev == base_ev
        assert all(np.array_equal(x, y) for x, y in zip(p, base_p))


def test_rejections(stream_session, cuda, weights):
    cfg, w = weights
    with pytest.raises(ValueError):
        FV.StreamServer(vadx.FireRedSession(W.firered_random_init(W.FireRedConfig(), 0), W.FireRedConfig()), 4)
    with pytest.raises(ValueError):
        FV.StreamServer(stream_session, vadx.FireRedSession.MAX_STREAMS_PER_CALL + 1)
    with pytest.raises(ValueError):
        FV.StreamServer(stream_session, 4, chunk_samples=399)
    S = 4
    server = FV.StreamServer(stream_session, S)
    ok = (torch.zeros((S, C), dtype=torch.int16), torch.zeros(S, dtype=torch.int32), torch.zeros(S, dtype=torch.bool))
    server.step(*ok).host_events()
    bad = [
        (torch.zeros((S, C), dtype=torch.int32), ok[1], ok[2]),
        (torch.zeros((S, C - 1), dtype=torch.int16), ok[1], ok[2]),
        (torch.zeros((S + 1, C), dtype=torch.int16), ok[1], ok[2]),
        (ok[0], torch.zeros(S, dtype=torch.int64), ok[2]),
        (ok[0], torch.zeros(S + 1, dtype=torch.int32), ok[2]),
        (ok[0], ok[1], torch.zeros(S, dtype=torch.float32)),
        (ok[0], torch.tensor([C + 1, 0, 0, 0], dtype=torch.int32), ok[2]),
        (ok[0], torch.tensor([-1, 0, 0, 0], dtype=torch.int32), ok[2]),
        (ok[0], torch.tensor([C - 1, 0, 0, 0], dtype=torch.int32), ok[2]),        # short, not last
        (ok[0], ok[1], None),
    ]
    for args in bad:
        with pytest.raises(ValueError):
            server.step(*args)
    # control words already on the device: the kernel holds the slot and the read-back raises
    raw = synth.synth_streams(1, 4 * C, seed=3)[0]
    clean, dirty = Stream(0, raw.copy()), Stream(0, raw.copy())
    run_ticks(server, _one_stream_plan(clean, 1))
    plan = _one_stream_plan(dirty, 1)
    srv2 = FV.StreamServer(stream_session, S)
    run_ticks(srv2, plan[:2])
    for n_bad, last_bad in ((C + 5, 0), (C - 7, 0), (-3, 1)):
        n = torch.zeros(S, dtype=torch.int32, device=cuda)
        n[1] = n_bad
        lst = torch.zeros(S, dtype=torch.uint8, device=cuda)
        lst[1] = last_bad
        t = srv2.step(torch.zeros((S, C), dtype=torch.int16, device=cuda), n, lst)
        with pytest.raises(PP.ServeTickError) as e:
            t.host_events()
        assert e.value.events == [] and e.value.error != 0
        assert t.frames.cpu().numpy().tolist() == [0] * S
    run_ticks(srv2, plan[2:])
    assert dirty.events == clean.events and dirty.frames == clean.frames
    assert np.array_equal(np.concatenate(dirty.probs), np.concatenate(clean.probs))
