"""Silero slot server (silero_vad.StreamServer, vadx_silero_serve_load / vadx_silero_serve_step): the iterator against
the reference VADIterator's record at kernel level, a long-lived slot, live churn against the oracle and the host
VADIterator, small shapes, placement independence, graph replay, rejections, and the session left as it was."""
import os

import numpy as np
import pytest
import torch

import vadx
from vadx import postprocess as PP, silero_vad as SV, synth, weights as W
from oracle.silero import OnnxWrapperOracle, SileroNetOracle

pytestmark = pytest.mark.gpu
BOUND = 5e-5      # the Silero forward's asserted bound (tests/test_gpu_silero.py)
WIN = 512
SCALE = 0.000030517578


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(os.path.join(golden_dir, "silero_iter.npz"))


@pytest.fixture(scope="module")
def wts():
    return W.silero_random_init(W.SileroConfig(), 0)


@pytest.fixture(scope="module")
def session(cuda, wts):
    return vadx.SileroSession(wts, W.SileroConfig())


class Replay:
    """the model surface VADIterator calls, replaying given probabilities"""

    def __init__(self, p):
        self.p, self.i = [float(v) for v in p], 0

    def reset_states(self):
        self.i = 0

    def __call__(self, chunk, sr):
        self.i += 1
        return torch.tensor([[self.p[self.i - 1]]])


def iterator_events(p, threshold=0.5, min_silence_duration_ms=100, speech_pad_ms=30, seconds=False, time_resolution=1):
    """[(window, kind, value)] of the host VADIterator replaying `p`; a stream that ends triggered gets the server's
    end-of-stream event (the windows consumed, in samples)"""
    it = SV.VADIterator(Replay(p), threshold=threshold, min_silence_duration_ms=min_silence_duration_ms,
                        speech_pad_ms=speech_pad_ms)
    ev = []
    for w in range(len(p)):
        r = it(torch.zeros(WIN), return_seconds=seconds, time_resolution=time_resolution)
        if r is not None:
            (k, v), = r.items()
            ev.append((w, PP.SERVE_START if k == "start" else PP.SERVE_END, v))
    if it.triggered:
        v = len(p) * WIN
        ev.append((len(p) - 1, PP.SERVE_END_OF_STREAM, round(v / 16000, time_resolution) if seconds else v))
    return ev


# ---------------------------------------------------------------- kernel level, given probabilities
def feed_track(p, W_, seg, slot, rs, short_last=True):
    """one track through slot `slot` of a model-less segmenter in W-window ticks, finalized with its last tick; the
    other slots hold, with garbage probabilities.  -> [(tick, kind, samples, seconds at resolution 2)]"""
    S = seg.S
    n_ticks = max(1, (len(p) + W_ - 1) // W_)
    out = []
    for k in range(n_ticks):
        f = min(W_, len(p) - k * W_)
        probs = rs.uniform(0, 1, size=(W_, S)).astype(np.float32)
        probs[:f, slot] = p[k * W_:k * W_ + f]
        n = np.zeros(S, np.int32)
        n[slot] = W_ * WIN if f == W_ else (f - 1) * WIN + (rs.randint(1, WIN + 1) if short_last else WIN)
        lst = np.zeros(S, np.uint8)
        lst[slot] = k == n_ticks - 1
        t = seg.step(torch.from_numpy(probs).cuda(), torch.from_numpy(n).cuda(), torch.from_numpy(lst).cuda())
        assert t.frames.cpu().numpy().tolist() == [f if s == slot else 0 for s in range(S)]
        ev, smp, sec = t.host_events(), t.host_samples(), t.host_seconds(2)
        assert all(s == slot for s, _, _ in ev)
        assert [(s, k_) for s, k_, _ in smp] == [(s, k_) for s, k_, _ in ev] == [(s, k_) for s, k_, _ in sec]
        out += [(k, kind, v, u) for (_, kind, v), (_, _, u) in zip(smp, sec)]
    return out


@pytest.mark.parametrize("i", range(3))
@pytest.mark.parametrize("W_", [1, 5, 7])
def test_kernel_reference_record(cuda, gold, i, W_):
    p = gold[f"it{i}_probs"]
    thr, min_sil, pad = gold[f"it{i}_params"]
    seg = PP.SileroSlotSegmenter(float(thr), int(min_sil), int(pad), n_slots=5, windows_per_tick=W_, device="cuda")
    got = feed_track(p, W_, seg, slot=3, rs=np.random.RandomState(i))
    ref_smp, ref_sec = gold[f"it{i}_smp"], gold[f"it{i}_sec"]
    mine = [e for e in got if e[1] != PP.SERVE_END_OF_STREAM]
    assert len(mine) == len(ref_smp) > 0
    for (tick, kind, smp, sec), (w, k_ref, v_smp), (_, _, v_sec) in zip(mine, ref_smp.tolist(), ref_sec.tolist()):
        assert tick == int(w) // W_ and kind == int(k_ref)
        assert smp == v_smp and sec == v_sec
    # the reference leaves a segment open at the end of the track; the server closes it with kind 2
    ends_triggered = int(ref_smp[-1, 1]) == 0
    eos = [e for e in got if e[1] == PP.SERVE_END_OF_STREAM]
    last_tick = (len(p) + W_ - 1) // W_ - 1
    assert eos == ([(last_tick, PP.SERVE_END_OF_STREAM, len(p) * WIN, round(len(p) * WIN / 16000, 2))]
                   if ends_triggered else [])


def alternating(rs, n_segments, lo=10, hi=40):
    runs = rs.randint(lo, hi, size=2 * n_segments)
    gate = np.concatenate([np.full(r, i % 2 == 0) for i, r in enumerate(runs)])
    return np.clip(np.where(gate, 0.85, 0.1) + rs.normal(0, 0.05, size=gate.shape), 0, 1).astype(np.float32)


def test_kernel_long_lived_slot(cuda):
    """> 1000 segments through one slot in one stream, nothing dropped, then a second stream in the same slot"""
    rs = np.random.RandomState(11)
    p = alternating(rs, 1100)
    W_, S, slot = 5, 4, 2
    seg = PP.SileroSlotSegmenter(n_slots=S, windows_per_tick=W_, device="cuda")
    for track in (p, p[:3001]):
        got = feed_track(track, W_, seg, slot, rs, short_last=False)
        ref = iterator_events(track)
        assert [(k, v) for _, k, v, _ in got] == [(k, v) for _, k, v in ref]
    assert sum(1 for _, k, _ in iterator_events(p) if k == PP.SERVE_END) > 1000


def test_kernel_rejection_keeps_other_slots_events(cuda):
    """a tick that rejects one slot's control words still reports every other slot's events on the exception; the
    rejected slot is held, so its events are those of the windows it did consume"""
    W_, S = 5, 3
    p = alternating(np.random.RandomState(4), 30)[:300]
    runs = []
    for bad in (False, True):
        seg = PP.SileroSlotSegmenter(n_slots=S, windows_per_tick=W_, device="cuda")
        ev, n_rejected = [], 0
        for k in range(len(p) // W_):
            probs = np.zeros((W_, S), np.float32)
            probs[:, 0] = probs[:, 1] = p[k * W_:(k + 1) * W_]
            n = np.array([W_ * WIN, W_ * WIN, 0], np.int32)
            if bad and k % 3 == 0:
                n[1] = W_ * WIN + 1
            t = seg.step(torch.from_numpy(probs).cuda(), torch.from_numpy(n).cuda(),
                         torch.zeros(S, dtype=torch.uint8, device=cuda))
            try:
                got = t.host_samples()
            except PP.ServeTickError as e:
                assert e.error == PP.SERVE_ERR_RANGE
                assert t.frames.cpu().numpy().tolist() == [W_, 0, 0]
                got, n_rejected = e.events, n_rejected + 1
            ev += got
        runs.append((ev, n_rejected))
    slot = lambda ev, s: [(k, v) for s_, k, v in ev if s_ == s]
    assert slot(runs[1][0], 0) == slot(runs[0][0], 0) == [(k, v) for _, k, v in iterator_events(p)
                                                         if k != PP.SERVE_END_OF_STREAM]
    assert len(slot(runs[0][0], 0)) > 4
    assert runs[0][1] == 0 and runs[1][1] == 20
    kept = np.concatenate([p[k * W_:(k + 1) * W_] for k in range(len(p) // W_) if k % 3])
    assert slot(runs[1][0], 1) == [(k, v) for _, k, v in iterator_events(kept) if k != PP.SERVE_END_OF_STREAM]


# ---------------------------------------------------------------- server driver
class Stream:
    def __init__(self, sid, audio):
        self.sid, self.audio, self.pos = sid, audio, 0
        self.windows, self.probs, self.events, self.samples = [], [], [], []
        self.done = False


def run_ticks(server, plan, garbage=None):
    """plan: list of ticks, each {slot: (stream, action)} with action 'feed', 'hold' or 'close' (n = 0, last = 1).
    Slots not named hold.  `garbage` (RandomState) fills every sample past n with noise."""
    S, L = server.S, server.chunk_samples
    out = []
    for tick in plan:
        chunk = np.zeros((S, L), np.int16)
        if garbage is not None:
            chunk = garbage.randint(-32768, 32767, size=(S, L)).astype(np.int16)
        n = np.zeros(S, np.int32)
        last = np.zeros(S, np.uint8)
        fed = {}
        for slot, (st, action) in tick.items():
            if action == "feed":
                m = min(L, len(st.audio) - st.pos)
                assert m > 0
                chunk[slot, :m] = st.audio[st.pos:st.pos + m]
                n[slot] = m
                st.pos += m
                # a stream that ends on a full chunk may instead be closed by a later tick with n_samples = 0
                last[slot] = st.pos == len(st.audio) and not (getattr(st, "close_after", False) and m == L)
                fed[slot] = st
            elif action == "close":
                last[slot] = 1
                fed[slot] = st
        t = server.step(torch.from_numpy(chunk).pin_memory(), torch.from_numpy(n).pin_memory(),
                        torch.from_numpy(last).pin_memory())
        ev, smp = t.host_events(), t.host_samples()
        slots = [s for s, _, _ in ev]
        assert slots == sorted(slots)
        probs, windows = t.probs.cpu().numpy(), t.frames.cpu().numpy()
        assert probs.shape == (S, server.W)
        for slot, st in fed.items():
            assert windows[slot] == (n[slot] + WIN - 1) // WIN
            if n[slot] > 0:
                st.windows.append(int(windows[slot]))
            st.probs.append(probs[slot, :windows[slot]].copy())
            if last[slot]:
                st.done = True
        for slot in range(S):
            if slot not in fed:
                assert windows[slot] == 0
        for (s, kind, w), (_, _, x) in zip(ev, smp):
            assert s in fed, (s, kind, w)
            fed[s].events.append((kind, w))
            fed[s].samples.append((kind, x))
        out.append(ev)
    return out


def churn_plan(streams, S, L, rs, p_hold=0.1, p_join=0.3):
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
                st._planned = fed_so_far + min(L, left)
                if st._planned == len(st.audio) and not getattr(st, "close_after", False):
                    del busy[slot]
            else:
                tick[slot] = (st, "close")
                del busy[slot]
        plan.append(tick)
    return plan


def make_streams(rs, n, L, seed):
    lengths = list(rs.randint(1, 12 * L, size=n))
    lengths[:7] = [1, 300, 511, L * 3 + 250, L * 4, L * 2, L + WIN]    # under one window; short last; exact multiples
    raw = synth.synth_streams(n, max(lengths), seed=seed)
    streams = [Stream(i, raw[i, :lengths[i]].copy()) for i in range(n)]
    for st in streams:
        st.close_after = len(st.audio) % L == 0 and rs.rand() < 0.7    # exact multiples: close with n_samples = 0
    streams[4].close_after = True
    return streams


def oracle_probs(wts, streams):
    """OnnxWrapperOracle.audio_forward over every stream at once: zero padding past a stream's end is what its short
    last window gets, and the network is causal, so each stream's first ceil(len/512) probabilities are its own"""
    cfg = W.SileroConfig()
    n = max(len(st.audio) for st in streams)
    x = np.zeros((len(streams), n), np.float32)
    for i, st in enumerate(streams):
        x[i, :len(st.audio)] = st.audio.astype(np.float32) * SCALE
    p = OnnxWrapperOracle(SileroNetOracle(wts, cfg)).audio_forward(torch.from_numpy(x)).numpy()
    return [p[i, :(len(st.audio) + WIN - 1) // WIN] for i, st in enumerate(streams)]


def check_churn(session, wts, measured, S, W_, n_streams, seed, what):
    rs = np.random.RandomState(seed)
    L = W_ * WIN
    streams = make_streams(rs, n_streams, L, seed=seed + 70)
    server = SV.StreamServer(session, S, windows_per_tick=W_)
    plan = churn_plan(streams, S, L, rs)
    assert any(a == "hold" for t in plan for _, a in t.values()) and any(a == "close" for t in plan for _, a in t.values())
    run_ticks(server, plan, garbage=np.random.RandomState(seed + 1))
    refs = oracle_probs(wts, streams)
    worst, n_ev, n_exact = 0.0, 0, 0
    for st, ref in zip(streams, refs):
        assert st.done and st.pos == len(st.audio)
        assert sum(st.windows) == (len(st.audio) + WIN - 1) // WIN, st.sid
        mine = np.concatenate(st.probs)
        assert mine.shape == ref.shape, st.sid
        worst = max(worst, float(np.abs(mine - ref).max()))
        assert st.samples == [(k, v) for _, k, v in iterator_events(mine)], st.sid
        n_ev += len(st.events)
        if min(np.abs(ref - 0.5).min(), np.abs(ref - 0.35).min()) > 1e-3:
            assert st.samples == [(k, v) for _, k, v in iterator_events(ref)], st.sid
            n_exact += 1
    print(f"{what}: {len(streams)} streams, {len(plan)} ticks, max abs err {worst:.2e}, events {n_ev}, "
          f"{n_exact} streams checked against the oracle's events")
    measured(f"silero StreamServer {what} probs vs OnnxWrapperOracle", worst, BOUND)
    assert n_ev > len(streams) // 2 and n_exact > 0


def test_live_churn_against_oracle(session, wts, measured):
    check_churn(session, wts, measured, 64, 5, 150, 5, "churn S=64 W=5")


@pytest.mark.parametrize("S,W_", [(48, 1), (8, 5), (16, 1)])
def test_small_shapes_against_oracle(session, wts, measured, S, W_):
    """W = 1 runs the per-window recurrence, n_slots <= 16 the skinny path"""
    check_churn(session, wts, measured, S, W_, 30, 40 + S + W_, f"S={S} W={W_}")


def _one_stream_plan(st, slot, L, holds=(), close_after=False):
    plan, pos, k = [], 0, 0
    while pos < len(st.audio):
        if k in holds:
            plan.append({slot: (st, "hold")})
        else:
            plan.append({slot: (st, "feed")})
            pos += L
        k += 1
    if close_after:
        plan.append({slot: (st, "close")})
    return plan


def _clone(st):
    c = Stream(st.sid, st.audio)
    c.close_after = getattr(st, "close_after", False)
    return c


def test_placement_independence(session):
    """the same stream in a fresh server, in a reused slot (garbage past n and in held chunks), and with holds"""
    S, slot, W_ = 16, 5, 5
    L = W_ * WIN
    raw = synth.synth_streams(3, 40 * L, seed=123)
    first, target = Stream(0, raw[0, :26 * L + 1000].copy()), Stream(1, raw[1, :38 * L + 77].copy())
    a = _clone(target)
    run_ticks(SV.StreamServer(session, S, W_), _one_stream_plan(a, slot, L))
    assert len(a.events) > 0
    reused = SV.StreamServer(session, S, W_)
    run_ticks(reused, _one_stream_plan(first, slot, L, holds=(2,)), garbage=np.random.RandomState(1))
    b = _clone(target)
    run_ticks(reused, _one_stream_plan(b, slot, L), garbage=np.random.RandomState(2))
    c = _clone(target)
    run_ticks(SV.StreamServer(session, S, W_), _one_stream_plan(c, slot, L, holds=(0, 3, 4, 7)),
              garbage=np.random.RandomState(3))
    for other in (b, c):
        assert other.events == a.events
        assert other.windows == a.windows
        assert np.array_equal(np.concatenate(other.probs), np.concatenate(a.probs))


def test_graph_replay_bit_identical_and_deterministic(session):
    """eager vs graph replay, two graph servers, and a second schedule through the same graph server"""
    S, W_ = 32, 5
    eager, g1, g2 = (SV.StreamServer(session, S, W_, graph=g) for g in (False, True, True))
    results = []
    for server in (eager, g1, g1, g2):
        rs = np.random.RandomState(21)
        streams = make_streams(rs, 60, W_ * WIN, seed=5)
        ev = run_ticks(server, churn_plan(streams, S, W_ * WIN, rs), garbage=np.random.RandomState(4))
        results.append((ev, [np.concatenate(s.probs) for s in streams]))
    base_ev, base_p = results[0]
    assert sum(len(e) for e in base_ev) > 0
    for ev, p in results[1:]:
        assert ev == base_ev
        assert all(np.array_equal(x, y) for x, y in zip(p, base_p))


def test_rejections(session, cuda):
    for bad in (dict(session=object(), n_slots=4), dict(n_slots=0), dict(n_slots=4, windows_per_tick=0),
                dict(n_slots=vadx.SileroSession.MAX_ROWS_PER_CALL // 5 + 1, windows_per_tick=5)):
        with pytest.raises(ValueError):
            SV.StreamServer(**{"session": session, **bad})
    S, W_ = 4, 5
    L = W_ * WIN
    server = SV.StreamServer(session, S, W_)
    ok = (torch.zeros((S, L), dtype=torch.int16), torch.zeros(S, dtype=torch.int32), torch.zeros(S, dtype=torch.bool))
    server.step(*ok).host_events()
    bad = [
        (torch.zeros((S, L), dtype=torch.float32), ok[1], ok[2]),
        (torch.zeros((S, L - 1), dtype=torch.int16), ok[1], ok[2]),
        (torch.zeros((S + 1, L), dtype=torch.int16), ok[1], ok[2]),
        (ok[0], torch.zeros(S, dtype=torch.int64), ok[2]),
        (ok[0], torch.zeros(S + 1, dtype=torch.int32), ok[2]),
        (ok[0], ok[1], torch.zeros(S, dtype=torch.float32)),
        (ok[0], torch.tensor([L + 1, 0, 0, 0], dtype=torch.int32), ok[2]),
        (ok[0], torch.tensor([-1, 0, 0, 0], dtype=torch.int32), ok[2]),
        (ok[0], torch.tensor([L - 1, 0, 0, 0], dtype=torch.int32), ok[2]),        # short, not last
        (ok[0], ok[1], None),
    ]
    for args in bad:
        with pytest.raises(ValueError):
            server.step(*args)
    # control words already on the device: the kernel holds the slot, the read-back raises with the other slots'
    # events, and the rejected slot then resumes as if the rejected ticks had been holds
    raw = synth.synth_streams(2, 12 * L, seed=3)
    clean, dirty, other = Stream(0, raw[0].copy()), Stream(0, raw[0].copy()), Stream(1, raw[1].copy())
    run_ticks(SV.StreamServer(session, S, W_), _one_stream_plan(clean, 1, L))
    alone = Stream(1, raw[1].copy())
    run_ticks(SV.StreamServer(session, S, W_), _one_stream_plan(alone, 2, L))
    srv2 = SV.StreamServer(session, S, W_)
    plan = _one_stream_plan(dirty, 1, L)
    run_ticks(srv2, [{**t, 2: (other, "feed")} for t in plan[:2]])
    for n_bad, last_bad in ((L + 5, 0), (L - 7, 0), (-3, 1)):
        n = torch.tensor([0, n_bad, L, 0], dtype=torch.int32, device=cuda)
        lst = torch.tensor([0, last_bad, 0, 0], dtype=torch.uint8, device=cuda)
        chunk = torch.zeros((S, L), dtype=torch.int16, device=cuda)
        chunk[2] = torch.from_numpy(other.audio[other.pos:other.pos + L]).to(cuda)
        other.pos += L
        t = srv2.step(chunk, n, lst)
        with pytest.raises(PP.ServeTickError) as e:
            t.host_samples()
        assert e.value.error != 0 and all(s == 2 for s, _, _ in e.value.events)
        other.samples += [(kind, v) for _, kind, v in e.value.events]
        other.probs.append(t.probs.cpu().numpy()[2].copy())
        assert t.frames.cpu().numpy().tolist() == [0, 0, W_, 0]
    rest = plan[2:]
    n_other = (len(other.audio) - other.pos) // L
    run_ticks(srv2, [{**(rest[i] if i < len(rest) else {}), **({2: (other, "feed")} if i < n_other else {})}
                     for i in range(max(len(rest), n_other))])
    assert dirty.events == clean.events and dirty.windows == clean.windows
    assert np.array_equal(np.concatenate(dirty.probs), np.concatenate(clean.probs))
    assert other.samples == alone.samples
    assert np.array_equal(np.concatenate(other.probs), np.concatenate(alone.probs))


def test_session_unchanged_by_serving(session):
    """speech_probs and the OnnxWrapper call give the same results before and after server ticks"""
    a = torch.from_numpy(synth.synth_streams(3, 40 * WIN + 100, seed=8)).float().cuda() * SCALE

    def probe():
        p = session.speech_probs(a).cpu().numpy()
        session.reset_states()
        o = [session(a[:, t * WIN:(t + 1) * WIN], 16000).cpu().numpy() for t in range(4)]
        return p, np.concatenate(o, axis=1)

    before = probe()
    streams = make_streams(np.random.RandomState(2), 20, 5 * WIN, seed=9)
    for graph in (False, True):
        server = SV.StreamServer(session, 16, graph=graph)
        run_ticks(server, churn_plan(streams if not graph else [_clone(s) for s in streams], 16, 5 * WIN,
                                     np.random.RandomState(3)))
        after = probe()
        assert np.array_equal(before[0], after[0]) and np.array_equal(before[1], after[1])


def test_session_usable_between_ticks(session):
    """speech_probs and the OnnxWrapper call between two ticks of a graph server give what they give alone, and the
    server's later ticks match those of a server nobody interrupted"""
    a = torch.from_numpy(synth.synth_streams(3, 40 * WIN + 100, seed=8)).float().cuda() * SCALE

    def probe():
        p = session.speech_probs(a).cpu().numpy()
        session.reset_states()
        o = [session(a[:, t * WIN:(t + 1) * WIN], 16000).cpu().numpy() for t in range(4)]
        return p, np.concatenate(o, axis=1)

    alone = probe()
    L = 5 * WIN
    streams = make_streams(np.random.RandomState(2), 20, L, seed=9)
    clones = [_clone(s) for s in streams]
    plan = churn_plan(streams, 16, L, np.random.RandomState(3))
    plan_c = churn_plan(clones, 16, L, np.random.RandomState(3))
    quiet, busy = SV.StreamServer(session, 16), SV.StreamServer(session, 16)
    ev_quiet = run_ticks(quiet, plan)
    ev_busy = []
    for k, tick in enumerate(plan_c):
        ev_busy += run_ticks(busy, [tick])
        if k in (0, 1, 2, len(plan_c) // 2):         # before, during and after the graph captures of both parities
            between = probe()
            assert np.array_equal(between[0], alone[0]) and np.array_equal(between[1], alone[1])
    assert ev_busy == ev_quiet and sum(len(e) for e in ev_quiet) > 0
    for s, c in zip(streams, clones):
        assert c.samples == s.samples and c.windows == s.windows
        assert np.array_equal(np.concatenate(c.probs), np.concatenate(s.probs))
