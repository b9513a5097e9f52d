"""MarbleNet slot server (marblenet_vad.StreamServer, vadx_marblenet_serve_step): the online VadPostprocessor alone
against the oracle, live streams against the offline run_vad, churn, a long-lived slot, placement independence, graph
replay, rejections, and the session left as it was."""
import dataclasses
import os

import numpy as np
import pytest
import torch

import vadx
from vadx import marblenet_vad as MV, postprocess as PP, synth, weights as W
from oracle import postproc as OP

pytestmark = pytest.mark.gpu


class ZeroNormal:
    """the reference's tail noise with the randomness taken out: the offline twin of the server's zero padding"""

    def normal(self, loc=0.0, scale=1.0, size=None):
        return np.zeros(size)


@pytest.fixture(scope="module")
def session(cuda):
    cfg = W.MarbleNetConfig()
    return vadx.MarbleNetSession(W.marblenet_random_init(cfg, 0), cfg)


@pytest.fixture(scope="module")
def sample(golden_dir):
    return np.load(os.path.join(golden_dir, "vad_sample_16k.npz"))["audio"].astype(np.int16)


@pytest.fixture(scope="module")
def post(session, sample):
    """MarbleNet's post-processor with the threshold at the median probability of the sample, so that the random-init
    model's tracks hold many segments"""
    p = session.run_batch(torch.from_numpy(sample[:16000 * 5].reshape(5, 16000)).cuda())[1].cpu().numpy()
    return dataclasses.replace(MV.POST_DEFAULT, prob_threshold=float(np.median(p)))


def pair(events):
    """[(kind, value)] of one slot -> [(start, end)]"""
    out, start = [], None
    for k, v in events:
        if k == PP.SERVE_START:
            assert start is None
            start = v
        else:
            assert start is not None
            out.append((start, v))
            start = None
    assert start is None
    return out


def reference(p, cfg, samples):
    """the reference's timestamps of one stream's probabilities (run_vad's post-processing, on the host)"""
    dec = OP.frame_decisions(p, *dataclasses.astuple(cfg)[:7])
    d = np.diff(np.concatenate(([0], dec, [0])).astype(np.int8))
    pairs = np.stack([np.flatnonzero(d == 1), np.flatnonzero(d == -1)], 1)
    return pairs, PP.segments_to_seconds(pairs, len(p), cfg, samples / 16000)


# ---------------------------------------------------------------- the machine alone, given probabilities
CFGS = [(5, 0.4, 20, 2000, 20, 5, 0), (3, 0.5, 10, 1000, 10, 3, 0), (5, 0.4, 20, 120, 20, 5, 0), (1, 0.5, 0, 2000, 0, 0, 0),
        (4, 0.45, 5, 60, 7, 4, 3), (1, 0.5, 3, 50, 0, 0, 2), (7, 0.35, 0, 33, 4, 9, 1), (2, 0.6, 1, 2000, 1, 1, 0),
        (5, 0.4, 1, 7, 1, 0, 0), (64, 0.4, 30, 500, 30, 5, 0),
        (3, 0.5, 10, 1000, 10, 3, 0), (3, 0.5, 10, 0, 10, 3, 0), (3, 0.5, 10, 1, 10, 3, 0), (3, 0.5, 10, 2, 10, 3, 0)]


def track(rs, n):
    lvl = np.clip(0.5 + np.cumsum(rs.normal(0, 0.07, n)), 0, 1)
    gate = np.sin(np.arange(n) / rs.uniform(3, 60) + rs.uniform(0, 6)) > rs.uniform(-0.7, 0.7)
    return np.clip(0.1 + 0.8 * gate * lvl + rs.normal(0, 0.08, n), 0, 1).astype(np.float32)


@pytest.mark.parametrize("cfg_t", CFGS)
def test_machine_matches_oracle(cuda, cfg_t):
    """random tracks tick by tick through the slots of a model-less segmenter, with holds, ragged last chunks and
    finalize with and without audio; slot 0 carries a constant 0.9 track (the split chain), slot 1 an alternating one"""
    F, L, S = 50, 16000, 6
    cfg = MV.POST_DEFAULT.__class__(*cfg_t, 0.02, 0.025, False)
    seg = PP.MarbleNetSlotSegmenter(cfg, S, F, L)
    rs = np.random.RandomState(sum(int(x * 100) for x in cfg_t))
    for trial in range(3):
        plans, probs = {}, {}
        for s in range(S):
            k = int(rs.randint(1, 40))
            p = np.full(k * F, 0.9, np.float32) if s == 0 else track(rs, k * F)
            if s == 1:
                p[::2], p[1::2] = 0.9, 0.1
            n_last = int(rs.choice([L, 1, rs.randint(1, L)]))
            ticks = [(L, 0, w) for w in range(k - 1)] + [(n_last, 1, k - 1)]
            if n_last == L and rs.rand() < 0.5:
                ticks[-1] = (L, 0, k - 1)
                ticks.append((0, 1, None))
            for _ in range(int(rs.randint(0, 4))):                 # holds anywhere
                ticks.insert(int(rs.randint(0, len(ticks))), (0, 0, None))
            plans[s], probs[s] = ticks, (p, (k - 1) * L + n_last)
        ev = {s: [] for s in range(S)}
        frames = {s: [] for s in range(S)}
        for t in range(max(len(p) for p in plans.values())):
            x = rs.rand(S, F + 3).astype(np.float32)                # garbage where a slot does not read
            n = np.zeros(S, np.int32)
            last = np.zeros(S, np.uint8)
            for s, p in plans.items():
                if t < len(p):
                    n[s], last[s], w = p[t]
                    if w is not None:
                        x[s, :F] = probs[s][0][w * F:(w + 1) * F]
            tk = seg.step(torch.from_numpy(x).cuda(), torch.from_numpy(n).cuda(), torch.from_numpy(last).cuda())
            for s, kind, v in tk.host_seconds():
                ev[s].append((kind, v))
            for s, kind, v in tk.host_events():
                frames[s].append((kind, v))
            assert tk.frames.cpu().tolist() == [F if n[s] > 0 else 0 for s in range(S)]
        for s in range(S):
            p, samples = probs[s]
            pairs, ts = reference(p, cfg, samples)
            assert pair(ev[s]) == ts, (cfg_t, trial, s)
            got = pair(frames[s])
            assert [a for a, _ in got] == pairs[:, 0].tolist(), (cfg_t, trial, s)
            assert [b for _, b in got[:-1]] == pairs[:-1, 1].tolist() if len(got) else True
        assert not seg.state.any()


def test_event_bound_with_max_speech_one(cuda):
    """max_speech = 1 on alternating and constant tracks: a tick stages up to its documented bound without overflow"""
    F, L = 50, 16000
    cfg = MV.POST_DEFAULT.__class__(1, 0.5, 0, 1, 0, 0, 0, 0.02, 0.025, False)
    seg = PP.MarbleNetSlotSegmenter(cfg, 2, F, L)
    assert seg.events_per_slot == 2 * (F + seg.delay) + 2
    p = np.zeros((2, 3 * F), np.float32)
    p[0, ::2] = 0.9
    p[1] = 0.9
    ev = {0: [], 1: []}
    for w in range(3):
        tk = seg.step(torch.from_numpy(np.ascontiguousarray(p[:, w * F:(w + 1) * F])).cuda(),
                      torch.tensor([L, L], dtype=torch.int32).cuda(), torch.tensor([w == 2] * 2).cuda())
        for s, kind, v in tk.host_seconds():
            ev[s].append((kind, v))
    for s in range(2):
        assert pair(ev[s]) == reference(p[s], cfg, 3 * L)[1]
    assert len(ev[0]) == 3 * F


def test_long_lived_slot(cuda):
    """one slot closes more than 1000 segments, then the slot serves a new stream"""
    F, L = 50, 16000
    cfg = MV.POST_DEFAULT
    seg = PP.MarbleNetSlotSegmenter(cfg, 2, F, L)
    pattern = np.tile(np.array([0.9] * 30 + [0.1] * 20, np.float32), 2)
    ends = 0
    k = 0
    while True:
        fin = k >= 1100
        x = np.stack([pattern[:F], pattern[:F]])          # one segment per tick
        t = seg.step(torch.from_numpy(x).cuda(), torch.tensor([L, 0], dtype=torch.int32).cuda(),
                     torch.tensor([fin, False]).cuda())
        ends += sum(1 for _, kind, _ in t.host_events() if kind != PP.SERVE_START)
        k += 1
        if fin:
            break
    assert ends > 1000
    rs = np.random.RandomState(5)
    p = track(rs, 7 * F)
    ev = []
    for w in range(7):
        t = seg.step(torch.from_numpy(np.stack([p[w * F:(w + 1) * F], pattern[:F]])).cuda(),
                     torch.tensor([L if w < 6 else 777, 0], dtype=torch.int32).cuda(), torch.tensor([w == 6, False]).cuda())
        ev += [(kind, v) for s, kind, v in t.host_seconds()]
    assert pair(ev) == reference(p, cfg, 6 * L + 777)[1]


# ---------------------------------------------------------------- end to end, against the offline path
def serve(server, streams, flush_last=False, probs=None):
    """streams: {slot: int16 audio}, all starting on the next tick; the other slots hold.  -> {slot: [(start, end)]};
    probs: {slot: list} receives each fed tick's probabilities of the slot"""
    S, L = server.S, server.L
    pos = {s: 0 for s in streams}
    ev = {s: [] for s in streams}
    done = set()
    while len(done) < len(streams):
        chunk = np.zeros((S, L), np.int16)
        n = np.zeros(S, np.int32)
        last = np.zeros(S, np.uint8)
        for s, a in streams.items():
            if s in done:
                continue
            k = min(L, len(a) - pos[s])
            n[s] = k
            chunk[s, :k] = a[pos[s]:pos[s] + k]
            pos[s] += k
            end = pos[s] == len(a)
            if end and (k < L or not flush_last or k == 0):
                last[s] = 1
        t = server.step(torch.from_numpy(chunk), torch.from_numpy(n), torch.from_numpy(last))
        for s, kind, v in t.host_seconds():
            ev[s].append((kind, v))
        if probs is not None:
            for s in streams:
                if n[s] > 0:
                    probs.setdefault(s, []).append(t.probs[s].cpu().numpy())
        done |= {s for s in streams if last[s]}
    return {s: pair(e) for s, e in ev.items()}


def offline(audio, session, L, post):
    return MV.run_vad(audio, session, post, input_audio_length=L, rng=ZeroNormal()).timestamps


@pytest.mark.parametrize("L", [16000, 32000, 20000])
def test_streams_equal_offline_run_vad(cuda, session, sample, post, L):
    server = MV.StreamServer(session, 6, window_samples=L, post=post)
    synth_a = synth.synth_streams(3, 5 * L, seed=L)
    streams = {
        0: sample,
        1: synth_a[0, :3 * L],                     # ends on a window: finalize without audio after it
        2: synth_a[1, :L * 2 // 3],               # shorter than one window
        3: synth_a[2, :2 * L + 1234],             # short last chunk
        4: synth_a[0, :1],                         # one sample
        5: sample[:L],                             # exactly one window
    }
    got_probs = {}
    got = serve(server, streams, flush_last=True, probs=got_probs)
    n_seg = 0
    for s, a in streams.items():
        ref = offline(a, session, L, post)
        assert got[s] == ref, (L, s)
        n_seg += len(ref)
        # each window's probabilities are bit-identical to run_batch over the same windows
        wins, _ = vadx.audio_io.align_non_overlapping(a, L, ZeroNormal())
        ref_p = session.run_batch(torch.from_numpy(wins).cuda())[1, :, :server.F].cpu().numpy()
        assert np.array_equal(np.stack(got_probs[s]), ref_p), (L, s)
    assert n_seg > 5
    # the same streams finalized on their last chunk, in other slots
    got = serve(server, {(s + 1) % 6: a for s, a in streams.items()}, flush_last=False)
    for s, a in streams.items():
        assert got[(s + 1) % 6] == offline(a, session, L, post), (L, s)
    assert not server.seg.state.any()


def test_churn(cuda, session, post):
    """streams join free slots, hold and leave at random; every stream's events equal its own offline run"""
    L, S = 16000, 5
    server = MV.StreamServer(session, S, post=post)
    rs = np.random.RandomState(11)
    pool = synth.synth_streams(12, 6 * L, seed=3)
    todo = [pool[i, :rs.randint(1, 6 * L)] for i in range(12)]
    live, done, nxt = {}, {}, 0                   # slot -> [stream id, received, events]
    while nxt < len(todo) or live:
        for s in range(S):
            if s not in live and nxt < len(todo) and rs.rand() < 0.5:
                live[s] = [nxt, 0, []]
                nxt += 1
        chunk = rs.randint(-9999, 9999, size=(S, L)).astype(np.int16)     # garbage where a slot does not read
        n = np.zeros(S, np.int32)
        last = np.zeros(S, np.uint8)
        for s, (i, received, _) in live.items():
            if rs.rand() < 0.15:
                continue          # hold
            a = todo[i]
            k = min(L, len(a) - received)
            n[s], last[s] = k, received + k == len(a)
            chunk[s, :k] = a[received:received + k]
            live[s][1] += k
        for s, kind, v in server.step(torch.from_numpy(chunk), torch.from_numpy(n), torch.from_numpy(last)).host_seconds():
            live[s][2].append((kind, v))
        for s in [s for s in live if last[s]]:
            i, _, ev = live.pop(s)
            done[i] = pair(ev)
    for i, a in enumerate(todo):
        assert done[i] == offline(a, session, L, post), i


def test_placement_and_graph_replay(cuda, session, sample, post):
    """the same stream in any slot gives the same events; graph replay is bit-identical to eager ticks"""
    a = sample[:9 * 16000 + 500]
    ref = None
    for graph in (True, False):
        for slot in (0, 3):
            got = serve(MV.StreamServer(session, 4, post=post, graph=graph), {slot: a})[slot]
            ref = got if ref is None else ref
            assert got == ref
    g, e = MV.StreamServer(session, 3, post=post, graph=True), MV.StreamServer(session, 3, post=post, graph=False)
    pool = synth.synth_streams(3, 5 * 16000, seed=9)
    for k in range(5):
        chunk = torch.from_numpy(np.ascontiguousarray(pool[:, k * 16000:(k + 1) * 16000]))
        n = torch.tensor([16000, 16000 if k < 4 else 300, 16000], dtype=torch.int32)
        last = torch.tensor([0, k == 4, k == 4], dtype=torch.uint8)
        tg, te = g.step(chunk, n, last), e.step(chunk, n, last)
        assert tg.host_events() == te.host_events()
        for x, y in ((g.scores, e.scores), (g.seg.state, e.seg.state), (g.seg.frames, e.seg.frames)):
            assert torch.equal(x.view(torch.uint8), y.view(torch.uint8))


def test_rejections(cuda, session, post):
    L = 16000
    server = MV.StreamServer(session, 3, post=post)
    chunk = torch.zeros((3, L), dtype=torch.int16)
    with pytest.raises(ValueError, match=r"n_samples must be in \[0, 16000\]"):
        server.step(chunk, torch.tensor([L + 1, 0, 0], dtype=torch.int32), torch.zeros(3, dtype=torch.uint8))
    with pytest.raises(ValueError, match="got a short chunk that is not their stream's last"):
        server.step(chunk, torch.tensor([100, 0, 0], dtype=torch.int32), torch.zeros(3, dtype=torch.uint8))
    with pytest.raises(ValueError, match="chunk must be an int16 tensor"):
        server.step(torch.zeros((3, L + 1), dtype=torch.int16), torch.zeros(3, dtype=torch.int32), torch.zeros(3, dtype=torch.uint8))
    # control words already on the device are checked by the serve kernel: slot 0 out of range, slot 1 short, slot 2 fine
    loud = torch.from_numpy(synth.synth_streams(3, L, seed=4))
    server.step(loud, torch.full((3,), L, dtype=torch.int32), torch.zeros(3, dtype=torch.uint8)).host_events()
    before = server.seg.state.clone()
    server.chunk.copy_(loud.cuda())
    server.n_samples.copy_(torch.tensor([L + 5, 100, L], dtype=torch.int32))
    server.last.zero_()
    with pytest.raises(PP.ServeTickError) as e:
        server.step().host_seconds()
    assert e.value.error == PP.SERVE_ERR_RANGE | PP.SERVE_ERR_SHORT
    assert all(s == 2 for s, _, _ in e.value.events)
    st = server.seg.state
    assert torch.equal(st[:2], before[:2]) and int(st[2, 0]) == 2 * server.F
    # the held slots carry on
    server.step(loud, torch.full((3,), L, dtype=torch.int32), torch.zeros(3, dtype=torch.uint8)).host_events()
    assert int(server.seg.state[0, 0]) == 2 * server.F and int(server.seg.state[1, 0]) == 2 * server.F
    # constructor rejections
    with pytest.raises(ValueError, match="n_slots must be at least 1"):
        MV.StreamServer(session, 0)
    with pytest.raises(ValueError, match="tail_adds_frame_length"):
        MV.StreamServer(session, 2, post=PP.FramePostConfig())
    with pytest.raises(ValueError, match="no frame"):
        MV.StreamServer(session, 2, window_samples=100)
    with pytest.raises(ValueError, match="16000 Hz"):
        cfg = W.MarbleNetConfig()
        MV.StreamServer(vadx.MarbleNetSession(W.marblenet_random_init(cfg, 0), cfg, in_sample_rate=8000), 2)


def test_session_is_not_disturbed(cuda, session, sample, post):
    a = torch.from_numpy(synth.synth_streams(3, 16000, seed=8)).cuda()

    def probe():
        return session.run_batch(a).cpu(), MV.run_vad(sample[:5 * 16000], session, post, input_audio_length=16000,
                                                      rng=ZeroNormal()).timestamps

    before = probe()
    serve(MV.StreamServer(session, 4, post=post), {1: sample[:3 * 16000], 2: sample[16000:3 * 16000]})
    after = probe()
    assert torch.equal(before[0], after[0]) and before[1] == after[1]
