"""FSMN slot server (fsmn_vad.StreamServer, vadx_fsmn_serve_load / vadx_fsmn_serve_step): the timestamp machine alone
against the oracle, live streams against the offline run_vad, churn, a long-lived slot, placement independence, graph
replay, rejections, and the session left as it was."""
import os

import numpy as np
import pytest
import torch

import vadx
from vadx import audio_io, fsmn_vad as FV, postprocess as PP, synth, weights as W
from oracle import postproc as OP

pytestmark = pytest.mark.gpu
D = 160 / 16000


class ZeroNormal:
    """the reference's tail noise with the randomness taken out: the offline twin of the server's zero padding"""

    def normal(self, loc=0.0, scale=1.0, size=None):
        return np.zeros(size)


@pytest.fixture(scope="module")
def wts():
    return W.fsmn_random_init(W.FsmnConfig(), 0)


@pytest.fixture(scope="module")
def sessions(cuda, wts):
    return {L: vadx.FsmnSession(wts, W.FsmnConfig(), chunk_len=L) for L in (16000, 7520, 512)}


@pytest.fixture(scope="module")
def sample(golden_dir):
    return np.load(os.path.join(golden_dir, "vad_sample_16k.npz"))["audio"].astype(np.int16)


LB_S = {16000: 0.3, 7520: 0.3, 512: 0.0}


def offline(audio, sess, lb_s):
    """run_vad(..., normalize=False) with zero padding.  A window of at most 16 frames takes the exact-fp32 skinny GEMMs
    in a one-stream forward but the tensor-core ones in a server's [n_slots][L] forward, so such sessions run the same
    offline computation with the recording in 8 rows of one forward."""
    if sess.T > 16:
        return FV.run_vad(audio, sess, lb_s, rng=ZeroNormal(), normalize=False).timestamps
    lb = FV.look_backward_frames(lb_s)
    aligned, stride, _ = audio_io.align_overlapping(np.asarray(audio, np.int16), sess.chunk_len, lb, 160, ZeroNormal())
    d = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(aligned, (8, aligned.shape[0])))).cuda()
    state, _ = FV.run_streams(sess, d, stride, lb_s)
    cnt, seg = state.segments()
    pairs = PP.take_segments(cnt, seg, 0)
    ts = PP.runs_to_timestamps(pairs, int(state.n_saved[0].item()), D)
    return PP.process_timestamps(ts, FV.FUSION_THRESHOLD, FV.MIN_SPEECH_DURATION)


def pair(events):
    """[(kind, seconds)] of one slot -> [(start, end)]"""
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


def plan(length, full_chunk, flush_last):
    """a stream's (n, last) per tick, fed in full chunks; flush_last: a stream that ends on a full chunk is finalized on
    the following tick without audio"""
    ticks, received = [], 0
    while received < length:
        n = min(full_chunk(received), length - received)
        received += n
        end = received == length
        if end and flush_last and n == full_chunk(received - n):
            ticks.append((n, False))
            ticks.append((0, True))
        else:
            ticks.append((n, end))
    return ticks


def serve(server, streams, flush_last=False):
    """streams: {slot: int16 audio}, all starting on the next tick; the other slots hold.  -> {slot: [(start, end)]}"""
    S, C = server.S, server.stride
    plans = {s: plan(len(a), server.full_chunk, flush_last) for s, a in streams.items()}
    pos = {s: 0 for s in streams}
    ev = {s: [] for s in streams}
    for k in range(max(len(p) for p in plans.values())):
        chunk = np.zeros((S, C), np.int16)
        n = np.zeros(S, np.int32)
        last = np.zeros(S, np.uint8)
        for s, p in plans.items():
            if k < len(p):
                n[s], last[s] = p[k]
                chunk[s, :n[s]] = streams[s][pos[s]:pos[s] + n[s]]
                pos[s] += n[s]
        for s, kind, v in server.step(torch.from_numpy(chunk), torch.from_numpy(n), torch.from_numpy(last)).host_seconds():
            ev[s].append((kind, v))
    return {s: pair(e) for s, e in ev.items()}


# ---------------------------------------------------------------- the machine alone, given flags
def flag_track(rs, n_windows, T):
    """runs of speech / silence flags with random lengths, cut into windows"""
    flags, v = [], rs.rand() < 0.5
    while len(flags) < n_windows * T:
        flags += [int(v)] * int(rs.geometric(rs.choice([0.05, 0.2, 0.6])))
        v = not v
    flags = np.array(flags[:n_windows * T], np.uint8)
    flags[rs.rand(flags.size) < 0.03] ^= 1
    return flags.reshape(n_windows, T)


@pytest.mark.parametrize("T,lb,fusion,min_dur", [(101, 30, 0.3, 0.2), (48, 30, 0.0, 0.0), (4, 0, 0.3, 0.2),
                                                 (4, 0, 0.0, 0.0), (101, 0, 0.05, 0.5), (21, 3, 0.02, 0.03)])
def test_machine_matches_oracle(cuda, T, lb, fusion, min_dur):
    """random flag tracks tick by tick through slots of a model-less segmenter, other slots fed garbage; a stream
    finalized with its last window or without audio after it"""
    L = (T - 1) * 160
    S = 5
    seg = PP.FsmnSlotSegmenter(S, T, L, lb, fusion_threshold=fusion, min_speech_duration=min_dur)
    rs = np.random.RandomState(T * 100 + lb)
    for trial in range(6):
        tracks = {s: flag_track(rs, rs.randint(1, 12), T) for s in range(S) if rs.rand() < 0.8}
        flush = trial % 2 == 1
        plans = {s: [] for s in tracks}
        for s, tr in tracks.items():
            received, fills = 0, []
            while received < L:
                fills.append(seg.full_chunk(received))
                received += fills[-1]
            p = [(n, None) for n in fills[:-1]] + [(fills[-1], 0)] + [(seg.stride, w) for w in range(1, len(tr))]
            if flush:
                p = [(n, w, False) for n, w in p] + [(0, None, True)]
            else:
                p = [(n, w, i == len(p) - 1) for i, (n, w) in enumerate(p)]
            plans[s] = p
        ev = {s: [] for s in tracks}
        for k in range(max(len(p) for p in plans.values())):
            score = rs.randint(0, 2, size=(S, T)).astype(np.uint8)
            n = np.zeros(S, np.int32)
            last = np.zeros(S, np.uint8)
            for s, p in plans.items():
                if k < len(p):
                    n[s], w, last[s] = p[k]
                    if w is not None:
                        score[s] = tracks[s][w]
            t = seg.step(torch.from_numpy(score).cuda(), torch.zeros(S, device="cuda"), torch.from_numpy(n).cuda(),
                         torch.from_numpy(last).cuda())
            for s, kind, v in t.host_seconds():
                ev[s].append((kind, v))
        for s, tr in tracks.items():
            ref = OP.fuse_timestamps(OP.runs_to_timestamps(OP.lookahead_hysteresis_flags(list(tr), lb, 0.5, 0.5), D),
                                     fusion, min_dur)
            assert pair(ev[s]) == ref, (trial, s)
        assert not seg.state.any()


def test_long_lived_slot(cuda):
    """one slot closes more than 1000 segments (no capacity anywhere), then the slot serves a new stream"""
    T, lb = 101, 0
    L = 16000
    seg = PP.FsmnSlotSegmenter(2, T, L, lb, fusion_threshold=0.0, min_speech_duration=0.0)
    pattern = np.tile(np.array([1, 1, 1, 0, 0], np.uint8), T)[:T]
    n_windows = 80
    ends = 0
    received = 0
    z = torch.zeros(2, device="cuda")
    k = 0
    while True:
        full = seg.full_chunk(received)
        received += full
        fin = k >= n_windows
        n = torch.tensor([full, 0], dtype=torch.int32)
        t = seg.step(torch.from_numpy(np.stack([np.roll(pattern, k), pattern])).cuda(), z, n.cuda(),
                     torch.tensor([fin, False]).cuda())
        ends += sum(1 for _, kind, _ in t.host_events() if kind != PP.SERVE_START)
        k += 1
        if fin:
            break
    assert ends > 1000
    rs = np.random.RandomState(5)
    tr = flag_track(rs, 4, T)
    ev = []
    received, w = 0, 0
    while w < len(tr):
        full = seg.full_chunk(received)
        received += full
        runs = received >= L
        t = seg.step(torch.from_numpy(np.stack([tr[w] if runs else pattern, pattern])).cuda(), z,
                     torch.tensor([full, 0], dtype=torch.int32).cuda(), torch.tensor([runs and w == len(tr) - 1, False]).cuda())
        ev += [(kind, v) for s, kind, v in t.host_seconds()]
        w += runs
    assert pair(ev) == OP.fuse_timestamps(OP.runs_to_timestamps(OP.lookahead_hysteresis_flags(list(tr), 0, 0.5, 0.5), D),
                                          0.0, 0.0)


# ---------------------------------------------------------------- end to end, against the offline path
@pytest.mark.parametrize("L", [16000, 7520, 512])
def test_streams_equal_offline_run_vad(cuda, sessions, sample, L):
    sess, lb_s = sessions[L], LB_S[L]
    server = FV.StreamServer(sess, 6, look_backward_s=lb_s)
    stride = server.stride
    synth_a = synth.synth_streams(3, 3 * L + 5 * stride, seed=L)
    streams = {
        0: sample,
        1: synth_a[0, :L + 3 * stride],            # ends on a window: finalize without audio
        2: synth_a[1, :L * 2 // 3],               # shorter than one window
        3: synth_a[2, :L + 2 * stride + 1234 % stride],   # short last chunk
        4: synth_a[0, :L],                         # exactly one window
        5: sample[:L + 7 * stride + 17],
    }
    got = serve(server, streams, flush_last=True)
    for s, a in streams.items():
        assert got[s] == offline(a, sess, lb_s), (L, s)
    # the same streams finalized on their last chunk, in other slots
    got = serve(server, {(s + 1) % 6: a for s, a in streams.items()}, flush_last=False)
    for s, a in streams.items():
        assert got[(s + 1) % 6] == offline(a, sess, lb_s), (L, s)
    assert not server.seg.state.any()


def test_churn(cuda, sessions):
    """streams join free slots, hold and leave at random; every stream's events equal its own offline run"""
    L = 7520
    sess, lb_s = sessions[L], LB_S[L]
    S = 5
    server = FV.StreamServer(sess, S, look_backward_s=lb_s)
    rs = np.random.RandomState(11)
    pool = synth.synth_streams(14, 6 * L, seed=3)
    todo = [pool[i, :rs.randint(100, 6 * L)] for i in range(14)]
    live = {}                     # slot -> [stream id, received, events]
    done = {}
    nxt = 0
    while nxt < len(todo) or live:
        for s in range(S):
            if s not in live and nxt < len(todo) and rs.rand() < 0.5:
                live[s] = [nxt, 0, []]
                nxt += 1
        chunk = np.zeros((S, server.stride), np.int16)
        n = np.zeros(S, np.int32)
        last = np.zeros(S, np.uint8)
        for s, (i, received, _) in live.items():
            if rs.rand() < 0.15:
                continue          # hold
            a = todo[i]
            k = min(server.full_chunk(received), len(a) - received)
            n[s], last[s] = k, received + k == len(a)
            chunk[s, :k] = a[received:received + k]
            live[s][1] += k
        chunk[n == 0] = rs.randint(-9999, 9999, size=chunk[n == 0].shape)      # never read
        for s, kind, v in server.step(torch.from_numpy(chunk), torch.from_numpy(n), torch.from_numpy(last)).host_seconds():
            live[s][2].append((kind, v))
        for s in [s for s in live if last[s]]:
            i, _, ev = live.pop(s)
            done[i] = pair(ev)
    for i, a in enumerate(todo):
        assert done[i] == offline(a, sess, lb_s), i


def test_placement_and_graph_replay(cuda, sessions, sample):
    """the same stream in any slot gives the same events; graph replay is bit-identical to eager ticks"""
    L = 16000
    sess = sessions[L]
    a = sample[:L + 9 * 11040 + 500]
    ref = None
    for graph in (True, False):
        for slot in (0, 3):
            server = FV.StreamServer(sess, 4, graph=graph)
            got = serve(server, {slot: a})[slot]
            ref = got if ref is None else ref
            assert got == ref
    g, e = FV.StreamServer(sess, 3, graph=True), FV.StreamServer(sess, 3, graph=False)
    rs = np.random.RandomState(2)
    for k in range(5):
        chunk = torch.from_numpy(rs.randint(-20000, 20000, size=(3, g.stride)).astype(np.int16))
        n = torch.tensor([g.full_chunk(min(k, 2) * g.stride if k < 2 else L)] * 3, dtype=torch.int32)
        last = torch.tensor([0, 0, k == 4], dtype=torch.uint8)
        tg, te = g.step(chunk, n, last), e.step(chunk, n, last)
        assert tg.host_events() == te.host_events()
        for x, y in ((g.window, e.window), (g.score, e.score), (g.noisy, e.noisy), (g.caches[(k + 1) & 1], e.caches[(k + 1) & 1]),
                     (g.seg.state, e.seg.state)):
            assert torch.equal(x.view(torch.uint8), y.view(torch.uint8))      # bitwise: noisy_dB is NaN in all-speech windows


def test_rejections(cuda, sessions):
    L = 16000
    server = FV.StreamServer(sessions[L], 3)
    C = server.stride
    chunk = torch.zeros((3, C), dtype=torch.int16)
    # host-side checks keep load_tick_inputs' messages
    with pytest.raises(ValueError, match=r"n_samples must be in \[0, 11040\]"):
        server.step(chunk, torch.tensor([C + 1, 0, 0], dtype=torch.int32), torch.zeros(3, dtype=torch.uint8))
    with pytest.raises(ValueError, match="chunk must be an int16 tensor"):
        server.step(torch.zeros((3, C + 1), dtype=torch.int16), torch.zeros(3, dtype=torch.int32), torch.zeros(3, dtype=torch.uint8))
    # tick 0: every slot fills its first stride samples
    server.step(chunk, torch.full((3,), C, dtype=torch.int32), torch.zeros(3, dtype=torch.uint8)).host_events()
    assert server.full_chunk(C) == L - C
    # tick 1: slot 0 oversteps its first window (range), slot 1 sends a short chunk that is not its last, slot 2 is fine
    loud = torch.from_numpy(synth.synth_streams(3, C, seed=4))
    before = server.seg.state.clone()
    with pytest.raises(PP.ServeTickError) as e:
        server.step(loud, torch.tensor([C, 100, L - C], dtype=torch.int32), torch.zeros(3, dtype=torch.uint8)).host_seconds()
    assert e.value.error == PP.SERVE_ERR_RANGE | PP.SERVE_ERR_SHORT
    assert all(s == 2 for s, _, _ in e.value.events)
    st = server.seg.state
    assert torch.equal(st[:2], before[:2]) and int(st[2, 0]) == L and int(st[2, 2]) == server.T - server.lb
    # the held slots carry on
    server.step(loud, torch.tensor([L - C, L - C, C], dtype=torch.int32), torch.zeros(3, dtype=torch.uint8)).host_events()
    assert int(server.seg.state[0, 0]) == L and int(server.seg.state[1, 0]) == L


def test_session_is_not_disturbed(cuda, wts, sample):
    L = 16000
    sess = vadx.FsmnSession(wts, W.FsmnConfig(), chunk_len=L)
    a = torch.from_numpy(synth.synth_streams(3, L, seed=8)).cuda()
    caches = sess.new_caches(3, "cuda")
    noise = torch.full((3,), 4.0, device="cuda")

    def probe():
        score, new, noisy, p, pw = sess.run_batch(a, caches, noise)
        r = FV.run_vad(sample[:5 * L], sess, normalize=False, rng=ZeroNormal())
        return [t.cpu() for t in [score, noisy, p, pw] + new], r.timestamps, r.saved

    before = probe()
    server = FV.StreamServer(sess, 4, one_minus_speech_threshold=0.9)
    serve(server, {1: sample[:3 * L], 2: sample[L:3 * L]})
    after = probe()
    assert all(torch.equal(x, y) for x, y in zip(before[0], after[0]))
    assert before[1] == after[1] and np.array_equal(before[2], after[2])
