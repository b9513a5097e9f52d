"""bench.py --dump-outputs: what it writes for one step of run_vad_streams (host-side, no device needed)."""
import os

import numpy as np
import torch

import bench


def fake_step(S=6, T=10, max_seg=6, seed=0):
    rs = np.random.RandomState(seed)
    probs = torch.from_numpy(rs.rand(S, T).astype(np.float32))
    dec = torch.from_numpy(rs.randint(0, 2, size=(S, T)).astype(np.int8))
    cnt = torch.from_numpy(np.arange(S, dtype=np.int32) % (max_seg + 2))        # includes counts above max_seg
    seg = torch.from_numpy(rs.randint(-99, 99, size=(S, max_seg, 2)).astype(np.int32))   # slots past the count: garbage
    n_valid = torch.from_numpy(np.full(S, T - 3, np.int32))
    return probs, dec, cnt, seg, n_valid


def test_dump_writes_float32_and_masks_unwritten_slots(tmp_path):
    probs, dec, cnt, seg, n_valid = fake_step()
    seg_before = seg.clone()
    bench.dump_outputs(str(tmp_path), probs, dec, cnt, seg, n_valid)
    assert torch.equal(seg, seg_before)                                         # the caller's tensors are left alone
    assert sorted(os.listdir(tmp_path)) == ["decisions.npy", "frame_probs.npy", "seg_count.npy", "segments.npy"]
    got = {k: np.load(tmp_path / f"{k}.npy") for k in ("frame_probs", "decisions", "seg_count", "segments")}
    assert all(a.dtype == np.float32 for a in got.values())
    assert np.array_equal(got["frame_probs"], probs.numpy())
    assert np.array_equal(got["seg_count"], cnt.numpy())
    assert np.array_equal(got["decisions"][:, :7], dec.numpy()[:, :7]) and not got["decisions"][:, 7:].any()
    for s in range(6):
        k = min(int(cnt[s]), 6)
        assert np.array_equal(got["segments"][s, :k], seg.numpy()[s, :k])
        assert (got["segments"][s, k:] == -1).all()


def test_dump_samples_the_same_streams_under_the_size_cap(tmp_path, monkeypatch):
    probs, dec, cnt, seg, n_valid = fake_step(S=40)
    per_stream = 4 * (10 + 10 + 1 + 12 + 1)
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 9 * per_stream)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), probs, dec, cnt, seg, n_valid)
    idx = np.load(tmp_path / "a" / "stream_index.npy")
    assert idx.shape == (9,) and np.array_equal(idx, np.load(tmp_path / "b" / "stream_index.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "frame_probs.npy"), probs.numpy()[idx.astype(int)])
    assert np.array_equal(np.load(tmp_path / "a" / "seg_count.npy"), cnt.numpy()[idx.astype(int)])
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 9 * per_stream + 5 * 128
