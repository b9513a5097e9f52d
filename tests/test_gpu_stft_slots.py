"""The tensor-core STFT's hop-row layout: every 128-slot tile holds its frames' hop rows once (T + Q - 1 slots per stream),
and frame t reads hop rows t .. t + Q - 1 as shifted operand rows.  Checked against a float64 framed DFT of the
pre-emphasised int16 signal at stream counts and lengths that put the stream boundaries, the halo slots and the last
partial tile everywhere a tile can have them."""
import numpy as np
import pytest
import torch

import vadx
from vadx import lib, synth, tables, weights as W

pytestmark = pytest.mark.gpu


def _ref_power(x, basis, nb, hop, pad_left, T, preemph=0.97):
    """float64 |DFT|^2 of the frames of y = x[i] - c x[i-1] (x[-1] = 0), zero outside [0, L)."""
    S, L = x.shape
    n_taps = basis.shape[0]
    xd = x.astype(np.float64)
    y = xd.copy()
    y[:, 1:] -= preemph * xd[:, :-1]
    span = (T - 1) * hop + n_taps
    yp = np.zeros((S, pad_left + max(L, span)), np.float64)
    yp[:, pad_left:pad_left + L] = y
    idx = np.arange(T)[:, None] * hop + np.arange(n_taps)[None, :]
    frames = yp[:, idx].reshape(S * T, n_taps)
    c = frames @ basis[:, :2 * nb].astype(np.float64)
    return c[:, 0::2] ** 2 + c[:, 1::2] ** 2


def _run_tc(cuda, x, basis, nb, hop, pad_left, T, fmt, ld=None):
    l = lib.load()
    S, L = x.shape
    n_taps = basis.shape[0]
    ld = ld or (nb + 3) // 4 * 4
    img = torch.from_numpy(lib.pack_stft_basis_tc(basis, nb, 0.97, 1.0, fmt)).to(cuda)
    xd = torch.from_numpy(x).to(cuda)
    out = torch.full((S * T, ld), float("nan"), device=cuda)
    tab, lo, hi = None, 0, T
    if pad_left > 0 or (T - 1) * hop - pad_left + n_taps > L:
        t, lo, hi = lib.pack_stft_dc_tc(basis, nb, 0.97, 1.0, L, hop, pad_left, T)
        tab = torch.from_numpy(t).to(cuda)
    lib.check(l.vadx_stft_power_tc_i16_ex(xd.data_ptr(), L, L, S, T, hop, n_taps, img.data_ptr(), nb, out.data_ptr(), ld,
                                          pad_left, None, None, lib.ptr(tab), lo, hi, 1.0, fmt, lib.stream_ptr()))
    torch.cuda.synchronize()
    return out[:, :nb].cpu().double().numpy()


def _check(got, ref, what):
    assert not np.isnan(got).any(), what
    rel = (np.abs(got - ref) / np.maximum(ref.max(axis=1, keepdims=True), 1e-30)).max()
    print(f"{what}: max err relative to the frame's strongest bin {rel:.2e}")
    # the same bound as the frame-per-row layout: fp32 TMEM accumulation over ~50 products per output
    assert rel <= 3e-5, (what, rel)


@pytest.mark.parametrize("S,T,fmt", [
    (128, 97, lib.TC_FMT_BF16),   # 99 slots per stream (odd): stream boundaries at all 128 phases of a tile, many tiles per CTA
    (5, 98, lib.TC_FMT_F16),      # the FireRed chunk: 500 slots, last tile partial (116 slots)
    (3, 8, lib.TC_FMT_BF16),      # T + Q - 1 = 10 slots: several streams inside one (partial) tile
    (2, 300, lib.TC_FMT_F16),     # one stream spans more than two tiles
    (1, 126, lib.TC_FMT_BF16),    # exactly one tile of slots, halo slots at its end
])
def test_stft_tc_slots_frames_inside(cuda, S, T, fmt):
    basis, first, nb = tables.interleaved_basis(400, 400, "povey", "v2")
    L = 400 + 160 * (T - 1)
    x = synth.synth_streams(S, L, seed=S * 1000 + T)
    got = _run_tc(cuda, x, basis, nb, 160, 0, T, fmt)
    _check(got, _ref_power(x, basis, nb, 160, 0, T), f"S={S} T={T} fmt={fmt}")


@pytest.mark.parametrize("hop", [16, 128, 240])
def test_stft_tc_slots_other_hops(cuda, hop):
    """hop = 16: a frame spans 26 hop rows (the widest halo); 128: Q = 4; 240 = 15 K16 columns, so the last ring stage of
    every tile is half full."""
    basis, first, nb = tables.interleaved_basis(400, 400, "povey", "v2")
    S, T = 7, 61
    L = (T - 1) * hop + 400
    L += (-L) % 8
    x = synth.synth_streams(S, L, seed=hop)
    got = _run_tc(cuda, x, basis, nb, hop, 0, T, lib.TC_FMT_BF16)
    _check(got, _ref_power(x, basis, nb, hop, 0, T), f"hop={hop}")


@pytest.mark.parametrize("S,L", [(9, 512), (37, 4800), (2, 16000)])
def test_stft_tc_slots_centre_padded(cuda, S, L):
    """Centre-padded frames (n_fft = 512, 400 taps): the first frames start in the zero pad, the last ones run past the end
    of the stream (L = 512: every frame but one does), and the hop rows behind a stream are zero beyond L."""
    basis, first, nb = tables.interleaved_basis(512, 400, "hann", "v2")
    pad_left = 256 - first
    T = L // 160 + 1
    x = synth.synth_streams(S, L, seed=S + L)
    got = _run_tc(cuda, x, basis, nb, 160, pad_left, T, lib.TC_FMT_F16, ld=260)
    _check(got, _ref_power(x, basis, nb, 160, pad_left, T), f"centre-padded S={S} L={L}")


def test_stft_tc_rejects_hop_not_multiple_of_16(cuda):
    basis, first, nb = tables.interleaved_basis(400, 400, "povey", "v2")
    x = synth.synth_streams(2, 16000, seed=3)
    T = 1 + (16000 - 400) // 168
    with pytest.raises(ValueError, match="multiple of 16"):
        _run_tc(cuda, x, basis, nb, 168, 0, T, lib.TC_FMT_BF16)


def test_firered_hop_168_runs_the_fp32_stft(cuda):
    """A FireRed config whose hop the tensor-core STFT cannot read as 16-sample slices takes the fp32 framed DFT."""
    from oracle.firered import FireRedOracle
    cfg = W.FireRedConfig(hop=168)
    w = W.firered_random_init(cfg, 0)
    chunks = synth.synth_chunks_fast(200, 16000, seed=5)
    d = torch.from_numpy(chunks).to(cuda)
    sess = vadx.FireRedSession(w, cfg, tensor_cores=True)
    lib.profile_enable(True)
    lib.profile_collect_kernels()
    p = sess.run_batch(d).cpu().numpy()
    k = lib.profile_collect_kernels()
    lib.profile_enable(False)
    assert "stft_power_tc_kernel" not in k and "gemm_f32_kernel(stft_power)" in k, sorted(k)
    ref = FireRedOracle(w, cfg).forward(chunks).numpy()
    assert p.shape == ref.shape
    assert np.abs(p - ref).max() <= 3e-4
