"""Host-side checks of the MarbleNet slot server's C entry points: the state-words and scratch-size queries and the
argument validation need no device."""
import ctypes as C

from vadx import lib, marblenet_vad as MV

CFG = MV.POST_DEFAULT.c_struct()


def _step(n_slots, F, L=16000, cfg=CFG, probs=None, scratch=None, need=None, size=0, ld=None):
    return lib.load().vadx_marblenet_serve_step(probs, F if ld is None else ld, F, None, None, n_slots, L, C.byref(cfg),
                                                0.02, None, None, None, None, None, None, scratch, size,
                                                C.byref(need) if need is not None else None, None)


def test_state_words_hold_the_delay_lines():
    l = lib.load()
    # 16 header words, the running-sum ring (3), the probability ring (D + 1 = 16: D = 10 + 3 + 2 + 0) and three bit rings
    assert l.vadx_marblenet_serve_state_words(C.byref(CFG)) == 16 + 3 + 16 + 3
    plain = lib.PostCfg(1, 0.5, 0, 1000, 0, 0, 0)
    assert l.vadx_marblenet_serve_state_words(C.byref(plain)) == 16 + 1 + 3
    wide = lib.PostCfg(64, 0.4, 30, 500, 30, 5, 0)                  # D = 30 + 64 + 4 = 98
    assert l.vadx_marblenet_serve_state_words(C.byref(wide)) == 16 + 64 + 99 + 1 + 3 + 1
    huge = lib.PostCfg(3, 0.5, 1 << 20, 1000, 10, 3, 0)
    assert l.vadx_marblenet_serve_state_words(C.byref(huge)) == -1
    assert b"delay" in l.vadx_last_error()


def test_scratch_size_query_grows_with_slots_and_frames():
    a, b, c = C.c_size_t(), C.c_size_t(), C.c_size_t()
    assert _step(64, 50, need=a) == 0
    assert _step(128, 50, need=b) == 0
    assert _step(64, 100, L=32000, need=c) == 0
    # staged events (2 (F + D) + 2 int32 pairs per slot, D = 15) dominate
    assert a.value >= 64 * (2 * (50 + 15) + 2) * 8 and b.value > a.value and c.value > a.value


def test_bad_shapes_are_rejected():
    n = C.c_size_t()
    l = lib.load()
    assert _step(0, 50, need=n) == -1
    assert b"bad shape" in l.vadx_last_error()
    assert _step(4, 0, need=n) == -1
    assert _step(4, 50, L=0, need=n) == -1
    assert b"bad shape" in l.vadx_last_error()
    assert _step(4, 50, cfg=lib.PostCfg(3, 0.5, 1 << 20, 1000, 10, 3, 0), need=n) == -1
    assert b"delay" in l.vadx_last_error()
    assert _step(4, 50, need=n) == 0
    assert _step(4, 50, scratch=1, need=n, size=8) == -1       # scratch too small
    assert b"scratch" in l.vadx_last_error()
    assert _step(4, 50, probs=16, scratch=16, size=n.value, ld=49) == -1
    assert b"null pointer" in l.vadx_last_error() or b"ld_probs" in l.vadx_last_error()


def test_null_pointers_are_rejected():
    n = C.c_size_t()
    assert _step(4, 50, need=n) == 0
    l = lib.load()
    # a scratch buffer of the queried size, but no probabilities, control words or outputs
    assert _step(4, 50, scratch=16, size=n.value) == -1
    assert b"null pointer" in l.vadx_last_error()
    assert l.vadx_marblenet_serve_state_words(None) == -1
    assert b"null pointer" in l.vadx_last_error()
