"""Host-side checks of the FSMN slot server's C entry points: the scratch-size query and the argument validation need
no device."""
import ctypes as C

from vadx import lib

CFG = lib.FsmnServeCfg(0.5, 0.5, 0.01, 0.3, 0.2, 1.0, 4.0)


def _step(n_slots, T, L=16000, stride=11040, lb=30, scratch=None, need=None, size=0):
    return lib.load().vadx_fsmn_serve_step(None, T, None, T, None, None, n_slots, L, stride, lb, C.byref(CFG), None, None,
                                           None, 0, 0, None, None, None, None, None, scratch, size,
                                           C.byref(need) if need is not None else None, None)


def _load(chunk, n, last, state, S, window, noise, L=16000, stride=11040, lb=30):
    return lib.load().vadx_fsmn_serve_load(chunk, n, last, state, S, L, stride, lb, 4.0, window, noise, None)


def test_state_words_hold_the_look_ahead_flags():
    l = lib.load()
    assert l.vadx_fsmn_serve_state_words(0) == 8
    assert l.vadx_fsmn_serve_state_words(30) == 9
    assert l.vadx_fsmn_serve_state_words(33) == 10


def test_scratch_size_query_grows_with_slots_and_frames():
    a, b, c = C.c_size_t(), C.c_size_t(), C.c_size_t()
    assert _step(64, 101, need=a) == 0
    assert _step(128, 101, need=b) == 0
    assert _step(64, 4, L=512, stride=352, lb=0, need=c) == 0
    # staged events (2T + 2 int32 pairs per slot) dominate
    assert a.value >= 64 * 204 * 8 and b.value > a.value and c.value < a.value


def test_bad_shapes_are_rejected():
    n = C.c_size_t()
    l = lib.load()
    assert _step(0, 101, need=n) == -1
    assert b"bad shape" in l.vadx_last_error()
    assert _step(4, 101, stride=0, need=n) == -1                 # stride <= 0
    assert _step(4, 101, stride=16000, need=n) == -1
    assert _step(4, 101, lb=101, need=n) == -1                   # look_backward must leave decisions per window
    assert b"bad shape" in l.vadx_last_error()
    assert _step(4, 101, need=n) == 0
    assert _step(4, 101, scratch=1, need=n, size=8) == -1       # scratch too small
    assert b"scratch" in l.vadx_last_error()
    assert _load(16, 16, 16, 16, 0, 16, 16) == -1               # n_slots = 0
    assert _load(16, 16, 16, 16, 4, 16, 16, stride=0) == -1      # stride <= 0
    assert _load(16, 16, 16, 16, 4, 16, 16, L=16004, stride=11044) == -1   # chunk_len % 8 != 0
    assert b"bad shape" in l.vadx_last_error()


def test_null_pointers_are_rejected():
    n = C.c_size_t()
    assert _step(4, 101, need=n) == 0
    l = lib.load()
    # a scratch buffer of the queried size, but no scores, control words or outputs
    assert _step(4, 101, scratch=16, size=n.value) == -1
    assert b"null pointer" in l.vadx_last_error()
    for i in range(4):
        args = [16, 16, 16, 16]
        args[i] = None
        assert _load(*args, 4, 16, 16) == -1
        assert b"null pointer" in l.vadx_last_error()
    assert _load(16, 16, 16, 16, 4, None, 16) == -1
    assert _load(16, 16, 16, 16, 4, 16, None) == -1
    assert b"null pointer" in l.vadx_last_error()


def test_misaligned_vector_buffers_are_rejected():
    """the load kernel moves 16-byte vectors: an offset chunk or window pointer is an argument error"""
    l = lib.load()
    assert _load(18, 16, 16, 16, 4, 16, 16) == -1
    assert b"16-byte aligned" in l.vadx_last_error()
    assert _load(16, 16, 16, 16, 4, 24, 16) == -1
    assert b"16-byte aligned" in l.vadx_last_error()
