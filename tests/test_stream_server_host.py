"""Host-side checks of the slot server's C entry points: the scratch-size query and the argument validation need no
device."""
import ctypes as C

from vadx import lib


def _step(n_slots, n_frames, chunk, scratch=None, need=None):
    cfg = lib.StreamPostCfg(5, 0.4, 5, 8, 2000, 20)
    return lib.load().vadx_stream_serve_step(None, n_frames, n_frames, None, None, n_slots, chunk, 400, 160,
                                             C.byref(cfg), None, None, None, 0, 0, None, None, None, None, None, scratch,
                                             0, C.byref(need) if need is not None else None, None)


def test_scratch_size_query_grows_with_slots_and_frames():
    a, b, c = C.c_size_t(), C.c_size_t(), C.c_size_t()
    assert _step(64, 14, 2560, need=a) == 0
    assert _step(128, 14, 2560, need=b) == 0
    assert _step(64, 28, 400 + 160 * 27, need=c) == 0
    # staged events (2T+1 int32 pairs per slot) dominate
    assert a.value >= 64 * 29 * 8 and b.value > a.value and c.value > a.value


def test_bad_shapes_are_rejected():
    n = C.c_size_t()
    assert _step(0, 14, 2560, need=n) == -1
    assert _step(4, 13, 2560, need=n) == -1                  # a full chunk gives 14 frames
    assert b"probs hold 13" in lib.load().vadx_last_error()
    assert _step(4, 14, 399, need=n) == -1                   # shorter than one frame
    assert _step(4, 14, 2560, scratch=1, need=n) == -1       # scratch too small
    l = lib.load()
    assert l.vadx_stream_serve_zero_tail(None, 2560, None, 4, 2560, 400, None) == -1
    assert b"null pointer" in l.vadx_last_error()
