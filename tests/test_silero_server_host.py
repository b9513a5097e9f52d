"""Host-side checks of the Silero slot server's C entry points: the scratch-size query and the argument validation need
no device."""
import ctypes as C

from vadx import lib


def _step(n_slots, W, scratch=None, need=None, ld=None, events=None):
    return lib.load().vadx_silero_serve_step(None, n_slots if ld is None else ld, None, None, n_slots, W, 0.5, 1600.0,
                                             None, None, None, None, None, events, None, None, None, scratch, 0,
                                             C.byref(need) if need is not None else None, None)


def test_scratch_size_query_grows_with_slots_and_windows():
    a, b, c = C.c_size_t(), C.c_size_t(), C.c_size_t()
    assert _step(64, 5, need=a) == 0
    assert _step(128, 5, need=b) == 0
    assert _step(64, 11, need=c) == 0
    # staged events (W + 1 int32 pairs per slot) dominate
    assert a.value >= 64 * 6 * 8 and b.value > a.value and c.value > a.value


def test_bad_shapes_are_rejected():
    n = C.c_size_t()
    l = lib.load()
    assert _step(0, 5, need=n) == -1
    assert b"bad shape" in l.vadx_last_error()
    assert _step(4, 0, need=n) == -1
    assert _step(4, 5, scratch=1, need=n) == -1              # scratch too small
    assert b"scratch" in l.vadx_last_error()
    assert l.vadx_silero_serve_load(1, 1, 0, 5, 1, None) == -1
    assert l.vadx_silero_serve_load(1, 1, 4, 0, 1, None) == -1
    assert b"bad shape" in l.vadx_last_error()


def test_null_pointers_are_rejected():
    n = C.c_size_t()
    assert _step(4, 5, need=n) == 0
    l = lib.load()
    # a scratch buffer of the queried size, but no probabilities, control words or outputs
    assert l.vadx_silero_serve_step(None, 4, None, None, 4, 5, 0.5, 1600.0, None, None, None, None, None, None, None,
                                    None, None, 1, n.value, None, None) == -1
    assert b"null pointer" in l.vadx_last_error()
    for args in ((None, 1, 4, 5, 1), (1, None, 4, 5, 1), (1, 1, 4, 5, None)):
        assert l.vadx_silero_serve_load(*args, None) == -1
        assert b"null pointer" in l.vadx_last_error()


def test_misaligned_vector_buffers_are_rejected():
    """the load kernel and the context roll move 16-byte vectors: an offset pointer is an argument error"""
    l = lib.load()
    assert l.vadx_silero_serve_load(18, 16, 4, 5, 16, None) == -1
    assert b"16-byte aligned" in l.vadx_last_error()
    assert l.vadx_silero_serve_load(16, 16, 4, 5, 20, None) == -1
    n = C.c_size_t()
    assert _step(4, 5, need=n) == 0
    assert l.vadx_silero_serve_step(16, 4, 16, 16, 4, 5, 0.5, 1600.0, 16, 20, None, None, 16, 16, 16, None, None, 16,
                                    n.value, None, None) == -1
    assert b"d_x must be 16-byte aligned" in l.vadx_last_error()
