"""Host side of the 64-channel-block BDC entries (csrc/bdc_wide.cu): the workspace arithmetic and the argument
refusals, all decided before any CUDA call, so no GPU is needed."""
import ctypes

import pytest

OK, INVALID, UNSUPPORTED, WORKSPACE = 0, -1, -2, -4


def _a4(n):
    return (n + 3) // 4 * 4


def _ws_floats(B, C, backward):
    k = C // 64
    P = k * (k + 1) // 2
    n = _a4(B * C) + _a4(B * k * C)                      # norms, per-tile row sums
    if backward:
        n += 2 * _a4(B * C) + _a4(B) + B * P * 4096 + _a4(B * P)  # dB row / column sums, total, S tiles, dt partials
    return n


@pytest.fixture(scope="module")
def h():
    from audio_fewshot_b200 import _lib
    return _lib.lib()


@pytest.mark.parametrize("C", list(range(128, 641, 64)))
@pytest.mark.parametrize("B", [0, 1, 3, 75, 2400, 10500, 70000])
def test_workspace_bytes(h, B, C):
    for backward in (0, 1):
        assert h.afs_bdc_wide_workspace_bytes(B, C, backward) == 4 * _ws_floats(B, C, backward)


def test_workspace_bytes_are_64_bit(h):
    n = 4 * _ws_floats(2 ** 31 - 1, 640, 1)
    assert n > 2 ** 50 and h.afs_bdc_wide_workspace_bytes(2 ** 31 - 1, 640, 1) == n


@pytest.mark.parametrize("C", [-64, 0, 1, 17, 63, 64, 65, 96, 127, 129, 700, 704, 1024])
def test_workspace_bytes_is_zero_for_unsupported_channel_counts(h, C):
    assert h.afs_bdc_wide_workspace_bytes(5, C, 0) == 0
    assert h.afs_bdc_wide_workspace_bytes(5, C, 1) == 0
    assert h.afs_bdc_wide_workspace_bytes(-1, 128, 0) == 0


def _fwd(h, x, B, C, M, t, out, ws, nbytes):
    return h.afs_bdc_wide_fwd(x, B, C, M, t, 1, out, ws, nbytes, None)


def _bwd(h, x, B, C, M, t, g, gx, gt, ws, nbytes):
    return h.afs_bdc_wide_bwd(x, B, C, M, t, 1, g, gx, gt, ws, nbytes, None)


def test_argument_refusals_before_any_cuda_call(h):
    """Pointers below are never dereferenced: every call is refused (or is a no-op) on the host."""
    p = ctypes.c_void_p(4096)  # a fake, 16-byte aligned address
    need_f = h.afs_bdc_wide_workspace_bytes(2, 128, 0)
    need_b = h.afs_bdc_wide_workspace_bytes(2, 128, 1)
    # null pointers
    for args in ((None, p, p), (p, None, p), (p, p, None)):
        x, t, out = args
        assert _fwd(h, x, 2, 128, 8, t, out, p, need_f) == INVALID
    for i in range(5):
        ptrs = [p] * 5
        ptrs[i] = None
        x, t, g, gx, gt = ptrs
        assert _bwd(h, x, 2, 128, 8, t, g, gx, gt, p, need_b) == INVALID
    # bad sizes
    for B, C, M in ((-1, 128, 8), (2, 128, 0), (2, 0, 8)):
        assert _fwd(h, p, B, C, M, p, p, p, need_f) == INVALID
        assert _bwd(h, p, B, C, M, p, p, p, p, p, need_b) == INVALID
    # channel counts outside 128, 192, ..., 640
    for C in (64, 65, 96, 127, 704, 1024):
        assert _fwd(h, p, 2, C, 8, p, p, p, need_f) == UNSUPPORTED
        assert _bwd(h, p, 2, C, 8, p, p, p, p, p, need_b) == UNSUPPORTED
    # B = 0 is a no-op, whatever the pointers
    assert _fwd(h, None, 0, 640, 8, None, None, None, 0) == OK
    assert _bwd(h, None, 0, 640, 8, None, None, None, None, None, 0) == OK
    # workspace: missing, one byte short, misaligned
    assert _fwd(h, p, 2, 128, 8, p, p, None, need_f) == WORKSPACE
    assert _fwd(h, p, 2, 128, 8, p, p, p, need_f - 1) == WORKSPACE
    assert _fwd(h, p, 2, 128, 8, p, p, ctypes.c_void_p(4100), need_f) == WORKSPACE
    assert _bwd(h, p, 2, 128, 8, p, p, p, p, None, need_b) == WORKSPACE
    assert _bwd(h, p, 2, 128, 8, p, p, p, p, p, need_b - 1) == WORKSPACE
    assert _bwd(h, p, 2, 128, 8, p, p, p, p, ctypes.c_void_p(4104), need_b) == WORKSPACE
    # the backward needs more than the forward
    assert _bwd(h, p, 2, 128, 8, p, p, p, p, p, need_f) == WORKSPACE
