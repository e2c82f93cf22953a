"""Argument checks of cl_pair_statistics (host only: every call here returns before any launch)."""
import ctypes as C

import pytest

OK, INVALID, UNSUPPORTED, WORKSPACE, ALIGNMENT = 0, -1, -2, -3, -4
BLOCKS, NQ = 296, 14                # linearity.cu kBlocks, kQ: the block partials the final kernel sums


@pytest.fixture(scope="module")
def lib():
    from camera_linearity_b200 import _lib, build
    build.build()
    return _lib.load(build_if_missing=False)


FAKE = 256                                  # a device address that is never dereferenced: validation fails first


def _limits(c, value):
    return (C.c_double * c)(*([value] * c))


def _call(lib, x=FAKE, xs=FAKE, y=FAKE, ys=FAKE, lower=None, upper=None, n=48, c=3, stats=FAKE, ws=FAKE,
          ws_bytes=None):
    if ws_bytes is None:
        ws_bytes = lib.cl_pair_statistics_workspace_bytes(c)
    return lib.cl_pair_statistics(x, xs, y, ys, 0.5, lower, upper, n, c, stats, ws, ws_bytes, None)


def test_workspace_bytes_formula(lib):
    # 296 block partials of 14 sums per channel, then the two shifts K (absolute, relative) per channel
    for c in range(1, 9):
        assert lib.cl_pair_statistics_workspace_bytes(c) == (BLOCKS * NQ * c + 2 * c) * 8
    for c in (0, -1):
        assert lib.cl_pair_statistics_workspace_bytes(c) == (BLOCKS * NQ + 2) * 8


def test_rejects_invalid_arguments(lib):
    assert _call(lib, c=0, n=48) == INVALID
    assert _call(lib, c=9, n=45) == INVALID               # more than CL_MAX_CHANNELS
    assert _call(lib, c=3, n=49) == INVALID               # n % C != 0
    assert _call(lib, n=-3) == INVALID
    assert _call(lib, lower=_limits(3, 0.1)) == INVALID   # lower without upper
    assert _call(lib, upper=_limits(3, 0.9)) == INVALID   # upper without lower
    assert _call(lib, x=None) == INVALID
    assert _call(lib, y=None) == INVALID
    assert _call(lib, stats=None) == INVALID


def test_rejects_a_missing_or_short_workspace(lib):
    for c in (1, 3, 8):
        need = lib.cl_pair_statistics_workspace_bytes(c)
        assert _call(lib, c=c, n=8 * c, ws_bytes=need - 1) == WORKSPACE
        assert _call(lib, c=c, n=8 * c, ws=None, ws_bytes=need) == WORKSPACE
        assert _call(lib, c=c, n=8 * c, ws=None, ws_bytes=0) == WORKSPACE
    # argument errors are reported before the workspace
    assert _call(lib, c=9, n=45, ws=None) == INVALID


def test_empty_image_is_checked_like_any_other(lib):
    # n = 0 has no early return: pointers, limits and workspace are checked as for any n (and, on a device, both
    # kernels run and every output is NaN: test_gpu_pair_statistics_paths.py::test_empty_image)
    assert _call(lib, n=0, x=None) == INVALID
    assert _call(lib, n=0, stats=None) == INVALID
    assert _call(lib, n=0, lower=_limits(3, 0.1)) == INVALID
    assert _call(lib, n=0, ws=None) == WORKSPACE
