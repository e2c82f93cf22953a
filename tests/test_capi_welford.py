"""Argument checks of the K3 Welford entry points (host only: every call here returns before any launch)."""
import pytest

OK, INVALID, UNSUPPORTED, WORKSPACE, ALIGNMENT = 0, -1, -2, -3, -4


@pytest.fixture(scope="module")
def lib():
    from camera_linearity_b200 import _lib, build
    build.build()
    return _lib.load(build_if_missing=False)


FAKE = 256                                  # a device address that is never dereferenced: validation fails first


def _stack(lib, frames=FAKE, f=10, n=48, c=3, lut=None, max_dn=255.0, ws=FAKE, ws_bytes=None):
    if ws_bytes is None:
        ws_bytes = lib.cl_welford_stack_workspace_bytes(f, n)
    return lib.cl_welford_stack(frames, f, n, c, lut, max_dn, FAKE, FAKE, FAKE, ws, ws_bytes, None)


def test_stack_workspace_bytes_formula(lib):
    # a 16-byte header (the tie counter) + one uint32 index per sample: every sample can be a rounding tie
    for f, n in ((1, 0), (600, 1), (600, 6220800), (10 ** 6, 2 ** 32 - 1), (3, 48)):
        assert lib.cl_welford_stack_workspace_bytes(f, n) == 16 + 4 * n
    assert lib.cl_welford_stack_workspace_bytes(10, -5) == 16


def test_stack_rejects_unsupported_sizes(lib):
    # the tie analysis holds for F <= 10^6, and the tie list stores 32-bit sample indices
    assert _stack(lib, f=10 ** 6 + 1) == UNSUPPORTED
    assert _stack(lib, f=10 ** 6 + 1, lut=FAKE) == UNSUPPORTED
    assert _stack(lib, n=2 ** 32, c=1) == UNSUPPORTED
    assert _stack(lib, n=3 * 2 ** 31, c=3) == UNSUPPORTED


def test_stack_rejects_a_short_or_misaligned_workspace(lib):
    need = lib.cl_welford_stack_workspace_bytes(10, 48)
    assert _stack(lib, ws_bytes=need - 1) == WORKSPACE
    assert _stack(lib, ws=None, ws_bytes=need) == WORKSPACE
    assert _stack(lib, ws=FAKE + 8, ws_bytes=need) == ALIGNMENT
    assert _stack(lib, ws=FAKE + 8, ws_bytes=need, lut=FAKE) == ALIGNMENT


def test_stack_rejects_invalid_arguments(lib):
    assert _stack(lib, n=49, c=3) == INVALID            # n % C != 0
    assert _stack(lib, c=0) == INVALID
    assert _stack(lib, n=45, c=9) == INVALID            # more than CL_MAX_CHANNELS
    assert _stack(lib, f=0) == INVALID
    assert _stack(lib, f=-1) == INVALID
    assert _stack(lib, n=-3) == INVALID
    assert _stack(lib, max_dn=0.0) == INVALID
    assert _stack(lib, frames=None) == INVALID
    # an empty image is a successful no-op, whatever the pointers
    assert lib.cl_welford_stack(None, 10, 0, 3, None, 255.0, None, None, None, None, 0, None) == OK


def test_update_and_finalize_checks(lib):
    # nothing to do: success without touching (null) pointers
    assert lib.cl_welford_update(None, 0, 48, 3, None, 255.0, None, None, 0, None) == OK
    assert lib.cl_welford_update(None, 5, 0, 3, None, 255.0, None, None, 7, None) == OK
    assert lib.cl_welford_finalize(None, None, 5, 0, 255.0, None, None, None) == OK
    # invalid arguments
    assert lib.cl_welford_update(FAKE, 5, 48, 0, None, 255.0, FAKE, FAKE, 0, None) == INVALID
    assert lib.cl_welford_update(FAKE, 5, 48, 9, None, 255.0, FAKE, FAKE, 0, None) == INVALID
    assert lib.cl_welford_update(FAKE, 5, 49, 3, None, 255.0, FAKE, FAKE, 0, None) == INVALID
    assert lib.cl_welford_update(FAKE, 5, 48, 3, None, 255.0, FAKE, FAKE, -1, None) == INVALID
    assert lib.cl_welford_update(FAKE, 5, 48, 3, None, 0.0, FAKE, FAKE, 0, None) == INVALID
    assert lib.cl_welford_update(FAKE, -1, 48, 3, None, 255.0, FAKE, FAKE, 0, None) == INVALID
    for null in range(3):
        p = [FAKE, FAKE, FAKE]
        p[null] = None
        assert lib.cl_welford_update(p[0], 5, 48, 3, None, 255.0, p[1], p[2], 0, None) == INVALID
    assert lib.cl_welford_finalize(None, FAKE, 5, 48, 255.0, FAKE, FAKE, None) == INVALID
    assert lib.cl_welford_finalize(FAKE, FAKE, -1, 48, 255.0, FAKE, FAKE, None) == INVALID
    assert lib.cl_welford_finalize(FAKE, FAKE, 5, -1, 255.0, FAKE, FAKE, None) == INVALID
