"""Argument checks of the 16-bit K3 Welford entry points (host only: every call here returns before any launch)."""
import pytest

OK, INVALID, UNSUPPORTED, WORKSPACE, ALIGNMENT = 0, -1, -2, -3, -4


@pytest.fixture(scope="module")
def lib():
    from camera_linearity_b200 import _lib, build
    build.build()
    return _lib.load(build_if_missing=False)


FAKE = 256                                  # a device address that is never dereferenced: validation fails first


def _stack(lib, frames=FAKE, f=10, n=48, c=3, lut=None, rows=0, max_dn=65535.0, mean=FAKE, sem=FAKE, mq=FAKE,
           ws=FAKE, ws_bytes=None):
    if ws_bytes is None:
        ws_bytes = lib.cl_welford_stack_workspace_bytes(f, n)
    return lib.cl_welford_stack_u16(frames, f, n, c, lut, rows, max_dn, mean, sem, mq, ws, ws_bytes, None)


def _update(lib, frames=FAKE, f=5, n=48, c=3, lut=None, rows=0, max_dn=65535.0, mean=FAKE, m2=FAKE, count0=0):
    return lib.cl_welford_update_u16(frames, f, n, c, lut, rows, max_dn, mean, m2, count0, None)


def test_symbols_and_signatures(lib):
    from camera_linearity_b200 import _lib
    for name in ("cl_welford_update_u16", "cl_welford_finalize_u16", "cl_welford_stack_u16"):
        assert name in _lib.SIGNATURES
        assert getattr(lib, name).argtypes == _lib.SIGNATURES[name][1]
    assert lib.cl_abi_version() == 1


def test_stack_frame_cap(lib):
    # the tie analysis of the 16-bit stack form holds for F <= 65536 (DESIGN.md, K3): beyond, the streaming form
    assert _stack(lib, f=65537, ws_bytes=10 ** 6) == UNSUPPORTED
    assert _stack(lib, f=65537, lut=FAKE, rows=65536, ws_bytes=10 ** 6) == UNSUPPORTED
    assert _stack(lib, n=2 ** 32, c=1, ws_bytes=2 ** 40) == UNSUPPORTED
    assert _stack(lib, f=65536, ws=FAKE + 8) == ALIGNMENT        # 65536 frames pass the cap


def test_stack_table_rows(lib):
    for rows in (0, -1, 65537):
        assert _stack(lib, lut=FAKE, rows=rows) == INVALID
    for rows in (1, 4096, 65536):
        assert _stack(lib, lut=FAKE, rows=rows, ws=FAKE + 8) == ALIGNMENT
    assert _stack(lib, lut=None, rows=-5, ws=FAKE + 8) == ALIGNMENT   # without a table the row count is ignored


def test_stack_workspace_and_alignment(lib):
    need = lib.cl_welford_stack_workspace_bytes(10, 48)
    assert need == 16 + 4 * 48                                     # the 8-bit formula suffices
    assert _stack(lib, ws_bytes=need - 1) == WORKSPACE
    assert _stack(lib, ws=None, ws_bytes=need) == WORKSPACE
    assert _stack(lib, ws=FAKE + 8) == ALIGNMENT
    assert _stack(lib, frames=FAKE + 1) == ALIGNMENT
    assert _stack(lib, mean=FAKE + 4) == ALIGNMENT
    assert _stack(lib, sem=FAKE + 4) == ALIGNMENT
    assert _stack(lib, mq=FAKE + 1) == ALIGNMENT
    assert _stack(lib, lut=FAKE + 4, rows=65536) == ALIGNMENT


def test_stack_invalid_arguments(lib):
    assert _stack(lib, n=49, c=3) == INVALID
    assert _stack(lib, c=0) == INVALID
    assert _stack(lib, n=45, c=9) == INVALID
    assert _stack(lib, f=0) == INVALID
    assert _stack(lib, n=-3) == INVALID
    assert _stack(lib, max_dn=0.0) == INVALID
    assert _stack(lib, frames=None) == INVALID
    assert lib.cl_welford_stack_u16(None, 10, 0, 3, None, 0, 65535.0, None, None, None, None, 0, None) == OK


def test_update_and_finalize_checks(lib):
    assert _update(lib, frames=None, f=0, mean=None, m2=None) == OK
    assert _update(lib, frames=None, n=0, mean=None, m2=None) == OK
    assert lib.cl_welford_finalize_u16(None, None, 5, 0, 65535.0, None, None, None) == OK
    assert _update(lib, c=0) == INVALID
    assert _update(lib, c=9) == INVALID
    assert _update(lib, n=49) == INVALID
    assert _update(lib, count0=-1) == INVALID
    assert _update(lib, max_dn=0.0) == INVALID
    assert _update(lib, f=-1) == INVALID
    for rows in (0, 65537):
        assert _update(lib, lut=FAKE, rows=rows) == INVALID
    for null in ("frames", "mean", "m2"):
        assert _update(lib, **{null: None}) == INVALID
    assert _update(lib, frames=FAKE + 1) == ALIGNMENT
    assert _update(lib, mean=FAKE + 4) == ALIGNMENT
    assert _update(lib, m2=FAKE + 4) == ALIGNMENT
    assert _update(lib, lut=FAKE + 4, rows=4096) == ALIGNMENT
    assert lib.cl_welford_finalize_u16(None, FAKE, 5, 48, 65535.0, FAKE, FAKE, None) == INVALID
    assert lib.cl_welford_finalize_u16(FAKE, FAKE, -1, 48, 65535.0, FAKE, FAKE, None) == INVALID
    assert lib.cl_welford_finalize_u16(FAKE, FAKE, 5, -1, 65535.0, FAKE, FAKE, None) == INVALID
    assert lib.cl_welford_finalize_u16(FAKE, FAKE, 5, 48, 65535.0, FAKE, FAKE + 1, None) == ALIGNMENT
    assert lib.cl_welford_finalize_u16(FAKE + 4, FAKE, 5, 48, 65535.0, FAKE, FAKE, None) == ALIGNMENT
