"""Argument checks of the 16-bit K4 entry points (host only: every call here fails before any launch)."""
import ctypes

import pytest

from camera_linearity_b200._lib import IcrfProblem, PeerGroup

INVALID = -1


@pytest.fixture(scope="module")
def lib():
    from camera_linearity_b200 import _lib, build
    build.build()
    return _lib.load(build_if_missing=False)


def _prob(datapoints, s=64):
    return IcrfProblem(s, 5, datapoints, 1, 1, datapoints - 1, 5, 0)


def test_tables_bytes_up_to_65536_points(lib):
    assert lib.cl_icrf_tables_bytes(ctypes.byref(_prob(65536))) == 2 * 64 * 65536 * 8
    assert lib.cl_icrf_tables_bytes(ctypes.byref(_prob(4096, 32))) == 2 * 32 * 4096 * 8
    assert lib.cl_icrf_tables_bytes(ctypes.byref(_prob(65537))) == 0
    assert lib.cl_icrf_energy_workspace_bytes(ctypes.byref(_prob(65536)), 400000) > 0
    assert lib.cl_icrf_energy_workspace_bytes(ctypes.byref(_prob(65537)), 400000) == 0
    # the exchange buffer depends on neither the curve length nor the sample type
    assert (lib.cl_icrf_exchange_bytes(ctypes.byref(_prob(65536)), 2)
            == lib.cl_icrf_exchange_bytes(ctypes.byref(_prob(256)), 2) > 0)


def test_u16_entry_points_reject_null_pointers_and_bad_lengths(lib):
    t = (ctypes.c_double * 5)(*[0.01, 0.02, 0.04, 0.08, 0.16])
    fake = ctypes.c_void_p(256)                  # never dereferenced: validation fails first
    peers = PeerGroup()
    peers.world, peers.rank = 1, 0
    peers.buffers[0] = 256
    for d in (1, 65537):
        p = _prob(max(d, 2))
        p.datapoints = d
        assert lib.cl_icrf_energy_partial_u16(ctypes.byref(p), fake, fake, None, t, 10, fake, fake, 1 << 20,
                                              None) == INVALID
        assert lib.cl_icrf_energy_population_u16(ctypes.byref(p), fake, fake, None, t, 10, fake, fake, fake, fake,
                                                 1 << 20, ctypes.byref(peers), None, None) == INVALID
        assert lib.cl_icrf_curves(ctypes.byref(p), fake, fake, fake, fake, fake, fake, None) == INVALID
    p = _prob(65536)
    assert lib.cl_icrf_energy_partial_u16(ctypes.byref(p), None, fake, None, t, 10, fake, fake, 1 << 20,
                                          None) == INVALID
    assert lib.cl_icrf_energy_partial_u16(ctypes.byref(p), fake, None, None, t, 10, fake, fake, 1 << 20,
                                          None) == INVALID
    assert lib.cl_icrf_energy_population_u16(ctypes.byref(p), fake, None, None, t, 10, fake, fake, fake, fake,
                                             1 << 20, ctypes.byref(peers), None, None) == INVALID
    assert lib.cl_icrf_energy_population_u16(ctypes.byref(p), fake, fake, None, t, 10, fake, fake, fake, fake,
                                             1 << 20, None, None, None) == INVALID
    assert lib.cl_icrf_curves(ctypes.byref(p), fake, None, fake, fake, fake, fake, None) == INVALID


def test_uint8_entry_points_still_stop_at_256_points(lib):
    t = (ctypes.c_double * 5)(*[0.01, 0.02, 0.04, 0.08, 0.16])
    fake = ctypes.c_void_p(256)
    peers = PeerGroup()
    peers.world, peers.rank = 1, 0
    peers.buffers[0] = 256
    p = _prob(257)
    assert lib.cl_icrf_energy_partial(ctypes.byref(p), fake, fake, None, t, 10, fake, fake, 1 << 20, None) == INVALID
    assert lib.cl_icrf_energy_population(ctypes.byref(p), fake, fake, None, t, 10, fake, fake, fake, fake, 1 << 20,
                                         ctypes.byref(peers), None, None) == INVALID
    assert lib.cl_abi_version() == 1
