"""Argument checks of cl_hdr_merge and its workspace size (host only: every call here returns before any launch)."""
import ctypes as C
import math

import pytest

OK, INVALID, UNSUPPORTED, WORKSPACE, ALIGNMENT = 0, -1, -2, -3, -4
TILE_SAMPLES = 512 * 3              # samples of one 512-pixel tile of the tile kernels (hdr_merge.cuh kStagedTilePx)
BUCKET_CAP, HOT_HEADER = 32, 4      # hdr_merge.cuh kBucketCap, kHotListHeader

FAKE = 256                          # a device address that is never dereferenced: validation fails first


@pytest.fixture(scope="module")
def lib():
    from camera_linearity_b200 import _lib, build
    build.build()
    return _lib.load(build_if_missing=False)


def _args(n=4, h=16, w=32, c=3, dn_bytes=1, t=None, std=True, std_lut=False, dark=False, scale=None, K=3,
          flat_bytes=0, algo=0):
    from camera_linearity_b200 import _lib
    a = _lib.HdrMergeArgs()
    a.n_exposures, a.height, a.width, a.channels, a.dn_bytes = n, h, w, c, dn_bytes
    a.bits = 256 if dn_bytes == 1 else 65536
    m = max(n, 1)
    keep = [(C.c_void_p * m)(*([FAKE] * m)),
            (C.c_void_p * m)(*([FAKE if std else None] * m)),
            (C.c_double * m)(*(t if t is not None else [0.01 * (k + 1) for k in range(m)])),
            (C.c_void_p * m)(*([FAKE] * m)),
            (C.c_double * m)(*([1.0] * m if scale is None else scale))]
    a.dn = C.cast(keep[0], C.POINTER(C.c_void_p))
    a.std = C.cast(keep[1], C.POINTER(C.c_void_p))
    a.exposure_s = C.cast(keep[2], C.POINTER(C.c_double))
    if dark:
        a.dark = C.cast(keep[3], C.POINTER(C.c_void_p))
        a.dark_scale = C.cast(keep[4], C.POINTER(C.c_double))
        a.dark_threshold = 0.05
    a.lut = a.dlut = FAKE
    a.std_lut = FAKE if std_lut else None
    a.median_kernel = K
    a.flat_bytes = flat_bytes
    if flat_bytes:
        a.flat = a.flat_std = a.flat_means = FAKE
    a.out_val = a.out_std = FAKE
    a.algo = algo
    return a, keep


def _call(lib, **kw):
    a, keep = _args(**kw)
    return lib.cl_hdr_merge(C.byref(a), FAKE, 1 << 30, None)


def test_rejects_invalid_arguments(lib):
    for n in (0, 33, -1):
        assert _call(lib, n=n) == INVALID, n
    for t in ([0.01, 0.0, 0.03, 0.04], [0.01, math.nan, 0.03, 0.04], [-0.0, 0.02, 0.03, 0.04]):
        assert _call(lib, t=t) == INVALID, t
    for scale in ([1.0, 0.0, 1.0, 1.0], [1.0, 1.0, -2.0, 1.0], [1.0, 1.0, 1.0, math.nan]):
        assert _call(lib, dark=True, scale=scale) == INVALID, scale
    for K in (0, 8, -3):
        assert _call(lib, K=K) == INVALID, K
    for fb in (3, 4, -1, 16):
        assert _call(lib, flat_bytes=fb) == INVALID, fb
    for algo in (-1, 5):
        assert _call(lib, algo=algo) == INVALID, algo
    assert _call(lib, c=0) == INVALID
    assert _call(lib, c=9) == INVALID
    assert _call(lib, dn_bytes=4) == INVALID
    assert _call(lib, std=False) == INVALID             # neither uncertainty images nor an STD table
    assert lib.cl_hdr_merge(None, FAKE, 1 << 30, None) == INVALID


def test_empty_image_returns_after_the_argument_checks(lib):
    # the largest accepted N, K and every flat type pass the checks; an empty image then returns before any launch
    assert _call(lib, n=32, h=0) == OK
    assert _call(lib, n=1, w=0, K=7, flat_bytes=8) == OK
    assert _call(lib, K=1, h=0, flat_bytes=2, dn_bytes=2) == OK
    assert _call(lib, n=0, h=0) == INVALID
    assert _call(lib, K=8, h=0) == INVALID


def _expected_workspace(n, h, w, c, dn_bytes, std_lut, algo):
    """merge_workspace() of hdr_merge.cu written out: the 16-bit tables (the larger of the generic kernel's
    {w} + {w g, dICRF} rows and the 16-bit kernel's interleaved rows), then for 8-bit C = 1 / 3 stacks the bucket
    counts, the work list and the bucket entries."""
    bits = 256 if dn_bytes == 1 else 65536
    tables = 0
    if bits > 256:
        generic = bits * 8 + bits * c * 16
        wide = bits * c * 32 if std_lut else generic
        tables = max(generic, wide)
    if dn_bytes == 1 and c in (1, 3) and algo != 1:
        samples = h * w * c
        tiles = samples // TILE_SAMPLES
        hot_cap = max(samples // 16, 65536)
        list_end = tables + tiles * 16 + (HOT_HEADER + hot_cap) * 4
        return list_end + 16 + tiles * BUCKET_CAP * 16
    return tables


@pytest.mark.parametrize("dn_bytes", [1, 2])
def test_workspace_bytes_formula(lib, dn_bytes):
    for c in (1, 2, 3, 4, 8):
        for h, w in ((1, 1), (16, 32), (33, 47), (512, 1), (1, 512), (2160, 3840), (4096, 4096)):
            for std_lut in (False, True):
                for algo in (0, 1, 2, 3, 4):
                    a, keep = _args(n=5, h=h, w=w, c=c, dn_bytes=dn_bytes, std=not std_lut, std_lut=std_lut, algo=algo)
                    got = lib.cl_hdr_merge_workspace_bytes(C.byref(a))
                    assert got == _expected_workspace(5, h, w, c, dn_bytes, std_lut, algo), (c, h, w, std_lut, algo)
    assert lib.cl_hdr_merge_workspace_bytes(None) == 0


def test_workspace_list_holds_one_entry_per_16_samples_and_at_least_65536(lib):
    # the work list of the tile kernels (bad pixels that miss their tile's bucket, cancelled single-pass samples)
    small = _expected_workspace(4, 32, 32, 3, 1, False, 0)
    big = _expected_workspace(4, 2048, 2048, 3, 1, False, 0)
    tiles_small, tiles_big = 32 * 32 * 3 // TILE_SAMPLES, 2048 * 2048 * 3 // TILE_SAMPLES
    assert small == tiles_small * 16 + (HOT_HEADER + 65536) * 4 + 16 + tiles_small * BUCKET_CAP * 16
    assert big == tiles_big * 16 + (HOT_HEADER + 2048 * 2048 * 3 // 16) * 4 + 16 + tiles_big * BUCKET_CAP * 16
