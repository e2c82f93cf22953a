"""K3 Welford: every dispatch path of csrc/welford.cu against exact or high-precision references.

* integer stack path (8-bit frames, no ICRF): Σd and Σd² are exact int64 sums (torch on the device), so the
  float64 mean must be the correctly rounded RN(Σd / (F·255)) bit for bit, the uint8 mean of every sample that is
  not a rounding tie is decided in integers, and the SEM is compared with sqrt(M2/(F−1))/sqrt(F) evaluated in
  extended precision from the exact M2 = (F·Σd² − (Σd)²) / (F·255²);
* ICRF stack path: every table value is an exact dyadic rational, so Σx and Σx² are exact Python integers;
* rounding ties and the streaming form: the reference's sequential recurrence (the oracle), because there the
  reference's own rounding noise is what the kernels must reproduce.
"""
import decimal
from fractions import Fraction

import numpy as np
import pytest
import torch

from oracle import welford as ow
from gpu_util import dev, host

pytestmark = pytest.mark.gpu
ops = pytest.importorskip("camera_linearity_b200.ops")
from camera_linearity_b200 import _lib  # noqa: E402

U = 2.0 ** -53                  # unit roundoff of float64
FRAME_BLOCK = 16384             # welford.cu kFrameBlock: above it the integer kernel keeps 64-bit Σd²
LANE_MODE_TIES = 256            # welford.cu kLaneModeTies: from here on one lane per tie


def _sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------------------------------------------------------------
# a. integer stack path
def _int_video(F, n, seed):
    """(F, n) uint8 on the device; eight sample groups: uniform noise, all 255, frames alternating 0/255 (the largest
    num = F·Σd² − (Σd)²), constant pixels (SEM exactly 0), low noise around a base (exact ties for even F), and
    uniform noise again.  The groups need not line up with the 16-sample vectors of the kernel."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    fr = torch.randint(0, 256, (F, n), generator=g, device="cuda", dtype=torch.uint8)
    q = n // 8
    fr[:, q:2 * q] = 255
    fr[:, 2 * q:3 * q] = ((torch.arange(F, device="cuda") % 2) * 255).to(torch.uint8)[:, None]
    fr[:, 3 * q:4 * q] = torch.randint(0, 256, (1, q), generator=g, device="cuda", dtype=torch.uint8)
    base = torch.randint(1, 255, (1, 2 * q), generator=g, device="cuda", dtype=torch.int16)
    noise = torch.randint(-1, 2, (F, 2 * q), generator=g, device="cuda", dtype=torch.int16)
    fr[:, 4 * q:6 * q] = (base + noise).to(torch.uint8)
    return fr


def _int_moments(fr):
    """exact Σd, Σd² per sample (int64 on the host) of a (F, n) uint8 device tensor, in bounded chunks of frames"""
    F, n = fr.shape
    s = torch.zeros(n, dtype=torch.int64, device=fr.device)
    s2 = torch.zeros_like(s)
    step = max(1, (1 << 27) // n)
    for f0 in range(0, F, step):
        x = fr[f0:f0 + step].to(torch.int64)
        s += x.sum(0)
        s2 += (x * x).sum(0)
    return host(s), host(s2)


def _sem_int_reference(num, F):
    """sqrt(M2/(F−1))/sqrt(F) = sqrt(num) / (255·F·sqrt(F−1)), num = F·Σd² − (Σd)² exact: in 64-bit-mantissa long
    double where the platform has it (3 roundings of 2^-64), else in 40-digit decimal on the distinct values."""
    if np.finfo(np.longdouble).nmant >= 63:
        ld = np.longdouble
        return np.sqrt(num.astype(ld)) / (ld(255 * F) * np.sqrt(ld(F - 1)))
    uniq, inv = np.unique(num, return_inverse=True)
    with decimal.localcontext() as ctx:
        ctx.prec = 40
        scale = decimal.Decimal(255 * F) * decimal.Decimal(F - 1).sqrt()
        vals = [decimal.Decimal(int(v)).sqrt() / scale for v in uniq]
    return np.array([float(v) for v in vals])[inv]     # (only 2^-53 coarser than the long double form)


SEM_INT_ULPS = 8    # the kernel's SEM: exact num, then ≤ 6 roundings (reciprocals of the uniform divisors, products,
                    # the square root and its reciprocal); each costs ≤ 2^-53 relative, halved under the root


def _check_integer_stack(fr, C, seed=0):
    """Run ops.welford_stack on (F, n) device frames viewed as (F, n/C, C) and check every output.  Returns the
    number of exact rounding ties."""
    F, n = fr.shape
    mean, sem, mean_u8 = ops.welford_stack(fr.view(F, n // C, C))
    mean, sem, mean_u8 = host(mean).ravel(), host(sem).ravel(), host(mean_u8).ravel()
    s, s2 = _int_moments(fr)
    # the mean is the correctly rounded quotient of two exact doubles -- as NumPy's division is
    expect = s.astype(np.float64) / float(F * 255)
    np.testing.assert_array_equal(mean.view(np.int64), expect.view(np.int64))
    # uint8 mean: rint(Σd / F) in integers except where Σd / F is exactly a half-integer
    tie = 2 * (s % F) == F
    np.testing.assert_array_equal(mean_u8[~tie], ((s[~tie] + F // 2) // F).astype(np.uint8))
    if tie.any():
        idx = np.nonzero(tie)[0]
        sub = host(fr[:, torch.from_numpy(idx).to(fr.device)])
        np.testing.assert_array_equal(mean_u8[idx], ow.welford(list(sub))["mean_u8"])
    if F == 1:
        assert np.isnan(sem).all()
        return int(tie.sum())
    num = F * s2 - s * s
    zero = num == 0
    assert (sem[zero] == 0).all(), "constant samples must have a SEM of exactly 0"
    ref = _sem_int_reference(num[~zero], F)
    err = np.abs(sem[~zero].astype(ref.dtype) - ref) / ref
    assert err.max() <= SEM_INT_ULPS * U, (F, float(err.max()))
    return int(tie.sum())


@pytest.mark.parametrize("C", [1, 2, 3, 4, 8])
def test_integer_stack_exact_small_images(C):
    # 768 samples = 48 vectors: slices = min(32, largest power of two <= F); F crosses kUnroll (8 frames in flight
    # per lane), the slice remainder and kFrameBlock (16384: the BIG kernel above it)
    n = 768
    ties = 0
    for F in (1, 2, 3, 7, 8, 9, 15, 16, 17, 255, 256, 257, FRAME_BLOCK, FRAME_BLOCK + 1, 20000):
        ties += _check_integer_stack(_int_video(F, n, seed=F * 10 + C), C)
    assert ties > 0                                # the low-noise group makes exact ties for small even F


@pytest.mark.parametrize("slices", [1, 2, 4, 8, 16, 32])
def test_integer_stack_exact_every_slice_count(slices):
    # The host picks the smallest power of two `slices` with n_vec·slices >= sm_count·1024 (capped at 32 and at F),
    # n_vec = n / 16.  n_vec = ceil(sm_count·1024 / slices) (rounded up to a multiple of 3 for C = 3) targets exactly
    # this count; F >= slices and, where it is cheap, F > 8·slices so the unrolled loop runs as well.  The checks do
    # not depend on the count actually chosen.
    want = _sm() * 1024
    n_vec = -(-want // slices)
    n_vec += -n_vec % 3
    F = {1: 17, 2: 17, 4: 37, 8: 73, 16: 257, 32: 300}[slices]
    _check_integer_stack(_int_video(F, 16 * n_vec, seed=slices), 3)


def test_integer_stack_big_kernel_with_fewer_slices():
    # F = 16385 (64-bit Σd²) on an image that targets 16 frame slices instead of 32: 2.5 GB of frames
    want = _sm() * 1024
    n_vec = -(-want // 16)
    n_vec += -n_vec % 3
    _check_integer_stack(_int_video(FRAME_BLOCK + 1, 16 * n_vec, seed=77), 3)


# ---------------------------------------------------------------------------------------------------------------------
# b. ICRF stack path
def _tables(C):
    d = np.arange(256) / 255.0
    c = np.arange(C)
    return {
        "smooth": d[:, None] ** (2.0 + 0.1 * c),
        "non_monotone": 0.5 + 0.4 * np.sin(7 * np.pi * d[:, None] + c),
        "above_one": 1.6 * d[:, None] ** (1.5 + 0.1 * c),        # mean·255 up to 408: the uint8 cast wraps
        "identity": np.repeat(d[:, None], C, axis=1),
    }


def _lut_exact(frames, table):
    """Exact integer ΣX, ΣX², X of frame 0 per sample (Python ints) and the scale D with x = X / D for every table
    value (all float64 values are dyadic rationals)."""
    F = frames.shape[0]
    C = table.shape[1]
    fr = frames.reshape(F, -1)
    vals = [Fraction(float(v)) for v in table.ravel()]
    D = max(v.denominator for v in vals)
    ti = np.array([v.numerator * (D // v.denominator) for v in vals], dtype=object).reshape(table.shape)
    x = ti[fr, np.arange(fr.shape[1]) % C]
    return x.sum(axis=0), (x * x).sum(axis=0), x[0], D


def _check_lut_stack(frames, table, out):
    """out = (mean, sem, mean_u8) of the kernel for host frames (F, ..., C).

    mean: the kernel returns x_first + RN(s1 / F), s1 = Σy = Σ(x − x_first) summed frame by frame: within 2 ulps of
    the correctly rounded exact mean plus the bound of recursive summation, F·2^-53·mean|y| (which dominates for
    dark pixels and when frame 0 is an outlier).
    sem: the kernel forms M2 = s2 − s1·(s1/F) from the shifted sums s1 = Σy, s2 = Σy².  Recursive summation of F
    terms errs by at most F·2^-53·s2 in s2 and (via s1) 2F·2^-53·s2 in s1²/F, so M2 is good to 3F·2^-53·κ relative,
    κ = s2 / M2 = Σ(x − x_first)² / Σ(x − mean)² (≈ 2 for noise, ≈ F when frame 0 is the only outlier: then log2 F
    more bits cancel), and the square root halves it: rtol = max(1e-13, 2·F·2^-53·κ), κ evaluated exactly.
    mean_u8: bit-exact against the reference recurrence."""
    F = frames.shape[0]
    mean, sem, mean_u8 = (host(t).ravel() for t in out)
    S, Q, X0, D = _lut_exact(frames, table)
    ref = np.array([float(Fraction(int(s), F * D)) for s in S])
    fr = frames.reshape(F, -1)
    x = table[fr, np.arange(fr.shape[1]) % table.shape[1]]
    tol = 2 * np.spacing(np.abs(ref)) + F * U * np.abs(x - x[0]).mean(axis=0)
    bad = np.abs(mean - ref) > tol
    assert not bad.any(), (F, mean[bad][:4], ref[bad][:4])
    o = ow.welford(list(frames), icrf=table)
    np.testing.assert_array_equal(mean_u8, o["mean_u8"].ravel())
    if F == 1:
        assert np.isnan(sem).all()
        return
    with decimal.localcontext() as ctx:
        ctx.prec = 40
        den = decimal.Decimal(F * F * (F - 1))
        for i, (s, q, x0) in enumerate(zip(S, Q, X0)):
            num = F * q - s * s                                   # F² M2 D², exact
            if num == 0:
                assert sem[i] == 0, (F, i, sem[i])
                continue
            kappa = Fraction(F * (q - 2 * x0 * s + F * x0 * x0), num)
            rtol = decimal.Decimal(max(1e-13, 2 * F * U * float(kappa)))
            r = (decimal.Decimal(num) / den).sqrt() / D
            assert abs(decimal.Decimal(float(sem[i])) - r) <= rtol * r, (F, i, float(sem[i]), float(r), float(kappa))


def _stack_capi(frames, table, frame_offset=0, out_offset=0):
    """cl_welford_stack called directly: frames `frame_offset` bytes into a larger buffer, mean / sem `out_offset`
    doubles into theirs (torch allocations are 512-byte aligned)."""
    lib = _lib.load()
    F = frames.shape[0]
    n = frames[0].size
    C = frames.shape[-1]
    buf = torch.zeros(F * n + 16, dtype=torch.uint8, device="cuda")
    buf[frame_offset:frame_offset + F * n] = dev(frames.reshape(-1))
    lut = dev(np.ascontiguousarray(table, dtype=np.float64)) if table is not None else None
    mean = torch.full((n + 2,), -1.0, dtype=torch.float64, device="cuda")
    sem = torch.full((n + 2,), -1.0, dtype=torch.float64, device="cuda")
    mean_u8 = torch.zeros(n + 16, dtype=torch.uint8, device="cuda")
    ws_bytes = lib.cl_welford_stack_workspace_bytes(F, n)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    st = lib.cl_welford_stack(buf.data_ptr() + frame_offset, F, n, C, lut.data_ptr() if lut is not None else None,
                              255.0, mean.data_ptr() + 8 * out_offset, sem.data_ptr() + 8 * out_offset,
                              mean_u8.data_ptr(), ws.data_ptr(), ws_bytes, torch.cuda.current_stream().cuda_stream)
    assert st == 0, st
    return mean[out_offset:out_offset + n], sem[out_offset:out_offset + n], mean_u8[:n]


LUT_FRAMES = (1, 2, 3, 4, 5, 7, 8, 9, 11, 12, 13, 300)


@pytest.mark.parametrize("C", [1, 2, 3, 4, 5, 6, 7, 8])
def test_lut_stack_every_table_copy_count(C):
    # C <= 3: 16 table copies, C = 4..6: 8, C = 7, 8: 4 (256·C·copies doubles within 96 KB of shared memory).
    # Layouts: n % 4 == 0 and aligned (the two-batch `full` loop), n % 4 != 0 (only for C not a multiple of 4) and the
    # frames one byte into their buffer (both the byte loop).  F crosses the two batches of 4 frames.
    rng = np.random.default_rng(C)
    rows_aligned = 28                    # n = 28·C, a multiple of 4
    rows_ragged = 27 if C % 2 else 29    # odd rows: n % 4 != 0 unless C is a multiple of 4
    for name, table in _tables(C).items():
        for F in LUT_FRAMES:
            layouts = [("aligned", rows_aligned, 0), ("byte_offset", rows_aligned, 1)]
            if C % 4:
                layouts.append(("ragged", rows_ragged, 0))
            for layout, rows, off in layouts:
                base = rng.integers(20, 236, (1, rows, C))
                frames = np.clip(base + rng.integers(-12, 13, (F, rows, C)), 0, 255).astype(np.uint8)
                if off:
                    out = _stack_capi(frames, table, frame_offset=off)
                else:
                    out = ops.welford_stack(dev(frames), dev(table))
                _check_lut_stack(frames, table, out)


@pytest.mark.parametrize("C", [1, 3, 5, 8])
def test_lut_stack_conditioning(C):
    rng = np.random.default_rng(100 + C)
    table = _tables(C)["smooth"]
    rows = 40
    for F in (3, 13, 300):
        # frame 0 is the only outlier: the shift by frame 0 then buys nothing and the sums cancel
        base = rng.integers(10, 120, (1, rows, C))
        frames = np.clip(base + rng.integers(-2, 3, (F, rows, C)), 0, 255).astype(np.uint8)
        frames[0] = 255 - base[0]
        _check_lut_stack(frames, table, ops.welford_stack(dev(frames), dev(table)))
        # a static dark pixel with a single one-DN flicker: one LUT step of x^2 near DN 1 is ~5e-5
        dark = rng.integers(0, 4, (1, rows, C))
        frames = np.repeat(dark, F, axis=0).astype(np.uint8)
        flick = rng.integers(0, F, (rows, C))
        r_i, c_i = np.meshgrid(np.arange(rows), np.arange(C), indexing="ij")
        frames[flick, r_i, c_i] += 1                  # (when the flicker is frame 0 it is the outlier case again)
        _check_lut_stack(frames, table, ops.welford_stack(dev(frames), dev(table)))
        # identical frames: SEM exactly 0 for every channel count (checked inside, num == 0)
        frames = np.repeat(rng.integers(0, 256, (1, rows, C)), F, axis=0).astype(np.uint8)
        out = ops.welford_stack(dev(frames), dev(table))
        assert not host(out[1]).any()
        _check_lut_stack(frames, table, out)


# ---------------------------------------------------------------------------------------------------------------------
# c. rounding-tie replay
def _half_table(C):
    """x = DN / 510: DN 2k, 2k+1, 2k+2 are k, k + 1/2, k + 1 in units of 1/255, so exact ties exist for odd F too"""
    return np.repeat((np.arange(256) / 510.0)[:, None], C, axis=1)


def _tie_video(rng, F, n, n_ties, icrf):
    """(F, n) uint8 video whose exact mean·255 is k + 1/2 on `n_ties` random samples and k + 1/2 + 1/F (or + 1/(2F)
    ... never within 1e-9 of a tie) elsewhere; each sample's frames in an independent random order.
    Returns (frames, tie indices, k per sample)."""
    tie = np.zeros(n, bool)
    tie[rng.choice(n, n_ties, replace=False)] = True
    if icrf:
        # a = F % 2 frames of 2k+1, b = (F − a)/2 of 2k+2, the rest 2k: mean·255 = k + (a/2 + b)/F = k + 1/2
        k = rng.integers(0, 127, n)
        a = F % 2
        b = (F - a) // 2
        col = np.zeros((F, n), np.uint8)
        col[:a] = 1
        col[a:a + b] = 2
        col[a + b, ~tie] = 2                          # one more 2k+2 frame: k + 1/2 + 1/F
        frames = (2 * k).astype(np.uint8)[None, :] + rng.permuted(col, axis=0)
    else:
        assert F % 2 == 0, "Σd / F is a half-integer only for even F"
        k = rng.integers(0, 255, n)
        col = np.zeros((F, n), np.uint8)
        col[:F // 2] = 1
        col[F // 2, ~tie] = 1                         # k + 1/2 + 1/F (exactly k + 1 for F = 2)
        frames = k.astype(np.uint8)[None, :] + rng.permuted(col, axis=0)
    return frames, np.nonzero(tie)[0], k


def _check_ties(frames, C, table, tie_idx, k):
    F = frames.shape[0]
    video = frames.reshape(F, -1, C)
    o = ow.welford(list(video), icrf=table)["mean_u8"].ravel()
    up = o[tie_idx] == k[tie_idx] + 1
    assert ((o[tie_idx] == k[tie_idx]) | up).all()
    assert up.any() and not up.all(), "the reference must round some ties down and some up"
    _, _, mean_u8 = ops.welford_stack(dev(video), dev(table) if table is not None else None)
    np.testing.assert_array_equal(host(mean_u8).ravel(), o)


@pytest.mark.parametrize("mode", ["integer", "icrf_lane", "icrf_warp"])
@pytest.mark.parametrize("F", [2, 10, 16, 17, 256, 257, 600])
def test_tie_replay_every_branch(mode, F):
    # integer and ICRF with C = 4 (the largest table the lane form holds): one warp per tie below 256 ties, one lane
    # per tie from 256 on; ICRF with C = 5: always one warp per tie.  F crosses kReplayBatch (16) and kReplayWindow (256).
    if mode == "integer" and F % 2:
        pytest.skip("without an ICRF Σd / F is never a half-integer for odd F")
    C = {"integer": 4, "icrf_lane": 4, "icrf_warp": 5}[mode]
    table = None if mode == "integer" else _half_table(C)
    rng = np.random.default_rng(F * 7 + C)
    for n, n_ties in ((1200, LANE_MODE_TIES - 1), (1200, LANE_MODE_TIES), (4800, 3000)):
        frames, tie_idx, k = _tie_video(rng, F, n, n_ties, table is not None)
        _check_ties(frames, C, table, tie_idx, k)


def test_tie_replay_lanes_several_passes_of_the_grid():
    # every sample of 10 × 480×640×3 is a tie: 921 600 ties > 2 · sm_count · 8 CTAs · 128 lanes, so each CTA of the
    # lane form loops over several blocks of ties (its __syncthreads inside that loop)
    rng = np.random.default_rng(11)
    n = 480 * 640 * 3
    assert n > 2 * _sm() * 8 * 128
    frames, tie_idx, k = _tie_video(rng, 10, n, n, False)
    _check_ties(frames, 3, None, tie_idx, k)


@pytest.mark.parametrize("C", [3, 6])
def test_icrf_near_ties(C):
    # samples whose exact mean·255 is k + 1/2 ± eps: eps = 1e-12 and 1e-10 are inside the kernel's 1e-9 window
    # (replayed), 1e-8 outside (decided by the kernel's own mean); all must match the reference
    rng = np.random.default_rng(C)
    F = 40
    epss = [s * e for e in (1e-12, 1e-10, 1e-8) for s in (1, -1)]
    table = np.repeat((np.arange(256) / 255.0)[:, None] ** 2, C, axis=1)
    ks = rng.integers(20, 200, len(epss))
    for j, (eps, kk) in enumerate(zip(epss, ks)):
        mid = (kk + 0.5 + eps) / 255.0
        table[2 * j] = mid - 3 / 255.0
        table[2 * j + 1] = mid + 3 / 255.0
    n = 600 * C
    kind = rng.integers(0, len(epss), n)
    col = np.zeros((F, n), np.int64)
    col[:F // 2] = 1
    frames = (2 * kind[None, :] + rng.permuted(col, axis=0)).astype(np.uint8).reshape(F, -1, C)
    o = ow.welford(list(frames), icrf=table)
    _, _, mean_u8 = ops.welford_stack(dev(frames), dev(table))
    np.testing.assert_array_equal(host(mean_u8), o["mean_u8"])


def test_tie_replay_at_65536_frames():
    # the replay and the 1e-9 window at large F: 300 exact ties (lane form) among noisy samples
    rng = np.random.default_rng(65536)
    F, C, n = 65536, 3, 1536
    table = _half_table(C)
    frames, tie_idx, k = _tie_video(rng, F, n, 300, True)
    noisy = np.setdiff1d(np.arange(n), tie_idx)[: n // 2]
    lvl = rng.integers(20, 230, noisy.size, dtype=np.int16)
    frames[:, noisy] = lvl[None, :] + rng.integers(-6, 7, (F, noisy.size), dtype=np.int16)   # stays in 14..235
    video = frames.reshape(F, -1, C)
    o = ow.welford(list(video), icrf=table)
    _, _, mean_u8 = ops.welford_stack(dev(video), dev(table))
    np.testing.assert_array_equal(host(mean_u8), o["mean_u8"])


# ---------------------------------------------------------------------------------------------------------------------
# d. streaming form
@pytest.mark.parametrize("C", [1, 2, 5, 8])
def test_streaming_update_with_icrf_resumed(C):
    rng = np.random.default_rng(C)
    rows = 29                                    # n % 4 != 0 for C = 1, 2, 5
    F, k0 = 61, 9
    table = _tables(C)["smooth"]
    frames = np.clip(rng.integers(20, 236, (1, rows, C)) + rng.integers(-9, 10, (F, rows, C)), 0, 255).astype(np.uint8)
    o0 = ow.welford(list(frames[:k0]), icrf=table)             # the state after k0 frames
    mean, m2 = dev(o0["mean"]), dev(o0["m2"])
    count = k0
    for size in (1, 7, 3, 16, 5, 20):                         # ragged chunks
        count = ops.welford_update(dev(frames[count:count + size]), mean, m2, count, dev(table))
    assert count == F
    o = ow.welford(list(frames), icrf=table)
    np.testing.assert_array_equal(host(mean).view(np.int64), o["mean"].view(np.int64))
    np.testing.assert_array_equal(host(m2).view(np.int64), o["m2"].view(np.int64))
    sem, mean_u8 = ops.welford_finalize(mean, m2, count)
    np.testing.assert_array_equal(host(sem).view(np.int64), o["sem"].view(np.int64))
    np.testing.assert_array_equal(host(mean_u8), o["mean_u8"])


def test_finalize_edges():
    # count = 1: sqrt(0 / 0) is NaN
    mean = dev(np.array([0.1, 0.5, 0.9]))
    sem, _ = ops.welford_finalize(mean, dev(np.zeros(3)), 1)
    assert np.isnan(host(sem)).all()
    # means whose RN(mean·255) is exactly k + 1/2: half-even, as np.around
    m = (np.arange(255) + 0.5) / 255.0
    m = m[m * 255.0 == np.arange(255) + 0.5]
    assert m.size > 100
    # out-of-range means wrap as NumPy's float -> uint8 cast does
    m = np.concatenate([m, np.array([256, 257, 300.4, 511.5, 766, -1, -2.5, -300, 1e6]) / 255.0])
    _, mean_u8 = ops.welford_finalize(dev(m), None, 10)
    np.testing.assert_array_equal(host(mean_u8), np.around(m * 255).astype(np.uint8))


def test_stack_and_streaming_forms_agree():
    # the two forms of the same video give the same uint8 mean bit for bit (ties included)
    rng = np.random.default_rng(21)
    for F, table in ((64, None), (17, None), (40, _tables(3)["smooth"]), (13, _tables(3)["above_one"])):
        frames = np.clip(rng.integers(20, 236, (1, 16, 24, 3)) + rng.integers(-1, 2, (F, 16, 24, 3)),
                         0, 255).astype(np.uint8)
        lut = dev(table) if table is not None else None
        _, _, u8_stack = ops.welford_stack(dev(frames), lut)
        mean = torch.zeros((16, 24, 3), dtype=torch.float64, device="cuda")
        m2 = torch.zeros_like(mean)
        ops.welford_update(dev(frames), mean, m2, 0, lut)
        _, u8_stream = ops.welford_finalize(mean, m2, F)
        assert torch.equal(u8_stack, u8_stream)


# ---------------------------------------------------------------------------------------------------------------------
# e. misaligned C-ABI buffers
def test_misaligned_outputs_and_frames_take_the_replay():
    # mean / sem 8 bytes (not 16) into their buffers, or frames one byte into theirs: the integer kernel needs
    # 16-byte vectors, so the whole image is replayed with the reference recurrence.  The uint8 mean is identical to
    # the aligned call; the float64 mean / SEM are then the reference's own (bit for bit), which differ from the
    # integer path's correctly rounded values by the reference's rounding noise only.
    rng = np.random.default_rng(5)
    F = 24
    frames = _tie_video(rng, F, 96, 30, False)[0].reshape(F, 32, 3)      # 30 exact ties among 96 samples
    o = ow.welford(list(frames))
    mean_a, sem_a, u8_a = _stack_capi(frames, None)
    for kw in ({"out_offset": 1}, {"frame_offset": 1}, {"frame_offset": 3, "out_offset": 1}):
        mean, sem, u8 = _stack_capi(frames, None, **kw)
        assert torch.equal(u8, u8_a), kw
        np.testing.assert_array_equal(host(u8), o["mean_u8"].ravel())
        np.testing.assert_array_equal(host(mean).view(np.int64), o["mean"].ravel().view(np.int64))
        np.testing.assert_array_equal(host(sem).view(np.int64), o["sem"].ravel().view(np.int64))
        np.testing.assert_allclose(host(mean), host(mean_a), rtol=1e-13, atol=0)
        np.testing.assert_allclose(host(sem), host(sem_a), rtol=1e-11, atol=0)


# ---------------------------------------------------------------------------------------------------------------------
# f. dispatch map
def test_dispatch_map():
    """One input per path of the dispatcher, with the kernel it must launch (template instance where there is
    one) as the profiler records it.  Keeps the tests above honest when the dispatcher changes."""
    rng = np.random.default_rng(0)
    act = torch.profiler.ProfilerActivity.CUDA

    def launched(fn):
        with torch.profiler.profile(activities=[act]) as prof:
            fn()
            torch.cuda.synchronize()
        return [e.name for e in prof.events()]

    def small(F, C=3, rows=256):
        return dev(np.clip(rng.integers(20, 236, (1, rows, C)) + rng.integers(-3, 4, (F, rows, C)), 0, 255)
                   .astype(np.uint8))

    probe = launched(lambda: ops.welford_stack(small(8)))
    if not any("welford" in name for name in probe):
        pytest.skip("the profiler records no device activity here")

    ties_few = _tie_video(rng, 10, 1200, 40, False)[0].reshape(10, -1, 4)
    ties_many = _tie_video(rng, 10, 1200, 600, False)[0].reshape(10, -1, 4)
    ties_warp = _tie_video(rng, 10, 1200, 600, True)[0].reshape(10, -1, 5)
    cases = [
        ("welford_stack_u8_kernel<false>", lambda: ops.welford_stack(small(FRAME_BLOCK, rows=16))),
        ("welford_stack_u8_kernel<true>", lambda: ops.welford_stack(small(FRAME_BLOCK + 1, rows=16))),
        ("welford_stack_lut_kernel<16>", lambda: ops.welford_stack(small(9, 3), dev(_tables(3)["smooth"]))),
        ("welford_stack_lut_kernel<8>", lambda: ops.welford_stack(small(9, 5), dev(_tables(5)["smooth"]))),
        ("welford_stack_lut_kernel<8>", lambda: ops.welford_stack(small(9, 6), dev(_tables(6)["smooth"]))),
        ("welford_stack_lut_kernel<4>", lambda: ops.welford_stack(small(9, 8), dev(_tables(8)["smooth"]))),
        ("welford_tie_replay_kernel", lambda: ops.welford_stack(dev(ties_few))),
        ("welford_tie_replay_kernel", lambda: ops.welford_stack(dev(ties_many))),
        ("welford_tie_replay_kernel", lambda: ops.welford_stack(dev(ties_warp), dev(_half_table(5)))),
        ("welford_replay_kernel", lambda: ops.welford_stack(small(9, 3, rows=7))),
        ("welford_replay_kernel", lambda: _stack_capi(host(small(9)), None, out_offset=1)),
        ("welford_update_kernel", lambda: ops.welford_update(small(9), torch.zeros((256, 3), dtype=torch.float64,
                                                                                    device="cuda"),
                                                             torch.zeros((256, 3), dtype=torch.float64, device="cuda"),
                                                             0, dev(_tables(3)["smooth"]))),
        ("welford_finalize_kernel", lambda: ops.welford_finalize(dev(np.full(5, 0.5)), dev(np.ones(5)), 9)),
    ]
    for kernel, fn in cases:
        names = [nm for nm in launched(fn) if "welford" in nm]
        assert any(kernel in nm for nm in names), (kernel, names)
        if kernel.startswith("welford_stack_lut_kernel"):
            # exactly one instance of the template runs
            assert sum("welford_stack_lut_kernel<" in nm for nm in names) == 1, names
