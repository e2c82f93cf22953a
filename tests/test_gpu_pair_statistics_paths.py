"""Pair statistics (csrc/linearity.cu): every kernel instance against exact references, with per-case error bounds.

Reference.  The per-sample values are the oracle's own, in float64 NumPy: thresholds, a, r, σa, σr (oracle/linearity.py)
and w = 1/σ.  Every sum over them is then exact: each float64 is an integer mantissa times a power of two, so Σw, Σw·v,
Σw·v² and Σσ are exact Python integers, and the mean μ = Σw·v / Σw and q = Σw(v − μ)² = Σw·v² − 2μΣw·v + μ²Σw over
the samples the variance counts are exact rationals.  The NaN / ±inf / 0 class of every output must equal the
oracle's (np.nansum / np.nanstd on the same values), sign included; the bounds below apply where both are finite.

Bounds, per case (u = 2⁻⁵³).
* δ bounds how far one per-sample term of the kernel can be from NumPy's.  a is the same operations in both.  The
  kernel takes w = rsqrt(q) (≤ 1 ulp, 2u) where NumPy rounds sqrt and then 1/·, and σ = q·rsqrt(q) where NumPy rounds
  sqrt once, and r = a·rcp(m·y) (2 roundings) where NumPy divides once.  Absolute difference: σa, wa ≤ 4u apart, wa·a
  ≤ 6u, so δ = 8u.  Relative difference: t2 = ((σy·x)·rcp)·(rcp·m) is 7 roundings against NumPy's 3 of
  (σy·x)/(m·y²), so t2² differs by ≤ 22u, qr by ≤ 24u, wr and σr by ≤ 16u and wr·r by ≤ 21u: δ = 24u there.
  Where a variance q_i = σ_i² or its parts (t1², t2²) are subnormal, each of those ≤ 4 roundings is exact only to
  η = 2⁻¹⁰⁷⁴ absolute, so sample i gets δ_i = δ + 4η/q_i (2⁻⁵⁰ at most for a normal q_i).  qa is the same operations
  in both, so only the relative difference's q_r really differs there.
* L bounds the longest addition chain of one output: ⌈n_c / (296 · lanes)⌉ per thread (n_c samples per channel,
  lanes = ⌊256/C⌋ threads per channel and block), lanes in the block reduction, ⌈296/32⌉ per lane of the final
  column sum and its 5 shuffle levels.
* Σw:    relative error ≤ b_w = Σw_i·δ_i / Σw + L·u;   error (mean σ): 2(δ + L·u) relative.
* mean:  |μ_k − μ| ≤ 2[Σ|w_i·v_i|(δ_i + L·u) / Σw + |μ|·b_w]  (with one δ: 2(δ + L·u)(Σ|w·v| / |Σw·v| + 1)|μ|).
* std:   the kernel forms q from shifted moments about its own K:  q = T2 − 2(μ − K)T1 + (μ − K)²T0, so
  |q_k − q| ≤ B_q = 2[(L + 8)·u·Σw(|v − K| + |μ − K|)² + 2Σδ_i·w|v||v − μ| + Σδ_i·w(v − μ)²]  and the std is within
  B_q / (2q) + b_w / 2 + 2u relative.  K is read from the workspace (the 2·C doubles behind the 296·14·C block
  partials).
Every case must also meet the 1e-11 bar of DESIGN §3: when K is far from μ (for example K = 0 under data 0.3 ± 1e-7)
B_q grows past it, so the bar is what shows the shift doing its job.  The one exception is a subnormal q_r: NumPy's
own σr there is rounded on the subnormal grid in its own operation order (~1e-4 relative at q_r ≈ 1e-310), and such a
sample carries ~1e150 times the weight of an ordinary one, so that case's relative outputs are held to their bound.
"""
import ctypes as C
import decimal
import math
import re
import zlib
from fractions import Fraction

import numpy as np
import pytest
import torch

from oracle import linearity as oli
from gpu_util import dev, host

pytestmark = pytest.mark.gpu
ops = pytest.importorskip("camera_linearity_b200.ops")
from camera_linearity_b200 import _lib  # noqa: E402

U = 2.0 ** -53
ETA = 2.0 ** -1074                          # the spacing of the subnormal float64 numbers
BLOCKS, THREADS, NQ = 296, 256, 14          # linearity.cu kBlocks, kThreads, kQ
SHIFT_SAMPLES = 16                          # linearity.cu kShiftSamples: a shift chunk is 16 · lanes_used samples
BAR = 1e-11
DELTA = (8 * U, 24 * U)                     # absolute, relative difference


def _lanes(c):
    return THREADS // c


# ---------------------------------------------------------------------------------------------------------------------
# the call, through the C ABI with a workspace the test owns
def _limits(c, lower, upper):
    if lower is None and upper is None:
        return None, None
    lower = [None] * c if lower is None else lower
    upper = [None] * c if upper is None else upper
    lo = (C.c_double * c)(*[-math.inf if v is None else float(v) for v in lower])
    hi = (C.c_double * c)(*[math.inf if v is None else float(v) for v in upper])
    return lo, hi


def _run(x, xs, y, ys, m, lower=None, upper=None):
    """(stats (2, 3, C), K (2, C)) of one cl_pair_statistics call on (n_c, C) float64 arrays"""
    lib = _lib.load()
    c = x.shape[-1]
    t = [None if a is None else dev(a) for a in (x, xs, y, ys)]
    ptr = [None if a is None else a.data_ptr() for a in t]
    lo, hi = _limits(c, lower, upper)
    stats = torch.empty((2, 3, c), dtype=torch.float64, device="cuda")
    nbytes = lib.cl_pair_statistics_workspace_bytes(c)
    ws = torch.full((nbytes // 8,), math.nan, dtype=torch.float64, device="cuda")
    st = lib.cl_pair_statistics(ptr[0], ptr[1], ptr[2], ptr[3], float(m), lo, hi, x.size, c, stats.data_ptr(),
                                ws.data_ptr(), nbytes, torch.cuda.current_stream().cuda_stream)
    assert st == 0
    torch.cuda.synchronize()
    return host(stats), host(ws[BLOCKS * NQ * c:]).reshape(2, c)


# ---------------------------------------------------------------------------------------------------------------------
# exact reference
def _ints(f):
    m, e = np.frexp(f)
    return (m * 2.0 ** 53).astype(np.int64).astype(object), e.astype(np.int64) - 53


def _exact_sum(m, e):
    """Σ m·2^e exactly (m: Python ints, e: int64 exponents)"""
    if len(m) == 0:
        return Fraction(0)
    e0 = int(e.min())
    return int(np.sum(np.left_shift(m, (e - e0).astype(object)))) * Fraction(2) ** e0


def _sqrt(fr):
    with decimal.localcontext() as ctx:
        ctx.prec = 40
        return float((decimal.Decimal(fr.numerator) / decimal.Decimal(fr.denominator)).sqrt())


def _exact(v, s):
    """exact mean and std of one channel, and the sums its bounds need; None where the exact form does not apply
    (an infinite weight, or nothing counted): the oracle's own finite values are then expected"""
    if s is None:
        w = np.ones_like(v)
        sw_set = ~np.isnan(v)
    else:
        w = 1.0 / s
        sw_set = ~np.isnan(w)
    var = np.isfinite(v) & np.isfinite(w)          # the samples whose terms are finite once μ is finite
    if not np.isfinite(w[sw_set]).all() or not var.any():
        return None
    mw, ew = _ints(w[var])
    mv, ev = _ints(v[var])
    s0 = _exact_sum(*_ints(w[sw_set]))
    t0, t1, t2 = _exact_sum(mw, ew), _exact_sum(mw * mv, ew + ev), _exact_sum(mw * mv * mv, ew + 2 * ev)
    if s0 == 0:
        return None
    mu = t1 / s0
    q = t2 - 2 * mu * t1 + mu * mu * t0
    return {"mean": float(mu), "std": _sqrt(q / s0), "q": float(q), "s0": float(s0), "w": w[var], "v": v[var],
            "var_of_sample": None if s is None else s[var] ** 2}


def _exact_error(s):
    sig = s[~np.isnan(s)]
    return float(_exact_sum(*_ints(sig)) / len(sig))


def _chain(n_c, lanes):
    """L: per thread, block reduction, the final kernel's per-lane column sum and its shuffle levels"""
    return math.ceil(n_c / (BLOCKS * lanes)) + lanes + math.ceil(BLOCKS / 32) + 5


def _bounds(ref, K, L, which):
    """(mean absolute, B_q, relative bound of Σw) of the module docstring, with the per-sample δ_i"""
    w, v, mu, s0 = ref["w"], ref["v"], ref["mean"], ref["s0"]
    d = np.full_like(w, DELTA[which])
    if ref["var_of_sample"] is not None:
        with np.errstate(divide="ignore"):
            d += 4 * ETA / ref["var_of_sample"]
    b_w = (float(np.sum(w * d)) + DELTA[which] * max(s0 - float(np.sum(w)), 0.0)) / s0 + L * U
    b_mean = 2 * (float(np.sum(np.abs(w * v) * (d + L * U))) / s0 + abs(mu) * b_w)
    bq = 2 * ((L + 8) * U * float(np.sum(w * (np.abs(v - K) + abs(mu - K)) ** 2))
              + 2 * float(np.sum(d * w * np.abs(v) * np.abs(v - mu))) + float(np.sum(d * w * (v - mu) ** 2)))
    return b_mean, bq, b_w


def _reference(x, xs, y, ys, m, lower=None, upper=None):
    """per-sample values exactly as the oracle computes them, and the oracle's statistics (the class reference)"""
    with np.errstate(all="ignore"):
        if lower is not None or upper is not None:
            x, xs = oli.apply_thresholds(x, xs, lower, upper)
            y, ys = oli.apply_thresholds(y, ys, lower, upper)
        (a, sa), (r, sr) = oli.compute_difference(x, xs, y, ys, m)
        cls = (oli.dimension_statistics(a, sa, axis=0), oli.dimension_statistics(r, sr, axis=0))
    return ((a, sa), (r, sr)), cls


def _same_class(got, want, what):
    assert np.isnan(got) == np.isnan(want), f"{what}: {got} vs oracle {want}"
    if not np.isnan(want):
        assert np.isinf(got) == np.isinf(want) and (got == 0) == (want == 0), f"{what}: {got} vs oracle {want}"
        assert np.sign(got) == np.sign(want), f"{what}: {got} vs oracle {want}"


def check(x, xs, y, ys, m, lower=None, upper=None, stats=None, K=None, bar=(BAR, BAR)):
    """run (unless given) and compare every output with the oracle's class and the exact value within its bound and
    the bar (absolute, relative difference; None: the bound only); returns (stats, K)"""
    if stats is None:
        stats, K = _run(x, xs, y, ys, m, lower, upper)
    c = x.shape[-1]
    vals, cls = _reference(x, xs, y, ys, m, lower, upper)
    use_std = xs is not None or ys is not None
    for which, ((v, s), st) in enumerate(zip(vals, cls)):
        for ch in range(c):
            got = stats[which, :, ch]
            want = [st["mean"][ch], st["std"][ch], st["error"][ch] if use_std else math.nan]
            tag = f"{'abs' if which == 0 else 'rel'} channel {ch}"
            for k, name in enumerate(("mean", "std", "error")):
                _same_class(got[k], want[k], f"{tag} {name}")
            L = _chain(v.shape[0], _lanes(c))
            if use_std and np.isfinite(want[2]) and want[2] > 0:
                e = abs(got[2] - _exact_error(s[:, ch])) / want[2]
                bound = 2 * (DELTA[which] + L * U)
                assert e <= bound and e <= (bar[which] or 1), f"{tag} error {got[2]!r} vs oracle {want[2]!r}: {e:.3g} > {bound:.3g}"
            ref = _exact(v[:, ch], None if s is None else s[:, ch]) if np.isfinite(want[0]) else None
            if ref is None:
                for k in range(2):
                    if np.isfinite(want[k]):
                        assert got[k] == want[k], f"{tag} {k}: {got[k]!r} vs oracle {want[k]!r}"
                continue
            b_mean, bq, b_w = _bounds(ref, K[which, ch], L, which)
            e = abs(got[0] - ref["mean"])
            assert e <= b_mean, f"{tag} mean {got[0]!r} vs exact {ref['mean']!r}: {e:.3g} > bound {b_mean:.3g}"
            if bar[which]:
                assert e <= bar[which] * abs(ref["mean"]), f"{tag} mean: {e / abs(ref['mean']):.3g} > {bar[which]}"
            if ref["std"] > 0:
                e = abs(got[1] - ref["std"]) / ref["std"]
                bound = bq / (2 * ref["q"]) + b_w / 2 + 2 * U
                assert e <= bound, f"{tag} std {got[1]!r} vs exact {ref['std']!r}: {e:.3g} > bound {bound:.3g}"
                assert e <= (bar[which] or 1), f"{tag} std: {e:.3g} relative > {bar[which]}"
            else:                                  # an exactly constant channel
                assert got[1] <= math.sqrt(bq / ref["s0"]), f"{tag} std {got[1]!r} of an exactly constant channel"
    return stats, K


# ---------------------------------------------------------------------------------------------------------------------
# data
INSTANCES = {            # name: (x_std, y_std, multiplier); the kernel instance each selects is pinned by the dispatch map
    "lean": (True, True, 0.7),
    "x_std_only": (True, False, 0.7),
    "y_std_only": (False, True, 0.7),
    "general_m_1e-120": (True, True, 1e-120),
    "general_m_1e120": (True, True, 1e120),
    "no_std": (False, False, 0.7),
}


def _pair(rng, n_c, c, instance, offset=0.05, spread=0.01):
    """x = m·y·(1 + offset ± spread): the absolute and relative differences have means well away from 0"""
    has_xs, has_ys, m = INSTANCES[instance]
    y = rng.uniform(0.2, 0.8, (n_c, c))
    x = m * y * (1 + offset + spread * rng.standard_normal((n_c, c)))
    xs = abs(m) * rng.uniform(1e-3, 2e-3, (n_c, c)) if has_xs else None
    ys = rng.uniform(1e-3, 2e-3, (n_c, c)) if has_ys else None
    return x, xs, y, ys, m


def _sizes(c):
    """samples per channel: fewer samples than lanes_used; inside one shift chunk; the unrolled loop's exact end
    (4 · 296 · lanes_used samples) and one pixel either side of it; ~1.2 M samples (several grid-stride rounds)"""
    lanes = _lanes(c)
    return {"below_lanes": lanes - 1, "in_shift_chunk": SHIFT_SAMPLES * lanes - 3,
            "unrolled_minus_1": 4 * BLOCKS * lanes - 1, "unrolled_exact": 4 * BLOCKS * lanes,
            "unrolled_plus_1": 4 * BLOCKS * lanes + 1, "1.2M": 1_200_000 // c + 1}


CHANNELS = (1, 2, 3, 4, 5, 7, 8)
GRID = ([(i, c, s) for i in INSTANCES for c in CHANNELS for s in ("below_lanes", "in_shift_chunk")]
        + [("lean", c, s) for c in CHANNELS for s in ("unrolled_minus_1", "unrolled_exact", "unrolled_plus_1")]
        + [(i, c, s) for i in INSTANCES if i != "lean" for c in (3, 8)
           for s in ("unrolled_minus_1", "unrolled_exact", "unrolled_plus_1")]
        + [(i, 3, "1.2M") for i in INSTANCES] + [("lean", 1, "1.2M"), ("lean", 8, "1.2M")])


@pytest.mark.parametrize("instance,c,size", GRID, ids=[f"{i}-C{c}-{s}" for i, c, s in GRID])
def test_paths(instance, c, size):
    rng = np.random.default_rng(zlib.crc32(f"{instance} {c} {size}".encode()))
    x, xs, y, ys, m = _pair(rng, _sizes(c)[size], c, instance)
    stats, K = check(x, xs, y, ys, m)
    assert np.isfinite(stats[:, :2]).all()
    if size == "1.2M":
        again, K2 = _run(x, xs, y, ys, m)
        assert np.array_equal(again, stats, equal_nan=True) and np.array_equal(K2, K)     # deterministic


# ---------------------------------------------------------------------------------------------------------------------
# thresholds
THRESHOLD_KINDS = ("per_channel_with_none", "first_chunk_dropped", "channel_dropped")


@pytest.mark.parametrize("kind", THRESHOLD_KINDS)
@pytest.mark.parametrize("c", (3, 8))
@pytest.mark.parametrize("instance", ("lean", "x_std_only", "no_std"))
def test_thresholds(instance, c, kind):
    rng = np.random.default_rng(c * 10 + THRESHOLD_KINDS.index(kind))
    n_c = 40_000
    x, xs, y, ys, m = _pair(rng, n_c, c, instance)
    lower = [0.25 + 0.01 * i if i % 3 != 1 else None for i in range(c)]
    upper = [0.75 - 0.01 * i if i % 3 != 2 else None for i in range(c)]
    if kind == "first_chunk_dropped":              # saturated top rows: every sample of the first shift chunk
        x[:SHIFT_SAMPLES * _lanes(c)] = 5.0
        lower, upper = [None] * c, [4.0] * c
    elif kind == "channel_dropped":                # nothing left in channel 1: every one of its outputs is NaN
        lower[1] = 10.0
    stats, _ = check(x, xs, y, ys, m, lower, upper)
    if kind == "channel_dropped":
        assert np.isnan(stats[:, :, 1]).all()
        assert np.isfinite(stats[:, :2, 0]).all()


# ---------------------------------------------------------------------------------------------------------------------
# degenerate samples, in the first shift chunk and scattered through the image
DEGENERATE = ("value_nan", "sigma_nan", "y_zero", "x_plus_inf", "x_minus_inf", "sigma_zero_one_side",
              "sigma_zero_both", "denormal_variance")


def _spoil(x, xs, y, ys, kind, idx, ch):
    sig = xs if xs is not None else ys
    if kind == "value_nan":
        x[idx, ch] = np.nan
    elif kind == "sigma_nan":
        sig[idx, ch] = np.nan
    elif kind == "y_zero":
        y[idx, ch] = 0.0
    elif kind == "x_plus_inf":
        x[idx, ch] = np.inf
    elif kind == "x_minus_inf":
        x[idx, ch] = -np.inf
    elif kind == "sigma_zero_one_side":
        sig[idx, ch] = 0.0
    elif kind == "sigma_zero_both":
        for s in (xs, ys):
            if s is not None:
                s[idx, ch] = 0.0
    elif kind == "denormal_variance":          # qa subnormal, just below 2^-1022; qr stays normal
        if xs is not None:
            xs[idx, ch] = 1e-154
        if ys is not None:
            ys[idx, ch] = 1e-154 if xs is not None else 1.3e-154


DEGENERATE_GRID = ([(i, k, p) for i in ("lean", "x_std_only", "y_std_only") for k in DEGENERATE
                    for p in ("first_chunk", "scattered")]
                   + [("no_std", "value_nan", p) for p in ("first_chunk", "scattered")])


@pytest.mark.parametrize("instance,kind,place", DEGENERATE_GRID, ids=["-".join(g) for g in DEGENERATE_GRID])
def test_degenerate_samples(instance, kind, place):
    c = 3
    rng = np.random.default_rng(DEGENERATE.index(kind) * 7 + len(place))
    n_c = 20_000
    x, xs, y, ys, m = _pair(rng, n_c, c, instance)
    chunk = SHIFT_SAMPLES * _lanes(c)
    idx = np.arange(3, chunk, 4) if place == "first_chunk" else np.arange(chunk + 11, n_c, 997)
    _spoil(x, xs, y, ys, kind, idx, 1)
    _spoil(x, xs, y, ys, kind, idx[::3], 2)
    if kind == "denormal_variance":
        qa, qr = _variances(x, xs, y, ys, m)
        assert (qa[idx, 1] > 0).all() and (qa[idx, 1] < TINY).all() and (qr[idx, 1] >= TINY).all()
    stats, _ = check(x, xs, y, ys, m)
    assert np.isfinite(stats[:, :2, 0]).all()


TINY = 2.0 ** -1022                         # the smallest normal float64


def _variances(x, xs, y, ys, m):
    """qa = σa², qr = σr² as the kernel and NumPy form them (their sums of squares, before the square root)"""
    xs0 = 0 if xs is None else xs
    ys0 = 0 if ys is None else ys
    with np.errstate(all="ignore"):
        return xs0 ** 2 + (m * ys0) ** 2, (xs0 / (m * y)) ** 2 + ((ys0 * x) / (m * y ** 2)) ** 2


@pytest.mark.parametrize("depth", ("deep", "just_below_normal"))
@pytest.mark.parametrize("instance", ("lean", "x_std_only", "y_std_only"))
def test_subnormal_absolute_variance(instance, depth):
    """Every sample of channel 1 has a subnormal qa (≈ 1e-318, or just below 2^-1022) and a normal qr: the multiplier
    1e-6 keeps σr a million times σa.  qa is the same operations in the kernel and in NumPy, so both sides meet
    1e-11.  The lean routine must hand every such sample to the general one: its rsqrt main path flushes a subnormal
    operand to 0."""
    rng = np.random.default_rng(17)
    n_c, c, m = 20_000, 3, 1e-6
    x, xs, y, ys, _ = _pair(rng, n_c, c, instance)
    x *= m / INSTANCES[instance][2]
    scale = {"deep": 1e-159, "just_below_normal": 0.8e-154}[depth] * rng.uniform(1.0, 1.2, n_c)
    if xs is not None:
        xs[:, 1] = scale
    if ys is not None:
        ys[:, 1] = scale / m
    qa, qr = _variances(x, xs, y, ys, m)
    assert (qa[:, 1] > 0).all() and (qa[:, 1] < TINY).all() and (qr[:, 1] >= TINY).all()
    assert (qa[:, 0] >= TINY).all()
    check(x, xs, y, ys, m)


@pytest.mark.parametrize("instance", ("lean", "x_std_only", "y_std_only"))
def test_subnormal_relative_variance(instance):
    """Every sample of channel 1 has a subnormal qr (≈ 1e-318) and a normal qa (multiplier 1e6).  The kernel's t1, t2
    are reassociated products, so on the subnormal grid its σr differs from NumPy's by up to ~4·2⁻¹⁰⁷⁴/qr: the
    relative outputs are held to their bound with that per-sample term, the absolute ones to 1e-11 as well."""
    rng = np.random.default_rng(18)
    n_c, c, m = 20_000, 3, 1e6
    x, xs, y, ys, _ = _pair(rng, n_c, c, instance)
    x *= m / INSTANCES[instance][2]
    scale = 1e-153 * rng.uniform(1.0, 1.2, n_c)
    if xs is not None:
        xs[:, 1] = scale
    if ys is not None:
        ys[:, 1] = scale / m
    qa, qr = _variances(x, xs, y, ys, m)
    assert (qr[:, 1] > 0).all() and (qr[:, 1] < TINY).all() and (qa[:, 1] >= TINY).all()
    check(x, xs, y, ys, m, bar=(BAR, None))


MULTIPLIER_GRID = [(i, m) for i in ("lean", "x_std_only", "no_std") for m in (0.0, math.nan)
                   if not (i == "no_std" and m == 0.0)]    # (an infinite relative mean without std: the tests below)


@pytest.mark.parametrize("instance,m", MULTIPLIER_GRID, ids=[f"{i}-m_{m}" for i, m in MULTIPLIER_GRID])
def test_degenerate_multiplier(instance, m):
    rng = np.random.default_rng(3)
    x, xs, y, ys, _ = _pair(rng, 5000, 3, instance)
    check(x, xs, y, ys, m)


# ---------------------------------------------------------------------------------------------------------------------
# the defects these tests were written for
@pytest.mark.parametrize("c", (1, 3))
def test_no_std_infinite_relative_mean(c):
    """One y == 0 (curve[0] = 0 linearises DN 0 to 0), no thresholds, no uncertainty images: the relative difference
    is +inf there, its mean +inf and np.nanstd NaN (inf − inf inside a plain sum)."""
    rng = np.random.default_rng(11)
    x, _, y, _, m = _pair(rng, 30_000, c, "no_std")
    y[12_345, 0] = 0.0
    stats, _ = check(x, None, y, None, m)
    assert stats[1, 0, 0] == np.inf and np.isnan(stats[1, 1, 0])
    assert np.isfinite(stats[0, :2, :]).all()


def test_no_std_opposite_infinities():
    """+inf and −inf values in one channel without uncertainty images: mean NaN and std NaN."""
    rng = np.random.default_rng(12)
    x, _, y, _, m = _pair(rng, 30_000, 2, "no_std")
    x[100, 1], x[20_000, 1] = np.inf, -np.inf
    stats, _ = check(x, None, y, None, m)
    assert np.isnan(stats[:, :2, 1]).all()
    assert np.isfinite(stats[:, :2, 0]).all()


@pytest.mark.parametrize("variant", ("x_inf", "ratio_overflow"))
def test_weighted_all_values_infinite(variant):
    """Both uncertainty images, every counted value +inf: the mean is +inf, and np.nansum of the all-NaN terms
    (inf − inf)² is 0, so the std is 0.  'x_inf' makes x itself infinite (the general routine counts every
    sample); 'ratio_overflow' keeps every input and variance normal and only the relative difference overflows, so
    the lean routine's own test |r| < inf is what sends the samples to the general one."""
    rng = np.random.default_rng(13)
    n_c, c = 20_000, 2
    x, xs, y, ys, m = _pair(rng, n_c, c, "lean")
    if variant == "x_inf":
        x[:] = np.inf
    else:
        m = 1e-20
        x = 1e150 * (1 + 1e-4 * rng.random((n_c, c)))
        y = 1e-140 * rng.uniform(0.5, 1.0, (n_c, c))
        xs, ys = 1e-7 * rng.uniform(1, 2, (n_c, c)), 1e-300 * rng.uniform(1, 2, (n_c, c))
    stats, _ = check(x, xs, y, ys, m)
    which = 0 if variant == "x_inf" else 1
    assert (stats[which, 0] == np.inf).all() and (stats[which, 1] == 0).all()


@pytest.mark.parametrize("c", (1, 3))
def test_shift_ignores_samples_the_variance_does_not_count(c):
    """Both uncertainty images.  The first shift chunk has valid values but NaN x_std and lies 1.0 above the rest,
    which spread by 1e-6: a K taken from those samples makes T2 − 2(μ−K)T1 + (μ−K)²T0 cancel ~12 digits."""
    rng = np.random.default_rng(14)
    n_c = 200_000 // c
    x, xs, y, ys, m = _pair(rng, n_c, c, "lean")
    chunk = SHIFT_SAMPLES * _lanes(c)
    x = m * y + 0.25 + 1e-6 * rng.standard_normal((n_c, c))
    x[:chunk] += 1.0
    xs[:chunk] = np.nan
    stats, K = check(x, xs, y, ys, m)
    assert np.all(np.abs(K[0] - 0.25) < 1e-6)


def test_shift_when_the_first_chunk_is_thresholded():
    """Every sample of the first shift chunk thresholded away (saturated top rows), data 0.3 ± 1e-7: K must come from
    the next chunk, not fall back to 0."""
    rng = np.random.default_rng(15)
    n_c, c = 100_000, 3
    x, xs, y, ys, m = _pair(rng, n_c, c, "lean")
    y = 0.5 * (1 + 1e-7 * rng.standard_normal((n_c, c)))
    x = m * y + 0.3 + 1e-7 * rng.standard_normal((n_c, c))
    x[:SHIFT_SAMPLES * _lanes(c)] = 5.0
    stats, K = check(x, xs, y, ys, m, [None] * c, [4.0] * c)
    assert np.all(np.abs(K[0] - 0.3) < 1e-6)


@pytest.mark.parametrize("instance", ("lean", "no_std"))
def test_shift_conditioning(instance):
    """Data 0.3 ± 1e-7 with an ordinary first chunk: q about K = 0 would lose ~13 digits; about the chunk mean it
    meets the 1e-11 bar."""
    rng = np.random.default_rng(16)
    n_c, c = 150_000, 3
    x, xs, y, ys, m = _pair(rng, n_c, c, instance)
    y = 0.5 * (1 + 1e-7 * rng.standard_normal((n_c, c)))
    x = m * y + 0.3 + 1e-7 * rng.standard_normal((n_c, c))
    stats, K = check(x, xs, y, ys, m)
    assert np.all(np.abs(K[0] - 0.3) < 1e-6)


def test_empty_image():
    """n = 0 has no early return.  Through ops an empty image fails the pointer check (an empty tensor's data pointer
    is null); through the C ABI with valid pointers both kernels run and every output is NaN (0 / 0)."""
    z = torch.zeros((0, 3), dtype=torch.float64, device="cuda")
    with pytest.raises(_lib.CamlinError) as err:
        ops.pair_statistics(z, None, z, None, 0.5)
    assert err.value.status == -1
    lib = _lib.load()
    buf = torch.zeros(8, dtype=torch.float64, device="cuda")
    nbytes = lib.cl_pair_statistics_workspace_bytes(3)
    ws = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda")
    for std in (None, buf.data_ptr()):
        stats = torch.zeros((2, 3, 3), dtype=torch.float64, device="cuda")
        n0 = _lib.launch_count()
        st = lib.cl_pair_statistics(buf.data_ptr(), std, buf.data_ptr(), std, 0.5, None, None, 0, 3, stats.data_ptr(),
                                    ws.data_ptr(), nbytes, torch.cuda.current_stream().cuda_stream)
        assert st == 0 and _lib.launch_count() - n0 == 2
        assert torch.isnan(stats).all()


# ---------------------------------------------------------------------------------------------------------------------
# which kernel each argument set launches
def _kernel_name(name):
    hit = re.search(r"(pair_stats_kernel<(?:true|false), ?(?:true|false)>|pair_final_kernel)", name)
    return hit.group(1).replace(", ", ",") if hit else None


DISPATCH = [
    ("both images", (True, True, 0.7), "pair_stats_kernel<true,true>"),
    ("both images, m = 1e-100", (True, True, 1e-100), "pair_stats_kernel<true,true>"),
    ("both images, m = -1e100", (True, True, -1e100), "pair_stats_kernel<true,true>"),
    ("both images, m = 1e-101", (True, True, 1e-101), "pair_stats_kernel<true,false>"),
    ("both images, m = 1e101", (True, True, 1e101), "pair_stats_kernel<true,false>"),
    ("both images, m = NaN", (True, True, math.nan), "pair_stats_kernel<true,false>"),
    ("x_std only", (True, False, 0.7), "pair_stats_kernel<true,false>"),
    ("y_std only", (False, True, 0.7), "pair_stats_kernel<true,false>"),
    ("no std", (False, False, 0.7), "pair_stats_kernel<false,false>"),
]


def test_dispatch_map():
    """One profiler session over every argument set, in order (a warm-up kernel first, so that no launch of interest
    is the session's first activity)."""
    rng = np.random.default_rng(0)
    y = rng.uniform(0.2, 0.8, (64, 3))
    x, s = 0.7 * y * 1.05, rng.uniform(1e-3, 2e-3, (64, 3))
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        torch.ones(1, device="cuda").add_(1)
        torch.cuda.synchronize()
        for _ in range(2):                    # with many modules loaded, tracing can start late in the session
            for _, (hx, hy, m), _ in DISPATCH:
                _run(x, s if hx else None, y, s if hy else None, m)
            torch.cuda.synchronize()
    events = sorted(prof.events(), key=lambda e: e.time_range.start)
    got = [n for n in (_kernel_name(e.name) for e in events) if n]
    if not events:
        pytest.skip("the profiler records no device activity here")
    want = [k for _, _, kernel in DISPATCH for k in (kernel, "pair_final_kernel")]
    assert got[-len(want):] == want                                       # the second pass, exactly
    first = got[: len(got) - len(want)]
    assert len(first) <= len(want) and first == want[len(want) - len(first):]
