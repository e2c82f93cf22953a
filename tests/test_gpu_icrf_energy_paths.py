"""K4 (``csrc/icrf_energy.cu``) path by path, against references whose own error is pinned layer by layer.

* Curves and tables: a NumPy restatement of ``build_curve``'s operation order (sequential k loop, separate multiply
  and add, shift, ``curve[0] = 0``) is exact, so ``curves``, the gates and the I / R tables in their
  ``[group][dn][lane]`` layout are asserted bit for bit; the ``pow`` parametrisation against mpmath within CUDA's
  2-ulp bound.
* Pair sums: each term from the kernel's own curve and the exposure doubles in ``np.longdouble`` (64-bit mantissa),
  summed in long double.  Valid counts are exact.  Each case carries an error bound derived from its data: per-term
  rounding of A, B, RN(1/t), RN(1/v) and the FMA (relative to u_ij = A_i B_j, not to |u_ij - 1|), with std the
  variance chain and ``rsqrt`` (1 ulp), and u * L * (sum of |everything added|, the masked 1.0s of the uniform loop
  included) for the lane recursion, the warp tree, the CTA reduction and the final subtraction.
* Finalize: a restatement of ``energy_of`` on ``pair_acc`` matches the energies bit for bit; the fused tail is
  bit-identical to partial + ``reduce_ctas_kernel`` + finalize; repeated runs are bit-identical.
"""
import re

import numpy as np
import pytest
import torch

from gpu_util import dev, host

pytestmark = pytest.mark.gpu
ops = pytest.importorskip("camera_linearity_b200.ops")

U = 2.0 ** -53
TIGHT = 1e-11                     # DESIGN §3, K4 energies
CLUSTER = 8                       # CTAs per candidate of curves_wide_kernel
LD = np.longdouble
assert np.finfo(LD).nmant >= 63, "the pair-sum reference needs an x87 long double"


def _basis(D, k=5):
    x = np.linspace(0, 1, D)
    q, _ = np.linalg.qr(np.stack([np.sin((j + 1) * np.pi * x) * x for j in range(k)], axis=1))
    return x, q


def _stack(rng, D, n_px, t, gamma=1 / 2.2, dtype=np.uint8):
    rad = rng.uniform(0, 1, (n_px, 1)) * 1.2 / t[-1]
    return np.rint((D - 1) * np.clip(rad * t[None, :], 0, 1) ** gamma).astype(dtype)


def _plan(dn, sd, t, mean, pca, lower, upper, params):
    """params (S, n_params); pixels (n_px, N).  Curves + tables built, nothing else run."""
    n_px, n = dn.shape
    plan = ops.IcrfEnergyPlan(dev(dn.reshape(n_px, 1, n)), None if sd is None else dev(sd.reshape(n_px, 1, n)), t,
                              mean, dev(pca), lower, upper, mean is not None, params.shape[0])
    plan.set_params(torch.from_numpy(np.ascontiguousarray(params)))
    plan.curves_and_tables()
    return plan


# ---- layer 1: curves, gates, tables ------------------------------------------------------------------------
def ref_curves(mean, pca, params):
    """build_curve with use_mean_icrf: sequential k loop, RN(pca * p) then RN(acc + .), then the shift."""
    S, D = params.shape[0], pca.shape[0]
    acc = np.zeros((S, D))
    for k in range(pca.shape[1]):
        acc = acc + pca[None, :, k] * params[:, k, None]
    v = mean[None, :] + acc
    v = v + (1.0 - v[:, -1:])
    v[:, 0] = 0.0
    return v


def ref_gates(v):
    with np.errstate(invalid="ignore"):
        bad = (v > 1).any(1) | (v < 0).any(1) | ~(v[:, 1:] > v[:, :-1]).all(1) | np.isnan(v).any(1)
    return ~bad


def uniform(lower, upper):
    return lower >= 1 and lower <= upper


def ref_tables(v, ok, lower, upper, use_std=False):
    S, D = v.shape
    lo, hi = v[:, lower, None], v[:, upper, None]
    with np.errstate(invalid="ignore", divide="ignore"):
        masked = (v < lo) | (v > hi)
        if uniform(lower, upper):
            inside = (np.arange(D) >= lower) & (np.arange(D) <= upper)
            benign = np.broadcast_to(np.where(inside, 1.0, 0.0), v.shape)
            I = np.where(ok[:, None], np.where(masked, 0.0, v), benign)
            r = 1.0 / v
            if use_std:                                    # 1/v = inf (subnormal v): weight 0 through R = 0
                r = np.where(np.isinf(r), 0.0, r)
            R = np.where(ok[:, None], np.where(masked, 0.0, r), benign)
        else:
            I = np.where(masked, np.nan, v)
            R = 1.0 / I
    lay = lambda a: a.reshape(S // 32, 32, D).transpose(0, 2, 1).ravel()        # [group][dn][lane]
    return np.concatenate([lay(I), lay(R)])


def _same_bits(a, b):
    """bit for bit, except that a NaN only has to be a NaN (the device's 1/NaN payload is its own)."""
    a, b = np.asarray(a), np.asarray(b)
    return np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(
        a[~np.isnan(a)].view(np.int64), b[~np.isnan(b)].view(np.int64))


def _boundary_problem(D, S, seed):
    """A basis with one spike column per CTA boundary of the wide kernel (position r * ceil(D / 8)), candidates that
    fail only across one boundary, equal neighbours there, NaN parameters and ordinary ones."""
    rng = np.random.default_rng(seed)
    x, q = _basis(D, 3)
    mean = x ** 2.2
    chunk = (D + CLUSTER - 1) // CLUSTER
    cuts = sorted({r * chunk for r in range(1, CLUSTER) if 1 < r * chunk < D - 1}) or [D // 2] * (D > 3)
    spikes = np.zeros((D, len(cuts)))
    for c, b in enumerate(cuts):
        spikes[b, c] = -1.0
    pca = np.hstack([q, spikes])
    k = q.shape[1]
    params = np.zeros((S, pca.shape[1]))
    params[:, :k] = rng.uniform(-0.03, 0.03, (S, k))
    for c, b in enumerate(cuts):
        step = mean[b] - mean[b - 1]                       # exact (Sterbenz): mean[b] - step == mean[b - 1]
        params[3 * c % S, :k] = 0.0
        params[3 * c % S, k + c] = 1.5 * step              # non-increasing across this boundary only
        params[(3 * c + 1) % S, :k] = 0.0
        params[(3 * c + 1) % S, k + c] = step              # equal neighbours
        params[(3 * c + 2) % S, :k] = 0.0
        params[(3 * c + 2) % S, k + c] = 0.5 * step        # a smaller dip: still increasing
    params[S - 1, 0] = np.nan
    params[S - 2, k - 1] = 3.0                             # oscillates: out of [0, 1] (D > 3)
    return mean, pca, params, cuts


@pytest.mark.parametrize("D", [2, 64, 200, 256, 257, 1000, 4096, 65536])
@pytest.mark.parametrize("limits", ["inner", "lower0", "swapped"])
def test_curves_gates_and_tables_bit_exact(D, limits):
    S = 64 if D <= 4096 else 32
    mean, pca, params, cuts = _boundary_problem(D, S, D)
    lower, upper = {"inner": (max(1, D // 50), D - 1 - D // 50), "lower0": (0, D - 1),
                    "swapped": (D - 1 - D // 50, max(1, D // 50) if D > 2 else 0)}[limits]
    if limits == "swapped" and D == 2:
        lower, upper = 1, 0
    dtype = np.uint8 if D <= 256 else np.uint16
    plan = _plan(np.zeros((1, 2), dtype), None, np.array([0.01, 0.02]), mean, pca, lower, upper, params)
    v = ref_curves(mean, pca, params)
    ok = ref_gates(v)
    assert _same_bits(host(plan.curves), v)
    assert np.array_equal(host(plan.valid) != 0, ok)
    tab = host(plan.tables).view(np.float64)
    assert _same_bits(tab, ref_tables(v, ok, lower, upper))
    if D > 3:                                              # every boundary candidate gated or not as intended
        for c in range(len(cuts)):
            assert not ok[3 * c % S] and not ok[(3 * c + 1) % S] and ok[(3 * c + 2) % S], c
        assert not ok[S - 2]
    assert not ok[S - 1] and ok.sum() >= 2


@pytest.mark.parametrize("D", [256, 4096])
def test_fused_de_trial_curves_build_the_same_tables(D):
    """cl_de_trial_curves(_wide): the curves and tables of the drawn trial vectors, bit for bit."""
    rng = np.random.default_rng(D)
    x, q = _basis(D)
    t = np.array([0.01, 0.02, 0.04])
    dn = _stack(rng, D, 300, t, dtype=np.uint8 if D <= 256 else np.uint16)
    lo, hi = 5 * D // 256, 250 * D // 256
    ev_params = np.zeros((40, 5))
    plan = _plan(dn, None, t, x ** 2.2, q, lo, hi, ev_params)
    unit = torch.from_numpy(rng.random((40, 5))).cuda()
    de = ops.DeviceDE.for_plan(plan, [-0.2] * 5, [0.2] * 5, unit, seed=3, tol=0.0)
    de.step_fused()
    torch.cuda.synchronize()
    params = host(plan.params)
    v = ref_curves(x ** 2.2, q, params)
    ok = ref_gates(v)
    assert ok.sum() > 5
    assert _same_bits(host(plan.curves), v)
    assert np.array_equal(host(plan.valid) != 0, ok)
    assert _same_bits(host(plan.tables).view(np.float64), ref_tables(v, ok, lo, hi))


@pytest.mark.parametrize("D", [256, 65536])
def test_pow_parametrisation_within_two_ulps(D):
    """linspace ** p[0] with a zero basis: the curve is the device pow itself (no shift: pow(1, p) = 1)."""
    mpmath = pytest.importorskip("mpmath")
    mpmath.mp.prec = 120
    pca = np.zeros((D, 2))
    params = np.zeros((32, 3))
    params[:, 0] = np.linspace(0.3, 3.1, 32)
    dtype = np.uint8 if D <= 256 else np.uint16
    plan = ops.IcrfEnergyPlan(dev(np.zeros((1, 1, 2), dtype)), None, [0.01, 0.02], None, dev(pca), 1, D - 1, False, 32)
    plan.set_params(torch.from_numpy(params))
    plan.curves_and_tables()
    c = host(plan.curves)
    xs = np.arange(D) * (1.0 / (D - 1))
    xs[-1] = 1.0
    pts = np.unique(np.r_[1:min(D, 300), np.linspace(1, D - 1, 700).astype(int)])
    for s in (0, 5, 13, 31):
        p = params[s, 0]
        for d in pts:
            want = float(mpmath.power(mpmath.mpf(float(xs[d])), mpmath.mpf(float(p))))
            got = c[s, d]
            assert abs(got - want) <= 2 * np.spacing(want), (s, d, got, want)
        assert c[s, 0] == 0.0


# ---- layer 2: pair sums --------------------------------------------------------------------------------------
def _warps(N, global_tables):
    return (16 if N <= 5 else 8) if global_tables else (16 if N <= 6 else 8)


def ref_pair_sums(curves, dn, sd, t, lower, upper, global_tables, sms, n_candidates, masked_term=True):
    """Exact-reference pair sums (S, P, 2) in long double and their per-case error bounds (S, P, 2).  Without
    ``masked_term`` the bound leaves out the masked 1.0s that the uniform no-std loop adds and subtracts again."""
    S = curves.shape[0]
    n_px, N = dn.shape
    P = N * (N - 1) // 2
    pairs = [(i, j) for i in range(N) for j in range(i + 1, N)]
    uni = uniform(lower, upper)
    # chain length: pixels per warp (+ subtraction), warp tree, lane-strided CTA sum, xor tree
    groups = n_candidates // 32
    chunks = max(1, (2 if global_tables else 1) * sms // groups)
    if chunks * 128 > n_px:
        chunks = max(1, -(-n_px // 128))
    per_cta = -(-n_px // chunks)
    L = -(-per_cta // _warps(N, global_tables)) + 1 + 4 + -(-chunks // 32) + 5 + 2
    tl = t.astype(LD)
    ref = np.zeros((S, P, 2), LD)
    bnd = np.zeros((S, P, 2))
    for s in range(S):
        v = curves[s]
        lo, hi = v[lower], v[upper]
        with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
            I = v[dn].astype(LD)                                 # (n_px, N)
            inr = (dn >= lower) & (dn <= upper) if uni else ~((v[dn] < lo) | (v[dn] > hi))
            for q, (i, j) in enumerate(pairs):
                both = inr[:, i] & inr[:, j]
                uij = (I[:, i] * tl[j]) / (tl[i] * I[:, j])
                a = np.abs(uij - 1)
                if sd is None:
                    take = both & ~np.isnan(a)
                    terms = np.where(take, a, 0)
                    ref[s, q, 0] = terms.sum()
                    ref[s, q, 1] = take.sum()
                    e_term = float(np.where(take, LD(4.1 * U) * np.abs(uij) + LD(1.1 * U) * a, 0).sum())
                    absum = float(terms.sum())
                    if uni and masked_term:
                        absum += 2.0 * (n_px - both.sum())           # the masked 1.0s and their subtraction
                    bnd[s, q, 0] = e_term + U * L * absum
                else:
                    si, sj = sd[:, i].astype(LD), sd[:, j].astype(LD)
                    var = (si * tl[j] / (tl[i] * I[:, j])) ** 2 + (uij * sj / I[:, j]) ** 2
                    take = both & np.isfinite(a) & (var > 0)
                    var = np.where(take, var, 1)
                    w = np.where(take, 1 / np.sqrt(var), 0)
                    at = np.where(take, a, 0)
                    ref[s, q, 0] = (at * w).sum()
                    ref[s, q, 1] = w.sum()
                    # var: 18 roundings relative, plus three on the subnormal grid (t1^2, t2^2, the fma) when the
                    # variance is subnormal; rsqrt within 1 ulp
                    w_rel = (18 * U + 3 * LD(2.0 ** -1074) / var) / 2 + LD(2.1 * U)
                    e_a = LD(5.1 * U) * np.where(take, np.abs(uij), 0) + LD(1.1 * U) * at
                    bnd[s, q, 0] = float((e_a * w + at * w * w_rel).sum() + U * L * (at * w).sum())
                    bnd[s, q, 1] = float((w * w_rel).sum() + U * L * w.sum())
    return ref, bnd


def ref_energy_of(acc, valid):
    """energy_of, operation for operation."""
    out = np.empty(acc.shape[0])
    for s in range(acc.shape[0]):
        if not valid[s]:
            out[s] = np.inf
            continue
        tot, cnt = 0.0, 0
        for q in range(acc.shape[1]):
            num, den = acc[s, q]
            if den == 0.0:
                continue
            with np.errstate(all="ignore"):
                r = num / den
            if r != r:
                continue
            tot += r
            cnt += 1
        e = tot / cnt if cnt else np.inf
        out[s] = np.inf if e != e else e
    return out


def _check(dn, sd, t, lower, upper, S=32, D=256, dtype=np.uint8, seed=0, params=None, mean=None, pca=None,
           bar=TIGHT, masked_term=True):
    """Runs both tails on one problem and checks all three layers.  Returns (max relative error of the energies,
    their largest derived bound)."""
    rng = np.random.default_rng(seed)
    if pca is None:
        x, pca = _basis(D)
        mean = x ** 2.2
    if params is None:
        params = rng.uniform(-0.04, 0.04, (S, pca.shape[1]))
        params[S // 2, 2] = 3.0                             # gated next to valid ones
    dn = dn.astype(dtype)
    plan = _plan(dn, sd, t, mean, pca, lower, upper, params)
    Sp = plan.prob.n_candidates
    curves, valid = host(plan.curves), host(plan.valid)
    allp = np.vstack([params, np.zeros((Sp - params.shape[0], pca.shape[1]))])
    v = ref_curves(mean, pca, allp)
    assert _same_bits(curves, v)
    assert np.array_equal(valid != 0, ref_gates(v))
    assert _same_bits(host(plan.tables).view(np.float64), ref_tables(v, valid != 0, lower, upper, sd is not None))
    acc = host(plan.partial()).copy()
    e_split = host(plan.finalize()).copy()
    e_fused = host(plan.population()).copy()
    acc_fused = host(plan.pair_acc).copy()
    # layer 3: the fused tail is the same reduction, finalize is energy_of
    assert np.array_equal(acc_fused.view(np.int64), acc.view(np.int64))
    assert np.array_equal(e_fused.view(np.int64), e_split.view(np.int64))
    assert np.array_equal(e_split.view(np.int64), ref_energy_of(acc, valid)[: params.shape[0]].view(np.int64))
    assert np.array_equal(host(plan.population()).view(np.int64), e_fused.view(np.int64))     # repeat run
    # layer 2: live candidates' pair sums against the long-double reference
    live = np.nonzero(valid[: params.shape[0]])[0]
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    ref, bnd = ref_pair_sums(curves[live], dn, sd, t, lower, upper, D > 256, sms, Sp, masked_term)
    got = acc[live]
    if sd is None:
        assert np.array_equal(got[..., 1], ref[..., 1].astype(np.float64)), "valid counts"
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(got), fin)
    err = np.abs(got.astype(LD) - ref).astype(np.float64)
    assert (err[fin] <= bnd[fin] + 1e-300).all(), float(np.max(err[fin] - bnd[fin]))
    # energies: nanmean of num / den over the pairs; bound from the pair-sum bounds
    with np.errstate(all="ignore"):
        r = ref[..., 0] / ref[..., 1]
        abs_q = (bnd[..., 0] + np.abs(r) * bnd[..., 1]) / ref[..., 1] + U * np.abs(r)     # of each num / den
    keep = (ref[..., 1] > 0) & ~np.isnan(r)
    P = ref.shape[1]
    e_ref = np.array([r[k][keep[k]].mean() if keep[k].any() else np.inf for k in range(len(live))])
    with np.errstate(all="ignore"):                          # the ratios are >= 0: their errors add up
        e_bnd = np.array([float(abs_q[k][keep[k]].sum() / r[k][keep[k]].sum()) + (P + 2) * U
                          if keep[k].any() else 0.0 for k in range(len(live))])
    e_got = e_split[live]
    assert np.array_equal(np.isinf(e_got), np.isinf(e_ref.astype(np.float64)))
    f = np.isfinite(e_ref) & (e_ref != 0)
    rel = (np.abs(e_got[f].astype(LD) - e_ref[f]) / np.abs(e_ref[f])).astype(np.float64)
    assert (rel <= e_bnd[f]).all()
    if bar is not None:
        assert (e_bnd[f] <= bar).all(), float(e_bnd[f].max())
    gated = np.nonzero(valid[: params.shape[0]] == 0)[0]
    assert np.isinf(e_split[gated]).all()
    return (float(rel.max()) if rel.size else 0.0), (float(e_bnd[f].max()) if f.any() else 0.0)


KINDS = {"u8": (np.uint8, 256), "u16_shared": (np.uint16, 256), "u16_global": (np.uint16, 4096)}


@pytest.mark.parametrize("kind", list(KINDS))
@pytest.mark.parametrize("lower0", [False, True])
@pytest.mark.parametrize("use_std", [False, True])
@pytest.mark.parametrize("N", [2, 3, 4, 5, 6, 7, 8])
def test_every_partial_instance(N, use_std, lower0, kind):
    dtype, D = KINDS[kind]
    rng = np.random.default_rng(N * 7 + use_std + 2 * lower0)
    t = 0.004 * 1.7 ** np.arange(N)
    dn = _stack(rng, D, 16 * 37 + 5, t, dtype=dtype)
    if lower0:
        dn[::9, 0] = 0                                       # DN 0: 0 / 0 skipped, x / 0 = inf kept
    sd = rng.uniform(0.002, 0.02, dn.shape) if use_std else None
    lo, hi = (0, D - 1) if lower0 else (5 * D // 256, 250 * D // 256)
    _check(dn, sd, t, lo, hi, S=32, D=D, dtype=dtype, seed=N)


@pytest.mark.parametrize("n_px", [1, 7, 15, 16 * 3, 16 * 31, 128 * 5 + 37, 148 * 128 + 19, 60_000])
@pytest.mark.parametrize("use_std", [False, True])
def test_pixel_counts(n_px, use_std):
    """1, fewer than WARPS, odd multiples of WARPS (the two-pixel loop ends on one pixel), counts that do not divide
    by the number of chunks, and many CTAs (~50 pixels per warp at 60 000; test_mostly_masked_stack_near_the_optimum
    runs ~320)."""
    rng = np.random.default_rng(n_px)
    t = 0.005 * 2.0 ** np.arange(5)
    dn = _stack(rng, 256, n_px, t)
    sd = rng.uniform(0.002, 0.02, dn.shape) if use_std else None
    _check(dn, sd, t, 5, 250, S=64 if n_px > 10_000 else 32, seed=1)


@pytest.mark.parametrize("S", [32, 45, 64, 96])
def test_candidate_counts(S):
    rng = np.random.default_rng(S)
    t = 0.005 * 2.0 ** np.arange(4)
    dn = _stack(rng, 256, 3000, t)
    _check(dn, None, t, 5, 250, S=S, seed=S)
    _check(dn, rng.uniform(0.002, 0.02, dn.shape), t, 5, 250, S=S, seed=S)


@pytest.mark.parametrize("limits", ["equal", "lower1", "upper_last", "swapped"])
@pytest.mark.parametrize("use_std", [False, True])
def test_data_limits(limits, use_std):
    rng = np.random.default_rng(3)
    t = 0.005 * 2.0 ** np.arange(4)
    dn = _stack(rng, 256, 4000, t)
    dn[::3] = 128                                            # lower == upper == 128: these pixels' pairs count
    sd = rng.uniform(0.002, 0.02, dn.shape) if use_std else None
    lo, hi = {"equal": (128, 128), "lower1": (1, 250), "upper_last": (5, 255), "swapped": (200, 50)}[limits]
    _check(dn, sd, t, lo, hi, seed=4)


@pytest.mark.parametrize("use_std", [False, True])
def test_swapped_limits_mask_every_sample(use_std):
    """1 <= upper < lower: every sample of a candidate that passes the gates is masked -> +inf and empty pairs."""
    rng = np.random.default_rng(5)
    x, q = _basis(256)
    t = 0.005 * 2.0 ** np.arange(5)
    dn = _stack(rng, 256, 2000, t)
    params = rng.uniform(-0.03, 0.03, (32, 5))
    plan = _plan(dn, rng.uniform(0.002, 0.02, dn.shape) if use_std else None, t, x ** 2.2, q, 200, 50, params)
    e = host(plan.population())
    assert host(plan.valid).sum() > 10
    assert np.isinf(e).all()
    assert not host(plan.pair_acc)[..., 1].any()


@pytest.mark.parametrize("eps", [1e-4, 1e-6, 1e-8])
def test_mostly_masked_stack_near_the_optimum(eps):
    """92 % of the pixels dark (outside the limits), the rest generated exactly by the linear curve, ~320 pixels per
    warp, the live candidates within eps of that curve: |d| ~ eps.  The uniform no-std loop adds 1.0 for every masked
    pair and subtracts the count at the end, so without std the case is held to the bound that counts those 1.0s
    (DESIGN §3: a finding).  With std the masked pairs add exact zeros: held to the bound of the valid terms alone.
    Neither is held to 1e-11: with |d| down to a fraction of eps the per-term conditioning (~5u / |d|, shared by every
    double evaluation, NumPy's included) makes each case's own bound larger than that at every eps here."""
    rng = np.random.default_rng(int(-np.log10(eps)))
    x, q = _basis(256)
    t = np.array([1.0, 2.0, 4.0])
    n = torch.cuda.get_device_properties(0).multi_processor_count * 16 * 320      # one CTA per SM at S = 32
    m = rng.integers(16, 64, n)
    dn = np.stack([m, 2 * m, 4 * m], axis=1)
    dark = rng.random(n) < 0.92
    dn[dark] = rng.integers(0, 8, (dark.sum(), 1)) * np.array([1, 2, 1])
    params = eps * rng.uniform(-1, 1, (32, 5))
    params[6:, 0] = np.nan                                  # gated: keeps the long-double reference small
    rel, b = _check(dn, None, t, 16, 255, params=params, mean=x, pca=q, bar=None)
    print(f"\neps={eps:g} no std: max relative error {rel:.3g}, bound {b:.3g}")
    sd = rng.uniform(0.002, 0.02, dn.shape)                 # masked pairs add exact zeros here
    rel, b = _check(dn, sd, t, 16, 255, params=params, mean=x, pca=q, bar=None, masked_term=False)
    print(f"eps={eps:g} std: max relative error {rel:.3g}, bound {b:.3g}")


WILD = ["zero_some", "zero_all", "nan", "negative", "inf", "tiny_inside", "tiny_outside", "huge_inside", "huge_outside",
        "denormal_scale"]


def _wild_case(kind):
    rng = np.random.default_rng(100 + WILD.index(kind))
    t = 0.005 * 2.0 ** np.arange(4)
    n = 148 * 128 * 4
    dn = _stack(rng, 256, n, t)
    sd = rng.uniform(0.002, 0.02, dn.shape)
    blk = slice(n // 2, n // 2 + 100)                        # inside one CTA among ordinary ones
    if kind == "zero_some":
        sd[blk, 1] = 0.0
    elif kind == "zero_all":
        sd[blk] = 0.0
    elif kind == "nan":
        sd[blk, 2] = np.nan
    elif kind == "negative":
        sd[blk, 0] = -0.01
    elif kind == "inf":
        sd[blk, 3] = np.inf
        sd[blk.start + 1, 2] = -np.inf
    elif kind == "tiny_inside":
        sd[blk] = 2.0 ** -332
    elif kind == "tiny_outside":
        sd[blk] = np.nextafter(2.0 ** -332, 0)
    elif kind == "huge_inside":
        sd[blk, 1] = np.nextafter(2.0 ** 332, 0)
    elif kind == "huge_outside":
        sd[blk, 1] = 2.0 ** 332
    elif kind == "denormal_scale":
        sd[blk] = 1e-160
    return dn, sd, t


@pytest.mark.parametrize("kind", WILD)
def test_wild_prescan(kind):
    """A subnormal variance keeps only a few significant bits in any double evaluation, NumPy's included: the
    denormal-scale case is held to its own bound, which carries three roundings on the subnormal grid."""
    dn, sd, t = _wild_case(kind)
    _check(dn, sd, t, 5, 250, S=32, seed=2, bar=None if kind == "denormal_scale" else TIGHT)


@pytest.mark.parametrize("ratio", ["inside", "outside"])
def test_exposure_ratio_window(ratio):
    rng = np.random.default_rng(9)
    big = 1e50 if ratio == "inside" else np.nextafter(1e50, np.inf)
    t = np.array([1.0, 2.0, big])
    dn = rng.integers(6, 250, (3000, 3))
    sd = rng.uniform(0.002, 0.02, dn.shape)
    sd[::11] = 1e-160                                        # denormal variances only the exact routine weighs
    _check(dn, sd, t, 5, 250, seed=9)


def test_subnormal_curve_value_inside_the_limits():
    """A candidate whose curve[lower] is subnormal: 1/v overflows.  Compared in class (NaN / inf) with the long-double
    reference and held to its bound on the other candidates."""
    D = 256
    x, q = _basis(D)
    mean = x.copy()
    mean[1] = 5e-310
    t = 0.005 * 2.0 ** np.arange(3)
    rng = np.random.default_rng(12)
    dn = rng.integers(1, 250, (2000, 3))
    dn[::7, 2] = 1
    params = np.zeros((32, 5))                                # candidate 0: the mean itself, curve[1] = 5e-310
    params[1:, 4] = np.linspace(1e-4, 3e-4, 31)
    sd = rng.uniform(0.002, 0.02, dn.shape)
    _check(dn, sd, t, 1, 250, params=params, mean=mean, pca=q, bar=None)


def test_partial_op_rejects_digital_numbers_without_a_curve_row():
    x, q = _basis(64)
    params = torch.zeros((32, 5), dtype=torch.float64, device="cuda")
    co = torch.ops.camera_linearity
    curves, valid, tables = co.icrf_energy_curves(params, dev(x), dev(q), 1, 60, 2, False)
    for dtype in (torch.uint8, torch.uint16):
        dn = torch.full((10, 2), 63, dtype=dtype, device="cuda")
        co.icrf_energy_partial(tables, dn, None, [0.01, 0.02], 32, 5, 64, True, 1, 60)
        dn[3, 1] = 64
        with pytest.raises(IndexError):
            co.icrf_energy_partial(tables, dn, None, [0.01, 0.02], 32, 5, 64, True, 1, 60)


def test_finalize_skips_empty_and_nan_pairs():
    """icrf_energy_finalize on crafted sums: den == 0 with num != 0 is skipped (an empty pair is NaN for nanmean),
    a NaN ratio is skipped, no pair left or a gate gives +inf, an infinite ratio is kept."""
    rng = np.random.default_rng(21)
    acc = rng.uniform(0.1, 2.0, (64, 3, 2))
    acc[0] = [[5.0, 0.0], [1.0, 2.0], [3.0, 4.0]]
    acc[1] = [[0.0, 0.0], [np.nan, 1.0], [2.0, 1.0]]
    acc[2] = [[1.0, 0.0], [0.0, 0.0], [7.0, 0.0]]
    acc[3] = [[np.inf, 1.0], [1.0, 1.0], [1.0, 1.0]]
    valid = np.ones(64, np.int32)
    valid[4] = 0
    e = host(torch.ops.camera_linearity.icrf_energy_finalize(dev(acc), dev(valid), 3))
    assert e[0] == (0.5 + 0.75) / 2 and e[1] == 2.0
    assert np.isinf(e[2]) and np.isinf(e[3]) and np.isinf(e[4])
    assert np.array_equal(e.view(np.int64), ref_energy_of(acc, valid).view(np.int64))


def _kernel_name(name):
    hit = re.search(r"(curves_wide_kernel|curves_kernel|reduce_ctas_kernel|finalize_kernel|energy_tail_kernel|"
                    r"energy_partial_kernel<[^>]*>)", name)
    return re.sub(r"\s+", "", hit.group(1)) if hit else None


def _partial_name(N, std, uni, dtype, global_tables):
    dn = "unsignedchar" if dtype == np.uint8 else "unsignedshort"
    b = lambda f: "true" if f else "false"
    return f"energy_partial_kernel<{N},{b(std)},{_warps(N, global_tables)},{b(uni)},{dn},{b(global_tables)}>"


def test_dispatch_map():
    """For each path: curves or curves_wide, the partial instance (N, std, warps, uniform masks, DN type, table
    location), then reduce + finalize, or the fused tail.  The whole sequence runs twice in one profiler session and
    the second pass must match exactly; of the first, the profiler may miss a leading part (with many modules loaded
    it starts tracing late), so it only has to be a suffix of the sequence."""
    rng = np.random.default_rng(0)
    runs = []
    for N in (2, 5, 6, 7, 8):
        for std in (False, True):
            for lower in (0, 5, "swapped"):
                for kind, (dtype, D) in KINDS.items():
                    t = 0.005 * 1.5 ** np.arange(N)
                    dn = _stack(rng, D, 300, t, dtype=dtype)
                    sd = rng.uniform(0.002, 0.02, dn.shape) if std else None
                    lo, hi = (D - 10, 5) if lower == "swapped" else (lower, D - 6)
                    plan = _plan(dn, sd, t, np.linspace(0, 1, D) ** 2.2, _basis(D)[1], lo, hi,
                                 rng.uniform(-0.03, 0.03, (32, 5)))
                    curve = "curves_wide_kernel" if D > 256 else "curves_kernel"
                    part = _partial_name(N, std, uniform(lo, hi), dtype, D > 256)
                    runs.append((plan, [curve, part, "reduce_ctas_kernel", "finalize_kernel", curve, part,
                                        "energy_tail_kernel"]))
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(2):
            for plan, _ in runs:
                plan.curves_and_tables()
                plan.partial()
                plan.finalize()
                plan.curves_and_tables()
                plan.population()
            torch.cuda.synchronize()
    events = sorted(prof.events(), key=lambda e: e.time_range.start)
    if not events:
        pytest.skip("the profiler records no device activity here")
    got = [n for n in (_kernel_name(e.name) for e in events) if n]
    want = [k for _, seq in runs for k in seq]
    assert got[-len(want):] == want
    first = got[: len(got) - len(want)]
    assert len(first) <= len(want) and first == want[len(want) - len(first):]
