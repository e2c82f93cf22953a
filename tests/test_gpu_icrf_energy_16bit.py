"""K4 for 16-bit (and 12-bit) cameras: uint16 samples and curves of up to 65536 points -- the cluster-built curves
and the partial kernel that gathers its tables from global memory -- against the oracle (``bits=D``), the uint8 path
and the unfused DE generation."""
import numpy as np
import pytest
import torch

from oracle import icrf_energy as oe
from gpu_util import assert_rel, host

pytestmark = pytest.mark.gpu
ops = pytest.importorskip("camera_linearity_b200.ops")
import camera_linearity_b200 as cl  # noqa: E402
from camera_linearity_b200 import ICRF_calibration_exposure as cal  # noqa: E402
from camera_linearity_b200.settings import GlobalSettings as gs  # noqa: E402

TIGHT = 1e-11
CLUSTER = 8                       # CTAs per candidate of the D > 256 curve kernel


def _basis(D):
    x = np.linspace(0, 1, D)
    q, _ = np.linalg.qr(np.stack([np.sin((k + 1) * np.pi * x) * x for k in range(5)], axis=1))
    return x, q


def _stack(rng, D, shape, t, gamma=1 / 2.2):
    rad = rng.uniform(0, 1, shape + (1,)) * 25
    return np.rint((D - 1) * np.clip(rad * t[None, None, :], 0, 1) ** gamma).astype(np.uint16)


def _oracle_curve(mean, pca, p):
    c = oe.candidate_curve(mean, pca, p, True, len(mean))
    c += 1 - c[-1]
    c[0] = 0
    return c


@pytest.mark.parametrize("D", [4096, 65536])
@pytest.mark.parametrize("n_exp", [2, 3, 5, 8])
@pytest.mark.parametrize("use_std", [False, True])
def test_energies_against_the_oracle(D, n_exp, use_std):
    rng = np.random.default_rng(D + n_exp)
    x, q = _basis(D)
    mean = x ** 2.2
    t = 0.004 * 1.9 ** np.arange(n_exp)
    dn = _stack(rng, D, (37, 23), t)
    sd = rng.uniform(0.002, 0.02, dn.shape) if use_std else None
    s = 40 + n_exp                                           # not a multiple of 32: padded internally
    params = rng.uniform(-0.04, 0.04, (5, s))
    params[:, 3] = [0, 0, 0, 0, 3.0]                          # gated
    lo, hi = 5 * D // 256, 250 * D // 256
    want = oe.energy_population(params, mean, q, dn, sd, lo, hi, True, t, bits=D)
    got = cl.EnergyEvaluator(mean, q, dn, sd, lo, hi, True, t, s)(params)
    assert np.isinf(want[3]) and np.isfinite(want).sum() > s // 2
    assert np.array_equal(np.isinf(got), np.isinf(want))
    assert_rel(got, want, TIGHT)


@pytest.mark.parametrize("D", [4096, 65536])
@pytest.mark.parametrize("use_std", [False, True])
def test_lower_zero_takes_the_nan_checking_path(D, use_std):
    rng = np.random.default_rng(7)
    x, q = _basis(D)
    t = 0.004 * 1.9 ** np.arange(4)
    dn = _stack(rng, D, (40, 30), t)
    dn[::5, ::3, 0] = 0                                        # DN 0: 0 / 0 pairs are skipped, x / 0 = inf kept
    sd = rng.uniform(0.002, 0.02, dn.shape) if use_std else None
    params = rng.uniform(-0.04, 0.04, (5, 33))
    with np.errstate(all="ignore"):
        want = oe.energy_population(params, x ** 2.2, q, dn, sd, 0, D - 1, True, t, bits=D)
    got = cl.EnergyEvaluator(x ** 2.2, q, dn, sd, 0, D - 1, True, t, 33)(params)
    assert np.array_equal(np.isinf(got), np.isinf(want))
    fin = np.isfinite(want)
    assert_rel(got[fin], want[fin], TIGHT)


def test_exponent_parametrisation_uses_device_pow():
    rng = np.random.default_rng(5)
    D = 65536
    x, q = _basis(D)
    t = 0.005 * 2.0 ** np.arange(5)
    dn = _stack(rng, D, (50, 40), t)
    params = np.vstack([rng.uniform(1.8, 2.6, 36), rng.uniform(-0.04, 0.04, (5, 36))])
    want = oe.energy_population(params, None, q, dn, None, 1285, 64250, False, t, bits=D)
    got = cl.EnergyEvaluator(None, q, dn, None, 1285, 64250, False, t, 36)(params)
    assert np.isfinite(want).sum() > 18
    assert np.array_equal(np.isinf(got), np.isinf(want))
    assert_rel(got, want, 1e-9)


def _cfg3_16(seed):
    rng = np.random.default_rng(seed)
    D = 65536
    x, q = _basis(D)
    t = 0.005 * 2.0 ** np.arange(5)
    dn = _stack(rng, D, (1000, 400), t)
    return rng, x ** 2.2, q, t, dn


@pytest.mark.parametrize("use_std", [False, True])
def test_cfg3_16_pair_sums_counts_and_oracle(use_std):
    """cfg3-16 size (S=64, 400k px x 5, D = 65536): valid counts exact, whole = sum of two halves, 3 candidates
    against the oracle on the full data."""
    rng, mean, q, t, dn = _cfg3_16(3 + use_std)
    sd = None
    if use_std:
        sd = rng.uniform(0.002, 0.02, dn.shape)
        sd[::97, ::13, 2] = 0.0                   # sigma == 0 -> the pair is skipped
    params = rng.uniform(-0.05, 0.05, (5, 64))
    params[:, 9] = [0, 0, 0, 0, 2.0]              # gated
    lo, hi = 5 * 257, 250 * 257
    whole = cl.EnergyEvaluator(mean, q, dn, sd, lo, hi, True, t, 64, shard=False)
    e = whole(params)
    assert np.isinf(e[9]) and np.isfinite(e).sum() >= 32
    acc = host(whole.plan.pair_acc).copy()
    if not use_std:
        ok = (dn >= lo) & (dn <= hi)              # a valid candidate is strictly increasing: masks by DN alone
        pairs = [(i, j) for i in range(5) for j in range(i + 1, 5)]
        counts = np.array([np.sum(ok[..., i] & ok[..., j]) for i, j in pairs])
        live = np.isfinite(e)
        assert np.array_equal(acc[: 64][live][..., 1], np.broadcast_to(counts, (live.sum(), 10)))
    halves = []
    for rows in (slice(0, 500), slice(500, None)):
        ev = cl.EnergyEvaluator(mean, q, dn[rows], None if sd is None else sd[rows], lo, hi, True, t, 64, shard=False)
        ev(params)
        halves.append(host(ev.plan.pair_acc).copy())
    live = np.isfinite(e)
    if not use_std:
        assert np.array_equal(acc[..., 1], halves[0][..., 1] + halves[1][..., 1])
    np.testing.assert_allclose(acc[: 64][live], (halves[0] + halves[1])[: 64][live], rtol=1e-12)
    ref = oe.energy_population(params[:, :3], mean, q, dn, sd, lo, hi, True, t, bits=65536)
    assert_rel(e[:3], ref, TIGHT)


def test_zero_nan_and_denormal_variances_take_the_exact_branch():
    rng = np.random.default_rng(11)
    D = 65536
    x, q = _basis(D)
    t = 0.004 * 1.9 ** np.arange(5)
    dn = _stack(rng, D, (64, 48), t, gamma=0.5)
    sd = rng.uniform(0.002, 0.02, dn.shape)
    sd[::7, ::5, :] = 0.0
    sd[1::7, ::5, 1:3] = 0.0
    sd[2::7, 1::5, :] = 2e-155
    sd[3::7, 2::5, 0] = 5e-155
    sd[4::7, 3::5, 1] = np.nan
    params = rng.uniform(-0.04, 0.04, (5, 37))
    with np.errstate(all="ignore"):
        want = oe.energy_population(params, x ** 2.0, q, dn, sd, 1285, 64250, True, t, bits=D)
    got = cl.EnergyEvaluator(x ** 2.0, q, dn, sd, 1285, 64250, True, t, 37)(params)
    assert np.isfinite(want).any()
    assert np.array_equal(np.isinf(got), np.isinf(want))
    assert_rel(got, want, 1e-9)


@pytest.mark.parametrize("D", [4096, 65536])
def test_curves_and_gates_including_a_step_across_a_cta_boundary(D):
    """plan.curves against the oracle's curve; `valid` against the oracle's gates.  Column 0 of the basis is a spike
    at the first point of the second CTA of the cluster, so the candidate with a large coefficient fails the
    monotonicity gate only across that boundary."""
    x, q = _basis(D)
    mean = x ** 2.2
    b = (D + CLUSTER - 1) // CLUSTER
    pca = q.copy()
    pca[:, 0] = 0.0
    pca[b, 0] = -1.0
    step = mean[b] - mean[b - 1]
    rng = np.random.default_rng(D)
    params = rng.uniform(-0.03, 0.03, (5, 40))
    params[0] = 0.0
    params[0, 1] = 1.5 * step                     # curve[b] < curve[b - 1]: gated by the cross-boundary step only
    params[0, 2] = 0.5 * step                     # a smaller dip: still strictly increasing
    params[0, 3] = 1.5 * step
    params[1:, 3] = [0, 0, 0, 3.0]                # gated by oscillation everywhere
    dn = _stack(rng, D, (16, 16), np.array([0.01, 0.02, 0.04]))
    ev = cl.EnergyEvaluator(mean, pca, dn, None, 5 * D // 256, 250 * D // 256, True, [0.01, 0.02, 0.04], 40)
    e = ev(params)
    curves, valid = host(ev.plan.curves), host(ev.plan.valid)
    for s in range(40):
        c = _oracle_curve(mean, pca, params[:, s])
        assert np.max(np.abs(curves[s] - c)) <= 1e-14, s
        steps = np.diff(c)
        if np.min(np.abs(steps)) > 1e-12 and np.all(np.abs(c[:-1] - 1) > 1e-12) and np.all(np.abs(c[1:]) > 1e-12):
            gate = bool(np.all(steps > 0) and c.max() <= 1 and c.min() >= 0)
            assert bool(valid[s]) == gate, s
    assert valid[1] == 0 and valid[2] == 1 and valid[3] == 0
    assert np.isinf(e[1]) and np.isfinite(e[2]) and np.isinf(e[3])
    curve1 = _oracle_curve(mean, pca, params[:, 1])
    bad = np.nonzero(np.diff(curve1) <= 0)[0]
    assert list(bad) == [b - 1]                   # the only failing step crosses the CTA boundary


def test_uint8_and_uint16_at_256_points_are_bit_identical():
    rng = np.random.default_rng(2)
    x, q = _basis(256)
    t = 0.005 * 2.0 ** np.arange(5)
    dn8 = _stack(rng, 256, (80, 60), t).astype(np.uint8)
    sd = rng.uniform(0.002, 0.02, dn8.shape)
    params = rng.uniform(-0.05, 0.05, (5, 50))
    for std in (None, sd):
        a = cl.EnergyEvaluator(x ** 2.2, q, dn8, std, 5, 250, True, t, 50)
        b = cl.EnergyEvaluator(x ** 2.2, q, dn8.astype(np.uint16), std, 5, 250, True, t, 50)
        assert b.plan.wide and not a.plan.wide
        ea, eb = a(params), b(params)
        assert np.array_equal(ea, eb)
        assert torch.equal(a.plan.pair_acc, b.plan.pair_acc)


def test_repeat_runs_are_bit_identical():
    rng, mean, q, t, dn = _cfg3_16(8)
    dn = dn[:200]
    sd = rng.uniform(0.002, 0.02, dn.shape)
    params = rng.uniform(-0.05, 0.05, (5, 64))
    ev = cl.EnergyEvaluator(mean, q, dn, sd, 1285, 64250, True, t, 64, shard=False)
    first = ev(params)
    acc = ev.plan.pair_acc.clone()
    for _ in range(3):
        assert np.array_equal(ev(params), first)
        assert torch.equal(ev.plan.pair_acc, acc)


def test_digital_numbers_beyond_the_curve_raise():
    x, q = _basis(4096)
    t = np.array([0.01, 0.02])
    dn = np.zeros((4, 4, 2), np.uint16)
    dn[1, 1, 1] = 40000                           # above 32767: an int16 view would make it negative
    with pytest.raises(IndexError):
        cl.EnergyEvaluator(x, q, dn, None, 5, 250, True, t, 1)
    dn[1, 1, 1] = 4096
    with pytest.raises(IndexError):
        cl.EnergyEvaluator(x, q, dn, None, 5, 250, True, t, 1)
    dn[1, 1, 1] = 4095
    cl.EnergyEvaluator(x, q, dn, None, 5, 250, True, t, 1)
    with pytest.raises(TypeError):
        ops.IcrfEnergyPlan(torch.zeros((4, 4, 2), dtype=torch.float32, device="cuda"), None, t, x,
                           torch.as_tensor(q, device="cuda"), 5, 250, True, 1)


def _camera16():
    D = 65536
    x = np.linspace(0, 1, D)
    mean = x ** 2.2
    pca = np.stack([0.1 * np.sin((k + 1) * np.pi * x) for k in range(5)], axis=1)
    p_true = np.array([0.12, -0.05, 0.03, 0.0, 0.01])
    curve = mean + pca @ p_true
    curve = curve + (1 - curve[-1])
    curve[0] = 0
    assert np.all(np.diff(curve) > 0)
    rng = np.random.default_rng(11)
    t = np.array([.005, .01, .02, .04, .08])
    rad = rng.uniform(0.5, 14, (64, 48, 1))
    # 1 % shot noise per exposure: at 16 bits the quantisation alone leaves the true curve an energy of ~4e-5, a
    # minimum too sharp for the DE's 1 % convergence test; with the noise it is ~1e-2, as for the 8-bit camera
    target = np.clip(rad * t[None, None, :] * rng.normal(1.0, 0.01, (64, 48, 5)), 0, 1)
    dn = np.minimum(np.searchsorted(curve, target), D - 1).astype(np.uint16)     # the camera's CRF
    return mean, pca, p_true, curve, dn, t


def test_fused_generation_and_cuda_graph_match_the_unfused_steps():
    from scipy.stats import qmc
    mean, pca, p_true, curve, dn, t = _camera16()
    lo, hi = 5 * 257, 250 * 257
    unit = torch.from_numpy(qmc.Sobol(d=5, seed=np.random.default_rng(9)).random(n=64)).cuda()
    ev_a = cl.EnergyEvaluator(mean, pca, dn, None, lo, hi, True, t, 64, shard=False)
    de_a = ops.DeviceDE(ev_a.device_energies, [-0.5] * 5, [0.5] * 5, unit, seed=9, tol=0.0)
    ev_b = cl.EnergyEvaluator(mean, pca, dn, None, lo, hi, True, t, 64, shard=False)
    de_b = ops.DeviceDE.for_plan(ev_b.plan, [-0.5] * 5, [0.5] * 5, unit, seed=9, tol=0.0)
    assert torch.equal(de_a.pop, de_b.pop) and torch.equal(de_a.energies, de_b.energies)
    for _ in range(24):
        de_a.step()
    de_b.run_graph(24, per_graph=8)
    torch.cuda.synchronize()
    assert torch.equal(de_a.pop, de_b.pop) and torch.equal(de_a.energies, de_b.energies)
    assert torch.equal(de_a.trial, de_b.trial) and torch.equal(ev_a.plan.params, ev_b.plan.params)
    assert de_a.poll()[1] == de_b.poll()[1] == 24
    rng = np.random.default_rng(4)
    sd = rng.uniform(0.002, 0.02, dn.shape)
    unit40 = unit[:40].clone()
    ev_c = cl.EnergyEvaluator(mean, pca, dn, sd, lo, hi, True, t, 40, shard=False)
    de_c = ops.DeviceDE(ev_c.device_energies, [-0.5] * 5, [0.5] * 5, unit40, seed=3, tol=0.0)
    ev_d = cl.EnergyEvaluator(mean, pca, dn, sd, lo, hi, True, t, 40, shard=False)
    de_d = ops.DeviceDE.for_plan(ev_d.plan, [-0.5] * 5, [0.5] * 5, unit40, seed=3, tol=0.0)
    for _ in range(8):
        de_c.step()
    de_d.run_graph(8, per_graph=8)
    for _ in range(16):
        de_c.step()
        de_d.step_fused()
    assert torch.equal(de_c.pop, de_d.pop) and torch.equal(de_c.energies, de_d.energies)


def test_both_drivers_recover_a_16bit_camera():
    mean, pca, p_true, curve, dn, t = _camera16()
    limits = [[-0.5, 0.5]] * 5
    x0 = [0.0] * 5
    lo, hi = 5 * 257, 250 * 257
    e_true = oe.energy(p_true, mean, pca, dn, None, lo, hi, True, t, bits=65536)
    for driver in ("scipy", "device"):
        c, p, e, it = cal.solve_channel(mean, pca, dn, None, t, limits, x0, data_limits=(lo, hi), seed=5,
                                        max_iterations=400, driver=driver)
        c = c + (1 - c[-1])
        assert e <= e_true * 1.05 + 1e-12, (driver, e, e_true)
        assert np.max(np.abs(c - curve)) < 5e-3, driver


def test_custom_op_chain_on_uint16_matches_the_evaluator():
    rng = np.random.default_rng(6)
    D = 65536
    x, q = _basis(D)
    t = 0.005 * 2.0 ** np.arange(4)
    dn = _stack(rng, D, (30, 20), t)
    sd = rng.uniform(0.002, 0.02, dn.shape)
    params = rng.uniform(-0.04, 0.04, (5, 64))
    want = cl.EnergyEvaluator(x ** 2.2, q, dn, sd, 1285, 64250, True, t, 64)(params)
    co = torch.ops.camera_linearity
    curves, valid, tables = co.icrf_energy_curves(torch.from_numpy(params.T.copy()).cuda(),
                                                  torch.from_numpy(x ** 2.2).cuda(), torch.from_numpy(q).cuda(),
                                                  1285, 64250, 4, True)
    assert curves.shape == (64, D)
    acc = co.icrf_energy_partial(tables, torch.from_numpy(dn.reshape(-1, 4)).cuda(),
                                 torch.from_numpy(sd.reshape(-1, 4)).cuda(), list(t), 64, 5, D, True, 1285, 64250)
    e = co.icrf_energy_finalize(acc, valid, 4)
    assert np.array_equal(host(e), want)


@pytest.fixture
def settings_16bit(tmp_path):
    keys = ("BIT_DEPTH", "BITS", "MAX_DN", "DATAPOINTS", "NUM_OF_CHS", "DATA_PATH", "PCA_FILES", "MEAN_ICRF_FILES",
            "NUM_OF_PCA_PARAMS")
    saved = {k: getattr(gs, k) for k in keys}
    yield tmp_path
    for k, v in saved.items():
        setattr(gs, k, v)


def test_calibration_end_to_end_on_16bit_tiffs(settings_16bit):
    import cv2 as cv
    tmp = settings_16bit
    mean, pca, p_true, curve, _, _ = _camera16()
    rng = np.random.default_rng(21)
    rad = rng.uniform(0.5, 14, (48, 40, 3))
    t_ms = [5, 10, 20, 40, 80]
    images = tmp / "acquired"
    images.mkdir()
    for ms in t_ms:
        target = np.clip(rad * ms / 1000, 0, 1)
        img = np.minimum(np.searchsorted(curve, target), 65535).astype(np.uint16)
        assert cv.imwrite(str(images / f"flat {ms}ms.tif"), img)
    np.savetxt(tmp / "pca.txt", pca)
    np.savetxt(tmp / "mean.txt", mean)
    gs.configure(BIT_DEPTH=16, DATAPOINTS=65536, NUM_OF_CHS=3, DATA_PATH=tmp, NUM_OF_PCA_PARAMS=5,
                 PCA_FILES=["pca.txt"] * 3, MEAN_ICRF_FILES=["mean.txt"] * 3)
    icrf, _, energies, _ = cal.calibration(-0.5, 0.5, data_spacing=1, data_limits=(5 * 257, 250 * 257),
                                           image_path=images, max_iterations=16, driver="device")
    assert icrf.shape == (65536, 3)
    assert np.all(np.isfinite(energies))
    assert icrf.min() >= 0 and icrf.max() <= 1
    assert np.all(np.diff(icrf, axis=0) >= 0)
    assert np.all(icrf[0] == 0)
