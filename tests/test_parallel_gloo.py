"""World-size-2 (gloo, CPU) test of the only collective on the path: the K4 pair sums are
all-reduced, then every rank finalises identically.  Sharding helpers for K1-K3 are checked too."""
import os
import socket
import sys
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

ROOT = Path(__file__).resolve().parents[1]


def pair_sums(curve, lo, hi, dn, std, t):
    """Per-pair (numerator, denominator) on a pixel shard with the oracle's formulae."""
    vals = curve[dn].astype(np.float64)
    vals = np.where((vals < lo) | (vals > hi), np.nan, vals).reshape(-1, dn.shape[-1])
    sd = None if std is None else std.reshape(-1, dn.shape[-1])
    n = dn.shape[-1]
    out = []
    with np.errstate(all="ignore"):
        for i in range(n):
            for j in range(i + 1, n):
                r = t[i] / t[j]
                scaled = vals[:, j] * r
                d = np.abs((vals[:, i] - scaled) / scaled)
                if sd is None:
                    ok = ~np.isnan(d)
                    out.append((d[ok].sum(), float(ok.sum())))
                else:
                    sig = np.sqrt((sd[:, i] / scaled) ** 2 + ((vals[:, i] * sd[:, j]) / (r * vals[:, j] ** 2)) ** 2)
                    ok = np.isfinite(d) & (sig != 0) & ~np.isnan(sig)
                    w = 1 / sig[ok]
                    out.append(((d[ok] * w).sum(), w.sum()))
    return np.array(out)


def _worker(rank, world, port, q):
    sys.path.insert(0, str(ROOT))
    # init_from_env selects the rank's GPU when CUDA is present: with fewer GPUs than ranks they share them
    n_dev = torch.cuda.device_count()
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank % n_dev if n_dev else rank))
    from camera_linearity_b200 import parallel
    from oracle import icrf_energy as oe
    r, w, _ = parallel.init_from_env(backend="gloo")
    assert (r, w) == (rank, world) and parallel.world_size() == world

    rng = np.random.default_rng(7)               # same data on every rank
    x = np.linspace(0, 1, 256)
    mean = x ** 2.2
    pca = np.stack([0.1 * np.sin((k + 1) * np.pi * x) for k in range(5)], axis=1)
    t = 0.005 * 2.0 ** np.arange(4)
    rad = rng.uniform(0, 1, (31, 17, 1)) * 25
    dn = np.rint(255 * np.clip(rad * t[None, None, :], 0, 1) ** (1 / 2.2)).astype(np.uint8)
    std = rng.uniform(0.002, 0.02, dn.shape)
    params = rng.uniform(-0.05, 0.05, (5, 6))
    flat_dn, flat_sd = dn.reshape(-1, 4), std.reshape(-1, 4)
    lo_px, hi_px = parallel.shard_range(flat_dn.shape[0])
    results = {}
    for use_std in (False, True):
        acc = np.zeros((6, 6, 2))
        gated = np.zeros(6, dtype=bool)
        for s in range(6):
            curve = oe.candidate_curve(mean, pca, params[:, s], True)
            curve += 1 - curve[-1]
            curve[0] = 0
            gated[s] = curve.max() > 1 or curve.min() < 0 or not np.all(curve[1:] > curve[:-1])
            acc[s] = pair_sums(curve, curve[5], curve[250], flat_dn[lo_px:hi_px],
                               flat_sd[lo_px:hi_px] if use_std else None, t)
        tensor = torch.from_numpy(acc)
        parallel.allreduce_pair_sums(tensor)     # the one collective of the path
        with np.errstate(all="ignore"):
            ratios = tensor.numpy()[..., 0] / tensor.numpy()[..., 1]
        energy = np.nanmean(ratios, axis=1)
        energy[gated] = np.inf                   # gates are applied after the reduction, on every rank
        expect = oe.energy_population(params, mean, pca, dn, std if use_std else None, 5, 250, True, t)
        results[use_std] = (energy, expect)
    torch.distributed.barrier()
    q.put((rank, lo_px, hi_px, results))
    torch.distributed.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.timeout(300)
def test_pair_sum_allreduce_world_size_2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        out = [q.get(timeout=240) for _ in procs]
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
    finally:                     # a rank left waiting for a failed peer would outlive the test
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join()
    out.sort()
    assert out[0][1] == 0 and out[0][2] == out[1][1] and out[1][2] == 31 * 17      # shards tile the pixels
    for _, _, _, results in out:
        for use_std in (False, True):
            energy, expect = results[use_std]
            np.testing.assert_allclose(energy, expect, rtol=1e-10)
    np.testing.assert_array_equal(out[0][3][True][0], out[1][3][True][0])           # identical on every rank


def test_shard_helpers():
    from camera_linearity_b200 import parallel
    for n in (0, 1, 7, 64, 2161):
        for w in (1, 2, 3, 8):
            spans = [parallel.shard_range(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            assert max(hi - lo for lo, hi in spans) - min(hi - lo for lo, hi in spans) <= 1
    lo, hi, src_lo, src_hi = parallel.shard_rows(2160, halo=1, rank_=3, world=8)
    assert (lo, hi) == (810, 1080) and (src_lo, src_hi) == (809, 1081)
    assert parallel.shard_rows(2160, halo=2, rank_=0, world=8)[2] == 0
    assert parallel.world_size() == 1 and parallel.rank() == 0


def test_numa_binding_is_best_effort_without_a_gpu():
    # no NVML device here: the helper must change nothing and say so
    import os
    from camera_linearity_b200 import parallel
    before = os.sched_getaffinity(0)
    assert parallel.bind_to_gpu_numa_node(0) in (False, True)
    assert os.sched_getaffinity(0) <= before and len(os.sched_getaffinity(0)) >= 1
