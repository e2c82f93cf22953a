"""The two-rank K4 run of test_gpu_multirank.py on a 16-bit problem: uint16 samples, D = 65536 (the cluster-built
curves and the global-table partial kernel) -- pair sums exchanged through peer memory or NCCL exactly as for uint8.
On a one-GPU box both ranks share cuda:0 and the process group is gloo."""
import os
import socket
import sys
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
LO, HI = 5 * 257, 250 * 257


def _problem():
    rng = np.random.default_rng(11)
    x = np.linspace(0, 1, 65536)
    mean = x ** 2.2
    pca, _ = np.linalg.qr(np.stack([np.sin((k + 1) * np.pi * x) * x for k in range(5)], axis=1))
    t = 0.005 * 2.0 ** np.arange(5)
    rad = rng.uniform(0, 1, (301, 211, 1)) * 25
    dn = np.rint(65535 * np.clip(rad * t[None, None, :], 0, 1) ** (1 / 2.2)).astype(np.uint16)
    std = rng.uniform(0.002, 0.02, dn.shape)
    params = rng.uniform(-0.05, 0.05, (5, 40))
    params[:, 5] = [0, 0, 0, 0, 3.0]             # gated candidate: +inf on every rank
    return mean, pca, t, dn, std, params


def _worker(rank, world, port, n_dev, q):
    sys.path.insert(0, str(ROOT))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank % n_dev))
    import camera_linearity_b200 as cl
    from camera_linearity_b200 import _lib, ops, parallel
    from scipy.stats import qmc
    backend = "nccl" if n_dev >= world else "gloo"
    parallel.init_from_env(backend=backend)
    dev = torch.device("cuda", rank % n_dev)
    torch.cuda.set_device(dev)
    mean, pca, t, dn, std, params = _problem()
    out = {"backend": backend}
    launches0 = _lib.launch_count()
    for use_std in (False, True):
        ev = cl.EnergyEvaluator(mean, pca, dn, std if use_std else None, LO, HI, True, t, params.shape[1], shard=True)
        assert ev.plan.wide and ev.sharded
        assert ev.plan.n_pixels in (dn.shape[0] * dn.shape[1] // 2, dn.shape[0] * dn.shape[1] // 2 + 1)
        out[use_std] = ev(params)
    out["launches"] = _lib.launch_count() - launches0
    # device-resident DE over the sharded objective: populations must stay bit-identical on both ranks
    ev = cl.EnergyEvaluator(mean, pca, dn, None, LO, HI, True, t, 64, shard=True)
    unit = qmc.Sobol(d=5, seed=np.random.default_rng(7)).random(n=64)
    de = ops.DeviceDE(ev.device_energies, [-0.5] * 5, [0.5] * 5, torch.from_numpy(unit).to(dev), seed=7, tol=0.0)
    for _ in range(12):
        de.step()
    torch.cuda.synchronize()
    out["pop"] = de.pop.cpu().numpy()
    out["energies"] = de.energies.cpu().numpy()
    out["exchange"] = ev.exchange
    if ev.exchange == "peer":
        # the fused generation replayed from a CUDA graph, pair sums pushed through peer memory: same walk
        ev2 = cl.EnergyEvaluator(mean, pca, dn, None, LO, HI, True, t, 64, shard=True)
        de2 = ops.DeviceDE.for_plan(ev2.plan, [-0.5] * 5, [0.5] * 5, torch.from_numpy(unit).to(dev), seed=7, tol=0.0)
        de2.run_graph(12, per_graph=4)
        torch.cuda.synchronize()
        out["pop_graph"] = de2.pop.cpu().numpy()
        # the NCCL route must give the same energies as the peer route
        ev3 = cl.EnergyEvaluator(mean, pca, dn, std, LO, HI, True, t, params.shape[1], shard=True, exchange="nccl")
        out["nccl_std"] = ev3(params)
    torch.distributed.barrier()
    q.put((rank, out))
    torch.distributed.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.timeout(600)
def test_k4_16bit_on_two_rank_shards_allreduce_and_finalize():
    from oracle import icrf_energy as oe
    n_dev = torch.cuda.device_count()
    assert n_dev >= 1
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, n_dev, q)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        out = [q.get(timeout=500) for _ in procs]
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
    finally:                     # a rank left waiting for a failed peer would outlive the test
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join()
    out.sort(key=lambda x: x[0])
    mean, pca, t, dn, std, params = _problem()
    for use_std in (False, True):
        expect = oe.energy_population(params, mean, pca, dn, std if use_std else None, LO, HI, True, t, bits=65536)
        assert np.isinf(expect[5])
        for _, res in out:
            e = res[use_std]
            assert np.array_equal(np.isinf(e), np.isinf(expect))
            fin = np.isfinite(expect)
            np.testing.assert_allclose(e[fin], expect[fin], rtol=1e-11)
        assert np.array_equal(out[0][1][use_std], out[1][1][use_std])         # identical finalize on every rank
    assert out[0][1]["launches"] > 0 and out[1][1]["launches"] > 0                  # the CUDA kernels ran on both
    assert np.array_equal(out[0][1]["pop"], out[1][1]["pop"])
    assert np.array_equal(out[0][1]["energies"], out[1][1]["energies"])
    assert out[0][1]["exchange"] == ("peer" if n_dev >= 2 else "nccl")
    if n_dev >= 2:
        assert np.array_equal(out[0][1]["pop_graph"], out[0][1]["pop"])
        assert np.array_equal(out[0][1]["pop_graph"], out[1][1]["pop_graph"])
        np.testing.assert_allclose(out[0][1]["nccl_std"], out[0][1][True], rtol=1e-13)
