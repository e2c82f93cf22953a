"""K4 at 16 bits on one GPU: cfg3-16 (bench.cfg3_problem() with uint16 samples and a 65536-point curve) next to the
8-bit cfg3, plus the oracle on one host core for the CPU baseline and a parity check at this size.

    python tools/run_k4_16bit.py --out DIR [--reps 50]

Writes DIR/k4_16bit.json (timings from CUDA events; per-kernel times from torch.profiler in a separate pass).
"""
import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

os.environ.setdefault("OMP_NUM_THREADS", "1")          # the oracle baseline is one host core
os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
os.environ.setdefault("MKL_NUM_THREADS", "1")

import numpy as np  # noqa: E402
import torch  # noqa: E402

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402
import camera_linearity_b200 as cl  # noqa: E402
from camera_linearity_b200 import ops  # noqa: E402
from oracle import icrf_energy as oe  # noqa: E402

D16 = 65536
S = 64


def cfg3_16_problem():
    """bench.cfg3_problem() at 16 bits, seed 3: 400 000 px x 5 exposures, 64 candidates, D = 65536."""
    x = np.linspace(0, 1, D16)
    pca, _ = np.linalg.qr(np.stack([np.sin((k + 1) * np.pi * x) * x for k in range(5)], axis=1))
    rng = np.random.default_rng(3)
    tt = 0.005 * 2.0 ** np.arange(5)
    rad = rng.uniform(0, 1, (1000, 400, 1)) * 25
    stack = np.rint(65535 * np.clip(rad * tt[None, None, :], 0, 1) ** (1 / 2.2)).astype(np.uint16)
    std = rng.uniform(0.002, 0.02, stack.shape)
    params = rng.uniform(-0.05, 0.05, (5, S))
    return x ** 2.2, pca, tt, stack, std, params, (5 * 257, 250 * 257)


def cfg3_problem():
    mean, pca, tt, stack, std, params = bench.cfg3_problem()
    return mean, pca, tt, stack, std, params, (5, 250)


def timed(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def kernel_times(fn, reps):
    """Mean device time per call of each kernel over `reps` calls (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if ev.device_type is not None and "cuda" in str(ev.device_type).lower() and ev.count:
            name = ev.key.replace("(anonymous namespace)::", "").replace("void ", "").split("(")[0]
            dt = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
            out[name[:120]] = {"us_per_call": dt / reps, "launches_per_call": ev.count / reps}
    return out


def measure(problem, dev, reps, label, table_rows_per_px):
    mean, pca, tt, stack, std, params, (lo, hi) = problem
    n_px, n_exp = stack.shape[0] * stack.shape[1], stack.shape[2]
    pairs = n_exp * (n_exp - 1) // 2
    p_dev = torch.from_numpy(np.ascontiguousarray(params.T)).to(dev)
    res = {}
    for name, sdv in (("nostd", None), ("std", std)):
        ev = cl.EnergyEvaluator(mean, pca, stack, sdv, lo, hi, True, tt, S, shard=False)
        e = ev.device_energies(p_dev).cpu().numpy()
        ms = timed(lambda: ev.device_energies(p_dev), reps)
        ms_curves = timed(ev.plan.curves_and_tables, reps)
        ms_pop = timed(ev.plan.population, reps)
        gathered = n_px * (S // 32) * table_rows_per_px * 256           # one 256-byte row per gather and warp
        r = {"ms_per_population": ms, "ms_curves_and_tables": ms_curves, "ms_partial_and_tail": ms_pop,
             "evals/s": S * 1e3 / ms, "pair_evals/s": S * n_px * pairs / ms * 1e3,
             "table_bytes_gathered_per_population": gathered,
             "gather_rate_GB/s (partial + tail time)": gathered / ms_pop / 1e6,
             "gated_candidates": int(np.isinf(e).sum()),
             "kernels": kernel_times(lambda: ev.device_energies(p_dev), reps=min(reps, 20))}
        from scipy.stats import qmc
        unit = qmc.Sobol(d=5, seed=np.random.default_rng(7)).random(n=S)
        de = ops.DeviceDE.for_plan(ev.plan, [-0.5] * 5, [0.5] * 5, torch.from_numpy(unit).to(dev), seed=7, tol=0.0)
        de.run_graph(8, per_graph=8)
        gen_ms = timed(lambda: de.run_graph(8, per_graph=8), reps=max(4, reps // 4), warm=2) / 8
        r["de_generation"] = {"ms": gen_ms, "evals/s": S * 1e3 / gen_ms,
                              "how": "cl_de_trial_curves + partial + fused tail with DE selection, CUDA graph of 8"}
        r["energies_first3"] = e[:3].tolist()
        res[name] = r
        del ev, de
    res["shape"] = f"{label}: S={S} x 5 PCs, {n_px} px x {n_exp} exposures, D={len(mean)}, {stack.dtype}"
    return res


def oracle_check(problem, res, label):
    """The oracle's energy for two candidates on one host core (CPU baseline), against the device's."""
    mean, pca, tt, stack, std, params, (lo, hi) = problem
    out = {}
    for name, sdv in (("nostd", None), ("std", std)):
        t0 = time.perf_counter()
        ref = oe.energy_population(params[:, :2], mean, pca, stack, sdv, lo, hi, True, tt, bits=len(mean))
        dt = time.perf_counter() - t0
        got = np.asarray(res[name]["energies_first3"][:2])
        same_gates = bool(np.array_equal(np.isinf(got), np.isinf(ref)))
        fin = np.isfinite(ref)
        rel = float(np.max(np.abs(got[fin] - ref[fin]) / np.abs(ref[fin]), initial=0.0))
        out[name] = {"cpu_evals/s": 2 / dt, "cpu_seconds_for_2": dt, "max_rel_diff": rel,
                     "ok": same_gates and rel <= 1e-11}
    return out


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        line = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        line = ""
    return {"query": q, "value": line, "torch_name": torch.cuda.get_device_name(0)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=50)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("run_k4_16bit.py measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    out = {"card_before": card()}
    p16 = cfg3_16_problem()
    out["cfg3_16"] = measure(p16, dev, args.reps, "cfg3-16", 2 * (5 - 1))
    p8 = cfg3_problem()
    out["cfg3_8bit"] = measure(p8, dev, args.reps, "cfg3", 2 * (5 - 1))
    out["oracle_cfg3_16"] = oracle_check(p16, out["cfg3_16"], "cfg3-16")
    out["card_after"] = card()
    out["ok"] = all(v["ok"] for v in out["oracle_cfg3_16"].values())
    Path(args.out).mkdir(parents=True, exist_ok=True)
    (Path(args.out) / "k4_16bit.json").write_text(json.dumps(out, indent=1))
    print(json.dumps({k: out[k] for k in ("card_before", "ok")}))
    for cfg in ("cfg3_16", "cfg3_8bit"):
        for name in ("nostd", "std"):
            r = out[cfg][name]
            print(cfg, name, f"pop {r['ms_per_population']:.4f} ms  curves {r['ms_curves_and_tables']:.4f} ms  "
                  f"partial+tail {r['ms_partial_and_tail']:.4f} ms  DE gen {r['de_generation']['ms']:.4f} ms  "
                  f"gated {r['gated_candidates']}")
    return 0 if out["ok"] else 1


if __name__ == "__main__":
    sys.exit(main())
