"""Measure K3 Welford for 16-bit cameras on the GPU and write DIR/k3_16bit.json.

    python tools/run_k3_16bit.py --out DIR [--reps 20]

Workloads (generated on the device from a seed):
  cfg4-16 : 64 frames of 4320 x 7680 x 1 uint16, MAX_DN 65535 -- the cfg5 sensor's dark-frame stack (a static
            scene plus noise), 4.25 GB of frames
  12bit   : 300 frames of 1080 x 1920 x 3 uint16, MAX_DN 4095 (12-bit data stored in uint16)
Per workload: the integer stack, the ICRF stack (65536-row table; 4096-row table where the DNs fit it) and the
streaming update, each through the C ABI on preallocated buffers and timed with CUDA events after a warm-up; a parity
check of a crop against the oracle; the oracle on one core over a few frames as the CPU baseline.  The 8-bit cfg4
stack (600 x 1080 x 1920 x 3 uint8) runs in the same process for context.  Bytes are algorithmic:
2 B per sample-frame plus 18 B per sample of output (f64 mean, f64 SEM, u16 mean; 17 B for uint8).
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from camera_linearity_b200 import _lib, ops  # noqa: E402
from oracle import welford as ow  # noqa: E402

HBM_GBPS = 6556.0        # MEASURED_PEAKS.json of the project's B200 runs (used when that file is absent)


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        line = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        line = ""
    return {"query": q, "value": line, "torch_name": torch.cuda.get_device_name(0)}


def hbm_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            v = json.loads(p.read_text())
            for k in ("hbm_gbps", "hbm_GBps", "hbm"):
                if k in v:
                    return float(v[k]), "MEASURED_PEAKS.json"
        except (ValueError, TypeError):
            pass
    return HBM_GBPS, "constant (MEASURED_PEAKS.json value of earlier runs)"


def make_frames(F, H, W, C, lo, hi, sigma, top, seed, dtype):
    """static scene uniform in [lo, hi] plus rounded Gaussian noise, clamped to [0, top]"""
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(seed)
    base = torch.randint(lo, hi + 1, (1, H, W, C), generator=g, device=dev, dtype=torch.int32)
    store = torch.int16 if dtype == torch.uint16 else torch.uint8
    frames = torch.empty((F, H, W, C), dtype=store, device=dev)
    step = max(1, F // 8)
    for f0 in range(0, F, step):
        k = min(step, F - f0)
        noise = torch.round(torch.randn((k, H, W, C), generator=g, device=dev) * sigma).to(torch.int32)
        frames[f0:f0 + k] = torch.clamp(base + noise, 0, top).to(store)   # int16 wraps 32768.. like uint16 bits
    return frames.view(dtype) if dtype == torch.uint16 else frames


def table(rows, C, seed):
    rng = np.random.default_rng(seed)
    x = np.linspace(0, 1, rows)[:, None] ** (2.0 + 0.1 * np.arange(C))
    return torch.from_numpy(np.ascontiguousarray(x + rng.uniform(0, 1e-7, (rows, C)))).to("cuda:0")


def timed(fn, reps, warmup=2):
    for _ in range(warmup):
        fn()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
    ev[0].record()
    for r in range(reps):
        fn()
        ev[r + 1].record()
    torch.cuda.synchronize()
    ms = [ev[r].elapsed_time(ev[r + 1]) for r in range(reps)]
    return {"ms_median": float(np.median(ms)), "ms_min": float(np.min(ms)), "ms_max": float(np.max(ms)), "reps": reps}


def stack_call(lib, frames, lut, max_dn, outs, ws):
    F = frames.shape[0]
    n = frames[0].numel()
    C = frames.shape[-1]
    mean, sem, mq = outs
    s = torch.cuda.current_stream().cuda_stream
    if frames.dtype == torch.uint16:
        st = lib.cl_welford_stack_u16(frames.data_ptr(), F, n, C, None if lut is None else lut.data_ptr(),
                                      0 if lut is None else lut.shape[0], max_dn, mean.data_ptr(), sem.data_ptr(),
                                      mq.data_ptr(), ws.data_ptr(), ws.numel(), s)
    else:
        st = lib.cl_welford_stack(frames.data_ptr(), F, n, C, None if lut is None else lut.data_ptr(), max_dn,
                                  mean.data_ptr(), sem.data_ptr(), mq.data_ptr(), ws.data_ptr(), ws.numel(), s)
    _lib.check(st, "welford stack")


def tie_count(ws):
    return int(ws[:4].view(torch.int32).item())


def parity(frames, lut, max_dn, outs, crop):
    """the crop's outputs of the full-image call against the oracle on the crop's frames"""
    h, w = crop
    sub = frames[:, :h, :w].cpu().numpy()
    o = ow.welford(list(sub), icrf=None if lut is None else lut.cpu().numpy(), max_dn=max_dn)
    mean, sem, mq = (t[:h, :w].cpu().numpy() for t in outs)
    rel_mean = float(np.max(np.abs(mean - o["mean"]) / np.maximum(np.abs(o["mean"]), 1e-300)))
    fin = np.isfinite(o["sem"]) & (o["sem"] > 0)
    rel_sem = float(np.max(np.abs(sem[fin] - o["sem"][fin]) / o["sem"][fin], initial=0.0))
    if mq.dtype == np.uint16:           # the R9 extension for uint16 frames (DESIGN.md section 3)
        with np.errstate(invalid="ignore"):
            expect_q = np.around(o["mean"] * max_dn).astype(np.uint16)
    else:
        expect_q = o["mean_u8"]
    same_q = bool(np.array_equal(mq, expect_q))
    return {"crop": [h, w], "mean_q_identical": same_q, "max_rel_mean": rel_mean, "max_rel_sem": rel_sem,
            "ok": same_q and rel_mean <= 1e-12 and rel_sem <= 1e-9}


def cpu_baseline(frames, lut, max_dn, n_frames):
    """the oracle (NumPy, one core) over the first n_frames frames of the whole image"""
    sub = frames[:n_frames].cpu().numpy()
    t0 = time.perf_counter()
    ow.welford(list(sub), icrf=None if lut is None else lut.cpu().numpy(), max_dn=max_dn)
    dt = time.perf_counter() - t0
    return {"frames": n_frames, "seconds": dt, "sample_frames_per_s": sub.size / dt}


def workload(lib, name, frames, max_dn, tables, reps, crop, peak):
    F = frames.shape[0]
    n = frames[0].numel()
    shape = tuple(frames.shape[1:])
    qdtype = frames.dtype
    outs = (torch.empty(shape, dtype=torch.float64, device="cuda:0"),
            torch.empty(shape, dtype=torch.float64, device="cuda:0"),
            torch.empty(shape, dtype=qdtype, device="cuda:0"))
    ws = torch.empty(lib.cl_welford_stack_workspace_bytes(F, n), dtype=torch.uint8, device="cuda:0")
    qbytes = 2 if qdtype == torch.uint16 else 1
    alg_bytes = qbytes * F * n + (16 + qbytes) * n
    res = {"frames": F, "shape": list(shape), "max_dn": max_dn, "algorithmic_bytes": alg_bytes,
           "hbm_floor_ms": alg_bytes / peak / 1e6}
    for label, lut in [("integer", None)] + [(f"icrf_{t.shape[0]}", t) for t in tables]:
        r = timed(lambda: stack_call(lib, frames, lut, float(max_dn), outs, ws), reps)
        r["ties_replayed"] = tie_count(ws)
        r["GBps"] = alg_bytes / r["ms_median"] / 1e6
        r["share_of_hbm_peak"] = r["GBps"] / peak
        r["parity"] = parity(frames, lut, max_dn, outs, crop)
        res[label] = r
        print(name, label, f"{r['ms_median']:.3f} ms  {r['GBps']:.0f} GB/s  ({100 * r['share_of_hbm_peak']:.1f} %)  "
              f"ties {r['ties_replayed']}  parity {r['parity']['ok']}", flush=True)
    if qdtype == torch.uint16:
        mean = torch.zeros(shape, dtype=torch.float64, device="cuda:0")
        m2 = torch.zeros_like(mean)
        for label, lut in [("stream", None)] + [(f"stream_icrf_{t.shape[0]}", t) for t in tables[:1]]:
            r = timed(lambda: ops.welford_update(frames, mean, m2, 0, lut, float(max_dn)), max(2, reps // 4), 1)
            r["GBps"] = (2 * F * n + 32 * n) / r["ms_median"] / 1e6
            res[label] = r
            print(name, label, f"{r['ms_median']:.3f} ms  {r['GBps']:.0f} GB/s", flush=True)
    res["cpu_oracle_1core"] = cpu_baseline(frames, None, max_dn, 2 if n > 10 ** 7 else 4)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("run_k3_16bit.py measures on a GPU; none is visible")
    torch.cuda.set_device(0)
    lib = _lib.load()
    peak, peak_src = hbm_peak()
    out = {"card_before": card(), "hbm_peak_GBps": peak, "hbm_peak_source": peak_src}
    fr = make_frames(64, 4320, 7680, 1, 256, 65279, 16.0, 65535, 1, torch.uint16)
    out["cfg4_16"] = workload(lib, "cfg4-16", fr, 65535, [table(65536, 1, 2)], args.reps, (32, 64), peak)
    del fr
    torch.cuda.empty_cache()
    fr = make_frames(300, 1080, 1920, 3, 20, 4075, 3.0, 4095, 3, torch.uint16)
    out["rgb12"] = workload(lib, "12bit", fr, 4095, [table(65536, 3, 4), table(4096, 3, 5)], args.reps, (8, 16),
                            peak)
    del fr
    torch.cuda.empty_cache()
    fr = make_frames(600, 1080, 1920, 3, 20, 230, 3.0, 255, 7, torch.uint8)
    out["cfg4_8bit"] = workload(lib, "cfg4", fr, 255, [], args.reps, (8, 16), peak)
    out["card_after"] = card()
    out["ok"] = all(v["parity"]["ok"] for w in ("cfg4_16", "rgb12", "cfg4_8bit") for k, v in out[w].items()
                    if isinstance(v, dict) and "parity" in v)
    Path(args.out).mkdir(parents=True, exist_ok=True)
    (Path(args.out) / "k3_16bit.json").write_text(json.dumps(out, indent=1))
    print(json.dumps({k: out[k] for k in ("card_before", "ok")}))
    return 0 if out["ok"] else 1


if __name__ == "__main__":
    sys.exit(main())
