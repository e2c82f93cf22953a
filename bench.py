#!/usr/bin/env python
"""Benchmark of the hot path: fused HDR merge throughput in Gpix*exposures/s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2|cfg1]
                    [--dump-outputs DIR]

One "step" = one fused HDR merge of one synthetic exposure stack (cfg2 of BASELINE.json /
SURVEY.md 8d by default: 16 exposures 3840x2160x3 uint8 + float64 uncertainty images, dark
frames for the exposures >= 0.05 s, flat field).  N > 1 (torchrun): every rank merges its own
stack -- stacks are independent units, no data-path collective -- so scaling is "weak" and
`value` = total pix*exposures of all ranks / max-over-ranks time.

`value`   : inputs resident in HBM, CUDA-event timed, per rank max.
`e2e`     : the same merge through the public API (ExposureSeries.process_HDR_image) from pinned
            HOST buffers, host->device copies and the device->host read of the result inside the
            timed region.
`roofline`: algorithmic bytes of the merge kernel / its CUDA-event duration vs the measured HBM
            peak (MEASURED_PEAKS.json, else the 6.65 TB/s fallback of B200_PROFILING.md).
`cpu_baseline`: the NumPy oracle port of the reference timed on a bounded row crop of the same
            workload on this box's host cores.
--impl reference: the oracle port (the reference is pure Python/NumPy and does not run at HEAD,
            see DESIGN.md) on all host cores, row tiles in a process pool.
--dump-outputs DIR: after the timed steps, what the last step computed as .npy files (`dump_outputs`).  The
            synthetic inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

WORKLOADS = {
    # name: (H, W, C, N, t0, ratio, corrections)
    "cfg1": dict(H=1536, W=2048, C=3, N=5, t0=0.005, ratio=2.0, corrections=False,
                 label="cfg1: 5-exposure 2048x1536x3 uint8 + f64 std, fixed ICRF"),
    "cfg2": dict(H=2160, W=3840, C=3, N=16, t0=0.001, ratio=1.6, corrections=True,
                 label="cfg2: 16-exposure 3840x2160x3 uint8 + f64 std, dark frames (t>=0.05s) + flat field"),
}
DARK_THRESHOLD = 0.05
KERNEL = 3
FF_MID = 0.2


def exposures_of(wl):
    return wl["t0"] * wl["ratio"] ** np.arange(wl["N"])


def icrf_tables(C):
    x = np.linspace(0, 1, 256)
    icrf = np.stack([x ** (2.0 + 0.1 * c) for c in range(C)], axis=1)
    diff = np.stack([np.gradient(icrf[:, c], 2 / 255) for c in range(C)], axis=1)
    return icrf, diff


def config_of(wl, world):
    """The `config` object of the JSON line -- identical in the GPU arm and the reference arm."""
    t = exposures_of(wl)
    n_dark = int(sum(1 for tk in t if wl["corrections"] and tk >= DARK_THRESHOLD))
    alg = algorithmic_bytes(wl, n_dark)
    return {"workload": wl["label"], "per_gpu_stack": f"{wl['N']}x{wl['H']}x{wl['W']}x{wl['C']}",
            "dark_frames": n_dark, "flat_field": bool(wl["corrections"]),
            "l2": f"inputs larger than L2 (no flush needed): {alg / 1e9:.2f} GB streamed per step vs 126 MB L2",
            "parallelism": f"independent stacks x{world}, no collective"}


# what cl_hdr_merge runs for an 8-bit RGB stack with float64 uncertainty images (include/camera_linearity.h, `algo`)
MERGE_KERNEL_OF_ALGO = {0: "merge_stream_kernel (single pass; the default)", 4: "merge_stream_kernel (single pass)",
                        2: "merge_staged_kernel<16> (two passes over the staged tile)", 1: "merge_generic_kernel"}


def std_table(C):
    """Synthetic camera STD table (image_set.py:365-385): shot-noise-like, sigma grows with the signal."""
    x = np.linspace(0, 1, 256)
    return 0.002 + 0.018 * np.sqrt(x)[:, None] * np.array([1.0, 0.9, 1.1, 1.0])[:C]


def algorithmic_bytes(wl, n_dark):
    n = wl["H"] * wl["W"] * wl["C"]
    b = wl["N"] * n * 9 + n_dark * n * 1 + n * 16
    if wl["corrections"]:
        b += n * 9
    return b


# ----------------------------------------------------------------------------- synthetic data
def make_stack_numpy(wl, rows, seed):
    """Host (NumPy) synthetic crop of `rows` rows: same generator family as the device one."""
    rng = np.random.default_rng(seed)
    H, W, C = rows, wl["W"], wl["C"]
    t = exposures_of(wl)
    rad = rng.uniform(0, 1, (H, W, C)) * 25
    dn = [np.rint(255 * np.clip(rad * tk, 0, 1) ** (1 / 2.2)).astype(np.uint8) for tk in t]
    std = [rng.uniform(0.002, 0.02, (H, W, C)) for _ in t]
    darks = [None] * wl["N"]
    flat = flat_std = None
    if wl["corrections"]:
        for k, tk in enumerate(t):
            if tk >= DARK_THRESHOLD:
                d = rng.poisson(2.0, (H, W, C)).astype(np.uint8)
                hot = rng.uniform(size=d.shape) < 0.001
                d[hot] = rng.integers(40, 200, int(hot.sum()))
                darks[k] = d
        flat = np.clip(np.rint(rng.normal(180, 6, (H, W, C))), 1, 255).astype(np.uint8)
        flat_std = rng.uniform(0.001, 0.01, (H, W, C))
    return dict(dn=dn, std=std, t=t, darks=darks, flat=flat, flat_std=flat_std)


def make_stack_device(wl, seed, dev):
    import torch
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    H, W, C = wl["H"], wl["W"], wl["C"]
    t = exposures_of(wl)
    rad = torch.rand((H, W, C), generator=g, device=dev, dtype=torch.float64) * 25
    dn, std, darks = [], [], []
    for tk in t:
        dn.append(torch.round(255 * torch.clamp(rad * tk, 0, 1) ** (1 / 2.2)).to(torch.uint8))
        std.append(torch.rand((H, W, C), generator=g, device=dev, dtype=torch.float64) * 0.018 + 0.002)
    flat = flat_std = None
    for tk in t:
        if wl["corrections"] and tk >= DARK_THRESHOLD:
            d = torch.poisson(torch.full((H, W, C), 2.0, device=dev), generator=g).to(torch.uint8)
            hot = torch.rand((H, W, C), generator=g, device=dev) < 0.001
            d[hot] = torch.randint(40, 200, (int(hot.sum()),), generator=g, device=dev, dtype=torch.uint8)
            darks.append(d)
        else:
            darks.append(None)
    if wl["corrections"]:
        flat = torch.clamp(torch.round(torch.randn((H, W, C), generator=g, device=dev) * 6 + 180), 1, 255).to(torch.uint8)
        flat_std = torch.rand((H, W, C), generator=g, device=dev, dtype=torch.float64) * 0.009 + 0.001
    del rad
    return dict(dn=dn, std=std, t=t, darks=darks, flat=flat, flat_std=flat_std)


# ----------------------------------------------------------------------------- CPU (oracle) arm
_CROP_CACHE = {}


def _oracle_merge_crop(args):
    """Merge one synthetic row crop with the NumPy oracle; returns the merge time only (the crop is
    generated once per (worker, seed) and cached, so generation stays outside the timing)."""
    wl_name, rows, seed = args
    wl = WORKLOADS[wl_name]
    from oracle import hdr_merge as om
    key = (wl_name, rows, seed)
    if key not in _CROP_CACHE:
        data = make_stack_numpy(wl, rows, seed)
        if wl["corrections"]:
            data["dark_val"] = [None if d is None else om.dark_value_image(d, 1.0) for d in data["darks"]]
            data["flat_val"] = data["flat"] / 255.0
        _CROP_CACHE[key] = data
    data = _CROP_CACHE[key]
    icrf, diff = icrf_tables(wl["C"])
    t0 = time.perf_counter()
    om.hdr_merge(data["dn"], data["std"], data["t"], icrf, diff, darks=data.get("dark_val"),
                 dark_threshold=DARK_THRESHOLD, kernel=KERNEL, flat_val=data.get("flat_val"),
                 flat_std=data["flat_std"], roi=(0, rows, 0, wl["W"]))
    return time.perf_counter() - t0


def cpu_baseline_single(wl_name, rows=96):
    wl = WORKLOADS[wl_name]
    dt = _oracle_merge_crop((wl_name, rows, 1234))
    pix_exp = rows * wl["W"] * wl["N"]
    return dict(value=pix_exp / dt / 1e9, unit="Gpix*exposures/s", cores=1, kind="port",
                sample=f"oracle (NumPy port of the reference + repairs R1-R8) on a {rows}-row crop "
                       f"({rows}x{wl['W']}x{wl['C']}, {wl['N']} exposures) of the workload, {dt:.2f} s, 1 core")


def run_reference_arm(args, wl_name):
    """`--impl reference`: the oracle port on all host cores.  Each step = one bounded row crop per
    worker process (the reference's NumPy code is single-threaded; row tiles are independent)."""
    import multiprocessing as mp
    wl = WORKLOADS[wl_name]
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cores = os.cpu_count() or 1
    rows = 48
    jobs = [(wl_name, rows, 100 + i) for i in range(cores)]
    times = []
    with mp.get_context("fork").Pool(cores) as pool:
        pool.map(_oracle_merge_crop, jobs)            # untimed: generates and caches the crops
        for step in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            pool.map(_oracle_merge_crop, jobs, chunksize=1)
            dt = time.perf_counter() - t0
            if step >= args.warmup:
                times.append(dt)
    total = sum(times)
    pix_exp_step = cores * rows * wl["W"] * wl["N"]
    value = pix_exp_step * len(times) / total / 1e9
    sample = (f"per step: {cores} worker processes x one {rows}-row crop ({rows}x{wl['W']}x{wl['C']}, "
              f"{wl['N']} exposures, dark frames + flat field as in the workload) through the NumPy oracle port "
              f"of the reference (+ repairs R1-R8); wall time of the parallel map, inputs pre-generated")
    line = {
        "impl": "reference", "metric": "HDR merge throughput", "value": value, "unit": "Gpix*exposures/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_of(wl, args.gpus),
        "cpu_baseline": {"value": value, "unit": "Gpix*exposures/s", "cores": cores, "kind": "port", "sample": sample,
                         "value_per_core": value / cores, "sample_rows_per_worker": rows, "workers": cores},
        "e2e": {"value": value, "unit": "Gpix*exposures/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock, power and throttle reasons through NVML in a background thread (every few
    ms, so that even a 100 ms timed region is covered); falls back to one nvidia-smi query."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, torch_device):
        self.samples = []
        self.reasons = set()
        self.sm_max = None
        self.power = []
        self.handle = None
        self.thread = None
        self.running = False
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            self.nv = pynvml
            uuid = str(getattr(torch.cuda.get_device_properties(torch_device), "uuid", ""))
            try:
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode() if uuid and not uuid.startswith("GPU-") else uuid.encode())
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(torch_device.index or 0)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.handle = None

    def _loop(self):
        nv = self.nv
        it = 0
        while self.running:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
                if it % 4 == 0:                      # the power query is the slow one
                    self.power.append(nv.nvmlDeviceGetPowerUsage(self.handle) / 1000.0)
            except Exception:
                pass
            it += 1
            time.sleep(0.001)

    def start(self):
        if self.handle is None:
            return
        import threading
        self.running = True
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def stop(self):
        if self.handle is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"], "samples": 0}
        self.running = False
        self.thread.join(timeout=2)
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.sm_max,
                "reasons": sorted(self.reasons), "samples": len(self.samples),
                "power_w_max": max(self.power) if self.power else None}


def measured_traffic(workload):
    """DRAM bytes (read + write) of one cl_hdr_merge call -- the merge kernel plus the dark scan / patch
    / fix-up kernels it launches -- from the committed ncu capture."""
    path = ROOT / "profiles" / "r02_traffic.json"
    try:
        entry = json.loads(path.read_text())[workload]
        return entry["dram_bytes_read"] + entry["dram_bytes_write"] + sum(entry.get("other_kernels", {}).values())
    except Exception:
        return None


def hbm_peak():
    path = ROOT / "MEASURED_PEAKS.json"
    if path.exists():
        try:
            return float(json.loads(path.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_SAMPLES = 1 << 20          # samples of the merged image kept by --dump-outputs: 8 MB per float64 array
DUMP_SEED = 0


def dump_outputs(directory, val, std, flat_means):
    """`--dump-outputs DIR`: the merged radiance and uncertainty of the last timed step, sampled at the same
    DUMP_SAMPLES flat indices of the (H, W, C) image (drawn once from a seeded generator, sorted), as
    DIR/hdr_val.npy and DIR/hdr_std.npy; the indices as DIR/hdr_sample_index.npy; the flat ROI means the step
    passed to the merge as DIR/flat_roi_means.npy.  All float64 (the indices are exact below 2**53)."""
    import torch
    directory = Path(directory)
    directory.mkdir(parents=True, exist_ok=True)
    n = val.numel()
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, min(n, DUMP_SAMPLES), replace=False))
    idx_dev = torch.from_numpy(idx).to(val.device)
    arrays = {"hdr_val": val.reshape(-1)[idx_dev], "hdr_std": std.reshape(-1)[idx_dev],
              "hdr_sample_index": idx, "flat_roi_means": flat_means}
    for name, a in arrays.items():
        if a is None:
            continue
        a = a.cpu().numpy() if isinstance(a, torch.Tensor) else a
        np.save(directory / f"{name}.npy", a.astype(np.float64))


# ----------------------------------------------------------------------------- ours
def run_ours(args, wl):
    import torch
    import torch.distributed as dist

    import camera_linearity_b200 as cl
    from camera_linearity_b200 import _lib, ops, parallel

    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"          # keep stdout to the one JSON line
    rank, world, local = parallel.init_from_env()
    numa_bound = parallel.bind_to_gpu_numa_node(local) if world > 1 else False   # pinned e2e buffers stay NUMA-local
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    cl.GlobalSettings.configure(IM_SIZE_X=wl["H"], IM_SIZE_Y=wl["W"], DARK_THRESHOLD=DARK_THRESHOLD,
                                MEDIAN_FILTER_KERNEL_SIZE=KERNEL, FF_MID_PERCENTAGE=FF_MID)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    data = make_stack_device(wl, 1000 + rank, dev)
    icrf_np, diff_np = icrf_tables(wl["C"])
    icrf, diff = torch.from_numpy(icrf_np).to(dev), torch.from_numpy(diff_np).to(dev)
    t = [float(x) for x in data["t"]]
    n_dark = sum(d is not None for d in data["darks"])
    out = (torch.empty((wl["H"], wl["W"], wl["C"]), dtype=torch.float64, device=dev),
           torch.empty((wl["H"], wl["W"], wl["C"]), dtype=torch.float64, device=dev))
    roi = cl.measurand._flat_roi()
    last = {}                                      # the flat ROI means of the latest step, for --dump-outputs

    def step():
        ev0 = torch.cuda.Event(enable_timing=True)
        ev1 = torch.cuda.Event(enable_timing=True)
        ev0.record()
        means = None
        if data["flat"] is not None:
            means = ops.flat_roi_means(data["flat"], data["flat_std"], roi)
        ops.hdr_merge(data["dn"], data["std"], t, icrf, diff, darks=data["darks"], dark_threshold=DARK_THRESHOLD,
                      median_kernel=KERNEL, flat=data["flat"], flat_std=data["flat_std"], flat_means=means,
                      algo=args.algo, out=out)
        last["flat_roi_means"] = means
        ev1.record()
        return ev0, ev1

    for _ in range(args.warmup):
        step()
    barrier()
    launches0 = _lib.launch_count()
    sampler = ClockSampler(dev)
    if rank == 0:
        sampler.start()
    start = torch.cuda.Event(enable_timing=True)
    stop = torch.cuda.Event(enable_timing=True)
    start.record()
    kernel_events = [step() for _ in range(args.steps)]
    stop.record()
    barrier()
    launches = _lib.launch_count() - launches0
    total_ms = start.elapsed_time(stop)
    kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in kernel_events]))
    tmax = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    total_ms = float(tmax.item())
    pix_exp = wl["H"] * wl["W"] * wl["N"]
    value = world * pix_exp * args.steps / (total_ms * 1e-3) / 1e9
    if args.dump_outputs is not None and rank == 0:     # before the STD-table loop below overwrites `out`
        dump_outputs(args.dump_outputs, out[0], out[1], last["flat_roi_means"])

    # ---- the same stack WITHOUT uncertainty images (sigma from the camera's STD table), device resident ----
    std_lut_np = std_table(wl["C"])
    std_lut_dev = torch.from_numpy(std_lut_np).to(dev)

    def step_table():
        means = None
        if data["flat"] is not None:
            means = ops.flat_roi_means(data["flat"], data["flat_std"], roi)
        ops.hdr_merge(data["dn"], None, t, icrf, diff, std_lut=std_lut_dev, darks=data["darks"],
                      dark_threshold=DARK_THRESHOLD, median_kernel=KERNEL, flat=data["flat"], flat_std=data["flat_std"],
                      flat_means=means, algo=args.algo, out=out)

    for _ in range(3):
        step_table()
    barrier()
    ta, tb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ta.record()
    for _ in range(args.steps):
        step_table()
    tb.record()
    barrier()
    tab_ms = torch.tensor([ta.elapsed_time(tb) / args.steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tab_ms, op=dist.ReduceOp.MAX)
    tab_ms = float(tab_ms.item())

    # ---- e2e: public API from pinned host buffers, H2D + D2H inside the timed region ----
    # Every step uploads the N exposures (uint8 DNs + float64 uncertainty images) from pinned host memory,
    # merges them through ExposureSeries.process_HDR_image and reads the float64 radiance + uncertainty back.
    # The dark frames and the flat field are per-camera CALIBRATION frames: they are uploaded once (outside
    # the timed region) and stay resident, as a long-running service would keep them.
    host = {k: [None if x is None else x.cpu().pin_memory() for x in data[k]] for k in ("dn", "std")}
    out_host = (torch.empty(out[0].shape, dtype=torch.float64).pin_memory(),
                torch.empty(out[0].shape, dtype=torch.float64).pin_memory())
    feats = lambda tk, subject: {"illumination": "bf", "magnification": "10x", "exposure": tk, "subject": subject}
    dark_sets = []
    for k, d in enumerate(data["darks"]):
        if d is not None:
            ds = cl.ImageSet(features=feats(t[k], "dark"))
            ds.set_digital_numbers(d)
            dark_sets.append(ds)
    flats = []
    if data["flat"] is not None:
        fs = cl.ImageSet(features=feats(0.0, "flat"), measurand=cl.Measurand(None, data["flat_std"]))
        fs.set_digital_numbers(data["flat"])
        flats.append(fs)
    data["dn"] = data["std"] = None
    del out
    torch.cuda.empty_cache()

    def e2e_step(out_host, use_table):
        sets = []
        for k in range(wl["N"]):
            std_k = None if use_table else host["std"][k].to(dev, non_blocking=True)
            s = cl.ImageSet(features=feats(t[k], "s"), measurand=cl.Measurand(None, std_k))
            s.set_digital_numbers(host["dn"][k])            # pinned host tensor -> device, asynchronous
            sets.append(s)
        series = cl.ExposureSeries(input_image_sets=sets)
        series.process_HDR_image(icrf, diff, dark_list=dark_sets, flat_list=flats, algo=args.algo,
                                 STD_data=std_lut_dev if use_table else None)
        m = series.merged_image_set.measurand
        out_host[0].copy_(m.val, non_blocking=True)
        out_host[1].copy_(m.std, non_blocking=True)

    # Two CUDA streams alternate between steps so that the device->host read of step i overlaps the
    # host->device copies of step i+1 (PCIe is full duplex); every step still moves all of its inputs
    # and reads back its whole result inside the timed region.
    n_e2e = max(2, args.steps)
    streams = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)]
    out_hosts = [out_host, (torch.empty_like(out_host[0]).pin_memory(), torch.empty_like(out_host[1]).pin_memory())]

    def e2e_run(count, use_table):
        for i in range(count):
            with torch.cuda.stream(streams[i % 2]):
                e2e_step(out_hosts[i % 2], use_table)
        for st in streams:
            st.synchronize()

    def e2e_measure(use_table):
        e2e_run(2, use_table)
        barrier()
        wall0 = time.perf_counter()
        e2e_run(n_e2e, use_table)
        barrier()
        ms = (time.perf_counter() - wall0) * 1e3
        tm = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        return float(tm.item())

    n_samp = wl["H"] * wl["W"] * wl["C"]
    d2h = n_samp * 16
    e2e_total_ms = e2e_measure(False)
    e2e_value = world * pix_exp * n_e2e / (e2e_total_ms * 1e-3) / 1e9
    h2d = wl["N"] * n_samp * 9
    # the same stack WITHOUT uncertainty images: sigma = STD_data[DN, c] (image_set.py:228-243, 365-385, the
    # reference's path whenever no '... STD.tif' exists) -> only the uint8 exposures cross PCIe
    e2e_tab_ms = e2e_measure(True)
    e2e_tab_value = world * pix_exp * n_e2e / (e2e_tab_ms * 1e-3) / 1e9
    h2d_tab = wl["N"] * n_samp
    del host, dark_sets, flats, data
    clocks = sampler.stop() if rank == 0 else None      # sampled through the timed steps, the STD-table loop and both e2e arms
    k4 = None
    if not args.no_extra:
        try:
            k4 = k4_block(dev, rank, world, cpu=not args.no_cpu)
        except Exception as exc:
            k4 = {"error": repr(exc)}
    extra = {}
    if rank == 0 and not args.no_extra:    # (before the cfg5 batch: that block leaves the GPU under its software power cap)
        try:
            extra = extra_kernels(dev)
        except Exception as exc:          # the headline must not die on an auxiliary measurement
            extra = {"error": repr(exc)}
    cfg5 = None
    if not args.no_extra and CFG5["stacks"] % world == 0:
        try:
            cfg5 = {"f64_std": cfg5_measure(dev, rank, world, 2, 3),
                    "std_table": cfg5_measure(dev, rank, world, 2, 3, std_table=True)}
        except Exception as exc:
            cfg5 = {"error": repr(exc)}

    if world > 1:
        try:                               # the line below must be printed whatever an auxiliary block left behind
            dist.barrier()
            dist.destroy_process_group()
        except Exception:
            pass
    if rank != 0:
        return
    peak, peak_src = hbm_peak()
    alg_bytes = algorithmic_bytes(wl, n_dark)
    ms_per_step = total_ms / args.steps
    achieved = alg_bytes / (ms_per_step * 1e-3) / 1e9      # whole step (ROI means + dark scan + merge + fix-up)
    cpu = cpu_baseline_single(args.workload) if world == 1 and not args.no_cpu else None
    line = {
        "metric": "HDR merge throughput", "value": value, "unit": "Gpix*exposures/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_of(wl, world),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": measured_traffic(args.workload) if args.algo != 1 else None, "traffic_source":
                     "ncu dram__bytes_read+write summed over the kernels of one step (merge kernel + dark scan / flat ROI / "
                     "fix-up), profiles/r02_traffic.json (tools/traffic_from_launches.py)", "peak_source": peak_src,
                     "kernel": (f"one step = cl_flat_roi_means + cl_hdr_merge (dark_scan + {MERGE_KERNEL_OF_ALGO[args.algo]}, "
                                "~94% of the time, + merge_fixup); achieved = algorithmic bytes / ms_per_step"
                                if args.algo != 1 else "merge_generic_kernel"),
                     "algorithmic_bytes_per_launch": alg_bytes, "step_ms_by_per_step_events": kernel_ms},
        "cpu_baseline": cpu,
        "e2e": {"value": e2e_value, "unit": "Gpix*exposures/s", "h2d_bytes_per_step": world * h2d,
                "d2h_bytes_per_step": world * d2h,
                "ms_per_step": e2e_total_ms / n_e2e, "steps": n_e2e,
                "api": "ExposureSeries.process_HDR_image on ImageSets built from pinned host tensors (ImageSet.set_digital_numbers "
                       "+ Measurand std); every step uploads the 16 exposures (uint8 + float64 uncertainty images) and reads the "
                       "float64 result back; the dark frames and the flat field are per-camera calibration frames, uploaded once "
                       "and kept resident; steps alternate between two CUDA streams (D2H of step i overlaps H2D of step i+1); "
                       "wall-clock timed",
                "numa_bound": bool(numa_bound)},
        "std_table_variant": {
            "what": "the same stack without uncertainty images: sigma = STD_data[DN, c] gathered inside the merge kernel "
                    "(image_set.py:228-243, 365-385 -- the reference's path whenever no '... STD.tif' exists)",
            "value": world * pix_exp / (tab_ms * 1e-3) / 1e9, "unit": "Gpix*exposures/s", "ms_per_step": tab_ms,
            "algorithmic_bytes_per_step": alg_bytes - wl["N"] * n_samp * 8,
            "kernel": "merge_stream_lut_kernel (single pass; tables {w, P1} and {x dg, e dg} in shared memory)",
            "bound": "sm (shared-memory table gathers + FP64), not HBM: "
                     f"{(alg_bytes - wl['N'] * n_samp * 8) / tab_ms / 1e6:.0f} GB/s of algorithmic traffic",
            "e2e": {"value": e2e_tab_value, "unit": "Gpix*exposures/s", "h2d_bytes_per_step": world * h2d_tab,
                    "d2h_bytes_per_step": world * d2h, "ms_per_step": e2e_tab_ms / n_e2e, "steps": n_e2e,
                    "api": "as `e2e`, with ExposureSeries.process_HDR_image(STD_data=...) and no uncertainty images: only "
                           "the uint8 exposures cross PCIe"}},
        "k4_icrf_fit": k4,
        "cfg5_sharded_batch": cfg5,
        "gpu_launches": int(launches),
        "clocks": clocks,
        "extra": extra,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------- cfg5: 64 stacks x 12 x 8K 16-bit
CFG5 = dict(H=4320, W=7680, N=12, stacks=64, t0=0.0005, ratio=1.7,
            label="cfg5: batch of 64 stacks x 12 exposures 7680x4320x1 uint16 + f64 std, 65536-row ICRF, sharded over the GPUs")


def cfg5_tables(dev):
    import torch
    x16 = np.linspace(0, 1, 65536)
    icrf = torch.from_numpy((x16 ** 2.1).reshape(-1, 1)).to(dev)
    diff = torch.from_numpy(np.gradient(x16 ** 2.1, 2 / 65535).reshape(-1, 1)).to(dev)
    stdlut = torch.from_numpy((0.002 + 0.02 * np.sqrt(x16)).reshape(-1, 1)).to(dev)
    return icrf, diff, stdlut


def cfg5_stack_device(seed, dev, with_std=True):
    import torch
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    H, W, N = CFG5["H"], CFG5["W"], CFG5["N"]
    t = [CFG5["t0"] * CFG5["ratio"] ** k for k in range(N)]
    rad = torch.rand((H, W, 1), generator=g, device=dev, dtype=torch.float32) * 25
    dn = [torch.round(65535 * torch.clamp(rad * tk, 0, 1) ** (1 / 2.2)).to(torch.int32).to(torch.uint16) for tk in t]
    del rad
    std = ([torch.rand((H, W, 1), generator=g, device=dev, dtype=torch.float64) * 0.018 + 0.002 for _ in t]
           if with_std else None)
    return dn, std, t


def cfg5_measure(dev, rank, world, steps, warmup, std_table=False, sample_clocks=True):
    """The sharded batch of BASELINE config 5: 64 stacks split over the ranks (8 per GPU at N = 8), no collective.
    Each rank keeps min(64 / world, 8) DISTINCT stacks resident (8 stacks = 36 GB) and merges its 64 / world stacks per
    step by cycling over them, so every merge reads data far larger than L2.  Strong scaling: the batch is fixed."""
    import torch
    import torch.distributed as dist
    from camera_linearity_b200 import ops
    per_rank = CFG5["stacks"] // world
    resident = min(per_rank, 8)
    icrf, diff, stdlut = cfg5_tables(dev)
    stacks = [cfg5_stack_device(5000 + 64 * rank + i, dev, with_std=not std_table) for i in range(resident)]
    n = CFG5["H"] * CFG5["W"]
    out = (torch.empty((CFG5["H"], CFG5["W"], 1), dtype=torch.float64, device=dev),
           torch.empty((CFG5["H"], CFG5["W"], 1), dtype=torch.float64, device=dev))
    kw = dict(std_lut=stdlut) if std_table else {}

    def step():
        for i in range(per_rank):
            dn, std, t = stacks[i % resident]
            ops.hdr_merge(dn, std, t, icrf, diff, out=out, **kw)

    for _ in range(warmup):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(dev) if (rank == 0 and sample_clocks) else None
    if sampler:
        sampler.start()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        step()
    b.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    block_clocks = sampler.stop() if sampler else None
    tm = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    ms_step = float(tm.item()) / steps
    pix_exp = CFG5["stacks"] * n * CFG5["N"]
    b_std = 0 if std_table else 8
    alg_stack = CFG5["N"] * n * (2 + b_std) + n * 16
    peak, _ = hbm_peak()
    del stacks, out
    torch.cuda.empty_cache()
    return {"workload": CFG5["label"], "uncertainty": "STD table (65536 rows, fused into the ICRF gather)" if std_table
            else "float64 uncertainty images", "value": pix_exp / (ms_step * 1e-3) / 1e9, "unit": "Gpix*exposures/s",
            "scaling": "strong", "ms_per_step": ms_step, "stacks_per_rank_per_step": per_rank,
            "distinct_resident_stacks_per_rank": resident, "ms_per_stack": ms_step / per_rank,
            "algorithmic_bytes_per_stack": alg_stack,
            "achieved_GB/s_per_gpu": alg_stack / (ms_step / per_rank) / 1e6,
            "frac_of_hbm_peak": alg_stack / (ms_step / per_rank) / 1e6 / peak,
            # this block keeps the GPU busy for hundreds of ms: the float64-image variant draws enough power for the
            # box's software power cap to lower the SM clock (one stack timed alone: 1.48 ms, tools/cfg5_sustained.py)
            "clocks": block_clocks,
            "bound": "L1 data pipe: one divergent 16-byte (32-byte with the STD table) table gather per sample-exposure "
                     "from a 1 MB (2 MB) table = one L1 wavefront per row, 1 per SM clock "
                     "(tools/microbench/gather_mix.cu; ncu: pipe 84 % busy), see DESIGN.md"}


def run_cfg5(args):
    """`--workload cfg5`: the sharded 16-bit batch as the main line (device-resident value, e2e from pinned host
    buffers, CPU port on a row crop)."""
    import torch
    import torch.distributed as dist
    import camera_linearity_b200 as cl
    from camera_linearity_b200 import _lib, ops, parallel
    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"
    rank, world, local = parallel.init_from_env()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if CFG5["stacks"] % world:
        raise SystemExit("cfg5 needs a GPU count that divides 64")
    steps = args.steps
    launches0 = _lib.launch_count()
    sampler = ClockSampler(dev)
    if rank == 0:
        sampler.start()
    main_res = cfg5_measure(dev, rank, world, steps, max(3, args.warmup))
    clocks = sampler.stop() if rank == 0 else None
    launches = _lib.launch_count() - launches0
    tab_res = cfg5_measure(dev, rank, world, steps, 3, std_table=True)

    # e2e: every stack of the rank's share is uploaded from pinned host memory (one pinned stack, re-sent: the
    # bytes are real, a 255 GB batch does not fit host memory), merged through ExposureSeries.process_HDR_image and
    # read back
    per_rank = CFG5["stacks"] // world
    icrf, diff, stdlut = cfg5_tables(dev)
    dn, std, t = cfg5_stack_device(777 + rank, dev)
    host_dn = [x.cpu().pin_memory() for x in dn]
    host_std = [x.cpu().pin_memory() for x in std]
    del dn, std
    torch.cuda.empty_cache()
    cl.GlobalSettings.configure(BIT_DEPTH=16)
    shape = (CFG5["H"], CFG5["W"], 1)
    outs = [(torch.empty(shape, dtype=torch.float64).pin_memory(), torch.empty(shape, dtype=torch.float64).pin_memory())
            for _ in range(2)]
    streams = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)]
    feats = lambda tk: {"illumination": "bf", "magnification": "10x", "exposure": tk, "subject": "s"}

    def e2e_stack(i):
        with torch.cuda.stream(streams[i % 2]):
            sets = []
            for k in range(CFG5["N"]):
                s_ = cl.ImageSet(features=feats(t[k]), measurand=cl.Measurand(None, host_std[k].to(dev, non_blocking=True)))
                s_.set_digital_numbers(host_dn[k])
                sets.append(s_)
            series = cl.ExposureSeries(input_image_sets=sets)
            series.process_HDR_image(icrf, diff, dark_list=[], flat_list=[])
            m = series.merged_image_set.measurand
            outs[i % 2][0].copy_(m.val, non_blocking=True)
            outs[i % 2][1].copy_(m.std, non_blocking=True)

    e2e_stacks = min(per_rank, 8)                      # a bounded share of the step, scaled to the whole step below
    for i in range(2):
        e2e_stack(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for i in range(e2e_stacks):
        e2e_stack(i)
    for st in streams:
        st.synchronize()
    if world > 1:
        dist.barrier()
    tm = torch.tensor([(time.perf_counter() - t0) * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    n = CFG5["H"] * CFG5["W"]
    e2e_value = world * e2e_stacks * n * CFG5["N"] / (float(tm.item()) * 1e-3) / 1e9
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    cpu = None
    if world == 1 and not args.no_cpu:
        from oracle import hdr_merge as om
        rows = 24
        rng = np.random.default_rng(5)
        tt = np.array(t)
        rad = rng.uniform(0, 1, (rows, CFG5["W"], 1)) * 25
        dn_h = [np.rint(65535 * np.clip(rad * tk, 0, 1) ** (1 / 2.2)).astype(np.uint16) for tk in tt]
        std_h = [rng.uniform(0.002, 0.02, (rows, CFG5["W"], 1)) for _ in tt]
        x16 = np.linspace(0, 1, 65536)
        t0 = time.perf_counter()
        om.hdr_merge(dn_h, std_h, tt, x16 ** 2.1, np.gradient(x16 ** 2.1, 2 / 65535), max_dn=65535)
        dt = time.perf_counter() - t0
        cpu = {"value": rows * CFG5["W"] * CFG5["N"] / dt / 1e9, "unit": "Gpix*exposures/s", "cores": 1, "kind": "port",
               "sample": f"oracle (NumPy port) on a {rows}-row crop of one stack ({rows}x{CFG5['W']}x1 uint16, 12 exposures), {dt:.2f} s"}
    peak, peak_src = hbm_peak()
    line = {
        "metric": "HDR merge throughput", "value": main_res["value"], "unit": "Gpix*exposures/s", "n_gpus": world,
        "steps": steps, "warmup": max(3, args.warmup), "ms_per_step": main_res["ms_per_step"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": CFG5["label"], "stacks_per_rank_per_step": main_res["stacks_per_rank_per_step"],
                   "distinct_resident_stacks_per_rank": main_res["distinct_resident_stacks_per_rank"],
                   "l2": "each merge streams 4.5 GB (8 distinct resident stacks per rank = 36 GB) vs 126 MB L2",
                   "parallelism": f"64 independent stacks over {world} GPU(s), no collective"},
        "roofline": {"bound": "hbm", "achieved": main_res["achieved_GB/s_per_gpu"], "peak": peak, "unit": "GB/s",
                     "frac": main_res["frac_of_hbm_peak"], "traffic": None, "peak_source": peak_src,
                     "kernel": "merge_wide_kernel<12,false> (+ build_wide_table_kernel, 1 MB)",
                     "algorithmic_bytes_per_launch": main_res["algorithmic_bytes_per_stack"], "note": main_res["bound"]},
        "cpu_baseline": cpu,
        "e2e": {"value": e2e_value, "unit": "Gpix*exposures/s", "h2d_bytes_per_step": CFG5["stacks"] * CFG5["N"] * n * 10,
                "d2h_bytes_per_step": CFG5["stacks"] * n * 16, "ms_per_step": float(tm.item()) / e2e_stacks * per_rank,
                "stacks_timed_per_rank": e2e_stacks,
                "api": "ExposureSeries.process_HDR_image per stack from pinned host tensors (uint16 exposures + float64 "
                       "uncertainty images uploaded, float64 result read back, two alternating streams); timed on "
                       f"{e2e_stacks} of the rank's {per_rank} stacks per step and scaled"},
        "std_table_variant": tab_res,
        "gpu_launches": int(launches), "clocks": clocks,
    }
    print(json.dumps(line))


def cfg3_problem():
    """cfg3 of BASELINE.json / SURVEY 8d: 400 000 pixels x 5 exposures (4.0 M pixel-pairs per evaluation), 64 candidates
    over 5 principal components (an all-valid population: most random candidates of a wide box hit the +inf gates)."""
    x = np.linspace(0, 1, 256)
    modes = np.stack([np.sin((k + 1) * np.pi * x) * x for k in range(5)], axis=1)
    pca, _ = np.linalg.qr(modes)
    rng = np.random.default_rng(3)
    tt = 0.005 * 2.0 ** np.arange(5)
    rad = rng.uniform(0, 1, (1000, 400, 1)) * 25
    stack = np.rint(255 * np.clip(rad * tt[None, None, :], 0, 1) ** (1 / 2.2)).astype(np.uint8)
    std = rng.uniform(0.002, 0.02, stack.shape)
    params = rng.uniform(-0.05, 0.05, (5, 64))
    return x ** 2.2, pca, tt, stack, std, params


def k4_block(dev, rank, world, cpu=True):
    """ICRF-fit loss evaluations per second on cfg3 with the pixels sharded over the `world` GPUs (collective: every
    rank calls it).  `population`: candidate curves + partial kernel + fused tail (CTA reduction, pair sums exchanged
    through peer memory, finalize) timed with CUDA events, max over ranks.  `de_generation`: the same inside the
    device-resident DE (3 launches per generation, 8 generations per CUDA-graph replay)."""
    import torch
    import torch.distributed as dist
    import camera_linearity_b200 as cl
    from camera_linearity_b200 import ops
    from scipy.stats import qmc
    mean, pca, tt, stack, std, params = cfg3_problem()
    out = {"shape": "cfg3: S=64 candidates x 5 PCs, 400k px x 5 exposures (4.0M pixel-pairs per eval), pixels sharded "
                    f"over {world} GPU(s)", "unit": "evals/s"}

    def sync_max(ms):
        tm = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        return float(tm.item())

    def timed(fn, reps, warm=3):
        for _ in range(warm):
            fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return sync_max(a.elapsed_time(b) / reps)

    for name, sdv in (("nostd", None), ("std", std)):
        ev = cl.EnergyEvaluator(mean, pca, stack, sdv, 5, 250, True, tt, 64, shard=True)
        p_dev = torch.from_numpy(np.ascontiguousarray(params.T)).to(dev)
        ms = timed(lambda: ev.device_energies(p_dev), reps=50)
        res = {"ms_per_population": ms, "evals/s": 64e3 / ms, "pair_evals/s": 64 * 400000 * 10 / ms * 1e3,
               "exchange": ev.exchange, "launches_per_population": 3 if ev.exchange != "nccl" else 5}
        unit = qmc.Sobol(d=5, seed=np.random.default_rng(7)).random(n=64)
        if ev.exchange != "nccl":
            de = ops.DeviceDE.for_plan(ev.plan, [-0.5] * 5, [0.5] * 5, torch.from_numpy(unit).to(dev), seed=7, tol=0.0)
            de.run_graph(8, per_graph=8)
            gen_ms = timed(lambda: de.run_graph(8, per_graph=8), reps=12, warm=2) / 8
            res["de_generation"] = {"ms": gen_ms, "evals/s": 64e3 / gen_ms, "generations/s": 1e3 / gen_ms,
                                    "how": "cl_de_trial_curves + partial + fused tail (reduce / exchange / finalize / DE selection), CUDA graph of 8 generations"}
        else:
            de = ops.DeviceDE(ev.device_energies, [-0.5] * 5, [0.5] * 5, torch.from_numpy(unit).to(dev), seed=7, tol=0.0)
            gen_ms = timed(de.step, reps=40, warm=3)
            res["de_generation"] = {"ms": gen_ms, "evals/s": 64e3 / gen_ms, "generations/s": 1e3 / gen_ms,
                                    "how": "generic step with an NCCL all-reduce between partial and finalize"}
        if world > 1 and ev.exchange == "peer":
            # the same objective with the pair sums all-reduced by NCCL between the partial and finalize launches
            # (round 1's path): what the peer-memory tail replaces
            ev_n = cl.EnergyEvaluator(mean, pca, stack, sdv, 5, 250, True, tt, 64, shard=True, exchange="nccl")
            ms_n = timed(lambda: ev_n.device_energies(p_dev), reps=50)
            de_n = ops.DeviceDE(ev_n.device_energies, [-0.5] * 5, [0.5] * 5, torch.from_numpy(unit).to(dev), seed=7, tol=0.0)
            gen_n = timed(de_n.step, reps=40, warm=3)
            res["nccl_allreduce_variant"] = {"ms_per_population": ms_n, "evals/s": 64e3 / ms_n,
                                             "de_generation_ms": gen_n, "de_evals/s": 64e3 / gen_n,
                                             "how": "curves, partial, reduce, ncclAllReduce(S x pairs x 2 f64), finalize "
                                                    "(+ de_trial, de_select): 7 launches per generation, host driven"}
            del ev_n, de_n
        out[name] = res
        del ev, de
    if cpu and rank == 0:
        # the reference's objective (oracle port of _energy_function, ICRF_calibration_exposure.py:148-201) on the same
        # pixels, one host core, a bounded number of candidates
        from oracle import icrf_energy as oe
        for name, sdv, n_cand in (("nostd", None, 3), ("std", std, 2)):
            t0 = time.perf_counter()
            oe.energy_population(params[:, :n_cand], mean, pca, stack, sdv, 5, 250, True, tt)
            dt = time.perf_counter() - t0
            out[name]["cpu_baseline"] = {"value": n_cand / dt, "unit": "evals/s", "cores": 1, "kind": "port",
                                         "sample": f"{n_cand} candidates of the population on the full 400k px x 5 stack, "
                                                   f"NumPy port of _energy_function, {dt:.2f} s"}
    return out


def extra_kernels(dev):
    """Short device-resident measurements of the other three kernels (reported, not the headline)."""
    import torch
    import camera_linearity_b200 as cl
    from camera_linearity_b200 import ops

    def timed(fn, reps=5, warm=2):
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

    out = {}
    g = torch.Generator(device=dev)
    g.manual_seed(7)
    icrf_np, diff_np = icrf_tables(3)
    icrf, diff = torch.from_numpy(icrf_np).to(dev), torch.from_numpy(diff_np).to(dev)
    peak, _ = hbm_peak()
    # K2 on the other single-stack configurations (device resident)
    for name, wl_name, corrections in (("k2_cfg1", "cfg1", False), ("k2_cfg2_no_corrections", "cfg2", False)):
        wl = dict(WORKLOADS[wl_name], corrections=corrections)
        data = make_stack_device(wl, 77, dev)
        tt = [float(x) for x in data["t"]]
        o = (torch.empty((wl["H"], wl["W"], 3), dtype=torch.float64, device=dev),
             torch.empty((wl["H"], wl["W"], 3), dtype=torch.float64, device=dev))
        # cfg1 is smaller than L2 x4: rotate over enough distinct stacks?  576 MB > 126 MB L2, fine.
        ms = timed(lambda: ops.hdr_merge(data["dn"], data["std"], tt, icrf, diff, out=o), reps=10, warm=3)
        nb = algorithmic_bytes(wl, 0)
        out[name] = {"ms": ms, "GB/s": nb / ms / 1e6, "frac_of_hbm_peak": nb / ms / 1e6 / peak,
                     "Gpix*exposures/s": wl["H"] * wl["W"] * wl["N"] / ms / 1e6, "algorithmic_bytes": nb}
        del data, o
    # K1: linearize one 4K RGB frame with std (25 B/sample)
    dn = torch.randint(0, 256, (2160, 3840, 3), generator=g, device=dev, dtype=torch.uint8)
    sd = torch.rand((2160, 3840, 3), generator=g, device=dev, dtype=torch.float64) * 0.02
    ms = timed(lambda: ops.linearize(dn, sd, icrf, diff))
    out["k1_linearize"] = {"ms": ms, "GB/s": dn.numel() * 25 / ms / 1e6, "frac_of_hbm_peak": dn.numel() * 25 / ms / 1e6 / peak,
                           "shape": "2160x3840x3 u8 + f64 std"}
    del dn, sd
    # linearity analysis of one exposure pair (next row 8f-1): 2160x3840x3 float64 val+std, one pass of 32 B/sample
    xv = torch.rand((2160, 3840, 3), generator=g, device=dev, dtype=torch.float64) + 0.05
    yv = torch.rand((2160, 3840, 3), generator=g, device=dev, dtype=torch.float64) + 0.05
    xs = torch.rand((2160, 3840, 3), generator=g, device=dev, dtype=torch.float64) * 0.02 + 0.001
    ys = torch.rand((2160, 3840, 3), generator=g, device=dev, dtype=torch.float64) * 0.02 + 0.001
    ms = timed(lambda: ops.pair_statistics(xv, xs, yv, ys, 0.5, [0.1] * 3, [0.9] * 3))
    out["pair_statistics"] = {"ms": ms, "GB/s": xv.numel() * 32 / ms / 1e6, "frac_of_hbm_peak": xv.numel() * 32 / ms / 1e6 / peak,
                              "shape": "one exposure pair 2160x3840x3 f64 val+std, every input read once (32 B/sample)"}
    # Measurand operators with propagation, fused (measurand.py:106-241): x * y and x / y on 4K RGB val+std pairs,
    # 32 B in + 16 B out per element
    import camera_linearity_b200 as cl
    mx, my = cl.Measurand(xv, xs), cl.Measurand(yv, ys)
    for name, fn in (("measurand_mul", lambda: mx * my), ("measurand_div", lambda: mx / my)):
        ms = timed(fn)
        out[name] = {"ms": ms, "GB/s": xv.numel() * 48 / ms / 1e6, "frac_of_hbm_peak": xv.numel() * 48 / ms / 1e6 / peak,
                     "shape": "2160x3840x3 f64 val+std (op) same, one fused pass"}
    del mx, my, xv, yv, xs, ys
    # K3: cfg4, 600 frames 1080x1920x3
    base = torch.randint(20, 231, (1, 1080, 1920, 3), generator=g, device=dev, dtype=torch.int16)
    frames = torch.empty((600, 1080, 1920, 3), dtype=torch.uint8, device=dev)
    for f0 in range(0, 600, 50):
        noise = torch.round(torch.randn((50, 1080, 1920, 3), generator=g, device=dev) * 3).to(torch.int16)
        frames[f0:f0 + 50] = torch.clamp(base + noise, 0, 255).to(torch.uint8)
    del noise
    ws = torch.empty(ops._lib.load().cl_welford_stack_workspace_bytes(600, frames[0].numel()), dtype=torch.uint8, device=dev)
    ms = timed(lambda: ops.welford_stack(frames, None, 255.0, ws), reps=5, warm=2)
    nb = frames.numel() + frames[0].numel() * 17
    out["k3_welford_stack"] = {"ms": ms, "GB/s": nb / ms / 1e6, "frac_of_hbm_peak": nb / ms / 1e6 / peak,
                               "Gpix*frames/s": 600 * 1080 * 1920 / ms / 1e6,
                               "shape": "cfg4: 600x1080x1920x3 u8"}
    ms = timed(lambda: ops.welford_stack(frames, icrf, 255.0, ws), reps=5, warm=2)       # linearised frames (ICRF given)
    out["k3_welford_stack_icrf"] = {"ms": ms, "GB/s": nb / ms / 1e6, "frac_of_hbm_peak": nb / ms / 1e6 / peak,
                                    "shape": "cfg4 with ICRF[frame, c] as the sample value"}
    # noise profiles (joint mean-DN / frame-DN histogram per channel, video_processing.py:77-106) over the same 600 frames
    mean_u8 = ops.welford_stack(frames, None, 255.0, ws)[2]
    hist = torch.zeros((256, 256, 3), dtype=torch.int64, device=dev)
    ms = timed(lambda: ops.noise_profiles(frames, mean_u8, hist), reps=3, warm=1)
    out["noise_profiles"] = {"ms": ms, "GB/s": frames.numel() / ms / 1e6, "frac_of_hbm_peak": frames.numel() / ms / 1e6 / peak,
                             "shape": "cfg4 frames against their uint8 mean frame, 1 B per sample-frame"}
    del hist, mean_u8
    # the reference's Welford recurrence (oracle port of video_processing.py:183-217) on a bounded number of frames
    from oracle import welford as ow
    n_f = 12
    host_frames = [f.cpu().numpy() for f in frames[:n_f]]
    t0 = time.perf_counter()
    ow.welford(host_frames)
    dt = time.perf_counter() - t0
    out["k3_welford_stack"]["cpu_baseline"] = {"value": n_f * 1080 * 1920 / dt / 1e9, "unit": "Gpix*frames/s", "cores": 1,
                                               "kind": "port", "sample": f"{n_f} frames 1080x1920x3, NumPy port of "
                                                                         f"welford_algorithm, {dt:.2f} s"}
    # K3 end to end through the public call: welford_algorithm over host frames (a frame source standing in for the
    # OpenCV decoder), i.e. host copy into the pinned staging buffers + H2D on the copy stream + cl_welford_update
    # per chunk + finalize; the result frames come back to the host.
    from camera_linearity_b200 import video_processing as vp
    n_in = 240
    host_video = frames[:n_in].cpu().numpy()

    def source(_path):
        for f in host_video:
            yield f
    for use_icrf in (False, True):
        vp.welford_algorithm(Path("synthetic.avi"), icrf_np if use_icrf else None, True, frame_source=source)   # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ret = vp.welford_algorithm(Path("synthetic.avi"), icrf_np if use_icrf else None, True, frame_source=source)
        ret["mean"].cpu(), ret["sem"].cpu()
        dt = time.perf_counter() - t0
        out["k3_welford_stack_icrf" if use_icrf else "k3_welford_stack"]["e2e"] = {
            "value": n_in * 1080 * 1920 / dt / 1e9, "unit": "Gpix*frames/s", "frames": n_in, "seconds": dt,
            "h2d_bytes": int(host_video.nbytes), "GB/s_host_to_result": host_video.nbytes / dt / 1e9,
            "api": "video_processing.welford_algorithm(frame_source=host frames): pinned double-buffered staging, "
                   "H2D on a copy stream, cl_welford_update per chunk, cl_welford_finalize; bound by the host-side copy "
                   "of each frame into the staging buffer (one core)"}
    del frames, ws
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS) + ["cfg5"])
    ap.add_argument("--algo", type=int, default=0, choices=[0, 1, 2, 4],
                    help="0 auto, 1 generic kernel, 2 staged two-pass kernel, 4 single-pass kernel")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float64; "
                         "a fixed, seeded sample of the merged image; cfg1 / cfg2 device arm, rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.impl != "ours" or args.workload == "cfg5"):
        ap.error("--dump-outputs is supported for the cfg1 / cfg2 device arm only")
    if args.workload == "cfg5" and args.impl == "ours":
        return run_cfg5(args)
    wl = WORKLOADS[args.workload if args.workload in WORKLOADS else "cfg2"]
    if args.impl == "reference":
        run_reference_arm(args, args.workload)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
