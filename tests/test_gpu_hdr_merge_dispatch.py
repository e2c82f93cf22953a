"""Which kernels cl_hdr_merge launches for each kind of stack and `algo`, and what it returns when it launches none.

Each case calls the C ABI directly on a small stack (a few 512-pixel tiles) and records the status, the library's launch
count and, under torch.profiler, the kernels (template instance included) and memsets in the order they ran."""
import ctypes as C
import re

import numpy as np
import pytest
import torch

from gpu_util import dev

pytestmark = pytest.mark.gpu
_lib = pytest.importorskip("camera_linearity_b200._lib")

OK, INVALID, UNSUPPORTED, WORKSPACE = 0, -1, -2, -3

SCAN = ["memset", "dark_scan_kernel"]          # dark scan: one memset clears the bucket counts and the work list
CLEAR = ["memset"]                             # work-list clear of the single-pass kernels without dark frames
FIXUP = ["merge_fixup_kernel"]
GEN8 = "merge_generic_kernel<unsigned char,true>"
GEN16 = ["build_tables_kernel", "merge_generic_kernel<unsigned short,false>"]
WIDE = "build_wide_table_kernel"


def _stack(dtype="u8", C_=3, N=4, H=32, W=64, std="images", darks=False, flat=False):
    """cl_hdr_merge_args of a synthetic stack and the tensors it points to.  std: "images" (float64 uncertainty image for
    every exposure), "table" (none: the STD table), "mixed" (images for the even exposures)."""
    rng = np.random.default_rng(N * 1000 + H * W * C_)
    u16 = dtype == "u16"
    max_dn, bits = (65535, 65536) if u16 else (255, 256)
    keep = []

    def d(x):
        t = dev(x)
        keep.append(t)
        return t

    t = 0.002 * 1.5 ** np.arange(N)
    dn = [d(rng.integers(0, max_dn + 1, (H, W, C_), dtype=np.uint16 if u16 else np.uint8)) for _ in range(N)]
    with_img = [std == "images" or (std == "mixed" and k % 2 == 0) for k in range(N)]
    sd = [d(rng.uniform(0.002, 0.02, (H, W, C_))) if w else None for w in with_img]
    x = np.linspace(0, 1, bits)
    lut = d(np.stack([x ** (2.0 + 0.1 * c) for c in range(C_)], axis=1))
    dlut = d(np.stack([np.gradient(x ** (2.0 + 0.1 * c), 2 / (bits - 1)) for c in range(C_)], axis=1))
    std_lut = d(np.tile(np.linspace(0.001, 0.02, bits)[:, None], (1, C_))) if std != "images" else None

    a = _lib.HdrMergeArgs()
    a.n_exposures, a.height, a.width, a.channels, a.dn_bytes, a.bits = N, H, W, C_, 2 if u16 else 1, bits
    arrays = [(C.c_void_p * N)(*[x.data_ptr() for x in dn]),
              (C.c_void_p * N)(*[x.data_ptr() if x is not None else None for x in sd]),
              (C.c_double * N)(*t)]
    a.dn = C.cast(arrays[0], C.POINTER(C.c_void_p))
    a.std = C.cast(arrays[1], C.POINTER(C.c_void_p))
    a.exposure_s = C.cast(arrays[2], C.POINTER(C.c_double))
    a.lut, a.dlut = lut.data_ptr(), dlut.data_ptr()
    a.std_lut = std_lut.data_ptr() if std_lut is not None else None
    if darks:                                   # a few hot pixels in every exposure's dark frame
        dk = []
        for _ in range(N):
            f = rng.poisson(2.0, (H, W, C_)).astype(np.uint16 if u16 else np.uint8)
            f.reshape(-1)[rng.choice(f.size, 40, replace=False)] = max_dn // 2
            dk.append(d(f))
        arrays.append((C.c_void_p * N)(*[x.data_ptr() for x in dk]))
        a.dark = C.cast(arrays[-1], C.POINTER(C.c_void_p))
        a.dark_threshold = 0.05
    a.median_kernel = 3
    if flat:
        a.flat_bytes = 2 if u16 else 1
        a.flat = d(rng.integers(max_dn // 2, max_dn, (H, W, C_), dtype=np.uint16 if u16 else np.uint8)).data_ptr()
        a.flat_std = d(rng.uniform(0.001, 0.01, (H, W, C_))).data_ptr()
        a.flat_means = d(np.concatenate([np.full(C_, 0.7), np.full(C_, 0.005)])).data_ptr()
    out_val = d(np.zeros((H, W, C_)))
    out_std = d(np.zeros((H, W, C_)))
    a.out_val, a.out_std = out_val.data_ptr(), out_std.data_ptr()
    return a, (keep, arrays)


def _name(event):
    if event.startswith("Memset"):
        return "memset"
    m = re.search(r"(\w+_kernel)(<[^>]*>)?", event)
    return (m.group(1) + (m.group(2) or "")).replace(", ", ",") if m else None


def _run(stack, algo, workspace="exact"):
    """(status, launches counted by the library, kernels and memsets in the order they ran).  workspace: "exact"
    (cl_hdr_merge_workspace_bytes bytes), "generous", "none", or "off16" (exact, 16- but not 32-byte aligned)."""
    lib = _lib.load()
    a = stack[0]
    a.algo = algo
    need = lib.cl_hdr_merge_workspace_bytes(C.byref(a))
    size = {"exact": need, "generous": 2 * need + 4096, "none": 0, "off16": need}[workspace]
    buf = torch.empty(size + 16, dtype=torch.uint8, device="cuda") if size else None
    ptr = None if buf is None else buf.data_ptr() + (16 if workspace == "off16" else 0)
    assert ptr is None or ptr % (16 if workspace == "off16" else 32) == 0
    stream = torch.cuda.current_stream().cuda_stream
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        st = lib.cl_hdr_merge(C.byref(a), ptr, size, stream)
        torch.cuda.synchronize()
    n1 = _lib.launch_count()
    events = sorted((e for e in prof.events() if _name(e.name)), key=lambda e: e.time_range.start)
    return st, n1 - n0, [_name(e.name) for e in events]


# (id, stack, algos, workspace, expected status, expected kernels)
RGB_DARK_FLAT = dict(N=16, darks=True, flat=True)
CASES = [
    ("u8_rgb_images_dark_flat", dict(RGB_DARK_FLAT), (0, 4), "exact", OK,
     SCAN + ["merge_stream_kernel<false>"] + FIXUP),
    ("u8_rgb_images_dark_flat_ragged", dict(RGB_DARK_FLAT, H=33), (0,), "exact", OK,
     SCAN + ["merge_stream_kernel<false>", GEN8] + FIXUP),
    ("u8_mono_table_n5", dict(C_=1, N=5, H=64, W=96, std="table"), (0, 4), "exact", OK,
     CLEAR + ["merge_stream_lut_kernel<true>"] + FIXUP),
    ("u8_rgb_images_n1", dict(N=1), (0,), "exact", OK, ["merge_staged_kernel<8,false>"]),
    ("u8_rgb_table_n1", dict(N=1, std="table"), (0,), "exact", OK, ["merge_staged_lut_kernel<8,false>"]),
    ("u8_rgb_images_n16_staged", dict(N=16), (2,), "exact", OK, ["merge_staged_kernel<16,false>"]),
    ("u8_rgb_images_n17_staged", dict(N=17), (2,), "exact", OK, ["merge_staged_kernel<32,false>"]),
    ("u8_mixed", dict(std="mixed"), (0,), "exact", OK, [GEN8]),
    ("u8_two_channels", dict(C_=2), (0,), "exact", OK, [GEN8]),
    ("u8_below_one_tile", dict(H=8, W=16), (0,), "exact", OK, [GEN8]),
    ("u8_rgb_images_no_workspace", dict(), (0,), "none", OK, ["merge_staged_kernel<8,false>"]),
    ("u16_images_n3", dict(dtype="u16", N=3, H=16, W=48), (0, 3), "exact", OK,
     [WIDE, "merge_wide_pipe_kernel<4,192,false>"]),
    ("u16_images_n5", dict(dtype="u16", N=5, H=16, W=48), (0, 3), "exact", OK,
     [WIDE, "merge_wide_pipe_kernel<8,192,false>"]),
    ("u16_images_n12", dict(dtype="u16", N=12, H=16, W=48), (0, 3), "exact", OK,
     [WIDE, "merge_wide_pipe_kernel<12,192,false>"]),
    ("u16_images_n16", dict(dtype="u16", N=16, H=16, W=48), (0, 3), "exact", OK,
     [WIDE, "merge_wide_pipe_kernel<16,128,false>"]),
    ("u16_table_n12", dict(dtype="u16", N=12, H=16, W=48, std="table"), (0, 3), "exact", OK,
     [WIDE, "merge_wide_pipe_kernel<12,128,true>"]),
    ("u16_mixed_n7", dict(dtype="u16", N=7, H=16, W=48, std="mixed"), (0, 3), "exact", OK,
     [WIDE, "merge_wide_kernel<8,true>"]),
    ("u16_n17", dict(dtype="u16", N=17, H=16, W=48), (0,), "exact", OK, GEN16),
    ("u16_workspace_not_32_aligned", dict(dtype="u16", N=5, H=16, W=48), (0,), "off16", OK, GEN16),
    ("u8_algo3", dict(), (3,), "exact", UNSUPPORTED, []),
    ("u16_n17_algo3", dict(dtype="u16", N=17, H=16, W=48), (3,), "exact", UNSUPPORTED, []),
    ("u16_no_workspace", dict(dtype="u16", N=5, H=16, W=48), (3, 0), "none", WORKSPACE, []),
    ("u8_n1_algo4", dict(N=1), (4,), "exact", UNSUPPORTED, []),
    ("u8_mixed_algo4", dict(std="mixed"), (4,), "exact", UNSUPPORTED, []),
    ("u8_rgb_no_workspace_algo4", dict(), (4,), "none", WORKSPACE, []),
    ("u8_mixed_algo2", dict(std="mixed"), (2,), "exact", UNSUPPORTED, []),
    ("u8_rgb_dark_no_workspace_algo2", dict(darks=True), (2,), "none", WORKSPACE, []),
    ("u16_algo_out_of_range", dict(dtype="u16", N=5, H=16, W=48), (7, -1), "exact", INVALID, []),
    ("u16_algo2_algo4", dict(dtype="u16", N=5, H=16, W=48), (2, 4), "exact", UNSUPPORTED, []),
    ("u16_algo2_algo4_no_workspace", dict(dtype="u16", N=5, H=16, W=48), (2, 4), "none", UNSUPPORTED, []),
]


@pytest.fixture(scope="module", autouse=True)
def _profiler_sees_kernels():
    st, _, names = _run(_stack(), 1)
    assert st == OK
    if not names:
        pytest.skip("the profiler records no device activity here")


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_dispatch_map(case):
    _, kw, algos, workspace, status, kernels = case
    stack = _stack(**kw)
    for algo in algos:
        st, launches, names = _run(stack, algo, workspace)
        assert (st, names) == (status, kernels), algo
        assert launches == sum(k != "memset" for k in kernels), (algo, launches)


SUCCESSES = [c for c in CASES if c[4] == OK and c[3] == "exact"]


@pytest.mark.parametrize("case", SUCCESSES, ids=[c[0] for c in SUCCESSES])
def test_exact_workspace_selects_what_a_generous_one_does(case):
    # a workspace of exactly cl_hdr_merge_workspace_bytes must be enough for every region cl_hdr_merge carves from it
    _, kw, algos, _, _, _ = case
    stack = _stack(**kw)
    for algo in algos:
        exact, generous = _run(stack, algo, "exact"), _run(stack, algo, "generous")
        assert exact[0] == generous[0] == OK
        assert exact[2] == generous[2], algo
