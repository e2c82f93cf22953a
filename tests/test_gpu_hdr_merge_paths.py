"""K2 (cl_hdr_merge) path by path: every kernel instance against an extended-precision evaluation of the merge formula of
hdr_merge.cuh on the exact double inputs the kernel reads, each sample within an error bound derived from its own data.

The reference takes, per sample and exposure, the (repaired) DN d and uncertainty s, the weight w = w[d] of
cl_gaussian_weight (the device function the kernels' tables are built with, checked against mpmath below), the table
values g = lut[d, c], dg = dlut[d, c] * s, kappa(d) = fma(d, -60/MAX, 30) rounded once, and rt = 1/t correctly rounded.
With S = sum w, x = kappa w g + w dg, e = kappa w^2 g, y = dg rt, it evaluates in long double

    val = sum(w g rt) / S,    std = sqrt(sum(((x - e / S) y)^2)) / S,
    A = sum (x y)^2,  B = sum (x y)(e y),  C = sum (e y)^2,  q = A - 2B/S + C/S^2   (the single-pass kernels' sums),

and the flat-field epilogue of flat_apply() on the exact reciprocal of the flat value.  Bad-pixel masks come from
NumPy's double comparison (what the host turns into an integer DN threshold), medians from integer / exact selection.
u = 2^-53 throughout; N is the exposure count."""
import json
import math
import re
import subprocess
import sys
import zlib
from fractions import Fraction
from pathlib import Path

import numpy as np
import pytest
import torch
from scipy.ndimage import median_filter

from oracle import hdr_merge as om
from gpu_util import dev, host

pytestmark = pytest.mark.gpu
ops = pytest.importorskip("camera_linearity_b200.ops")
if np.finfo(np.longdouble).nmant < 63:
    pytest.skip("the reference needs an 80-bit long double", allow_module_level=True)

LD = np.longdouble
U = 2.0 ** -53
TIGHT = 1e-11                  # every ordinary case also meets this, whatever its own bound
STREAM = 1e-9                  # single-pass uncertainty of a sample the fix-up rule does not flag
CANCEL = 1e-6                  # hdr_merge.cuh kStreamCancel
TILE = 512 * 3                 # samples per tile of the tile kernels
GEN8 = "merge_generic_kernel<unsigned char,true>"
GEN16 = "merge_generic_kernel<unsigned short,false>"


# ---------------------------------------------------------------------------------------------------------------------
# helpers

def _name(event):
    m = re.search(r"(\w+_kernel)(<[^>]*>)?", event)
    return (m.group(1) + (m.group(2) or "")).replace(", ", ",") if m else None


def _profiled(fn):
    """(fn(), names of the kernels it launched, in order)"""
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    events = sorted((e for e in prof.events() if _name(e.name)), key=lambda e: e.time_range.start)
    return out, [_name(e.name) for e in events]




def _profiled_cases(cases):
    """{id: kernels launched by run()} for (id, run) in cases, from ONE profiler session (the number of sessions a
    process can open with device activity recorded is limited): a gaussian_weight_kernel launch separates the cases.
    None when the profiler records no device activity here."""
    marker = torch.zeros(1, dtype=torch.float64, device="cuda")

    def all_cases():
        for _, run in cases:
            run()
            torch.cuda.synchronize()
            ops.gaussian_weight(marker)
    _, names = _profiled(all_cases)
    if not names:
        return None
    out, cur = {}, []
    ids = iter(i for i, _ in cases)
    for nm in (x for x in names if "at::" not in x):          # (PyTorch's own copy / fill kernels)
        if nm == "gaussian_weight_kernel":
            out[next(ids)] = cur
            cur = []
        else:
            cur.append(nm)
    assert len(out) == len(cases)
    return out


def _dev_dn(a):
    return dev(a) if a.dtype == np.uint8 else dev(a.view(np.int16)).view(torch.uint16)


_W, _KAPPA = {}, {}


def _weights(max_dn):
    """w[d] = cl_gaussian_weight(d / MAX) for every DN: the values the kernels' tables hold"""
    if max_dn not in _W:
        w, _ = ops.gaussian_weight(dev(np.arange(max_dn + 1) / float(max_dn)))
        _W[max_dn] = host(w)
    return _W[max_dn]


def _kappa(max_dn):
    """kappa(d) = fma(d, -60 / MAX, 30), rounded once"""
    if max_dn not in _KAPPA:
        ks = Fraction(-60.0 / max_dn)
        _KAPPA[max_dn] = np.array([float(d * ks + 30) for d in range(max_dn + 1)])
    return _KAPPA[max_dn]


def _tables(c, bits, rng=None, std_kind=None):
    x = np.linspace(0, 1, bits)
    lut = np.stack([x ** (2.0 + 0.1 * k) for k in range(c)], axis=1)
    dlut = np.stack([np.gradient(lut[:, k], 2 / (bits - 1)) for k in range(c)], axis=1)
    std_lut = None
    if std_kind == "monotone":
        std_lut = np.stack([0.002 + 0.02 * np.sqrt(x) * (1 + 0.1 * k) for k in range(c)], axis=1)
    elif std_kind == "wild":
        std_lut = 0.002 + 0.02 * (0.3 + np.abs(np.sin(9 * x)))[:, None] * rng.uniform(0.5, 1.5, (bits, c))
    return lut, dlut, std_lut


def _repair(dn, sg, hot, K):
    """bad-pixel repair of one exposure: the K x K median (scipy 'reflect', rank K*K//2) of the DNs and of the
    uncertainties where `hot`"""
    med_d = median_filter(dn, size=(K, K), axes=(0, 1), mode="reflect")
    med_s = median_filter(sg, size=(K, K), axes=(0, 1), mode="reflect")
    return np.where(hot, med_d, dn), np.where(hot, med_s, sg)


class Ref:
    """Extended-precision evaluation of the merge formula (module docstring) and the per-sample error bounds."""

    def __init__(self, d, s, t, lut, dlut, max_dn):
        n = len(d)
        self.n = n
        shape = d[0].shape
        c = np.broadcast_to(np.arange(shape[-1]), shape)
        wt, kt = _weights(max_dn), _kappa(max_dn)
        f = lambda v: np.asarray(v, dtype=np.float64)
        S = sum(LD(1) * wt[dk] for dk in d)
        rS = f(1 / S)
        z0 = np.zeros(shape, dtype=LD)
        val, q, A, B, C = z0.copy(), z0.copy(), z0.copy(), z0.copy(), z0.copy()
        z64 = np.zeros(shape)
        var2, aXmX, cross, aE2, aEq, sXE = z64.copy(), z64.copy(), z64.copy(), z64.copy(), z64.copy(), z64.copy()
        for k, dk in enumerate(d):                 # one exposure at a time: dense windows stay small in memory
            w, g, kap = LD(1) * wt[dk], LD(1) * lut[dk, c], LD(1) * kt[dk]
            dg = LD(1) * dlut[dk, c] * s[k]
            rt = LD(1.0 / float(t[k]))
            x = kap * w * g + w * dg
            e = kap * w * w * g
            y = dg * rt
            X, E, Z = x * y, e * y, (x - e / S) * y
            val += w * g * rt
            q += Z * Z
            A += X * X
            B += X * E
            C += E * E
            ay, absq = np.abs(f(y)), np.abs(f(Z))
            parts = np.abs(f(kap * w * g)) + np.abs(f(w * dg))
            # two-pass: |dz| <= (N + 5) u (|kappa w g| + |w dg| + |e rS|), |dq| <= |y| (|dz| + 3.02 u |z|)
            dq = ay * ((n + 5) * U * (parts + np.abs(f(e)) * rS) + 3.02 * U * np.abs(f(x - e / S)))
            var2 += 2 * absq * dq + dq ** 2
            # single-pass: |X^ - X| <= 6.1 u mX, mX = (|kappa w g| + |w dg|) |y|; the same for E with |E|
            mX, aX, aE = parts * ay, np.abs(f(X)), np.abs(f(E))
            aXmX += aX * mX
            cross += aX * aE + aE * mX
            aE2 += aE * aE
            aEq += aE * absq
            sXE += aX * aE
        self.S = S
        self.val = val / S
        self.q, self.A, self.B, self.C = q, A, B, C
        self.std = np.sqrt(q) / S
        q64, A64, C64 = f(q), f(A), f(C)
        with np.errstate(divide="ignore", invalid="ignore"):
            self.rel_std2 = 1.01 * (0.5 * (var2 / q64 + (n + 0.01) * U) + (n + 2.1) * U)
        self.rel_val = (2 * n + 4) * U
        # single-pass: the sums round N times each, expanded_variance three times, rS carries (N + 0.01) u
        dqs = U * (12.2 * aXmX + (n + 1) * A64 + 2 * rS * (6.1 * cross + (n + 1) * sXE)
                   + rS * rS * (12.2 * aE2 + (n + 1) * C64) + 2 * (n + 0.01) * rS * aEq + q64)
        self.dq1 = 1.01 * dqs
        with np.errstate(divide="ignore", invalid="ignore"):
            self.rel_q1 = 1.01 * dqs / q64
            self.rel_std1 = 0.5 * self.rel_q1 + 1.01 * (n + 2.1) * U
        # the scale of the single-pass rounding error, which the fix-up rule compares q with (expansion_cancelled)
        self.scale = A64 + 2 * np.abs(f(B)) * rS + C64 * rS * rS

    def flat(self, fval, fstd, m, ms, single_pass):
        """flat_apply() on the exact reciprocal of the flat value: (val', std', rel bound val', rel bound std')"""
        rf = 1 / (LD(1) * fval)
        mm, mms = LD(1) * m, LD(1) * ms
        var = self.std * self.std
        vr = self.val * rf
        t1 = var * (rf * mm) ** 2
        t2 = (vr * rf * fstd * mm) ** 2
        t3 = (vr * mms) ** 2
        rad = t1 + t2 + t3
        f = lambda v: np.asarray(v, dtype=np.float64)
        rel_var = (self.rel_q1 + (2 * self.n + 3) * U) if single_pass else 2 * self.rel_std2 + 3 * U
        rv = self.rel_val
        with np.errstate(all="ignore"):
            rel = 1.01 * (0.5 * ((rel_var + 6 * U) * f(t1) + 2 * (rv + 6 * U) * f(t2) + 2 * (rv + 3 * U) * f(t3))
                          / f(rad) + 2 * U)
        return f(vr * mm), f(np.sqrt(rad)), rv + 4 * U, rel


def _rel_err(got, ref):
    ref = np.asarray(ref, dtype=np.longdouble)
    with np.errstate(all="ignore"):
        return np.asarray(np.abs(got - ref) / np.abs(ref), dtype=np.float64)


def _same_class(got, exp):
    """NaN / +inf / -inf / 0 class of every output as the oracle's"""
    for pred in (np.isnan, np.isposinf, np.isneginf, lambda a: a == 0):
        np.testing.assert_array_equal(pred(got), pred(exp))


def _check(got, ref, bound, tight=TIGHT, where=None):
    """finite, non-zero samples: within their own bound and within `tight`; returns the worst relative error"""
    ok = np.isfinite(got) & (np.asarray(ref, dtype=np.float64) != 0) & np.isfinite(np.asarray(ref, dtype=np.float64))
    if where is not None:
        ok &= where
    err = _rel_err(got[ok], ref[ok])
    b = np.broadcast_to(bound, got.shape)[ok]
    bad = err > b
    assert not bad.any(), f"{int(bad.sum())} samples beyond their bound, e.g. err {err[bad][:4]} bound {b[bad][:4]}"
    if tight is not None:
        assert err.max(initial=0.0) <= tight, err.max()
    return float(err.max(initial=0.0))


# ---------------------------------------------------------------------------------------------------------------------
# the weight table

@pytest.mark.parametrize("max_dn", [255, 65535])
def test_gaussian_weight_of_every_dn_within_one_ulp(max_dn):
    """w[d] = exp(-30 (d/MAX - 0.5)^2) for every DN, the argument in NumPy's double operations: within 1 ulp of mpmath's
    exp of that argument (the merge kernels build their tables with the same device function)."""
    mpmath = pytest.importorskip("mpmath")
    v = np.arange(max_dn + 1) / float(max_dn)
    c = v - 0.5
    arg = -30.0 * (c * c)
    w = _weights(max_dn)
    mpmath.mp.prec = 120
    ref = np.array([float(mpmath.exp(mpmath.mpf(float(a)))) for a in arg])
    ulps = np.abs(w - ref) / np.spacing(ref)
    assert ulps.max() <= 1.0, (int(np.argmax(ulps)), float(ulps.max()))
    with np.errstate(all="ignore"):
        ew, _ = om.gaussian_weight(v)
    assert np.max(np.abs(w - ew) / ew) < 12 * U      # the oracle's np.e ** x: e rounded, times |x| <= 7.5


# ---------------------------------------------------------------------------------------------------------------------
# every kernel instance

def _stack(rng, n, h, w, c, max_dn, std_kind, darks, K, flat, thr=0.03, edge_flat=False):
    """a seeded stack with what each case needs; returns (kwargs for ops.hdr_merge, host data for the reference)"""
    dt = np.uint8 if max_dn == 255 else np.uint16
    t = 0.002 * 1.5 ** np.arange(n)
    rad = rng.uniform(0, 1, (h, w, c)) * 25
    dn = [np.rint(max_dn * np.clip(rad * tk, 0, 1) ** (1 / 2.2)).astype(dt) for tk in t]
    bits = max_dn + 1
    lut, dlut, std_lut = _tables(c, bits, rng, {"images": None, "mixed": "monotone"}.get(std_kind, std_kind))
    if std_kind == "images":
        sg_img = [rng.uniform(0.002, 0.02, (h, w, c)) for _ in t]
        std_dev = [dev(s) for s in sg_img]
    elif std_kind == "mixed":
        sg_img = [rng.uniform(0.002, 0.02, (h, w, c)) if k % 3 == 0 else None for k in range(n)]
        std_dev = [None if s is None else dev(s) for s in sg_img]
    else:
        sg_img = [None] * n
        std_dev = None
    cidx = np.broadcast_to(np.arange(c), (h, w, c))
    sg = [s if s is not None else std_lut[d, cidx] for s, d in zip(sg_img, dn)]
    kw = dict(std_lut=None if std_lut is None else dev(std_lut), median_kernel=K)
    d_rep, s_rep = list(dn), list(sg)
    if darks:
        dk = []
        for k in range(n):
            if k % 2 == 0 and k < n - 1 and n > 1:
                dk.append(None)
                continue
            f = rng.poisson(2.0, (h, w, c)).astype(dt)
            hot = rng.uniform(size=f.shape) < 0.02
            f[hot] = rng.integers(max_dn // 20, max_dn, int(hot.sum()))
            f.reshape(-1)[:c] = max_dn                     # image corner
            f.reshape(-1)[-c:] = max_dn
            dk.append(f)
        scales = [1.0 if k % 3 else 1.25 for k in range(n)]
        for k, f in enumerate(dk):
            if f is not None:
                hot = om.dark_value_image(f, scales[k], max_dn=max_dn) > thr
                d_rep[k], s_rep[k] = _repair(dn[k], sg[k], hot, K)
        kw.update(darks=[None if f is None else _dev_dn(f) for f in dk], dark_scales=scales, dark_threshold=thr)
    fl = None
    if flat:
        if flat == 8:
            fv = rng.uniform(0.4, 1.0, (h, w, c))
            fv.reshape(-1)[:5] = [0.0, 1.0, 1e-300, 0.5, 1.0 - 2 ** -52]
            fdev = dev(fv)
        else:
            fdt = np.uint8 if flat == 1 else np.uint16
            fmax = 255 if flat == 1 else 65535
            fd = rng.integers(fmax // 2, fmax + 1, (h, w, c)).astype(fdt)
            if edge_flat:
                fd.reshape(-1)[::7] = 0
                fd.reshape(-1)[3::7] = fmax
            fdev = _dev_dn(fd)
            fv = fd / float(max_dn)          # the kernels scale an integer flat by the stack's MAX
        fs = rng.uniform(0.001, 0.01, (h, w, c))
        means = np.concatenate([rng.uniform(0.6, 0.9, c), rng.uniform(0.002, 0.006, c)])
        kw.update(flat=fdev, flat_std=dev(fs), flat_means=dev(means))
        fl = (fv, fs, means[cidx], means[c + cidx])
    host_data = dict(dn=[_dev_dn(d) for d in dn], std=std_dev, t=[float(x) for x in t], icrf=dev(lut), dlut=dev(dlut),
                     d_rep=d_rep, s_rep=s_rep, lut=lut, dl=dlut, flat=fl, max_dn=max_dn, sg=sg, dn_h=dn)
    return kw, host_data


def _oracle(hd, kw):
    """the NumPy oracle on the same repaired inputs: only its NaN / inf / 0 class is used"""
    d, s = hd["d_rep"], hd["s_rep"]
    lut, dl = hd["lut"], hd["dl"]
    c = lut.shape[1]
    with np.errstate(all="ignore"):
        ev, es = om.hdr_merge(d, s, np.array(hd["t"]), lut[:, 0] if c == 1 else lut, dl[:, 0] if c == 1 else dl,
                              max_dn=hd["max_dn"])
        if hd["flat"] is not None:
            fv, fs, m, ms = hd["flat"]
            ev, es = om.normalize_by_map(ev, es, fv, fs, None, means=(m, ms))
    return ev, es


def _run_case(kw, hd, algo, single_pass):
    v, s = ops.hdr_merge(hd["dn"], hd["std"], hd["t"], hd["icrf"], hd["dlut"], algo=algo, **kw)
    v, s = host(v), host(s)
    r = Ref(hd["d_rep"], hd["s_rep"], hd["t"], hd["lut"], hd["dl"], hd["max_dn"])
    if hd["flat"] is None:
        rv, rs, bv, bs2, bs1 = r.val, r.std, r.rel_val, r.rel_std2, r.rel_std1
    else:
        rv, rs, bv, bs2 = r.flat(*hd["flat"], False)
        bs1 = r.flat(*hd["flat"], True)[3]
    ev, es = _oracle(hd, kw)
    _same_class(v, ev)
    _same_class(s, es)
    _check(v, rv, bv)
    if single_pass:
        # the fix-up pass gives flagged samples the two-pass bits; every other sample meets its own bound and STREAM
        v1, s1 = (host(x) for x in ops.hdr_merge(hd["dn"], hd["std"], hd["t"], hd["icrf"], hd["dlut"], algo=1, **kw))
        assert np.array_equal(v, v1, equal_nan=True)
        two_pass = s == s1
        _check(s, rs, bs2, where=two_pass)
        _check(s, rs, bs1, tight=STREAM, where=~two_pass)
    else:
        _check(s, rs, bs2)
    return r


# (id, stack arguments, algo, expected kernel instance, single pass)
def _inst(id_, algo, kernel, single=False, **kw):
    base = dict(n=4, h=19, w=23, c=3, max_dn=255, std_kind="images", darks=False, K=3, flat=0)
    base.update(kw)
    return pytest.param(base, algo, kernel, single, id=id_)


INSTANCES = (
    [_inst(f"generic_u8_c{c}", 1, GEN8, c=c, darks=c % 2 == 1, flat=1 if c < 5 else 8) for c in range(1, 9)]
    + [_inst("generic_u8_c4_table_wild", 1, GEN8, c=4, std_kind="wild", darks=True, flat=2),
       _inst("generic_u16_images", 1, GEN16, n=5, max_dn=65535, c=2),
       _inst("generic_u16_table", 1, GEN16, n=6, max_dn=65535, c=3, std_kind="monotone", darks=True, flat=2),
       _inst("generic_u16_n20_dark_flat", 0, GEN16, n=20, max_dn=65535, c=1, darks=True, flat=2, h=21, w=37)]
    + [_inst(f"staged_{n}_{'mono' if c == 1 else 'rgb'}", 2, f"merge_staged_kernel<{tn},{str(c == 1).lower()}>",
             n=n, c=c, h=24 if c == 3 else 40, w=75 if c == 3 else 101, darks=n <= 16, flat=1 if n <= 16 else 0, K=5)
       for n, tn in ((1, 8), (5, 8), (16, 16), (17, 32), (32, 32)) for c in (3, 1)]
    + [_inst(f"staged_table_{n}_{'mono' if c == 1 else 'rgb'}", 2, f"merge_staged_lut_kernel<{tn},{str(c == 1).lower()}>",
             n=n, c=c, h=24 if c == 3 else 40, w=75 if c == 3 else 101, std_kind="wild", darks=True, flat=1)
       for n, tn in ((6, 8), (13, 16)) for c in (3, 1)]
    + [_inst(f"single_pass_{kind}_{n}_{'mono' if c == 1 else 'rgb'}", 4,
             f"merge_stream{'_lut' if kind == 'table' else ''}_kernel<{str(c == 1).lower()}>", single=True,
             n=n, c=c, h=33 if c == 3 else 45, w=64 if c == 3 else 101, std_kind="images" if kind == "images" else "wild",
             darks=n == 32, flat=(1 if n == 32 else (8 if n == 17 else 0)))
       for kind in ("images", "table") for n in (2, 16, 17, 32) for c in (3, 1)]
    + [_inst("single_pass_flat_u16_bytes", 4, "merge_stream_kernel<false>", single=True, n=5, h=32, w=48, flat=2),
       _inst("single_pass_flat_edges", 4, "merge_stream_kernel<false>", single=True, n=5, h=32, w=48, flat=1,
             edge_flat=True),
       _inst("staged_flat_edges", 2, "merge_staged_kernel<8,false>", n=5, h=32, w=48, flat=1, edge_flat=True),
       _inst("generic_flat_edges", 1, GEN8, n=5, h=17, w=29, flat=1, edge_flat=True),
       _inst("single_pass_mono_rows_cross_tiles", 4, "merge_stream_kernel<true>", single=True, n=3, c=1, h=37, w=83,
             darks=True, K=3)]
    + [_inst(f"wide_pipe_{n}_{tab}", 3, f"merge_wide_pipe_kernel<{tn},{th},{str(tab == 'table').lower()}>",
             n=n, max_dn=65535, c=3 if n % 2 else 1, h=17, w=45, std_kind="images" if tab == "images" else "monotone",
             darks=n > 4, flat=2 if n > 8 else 0)
       for tab in ("images", "table")
       for n, tn, th in ((3, 4, 192), (7, 8, 192), (10, 12, 192 if tab == "images" else 128), (16, 16, 128))]
    + [_inst(f"wide_mixed_{n}", 3, f"merge_wide_kernel<{tn},true>", n=n, max_dn=65535, c=3, h=17, w=45,
             std_kind="mixed", darks=True, flat=2)
       for n, tn in ((5, 8), (11, 12), (14, 16))]
)


def _instance_stack(args):
    rng = np.random.default_rng(zlib.crc32(repr(sorted(args.items())).encode()))
    return _stack(rng, **args)


def collect_kernel_names():
    """{"instances": {case id: kernels}, "roi": {C: kernels}} of every instance case and of cl_flat_roi_means for
    C = 1 ... 8, each group from one profiler session; None for a group when the profiler records nothing.  Run in a
    process of its own (test_every_case_launches_its_kernel_instance) so that the answer does not depend on how many
    profiler sessions the test process has already opened."""
    _weights(255), _weights(65535)                  # (their gaussian_weight launches must not land in a session)
    cases = []
    for p in INSTANCES:
        args, algo = p.values[0], p.values[1]
        kw, hd = _instance_stack(args)
        cases.append((p.id, lambda kw=kw, hd=hd, algo=algo: ops.hdr_merge(hd["dn"], hd["std"], hd["t"], hd["icrf"],
                                                                           hd["dlut"], algo=algo, **kw)))
    flat = torch.full((8, 8, 8), 0.5, dtype=torch.float64, device="cuda")
    planes = [flat[..., :c].contiguous() for c in range(1, 9)]
    roi = _profiled_cases([(str(c), lambda c=c: ops.flat_roi_means(planes[c - 1], planes[c - 1], (0, 8, 0, 8)))
                           for c in range(1, 9)])
    return {"instances": _profiled_cases(cases), "roi": roi}


def test_every_case_launches_its_kernel_instance():
    """Which kernel instance each case of test_kernel_instance_against_reference runs (and the generic kernel on the
    ragged tail of a tile stack), and roi_partial_kernel<1 | 3 | 0> for C = 1, 3 and the rest, named by torch.profiler
    in a fresh process.  Skipped, visibly, where the profiler records no device activity."""
    tests_dir = Path(__file__).resolve().parent
    code = ("import json, sys; sys.path[:0] = [sys.argv[1], sys.argv[2]]; import test_gpu_hdr_merge_paths as m; "
            "print('NAMES ' + json.dumps(m.collect_kernel_names()))")
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, "-c", code, str(tests_dir), str(tests_dir.parent)], capture_output=True,
                       text=True, timeout=900, cwd=tests_dir.parent)
    assert r.returncode == 0, r.stderr[-3000:]
    names = json.loads(next(line for line in r.stdout.splitlines() if line.startswith("NAMES "))[6:])
    if names["instances"] is None or names["roi"] is None:
        pytest.skip("the profiler records no device activity here")
    for p in INSTANCES:
        args, algo, kernel = p.values[0], p.values[1], p.values[2]
        got = names["instances"][p.id]
        assert kernel in got, (p.id, got)
        if algo in (2, 4) and (args["h"] * args["w"] * args["c"]) % TILE:
            assert GEN8 in got, (p.id, got)            # the ragged tail
    for c in range(1, 9):
        assert names["roi"][str(c)] == [f"roi_partial_kernel<{c if c in (1, 3) else 0}>"], (c, names["roi"][str(c)])


@pytest.mark.parametrize("args,algo,kernel,single", INSTANCES)
def test_kernel_instance_against_reference(args, algo, kernel, single):
    """One kernel instance on a seeded stack (test_every_case_launches_its_kernel_instance checks that `kernel` is what
    runs): radiance within (2N + 4) u (+ 4 u with a flat),
    two-pass uncertainty within 1.01 (|dvar| / 2 var + (N + 2.1) u) with |dq_k| <= |y|((N + 5) u (|kappa w g| + |w dg|
    + |e rS|) + 3.02 u |z|) propagated through the sum of squares, both also within 1e-11; single-pass uncertainty of
    an unflagged sample within |dq| / 2q + (N + 2.1) u with |dq| <= u (L (A + 2|B| rS + C rS^2) + perturbation
    terms) (Ref) and within 1e-9, a flagged one bit-identical to the two-pass kernel; the flat epilogue adds its own
    terms (Ref.flat); NaN / inf / 0 class as the oracle's."""
    kw, hd = _instance_stack(args)
    _run_case(kw, hd, algo, single)


# ---------------------------------------------------------------------------------------------------------------------
# the single-pass fix-up rule: samples around q = kStreamCancel * A

def _workspace(n_samples):
    """a workspace laid out as merge_workspace() does for an 8-bit tile stack, and the byte offset of its work list"""
    tiles = n_samples // TILE
    hot_cap = max(n_samples // 16, 65536)
    list_off = tiles * 16
    total = list_off + (4 + hot_cap) * 4 + 16 + tiles * 32 * 16
    return torch.zeros(total, dtype=torch.uint8, device="cuda"), list_off, hot_cap


def _work_list(ws, list_off):
    lst = host(ws[list_off:].view(torch.int32))
    return int(lst[0]), lst[4:4 + int(lst[0])]


def _window_stack(rng, n, h, w, c, mode, dense=False):
    """DNs in 140 ... 254 (kappa < 0) and uncertainties chosen so that x_k - e_k / S cancels to a ratio sqrt(rho) of
    x_k in every exposure: q / A lands near rho, and C rS^2 ~ B rS ~ A (the expansion's worst case).  With
    w_k / S = p_k:  x_k - e_k / S = w_k kappa g (1 - p_k) + w_k dg, which is -w_k kappa g (1 - p_k) eps_k for
    dg = -kappa g (1 - p_k)(1 + eps_k), eps_k = sqrt(rho) p_k / ((1 - p_k)(1 + sqrt(rho))).  rho is log-uniform over
    [1e-7, 1e-4]; dense: a quarter of the samples uniform in q / A in [1e-6, 1.5e-6] (where a test against A alone
    would have let them through) and the rest uniform in q / scale in [1e-6, 1.5e-6], just above the threshold.
    mode "table": every exposure of a sample has the same DN, so p_k = 1/N and the uncertainty is a function of
    (DN, channel): the camera's STD table."""
    shape = (h, w, c)
    cidx = np.broadcast_to(np.arange(c), shape)
    lut, dlut, _ = _tables(c, 256)
    wt, kt = _weights(255), _kappa(255)
    t = 0.002 * 1.5 ** np.arange(n)

    def uncertainties(d, rho):
        S = sum(wt[dk] for dk in d)
        sg = []
        for dk in d:
            p = wt[dk] / S
            eps = np.sqrt(rho) * p / ((1 - p) * (1 + np.sqrt(rho)))
            sg.append(-kt[dk] * lut[dk, cidx] * (1 - p) * (1 + eps) / dlut[dk, cidx])
        return sg

    if mode == "images":
        d = [rng.integers(140, 255, shape).astype(np.uint8) for _ in range(n)]
        if not dense:
            return d, uncertainties(d, 10.0 ** rng.uniform(-7, -4, shape)), t, lut, dlut, None
        # scale / A of each sample (it hardly depends on rho this close to the threshold), in double
        sg = uncertainties(d, np.full(shape, 1e-6))
        S = sum(wt[dk] for dk in d)
        A = B = C = 0.0
        for k, dk in enumerate(d):
            g, dg = lut[dk, cidx], dlut[dk, cidx] * sg[k]
            y = dg / t[k]
            X, E = (kt[dk] * wt[dk] * g + wt[dk] * dg) * y, kt[dk] * wt[dk] ** 2 * g * y
            A, B, C = A + X * X, B + X * E, C + E * E
        ratio = (A + 2 * np.abs(B) / S + C / S ** 2) / A
        rho = rng.uniform(1e-6, 1.5e-6, shape) * np.where(rng.uniform(size=shape) < 0.25, 1.0, ratio)
        return d, uncertainties(d, rho), t, lut, dlut, None
    p = 1.0 / n
    rho_tab = 10.0 ** rng.uniform(-7, -4, (256, c))
    eps = np.sqrt(rho_tab) * p / ((1 - p) * (1 + np.sqrt(rho_tab)))
    dd = np.arange(256)[:, None]
    std_lut = np.where(dd >= 140, -kt[dd] * lut * (1 - p) * (1 + eps) / np.where(dlut > 0, dlut, 1.0), 0.01)
    d0 = rng.integers(140, 255, shape).astype(np.uint8)
    d = [d0] * n
    sg = [std_lut[d0, cidx]] * n
    return d, sg, t, lut, dlut, std_lut


WINDOW = ([pytest.param(n, mode, 3, False, id=f"{mode}_n{n}_c3") for mode in ("images", "table") for n in (2, 8, 16, 32)]
          + [pytest.param(16, "images", 1, False, id="images_n16_c1"), pytest.param(8, "table", 1, False, id="table_n8_c1"),
             pytest.param(32, "images", 3, True, id="dense_images_n32_c3"),
             pytest.param(16, "images", 3, True, id="dense_images_n16_c3")])


@pytest.mark.parametrize("n,mode,c,dense", WINDOW)
def test_single_pass_threshold_window(n, mode, c, dense):
    """Samples whose expanded variance keeps q / A in [1e-7, 1e-4], on the single-pass kernel with uncertainty images
    (stream_mode 1) and with the STD table (stream_mode 2); the dense cases put 147 000 samples just above the
    threshold and 49 000 at q / A in [1e-6, 1.5e-6].  The fix-up rule flags q < 1e-6 scale, scale = A + 2|B| rS + C rS^2
    (expansion_cancelled).  The flag decision itself, read from the work list: every sample that is below the threshold
    whatever the rounding (q + |dq| < 1e-6 (scale - |dscale|)(1 - u)) is on it, every sample that is above it whatever
    the rounding is not.  Flagged samples carry the two-pass bits; every other sample is within its own bound
    |dq| / 2q + (N + 2.1) u, |dq| <= u (L scale + perturbation terms) (Ref), and within STREAM = 1e-9 -- for which
    the bound alone, ~L u 1e6 / 2 at q = 1e-6 scale, does not vouch: this is measured.
    The reference is the long-double Ref, not exact rational sums: the construction cancels x - e / S to at worst
    sqrt(1e-7) ~ 3e-4 of x, so long double's 2^-64 leaves the reference uncertainty within ~2e-16 relative, six
    orders below the errors measured here."""
    rng = np.random.default_rng(7000 + 10 * n + c + (1 if mode == "table" else 0) + (5 if dense else 0))
    h, w = (256, 256) if dense else ((32, 96) if c == 3 else (96, 96))
    d, sg, t, lut, dlut, std_lut = _window_stack(rng, n, h, w, c, mode, dense)
    ws, list_off, hot_cap = _workspace(h * w * c)
    args = ([dev(x) for x in d], None if mode == "table" else [dev(x) for x in sg], [float(x) for x in t], dev(lut),
            dev(dlut))
    kw = dict(std_lut=None if std_lut is None else dev(std_lut))
    v4, s4 = ops.hdr_merge(*args, algo=4, workspace=ws, **kw)
    count, flagged = _work_list(ws, list_off)
    assert count <= hot_cap
    v4, s4 = host(v4), host(s4)
    v1, s1 = (host(x) for x in ops.hdr_merge(*args, algo=1, **kw))
    assert np.array_equal(v4, v1)
    r = Ref(d, sg, t, lut, dlut, 255)
    f = lambda a: np.asarray(a, dtype=np.float64).reshape(-1)
    q, A, scale, dq = f(r.q), f(r.A), f(r.scale), f(r.dq1)
    dscale = dq + 4 * U * scale
    rho, rel = q / A, q / scale
    surely_below = q + dq < CANCEL * (scale - dscale) * (1 - U)
    surely_above = q - dq >= CANCEL * (scale + dscale) * (1 + U)
    is_flagged = np.zeros(q.size, dtype=bool)
    is_flagged[flagged] = True
    assert len(set(flagged.tolist())) == count
    assert is_flagged[surely_below].all(), int((~is_flagged[surely_below]).sum())
    assert not is_flagged[surely_above].any(), int(is_flagged[surely_above].sum())
    just_above = ((rel > 1e-6) & (rel < 1.5e-6) & surely_above).sum()
    if dense:
        assert just_above > 100_000, just_above
        assert ((rho > 1e-6) & (rho < 1.5e-6) & surely_below).sum() > 40_000
    else:
        assert surely_below.sum() > 200 and surely_above.sum() > 200
        assert just_above > 20
    s4f, s1f = s4.reshape(-1), s1.reshape(-1)
    assert np.array_equal(s4f[is_flagged], s1f[is_flagged])
    _check(s1f, f(r.std), f(r.rel_std2), tight=None)
    err = _rel_err(s4f[~is_flagged], np.asarray(r.std, dtype=LD).reshape(-1)[~is_flagged])
    bound = f(r.rel_std1)[~is_flagged]
    assert (err <= bound).all(), (float(err.max()), int((err > bound).sum()))
    worst = float(err.max())
    k = int(np.argmax(err))
    print(f"\nsingle-pass window {mode} N={n} C={c}{' dense' if dense else ''}: {int(is_flagged.sum())} of {q.size} "
          f"flagged; worst unflagged std error {worst:.3e} at q/A = {rho[~is_flagged][k]:.4e}, q/scale = "
          f"{rel[~is_flagged][k]:.4e}, its bound {bound[k]:.3e}")
    assert worst <= STREAM, worst


# ---------------------------------------------------------------------------------------------------------------------
# bad pixels

def _hd(dn, sg, t, lut, dlut, d_rep, s_rep, max_dn=255, std_images=True):
    dev_sg = [dev(x) for x in sg] if std_images else None
    return dict(dn=[_dev_dn(x) for x in dn], std=dev_sg, t=[float(x) for x in t], icrf=dev(lut), dlut=dev(dlut),
                d_rep=d_rep, s_rep=s_rep, lut=lut, dl=dlut, flat=None, max_dn=max_dn)


@pytest.mark.parametrize("scale", [1.0, 1.37])
def test_every_integer_dark_threshold(scale):
    """The host turns dark_threshold into hot_dn, the lowest dark DN whose value (d / 255) [* scale] exceeds it, and
    dark_scan_kernel tests four bytes at once (bytes_ge: one branch for hot_dn <= 128, one above).  Thresholds exactly
    at, and one ulp either side of, the value of every DN reach every hot_dn from 0 to 256; the dark frame holds every
    DN value; 1581 samples = one tile + a ragged 45 (n % 16 != 0).  The output of every sample must be the repaired or
    the unrepaired one as NumPy's comparison says, on the generic kernel and on the scan + tile kernel."""
    rng = np.random.default_rng(256 + int(scale * 100))
    h, w, c, n = 17, 31, 3, 2
    t = np.array([0.004, 0.009])
    lut, dlut, _ = _tables(c, 256)
    dn = [rng.integers(0, 256, (h, w, c)).astype(np.uint8) for _ in range(n)]
    sg = [rng.uniform(0.002, 0.02, (h, w, c)) for _ in range(n)]
    dark = rng.permutation(np.arange(h * w * c) % 256).astype(np.uint8).reshape(h, w, c)
    K = 3
    d_hot, s_hot = _repair(dn[1], sg[1], np.ones(dn[1].shape, dtype=bool), K)
    cold = Ref(dn, sg, t, lut, dlut, 255)
    hot = Ref([dn[0], d_hot], [sg[0], s_hot], t, lut, dlut, 255)
    dval = om.dark_value_image(dark, scale)
    distinct = _rel_err(np.asarray(cold.std, dtype=np.float64), hot.std) > 1e-6
    assert distinct.mean() > 0.8
    args = ([dev(x) for x in dn], [dev(x) for x in sg], [float(x) for x in t], dev(lut), dev(dlut))
    dev_dark = [None, dev(dark)]
    levels = np.arange(256) / 255.0
    if scale != 1.0:
        levels = levels * np.array([scale])
    thresholds = [-1.0] + [x for lv in levels for x in (np.nextafter(lv, -np.inf), lv, np.nextafter(lv, np.inf))]
    seen = set()
    for thr in thresholds:
        thr = float(thr)
        mask = dval > thr
        ok_dn = np.flatnonzero(levels > thr)
        seen.add(int(ok_dn[0]) if ok_dn.size else 256)
        ev = np.where(mask, hot.val, cold.val)
        es = np.where(mask, hot.std, cold.std)
        for algo in (1, 4):
            v, s = ops.hdr_merge(*args, algo=algo, darks=dev_dark, dark_scales=[1.0, scale], dark_threshold=thr,
                                 median_kernel=K)
            v, s = host(v), host(s)
            assert _rel_err(v, ev).max() <= TIGHT, (thr, algo)
            bad = _rel_err(s, es) > 1e-9
            assert not bad.any(), (thr, algo, int(bad.sum()), dark[bad][:8])
    assert seen == set(range(257))


def _narrow_case(rng, shape, K, n=3, ties=True):
    h, w, c = shape
    t = 0.003 * 1.6 ** np.arange(n)
    lut, dlut, _ = _tables(c, 256)
    vals = np.array([40, 41, 120, 200], dtype=np.uint8)
    dn = [(rng.choice(vals, shape) if ties else rng.integers(0, 256, shape)).astype(np.uint8) for _ in range(n)]
    sg = [rng.choice([0.004, 0.005, 0.011], shape) for _ in range(n)]
    darks, d_rep, s_rep = [None], [dn[0]], [sg[0]]
    thr = 0.1
    for k in range(1, n):
        f = np.where(rng.uniform(size=shape) < 0.3, 200, 3).astype(np.uint8)
        f.reshape(h, w, c)[0, 0] = 200
        f.reshape(h, w, c)[-1, -1] = 200
        f.reshape(h, w, c)[0, -1] = 200
        f.reshape(h, w, c)[-1, 0] = 200
        darks.append(f)
        dr, sr = _repair(dn[k], sg[k], om.dark_value_image(f, 1.0) > thr, K)
        d_rep.append(dr)
        s_rep.append(sr)
    kw = dict(darks=[None if f is None else dev(f) for f in darks], dark_threshold=thr, median_kernel=K)
    return kw, _hd(dn, sg, t, lut, dlut, d_rep, s_rep)


NARROW = [(1536, 1, 1), (1, 1536, 1), (768, 2, 1), (2, 768, 1), (512, 1, 3), (1, 512, 3), (3, 5, 3), (5, 4, 1)]


@pytest.mark.parametrize("K", range(1, 8))
def test_median_kernels_at_image_edges(K):
    """Bad-pixel repair with K = 1 ... 7 (even K: the window is [-K/2, K/2 - 1], rank K*K/2) at image corners, on images
    1 and 2 pixels wide or high and narrower than K (reflect_index reflects more than once), with ties among the DNs
    and the uncertainties; K = 3 on the tile kernels takes the 9-element selection network, every other K the
    selection sort.  Generic, staged and single-pass kernels where the stack is a tile stack."""
    rng = np.random.default_rng(4000 + K)
    for shape in NARROW:
        kw, hd = _narrow_case(rng, shape, K)
        tile = shape[0] * shape[1] * shape[2] >= TILE
        for algo in ((1, 2, 4) if tile else (1,)):
            _run_case(kw, hd, algo, single_pass=algo == 4)


def _spiky_stack(rng, h, w, c, n):
    t = 0.003 * 1.6 ** np.arange(n)
    lut, dlut, _ = _tables(c, 256)
    dn = [rng.integers(100, 110, (h, w, c)).astype(np.uint8) for _ in range(n)]
    sg = [rng.uniform(0.002, 0.02, (h, w, c)) for _ in range(n)]
    return t, lut, dlut, dn, sg


@pytest.mark.parametrize("algo", [2, 4])
def test_bucket_of_exactly_32_and_33_bad_pairs(algo):
    """A tile's bucket holds kBucketCap = 32 bad (sample, exposure) pairs; the 33rd goes to the work list.  Tile 0 has
    exactly 32 pairs, tile 1 exactly 33, tile 2 none; every bad sample is a spike (DN 250 among 100 ... 109), so a
    missed repair shows.  The work list of the staged kernel holds exactly the one overflowing pair."""
    rng = np.random.default_rng(3233)
    h, w, c, n = 3, 512, 3, 3                  # one 512-pixel row per tile
    t, lut, dlut, dn, sg = _spiky_stack(rng, h, w, c, n)
    darks = [np.zeros((h, w, c), dtype=np.uint8) for _ in range(n)]
    for row, pairs in ((0, 32), (1, 33)):
        cells = rng.choice(w * c, pairs, replace=False)
        for j, cell in enumerate(cells):
            k = j % n
            darks[k][row].reshape(-1)[cell] = 255
            dn[k][row].reshape(-1)[cell] = 250
    d_rep, s_rep = [], []
    for k in range(n):
        dr, sr = _repair(dn[k], sg[k], om.dark_value_image(darks[k], 1.0) > 0.5, 3)
        d_rep.append(dr)
        s_rep.append(sr)
    hd = _hd(dn, sg, t, lut, dlut, d_rep, s_rep)
    kw = dict(darks=[dev(f) for f in darks], dark_threshold=0.5, median_kernel=3)
    _run_case(kw, hd, algo, single_pass=algo == 4)
    ws, list_off, _ = _workspace(h * w * c)
    ops.hdr_merge(hd["dn"], hd["std"], hd["t"], hd["icrf"], hd["dlut"], algo=algo, workspace=ws, **kw)
    count, lst = _work_list(ws, list_off)
    if algo == 2:
        assert count == 1 and lst[0] // (w * c) == 1, (count, lst)
    else:
        assert count >= 1 and (lst // (w * c) == 1).sum() >= 1


@pytest.mark.parametrize("algo", [2, 4])
def test_work_list_overflow(algo):
    """Every dark sample above the threshold: 11 tiles x (4 x 1536 - 32) = 67 232 pairs miss their buckets, more than
    the 65 536 the work list holds, so merge_fixup_kernel rescans the image."""
    rng = np.random.default_rng(65536 + algo)
    h, w, c, n = 88, 64, 3, 4
    t, lut, dlut, dn, sg = _spiky_stack(rng, h, w, c, n)
    dn = [rng.integers(0, 256, (h, w, c)).astype(np.uint8) for _ in range(n)]
    darks = [rng.integers(0, 50, (h, w, c)).astype(np.uint8) for _ in range(n)]
    d_rep, s_rep = [], []
    for k in range(n):
        dr, sr = _repair(dn[k], sg[k], np.ones(dn[k].shape, dtype=bool), 3)
        d_rep.append(dr)
        s_rep.append(sr)
    hd = _hd(dn, sg, t, lut, dlut, d_rep, s_rep)
    kw = dict(darks=[dev(f) for f in darks], dark_threshold=-1.0, median_kernel=3)
    _run_case(kw, hd, algo, single_pass=algo == 4)
    ws, list_off, hot_cap = _workspace(h * w * c)
    ops.hdr_merge(hd["dn"], hd["std"], hd["t"], hd["icrf"], hd["dlut"], algo=algo, workspace=ws, **kw)
    assert _work_list(ws, list_off)[0] > hot_cap


# ---------------------------------------------------------------------------------------------------------------------
# flat-field ROI means

def _exact_mean(a):
    """correctly rounded mean of the doubles in `a` (exact rational sum)"""
    if a.size == 0:
        return math.nan
    vals, counts = np.unique(a, return_counts=True)
    total = sum((Fraction(float(v)) * int(k) for v, k in zip(vals, counts)), Fraction(0))
    return float(total / a.size)


@pytest.mark.parametrize("fbytes", [1, 2, 8])
@pytest.mark.parametrize("c", [1, 3, 2, 5, 8])
def test_roi_means_against_exact_means(c, fbytes):
    """cl_flat_roi_means (roi_partial_kernel<1>, <3> and <0>, run-time C) on uint8 / uint16 / float64 flats against the
    exact means of the flat values (d / MAX as NumPy rounds it) and of the flat uncertainties: within (L + 2) u with
    L = ceil(pixels / (444 x 256)) + 32 additions on the longest chain (thread, warp tree, block, partials); a ROI
    clamped to the image and an empty ROI (NaN, like np.mean of an empty slice)."""
    rng = np.random.default_rng(100 * c + fbytes)
    h, w = (700, 900) if c == 3 else (37, 53)
    max_dn = 65535 if fbytes == 2 else 255
    if fbytes == 8:
        fv = rng.uniform(0.3, 1.0, (h, w, c))
        flat = dev(fv)
    else:
        fd = rng.integers(0, max_dn + 1, (h, w, c)).astype(np.uint8 if fbytes == 1 else np.uint16)
        flat = _dev_dn(fd)
        fv = fd / float(max_dn)
    fs = rng.uniform(0.001, 0.01, (h, w, c))
    for roi in ((h // 4, 3 * h // 4, w // 5, 4 * w // 5), (0, h, 0, w), (h - 3, h + 50, w // 2, w + 9), (5, 5, 0, w),
                (3, 9, 7, 7), (h - 1, h, w - 1, w)):
        r0, r1, c0, c1 = roi
        m = host(ops.flat_roi_means(flat, dev(fs), roi, max_dn=float(max_dn)))
        sub_v, sub_s = fv[r0:r1, c0:c1], fs[r0:r1, c0:c1]
        exp = np.array([_exact_mean(sub_v[..., k]) for k in range(c)] + [_exact_mean(sub_s[..., k]) for k in range(c)])
        if sub_v.size == 0:
            assert np.isnan(m).all(), (roi, m)
            continue
        L = math.ceil(sub_v[..., 0].size / (444 * 256)) + 32
        err = np.abs(m - exp) / np.abs(exp)
        assert (err <= (L + 2) * U).all(), (roi, err)
