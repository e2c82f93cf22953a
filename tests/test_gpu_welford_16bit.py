"""K3 Welford for 16-bit cameras: every path of csrc/welford_u16.cu against exact or high-precision references.

* integer stack path (uint16 frames, no ICRF): Σd and Σd² are exact integers, so the float64 mean must be the
  correctly rounded RN(Σd / (F·MAX_DN)) bit for bit, the uint16 mean of every non-tie sample is rint(Σd / F) decided
  in integers, and the SEM is compared with sqrt(num) / (MAX_DN·F·sqrt(F−1)) from the exact num = F·Σd² − (Σd)²,
  which needs all 64 bits (int64 overflows at F = 65536 with full-scale data);
* ICRF stack path: every table value is an exact dyadic rational, so Σx and Σx² are exact Python fractions;
* ties, replays and the streaming form: the reference's sequential recurrence (the oracle), whose own rounding noise
  is what the kernels must reproduce.
"""
import decimal
from fractions import Fraction

import numpy as np
import pytest
import torch

from oracle import welford as ow
from gpu_util import dev, host

pytestmark = pytest.mark.gpu
ops = pytest.importorskip("camera_linearity_b200.ops")
from camera_linearity_b200 import _lib  # noqa: E402

U = 2.0 ** -53
MAX_FRAMES = 65536              # welford_u16.cu kU16MaxFrames
SEM_ULPS = 8                    # exact num rounded once to double, then <= 6 roundings (reciprocals of the uniform
                                # divisors, products, the square root and its reciprocal); halved under the root


def _reference(frames, icrf=None, max_dn=65535):
    """The reference recurrence (oracle.welford) with the R9 extension for uint16 frames (DESIGN.md section 3): the
    quantised mean and std frames are np.around(...).astype(np.uint16) of the oracle's float64 mean / SEM, where
    the reference's literal uint8 cast would wrap every 16-bit mean modulo 256."""
    o = ow.welford(frames, icrf=icrf, max_dn=max_dn)
    with np.errstate(invalid="ignore"):
        o["mean_q"] = np.around(o["mean"] * max_dn).astype(np.uint16)
        o["std_q"] = None if o["sem"] is None else np.around(o["sem"]).astype(np.uint16)
    return o


def _sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _moments(fr):
    """exact Σd (int64) and Σd² (uint64) per sample of a (F, n) uint16 host array"""
    F, n = fr.shape
    s = np.zeros(n, dtype=np.int64)
    s2 = np.zeros(n, dtype=np.uint64)
    for f0 in range(0, F, 4096):
        x = fr[f0:f0 + 4096].astype(np.int64)
        s += x.sum(0)
        s2 += (x * x).sum(0).astype(np.uint64)
    return s, s2


def _num(s, s2, F):
    """num = F·Σd² − (Σd)² as uint64: exact, because the true value lies in [0, 2^64) (checked in Python integers
    on the largest sample) and uint64 arithmetic is exact modulo 2^64"""
    su = s.astype(np.uint64)
    num = np.uint64(F) * s2 - su * su
    k = int(np.argmax(s2))
    assert 0 <= F * int(s2[k]) - int(s[k]) ** 2 == int(num[k]) < 2 ** 64
    return num


def _sem_reference(num, F, max_dn):
    """sqrt(num) / (MAX_DN·F·sqrt(F−1)) in 64-bit-mantissa long double (num < 2^64 is exact there), else in 40-digit
    decimal on the distinct values"""
    if np.finfo(np.longdouble).nmant >= 63:
        ld = np.longdouble
        x = (num >> np.uint64(32)).astype(ld) * ld(2.0 ** 32) + (num & np.uint64(0xFFFFFFFF)).astype(ld)
        return np.sqrt(x) / (ld(max_dn) * ld(F) * np.sqrt(ld(F - 1)))
    uniq, inv = np.unique(num, return_inverse=True)
    with decimal.localcontext() as ctx:
        ctx.prec = 40
        scale = decimal.Decimal(max_dn) * decimal.Decimal(F) * decimal.Decimal(F - 1).sqrt()
        vals = [decimal.Decimal(int(v)).sqrt() / scale for v in uniq]
    return np.array([float(v) for v in vals])[inv]


def _video(rng, F, n, top):
    """(F, n) uint16: uniform noise, all `top`, frames alternating 0 / `top` (the largest num), constant samples
    (SEM exactly 0), low noise around a base (exact ties for even F), uniform noise again."""
    fr = rng.integers(0, top + 1, (F, n)).astype(np.uint16)
    q = n // 8
    fr[:, q:2 * q] = top
    fr[:, 2 * q:3 * q] = ((np.arange(F) % 2) * top)[:, None]
    fr[:, 3 * q:4 * q] = rng.integers(0, top + 1, (1, q))
    base = rng.integers(1, top, (1, 2 * q))
    fr[:, 4 * q:6 * q] = base + rng.integers(-1, 2, (F, 2 * q))
    return fr


def _check_integer_stack(fr, C, max_dn):
    """ops.welford_stack on (F, n) frames viewed as (F, n/C, C); every output against its exact reference.
    Returns the number of exact ties."""
    F, n = fr.shape
    mean, sem, mean_q = ops.welford_stack(dev(fr).view(F, n // C, C), None, max_dn)
    assert mean_q.dtype == torch.uint16
    mean, sem, mean_q = host(mean).ravel(), host(sem).ravel(), host(mean_q).ravel()
    s, s2 = _moments(fr)
    expect = s.astype(np.float64) / float(F * max_dn)          # correctly rounded: both operands are exact doubles
    np.testing.assert_array_equal(mean.view(np.int64), expect.view(np.int64))
    tie = 2 * (s % F) == F
    np.testing.assert_array_equal(mean_q[~tie], ((s[~tie] + F // 2) // F).astype(np.uint16))
    if tie.any():
        idx = np.nonzero(tie)[0]
        np.testing.assert_array_equal(mean_q[idx], _reference(list(fr[:, idx]), max_dn=max_dn)["mean_q"])
    if F == 1:
        assert np.isnan(sem).all()
        return int(tie.sum())
    num = _num(s, s2, F)
    zero = num == 0
    assert (sem[zero] == 0).all(), "constant samples must have a SEM of exactly 0"
    ref = _sem_reference(num[~zero], F, max_dn)
    err = np.abs(sem[~zero].astype(ref.dtype) - ref) / ref
    assert err.max() <= SEM_ULPS * U, (F, float(err.max()))
    return int(tie.sum())


# ---------------------------------------------------------------------------------------------------------------------
# a. integer stack path
@pytest.mark.parametrize("max_dn", [65535, 4095])
@pytest.mark.parametrize("C", [1, 2, 3, 4, 8])
def test_integer_stack_exact(max_dn, C):
    rng = np.random.default_rng(C * 7 + max_dn)
    ties = 0
    for F in (1, 2, 3, 7, 8, 9, 16, 17, 64, 257, 1000):
        ties += _check_integer_stack(_video(rng, F, 768, max_dn), C, max_dn)
    assert ties > 0


@pytest.mark.parametrize("slices", [1, 2, 4, 8, 16, 32])
def test_integer_stack_every_slice_count(slices):
    # the host picks the smallest power of two `slices` with n_vec·slices >= sm_count·1024 (capped at 32 and at F),
    # n_vec = n / 8: this n_vec targets exactly `slices`; F > 8·slices runs the unrolled loop as well
    n = 8 * -(-_sm() * 1024 // slices)
    n -= n % 24                               # a multiple of 8 and of C = 3
    F = 8 * slices + 3 if slices < 32 else 40
    rng = np.random.default_rng(slices)
    _check_integer_stack(_video(rng, F, n, 65535), 3, 65535)


def test_integer_stack_at_the_frame_limit():
    # F = 65536: full-scale alternating frames (the largest num), full-scale constant samples (F·Σd² and (Σd)² reach
    # 2^64 − 2^49 + 2^32: int64 overflows, uint64 only just holds them) and samples whose Σd/F is a tie or one of the
    # nearest non-ties k + ½ ± 1/F, against the oracle
    F = MAX_FRAMES
    rng = np.random.default_rng(5)
    n = 48
    fr = rng.integers(30000, 30010, (F, n)).astype(np.uint16)
    fr[:, :8] = ((np.arange(F) % 2) * 65535)[:, None]
    fr[:, 8:16] = 65535                               # F·Σd² = (Σd)² = 2^64 − 2^49 + 2^32: num = 0
    s = fr.astype(np.int64).sum(0)
    for i, off in zip(range(16, n), [-1, 0, 1] * 20):
        target = (s[i] // F) * F + F // 2 + off       # Σd/F = k + ½ + off/F
        delta = int(target - s[i])
        fr[:abs(delta), i] += np.uint16(1) if delta > 0 else np.uint16(0xFFFF)   # ±1 DN on |delta| frames
    s, s2 = _moments(fr)
    assert ((2 * (s[16:] % F) - F) == np.tile([-2, 0, 2], 11)[:n - 16]).all()
    assert F * int(s2[8]) == int(s[8]) ** 2 == 2 ** 64 - 2 ** 49 + 2 ** 32
    assert int(_num(s, s2, F)[0]) == F * F // 4 * 65535 ** 2
    _check_integer_stack(fr, 1, 65535)
    out = ops.welford_stack(dev(fr).view(F, n, 1), None, 65535.0)[2]
    np.testing.assert_array_equal(host(out).ravel(), _reference(list(fr), max_dn=65535)["mean_q"])


def test_stack_above_the_frame_limit_takes_the_streaming_form(monkeypatch):
    import camera_linearity_b200 as cl
    from camera_linearity_b200.settings import GlobalSettings as gs
    F = MAX_FRAMES + 1
    rng = np.random.default_rng(6)
    fr = rng.integers(0, 65536, (F, 2, 4, 2)).astype(np.uint16)
    with pytest.raises(_lib.CamlinError) as e:
        ops.welford_stack(dev(fr), None, 65535.0)
    assert e.value.status == -2
    monkeypatch.setattr(gs, "MAX_DN", 65535)
    r = cl.welford_stack(fr)
    o = _reference(list(fr), max_dn=65535)
    assert r["mean"].dtype == torch.uint16 and r["std"].dtype == torch.uint16
    np.testing.assert_array_equal(host(r["mean"]), o["mean_q"])
    np.testing.assert_array_equal(host(r["std"]), o["std_q"])
    np.testing.assert_array_equal(host(r["mean_f64"]), o["mean"])
    np.testing.assert_array_equal(host(r["sem"]), o["sem"])


# ---------------------------------------------------------------------------------------------------------------------
# b. ICRF stack path
def _dyadic_table(rng, rows, C, bits=40):
    """(rows, C) float64 of exact dyadic values k / 2^bits, smooth-ish and in (0, 1)"""
    x = np.linspace(0, 1, rows)[:, None] ** (2.0 + 0.1 * np.arange(C))
    jitter = rng.integers(0, 2 ** 10, (rows, C)) / 2.0 ** 30
    return np.round((x * 0.9 + jitter) * 2.0 ** bits) / 2.0 ** bits


def _check_lut_stack(frames, table, max_dn):
    """frames (F, n/C, C) uint16; checks float64 outputs against exact rational sums and the uint16 mean against
    the oracle for every sample"""
    F = frames.shape[0]
    C = table.shape[1]
    mean, sem, mean_q = ops.welford_stack(dev(frames), dev(table), float(max_dn))
    mean, sem, mean_q = host(mean).ravel(), host(sem).ravel(), host(mean_q).ravel()
    o = _reference(list(frames), icrf=table, max_dn=max_dn)
    np.testing.assert_array_equal(mean_q, o["mean_q"].ravel())
    fr = frames.reshape(F, -1)
    n = fr.shape[1]
    ch = np.arange(n) % C
    for i in range(0, n, max(1, n // 97)):            # exact references on a spread of samples
        xs = [Fraction(float(table[d, ch[i]])) for d in fr[:, i]]
        m = sum(xs) / F
        m_abs = max(abs(x) for x in xs)
        assert abs(Fraction(float(mean[i])) - m) <= 2 * U * abs(m) + (F + 2) * U * m_abs
        if F > 1:
            m2 = sum((x - m) ** 2 for x in xs)
            if m2 == 0:
                assert sem[i] == 0
                continue
            y2 = sum((x - xs[0]) ** 2 for x in xs)
            kappa = float(y2 / m2)
            exact = (float(m2) / (F - 1)) ** 0.5 / F ** 0.5
            assert abs(sem[i] - exact) <= max(1e-13, 4 * F * U * kappa) * exact, (i, sem[i], exact)


@pytest.mark.parametrize("rows,max_dn", [(65536, 65535), (4096, 4095)])
@pytest.mark.parametrize("C", [1, 3, 8])
def test_lut_stack_exact(rows, max_dn, C):
    rng = np.random.default_rng(rows + C)
    table = _dyadic_table(rng, rows, C)
    for F, n in ((1, 96), (2, 96), (9, 600), (64, 1200), (33, 4 * C + C)):   # the last is ragged (n % 4 != 0)
        frames = rng.integers(0, rows, (F, n // C, C)).astype(np.uint16)
        _check_lut_stack(frames, table, max_dn)


def test_lut_stack_static_pixels():
    # a nearly static scene on a table with small steps: the first-frame shift keeps the SEM accurate
    rng = np.random.default_rng(11)
    table = _dyadic_table(rng, 65536, 1)
    base = rng.integers(100, 65000, (1, 500, 1))
    frames = (base + rng.integers(-1, 2, (200, 500, 1))).astype(np.uint16)
    frames[:, :20] = base[:, :20]                     # identical frames: SEM exactly 0
    _check_lut_stack(frames, table, 65535)


def _near_tie_case(rng, deltas, max_dn=4096.0, F=4):
    """frames alternate DNs a_i, b_i whose table values average to (m_i + ½ + δ_i) / max_dn exactly"""
    n = len(deltas)
    table = np.zeros((65536, 1))
    a, b = 2 * np.arange(n) + 1, 2 * np.arange(n) + 2
    m = rng.integers(100, 4000, n)
    e = rng.integers(1, 2 ** 20, n) / 2.0 ** 32
    table[a, 0] = (m + 0.5 + deltas + e) / max_dn
    table[b, 0] = (m + 0.5 + deltas - e) / max_dn
    assert np.array_equal((table[a, 0] + table[b, 0]) / 2 * max_dn, m + 0.5 + deltas)   # exact
    frames = np.where((np.arange(F) % 2)[:, None] == 0, a, b).astype(np.uint16)[:, :, None]
    return frames, table


def test_lut_stack_near_ties_inside_and_outside_the_window():
    rng = np.random.default_rng(12)
    F, max_dn = 4, 4096.0
    w = U * 1.0 * max_dn * (4 * F + 16)                # the kernel's window for |x| <= 1
    deltas = np.array([d * s for d in (0.0, 2.0 ** -40, w / 8, w / 2, 2 * w, 8 * w, 2.0 ** -20) for s in (1, -1)])
    deltas = np.round(deltas * 2.0 ** 41) / 2.0 ** 41        # m + ½ + δ ± e stays exact (m < 2^12)
    frames, table = _near_tie_case(rng, np.repeat(deltas, 8), max_dn, F)
    mean, _, mean_q = ops.welford_stack(dev(frames), dev(table), max_dn)
    o = _reference(list(frames), icrf=table, max_dn=max_dn)
    np.testing.assert_array_equal(host(mean_q), o["mean_q"])


def test_lut_stack_dn_without_a_row_raises():
    rng = np.random.default_rng(13)
    table = _dyadic_table(rng, 4096, 3)
    frames = rng.integers(0, 4096, (5, 40, 3)).astype(np.uint16)
    ops.welford_stack(dev(frames), dev(table), 4095.0)         # every DN has its row
    frames[3, 7, 1] = 4096
    with pytest.raises(IndexError):
        ops.welford_stack(dev(frames), dev(table), 4095.0)
    with pytest.raises(IndexError):
        ops.welford_update(dev(frames), torch.zeros((40, 3), dtype=torch.float64, device="cuda"),
                           torch.zeros((40, 3), dtype=torch.float64, device="cuda"), 0, dev(table), 4095.0)
    with pytest.raises(IndexError):
        np.asarray(table)[frames[3, 7, 1], 1]                   # as NumPy raises
    with pytest.raises(ValueError):
        ops.welford_stack(dev(frames), dev(np.zeros((65537, 3))), 4095.0)


# ---------------------------------------------------------------------------------------------------------------------
# c. replays
def _tie_video(rng, F, n, n_ties):
    """(F, n) uint16 whose first n_ties samples have Σd/F exactly k + ½ (F even), in random frame order"""
    fr = rng.integers(1000, 60000, (F, n)).astype(np.uint16)
    for i in range(n_ties):
        base = rng.integers(1000, 60000)
        col = np.full(F, base, dtype=np.int64)
        col[: F // 2] += 1                            # Σd = F·base + F/2
        col += np.repeat(rng.integers(-50, 51, F // 2), 2) * np.tile([1, -1], F // 2)
        fr[:, i] = rng.permutation(col)
    return fr


@pytest.mark.parametrize("n_ties", [5, 3000])
def test_tie_replay(n_ties):
    rng = np.random.default_rng(n_ties)
    F = 10
    fr = _tie_video(rng, F, 4000, n_ties)
    _, _, mean_q = ops.welford_stack(dev(fr).view(F, -1, 4), None, 65535.0)
    o = _reference(list(fr[:, :n_ties]), max_dn=65535)["mean_q"]
    np.testing.assert_array_equal(host(mean_q).ravel()[:n_ties], o)
    if n_ties > 100:
        assert len(set((o % 2).tolist())) == 2      # the reference rounds some ties up and some down


def _stack_capi(frames, table, frame_offset=0, out_offset=0, max_dn=65535.0):
    """cl_welford_stack_u16 called directly: frames `frame_offset` samples into a larger buffer, mean / sem / mean_q
    `out_offset` elements into theirs"""
    lib = _lib.load()
    F, n = frames.shape[0], frames[0].size
    C = frames.shape[-1]
    buf = torch.empty(F * n + frame_offset, dtype=torch.uint16, device="cuda")
    buf[frame_offset:] = dev(frames.reshape(-1))
    mean = torch.zeros(n + out_offset, dtype=torch.float64, device="cuda")
    sem = torch.zeros_like(mean)
    mq = torch.empty(n + out_offset, dtype=torch.uint16, device="cuda")
    lut = dev(table)
    ws_bytes = lib.cl_welford_stack_workspace_bytes(F, n)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    st = lib.cl_welford_stack_u16(buf.data_ptr() + 2 * frame_offset, F, n, C,
                                  lut.data_ptr() if lut is not None else None, 0 if table is None else len(table),
                                  max_dn, mean.data_ptr() + 8 * out_offset, sem.data_ptr() + 8 * out_offset,
                                  mq.data_ptr() + 2 * out_offset, ws.data_ptr(), ws_bytes,
                                  torch.cuda.current_stream().cuda_stream)
    assert st == 0
    return host(mean[out_offset:]), host(sem[out_offset:]), host(mq[out_offset:])


@pytest.mark.parametrize("frame_offset,out_offset,n", [(0, 0, 96 * 3 + 3), (1, 0, 96 * 3), (0, 1, 96 * 3)])
def test_whole_image_replay(frame_offset, out_offset, n):
    rng = np.random.default_rng(n + frame_offset)
    F = 12
    frames = _tie_video(rng, F, n, 20).reshape(F, n // 3, 3)
    mean, sem, mq = _stack_capi(frames, None, frame_offset, out_offset)
    o = _reference(list(frames), max_dn=65535)
    np.testing.assert_array_equal(mq, o["mean_q"].ravel())
    np.testing.assert_array_equal(mean, o["mean"].ravel())            # the reference recurrence, bit for bit
    np.testing.assert_array_equal(sem, o["sem"].ravel())
    if n % 8 == 0:                                                    # the aligned call: same uint16 mean
        _, _, mq_a = ops.welford_stack(dev(frames), None, 65535.0)
        np.testing.assert_array_equal(mq, host(mq_a).ravel())


# ---------------------------------------------------------------------------------------------------------------------
# d. streaming form and finalize
@pytest.mark.parametrize("rows", [None, 65536, 4096])
def test_streaming_update_bit_identical(rows):
    rng = np.random.default_rng(21)
    C = 3
    top = 65535 if rows in (None, 65536) else rows - 1
    table = None if rows is None else _dyadic_table(rng, rows, C)
    frames = rng.integers(0, top + 1, (70, 9, 7, C)).astype(np.uint16)
    k0 = 5
    o0 = _reference(list(frames[:k0]), icrf=table, max_dn=top)
    mean, m2 = dev(o0["mean"].copy()), dev(o0["m2"].copy())
    count = k0
    for size in (1, 32, 32):                         # resumed across chunks from count0 > 0
        count = ops.welford_update(dev(frames[count:count + size]), mean, m2, count, dev(table), float(top))
    o = _reference(list(frames), icrf=table, max_dn=top)
    np.testing.assert_array_equal(host(mean), o["mean"])
    np.testing.assert_array_equal(host(m2), o["m2"])
    sem, mq = ops.welford_finalize(mean, m2, count, float(top), torch.uint16)
    np.testing.assert_array_equal(host(sem), o["sem"])
    np.testing.assert_array_equal(host(mq), o["mean_q"])


def test_finalize_edges():
    m = np.array([np.nan, -1.0, 65536 + 5, 70000.5, 2.0 ** 31 + 7, -70000.0, np.inf, 1e300, 3.5, 4.5, -0.5,
                  65535.49, 65535.5]) / 65535.0
    with np.errstate(invalid="ignore"):
        expect = np.around(m * 65535.0).astype(np.uint16)
    _, mq = ops.welford_finalize(dev(m), None, 10, 65535.0, torch.uint16)
    np.testing.assert_array_equal(host(mq), expect)
    sem, _ = ops.welford_finalize(dev(np.full(3, 0.5)), dev(np.zeros(3)), 1, 65535.0, torch.uint16)
    assert np.isnan(host(sem)).all()
    with pytest.raises(TypeError):
        ops.welford_finalize(dev(m), None, 10, 65535.0, torch.int16)


def test_stack_and_streaming_agree():
    rng = np.random.default_rng(22)
    F = 40
    frames = _tie_video(rng, F, 960, 100).reshape(F, -1, 3)
    for table in (None, _dyadic_table(rng, 65536, 3)):
        lut = dev(table)
        _, _, q_stack = ops.welford_stack(dev(frames), lut, 65535.0)
        mean = torch.zeros((320, 3), dtype=torch.float64, device="cuda")
        m2 = torch.zeros_like(mean)
        ops.welford_update(dev(frames), mean, m2, 0, lut, 65535.0)
        _, q_stream = ops.welford_finalize(mean, m2, F, 65535.0, torch.uint16)
        np.testing.assert_array_equal(host(q_stack), host(q_stream))


# ---------------------------------------------------------------------------------------------------------------------
# e. public calls
def test_welford_algorithm_uint16_frames(monkeypatch):
    # at the parent commit the uint8 staging buffer wrapped every sample modulo 256
    import camera_linearity_b200 as cl
    from camera_linearity_b200.settings import GlobalSettings as gs
    monkeypatch.setattr(gs, "MAX_DN", 65535)
    rng = np.random.default_rng(31)
    frames = rng.integers(200, 65536, (75, 6, 10, 3)).astype(np.uint16)       # 3 chunks of 32 frames
    r = cl.welford_algorithm("mem", None, True, frame_source=lambda p: list(frames) + [None])
    o = _reference(list(frames), max_dn=65535)
    assert r["mean"].dtype == torch.uint16 and r["count"] == 75
    np.testing.assert_array_equal(host(r["mean"]), o["mean_q"])
    np.testing.assert_array_equal(host(r["std"]), o["std_q"])
    np.testing.assert_array_equal(host(r["mean_f64"]), o["mean"])
    np.testing.assert_array_equal(host(r["sem"]), o["sem"])
    s = cl.welford_stack(frames)
    np.testing.assert_array_equal(host(s["mean"]), o["mean_q"])
    np.testing.assert_array_equal(host(s["std"]), o["std_q"])
    mixed = list(frames[:3]) + [frames[3].astype(np.uint8)]
    with pytest.raises(TypeError):
        cl.welford_algorithm("mem", None, True, frame_source=lambda p: mixed + [None])
    with pytest.raises(TypeError):
        cl.compute_noise_profiles(["mem"], frame_source=lambda p: list(frames[:4]) + [None])


def test_custom_ops_uint16():
    K = torch.ops.camera_linearity
    rng = np.random.default_rng(32)
    frames = rng.integers(0, 4096, (17, 5, 8, 3)).astype(np.uint16)
    o = _reference(list(frames), max_dn=4095)
    mean, sem, mq = K.welford_stack(dev(frames), None, 4095.0)
    np.testing.assert_array_equal(host(mq), o["mean_q"])
    m = torch.zeros((5, 8, 3), dtype=torch.float64, device="cuda")
    m2 = torch.zeros_like(m)
    K.welford_update(dev(frames[:9]), m, m2, 0, None, 4095.0)
    K.welford_update(dev(frames[9:]), m, m2, 9, None, 4095.0)
    sem, mq = K.welford_finalize_u16(m, m2, 17, 4095.0)
    assert mq.dtype == torch.uint16
    np.testing.assert_array_equal(host(m), o["mean"])
    np.testing.assert_array_equal(host(sem), o["sem"])
    np.testing.assert_array_equal(host(mq), o["mean_q"])
    with pytest.raises(TypeError):
        ops.welford_stack(dev(frames.astype(np.int32)))


def test_dispatch_map():
    rng = np.random.default_rng(0)
    act = torch.profiler.ProfilerActivity.CUDA

    def launched(fn):
        with torch.profiler.profile(activities=[act]) as prof:
            fn()
            torch.cuda.synchronize()
        return [e.name for e in prof.events()]

    def small(F, C=3, rows=256, top=65535):
        return dev(rng.integers(0, top + 1, (F, rows, C)).astype(np.uint16))

    probe = launched(lambda: ops.welford_stack(small(8)))
    if not any("welford" in name for name in probe):
        pytest.skip("the profiler records no device activity here")
    t16 = dev(_dyadic_table(rng, 65536, 3))
    t12 = dev(_dyadic_table(rng, 4096, 3))
    ties = dev(_tie_video(rng, 10, 1200, 40).reshape(10, -1, 4))
    zeros = lambda: torch.zeros((256, 3), dtype=torch.float64, device="cuda")  # noqa: E731
    cases = [
        ("welford_stack_u16_kernel", lambda: ops.welford_stack(small(9))),
        ("welford_stack_lut_u16_kernel<true>", lambda: ops.welford_stack(small(9), t16)),
        ("welford_stack_lut_u16_kernel<false>", lambda: ops.welford_stack(small(9, top=4095), t12)),
        ("welford_replay_u16_kernel", lambda: ops.welford_stack(ties)),
        ("welford_replay_u16_kernel", lambda: ops.welford_stack(small(9, 3, rows=7))),
        ("welford_update_u16_kernel", lambda: ops.welford_update(small(9), zeros(), zeros(), 0, t16)),
        ("welford_finalize_u16_kernel", lambda: ops.welford_finalize(zeros(), zeros(), 9, 65535.0, torch.uint16)),
    ]
    for kernel, fn in cases:
        names = [nm for nm in launched(fn) if "welford" in nm]
        assert any(kernel in nm for nm in names), (kernel, names)
        assert not any("u8_kernel" in nm or "welford_stack_lut_kernel" in nm for nm in names), names
