"""The step kernel's arithmetic helpers (csrc/hlynr_device.cuh) one by one on the device, against float64 or exact references,
exhaustively where the input space allows.

The step kernel is otherwise tested end to end against the C oracle, whose libm calls the kernel replaces with hand-written
approximations; whole trajectories at the parity tolerances cannot see a subtly wrong approximation, nor the rare inputs
(arguments at +-1 and +-0, the last uniforms before 1, octant boundaries, the flush-to-zero limits) where one breaks.  Here
tests/device_probe.cu, built into a temporary directory, runs each helper element by element:

  * exact claims are checked bit for bit: cdiv (correctly rounded for the constants the kernel divides by), dot3 / dot2 (float
    products, double accumulator, one final rounding), any_nonfinite / nan_guard;
  * the fp64 build's reciprocal, quotient and square root (drcp / dvd / nrcp / sqr) within 2 ulp of the correctly rounded
    result over the normal range, and their behaviour outside it pinned;
  * the float approximations (fast_atan2, fast_asin, euler_over_pi, fast_pair, box_muller, quat_step, isa_props) within the
    worst error measured on a B200, which is what the comments in hlynr_device.cuh state;
  * the launch quaternion of the reset kernel, through the simulator, against float64 acos / sin / cos of the exported positions.
The worst observed value of each bounded helper is printed as a `device_math` line (run pytest with -s to see it)."""
import ctypes as C
import json
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

from hlynr_intercept_b200 import build as _build

F32, F64 = np.float32, np.float64
PROBE_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "device_probe.cu")
DT = 0.01   # every shipped configuration's dt

# Bounds: the worst error measured on a B200 at its 1000 W power limit (printed by the tests; the figure after each colon),
# rounded up.  The same figures are in hlynr_device.cuh.
ATAN2_ABS = 3.6e-7      # fast_atan2, rad: 3.36e-7 (all octants, 2^-126 <= max(|x|, |y|) < 2^126)
ASIN_ABS = 2.6e-7       # fast_asin, rad: 2.38e-7
EULER_ABS = 1.5e-7      # euler_over_pi against float64 atan2 / asin of its own float32 arguments, over pi: 1.23e-7
PAIR_SMALL_R = 0.1      # fast_pair: below this radius (u within 0.005 of 1) the absolute error of __log2f dominates ...
PAIR_ABS = 2.5e-6       # ... above it |z - z64| <= PAIR_ABS: 2.07e-6
PAIR_ERR_R = 1e-7       # ... below it |z - z64| r64 <= PAIR_ERR_R: 7.5e-8 (|z - z64| = 2.2e-4 at the smallest radius, 3.5e-4)
BM_REL = 2e-7           # box_muller, |z - z64| / r64: 1.76e-7
QUAT_ABS_F = 2e-7       # quat_step, fp32 build, per component: 1.72e-7
QUAT_ABS_D = 1.2e-7     # quat_step, fp64 build, per component (the result is float32): 9.3e-8
ISA_REL_F = 1.5e-6      # isa_props, fp32 build, relative: 1.27e-6
ISA_ULP_D = 12          # isa_props, fp64 build, ulp: 11
LAUNCH_ABS_F = 3e-7     # launch quaternion, fp32 build (sqrt identities), plus |eps| / al (test_launch_quaternion)

WORST = {}


def _note(key, value):
    WORST[key] = max(WORST.get(key, 0.0), float(value))


def _report(name):
    print("device_math", json.dumps({"test": name, **WORST}))
    WORST.clear()


# ---------------------------------------------------------------------------------------------------------------------------
# the probe library
# ---------------------------------------------------------------------------------------------------------------------------
_SIGS = {   # name -> argument types (p pointer, f float, d double) before the (int64 n, stream) every launcher ends with
    "cdiv_f": "pffp", "cdiv_d": "pddp", "drcp": "pp", "nrcp_d": "pp", "dvd_d": "ppp", "sqr_d": "pp",
    "dot3_f": "ppp", "dot3_d": "ppp", "dot2_f": "ppp", "fast_atan2": "ppp", "fast_asin": "pp", "euler_over_pi": "pp",
    "fast_pair": "pppp", "box_muller": "pppp", "quat_step_f": "ppf", "quat_step_d": "ppd",
    "isa_props_f": "pppp", "isa_props_d": "pppp", "any_nonfinite_f": "pp", "any_nonfinite_d": "pp",
    "nan_guard_f": "pfp", "nan_guard_d": "pdp",
}
_CT = {"p": C.c_void_p, "f": C.c_float, "d": C.c_double}


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    """tests/device_probe.cu compiled with the library's flags into a temporary directory and loaded with ctypes."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    so = str(tmp_path_factory.mktemp("device_probe") / "device_probe.so")
    res = subprocess.run([nvcc] + _build.NVCC_FLAGS + ["-o", so, PROBE_SRC], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert res.returncode == 0, "nvcc failed:\n" + res.stdout
    lib = C.CDLL(so)
    for name, sig in _SIGS.items():
        fn = getattr(lib, "probe_" + name)
        fn.argtypes = [_CT[c] for c in sig] + [C.c_int64, C.c_void_p]
        fn.restype = C.c_int
    return lib


def test_probe_compiles_for_sm_100a(probe):
    """The probe builds against the current header for sm_100a and exports every launcher (no GPU needed)."""
    for name in _SIGS:
        assert getattr(probe, "probe_" + name)


def _run(probe, name, n, *args):
    """Launch probe_<name> on the current stream with torch tensors (as device pointers) and scalars, then synchronise."""
    import torch

    conv = [C.c_void_p(a.data_ptr()) if isinstance(a, torch.Tensor) else a for a in args]
    err = getattr(probe, "probe_" + name)(*conv, int(n), C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert err == 0, (name, err)
    torch.cuda.synchronize()


def _dev(a):
    import torch

    a = np.ascontiguousarray(a)
    if a.dtype == np.uint32:
        return torch.from_numpy(a.view(np.int32)).cuda()
    return torch.from_numpy(a).cuda()


def _out(n, dtype):
    import torch

    return torch.empty(n, dtype={F32: torch.float32, F64: torch.float64, np.uint8: torch.uint8}[dtype], device="cuda")


def _host(t):
    return t.cpu().numpy()


def _same_bits(got, want):
    """Bitwise equality, with every NaN equal to every NaN (payloads are not part of any helper's contract)."""
    got, want = np.asarray(got), np.asarray(want)
    it = np.int32 if got.dtype == F32 else np.int64
    return (got.view(it) == want.view(it)) | (np.isnan(got) & np.isnan(want))


def _ulps(got, want):
    """Distance in units in the last place through the integer view (both finite, same type)."""
    it = np.int32 if got.dtype == F32 else np.int64
    g, w = got.view(it).astype(np.int64), want.view(it).astype(np.int64)
    # map the sign-magnitude encoding onto a monotone integer line
    top = np.int64(1) << (31 if it == np.int32 else 63)
    g = np.where(g < 0, -(g + top), g)
    w = np.where(w < 0, -(w + top), w)
    return np.abs(g - w)


def _binade(e, dtype=F32, step=1):
    """Every (step-th) float32 / float64 of the binade [2^e, 2^(e+1))."""
    if dtype == F32:
        m = np.arange(0, 1 << 23, step, dtype=np.uint32)
        return ((np.uint32(e + 127) << np.uint32(23)) | m).view(F32)
    m = np.arange(0, 1 << 52, step, dtype=np.uint64)
    return ((np.uint64(e + 1023) << np.uint64(52)) | m).view(F64)


def _log_uniform(rng, n, lo, hi):
    """n doubles 2^U(lo, hi) with uniform random mantissas and random signs."""
    x = np.ldexp(1.0 + rng.random(n), rng.integers(lo, hi, n))
    return np.where(rng.random(n) < 0.5, -x, x)


def _rn32_sum(a, b):
    """float32(a + b), correctly rounded, for float64 arrays a, b whose exact sum may not be a double (TwoSum + a tie fix-up):
    the exact emulation of fmaf(x, y, c) is _rn32_sum(f64(x) * f64(y), f64(c)) (a float32 product is exact in float64)."""
    s = a + b
    bb = s - a
    err = (a - (s - bb)) + (b - bb)
    r = s.astype(F32)
    lo = np.where(r.astype(F64) > s, np.nextafter(r, F32(-np.inf)), r)
    hi = np.nextafter(lo, F32(np.inf))
    tie = (s == (lo.astype(F64) + hi.astype(F64)) / 2) & (err != 0)
    return np.where(tie & (err > 0), hi, np.where(tie & (err < 0), lo, r))


def _fmaf(x, y, c):
    return _rn32_sum(x.astype(F64) * y.astype(F64), np.asarray(c, F32).astype(F64))


gpu = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------------------------
# cdiv: x / c by Markstein's correction with rc = RN(1 / c)
# ---------------------------------------------------------------------------------------------------------------------------
# The constants the kernel divides by (hlynr_device.cuh tick_interceptor / tick_outcome): 500 with rc = R(1.0 / 500.0), 100 with
# rc = R(0.01), dt with rc = KParams::rc_dt = (R)(1.0 / (double)(R)dt) (hlynr_capi.cu make_kparams).
def _cdiv_constants(dtype):
    dt = dtype(DT)
    return [(dtype(500.0), dtype(1.0 / 500.0)), (dtype(100.0), dtype(0.01)), (dt, dtype(1.0 / F64(dt)))]


@gpu
@pytest.mark.parametrize("k", range(3), ids=["c500", "c100", "dt"])
def test_cdiv_float_is_correctly_rounded(probe, k):
    c, rc = _cdiv_constants(F32)[k]
    tiny = np.arange(1, 1 << 16, dtype=np.uint32).view(F32)                        # subnormals
    big = F32(np.finfo(F32).max * 0.5 * min(1.0, float(c))) / np.arange(1, 4097, dtype=F32)   # |x / c| < FLT_MAX
    x = np.concatenate([_binade(0), _binade(13), _binade(-20, step=3), tiny, big, np.array([1, 2, 3, 1e-30, 1e30], F32)])
    x = np.concatenate([x, -x]).astype(F32)
    y = _out(x.size, F32)
    _run(probe, "cdiv_f", x.size, _dev(x), c, rc, y)
    got = _host(y)
    want = (x.astype(F64) / F64(c)).astype(F32)   # correctly rounded: 53 >= 2 * 24 + 2
    normal = np.abs(want) >= np.finfo(F32).tiny
    bad = np.flatnonzero(~_same_bits(got, want) & normal)
    assert bad.size == 0, f"c={c!r}: {bad.size} misrounded, e.g. x={x[bad[:4]]!r} got {got[bad[:4]]!r} want {want[bad[:4]]!r}"
    assert normal.sum() > 3 << 23 and _ulps(got[~normal], want[~normal]).max() <= 1   # subnormal quotients: within 1 ulp
    # +-0: the residual fma(-q, c, x) of a zero is +0, so the quotient of -0 is +0 (a zero either way)
    z = _out(2, F32)
    _run(probe, "cdiv_f", 2, _dev(np.array([0.0, -0.0], F32)), c, rc, z)
    assert (_host(z) == 0).all()


@gpu
@pytest.mark.parametrize("k", range(3), ids=["c500", "c100", "dt"])
def test_cdiv_double_is_correctly_rounded(probe, k):
    from fractions import Fraction

    c, rc = _cdiv_constants(F64)[k]
    rng = np.random.default_rng(11 + k)
    x = [_log_uniform(rng, 4 << 20, -60, 60)]
    # hard cases: exact quotients k c and their neighbours, and dividends whose quotient lies next to a rounding midpoint
    kc = np.arange(1, 20001, dtype=F64) * c
    x += [kc, np.nextafter(kc, 0), np.nextafter(kc, np.inf)]
    mids = []
    for q in np.ldexp(1.0 + rng.random(4000), rng.integers(-30, 30, 4000)):
        x0 = float((Fraction(float(q)) + Fraction(math.ulp(q)) / 2) * Fraction(float(c)))
        mids += [x0, math.nextafter(x0, 0), math.nextafter(x0, math.inf)]
    x = np.concatenate(x + [np.array(mids)])
    x = np.concatenate([x, -x])
    y = _out(x.size, F64)
    _run(probe, "cdiv_d", x.size, _dev(x), float(c), float(rc), y)
    got, want = _host(y), x / c
    bad = np.flatnonzero(~_same_bits(got, want))
    assert bad.size == 0, f"c={c!r}: {bad.size} misrounded, e.g. x={x[bad[:4]]!r} got {got[bad[:4]]!r} want {want[bad[:4]]!r}"


# ---------------------------------------------------------------------------------------------------------------------------
# fp64 build: reciprocal / quotient / square root from the MUFU approximations plus Newton steps
# ---------------------------------------------------------------------------------------------------------------------------
@gpu
def test_fp64_reciprocal_and_quotient_within_2_ulp(probe):
    rng = np.random.default_rng(5)
    n = 4 << 20
    b = _log_uniform(rng, n, -1021, 1022)                 # 1 / b normal
    b = np.concatenate([b, np.ldexp(1.0, np.arange(-1022, 1022)), np.ldexp(np.nextafter(2.0, 0), np.arange(-1022, 1022))])
    a = _log_uniform(rng, b.size, -400, 400)
    with np.errstate(over="ignore", under="ignore"):
        q = np.abs(a / b)
    keep = (q > 2.0 ** -1021) & (q < 2.0 ** 1022)         # a / b normal
    a, bq = a[keep], b[keep]
    worst = {}
    for name, args, want in (("drcp", (b,), 1.0 / b), ("nrcp_d", (b,), 1.0 / b), ("dvd_d", (a, bq), a / bq)):
        y = _out(want.size, F64)
        _run(probe, name, want.size, *[_dev(v) for v in args], y)
        u = _ulps(_host(y), want)
        worst[name] = int(u.max())
        _note(name + "_ulp", u.max())
    _report("fp64_reciprocal")
    assert max(worst.values()) <= 2, worst


# Outside the normal range (the kernel's divisors are positive and finite: clamped speeds, masses, norms tested > 1e-6):
# rcp.approx.ftz.f64 flushes a subnormal input to zero and a subnormal result to zero.
_RCP_EDGES = [(0.0, np.nan), (-0.0, np.nan), (5e-324, np.nan), (2.0 ** -1030, np.nan), (2.0 ** 1022 * 1.5, 0.0),
              (-np.finfo(F64).max, -0.0), (np.inf, np.nan), (-np.inf, np.nan), (np.nan, np.nan)]


@gpu
def test_fp64_reciprocal_edges(probe):
    b = np.array([e[0] for e in _RCP_EDGES])
    want = np.array([e[1] for e in _RCP_EDGES])
    for name in ("drcp", "nrcp_d"):
        y = _out(b.size, F64)
        _run(probe, name, b.size, _dev(b), y)
        got = _host(y)
        assert _same_bits(got, want).all(), (name, list(zip(b, got)))
    y = _out(b.size, F64)
    _run(probe, "dvd_d", b.size, _dev(np.full(b.size, 3.0)), _dev(b), y)
    assert _same_bits(_host(y), 3.0 * want).all(), list(zip(b, _host(y)))


@gpu
def test_fp64_sqrt_within_3_ulp(probe):
    rng = np.random.default_rng(7)
    e = np.arange(-1022, 1024)
    m = rng.integers(0, 1 << 52, (e.size, 1500), dtype=np.uint64)
    a = (((e + 1023).astype(np.uint64)[:, None] << np.uint64(52)) | m).view(F64).ravel()
    p2 = np.ldexp(1.0, e)
    a = np.concatenate([a, p2, np.nextafter(p2, 0), np.nextafter(p2, np.inf), [np.finfo(F64).max]])
    a = a[(a >= 2.3e-308) & np.isfinite(a)]
    y = _out(a.size, F64)
    _run(probe, "sqr_d", a.size, _dev(a), y)
    u = _ulps(_host(y), np.sqrt(a))
    _note("sqr_ulp", u.max())
    _report("fp64_sqrt")
    assert u.max() <= 3, (int(u.max()), a[np.argmax(u)])


@gpu
def test_fp64_sqrt_edges(probe):
    """sqr outside [2.3e-308, DBL_MAX]: +0 for zero, subnormal, small normal, negative and NaN input; NaN for +inf."""
    a = np.array([0.0, -0.0, 5e-324, 2.2e-308, 2.2250738585072014e-308, 2.29e-308, -1.0, -np.inf, np.nan, np.inf])
    want = np.array([0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, np.nan])
    y = _out(a.size, F64)
    _run(probe, "sqr_d", a.size, _dev(a), y)
    assert _same_bits(_host(y), want).all(), list(zip(a, _host(y)))


# ---------------------------------------------------------------------------------------------------------------------------
# dot3 / dot2: np.dot on float32 vectors (float products, double accumulator in order, one final rounding); fp64: exact ops
# ---------------------------------------------------------------------------------------------------------------------------
def _dot_inputs(rng, k, n):
    a = _log_uniform(rng, n * k, -40, 40).reshape(n, k)
    b = _log_uniform(rng, n * k, -40, 40).reshape(n, k)
    # cancelling: a product pair that cancels exactly next to a small third product, in every position
    big, small = np.ldexp(1.0 + rng.random(n), rng.integers(20, 60, n)), np.ldexp(1.0 + rng.random(n), rng.integers(-30, 0, n))
    cols = [big, -big, small] if k == 3 else [big, -big * (1 + 2.0 ** -20)]
    perms = ((0, 1, 2), (0, 2, 1), (1, 0, 2), (1, 2, 0), (2, 0, 1), (2, 1, 0)) if k == 3 else ((0, 1), (1, 0))
    canc = [np.stack([cols[j] for j in perm], axis=1) for perm in perms]
    # overflowing products (inf, inf - inf = NaN) and products below the float range
    huge = np.array([[1e20, 1e20, 1.0], [1e20, -1e20, 3.0], [1e-30, 1e-30, 1.0], [3e38, 2.0, -3e38]])[:, :k]
    ones = np.ones_like(huge)
    a = np.concatenate([a] + canc + [huge, huge])
    b = np.concatenate([b] + [np.ones((n, k))] * len(canc) + [huge, ones])
    return a, b


@gpu
def test_dot3_dot2_float_bit_exact(probe):
    rng = np.random.default_rng(3)
    for k, name in ((3, "dot3_f"), (2, "dot2_f")):
        a, b = _dot_inputs(rng, k, 1 << 20)
        a, b = a.astype(F32), b.astype(F32)
        with np.errstate(over="ignore", invalid="ignore"):
            p = (a * b).astype(F64)      # float32 products (no FMA in numpy), widened exactly
            s = p[:, 0] + p[:, 1]
            if k == 3:
                s = s + p[:, 2]
            want = s.astype(F32)
        y = _out(a.shape[0], F32)
        _run(probe, name, a.shape[0], _dev(a.ravel()), _dev(b.ravel()), y)
        got = _host(y)
        bad = np.flatnonzero(~_same_bits(got, want))
        assert bad.size == 0, (name, bad.size, a[bad[:3]], b[bad[:3]], got[bad[:3]], want[bad[:3]])


@gpu
def test_dot3_double_bit_exact(probe):
    rng = np.random.default_rng(4)
    a, b = _dot_inputs(rng, 3, 1 << 20)
    a = np.concatenate([a, np.ldexp(a[:1000], 900)])    # double products that overflow
    b = np.concatenate([b, np.ldexp(b[:1000], 200)])
    with np.errstate(over="ignore", invalid="ignore"):
        want = (a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1]) + a[:, 2] * b[:, 2]
    y = _out(a.shape[0], F64)
    _run(probe, "dot3_d", a.shape[0], _dev(a.ravel()), _dev(b.ravel()), y)
    assert _same_bits(_host(y), want).all()


# ---------------------------------------------------------------------------------------------------------------------------
# fast_atan2 / fast_asin / euler_over_pi
# ---------------------------------------------------------------------------------------------------------------------------
def _atan2_cases():
    """(y, x) float32: all 8 octants over a dense grid of ratios in [0, 1], the axes, +-0, subnormal minors, and the grid
    scaled through the domain 2^-126 <= max(|x|, |y|) < 2^126."""
    r = np.concatenate([_binade(e, step=97) for e in range(-30, 0)] + [np.array([0.0, 1.0, 1e-30, 1e-40, 1e-45], F32)])
    ys, xs = [], []
    for sx in (1, -1):
        for sy in (1, -1):
            for swap in (False, True):
                a, b = (r * sy, np.full_like(r, sx)) if not swap else (np.full_like(r, sy), r * sx)
                ys.append(a); xs.append(b)
    y, x = np.concatenate(ys), np.concatenate(xs)
    sub = np.random.default_rng(9).choice(y.size, 1 << 18, replace=False)
    sc = np.ldexp(F32(1), np.random.default_rng(10).integers(-126, 126, sub.size)).astype(F32)
    y = np.concatenate([y, y[sub] * sc, np.array([0.0, -0.0], F32), np.full(2, 1.5 * 2.0 ** 125, F32)])
    x = np.concatenate([x, x[sub] * sc, np.zeros(2, F32), np.array([2.0 ** 125, -2.0 ** 125], F32)])
    return y.astype(F32), x.astype(F32)


_ATAN_C = [F32(c) for c in (-0.004780525807291269, 0.024557389318943024, -0.05990511178970337, 0.09942789375782013,
                            -0.14029431343078613, 0.1997137814760208, -0.3333209455013275, 0.9999999403953552)]


def _fast_atan2_f32(y, x):
    """fast_atan2's op sequence in float32 for max(|x|, |y|) a power of two, where rcp.approx is exact."""
    ax, ay = np.abs(x), np.abs(y)
    mx, mn = np.maximum(ax, ay), np.minimum(ax, ay)
    a = np.where(mx > 0, mn * (F32(1) / mx), F32(0)).astype(F32)
    s = a * a
    p = np.full_like(s, _ATAN_C[0])
    for c in _ATAN_C[1:]:
        p = _fmaf(p, s, c)
    r = p * a
    r = np.where(ay > ax, F32(1.57079632679489662) - r, r)
    r = np.where(x < 0, F32(3.14159265358979324) - r, r)
    return np.copysign(r, y).astype(F32)


@gpu
def test_fast_atan2_error_bound(probe):
    y, x = _atan2_cases()
    r = _out(y.size, F32)
    _run(probe, "fast_atan2", y.size, _dev(y), _dev(x), r)
    got = _host(r)
    want = np.arctan2(y.astype(F64), x.astype(F64))
    err = np.abs(got - want)
    _note("atan2_abs", err.max())
    _report("fast_atan2")
    assert err.max() <= ATAN2_ABS, (err.max(), y[np.argmax(err)], x[np.argmax(err)])
    assert (np.signbit(got) == np.signbit(want)).all()
    # where the reciprocal is exact the helper is plain float32 arithmetic: bit for bit (pins every coefficient to the bit)
    mx = np.maximum(np.abs(x), np.abs(y))
    exact = (mx > 0) & (np.frexp(mx)[0] == 0.5)
    bad = np.flatnonzero(~_same_bits(got[exact], _fast_atan2_f32(y[exact], x[exact])))
    assert exact.sum() > 1 << 20 and bad.size == 0, (bad.size, y[exact][bad[:3]], x[exact][bad[:3]])
    # outside the domain: 1 / max(|x|, |y|) flushes to zero from 2^126 on, so atan2(1e38, 2e38) is 0 instead of 0.46; and
    # x = -0 counts as positive, so atan2(+-0, -0) is +-0 instead of +-pi (euler_over_pi's cos terms 1 - 2 v are never -0)
    edge = _out(3, F32)
    _run(probe, "fast_atan2", 3, _dev(np.array([1e38, 0.0, -0.0], F32)), _dev(np.array([2e38, -0.0, -0.0], F32)), edge)
    assert _same_bits(_host(edge), np.array([0.0, 0.0, -0.0], F32)).all(), _host(edge)


@gpu
def test_fast_asin_error_bound(probe):
    near = np.arange(F32(0.99).view(np.int32), F32(1).view(np.int32) + 1, dtype=np.int32).view(F32)   # every float32 in [0.99, 1]
    x = np.concatenate([near, -near, np.linspace(-1, 1, 1 << 21, dtype=F32), np.array([0.0, -0.0, 1e-40, -1e-40, 1e-20], F32)])
    r = _out(x.size, F32)
    _run(probe, "fast_asin", x.size, _dev(x), r)
    got = _host(r)
    err = np.abs(got - np.arcsin(x.astype(F64)))
    _note("asin_abs", err.max())
    _report("fast_asin")
    assert err.max() <= ASIN_ABS, (err.max(), x[np.argmax(err)])
    assert got[x == 1][0] == F32(np.pi / 2) and got[x == -1][0] == -F32(np.pi / 2)


def _euler_args(q):
    """The float32 arguments euler_over_pi forms (exact emulation of its fmaf / products), as float64."""
    w, x, y, z = (q[:, i] for i in range(4))
    two = F32(2)
    sinr = two * _fmaf(w, x, y * z)
    cosr = F32(1) - two * _fmaf(x, x, y * y)
    sinp = two * _fmaf(w, y, -(z * x))
    siny = two * _fmaf(w, z, x * y)
    cosy = F32(1) - two * _fmaf(y, y, z * z)
    return [v.astype(F32).astype(F64) for v in (sinr, cosr, sinp, siny, cosy)]


@gpu
def test_euler_over_pi(probe):
    rng = np.random.default_rng(12)
    q = rng.normal(size=(1 << 20, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    # gimbal lock: pitch +-90 degrees (sinp = +-1), just short of it and just past it through rounding; random roll and yaw
    lock = []
    for pitch in (np.pi / 2, -np.pi / 2):
        for eps in (0.0, 1e-7, -1e-7, 1e-4, -1e-4, 3e-3):
            r2, y2 = rng.uniform(-np.pi, np.pi, (2, 4096)) / 2
            p2 = np.full(4096, (pitch + eps) / 2)
            cr, sr, cp, sp, cy, sy = np.cos(r2), np.sin(r2), np.cos(p2), np.sin(p2), np.cos(y2), np.sin(y2)
            lock.append(np.stack([cr * cp * cy + sr * sp * sy, sr * cp * cy - cr * sp * sy, cr * sp * cy + sr * cp * sy,
                                  cr * cp * sy - sr * sp * cy], axis=1))
    # roll and yaw at +-pi: a rotation by pi about x or z, with +-0 components
    flips = np.array([[0, 1, 0, 0], [0, -1, 0, 0], [0, 0, 0, 1], [0, 0, 0, -1], [-0.0, 1, 0, 0], [0, 1, -0.0, -0.0], [1, 0, 0, 0],
                      [0, 0, 1, 0]], F64)
    q = np.concatenate([q] + lock + [flips]).astype(F32)
    r = _out(3 * q.shape[0], F32)
    _run(probe, "euler_over_pi", q.shape[0], _dev(q.ravel()), r)
    got = _host(r).reshape(-1, 3).astype(F64)
    sinr, cosr, sinp, siny, cosy = _euler_args(q)
    want = np.stack([np.arctan2(sinr, cosr), np.arcsin(np.clip(sinp, -1, 1)), np.arctan2(siny, cosy)], axis=1) / np.pi
    d = np.abs(got - want)
    d[:, [0, 2]] = np.minimum(d[:, [0, 2]], 2 - d[:, [0, 2]])   # -1 and +1 are the same angle
    _note("euler_abs", d.max())
    _report("euler_over_pi")
    assert d.max() <= EULER_ABS, (d.max(), q[np.argmax(d.max(axis=1))])
    assert (np.abs(got) <= 1).all()


# ---------------------------------------------------------------------------------------------------------------------------
# normal draws: fast_pair (per tick) and box_muller (reset path) against float64 Box-Muller (include/hlynr_rng.h)
# ---------------------------------------------------------------------------------------------------------------------------
def _bm64(xa, xb):
    r = np.sqrt(-2.0 * np.log(((xa >> 8).astype(F64) + 1) * 2.0 ** -24))
    t = np.pi * 2.0 * ((xb >> 8).astype(F64) * 2.0 ** -24)
    return r, r * np.cos(t), r * np.sin(t)


def _pair_sweeps():
    """(xa, xb) word pairs: every one of the 2^24 radius words with a few angle words, and every angle word with a few radius
    words (the low 8 bits of a word are not used by the draw; they are set to show that)."""
    every = (np.arange(1 << 24, dtype=np.uint32) << np.uint32(8)) | np.uint32(0xA5)
    angles = np.array([0, 1 << 22, 1 << 23, 3 << 22, (1 << 24) - 1, 12345678], np.uint32) << np.uint32(8)
    radii = np.array([0, 1 << 23, (1 << 24) - 2, (1 << 24) - 1, 777], np.uint32) << np.uint32(8)
    for b in angles:
        yield every, np.full_like(every, b)
    for a in radii:
        yield np.full_like(every, a), every


@gpu
@pytest.mark.parametrize("name", ["fast_pair", "box_muller"])
def test_normal_pairs(probe, name):
    z0, z1 = _out(1 << 24, F32), _out(1 << 24, F32)
    nonfinite = 0
    for xa, xb in _pair_sweeps():
        _run(probe, name, xa.size, _dev(xa), _dev(xb), z0, z1)
        g0, g1 = _host(z0).astype(F64), _host(z1).astype(F64)
        nonfinite += int((~np.isfinite(g0) | ~np.isfinite(g1)).sum())
        r, w0, w1 = _bm64(xa, xb)
        err = np.maximum(np.abs(g0 - w0), np.abs(g1 - w1))
        small = r < PAIR_SMALL_R
        _note(name + "_abs", np.nanmax(err[~small], initial=0))
        _note(name + "_abs_times_r_small_r", np.nanmax(err[small] * r[small], initial=0))
        with np.errstate(invalid="ignore", divide="ignore"):
            _note(name + "_rel", np.nanmax(np.where(r > 0, err / r, 0)))
    _note(name + "_nonfinite", nonfinite)
    worst = dict(WORST)
    _report(name)
    assert nonfinite == 0
    if name == "fast_pair":
        assert worst["fast_pair_abs"] <= PAIR_ABS and worst["fast_pair_abs_times_r_small_r"] <= PAIR_ERR_R, worst
    else:
        assert worst["box_muller_rel"] <= BM_REL, worst


# ---------------------------------------------------------------------------------------------------------------------------
# quat_step against the float64 axis-angle product (environment.py:937-956)
# ---------------------------------------------------------------------------------------------------------------------------
def _quat64(q, w, dt):
    q = q.astype(F64)
    wn = np.linalg.norm(w, axis=1)
    h = wn * dt / 2
    with np.errstate(invalid="ignore", divide="ignore"):
        ax = w / wn[:, None]
    ch, sh = np.cos(h), np.sin(h)
    w1, x1, y1, z1 = ch, ax[:, 0] * sh, ax[:, 1] * sh, ax[:, 2] * sh
    w2, x2, y2, z2 = (q[:, i] for i in range(4))
    out = np.stack([w1 * w2 - x1 * x2 - y1 * y2 - z1 * z2, w1 * x2 + x1 * w2 + y1 * z2 - z1 * y2,
                    w1 * y2 - x1 * z2 + y1 * w2 + z1 * x2, w1 * z2 + x1 * y2 - y1 * x2 + z1 * w2], axis=1)
    out /= np.linalg.norm(out, axis=1, keepdims=True)
    return np.where((wn * dt > 1e-6)[:, None], out, q)


@gpu
@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_quat_step(probe, prec):
    R = F32 if prec == "fp32" else F64
    rng = np.random.default_rng(21)
    n = 1 << 20
    q = rng.normal(size=(n, 4))
    q = (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(F32)
    a = rng.uniform(-1, 1, (n, 3))                                   # actions in [-1, 1]: |w| <= 20 sqrt(3)
    u = rng.normal(size=(n, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    k = n // 8
    a[:k] = u[:k] * (1.0 / 20 / DT) * rng.choice([0.98, 0.999, 1.001, 1.02, 1.5], k)[:, None]   # h = |a| 20 dt / 2 around 0.5
    a[k:2 * k] = u[k:2 * k] * (1e-6 / DT / 20) * rng.choice([0.5, 0.9, 1.1, 2.0], k)[:, None]  # |w| dt around the 1e-6 threshold
    w = (a.astype(R) * R(20.0)).astype(R)                            # mul(a3, R(20.0)) in the kernel
    dev_q = _dev(q.ravel())
    _run(probe, "quat_step_" + ("f" if R == F32 else "d"), n, dev_q, _dev(w.ravel()), R(DT))
    got = _host(dev_q).reshape(n, 4).astype(F64)
    want = _quat64(q, w.astype(F64), F64(R(DT)))
    # away from the threshold's own rounding (|w| dt within 1e-3 of 1e-6 relative) the decision must agree
    wdt = np.linalg.norm(w.astype(F64), axis=1) * F64(R(DT))
    clear = np.abs(wdt / 1e-6 - 1) > 1e-3
    d = np.abs(got - want)[clear].max(axis=1)
    norm_err = np.abs(np.linalg.norm(got, axis=1) - 1)
    _note(f"quat_{prec}_abs", d.max())
    _note(f"quat_{prec}_norm", norm_err.max())
    _report(f"quat_step_{prec}")
    assert d.max() <= (QUAT_ABS_F if R == F32 else QUAT_ABS_D), d.max()
    assert norm_err.max() <= 2 * 2.0 ** -23                          # unit norm within 2 float ulp of 1
    assert (got[wdt < 0.999e-6] == q[wdt < 0.999e-6]).all()          # below the threshold: untouched


# ---------------------------------------------------------------------------------------------------------------------------
# isa_props (+ isa_above_11km) against AtmosphericModel (physics_models.py:154-177) in float64
# ---------------------------------------------------------------------------------------------------------------------------
def _isa64(T0, alt):
    g0, Rg, L = 9.80665, 287.05, 0.0065
    T = np.where(alt <= 11000, T0 - L * alt, np.where(alt <= 20000, 216.65, 216.65 * np.exp(-(alt - 20000) / 10000.0)))
    base = 22632.0 * np.exp(-g0 * 9000.0 / (Rg * 216.65))
    with np.errstate(invalid="ignore"):
        P = np.where(alt <= 11000, 101325.0 * (np.maximum(T0 - L * alt, 1e-300) / T0) ** (g0 / (Rg * L)),
                     np.where(alt <= 20000, 22632.0 * np.exp(-g0 * (alt - 11000) / (Rg * 216.65)), base * np.exp(-(alt - 20000) / 6000.0)))
    return P / (Rg * T), np.sqrt(1.4 * Rg * T)


@gpu
@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_isa_props(probe, prec):
    R = F32 if prec == "fp32" else F64
    rng = np.random.default_rng(31)
    edges = []
    for b in (R(11000), R(20000), R(0)):
        v = b
        for _ in range(3):
            v = np.nextafter(v, R(-np.inf))
            edges.append(v)
        v = b
        for _ in range(3):
            v = np.nextafter(v, R(np.inf))
            edges.append(v)
        edges.append(b)
    alt = np.concatenate([np.linspace(-500, 30000, 1 << 20), rng.uniform(-500, 30000, 1 << 20), np.array(edges, F64)]).astype(R)
    # T0: the standard 288.15 K, and the domain-randomised walk around it (hlynr_device.cuh spawn: T0 += dr_var[1] z per reset)
    T0 = np.where(rng.random(alt.size) < 0.25, 288.15, 288.15 + rng.normal(0, 15, alt.size)).astype(R)
    rho, cs = _out(alt.size, R), _out(alt.size, R)
    _run(probe, "isa_props_" + ("f" if R == F32 else "d"), alt.size, _dev(T0), _dev(alt), rho, cs)
    got_rho, got_cs = _host(rho), _host(cs)
    want_rho, want_cs = _isa64(T0.astype(F64), alt.astype(F64))
    if R == F32:
        rel = np.maximum(np.abs(got_rho / want_rho - 1), np.abs(got_cs / want_cs - 1))
        _note("isa_fp32_rel", rel.max())
        bound_ok = rel.max() <= ISA_REL_F
    else:
        u = np.maximum(_ulps(got_rho, want_rho), _ulps(got_cs, want_cs))
        _note("isa_fp64_ulp", u.max())
        bound_ok = u.max() <= ISA_ULP_D
    # across both layer boundaries at T0 = 288.15 K the device jumps as the reference does: at 11 km the reference's
    # 22632 Pa is 1.3e-5 above 101325 (216.65 / 288.15)^5.2559; at 20 km it is continuous
    for b in (R(11000), R(20000)):
        a2 = np.array([b, np.nextafter(b, R(np.inf))], R)
        T02 = np.full(2, 288.15, R)
        r2, c2 = _out(2, R), _out(2, R)
        _run(probe, "isa_props_" + ("f" if R == F32 else "d"), 2, _dev(T02), _dev(a2), r2, c2)
        ref_rho = _isa64(T02.astype(F64), a2.astype(F64))[0]
        jump, ref_jump = _host(r2)[1] / _host(r2)[0] - 1, ref_rho[1] / ref_rho[0] - 1
        _note(f"isa_{prec}_jump_{int(b)}_vs_reference", abs(jump - ref_jump))
        assert abs(jump - ref_jump) <= (2 * ISA_REL_F if R == F32 else 1e-13), (b, jump, ref_jump)
    worst = dict(WORST)
    _report(f"isa_props_{prec}")
    assert bound_ok, worst


# ---------------------------------------------------------------------------------------------------------------------------
# any_nonfinite / nan_guard: exact
# ---------------------------------------------------------------------------------------------------------------------------
def _special_values(R):
    it, ut = (np.int32, np.uint32) if R == F32 else (np.int64, np.uint64)
    nexp, mbits = (256, 23) if R == F32 else (2048, 52)
    rng = np.random.default_rng(41)
    m = rng.integers(0, 1 << mbits, nexp * 4, dtype=np.uint64).astype(ut)
    e = np.repeat(np.arange(nexp, dtype=np.uint64), 4).astype(ut)
    v = ((e << ut(mbits)) | m).view(R)                              # every exponent, incl. subnormals, inf and NaN payloads
    top = ut(nexp - 1) << ut(mbits)
    payloads = np.array([1, 2, 1 << (mbits - 1), (1 << mbits) - 1, 12345], np.uint64).astype(ut) | top
    extra = np.concatenate([np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1.0, np.finfo(R).max, np.finfo(R).tiny], R),
                            np.array([1, 2, (1 << mbits) - 1], np.uint64).astype(ut).view(R),   # subnormals
                            payloads.view(R)])
    v = np.concatenate([v, extra, -extra])
    return v.astype(R)


@gpu
@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_any_nonfinite_and_nan_guard_exact(probe, prec):
    R = F32 if prec == "fp32" else F64
    sfx = "f" if R == F32 else "d"
    v = _special_values(R)
    rng = np.random.default_rng(43)
    # triples: the value in each of the three positions next to finite companions, and three random values
    fin = v[np.isfinite(v)]
    trip = []
    for pos in range(3):
        t = rng.choice(fin, (v.size, 3))
        t[:, pos] = v
        trip.append(t)
    trip.append(rng.choice(v, (v.size * 4, 3)))
    trip = np.concatenate(trip).astype(R)
    y = _out(trip.shape[0], np.uint8)
    _run(probe, "any_nonfinite_" + sfx, trip.shape[0], _dev(trip.ravel()), y)
    assert (_host(y).astype(bool) == ~np.isfinite(trip).all(axis=1)).all()
    lim = R(20.0)
    g = _out(v.size, R)
    _run(probe, "nan_guard_" + sfx, v.size, _dev(v), lim, g)
    want = np.nan_to_num(v, nan=0.0, posinf=lim, neginf=-lim)
    it = np.int32 if R == F32 else np.int64
    assert (_host(g).view(it) == want.view(it)).all()


# ---------------------------------------------------------------------------------------------------------------------------
# the launch quaternion of a reset (environment.py:492-530), through the simulator
# ---------------------------------------------------------------------------------------------------------------------------
def _spawn_cfg(where):
    from hlynr_intercept_b200 import config

    e = config.baseline_config("cfg4")
    # missile_spawn velocities only set the speed range; the interceptor box sets where the line of sight starts
    ip = [[-200, -200, 500], [200, 200, 800]]
    if where == "generic":
        mp = [[-3000, -3000, 0], [3000, 3000, 3000]]
    elif where == "near_up":     # within 1e-3 rad of +Z: |horizontal offset| <= 0.7 m over >= 1000 m
        ip, mp = [[10, 20, 0], [10.5, 20.5, 1]], [[10, 20, 1500], [10.5, 20.5, 2500]]
    elif where == "near_down":
        ip, mp = [[10, 20, 2000], [10.5, 20.5, 2001]], [[10, 20, 100], [10.5, 20.5, 900]]
    elif where == "up":          # exactly vertical, aligned with +Z
        ip, mp = [[10, 20, 0], [10, 20, 5]], [[10, 20, 1500], [10, 20, 2500]]
    else:                        # exactly vertical, anti-aligned
        ip, mp = [[10, 20, 2000], [10, 20, 2001]], [[10, 20, 100], [10, 20, 900]]
    e["interceptor_spawn"] = dict(position=ip, velocity=[[20, 20, 40], [40, 40, 80]])
    e["missile_spawn"] = dict(position=mp, velocity=[[-110, -110, -55], [-160, -160, -75]])
    return e


def _launch_quat64(ipos, mpos):
    """float64 acos / sin / cos of the float32 line of sight, as spawn_values forms it: rv = f32(m - i), rd = |rv| (float32
    products, double sum, float32 sqrt), f = f32(rv / rd), then float64."""
    rv = (mpos.astype(F32) - ipos.astype(F32)).astype(F32)
    p = (rv * rv).astype(F64)
    rd = np.sqrt(((p[:, 0] + p[:, 1]) + p[:, 2]).astype(F32).astype(F64)).astype(F32)
    f = (rv.astype(F64) / rd.astype(F64)[:, None]).astype(F32).astype(F64)
    ax, ay = -f[:, 1], f[:, 0]
    al = np.sqrt(ax * ax + ay * ay + 0.0)
    h = np.arccos(np.clip(f[:, 2], -1, 1)) / 2
    with np.errstate(invalid="ignore", divide="ignore"):
        q = np.stack([np.cos(h), ax / al * np.sin(h), ay / al * np.sin(h), np.zeros_like(h)], axis=1)
    ident, flip = np.array([1.0, 0, 0, 0]), np.array([0.0, 1, 0, 0])
    q = np.where((al > 1e-6)[:, None], q, np.where((f[:, 2] > 0)[:, None], ident, flip))
    return np.where((rd > 1e-6)[:, None], q, ident), al, (f * f).sum(axis=1) - 1


@gpu
@pytest.mark.parametrize("prec", ["fp32", "fp64"])
@pytest.mark.parametrize("where", ["generic", "near_up", "near_down", "up", "down"])
def test_launch_quaternion(where, prec):
    import torch

    from hlynr_intercept_b200.sim import HlynrSim

    sim = HlynrSim(_spawn_cfg(where), n_envs=4099, seed=77, precision=prec, warn_dead=False)
    try:
        obs = sim.reset().cpu().numpy()
        torch.cuda.synchronize()
        st = sim.export_state()
    finally:
        sim.close()
    got = st["quat"].astype(F64)
    want, al, eps = _launch_quat64(st["ipos"], st["mpos"])
    if where in ("up", "down"):
        assert (al == 0).all()
        assert (got == want).all(), got[:3]      # the reference's quirk: aligned -> identity, anti-aligned -> (0, 1, 0, 0)
    elif where != "generic":
        assert (al > 1e-6).mean() > 0.9 and (al < 1.1e-3).all()
    d = np.abs(got - want)
    if prec == "fp32":   # the sqrt identities differ from acos / sin / cos by up to about eps / (2 al), |f|^2 = 1 + eps
        bound = LAUNCH_ABS_F + (np.abs(eps) / np.maximum(al, 1e-300))[:, None]
    else:   # the float32 rounding of a float64 value within 1e-12 of the reference
        bound = np.spacing(np.abs(want).astype(F32)).astype(F64) / 2 + 1e-12
    _note(f"launch_{prec}_abs", d.max())
    _note(f"launch_{prec}_share_of_bound", (d / bound).max())
    assert (d <= bound).all(), (where, d.max())
    # the reset observation's Euler channels against float64 atan2 / asin of the same quaternion
    sinr, cosr, sinp, siny, cosy = _euler_args(st["quat"].astype(F32))
    eul = np.stack([np.arctan2(sinr, cosr), np.arcsin(np.clip(sinp, -1, 1)), np.arctan2(siny, cosy)], axis=1) / np.pi
    de = np.abs(obs[:, 9:12].astype(F64) - eul)
    de[:, [0, 2]] = np.minimum(de[:, [0, 2]], 2 - de[:, [0, 2]])
    _note(f"launch_{prec}_euler_abs", de.max())
    _report(f"launch_quaternion_{where}_{prec}")
    assert de.max() <= EULER_ABS, de.max()
