"""The fast-math primitives of csrc/fastmath.cuh, one by one on the device, against high-precision references.

tests/fastmath_harness.cu evaluates each primitive element-wise (the header included as it is); it is compiled here for sm_100a with
the library's flags and loaded with ctypes, and torch tensors carry the buffers. References: 200-bit mpmath on ~2e4 chosen points per
function (the edges where such code goes wrong), long double (atan2l / sinl / cosl precision) on 1e6 random points. Errors are in
ulps of the correctly rounded result, or absolute where the header states an absolute bound; every asserted bound is the one the
header states, and each test prints its measured worst case next to it.

The end-to-end EKF tests cannot see these: the FAST kernels sit ~1e-13 from the oracle against a 1e-9 tolerance, so a primitive
could be 1000x worse than its documented accuracy (a wrong table bit, a dropped Newton step) with every one of them green."""
import ctypes
import subprocess
from pathlib import Path

import mpmath
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
CSRC = ROOT / "shermbot-navigation_b200" / "csrc"
HARNESS = Path(__file__).resolve().parent / "fastmath_harness.cu"

# the bounds stated in fastmath.cuh
RCP_ULP = 1.0            # rcp_fast, div_fast: <= 1 ulp for normal operands
RSQRT_ULP = 1.0          # rsqrt_fast: <= 1 ulp
RSQRT1_REL = 1.3e-12     # rsqrt_1: relative error <= 1.3e-12
ATAN2_FAST_ULP = 2.0     # atan2_fast / atan2_tab: <= 2 ulp on the documented domain
ATAN2_UNIT_ABS = 4.9e-16  # atan2_unit: worst absolute error 4.9e-16 (rs within an ulp of the exact value)
WRAP_ULP = 1.0           # wrap_angle: normalize_angle (and the exact reduction) to 1 ulp on |a| <= 2 pi + 1
SINCOS_ULP = 1.7         # sincos_fast: |a| <= 1e3
SINCOS_ULP_1E6 = 2.0     # sincos_fast: |a| ~ 1e6, the end of the exact reduction
SINCOS_SMALL_ULP = 1.0   # sincos_small: |a| <= 0.25

mpmath.mp.prec = 200
M = mpmath.mpf


@pytest.fixture(scope="module")
def fm(tmp_path_factory):
    """Compile the harness with the library's architecture and flags, load it, and return a caller: fm(name, *inputs, nout=1) copies
    the float64 inputs to the device, launches, and returns the outputs as numpy arrays."""
    import torch
    from shermbot_navigation_b200 import build
    out = tmp_path_factory.mktemp("fastmath") / "libfastmath_harness.so"
    cmd = [build.nvcc(), "-O3", "-std=c++17", *build.ARCH, "--expt-relaxed-constexpr", "-shared", "-Xcompiler", "-fPIC",
           f"-I{ROOT / 'include'}", f"-I{CSRC}", "-o", str(out), str(HARNESS)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    lib = ctypes.CDLL(str(out))
    dev = torch.device("cuda", 0)

    def call(name, *inputs, nout=1):
        ins = [torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev) for a in inputs]
        n = ins[0].numel()
        outs = [torch.empty(n, dtype=torch.float64, device=dev) for _ in range(nout)]
        fn = getattr(lib, "fm_" + name)
        fn.restype = ctypes.c_int
        rc = fn(*[ctypes.c_void_p(t.data_ptr()) for t in ins + outs], ctypes.c_long(n))
        assert rc == 0, f"{name}: launch failed with cudaError {rc}"
        torch.cuda.synchronize()
        res = [t.cpu().numpy() for t in outs]
        return res[0] if nout == 1 else res
    return call


def ulps_ld(got, ref_ld):
    """|got - ref| in ulps of the correctly rounded value, the reference in long double."""
    cr = ref_ld.astype(np.float64)
    return np.abs((got.astype(np.longdouble) - ref_ld) / np.spacing(np.abs(cr)).astype(np.longdouble)).astype(np.float64)


def ulps_mp(got, refs):
    """|got - ref| in ulps of the correctly rounded value, refs a list of mpf."""
    return np.array([float(abs(M(float(g)) - r) / M(float(np.spacing(abs(float(r)))))) for g, r in zip(got, refs)])


def abs_mp(got, refs):
    return np.array([float(abs(M(float(g)) - r)) for g, r in zip(got, refs)])


def report(name, worst, bound, unit, where=None):
    at = f" at {where!r}" if where is not None else ""
    print(f"[{name}] worst {worst:.4g} {unit}{at} (bound {bound:g} {unit})")
    assert worst <= bound, f"{name}: {worst} {unit} > {bound}"


def pow2_neighbours(lo_exp, hi_exp, step):
    """Powers of two (both signs) and the values 1..3 ulp on either side of them."""
    p = np.ldexp(1.0, np.arange(lo_exp, hi_exp + 1, step))
    up = [p]
    dn = [p]
    for _ in range(3):
        up.append(np.nextafter(up[-1], np.inf))
        dn.append(np.nextafter(dn[-1], 0.0))
    x = np.concatenate(up + dn[1:])
    return np.concatenate([x, -x])


def log_uniform(rng, lo, hi, n, signed=True):
    v = 10.0 ** rng.uniform(lo, hi, n)
    return v * rng.choice([-1.0, 1.0], n) if signed else v


# ------------------------------------------------------------------------------------------------------------ rcp, div, rsqrt

def test_rcp_fast(fm):
    rng = np.random.default_rng(1)
    x = np.concatenate([log_uniform(rng, -300, 300, 1_000_000), pow2_neighbours(-996, 996, 1)])
    got = fm("rcp_fast", x)
    e = ulps_ld(got, 1 / x.astype(np.longdouble))
    report("rcp_fast vs 1/x (long double), normal x in 1e-300..1e300", e.max(), RCP_ULP, "ulp", x[e.argmax()])
    sel = np.concatenate([pow2_neighbours(-990, 990, 30), log_uniform(rng, -300, 300, 20_000)])[:20_000]
    g2 = fm("rcp_fast", sel)
    e2 = ulps_mp(g2, [1 / M(float(v)) for v in sel])
    report("rcp_fast vs mpmath", e2.max(), RCP_ULP, "ulp", sel[e2.argmax()])


def test_div_fast(fm):
    rng = np.random.default_rng(2)
    n = 1_000_000
    b = np.concatenate([log_uniform(rng, -150, 150, n), pow2_neighbours(-498, 498, 2)])
    a = log_uniform(rng, -150, 150, b.size)
    a[:1000] = b[:1000] * rng.integers(-1000, 1000, 1000)   # exact quotients (integers)
    got = fm("div_fast", a, b)
    e = ulps_ld(got, a.astype(np.longdouble) / b.astype(np.longdouble))
    report("div_fast vs a/b (long double), quotients in 1e-300..1e300", e.max(), RCP_ULP, "ulp", (a[e.argmax()], b[e.argmax()]))
    assert np.array_equal(got[:1000], a[:1000] / b[:1000])
    sa, sb = a[-20_000:], b[-20_000:]
    g2 = fm("div_fast", sa, sb)
    e2 = ulps_mp(g2, [M(float(p)) / M(float(q)) for p, q in zip(sa, sb)])
    report("div_fast vs mpmath", e2.max(), RCP_ULP, "ulp")


def test_rsqrt(fm):
    rng = np.random.default_rng(3)
    x = np.concatenate([log_uniform(rng, -300, 300, 1_000_000, signed=False), np.abs(pow2_neighbours(-996, 996, 1))])
    ref = 1 / np.sqrt(x.astype(np.longdouble))
    g = fm("rsqrt_fast", x)
    e = ulps_ld(g, ref)
    report("rsqrt_fast vs 1/sqrt(x) (long double)", e.max(), RSQRT_ULP, "ulp", x[e.argmax()])
    g1 = fm("rsqrt_1", x)
    rel = np.abs((g1.astype(np.longdouble) - ref) / ref).astype(np.float64)
    report("rsqrt_1 relative", rel.max(), RSQRT1_REL, "rel", x[rel.argmax()])
    sel = np.concatenate([np.abs(pow2_neighbours(-990, 990, 20)), log_uniform(rng, -300, 300, 20_000, signed=False)])[:20_000]
    refs = [1 / mpmath.sqrt(M(float(v))) for v in sel]
    e2 = ulps_mp(fm("rsqrt_fast", sel), refs)
    report("rsqrt_fast vs mpmath", e2.max(), RSQRT_ULP, "ulp", sel[e2.argmax()])
    g1 = fm("rsqrt_1", sel)
    rel2 = max(float(abs(M(float(g)) - r) / r) for g, r in zip(g1, refs))
    report("rsqrt_1 vs mpmath, relative", rel2, RSQRT1_REL, "rel")


# ------------------------------------------------------------------------------------------------------------ atan2

def atan2_edges(rng):
    """(y, x) edge sets: both axes, |x| == |y| in the four quadrants, +-0 in either argument (the other non-zero), ratios exactly at
    (k +- 1/2) / 64 and their neighbours (the fp32 estimate may pick either table point), mn / mx below 2^-30, magnitudes 1e-8 .. 1e4."""
    mags = np.concatenate([10.0 ** np.arange(-8, 5), rng.uniform(1e-8, 1e4, 20), np.ldexp(1.0, np.arange(-26, 14))])
    ys, xs = [], []
    for m in mags:
        for sy, sx in ((1, 1), (1, -1), (-1, 1), (-1, -1)):
            ys += [0.0, sy * m, sy * m, 0.0 * sy, sy * m]
            xs += [sx * m, 0.0, sx * m, sx * m, 0.0 * sx]
    # ratios at the midpoints between table points and around them: mn / mx = (2k + 1) / 128 (exact), +-1..2 ulp of mn
    for k in range(64):
        for scale in (1.0, 2.0 ** -20, 2.0 ** 10, 1e-7 / 128, 3.1):
            mx = 128.0 * scale
            mn0 = (2 * k + 1) * scale
            for mn in (np.nextafter(np.nextafter(mn0, 0), 0), np.nextafter(mn0, 0), mn0, np.nextafter(mn0, np.inf),
                       np.nextafter(np.nextafter(mn0, np.inf), np.inf)):
                for sy, sx in ((1, 1), (1, -1), (-1, 1), (-1, -1)):
                    ys += [sy * mn, sy * mx]
                    xs += [sx * mx, sx * mn]
    # tiny ratios
    r = np.ldexp(rng.uniform(1, 2, 400), rng.integers(-60, -30, 400))
    mx = 10.0 ** rng.uniform(-8, 4, 400)
    sg = rng.choice([-1.0, 1.0], (400, 2))
    ys += list(sg[:, 0] * r * mx) + list(sg[:, 0] * mx)
    xs += list(sg[:, 1] * mx) + list(sg[:, 1] * r * mx)
    # every table point itself and random ratios at magnitudes 1e-8 .. 1e4
    t = np.concatenate([np.arange(65) / 64.0, rng.uniform(0, 1, 4000)])
    mx = 10.0 ** rng.uniform(-8, 4, t.size)
    ang = rng.integers(0, 8, t.size)
    sw, sx, sy = ang & 1, np.where(ang & 2, -1.0, 1.0), np.where(ang & 4, -1.0, 1.0)
    ys += list(np.where(sw, mx, t * mx) * sy)
    xs += list(np.where(sw, t * mx, mx) * sx)
    return np.array(ys), np.array(xs)


def atan2_random(rng, n=1_000_000):
    ang = rng.uniform(-np.pi, np.pi, n)
    rad = 10.0 ** rng.uniform(-8, 4, n)
    return rad * np.sin(ang), rad * np.cos(ang)


def mp_atan2(y, x):
    """mpmath's atan2 with libm's signed zeros (mpmath has no -0: atan2(-0, x < 0) must be -pi)."""
    r = mpmath.atan2(M(float(y)), M(float(x)))
    return -r if y == 0.0 and np.signbit(y) else r


def ignore_zero_sign(v):
    return np.where(v == 0.0, 0.0, v)


def test_atan2_fast_and_tab(fm):
    """atan2_fast against atan2l and mpmath on the edge sets, <= 2 ulp; a zero argument counts as +0 (documented: the sign tests are
    x < 0, y < 0). scan_moment.cuh's atan2_tab (the same code on shared-memory copies of the tables) gives the same bits on every
    input."""
    rng = np.random.default_rng(4)
    ye, xe = atan2_edges(rng)
    yr, xr = atan2_random(rng)
    y, x = np.concatenate([ye, yr]), np.concatenate([xe, xr])
    got = fm("atan2_fast", y, x)
    tab = fm("atan2_tab", y, x)
    assert np.array_equal(got.view(np.int64), tab.view(np.int64)), "atan2_tab differs from atan2_fast"
    yl, xl = ignore_zero_sign(y).astype(np.longdouble), ignore_zero_sign(x).astype(np.longdouble)
    e = ulps_ld(got, np.arctan2(yl, xl))
    i = e.argmax()
    report(f"atan2_fast vs atan2l, {y.size} points", e.max(), ATAN2_FAST_ULP, "ulp", (y[i], x[i]))
    sel = np.arange(min(ye.size, 20_000))
    refs = [mpmath.atan2(M(float(ignore_zero_sign(y[j]))), M(float(ignore_zero_sign(x[j])))) for j in sel]
    e2 = ulps_mp(got[sel], refs)
    report(f"atan2_fast vs mpmath, {sel.size} edge points", e2.max(), ATAN2_FAST_ULP, "ulp", (y[sel][e2.argmax()], x[sel][e2.argmax()]))
    print(f"[atan2_fast] worst absolute error {abs_mp(got[sel], refs).max():.3g}")


def test_atan2_fast_domain(fm):
    """The documented domain max(|x|, |y|) in [2^-100, 2^100]: the bound holds at its ends. Outside it (the fp32 estimate of mn / mx
    overflows, is denormal, or __fdividef returns 0) the result is a finite number; the error there is reported, not asserted."""
    rng = np.random.default_rng(5)
    t = np.concatenate([np.arange(65) / 64.0, rng.uniform(0, 1, 500)])
    ys, xs = [], []
    for mx in (2.0 ** -100, 2.0 ** 100, np.nextafter(2.0 ** 100, 0), 1e-30, 1e30):
        for sy, sx in ((1, 1), (1, -1), (-1, 1), (-1, -1)):
            ys += list(sy * t * mx) + list(sy * np.full(t.size, mx))
            xs += list(sx * np.full(t.size, mx)) + list(sx * t * mx)
    y, x = np.array(ys), np.array(xs)
    keep = (y != 0.0) | (x != 0.0)
    y, x = y[keep], x[keep]
    got = fm("atan2_fast", y, x)
    e = ulps_mp(got, [mpmath.atan2(M(float(a)), M(float(b))) for a, b in zip(y, x)])
    report("atan2_fast at the ends of its domain", e.max(), ATAN2_FAST_ULP, "ulp", (y[e.argmax()], x[e.argmax()]))
    out = {}
    for mx in (1e300, 2.0 ** 127, 3.3e38, 2.0 ** -110, 1e-40, 1e-300, 5e-324 * 1e6):   # the last one is denormal: NaN (rcp_fast flushes it)
        yy = np.concatenate([t * mx, np.full(t.size, mx)])
        xx = np.concatenate([np.full(t.size, mx), t * mx])
        keep = (yy != 0.0) | (xx != 0.0)
        yy, xx = yy[keep], xx[keep]
        g = fm("atan2_fast", yy, xx)
        gt = fm("atan2_tab", yy, xx)
        assert np.array_equal(g.view(np.int64), gt.view(np.int64)), mx
        assert np.isfinite(g).all() or mx < 2.2250738585072014e-308, mx
        out[mx] = np.abs(g - np.arctan2(yy, xx)).max()
    print("[atan2_fast outside its domain, max abs error by max(|x|, |y|)] " + ", ".join(f"{k:.3g}: {v:.2g}" for k, v in out.items()))


def test_atan2_unit(fm):
    """atan2_unit against atan2l and mpmath: absolute error <= 4.9e-16 (the header's bound) with rs the correctly rounded
    1 / sqrt(x^2 + y^2) and with rs one ulp off either way; signed zeros follow libm (sign-bit tests)."""
    rng = np.random.default_rng(6)
    ye, xe = atan2_edges(rng)
    yr, xr = atan2_random(rng)
    y, x = np.concatenate([ye, yr]), np.concatenate([xe, xr])
    yl, xl = y.astype(np.longdouble), x.astype(np.longdouble)
    rs0 = (1 / np.sqrt(xl * xl + yl * yl)).astype(np.float64)
    ref = np.arctan2(yl, xl)
    worst = (0.0, None)
    for rs in (rs0, np.nextafter(rs0, 0), np.nextafter(rs0, np.inf)):
        got = fm("atan2_unit", y, x, rs)
        err = np.abs(got.astype(np.longdouble) - ref).astype(np.float64)
        if err.max() > worst[0]:
            worst = (err.max(), (y[err.argmax()], x[err.argmax()]))
    report(f"atan2_unit vs atan2l, {y.size} points x 3 rs", worst[0], ATAN2_UNIT_ABS, "abs", worst[1])
    sel = np.arange(min(ye.size, 20_000))
    got = fm("atan2_unit", y[sel], x[sel], rs0[sel])
    refs = [mp_atan2(y[j], x[j]) for j in sel]
    e2 = abs_mp(got, refs)
    report(f"atan2_unit vs mpmath, {sel.size} edge points", e2.max(), ATAN2_UNIT_ABS, "abs", (y[sel][e2.argmax()], x[sel][e2.argmax()]))
    # signed zeros: the result's sign is libm's (atan2(-0, x < 0) = -pi, atan2(+-0, x > 0) = +-0)
    z = np.array([0.0, -0.0, 0.0, -0.0, 1.0, -1.0, 1.0, -1.0])
    w = np.array([-1.0, -1.0, 1.0, 1.0, 0.0, 0.0, -0.0, -0.0])
    got = fm("atan2_unit", z, w, np.ones(8))
    assert np.array_equal(np.signbit(got), np.signbit(np.arctan2(z, w))) and np.abs(got - np.arctan2(z, w)).max() <= ATAN2_UNIT_ABS


# ------------------------------------------------------------------------------------------------------------ wrap_angle

def test_wrap_angle(fm, orc):
    """wrap_angle against rigid2d::normalize_angle (the oracle's) on |a| <= 2 pi + 1, the neighbourhoods (+-8 ulp) of +-pi and +-2 pi
    included: within 1 ulp, and on the same side of the cut as normalize_angle at +-pi; against the exact reduction (mpmath) within
    1 ulp (it is 0.5 ulp from a - k (2 pi hi + 2 pi lo), and that split is 1e-32 from 2 pi). Outside the domain (|a| = 3 pi) the
    result may leave [-pi, pi]: reported only."""
    rng = np.random.default_rng(7)
    P = 2 * np.pi + 1
    cen = np.array([np.pi, -np.pi, 2 * np.pi, -2 * np.pi, 0.0, P, -P])
    near = (cen[:, None] + np.arange(-8, 9)[None, :] * np.spacing(np.abs(cen) + 1e-300)[:, None]).ravel()
    pts = np.concatenate([near, rng.uniform(-P, P, 20_000 - near.size)])
    got = fm("wrap_angle", pts)
    nrm = np.array([orc.normalize_angle(float(v)) for v in pts])
    e = np.abs(got - nrm) / np.spacing(np.abs(nrm))
    report("wrap_angle vs normalize_angle, |a| <= 2 pi + 1", e.max(), WRAP_ULP, "ulp", pts[e.argmax()])
    assert np.array_equal(np.sign(got[np.abs(nrm) > 3]), np.sign(nrm[np.abs(nrm) > 3])), "a tie at +-pi lands on the other side"
    assert (np.abs(got) <= np.pi).all()
    exact = []
    for v in pts:
        m = M(float(v))
        exact.append(m - mpmath.nint(m / (2 * mpmath.pi)) * 2 * mpmath.pi)
    e2 = ulps_mp(got, exact)
    report("wrap_angle vs exact reduction (mpmath)", e2.max(), WRAP_ULP, "ulp", pts[e2.argmax()])
    big = rng.uniform(-P, P, 1_000_000)
    gb = fm("wrap_angle", big)
    bl = big.astype(np.longdouble)
    two_pi = 2 * np.pi
    ref = bl - np.rint(big / two_pi).astype(np.longdouble) * (np.longdouble(two_pi) + np.longdouble(2.4492935982947064e-16))
    # the long double reference itself is good to ~4e-19 absolute
    eb = ((np.abs(gb.astype(np.longdouble) - ref) - np.longdouble(4e-19)) / np.spacing(np.abs(gb)).astype(np.longdouble)).astype(np.float64)
    report("wrap_angle vs long double, 1e6 random", eb.max(), WRAP_ULP, "ulp", big[eb.argmax()])
    far = np.array([3 * np.pi, -3 * np.pi, 7.0, -20.0, 100.0])
    print("[wrap_angle outside |a| <= 2 pi + 1] " + ", ".join(f"{a!r} -> {w!r} (normalize_angle {orc.normalize_angle(float(a))!r})"
                                                             for a, w in zip(far, fm("wrap_angle", far))))


# ------------------------------------------------------------------------------------------------------------ sin / cos

def sincos_points(rng):
    q = np.arange(-64, 65) * (np.pi / 4)
    near = (q[:, None] + np.arange(-8, 9)[None, :] * np.spacing(np.maximum(np.abs(q), 1e-300))[:, None]).ravel()
    return np.concatenate([rng.uniform(-50, 50, 500_000), rng.uniform(-1e3, 1e3, 500_000), near,
                           (q[:, None] + rng.uniform(-1e-6, 1e-6, (q.size, 16))).ravel()])


def test_sincos_fast(fm):
    """sincos_fast on [-1e3, 1e3] (and [-50, 50], the multiples of pi / 4 and their neighbours): <= 1.7 ulp of the correctly rounded
    sin / cos (the header's bound; it is not 1 ulp); at |a| ~ 1e6, its documented limit: <= 2 ulp."""
    rng = np.random.default_rng(8)
    a = sincos_points(rng)
    s, c = fm("sincos_fast", a, nout=2)
    al = a.astype(np.longdouble)
    es, ec = ulps_ld(s, np.sin(al)), ulps_ld(c, np.cos(al))
    report("sincos_fast sin vs sinl", es.max(), SINCOS_ULP, "ulp", a[es.argmax()])
    report("sincos_fast cos vs cosl", ec.max(), SINCOS_ULP, "ulp", a[ec.argmax()])
    k = np.arange(-200, 201)
    base = np.concatenate([k * (np.pi / 4), k * (np.pi / 2)])
    sel = (base[:, None] + np.arange(-4, 5)[None, :] * np.spacing(np.maximum(np.abs(base), 1e-300))[:, None]).ravel()
    sel = np.concatenate([sel[sel != 0.0], rng.uniform(-50, 50, 20_000 - sel.size)])
    s, c = fm("sincos_fast", sel, nout=2)
    ms = [M(float(v)) for v in sel]
    e2 = max(ulps_mp(s, [mpmath.sin(v) for v in ms]).max(), ulps_mp(c, [mpmath.cos(v) for v in ms]).max())
    report("sincos_fast vs mpmath", e2, SINCOS_ULP, "ulp")
    big = np.concatenate([1e6 + rng.uniform(-1, 1, 100_000), -1e6 + rng.uniform(-1, 1, 100_000)])
    s, c = fm("sincos_fast", big, nout=2)
    bl = big.astype(np.longdouble)
    report("sincos_fast at |a| ~ 1e6", max(ulps_ld(s, np.sin(bl)).max(), ulps_ld(c, np.cos(bl)).max()), SINCOS_ULP_1E6, "ulp")


def test_sincos_small(fm):
    """sincos_small on both sides of 0.25: the series for |a| <= 0.25 (<= 1 ulp; the truncation alone is below 3e-18), and for
    |a| > 0.25 exactly sincos_fast's bits."""
    rng = np.random.default_rng(9)
    q = 0.25
    edge = np.array([0.0, -0.0, 1e-300, 1e-20, 1e-8, 1e-3, -1e-3, 0.02, -0.02, q, -q, np.nextafter(q, 0), np.nextafter(-q, 0),
                     np.nextafter(q, 1), np.nextafter(-q, -1), 0.26, -0.26, 0.9, -0.9, 3.0, -3.0])
    inside = np.concatenate([rng.uniform(-q, q, 1_000_000), edge[np.abs(edge) <= q]])
    s, c = fm("sincos_small", inside, nout=2)
    al = inside.astype(np.longdouble)
    nz = inside != 0.0
    es, ec = ulps_ld(s[nz], np.sin(al[nz])), ulps_ld(c, np.cos(al))
    report("sincos_small sin, |a| <= 0.25", es.max(), SINCOS_SMALL_ULP, "ulp", inside[nz][es.argmax()])
    report("sincos_small cos, |a| <= 0.25", ec.max(), SINCOS_SMALL_ULP, "ulp", inside[ec.argmax()])
    assert np.array_equal(s[~nz], inside[~nz]) and (c[~nz] == 1.0).all()
    sel = np.concatenate([edge[np.abs(edge) <= q], rng.uniform(-q, q, 20_000)])
    sel = sel[sel != 0.0]
    s, c = fm("sincos_small", sel, nout=2)
    ms = [M(float(v)) for v in sel]
    e2 = max(ulps_mp(s, [mpmath.sin(v) for v in ms]).max(), ulps_mp(c, [mpmath.cos(v) for v in ms]).max())
    report("sincos_small vs mpmath, |a| <= 0.25", e2, SINCOS_SMALL_ULP, "ulp")
    outside = np.concatenate([edge[np.abs(edge) > q], rng.uniform(0.25, 3.5, 10_000) * rng.choice([-1.0, 1.0], 10_000)])
    outside = outside[np.abs(outside) > q]
    s, c = fm("sincos_small", outside, nout=2)
    s2, c2 = fm("sincos_fast", outside, nout=2)
    assert np.array_equal(s, s2) and np.array_equal(c, c2), "|a| > 0.25 must take sincos_fast"
