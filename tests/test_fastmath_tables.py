"""The constant tables of csrc/fastmath.cuh against 200-bit mpmath, and sincos_fast (a __host__ __device__ function of pure fma
arithmetic) compiled for the host, against long-double and mpmath references.

The FAST EKF kernels agree with the oracle to ~1e-13, far inside the project's 1e-9 tolerance, so a wrong table entry or a lost
polynomial term would not show in the end-to-end tests. These tests read the tables from the header text itself (no copy of them
lives here) and pin every entry: a flipped last bit fails. They need no GPU: g++ compiles the header's own sincos_fast."""
import ast
import ctypes
import re
import shutil
import subprocess
from pathlib import Path

import mpmath
import numpy as np
import pytest

HEADER = Path(__file__).resolve().parent.parent / "shermbot-navigation_b200" / "csrc" / "fastmath.cuh"
mpmath.mp.prec = 200
M = mpmath.mpf


def _cexpr(s):
    """A C constant expression of the header (literals, unary minus, * and /), folded in IEEE double as the compiler folds it."""
    def ev(n):
        if isinstance(n, ast.Expression):
            return ev(n.body)
        if isinstance(n, ast.Constant) and isinstance(n.value, (int, float)):
            return float(n.value)
        if isinstance(n, ast.UnaryOp) and isinstance(n.op, ast.USub):
            return -ev(n.operand)
        if isinstance(n, ast.BinOp) and isinstance(n.op, (ast.Div, ast.Mult)):
            a, b = ev(n.left), ev(n.right)
            return a / b if isinstance(n.op, ast.Div) else a * b
        raise ValueError(f"unexpected constant expression {s!r}")
    return ev(ast.parse(s.strip(), mode="eval"))


def _array(text, name):
    m = re.search(r"__constant__\s+\w+\s+" + name + r"\[(\d+)\]\s*=\s*\{(.*?)\};", text, re.S)
    assert m, name
    return int(m.group(1)), m.group(2)


def _rows(body):
    return [[_cexpr(v) for v in row.split(",")] for row in re.findall(r"\{([^{}]*)\}", body)]


@pytest.fixture(scope="module")
def tables():
    text = HEADER.read_text()
    out = {}
    for name in ("kAtanTab", "kAtanUnit"):
        n, body = _array(text, name)
        rows = _rows(body)
        assert len(rows) == n == 65, name
        out[name] = rows
    for name in ("kFastK", "kFastK2", "kSinK", "kCosK"):
        n, body = _array(text, name)
        vals = [_cexpr(v) for v in body.split(",")]
        assert len(vals) == n, name
        out[name] = vals
    # the octant table is written with a macro: NUSLAM_Q(k) = (k) * pi/4 hi, (k) * pi/4 lo
    q = re.search(r"#define NUSLAM_Q\(k\) \(\(k\) \* ([-+.e\d]+)\), \(\(k\) \* ([-+.e\d]+)\)", text)
    assert q
    out["pi4"] = (float(q.group(1)), float(q.group(2)))
    n, body = _array(text, "kAtanOct")
    rows = re.findall(r"\{NUSLAM_Q\(([-.\d]+)\),\s*([-.\d]+),\s*([-.\d]+)\}", body)
    assert len(rows) == n == 8
    out["kAtanOct"] = [(float(k) * out["pi4"][0], float(k) * out["pi4"][1], float(s), float(k)) for k, s, _ in rows]
    return out


def _rounded(v):
    """v (mpf) correctly rounded to double."""
    return float(mpmath.mpf(v))


def test_atan_table(tables):
    """kAtanTab[k] = atan(k / 64) as hi + lo: hi correctly rounded, hi + lo within 1e-32; kAtanUnit carries the same (hi, lo) and
    cos / sin of atan(k / 64), each correctly rounded."""
    worst = 0.0
    for k, (hi, lo) in enumerate(tables["kAtanTab"]):
        a = mpmath.atan(M(k) / 64)
        assert hi == _rounded(a), k
        err = abs(M(hi) + M(lo) - a)
        worst = max(worst, float(err))
        assert err < M("1e-32"), (k, float(err))
    print(f"[kAtanTab] 65 rows: hi correctly rounded, worst |hi + lo - atan(k/64)| = {worst:.2e} (bound 1e-32)")
    for k, (hi, lo, c, s) in enumerate(tables["kAtanUnit"]):
        assert (hi, lo) == tuple(tables["kAtanTab"][k]), k
        t = M(k) / 64
        assert c == _rounded(1 / mpmath.sqrt(1 + t * t)), ("cos", k)
        assert s == _rounded(t / mpmath.sqrt(1 + t * t)), ("sin", k)


def test_octant_table(tables):
    """kAtanOct[swap | xneg << 1 | yneg << 2] = (A hi, A lo, S): atan2(y, x) = A + S atan(min / max) in each octant; pi / 4 split into
    a correctly rounded hi and a lo within 1e-32."""
    hi, lo = tables["pi4"]
    pi4 = mpmath.pi / 4
    assert hi == _rounded(pi4) and abs(M(hi) + M(lo) - pi4) < M("1e-32")
    for idx, (ahi, alo, s, k) in enumerate(tables["kAtanOct"]):
        assert ahi + alo == ahi and abs(M(ahi) + M(alo) - k * pi4) < M("1e-31")   # k * (hi, lo) is exact for k = 0, +-2, +-4
        sw, xneg, yneg = idx & 1, (idx >> 1) & 1, (idx >> 2) & 1
        mn, mx = M(3) / 10, M(1)
        ax, ay = (mn, mx) if sw else (mx, mn)
        x, y = (-ax if xneg else ax), (-ay if yneg else ay)
        want = mpmath.atan2(y, x)
        got = M(ahi) + M(alo) + s * mpmath.atan(mn / mx)
        assert abs(got - want) < M("1e-30"), (idx, float(got), float(want))


def test_scalar_constants(tables):
    """kFastK (atan series, 2 pi as hi + lo, 1 / 2 pi, 1e300, pi), kFastK2 (asin series), kSinK / kCosK (Taylor series of sin / cos):
    every coefficient is the correctly rounded value of what it stands for."""
    K = tables["kFastK"]
    assert K[0] == _rounded(M(-1) / 7) and K[1] == _rounded(M(1) / 5) and K[2] == _rounded(M(-1) / 3)
    assert K[3] == _rounded(2 * mpmath.pi) and abs(M(K[3]) + M(K[4]) - 2 * mpmath.pi) < M("1e-32")
    assert K[5] == _rounded(1 / (2 * mpmath.pi)) and K[6] == 1e300 and K[7] == _rounded(mpmath.pi)
    assert tables["kFastK2"][:3] == [_rounded(M(15) / 336), _rounded(M(3) / 40), _rounded(M(1) / 6)]
    assert tables["kSinK"] == [_rounded((-1) ** j / mpmath.factorial(2 * j + 1)) for j in range(1, 7)]
    assert tables["kCosK"] == [_rounded((-1) ** j / mpmath.factorial(2 * j)) for j in range(1, 8)]


def test_sincos_small_truncation(tables):
    """The header's bound on sincos_small's series: truncation error below 3e-18 for |a| <= 0.25 (exact arithmetic, the table's
    coefficients)."""
    a = M(1) / 4
    ps = sum(M(c) * a ** (2 * j + 3) for j, c in enumerate(tables["kSinK"])) + a
    pc = sum(M(c) * a ** (2 * j + 2) for j, c in enumerate(tables["kCosK"])) + 1
    es, ec = abs(ps - mpmath.sin(a)), abs(pc - mpmath.cos(a))
    print(f"[sincos_small] truncation at |a| = 0.25: sin {float(es):.2e}, cos {float(ec):.2e} (bound 3e-18)")
    assert es < 3e-18 and ec < 3e-18


# ---------------------------------------------------------------------------------------------------------------- sincos_fast on the host

SINCOS_BOUND_ULP = 1.7       # the header's bounds (fastmath.cuh, sincos_fast), in ulps of the correctly rounded value: |a| <= 1e3
SINCOS_BOUND_ULP_1E6 = 2.0   # |a| ~ 1e6, the end of the exact reduction


@pytest.fixture(scope="module")
def sincos_host(tmp_path_factory):
    """The header's sincos_fast, cut out of the header text and compiled by g++ with hardware fma (its arithmetic is fma, *, rint only,
    so the host computes the bits the device computes)."""
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("g++ not found")
    text = HEADER.read_text()
    m = re.search(r"__host__ __device__ __forceinline__ void sincos_fast\(.*?\n\}\n", text, re.S)
    assert m
    src = "\n".join(["#include <cmath>", "using std::fma; using std::rint;", "#define __host__", "#define __device__",
                     "#define __forceinline__ inline", m.group(0),
                     'extern "C" void sincos_fast_n(const double * a, double * s, double * c, long n)',
                     "{ for (long i = 0; i < n; ++i) sincos_fast(a[i], s + i, c + i); }", ""])
    d = tmp_path_factory.mktemp("sincos_host")
    (d / "sincos.cpp").write_text(src)
    lib = d / "libsincos.so"
    flags = ["-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC"]
    if subprocess.run([gxx, "-mfma", "-x", "c++", "-E", "-", "-o", "/dev/null"], input="", capture_output=True, text=True).returncode == 0:
        flags.append("-mfma")   # std::fma is exact with or without it; -mfma makes it one instruction
    subprocess.run([gxx, *flags, "-o", str(lib), str(d / "sincos.cpp")], check=True)
    dll = ctypes.CDLL(str(lib))
    fn = dll.sincos_fast_n
    fn.restype = None
    fn.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_long]

    def run(a):
        a = np.ascontiguousarray(a, dtype=np.float64)
        s, c = np.empty_like(a), np.empty_like(a)
        fn(a.ctypes.data, s.ctypes.data, c.ctypes.data, a.size)
        return s, c
    return run


def ulp_err_ld(got, ref_ld):
    """|got - ref| in ulps of the correctly rounded value (ref in long double)."""
    cr = ref_ld.astype(np.float64)
    ulp = np.spacing(np.abs(cr)).astype(np.longdouble)
    return np.abs((got.astype(np.longdouble) - ref_ld) / ulp).astype(np.float64)


def sincos_points(rng):
    """[-50, 50] and [-1e3, 1e3] at random, the neighbourhoods of multiples of pi / 4 (the reduction's and the quadrant logic's
    edges), and tiny arguments."""
    q = np.arange(-64, 65) * (np.pi / 4)
    near = (q[:, None] + np.arange(-8, 9)[None, :] * np.spacing(np.maximum(np.abs(q), 1e-300))[:, None]).ravel()
    near = np.concatenate([near, (q[:, None] + rng.uniform(-1e-6, 1e-6, (q.size, 16))).ravel()])
    tiny = np.concatenate([[0.0, -0.0, 1e-300, -1e-300, 1e-20, 2.0 ** -27], rng.uniform(-1e-4, 1e-4, 500)])
    return np.concatenate([rng.uniform(-50, 50, 500_000), rng.uniform(-1e3, 1e3, 500_000), near, tiny])


def test_sincos_fast_host_longdouble(sincos_host):
    """sincos_fast on [-1e3, 1e3] and around multiples of pi / 4 against sinl / cosl: within the header's 1.7 ulp of the correctly
    rounded value. (It is NOT within 1 ulp: the fdlibm kernels are ~0.5 ulp from sin / cos of the reduced argument, and the
    reduced argument is rounded once more.)"""
    a = sincos_points(np.random.default_rng(5))
    s, c = sincos_host(a)
    al = a.astype(np.longdouble)
    es, ec = ulp_err_ld(s, np.sin(al)), ulp_err_ld(c, np.cos(al))
    nz = a != 0.0
    ws, wc = es[nz].max(), ec.max()
    print(f"[sincos_fast host, {a.size} points] worst sin {ws:.3f} ulp at {a[nz][es[nz].argmax()]!r}, cos {wc:.3f} ulp at {a[ec.argmax()]!r} "
          f"(bound {SINCOS_BOUND_ULP} ulp)")
    assert ws <= SINCOS_BOUND_ULP and wc <= SINCOS_BOUND_ULP
    assert np.array_equal(s[~nz], a[~nz]) and (c[~nz] == 1.0).all()   # sin(+-0) = +-0


def test_sincos_fast_host_mpmath(sincos_host):
    """~2e4 chosen points against 200-bit mpmath: multiples of pi / 4 and pi / 2 and their neighbours (where sin or cos is near 0 and
    the reduction cancels), [-50, 50], and the documented range limit |a| ~ 1e6."""
    rng = np.random.default_rng(6)
    k = np.arange(-200, 201)
    base = np.concatenate([k * (np.pi / 4), k * (np.pi / 2)])
    pts = np.concatenate([(base[:, None] + np.arange(-4, 5)[None, :] * np.spacing(np.maximum(np.abs(base), 1e-300))[:, None]).ravel(),
                          rng.uniform(-50, 50, 8000)])
    pts = pts[pts != 0.0]
    s, c = sincos_host(pts)
    worst = 0.0
    for a, sv, cv in zip(pts, s, c):
        ma = M(float(a))
        for got, ref in ((sv, mpmath.sin(ma)), (cv, mpmath.cos(ma))):
            cr = float(ref)
            worst = max(worst, float(abs(M(float(got)) - ref) / M(float(np.spacing(abs(cr))))))
    print(f"[sincos_fast host vs mpmath, {pts.size} points] worst {worst:.3f} ulp (bound {SINCOS_BOUND_ULP})")
    assert worst <= SINCOS_BOUND_ULP
    # the documented limit: up to |a| ~ 1e6 the three-piece reduction is exact, and the error stays within 2 ulp
    big = np.concatenate([1e6 + rng.uniform(-1, 1, 2000), -1e6 + rng.uniform(-1, 1, 2000)])
    s, c = sincos_host(big)
    bl = big.astype(np.longdouble)
    wb = max(ulp_err_ld(s, np.sin(bl)).max(), ulp_err_ld(c, np.cos(bl)).max())
    print(f"[sincos_fast host at |a| ~ 1e6] worst {wb:.3f} ulp (bound {SINCOS_BOUND_ULP_1E6})")
    assert wb <= SINCOS_BOUND_ULP_1E6
