"""The scan detector on the paths that the tube workload of tests/test_scan_gpu.py never reaches.

Both arithmetics (the moment route of scan_moment.cuh and the oracle-order Jacobi pipeline of scan_detect.cuh) choose among about a
dozen code paths by cluster size, cluster count, batch size, range gate and pointer alignment. The scenes below are built to reach
each of them:

* whole-scan arcs seen from inside a circle (clusters of more than 126 points: k_scan_fit_big<kBeams + 2, 2, false>, and the moment
  route's multi-batch point loop), some wrapping past beam 359;
* crowded scans (more than 32 pre-erase or kept clusters: the pipeline's slow list, the latency kernel's second round of 32 clusters,
  the moment route's hand-over) with more published circles than max_circles (the three truncation sites);
* a conditioning sweep of tubes seen from outside, radii straddling the 1 m gate, nearly collinear arcs, and "V" clusters whose
  inscribed-angle std lies within 1e-6 degrees of the 10 degree threshold (the moment route's guards);
* range gates float cannot represent, ranges a few ulps either side of them, neighbour differences within one ulp of 0.04, and wide
  gates with huge, infinite and NaN ranges (the big_gate branch);
* unaligned range and cluster_of_beam buffers, no cluster_of_beam, host against device memory;
* a batch of kScanChunk + 300 scans (two pipeline chunks).

Every GPU test runs in both fit modes, at a batch of at most 256 scans (the Jacobi latency path) and mixed into 4096 scenario scans
(the throughput path). The checker is the oracle; the bar is the suite's: cluster ids, cluster and circle counts exact, circles within
1e-9 relative. Scenes are plain numpy: ranges are analytic ray / circle (or ray / segment) distances stored as float32, as
synth.simulate_scans stores them."""
import functools

import numpy as np
import pytest

from shermbot_navigation_b200 import synth
from test_scan_gpu import compare_scans

BEAMS = 360
ANG = np.deg2rad(np.arange(BEAMS))
UX, UY = np.cos(ANG), np.sin(ANG)
GATE = (synth.MIN_RANGE, synth.MAX_RANGE)
SCAN_CHUNK = 262144          # kScanChunk of scan_detect.cuh
LATENCY_MAX = 256            # batches up to this size take the one-launch latency path in Jacobi mode
SIZE_CLASSES = ((1, 12), (13, 32), (33, 126), (127, BEAMS + 1))   # the Jacobi pipeline's fit classes (points per kept cluster)


# ------------------------------------------------------------------------------------------------------------------ scene builders

def _store(t, max_range, noise=0.0, rng=None, fill=None):
    """Distances -> float32 ranges the way synth.simulate_scans stores them: optional Gaussian noise, then anything that is not a
    finite hit within max_range becomes the fill value max_range + 1."""
    t = np.asarray(t, dtype=np.float64)
    if noise > 0:
        t = t + rng.normal(0.0, noise, t.shape)
    fill = max_range + 1.0 if fill is None else fill
    return np.where(np.isfinite(t) & (t <= max_range), t, fill).astype(np.float32)


def inside_circle(cx, cy, R):
    """Distance along every beam from the origin to a circle (centre (cx, cy), radius R) that contains the origin."""
    p = cx * UX + cy * UY
    return p + np.sqrt(p * p - (cx * cx + cy * cy) + R * R)


def outside_circle(cx, cy, rho):
    """Distance along every beam to a tube (centre (cx, cy), radius rho) that does not contain the origin; inf where the beam misses."""
    p = cx * UX + cy * UY
    disc = rho * rho - (cx * cx + cy * cy) + p * p
    with np.errstate(invalid="ignore"):
        t = p - np.sqrt(disc)
    return np.where((disc >= 0) & (t > 0), t, np.inf)


def segments(segs):
    """Distance along every beam to the nearest of the segments (x0, y0, x1, y1); inf where the beam misses them all."""
    best = np.full(BEAMS, np.inf)
    for x0, y0, x1, y1 in segs:
        ex, ey = x1 - x0, y1 - y0
        den = UX * ey - UY * ex
        with np.errstate(divide="ignore", invalid="ignore"):
            t = (x0 * ey - y0 * ex) / den
            s = (x0 * UY - y0 * UX) / den
        ok = (np.abs(den) > 1e-12) & (t > 0) & (s >= 0) & (s <= 1)
        best = np.where(ok & (t < best), t, best)
    return best


def _window(start, length):
    w = np.zeros(BEAMS, dtype=bool)
    w[(start + np.arange(length)) % BEAMS] = True
    return w


def arc_scan(R, length, start, noise=0.0, seed=0, max_range=1.0):
    """An arc of `length` beams from inside a circle of radius R, centred on beam start + length / 2; every other beam is fill. The
    robot sits off the circle's centre by the smallest offset that keeps the whole arc inside the range window (None: impossible)."""
    w = _window(start, length)
    psi = np.deg2rad(start + length / 2.0)
    margin = 4 * noise
    for d in np.concatenate([np.linspace(0.0, 1e-3, 41), np.linspace(1e-3, max(R - 0.1, 1e-3), 600)]):
        t = inside_circle(-d * np.cos(psi), -d * np.sin(psi), R)
        tw = t[w]
        if tw.max() + margin <= max_range and tw.min() - margin >= 0.08:
            t = np.where(w, t, np.inf)
            return _store(t, max_range, noise, np.random.default_rng(seed))
    return None


# radii: the span of the task, the gate at 1 m to rounding, 1 +- 1e-5 and 0.999; lengths 127 .. 330 beams; starts near 359 wrap
ARC_RADII = (0.3, 0.45, 0.6, 0.8, 0.95, 0.999, 1 - 1e-5, 1 - 1e-7, 1 + 1e-7, 1 + 1e-5, 1.05, 1.2)
ARC_LENGTHS = (127, 150, 180, 210, 250, 300, 330)


def arc_scans(noise):
    scans, near = [], []
    for i, R in enumerate(ARC_RADII):
        for j, L in enumerate(ARC_LENGTHS):
            start = (37 * i + 101 * j) % BEAMS if (i + j) % 3 else BEAMS - L // 3   # every third arc wraps past beam 359
            s = arc_scan(R, L, start, noise, seed=1000 * i + j)
            if s is not None:
                scans.append(s)
                near.append(noise == 0 and abs(R - 1) < 1e-6)
    return np.stack(scans), np.array(near)


def _levels(n, lo=0.25, step=0.07, k=6):
    """n constant ranges, neighbours (cyclically) at least `step` apart: lo + step * (0, 2, 4, 1, 3, 5, ...)."""
    order = np.array([0, 2, 4, 1, 3, 5][:k])
    lv = lo + step * order[np.arange(n) % k]
    if n % k == 1:
        lv[-1] = lo + step * 3   # keep the last level away from the first (no wrap onto cluster 0)
    return lv


def crowded_scans():
    """Constant-range arcs (each a published circle about the robot) and small clusters in every mix the clustering walk and the
    erase loop distinguish: 33 - 40 kept arcs; more than 32 pre-erase clusters of which at most 32 are kept (one- and two-beam
    clusters between arcs); more than 32 kept clusters of which only a few are circles (3-beam clusters: circleFit rejects N < 4)."""
    scans = []
    rng = np.random.default_rng(7)
    for nk in (33, 34, 36, 38, 40, 45):
        sizes = np.full(nk, BEAMS // nk)
        sizes[: BEAMS - sizes.sum()] += 1
        r = np.repeat(_levels(nk), sizes)
        scans.append(np.roll(r, rng.integers(0, BEAMS)).astype(np.float32))
    for group, arc_len in (((1,), 12), ((1,), 14), ((2,), 16), ((1,), 8), ((1, 2), 9), ((2, 1), 7), ((1, 1), 6)):
        # arc, small, [small], arc, ...: the first small after a kept cluster is erased, the one after it is never examined (kept)
        parts = []
        k = 0
        while sum(len(p) for p in parts) + arc_len + sum(group) + 4 <= BEAMS:
            parts.append(np.full(arc_len, 0.3 + 0.07 * (k % 2)))
            for g, sz in enumerate(group):
                parts.append(np.full(sz, 0.55 + 0.1 * g + 0.2 * (k % 2)))
            k += 1
        r = np.concatenate(parts)
        scans.append(np.concatenate([r, np.full(BEAMS - len(r), 2.0)]).astype(np.float32))
    for n_arcs in (1, 3, 5, 20):
        parts = []
        k = 0
        for a in range(n_arcs):
            parts.append(np.full(10, 0.8 - 0.05 * (a % 2)))
        while sum(len(p) for p in parts) + 3 <= BEAMS - 2:
            parts.append(np.full(3, _levels(6)[k % 6] if k % 6 != 5 else 0.6))   # 3-beam clusters: classified, circleFit id -1
            k += 1
        r = np.concatenate(parts)
        scans.append(np.concatenate([r, np.full(BEAMS - len(r), 2.0)]).astype(np.float32))
    # the crowded scans with 1e-3 noise on the arcs' ranges (keeps the clusters: levels are 0.07 apart)
    noisy = [(s + np.where(s < 1.0, rng.normal(0, 1e-3, BEAMS), 0.0)).astype(np.float32) for s in scans[:6]]
    return np.stack(scans + noisy)


def tube_scans(noise, seed=11):
    """Tubes seen from outside: radius 0.01 .. 1.2 at distances from just outside the tube up to the range gate (spans of 4 beams to
    most of a half circle), one or two per scan, at random bearings."""
    rng = np.random.default_rng(seed)
    scans = []
    for rho in np.geomspace(0.01, 1.2, 14):
        for gap in (0.07, 0.15, 0.3, 0.5, 0.7, 0.9):
            psi = rng.uniform(0, 2 * np.pi)
            D = rho + gap
            t = outside_circle(D * np.cos(psi), D * np.sin(psi), rho)
            if gap < 0.5 and rho < 0.3:   # a second tube on the far side
                D2, psi2 = rho + 0.6, psi + np.pi
                t = np.minimum(t, outside_circle(D2 * np.cos(psi2), D2 * np.sin(psi2), rho))
            s = _store(t, 1.0, noise, rng)
            if (s <= 1.0).sum() >= 4:
                scans.append(s)
    return np.stack(scans)


def gate_tube_scans():
    """Noise-free tubes and arcs whose radius is within 1e-5 of the 1 m publication gate (R within 1e-6 of it: the moment route must
    hand the scan over), R = 0.999, and nearly collinear arcs of R = 5 .. 50 m (classified circles, then gated)."""
    rng = np.random.default_rng(13)
    scans, near = [], []
    for rho in (1 - 1e-5, 1 - 1e-7, 1.0, 1 + 1e-7, 1 + 1e-5, 0.999, 1 - 5e-7, 1 + 5e-7):
        for gap in (0.08, 0.2, 0.45):
            psi = rng.uniform(0, 2 * np.pi)
            D = rho + gap
            scans.append(_store(outside_circle(D * np.cos(psi), D * np.sin(psi), rho), 1.0))
            near.append(abs(rho - 1) < 1e-6)
    for rho in (5.0, 10.0, 20.0, 50.0):
        for gap in (0.2, 0.5, 0.8):
            psi = rng.uniform(0, 2 * np.pi)
            D = rho + gap
            scans.append(_store(outside_circle(D * np.cos(psi), D * np.sin(psi), rho), 1.0))
            near.append(False)
    return np.stack(scans), np.array(near)


def v_scan(delta, Dc, a1, a2, psi):
    """A "V" of two segments meeting at a corner at distance Dc in direction psi, its arms (lengths a1, a2) tilted by delta towards
    the robot: delta = 0 is a straight wall, larger delta a deeper V with a larger spread of inscribed angles."""
    c, s = np.cos(psi), np.sin(psi)
    rot = lambda x, y: (c * x - s * y, s * x + c * y)
    C = rot(Dc, 0.0)
    E1 = rot(Dc - a1 * np.sin(delta), a1 * np.cos(delta))
    E2 = rot(Dc - a2 * np.sin(delta), -a2 * np.cos(delta))
    return _store(segments([(*C, *E1), (*C, *E2)]), 1.0)


def _v_cluster(orc, ranges):
    cl = orc.cluster_points(ranges, *GATE)
    return max(cl, key=lambda c: len(c[0]))[1]


def inscribed_std(pts):
    """classifyCluster's statistic (circle_fit_library.cpp:208-250) in numpy: population std of the inscribed angles, degrees."""
    p2, p3, p1 = pts[0], pts[-1], pts[1:-1]
    num = p2[1] * (p1[:, 0] - p3[0]) + p1[:, 1] * (p3[0] - p2[0]) + p3[1] * (p2[0] - p1[:, 0])
    den = (p2[0] - p1[:, 0]) * (p1[:, 0] - p3[0]) + (p2[1] - p1[:, 1]) * (p1[:, 1] - p3[1])
    ang = np.rad2deg(np.arctan2(num, den))
    return float(np.sqrt(((ang - ang.mean()) ** 2).mean()))


V_SHAPES = ((0.6, 0.25, 0.2, 0.9), (0.8, 0.15, 0.3, 2.0), (0.5, 0.3, 0.2, 4.0), (0.7, 0.2, 0.2, 5.5), (0.9, 0.1, 0.25, 1.1),
            (0.45, 0.2, 0.35, 3.3))


@functools.lru_cache(maxsize=None)
def v_scans(flavour):
    """For each V shape, the two scans either side of the classifier's threshold: the corner tilt is bisected on the oracle's
    classifyCluster over the float-rounded points until the two tilts are adjacent doubles (their ranges then differ by an ulp or
    so), which puts the inscribed-angle std of both within about 1e-6 degrees of 10."""
    import oracle
    orc = oracle.load(flavour)
    scans = []
    for Dc, a1, a2, psi in V_SHAPES:
        lo, hi = 0.0, np.deg2rad(40.0)
        assert orc.classify_cluster(_v_cluster(orc, v_scan(lo, Dc, a1, a2, psi)))
        assert not orc.classify_cluster(_v_cluster(orc, v_scan(hi, Dc, a1, a2, psi)))
        while True:
            mid = 0.5 * (lo + hi)
            if mid <= lo or mid >= hi:
                break
            if orc.classify_cluster(_v_cluster(orc, v_scan(mid, Dc, a1, a2, psi))):
                lo = mid
            else:
                hi = mid
        scans += [_v_tune(orc, v_scan(lo, Dc, a1, a2, psi), True), _v_tune(orc, v_scan(hi, Dc, a1, a2, psi), False)]
    return np.stack(scans)


def _v_tune(orc, r, circle):
    """Bring the std still closer to 10 degrees without crossing it: move single ranges of the cluster by one float ulp, greedily."""
    beams = max(orc.cluster_points(r, *GATE), key=lambda c: len(c[0]))[0]
    pts = lambda q: np.stack([q[beams].astype(np.float64) * UX[beams], q[beams].astype(np.float64) * UY[beams]], axis=1)
    best, cur = r, abs(inscribed_std(pts(r)) - 10.0)
    for _ in range(40):
        if cur < 1e-8:
            break
        step = None
        for b in beams:
            for k in (-1, 1):
                q = best.copy()
                q[b] = _ulps(q[b], k)
                s = inscribed_std(pts(q))
                if (s < 10.0) == circle and abs(s - 10.0) < cur:
                    step, cur = q, abs(s - 10.0)
        if step is None:
            break
        best = step
    return best if orc.classify_cluster(_v_cluster(orc, best)) == circle else r


def _ulps(v, k):
    """The float k ulps above (k > 0) or below the float nearest to v."""
    f = np.float32(v)
    for _ in range(abs(k)):
        f = np.nextafter(f, np.float32(np.inf if k > 0 else -np.inf), dtype=np.float32)
    return f


def gate_edge_scans(lo, hi, n=24, seed=17):
    """Runs of 3 - 12 beams whose ranges are drawn from the floats within 3 ulps of a gate (so some beams of a run are out of range
    and are skipped, while their neighbours compare against them), separated by fill; and staircases whose steps lie within one float
    ulp of 0.04 on either side (similar / not similar decided by the double difference)."""
    rng = np.random.default_rng(seed)
    fill = np.float32(hi + 1.0)
    near = {g: np.array([_ulps(g, k) for k in range(-3, 4)], dtype=np.float32) for g in (lo, hi) if g > 0}
    scans = []
    for k in range(n):
        r = np.full(BEAMS, fill, np.float32)
        b = int(rng.integers(0, 3))
        while b < BEAMS - 14:
            L = int(rng.integers(3, 13))
            vals = near[list(near)[int(rng.integers(0, len(near)))]]
            r[b:b + L] = vals[rng.integers(0, len(vals), L)]
            b += L + int(rng.integers(1, 4))
        scans.append(r)
    top = min(max(hi, lo + 0.8), 1e3)   # (a staircase may leave a narrow window: its beams beyond the gate are skipped)
    for k in range(n):
        r = np.full(BEAMS, fill, np.float32)
        b = 0
        while b < BEAMS - 40:
            v = np.float32(max(lo, 1e-3) + rng.uniform(0.001, 0.02))
            while b < BEAMS - 1 and float(v) + 0.05 < top:
                r[b] = v
                target = float(v) + 0.04
                lo_f = np.float32(target)
                lo_f = lo_f if float(lo_f) < target else np.nextafter(lo_f, np.float32(-np.inf), dtype=np.float32)
                hi_f = np.nextafter(lo_f, np.float32(np.inf), dtype=np.float32)
                v = lo_f if rng.random() < 0.5 else hi_f
                b += 1
            b += int(rng.integers(2, 6))
        scans.append(r)
    return np.stack(scans)


WIDE_VALUES = (0.03, 0.5, 1.0, 31.9, 32.0, 39.99, 40.0, 40.01, 63.99, 64.0, 64.02, 100.0, 999.0, 1e3, 9999.0, 1e4, 1.0001e4, 3e4,
               np.inf, -np.inf, np.nan)


def wide_gate_scans(hi, n=24, seed=19):
    """For wide gates (min_range 0): runs near and beyond the gate, near the 32 m / 64 m magnitude limits of the moment route's float
    decisions, +-inf and NaN; constant-range arcs of 30 m (circles, gated); staircases of 0.04 +- an ulp at 70 m."""
    rng = np.random.default_rng(seed)
    vals = list(WIDE_VALUES)
    for g in (40.0, 64.0, hi):
        vals += [float(_ulps(g, k)) for k in (-2, -1, 1, 2)]
    vals = np.array(vals, dtype=np.float32)
    scans = []
    for k in range(n):
        r = np.full(BEAMS, np.float32(np.inf), np.float32)
        b = 0
        while b < BEAMS - 12:
            L = int(rng.integers(1, 12))
            base = vals[int(rng.integers(0, len(vals)))]
            run = np.full(L, base, np.float32)
            if np.isfinite(base) and rng.random() < 0.5:
                run = (base + rng.uniform(-0.03, 0.03, L).astype(np.float32)).astype(np.float32)   # similar neighbours at that magnitude
            r[b:b + L] = run
            b += L + int(rng.integers(1, 3))
        scans.append(r)
    arc = np.full(BEAMS, np.float32(np.inf), np.float32)
    arc[10:50] = np.float32(30.0)
    arc[100:140] = np.float32(70.0)
    v = np.float32(70.2)
    for b in range(200, 300):
        arc[b] = v
        lo_f = np.float32(float(v) + 0.04)
        lo_f = lo_f if float(lo_f) < float(v) + 0.04 else np.nextafter(lo_f, np.float32(-np.inf), dtype=np.float32)
        v = lo_f if b % 3 else np.nextafter(lo_f, np.float32(np.inf), dtype=np.float32)
    scans.append(arc)
    return np.stack(scans)


GATES = ((0.05, 1.0), (0.12, 3.5), (0.05, 0.12), (0.02, 0.05), (1.0, 3.5), (0.12, 1.0))
WIDE_GATES = ((0.0, 40.0), (0.0, 1e4))


# ------------------------------------------------------------------------------------------------------------------ helpers

@functools.lru_cache(maxsize=None)
def scenario():
    return synth.scan_scenario(4096, seed=47, noise_sigma=0.001)["ranges"]


def batches(special, kind):
    """The special scans alone (at most 256 per call: the latency path), or mixed into 4096 scenario scans: a third at the start, a
    third in the middle and the rest at the end. Returns the batch and the positions of the special scans in it."""
    special = np.asarray(special, dtype=np.float32)
    n = len(special)
    if kind == "alone":
        assert n <= LATENCY_MAX
        return special, np.arange(n)
    base = scenario()
    a, b = n // 3, 2 * n // 3
    mid = len(base) // 2
    out = np.concatenate([special[:a], base[:mid], special[a:b], base[mid:], special[b:]])
    pos = np.concatenate([np.arange(a), a + mid + np.arange(b - a), a + len(base) + (b - a) + np.arange(n - b)])
    return out, pos


def run(orc, ranges, lo, hi, kmax=16):
    from shermbot_navigation_b200 import circle_fit
    want = orc.scan_detect_batch(ranges, lo, hi, kmax=kmax, nthreads=0)
    got = circle_fit.scan_detect(ranges, lo, hi, max_circles=kmax)
    worst = compare_scans(got, want)
    return got, want, worst


def same_bits(a, b, ref):
    """Every defined output of two scan_detect calls bit for bit: cluster ids (when both have them), counts, and the circle slots
    the call writes (the first min(n_circles, max_circles) of each scan; the rest are not outputs)."""
    for key in ("cluster_of_beam", "n_clusters", "n_circles"):
        if a[key] is not None and b[key] is not None:
            assert np.array_equal(a[key], b[key]), key
    kmax = ref["circles"].shape[1]
    k = np.clip(ref["n_circles"], 0, kmax)
    written = np.arange(kmax)[None, :] < k[:, None]
    ca, cb = a["circles"].view(np.int64)[written], b["circles"].view(np.int64)[written]
    assert np.array_equal(ca, cb), "circles differ"


def _np(out):
    return {k: (v.cpu().numpy() if v is not None and hasattr(v, "cpu") else v) for k, v in out.items()}


def published_sizes(want):
    """Points of every published circle's cluster (cluster ids per beam, beam 359 of the wrap rule included)."""
    sizes = []
    kmax = want["circles"].shape[1]
    for s in np.nonzero(want["n_circles"] > 0)[0]:
        for q in want["circles"][s, : min(int(want["n_circles"][s]), kmax), 3].astype(int):
            sizes.append(int((want["cluster_of_beam"][s] == q).sum()))
    return np.array(sizes, dtype=int)


@pytest.fixture(params=["moment", "jacobi"])
def fit_mode(request, cuda_lib):
    """Both circle-fit arithmetics of the batched path; the previous mode is restored afterwards."""
    from shermbot_navigation_b200 import circle_fit
    prev = circle_fit.set_fit(request.param)
    yield request.param
    circle_fit.set_fit(prev)


@pytest.fixture(params=["alone", "mixed"])
def batch(request):
    return request.param


# ------------------------------------------------------------------------------------------------------------------ CPU: the scenes

def test_scenes_reach_their_paths(orc):
    """The scenes through the oracle alone: they must keep reaching what the GPU tests claim to exercise, so that a change to a
    builder cannot quietly turn them back into easy data."""
    sizes = []
    for noise in (0.0, 1e-3):
        a, near = arc_scans(noise)
        w = orc.scan_detect_batch(a, *GATE, nthreads=0)
        big = published_sizes(w)
        sizes.append(big)
        assert (big > 126).sum() >= 20, f"noise {noise}: {(big > 126).sum()} published clusters of > 126 points"
        assert (big > 200).sum() >= 5 and len(a) <= LATENCY_MAX
        if noise == 0:
            assert near.sum() >= 4
            wr = w["cluster_of_beam"][:, BEAMS - 1]
            assert ((wr == 0) & (w["n_circles"] > 0)).sum() >= 5, "published arcs that wrap past beam 359"
    cr = crowded_scans()
    w = orc.scan_detect_batch(cr, *GATE, kmax=64, nthreads=0)
    sizes.append(published_sizes(w))
    assert ((w["n_clusters"] > 32) & (w["n_circles"] > 32)).sum() >= 4, "scans with more than 32 kept clusters, all published"
    assert ((w["n_clusters"] > 32) & (w["n_circles"] > 0) & (w["n_circles"] <= 5)).sum() >= 3, "> 32 kept clusters, few circles"
    # more than 32 pre-erase clusters (closers) while at most 32 are kept
    inr = (cr >= np.float32(GATE[0])) & (cr <= np.float32(GATE[1]))
    closers = (inr & ~(np.abs(cr.astype(np.float64) - np.roll(cr, -1, axis=1)) < 0.04)).sum(axis=1)
    assert ((closers > 32) & (w["n_clusters"] <= 32) & (w["n_circles"] > 16)).sum() >= 2
    assert (w["n_circles"] > 16).sum() >= 6 and (w["n_circles"] > 1).sum() >= 10, "more circles than max_circles"
    for noise in (0.0, 1e-3):
        t = tube_scans(noise)
        w = orc.scan_detect_batch(t, *GATE, nthreads=0)
        sizes.append(published_sizes(w))
        assert len(t) <= LATENCY_MAX and (w["n_circles"] > 0).mean() > 0.5
    g, near = gate_tube_scans()
    w = orc.scan_detect_batch(g, *GATE, nthreads=0)
    sizes.append(published_sizes(w))
    R = w["circles"][:, 0, 2]
    assert ((w["n_circles"] > 0) & near & (np.abs(R - 1) < 1e-6)).sum() >= 3, "published circles within 1e-6 of the 1 m gate"
    # classified circles of R > 1 m that the gate drops (the nearly collinear arcs, the tubes just above 1 m)
    gated = 0
    for s in g:
        for _, pts in orc.cluster_points(s, *GATE):
            if len(pts) >= 4 and orc.classify_cluster(pts):
                mid, _, _, r = orc.circle_fit(pts)
                gated += mid == 0 and r > 5
    assert gated >= 6, gated
    sizes = np.concatenate(sizes)
    for lo, hi in SIZE_CLASSES:
        n = int(((sizes >= lo) & (sizes <= hi)).sum())
        assert n >= 20, f"only {n} published circles of {lo}..{hi} points"
    # V clusters: both sides of the threshold, within 1e-6 degrees of it (the moment route's guard on var within 2e-5 of 100)
    v = v_scans(orc.kind)
    stds = np.array([inscribed_std(_v_cluster(orc, s)) for s in v])
    cls = np.array([orc.classify_cluster(_v_cluster(orc, s)) for s in v])
    assert cls[0::2].all() and not cls[1::2].any()
    assert (np.abs(stds - 10.0) < 1e-6).sum() >= 4, stds - 10.0
    # range gates: ranges within 2 ulps of each gate, on both sides, in range and out of it
    for lo, hi in GATES:
        e = gate_edge_scans(lo, hi)
        for gv in (lo, hi):
            f = np.float32(gv)
            ulp = np.abs(np.nextafter(f, np.float32(np.inf), dtype=np.float32) - f)
            d = e.astype(np.float64) - gv
            assert ((d > 0) & (d < 2 * ulp)).sum() > 20 and ((d < 0) & (d > -2 * ulp)).sum() > 20, (lo, hi, gv)
        # steps within one float ulp of 0.04, both below and above (decided by the double comparison)
        st = np.abs(e[:, 1:].astype(np.float64) - e[:, :-1])
        ulp = np.spacing(e[:, 1:].astype(np.float32)).astype(np.float64)
        dd = st - 0.04
        assert ((dd < 0) & (dd > -ulp)).sum() > 50 and ((dd > 0) & (dd < ulp)).sum() > 50, (lo, hi)
        w = orc.scan_detect_batch(e, lo, hi, nthreads=0)
        assert (w["n_clusters"] > 0).mean() > 0.5
    for lo, hi in WIDE_GATES:
        e = wide_gate_scans(hi)
        assert np.isnan(e).any() and np.isposinf(e).any() and np.isneginf(e).any()
        inr = (e >= lo) & (e <= hi)
        assert (inr & (e > min(hi, 64.0) - 1)).any() and (~inr & np.isfinite(e) & (e > hi)).any()
        w = orc.scan_detect_batch(e, lo, hi, nthreads=0)
        assert (w["n_clusters"] > 0).mean() > 0.5


# ------------------------------------------------------------------------------------------------------------------ GPU

@pytest.mark.gpu
@pytest.mark.parametrize("noise", [0.0, 1e-3])
def test_whole_scan_arcs(orc, fit_mode, batch, noise):
    """Arcs of 127 - 330 beams from inside circles of R = 0.3 .. 1.2 (1 +- 1e-7, 1 +- 1e-5 and 0.999 included), some wrapping past
    beam 359: the only clusters that reach k_scan_fit_big<kBeams + 2, 2, false> and the moment route's multi-batch point loop."""
    from shermbot_navigation_b200 import circle_fit
    arcs, near = arc_scans(noise)
    r, pos = batches(arcs, batch)
    got, want, worst = run(orc, r, *GATE)
    fb = circle_fit.last_fallbacks() if fit_mode == "moment" else 0
    print(f"[arcs noise={noise} fit={fit_mode} {batch}] {len(r)} scans, {int(want['n_circles'][pos].clip(0).sum())} published arcs, "
          f"worst rel {worst:.2e}, re-run in oracle order {fb}")
    if fit_mode == "moment" and near.any():
        circle_fit.scan_detect(arcs[near], *GATE)
        assert circle_fit.last_fallbacks() > 0, "arcs within 1e-6 of the 1 m gate must be handed to the oracle-order kernel"


@pytest.mark.gpu
@pytest.mark.parametrize("max_circles", [1, 16, 64])
def test_crowded_scans(orc, fit_mode, batch, max_circles):
    """33 - 45 kept clusters per scan, more than 32 pre-erase clusters with at most 32 kept, more than 32 kept with a few circles:
    the pipeline's slow list, the latency kernel's second round of 32, the moment route's hand-over, and max_circles truncation in
    k_scan_publish, k_scan_moment and the inline path (n_circles counts every published circle)."""
    r, pos = batches(crowded_scans(), batch)
    got, want, worst = run(orc, r, *GATE, kmax=max_circles)
    assert (want["n_circles"][pos] > max_circles).any() or max_circles == 64
    print(f"[crowded max_circles={max_circles} fit={fit_mode} {batch}] {len(r)} scans, most circles in a scan "
          f"{int(want['n_circles'].max())}, worst rel {worst:.2e}")


@pytest.mark.gpu
def test_conditioning_sweep(orc, fit_mode, batch):
    """Tubes of radius 0.01 .. 1.2 from just outside to the gate (noise-free and 1e-3), radii within 1e-5 of the 1 m gate, nearly
    collinear arcs of 5 - 50 m, and V clusters either side of the 10 degree threshold. In moment mode the scans near a gate must be
    handed to the oracle-order kernel."""
    from shermbot_navigation_b200 import circle_fit
    gate, near = gate_tube_scans()
    v = v_scans(orc.kind)
    special = np.concatenate([tube_scans(0.0), tube_scans(1e-3, seed=12), gate, v])
    assert len(special) <= LATENCY_MAX
    r, pos = batches(special, batch)
    got, want, worst = run(orc, r, *GATE)
    fb = circle_fit.last_fallbacks() if fit_mode == "moment" else 0
    print(f"[conditioning fit={fit_mode} {batch}] {len(r)} scans, worst rel {worst:.2e}, re-run in oracle order {fb}")
    if fit_mode == "moment":
        circle_fit.scan_detect(gate[near], *GATE)
        fb_gate = circle_fit.last_fallbacks()
        circle_fit.scan_detect(v, *GATE)
        fb_v = circle_fit.last_fallbacks()
        print(f"  handed over: {fb_gate} / {int(near.sum())} tubes within 1e-6 of R = 1, {fb_v} / {len(v)} V clusters")
        assert fb_gate > 0 and fb_v > 0


@pytest.mark.gpu
@pytest.mark.parametrize("gate", GATES + WIDE_GATES, ids=lambda g: f"{g[0]}-{g[1]}")
def test_range_gate_edges(orc, fit_mode, batch, gate):
    """Gates float cannot represent (0.05, 0.12) and ones it can (1.0, 3.5), ranges within 3 ulps of them, neighbour steps within an
    ulp of 0.04; wide gates (40 m, 1e4 m) with huge, infinite and NaN ranges (the moment route's big_gate branch)."""
    lo, hi = gate
    special = wide_gate_scans(hi) if lo == 0.0 else gate_edge_scans(lo, hi)
    r, pos = batches(special, batch)
    got, want, worst = run(orc, r, lo, hi)
    print(f"[gate {lo}..{hi} fit={fit_mode} {batch}] {len(r)} scans, {int(want['n_clusters'][pos].sum())} clusters, worst rel {worst:.2e}")


@pytest.mark.gpu
def test_unaligned_and_host_buffers(orc, fit_mode, batch):
    """Ranges at a 4-byte offset (the moment route's scalar loads), cluster_of_beam at a 2-byte offset (its element-wise stores),
    no cluster_of_beam, and host memory: each equal to the aligned device call bit for bit."""
    import torch
    from shermbot_navigation_b200 import circle_fit, nuslam
    special = np.concatenate([arc_scans(1e-3)[0][:40], crowded_scans(), tube_scans(1e-3)[:40], v_scans(orc.kind)])
    r, pos = batches(special, batch)
    S = len(r)
    kmax = 16
    ref = _np(circle_fit.scan_detect(torch.tensor(r, device="cuda"), *GATE, max_circles=kmax))
    compare_scans(ref, orc.scan_detect_batch(r, *GATE, kmax=kmax, nthreads=0))
    # ranges: a contiguous slice of a larger tensor, 4 bytes past a 16-byte boundary
    big = torch.zeros(S * BEAMS + 4, dtype=torch.float32, device="cuda")
    big[1:1 + S * BEAMS] = torch.tensor(r.reshape(-1), device="cuda")
    r_off = big[1:1 + S * BEAMS].view(S, BEAMS)
    assert r_off.data_ptr() % 16 == 4 and r_off.is_contiguous()
    same_bits(_np(circle_fit.scan_detect(r_off, *GATE, max_circles=kmax)), ref, ref)
    # cluster_of_beam 2 bytes past an 8-byte boundary, through the C entry point on device pointers; the guard words stay untouched
    dev = torch.device("cuda")
    cob_buf = torch.full((S * BEAMS + 8,), 0x5A5A, dtype=torch.int16, device=dev)
    ncl = torch.empty(S, dtype=torch.int32, device=dev)
    nci = torch.empty(S, dtype=torch.int32, device=dev)
    circ = torch.zeros((S, kmax, 4), dtype=torch.float64, device=dev)
    rd = torch.tensor(r, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    nuslam._check(circle_fit.lib().nuslam_scan_detect(rd.data_ptr(), S, GATE[0], GATE[1], cob_buf.data_ptr() + 2, ncl.data_ptr(),
                                                      nci.data_ptr(), circ.data_ptr(), kmax, nuslam.NUSLAM_DEVICE, dev.index or 0, st),
                  "nuslam_scan_detect")
    torch.cuda.synchronize()
    cb = cob_buf.cpu().numpy()
    assert (cb[0] == 0x5A5A) and (cb[1 + S * BEAMS:] == 0x5A5A).all()
    same_bits(dict(cluster_of_beam=cb[1:1 + S * BEAMS].reshape(S, BEAMS), n_clusters=ncl.cpu().numpy(), n_circles=nci.cpu().numpy(),
                   circles=circ.cpu().numpy()), ref, ref)
    # no cluster_of_beam
    nob = _np(circle_fit.scan_detect(torch.tensor(r, device="cuda"), *GATE, max_circles=kmax, want_cluster_of_beam=False))
    assert nob["cluster_of_beam"] is None
    same_bits(nob, ref, ref)
    # host memory
    same_bits(circle_fit.scan_detect(r, *GATE, max_circles=kmax), ref, ref)


@pytest.mark.gpu
def test_chunk_boundary(orc, fit_mode):
    """kScanChunk + 300 scans: tiles of 4096 scenario scans with the special scans at both sides of the chunk boundary (262143,
    262144) and at the end. Every tile must equal the first bit for bit, and the first tile and the special scans the oracle."""
    import torch
    from shermbot_navigation_b200 import circle_fit
    base = scenario()
    special = np.concatenate([arc_scans(0.0)[0][::9], crowded_scans()[::3], gate_tube_scans()[0][::4], v_scans(orc.kind)[:4]])
    m = len(special)
    S = SCAN_CHUNK + 300
    rows = np.arange(S) % len(base)
    r = base[rows]
    h = m // 2
    at = np.concatenate([SCAN_CHUNK - h + np.arange(h), SCAN_CHUNK + np.arange(m - h - 3), S - 3 + np.arange(3)])
    assert SCAN_CHUNK - 1 in at and SCAN_CHUNK in at and S - 1 in at and len(at) == m
    r[at] = special
    got = circle_fit.scan_detect(torch.tensor(r, device="cuda"), *GATE)
    torch.cuda.synchronize()
    del r
    g = _np(got)
    twin = np.ones(S, dtype=bool)
    twin[at] = False
    twin[: len(base)] = False
    for key in ("cluster_of_beam", "n_clusters", "n_circles"):
        assert np.array_equal(g[key][twin], g[key][rows[twin]]), key
    assert np.array_equal(g["circles"][twin], g["circles"][rows[twin]], equal_nan=True)
    first = {k: v[: len(base)] for k, v in g.items()}
    compare_scans(first, orc.scan_detect_batch(base, *GATE, nthreads=0))
    sp = {k: v[at] for k, v in g.items()}
    want = orc.scan_detect_batch(special, *GATE, nthreads=0)
    worst = compare_scans(sp, want)
    print(f"[chunk boundary fit={fit_mode}] {S} scans, {m} special scans at {at[0]}..{at[m - 4]} and the last 3, worst rel {worst:.2e}")
