"""NUSLAM_OPT_NEAREST_NEIGHBOUR: associateLandmark by individual-compatibility nearest neighbour, in the oracle-order kernels (STRICT,
FAST with options set, the large-map tail) and in large-map mode (per-CTA (d, k) minima, then a scan of the slots). Checked against a
numpy restatement of the rule (NnEkf below, on top of tests/sane_reference.py), between modes, between the fused and the unfused scan
step, and on hand-built states for ties, full maps and singular candidates. Tolerances as in test_options_gpu.py: ids exactly equal,
x / Sigma within 1e-9 relative."""
import numpy as np
import pytest

from sane_reference import JOSEPH, PRE_MOTION, WRAP, SaneEkf
from shermbot_navigation_b200 import synth, tube_world
from test_large_options_gpu import picked
from test_large_scan_gpu import ranges_of, ring_run, ring_tubes, touched

pytestmark = pytest.mark.gpu
TOL = 1e-9
NN = 8
MAP_FULL, SINGULAR = 1, 2
ID_EXCEPTION = -1000
CHI2 = (9.21, 60.0)   # 99 % gate at 2 dof, new-landmark threshold
DEFAULT = (0.01, 60.0)


def rel(a, b):
    return np.abs(a - b).max() / max(np.abs(a).max(), np.abs(b).max(), 1e-300)


class Thrown(Exception):
    def __init__(self, bit):
        self.bit = bit


class NnEkf(SaneEkf):
    """SaneEkf with the nearest-neighbour rule, and the engine's status contract where the reference would throw: the measurement gets
    ID_EXCEPTION, the rest of the scan 0, and the filter stays frozen from then on."""
    status = 0

    def associate(self, z):
        if self.seen == 0:
            self.seen = 1
            return 1
        best, kbest = 0.0, 0
        for k in range(1, self.seen + 1):
            zhat, H = self.model(k)
            psi = H @ self.S @ H.T + self.R
            if psi[0, 0] * psi[1, 1] - psi[0, 1] * psi[1, 0] == 0.0:
                raise Thrown(SINGULAR)
            dz = self.innovation(z, zhat)
            d = float(dz @ np.linalg.inv(psi) @ dz)
            if d == d and (kbest == 0 or d < best):
                best, kbest = d, k
        if kbest and best < self.amin:
            return kbest
        if kbest and best < self.amax:
            return -1
        if 3 + 2 * self.seen >= self.len:
            raise Thrown(MAP_FULL)
        self.seen += 1
        return self.seen

    def step(self, tw, zs, ids=None):
        if self.status:
            return [0] * len(zs)
        snapshot = self.seen
        self.predict(tw[0], tw[1])
        out = []
        for i, z in enumerate(zs):
            try:
                j = self.associate(z)
            except Thrown as e:
                self.status |= e.bit
                return out + [ID_EXCEPTION] + [0] * (len(zs) - i - 1)
            out.append(j)
            if j > snapshot:
                self.init_landmark(z, j)
            elif j < 0:
                continue
            self.update(z, j)
        return out


def engine(cuda_lib, robot, n, options, thresholds, mode=None, Q=synth.Q_DEFAULT, R=synth.R_DEFAULT, prior=100.0):
    kw = {} if mode is None else {"mode": mode}
    return cuda_lib.BatchedExtendedKalman(robot, n_landmarks=n, Q=Q, R=R, options=options, assoc_min=thresholds[0], assoc_max=thresholds[1],
                                          landmark_prior=prior, **kw)


def run_numpy(cuda_lib, sc, z, options, thresholds, mode=None):
    """Unknown ids from scratch on the engine and on NnEkf; returns (ids engine, ids numpy, engine state, numpy filters)."""
    T, B = z.shape[:2]
    eng = engine(cuda_lib, sc["robot0"][:B], sc["n"], options, thresholds, mode)
    refs = [NnEkf(sc["n"], sc["robot0"][b], sc["Q"], sc["R"], prior=100.0, options=options, amin=thresholds[0], amax=thresholds[1])
            for b in range(B)]
    got, want = [], []
    for t in range(T):
        got.append(eng.step(sc["twists"][t, :B], z[t], None, return_ids=True))
        want.append([f.step(sc["twists"][t, b], z[t, b]) for b, f in enumerate(refs)])
    state = eng.get_state()
    eng.close()
    return np.stack(got), np.array(want, dtype=np.int32), state, refs


def check_against_numpy(state, refs, ids, ids_np, tag):
    x, s, seen, status = state
    assert np.array_equal(ids, ids_np), tag
    assert np.array_equal(seen, [f.seen for f in refs]) and np.array_equal(status, [f.status for f in refs]), tag
    ex = max(rel(x[b], refs[b].x) for b in range(len(refs)))
    es = max(rel(s[b][np.ix_(touched(seen[b]), touched(seen[b]))], refs[b].S[np.ix_(touched(seen[b]), touched(seen[b]))]) for b in range(len(refs)))
    print(f"[{tag}] matched {(ids > 0).sum()}, ambiguous {(ids == -1).sum()}, seen {seen.tolist()}, status {status.tolist()}: "
          f"x rel {ex:.2e}, Sigma rel {es:.2e}")
    assert ex < TOL and es < TOL, tag


@pytest.mark.parametrize("options", [NN, NN | WRAP, NN | WRAP | JOSEPH | PRE_MOTION])
@pytest.mark.parametrize("thresholds", [DEFAULT, CHI2])
@pytest.mark.parametrize("geometry", ["benign", "adversarial"])
def test_nn_strict_matches_numpy_and_fast_equals_strict(cuda_lib, options, thresholds, geometry):
    """n = 12, unknown ids from scratch: STRICT against the numpy rule; a FAST handle with the same options runs the same kernels."""
    B, T, n = 6, 20, 12
    sc = synth.ekf_scenario(B, T, n=n, seed=7, geometry=geometry, shuffle_order=True)
    ids, ids_np, state, refs = run_numpy(cuda_lib, sc, sc["z"], options, thresholds, mode="strict")
    check_against_numpy(state, refs, ids, ids_np, f"strict opt {options} {thresholds} {geometry}")
    ids_f, _, state_f, _ = run_numpy(cuda_lib, sc, sc["z"], options, thresholds, mode="fast")
    assert np.array_equal(ids_f, ids)
    for u, v in zip(state_f, state):
        assert np.array_equal(u, v)


def landmark_state(n, lm, robot=(0.1, 0.05, -0.02), seen=None, var=1e-3, robot_var=1e-4):
    """One filter's x / Sigma ([row, col]) with landmarks lm (k x 2) in slots 1..k, diagonal Sigma."""
    length = 3 + 2 * n
    x = np.zeros(length)
    x[:3] = robot
    x[3:3 + 2 * len(lm)] = np.asarray(lm, dtype=np.float64).ravel()
    s = np.diag(np.full(length, var))
    s[:3, :3] = robot_var * np.eye(3)
    return x, s, len(lm) if seen is None else seen


def polar(x, p):
    dx, dy = p[0] - x[1], p[1] - x[2]
    return np.array([np.hypot(dx, dy), synth.wrap_pi(np.arctan2(dy, dx) - x[0])])


def set_states(eng, states, status=None):
    x = np.stack([s[0] for s in states])
    s = np.stack([s[1] for s in states])
    seen = np.array([s[2] for s in states], dtype=np.int32)
    eng.set_state(x, s, seen, np.zeros(len(states), np.int32) if status is None else np.asarray(status, np.int32))


@pytest.mark.parametrize("mode,n,pairs", [("strict", 40, [(3, 35), (7, 8)]), ("large", 160, [(3, 140), (7, 8)])])
def test_nn_ties_go_to_the_lower_id(cuda_lib, mode, n, pairs):
    """Two landmarks at identical coordinates with identical Sigma blocks have bit-equal distances: the lower id wins, in the single
    call and in the step, whether the pair shares a warp chunk / CTA or not. Landmark 1 lies at an ambiguous distance (under the
    reference's rule it would decide first)."""
    zero = np.zeros((len(pairs), 3))
    states, zs = [], []
    rng = np.random.default_rng(3)
    for lo, hi in pairs:
        lm = rng.uniform(-2, 2, size=(hi, 2))
        lm[hi - 1] = lm[lo - 1]
        x, s, seen = landmark_state(n, lm)
        z = polar(x, lm[lo - 1])
        # landmark 1 on the same bearing, farther by 0.3 sigma-units of range too many for a match: d between the thresholds
        lm1 = lm[lo - 1] + 0.17 * (lm[lo - 1] - x[1:3]) / np.linalg.norm(lm[lo - 1] - x[1:3])
        x[3:5] = lm1
        states.append((x, s, seen))
        zs.append(z)
    zs = np.array(zs)
    for opts in (NN, NN | WRAP):
        eng = engine(cuda_lib, zero, n, opts, CHI2, mode=mode, Q=1e-6 * np.eye(3))
        set_states(eng, states)
        assert list(eng.associateLandmark(zs)) == [lo for lo, _ in pairs]
        ref = engine(cuda_lib, zero, n, 0, CHI2, mode=mode, Q=1e-6 * np.eye(3))
        set_states(ref, states)
        assert list(ref.associateLandmark(zs)) == [-1] * len(pairs), "landmark 1 is ambiguous: the reference's rule stops there"
        ids = eng.step(np.zeros((len(pairs), 3)), zs[:, None], None, return_ids=True)
        assert list(ids[:, 0]) == [lo for lo, _ in pairs]
        _, _, seen, status = eng.get_state()
        assert not status.any() and np.array_equal(seen, [s[2] for s in states])
        eng.close()
        ref.close()


@pytest.mark.parametrize("mode", ["strict", "large"])
def test_nn_full_map(cuda_lib, mode):
    """seen == n: a measurement of a known landmark matches and updates; a far one flags MAP_FULL, gets ID_EXCEPTION and freezes the
    filter (the next step changes nothing). Single call and step."""
    n = 12
    a = 2 * np.pi * np.arange(n) / n
    lm = 1.5 * np.stack([np.cos(a), np.sin(a)], axis=1)
    x, s, seen = landmark_state(n, lm)
    zk = polar(x, lm[4]) + np.array([0.01, -0.005])
    zfar = np.array([6.0, 0.3])
    z = np.array([zk, zfar])
    zero = np.zeros((2, 3))
    for opts in (NN, NN | WRAP):
        eng = engine(cuda_lib, zero, n, opts, CHI2, mode=mode)
        set_states(eng, [(x, s, seen)] * 2)
        assert list(eng.associateLandmark(z)) == [5, ID_EXCEPTION]
        _, _, sn, st = eng.get_state()
        assert list(st) == [0, MAP_FULL] and list(sn) == [n, n]
        set_states(eng, [(x, s, seen)] * 2)
        tw = np.tile([0.01, 0.02, 0.0], (2, 1))
        # filter 0: the known landmark, then the far one; filter 1: the far one first, then the known one (never reached)
        ids = eng.step(tw, np.array([[zk, zfar], [zfar, zk]]), None, return_ids=True)
        assert ids.tolist() == [[5, ID_EXCEPTION], [ID_EXCEPTION, 0]]
        x1, s1, sn, st = eng.get_state()
        assert list(st) == [MAP_FULL, MAP_FULL] and list(sn) == [n, n]
        ref = NnEkf(n, x[:3], synth.Q_DEFAULT, synth.R_DEFAULT, options=opts, amin=CHI2[0], amax=CHI2[1])
        ref.x, ref.S, ref.seen = x.copy(), s.copy(), seen
        assert ref.step(tw[0], [zk, zfar]) == [5, ID_EXCEPTION]
        assert rel(x1[0], ref.x) < TOL and rel(s1[0], ref.S) < TOL, "the match before the exception was applied"
        assert abs(x1[0][3 + 8] - x[3 + 8]) > 0
        ids = eng.step(tw, z[None].repeat(2, axis=0), None, return_ids=True)
        assert not ids.any()
        x2, s2, _, _ = eng.get_state()
        assert np.array_equal(x2, x1) and np.array_equal(s2, s1), "a filter flagged MAP_FULL stays frozen"
        eng.close()


@pytest.mark.parametrize("mode", ["strict", "large"])
def test_nn_singular_candidate(cuda_lib, mode):
    """R = 0, Q = 0, a zero robot block and a zero Sigma block at landmark 2: psi of candidate 2 is singular. The nearest-neighbour rule
    reaches it even when candidate 1 matches exactly (the reference's rule stops at 1), so SINGULAR and the exception. The single call
    still associates a filter that is already flagged."""
    n = 12
    lm = np.array([[1.0, 0.2], [0.3, 1.1], [-0.8, 0.4]])
    x, s, seen = landmark_state(n, lm)
    s[:3, :3] = 0.0
    s[5:7, 5:7] = 0.0
    ok = landmark_state(n, lm)
    z = np.array([polar(x, lm[0]), polar(ok[0], lm[2])])
    zero = np.zeros((2, 3))
    Q, R = np.zeros((3, 3)), np.zeros((2, 2))
    eng = engine(cuda_lib, zero, n, NN | WRAP, CHI2, mode=mode, Q=Q, R=R)
    ref = engine(cuda_lib, zero, n, 0, CHI2, mode=mode, Q=Q, R=R)
    for e in (eng, ref):
        set_states(e, [(x, s, seen), ok], status=[0, SINGULAR])
    assert list(ref.associateLandmark(z)) == [1, 3]
    assert list(eng.associateLandmark(z)) == [ID_EXCEPTION, 3], "filter 1 is flagged already and still associates"
    assert list(eng.get_state()[3]) == [SINGULAR, SINGULAR]
    set_states(eng, [(x, s, seen), ok])
    ids = eng.step(zero, z[:, None], None, return_ids=True)
    assert list(ids[:, 0]) == [ID_EXCEPTION, 3]
    assert list(eng.get_state()[3]) == [SINGULAR, 0]
    eng.close()
    ref.close()


@pytest.mark.parametrize("geometry", ["benign", "adversarial"])
def test_nn_large_matches_numpy(cuda_lib, geometry):
    """n = 96 (large-map mode chosen by the engine), 20 measurements per step (two passes), from scratch: first touches and new landmarks
    go through the oracle-order tail, which must apply the nearest-neighbour rule too."""
    B, T, n = 3, 8, 96
    sc = synth.ekf_scenario(B, T, n=n, seed=41, geometry=geometry, shuffle_order=True)
    z, _ = picked(sc, np.linspace(1, n, 20).astype(np.int32))
    opts = NN | WRAP | JOSEPH
    ids, ids_np, state, refs = run_numpy(cuda_lib, sc, z, opts, CHI2)
    check_against_numpy(state, refs, ids, ids_np, f"large opt {opts} {geometry}")
    assert (ids[1:] > 0).sum() > 0


@pytest.mark.parametrize("options", [NN | WRAP, NN | WRAP | JOSEPH | PRE_MOTION])
def test_nn_large_equals_strict(cuda_lib, options):
    """n = 40 on a large-map handle and on a STRICT handle, from scratch (new landmarks through the oracle-order tail): ids identical,
    states within 1e-9. Finite prior: with INT_MAX and no JOSEPH the first touch leaves Sigma asymmetric at 1e-6 and the delayed
    form's rounding is amplified past 1e-9 (whatever the association rule)."""
    B, T, n = 4, 6, 40
    sc = synth.ekf_scenario(B, T, n=n, seed=62, geometry="adversarial", shuffle_order=True)
    out = {}
    for mode in ("large", "strict"):
        eng = engine(cuda_lib, sc["robot0"], n, options, CHI2, mode=mode)
        ids = np.stack([eng.step(sc["twists"][t], sc["z"][t], None, return_ids=True) for t in range(T)])
        out[mode] = (ids,) + eng.get_state()
        eng.close()
    (il, xl, sl, nl, stl), (is_, xs, ss, ns, sts) = out["large"], out["strict"]
    assert np.array_equal(il, is_) and np.array_equal(nl, ns) and np.array_equal(stl, sts)
    es = max(rel(sl[b][np.ix_(touched(ns[b]), touched(ns[b]))], ss[b][np.ix_(touched(ns[b]), touched(ns[b]))]) for b in range(B))
    print(f"[large == strict NN, options {options}] seen {ns.tolist()}, status {sts.tolist()}: x rel {rel(xl, xs):.2e}, Sigma rel {es:.2e}")
    assert rel(xl, xs) < TOL and es < TOL
    assert all((il[:, b] > 0).sum() > ns[b] for b in range(B)), "some measurements matched a landmark opened before"


def test_nn_4096_built_map(cuda_lib):
    """A built 4 096-landmark map (tubes on a 0.6 m grid, 4 000 seen), NN | WRAP at 9.21 / 60: every marker of the fused scan step
    matches the tube it came from, and the single call on a second handle (predict, then associateLandmark / update marker by marker)
    returns the same ids."""
    import torch
    from shermbot_navigation_b200 import circle_fit
    n, seen_n, spacing, T = 4096, 4000, 0.6, 4
    dev = torch.device("cuda")
    side = int(np.ceil(np.sqrt(seen_n)))
    gx, gy = np.meshgrid(np.arange(side) * spacing, np.arange(side) * spacing)
    lm = (np.stack([gx.ravel(), gy.ravel()], axis=1)[:seen_n] - spacing * (side - 1) / 2).copy()
    tw = np.tile(np.array([0.002, 0.005, 0.0]), (T, 1))
    tw[0] = 0.0
    poses = [np.array([0.3, 0.01, -0.02])]
    for t in range(1, T):
        th, px, py = poses[-1]
        q, th1 = tw[t, 1] / tw[t, 0], th + tw[t, 0]
        poses.append(np.array([th1, px - q * np.sin(th) + q * np.sin(th1), py + q * np.cos(th) - q * np.cos(th1)]))
    length = 3 + 2 * n
    g = np.random.default_rng(5)
    x0 = torch.zeros((1, length), dtype=torch.float64, device=dev)
    x0[0, :3] = torch.tensor(poses[0], device=dev)
    x0[0, 3:3 + 2 * seen_n] = torch.tensor((lm + g.normal(0, 1e-4, lm.shape)).ravel(), device=dev)
    Q, R = 1e-8 * np.eye(3), 1e-3 * np.eye(2)
    engs, states = [], []
    for _ in range(2):
        e = cuda_lib.BatchedExtendedKalman(poses[0][None], n_landmarks=n, Q=Q, R=R, options=NN | WRAP, assoc_min=CHI2[0], assoc_max=CHI2[1],
                                           stream=torch.cuda.current_stream(dev).cuda_stream)
        sig = torch.zeros((1, length, length), dtype=torch.float64, device=dev)
        d = torch.full((length,), 1e-4, dtype=torch.float64, device=dev)
        d[:3] = 1e-6
        sig[0].diagonal().copy_(d)
        st = (x0.clone(), sig, torch.full((1,), seen_n, dtype=torch.int32, device=dev), torch.zeros(1, dtype=torch.int32, device=dev))
        e.bind_state(*st)
        engs.append(e)
        states.append(st)
    fused, single = engs
    markers = 0
    for t in range(T):
        ranges = synth.simulate_scans(poses[t][None], lm[np.hypot(lm[:, 0] - poses[t][1], lm[:, 1] - poses[t][2]) < 1.2])
        det = circle_fit.scan_detect(ranges, tube_world.MIN_RANGE, tube_world.MAX_RANGE, max_circles=16, want_cluster_of_beam=False)
        cnt = int(det["n_circles"][0])
        assert 1 <= cnt <= 16
        nm, z, ids = fused.scan_step(torch.tensor(tw[t:t + 1], device=dev), torch.tensor(ranges, device=dev), tube_world.MIN_RANGE,
                                     tube_world.MAX_RANGE, 16, return_all=True)
        ids = ids.cpu().numpy()[0]
        th, px, py = poses[t]
        for i in range(cnt):
            cx, cy = det["circles"][0, i, 0], det["circles"][0, i, 1]
            wx, wy = px + np.cos(th) * cx - np.sin(th) * cy, py + np.sin(th) * cx + np.cos(th) * cy
            assert ids[i] == int(np.argmin(np.hypot(lm[:, 0] - wx, lm[:, 1] - wy))) + 1, (t, i)
        assert not ids[cnt:].any()
        single.predict(torch.tensor(tw[t:t + 1], device=dev))
        for i in range(cnt):
            zi = z[:, i].contiguous()
            got = single.associateLandmark(zi)
            assert int(got[0]) == ids[i], (t, i)
            single.update(zi, got)
        markers += cnt
    torch.cuda.synchronize()
    assert int(states[0][3][0]) == 0 and int(states[1][3][0]) == 0 and int(states[0][2][0]) == seen_n
    ex = float((states[0][0] - states[1][0]).abs().max() / states[1][0].abs().max())
    print(f"[NN 4096] {markers} markers over {T} scans all matched their tube; fused vs single-call state x rel {ex:.2e}")
    assert ex < 1e-9
    for e in engs:
        e.close()


@pytest.mark.parametrize("mode,n", [("strict", 40), ("large", 96)])
def test_nn_scan_step_bit_identical(cuda_lib, mode, n):
    """The fused scan step with NN | WRAP equals detect -> cartesian2polar -> step(ids = None) bit for bit at ragged marker counts; each
    filter's unfused step runs on a one-filter handle with its own count."""
    from shermbot_navigation_b200 import circle_fit
    counts = [(0, 0), (5, 0), (10, 8), (13, 13)]
    B, T, m = len(counts), 4, 20
    tubes = ring_tubes(counts, [0.05, 0.05, 0.05, 0.3])
    poses, tw = ring_run(T, B)
    Q = 1e-4 * np.eye(3)
    fused = engine(cuda_lib, poses[0], n, NN | WRAP, CHI2, mode=mode, Q=Q, prior=None)
    plain = [engine(cuda_lib, poses[0][b:b + 1], n, NN | WRAP, CHI2, mode=mode, Q=Q, prior=None) for b in range(B)]
    matched = 0
    for t in range(T):
        ranges = ranges_of(poses[t], tubes)
        seen0 = fused.getSeenLandmarks()
        nm, z, ids = fused.scan_step(tw[t], ranges, tube_world.MIN_RANGE, tube_world.MAX_RANGE, m, return_all=True)
        det = circle_fit.scan_detect(ranges, tube_world.MIN_RANGE, tube_world.MAX_RANGE, max_circles=m, want_cluster_of_beam=False)
        assert np.array_equal(nm, det["n_circles"]), t
        mv = np.clip(nm, 0, m)
        for b in range(B):
            if mv[b] == 0:
                plain[b].predict(tw[t][b:b + 1])
                assert not ids[b].any(), (t, b)
            else:
                z2 = cuda_lib.cartesian2polar(np.ascontiguousarray(det["circles"][b, :mv[b], :2])).reshape(1, mv[b], 2)
                ids2 = plain[b].step(tw[t][b:b + 1], z2, None, return_ids=True)
                assert np.array_equal(z[b, :mv[b]], z2[0]), (t, b)
                assert np.array_equal(ids[b, :mv[b]], ids2[0]) and not ids[b, mv[b]:].any(), (t, b)
        for b in range(B):
            for u, v in zip(fused.get_state(), plain[b].get_state()):
                assert np.array_equal(u[b], v[0]), (t, b)
        matched += int(((ids > 0) & (ids <= seen0[:, None])).sum())
    print(f"[NN scan step {mode}] seen {fused.getSeenLandmarks().tolist()}, status {fused.getStatus().tolist()}")
    assert matched > 0
    for e in [fused] + plain:
        e.close()


def test_default_handles_unaffected_and_unknown_bits_refused(cuda_lib):
    """Default (options 0) FAST, STRICT and large-map handles compute the same bits before and after NN handles ran in the same process;
    an option bit beyond NEAREST_NEIGHBOUR is still refused."""
    from shermbot_navigation_b200 import nuslam
    B, T = 4, 6
    sc12 = synth.ekf_scenario(B, T, n=12, seed=9, geometry="adversarial", shuffle_order=True)
    sc96 = synth.ekf_scenario(B, T, n=96, seed=9, geometry="adversarial", shuffle_order=True)
    z96, _ = picked(sc96, np.linspace(1, 96, 20).astype(np.int32))

    def run(options):
        out = []
        for mode, sc, z in (("fast", sc12, sc12["z"]), ("strict", sc12, sc12["z"]), (None, sc96, z96)):
            kw = {} if mode is None else {"mode": mode}
            eng = cuda_lib.BatchedExtendedKalman(sc["robot0"], n_landmarks=sc["n"], Q=sc["Q"], R=sc["R"], options=options, **kw)
            ids = [eng.step(sc["twists"][t], z[t], None, return_ids=True) for t in range(T)]
            out.append((np.stack(ids),) + eng.get_state())
            eng.close()
        return out

    before = run(0)
    for options in (NN, NN | WRAP | JOSEPH | PRE_MOTION):
        run(options)
    after = run(0)
    for a, b in zip(before, after):
        for u, v in zip(a, b):
            assert np.array_equal(u, v)
    with pytest.raises(nuslam.NuslamError, match=r"code 1\)"):
        cuda_lib.BatchedExtendedKalman(np.zeros((1, 3)), n_landmarks=12, options=16)
    assert nuslam.OPT_NEAREST_NEIGHBOUR == NN
