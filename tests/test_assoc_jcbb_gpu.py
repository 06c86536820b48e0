"""NUSLAM_OPT_JOINT_COMPATIBILITY: a step's measurements associated by joint compatibility branch and bound in the oracle-order kernels
(STRICT, and FAST handles with options, which run the same kernels). Checked against a dense numpy restatement of the rule (JcbbEkf
below, on top of tests/sane_reference.py: the joint S built whole and factored by np.linalg.cholesky, the search order, tie rules,
pruning and test budget of include/nuslam_b200.h), against nearest neighbour where the two rules coincide (one measurement), and on
hand-built states: a pose error that nearest neighbour cannot see, the joint threshold, the budget, singular candidates and full maps.
Tolerances as in test_assoc_nn_gpu.py: ids and status exactly equal, x / Sigma within 1e-9 relative."""
import math

import numpy as np
import pytest
from scipy.stats import chi2

from sane_reference import JOSEPH, PRE_MOTION, WRAP
from shermbot_navigation_b200 import synth, tube_world
from test_assoc_nn_gpu import (CHI2, ID_EXCEPTION, MAP_FULL, NN, SINGULAR, TOL, NnEkf, Thrown, check_against_numpy, engine, landmark_state,
                               polar, rel, set_states)
from test_large_options_gpu import picked
from test_large_scan_gpu import ranges_of, ring_run, ring_tubes

pytestmark = pytest.mark.gpu
JC = 32
TRUNCATED = 8
MAX_TESTS = 4096
GATE_95 = (5.99, 60.0)


def joint_thresholds(amin):
    """T[p] = chi2_{2p}^-1(1 - exp(-amin / 2)), T[1] = amin."""
    conf = -math.expm1(-0.5 * amin)
    return [0.0, amin] + [float(chi2.ppf(conf, 2 * p)) for p in range(2, 17)]


class Truncated(Exception):
    pass


class JcbbEkf(NnEkf):
    """NnEkf with the steps' measurements associated jointly (the single associateLandmark call stays nearest neighbour)."""

    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        self.T = joint_thresholds(self.amin)
        self.truncated = False

    def joint_d2(self, zs, pairs, dist):
        if len(pairs) == 1:
            i, k = pairs[0]
            return dist[i][k - 1]
        Hs, nus = [], []
        for i, k in pairs:
            zhat, H = self.model(k)
            Hs.append(H)
            nus.append(self.innovation(zs[i], zhat))
        H, nu = np.vstack(Hs), np.concatenate(nus)
        S = H @ self.S @ H.T + np.kron(np.eye(len(pairs)), self.R)
        try:
            L = np.linalg.cholesky(S)
        except np.linalg.LinAlgError:
            return math.nan
        y = np.linalg.solve(L, nu)
        return float(y @ y)

    def associate_joint(self, zs):
        m, seen0 = len(zs), self.seen
        dist = [[0.0] * seen0 for _ in range(m)]
        for i in range(m):
            for k in range(1, seen0 + 1):
                zhat, H = self.model(k)
                psi = H @ self.S @ H.T + self.R
                if psi[0, 0] * psi[1, 1] - psi[0, 1] * psi[1, 0] == 0.0:
                    raise Thrown(SINGULAR)
                dz = self.innovation(zs[i], zhat)
                dist[i][k - 1] = float(dz @ np.linalg.inv(psi) @ dz)
        cand = [sorted((k for k in range(1, seen0 + 1) if dist[i][k - 1] < self.amin), key=lambda k: (dist[i][k - 1], k)) for i in range(m)]
        best = {"p": 0, "d2": 0.0, "hyp": [0] * m}
        hyp = [0] * m
        self.tests = 0

        def node(i, pairs, d2):
            if len(pairs) + (m - i) < best["p"]:
                return
            if i == m:
                if len(pairs) > best["p"] or (len(pairs) == best["p"] and d2 < best["d2"]):
                    best.update(p=len(pairs), d2=d2, hyp=list(hyp))
                return
            used = {k for _, k in pairs}
            for k in cand[i]:
                if k in used:
                    continue
                if self.tests == MAX_TESTS:
                    raise Truncated
                self.tests += 1
                t = self.joint_d2(zs, pairs + [(i, k)], dist)
                if t < self.T[len(pairs) + 1]:
                    hyp[i] = k
                    node(i + 1, pairs + [(i, k)], t)
            hyp[i] = 0
            node(i + 1, pairs, d2)

        if m and seen0:
            try:
                node(0, [], 0.0)
            except Truncated:
                self.status |= TRUNCATED
        out = []
        for r in range(m):
            if best["hyp"][r]:
                out.append(best["hyp"][r])
            elif any(d < self.amax for d in dist[r]):
                out.append(-1)
            elif self.seen >= self.n:
                self.status |= MAP_FULL
                return out + [ID_EXCEPTION] + [0] * (m - r - 1)
            else:
                self.seen += 1
                out.append(self.seen)
        return out

    def step(self, tw, zs, ids=None):
        if self.status & (MAP_FULL | SINGULAR):
            return [0] * len(zs)
        snapshot = self.seen
        self.predict(tw[0], tw[1])
        try:
            jids = self.associate_joint(list(zs))
        except Thrown as e:
            self.status |= e.bit
            return [ID_EXCEPTION] + [0] * (len(zs) - 1)
        out = []
        for i, (z, j) in enumerate(zip(zs, jids)):
            out.append(j)
            if j == ID_EXCEPTION:
                return out + [0] * (len(zs) - i - 1)
            if j > snapshot:
                self.init_landmark(z, j)
            elif j < 0:
                continue
            self.update(z, j)
        return out


def run_joint(cuda_lib, sc, z, options, thresholds, mode):
    T, B = z.shape[:2]
    eng = engine(cuda_lib, sc["robot0"][:B], sc["n"], options, thresholds, mode)
    refs = [JcbbEkf(sc["n"], sc["robot0"][b], sc["Q"], sc["R"], prior=100.0, options=options, amin=thresholds[0], amax=thresholds[1])
            for b in range(B)]
    got, want = [], []
    for t in range(T):
        got.append(eng.step(sc["twists"][t, :B], z[t], None, return_ids=True))
        want.append([f.step(sc["twists"][t, b], z[t, b]) for b, f in enumerate(refs)])
    state = eng.get_state()
    eng.close()
    return np.stack(got), np.array(want, dtype=np.int32), state, refs


@pytest.mark.parametrize("options", [JC | WRAP, JC | WRAP | JOSEPH | PRE_MOTION])
@pytest.mark.parametrize("thresholds", [CHI2, GATE_95])
@pytest.mark.parametrize("geometry", ["benign", "adversarial"])
def test_jcbb_matches_numpy_and_fast_equals_strict(cuda_lib, options, thresholds, geometry):
    """16 filters x 20 steps of 12 measurements, unknown ids from scratch: STRICT against the numpy rule; a FAST handle with the same
    options gives the same bits."""
    B, T, n = 16, 20, 12
    sc = synth.ekf_scenario(B, T, n=n, seed=11, geometry=geometry, shuffle_order=True)
    ids, ids_np, state, refs = run_joint(cuda_lib, sc, sc["z"], options, thresholds, "strict")
    check_against_numpy(state, refs, ids, ids_np, f"jcbb opt {options} {thresholds} {geometry}")
    assert (ids[1:] > 0).sum() > 0
    ids_f, _, state_f, _ = run_joint(cuda_lib, sc, sc["z"], options, thresholds, "fast")
    assert np.array_equal(ids_f, ids)
    for u, v in zip(state_f, state):
        assert np.array_equal(u, v)


@pytest.mark.parametrize("geometry", ["benign", "adversarial"])
def test_jcbb_one_measurement_is_nearest_neighbour(cuda_lib, geometry):
    """Steps with m = 1 and single associateLandmark calls on a JOINT handle give the bits of a NEAREST_NEIGHBOUR handle."""
    B, T, n = 16, 30, 12
    sc = synth.ekf_scenario(B, T, n=n, seed=5, geometry=geometry, shuffle_order=True)
    outs = []
    for opts in (JC | WRAP, NN | WRAP):
        eng = engine(cuda_lib, sc["robot0"], n, opts, CHI2, "strict")
        ids = [eng.step(sc["twists"][t], sc["z"][t][:, :1], None, return_ids=True) for t in range(T)]
        single = [eng.associateLandmark(np.ascontiguousarray(sc["z"][t][:, 1])) for t in range(3)]
        outs.append((np.stack(ids), np.stack(single)) + eng.get_state())
        eng.close()
    for u, v in zip(*outs):
        assert np.array_equal(u, v)
    assert (outs[0][0] > 0).sum() > 0


def row_state(shift):
    """Five landmarks 0.3 m apart on a row 2 m ahead, the robot's lateral position uncertain (sigma 0.2 m), measured from a pose shifted
    by `shift` along the row, in the order of landmarks 2, 3, 4, 5, 1: each of the first four measurements lies closer to the landmark
    next to its own."""
    n = 12
    lm = np.stack([np.full(5, 2.0), 0.3 * np.arange(-2, 3)], axis=1)
    x, s, seen = landmark_state(n, lm, robot=(0.0, 0.0, 0.0), var=1e-4)
    s[:3, :3] = np.diag([1e-6, 1e-6, 0.04])
    truth = x.copy()
    truth[2] = shift
    z = np.array([polar(truth, lm[j]) for j in (1, 2, 3, 4, 0)])
    return (x, s, seen), z


def test_jcbb_beats_nearest_neighbour_on_a_common_pose_error(cuda_lib):
    """A lateral pose error of 0.2 m along a row of landmarks 0.3 m apart: nearest neighbour pairs the first measurement with the
    neighbouring landmark, its update drags the pose further off, and every later measurement follows (ids crossed by one); joint
    compatibility pairs every measurement with its own landmark, since only that hypothesis pairs all five."""
    state, z = row_state(0.2)
    zero = np.zeros((1, 3))
    got = {}
    for opts in (JC | WRAP, NN | WRAP):
        eng = engine(cuda_lib, zero, 12, opts, CHI2, mode="strict", Q=1e-12 * np.eye(3))
        set_states(eng, [state])
        got[opts] = eng.step(zero, z[None], None, return_ids=True)[0].tolist()
        assert not eng.getStatus().any()
        eng.close()
    print(f"[row] JCBB {got[JC | WRAP]}, NN {got[NN | WRAP]}")
    truth = [2, 3, 4, 5, 1]
    assert got[JC | WRAP] == truth
    assert got[NN | WRAP][:4] == [1, 2, 3, 4]
    ref = JcbbEkf(12, np.zeros(3), 1e-12 * np.eye(3), synth.R_DEFAULT, options=JC | WRAP, amin=CHI2[0], amax=CHI2[1])
    ref.x, ref.S, ref.seen = state[0].copy(), state[1].copy(), state[2]
    assert ref.step(zero[0], z) == truth


def test_jcbb_joint_threshold(cuda_lib):
    """Two landmarks with independent covariance blocks (zero robot covariance, Q = 0): the joint D^2 of the two pairings is d_1 + d_2,
    placed at T_2 (1 -+ 1e-6) with T_2 from scipy. Below it both measurements pair; above it only one pairing survives, the one with
    the smaller D^2 (measurement 2), and measurement 1 is ambiguous."""
    n, amin = 12, CHI2[0]
    T2 = joint_thresholds(amin)[2]
    lm = np.array([[1.5, 0.4], [-0.7, 1.2]])
    v, R = 1e-3, synth.R_DEFAULT
    states, zs = [], []
    for f in (1 - 1e-6, 1 + 1e-6):
        x, s, seen = landmark_state(n, lm, robot=(0.0, 0.0, 0.0), var=v)
        s[:3, :3] = 0.0
        z = []
        for j, share in ((0, 0.55), (1, 0.45)):
            zz = polar(x, lm[j])
            zz[0] += math.sqrt(share * f * T2 * (v + R[0, 0]))
            z.append(zz)
        ref = JcbbEkf(n, np.zeros(3), np.zeros((3, 3)), R, options=JC | WRAP, amin=amin, amax=CHI2[1])
        ref.x, ref.S, ref.seen = x.copy(), s.copy(), seen
        dist = [[0.0] * seen for _ in z]
        for i in range(2):
            zhat, H = ref.model(i + 1)
            dz = ref.innovation(z[i], zhat)
            dist[i][i] = float(dz @ np.linalg.inv(H @ ref.S @ H.T + R) @ dz)
        d2 = ref.joint_d2(z, [(0, 1), (1, 2)], dist)
        assert abs(d2 / (f * T2) - 1) < 1e-10 and max(dist[0][0], dist[1][1]) < amin
        states.append((x, s, seen))
        zs.append(z)
    eng = engine(cuda_lib, np.zeros((2, 3)), n, JC | WRAP, CHI2, mode="strict", Q=np.zeros((3, 3)))
    set_states(eng, states)
    ids = eng.step(np.zeros((2, 3)), np.array(zs), None, return_ids=True)
    assert ids.tolist() == [[1, 2], [-1, 2]]
    assert not eng.getStatus().any()
    eng.close()


def crowded_state(n=20, k=14, seed=4):
    """k landmarks within a few centimetres, each with a variance of 1 m^2: every measurement is compatible with every landmark, alone
    and jointly."""
    g = np.random.default_rng(seed)
    lm = np.array([2.0, 0.5]) + g.uniform(-0.03, 0.03, size=(k, 2))
    x, s, seen = landmark_state(n, lm, var=1.0)
    z = np.array([polar(x, p) + g.normal(0, 0.01, 2) for p in lm])
    return (x, s, seen), z


def test_jcbb_budget(cuda_lib):
    """12 measurements of a crowded cluster of 14 landmarks exhaust the 4 096 joint tests: ASSOC_TRUNCATED, the best hypothesis found
    so far (as numpy finds it), and the filter keeps running; the same state with 3 measurements is searched to the end."""
    state, z = crowded_state()
    tw = np.zeros((1, 3))
    Q = 1e-6 * np.eye(3)
    for m, truncated in ((12, True), (3, False)):
        eng = engine(cuda_lib, tw, 20, JC | WRAP, CHI2, mode="strict", Q=Q)
        set_states(eng, [state])
        ids = eng.step(tw, z[None, :m], None, return_ids=True)[0]
        ref = JcbbEkf(20, np.zeros(3), Q, synth.R_DEFAULT, options=JC | WRAP, amin=CHI2[0], amax=CHI2[1])
        ref.x, ref.S, ref.seen = state[0].copy(), state[1].copy(), state[2]
        want = ref.step(tw[0], z[:m])
        print(f"[budget m = {m}] ids {ids.tolist()}, numpy {want} after {ref.tests} tests, status {ref.status}")
        assert ids.tolist() == want and (ids > 0).all()
        x1, s1, seen1, st = eng.get_state()
        assert int(st[0]) == (TRUNCATED if truncated else 0) == ref.status
        assert rel(x1[0], ref.x) < TOL and rel(s1[0], ref.S) < TOL
        # a truncated filter is not frozen: the next step still updates it
        ids2 = eng.step(np.array([[0.0, 0.01, 0.0]]), z[None, :m], None, return_ids=True)[0]
        x2, _, _, st2 = eng.get_state()
        assert (ids2 > 0).all() and not np.array_equal(x2, x1) and int(st2[0]) & ~TRUNCATED == 0
        eng.close()


def test_jcbb_singular_candidate(cuda_lib):
    """R = 0, Q = 0, a zero robot block and a zero Sigma block at landmark 2: psi of candidate 2 is singular for every measurement.
    SINGULAR, the first measurement gets the exception and the others 0, no update (the prediction stands), and the filter is frozen."""
    n = 12
    lm = np.array([[1.0, 0.2], [0.3, 1.1], [-0.8, 0.4]])
    x, s, seen = landmark_state(n, lm)
    s[:3, :3] = 0.0
    s[5:7, 5:7] = 0.0
    z = np.array([polar(x, lm[0]), polar(x, lm[2])])
    zero = np.zeros((1, 3))
    eng = engine(cuda_lib, zero, n, JC | WRAP, CHI2, mode="strict", Q=np.zeros((3, 3)), R=np.zeros((2, 2)))
    set_states(eng, [(x, s, seen)])
    ids = eng.step(zero, z[None], None, return_ids=True)
    assert ids.tolist() == [[ID_EXCEPTION, 0]]
    x1, s1, seen1, st = eng.get_state()
    assert list(st) == [SINGULAR] and list(seen1) == [seen]
    assert np.array_equal(x1[0], x) and np.array_equal(s1[0], s)
    assert not eng.step(zero, z[None], None, return_ids=True).any()
    eng.close()


def test_jcbb_full_map(cuda_lib):
    """seen == n: filter 0 measures a known landmark, then a far one: the match is applied, the far one flags MAP_FULL with the
    exception. Filter 1 measures the known landmark only: the match succeeds on the full map."""
    n = 12
    a = 2 * np.pi * np.arange(n) / n
    lm = 1.5 * np.stack([np.cos(a), np.sin(a)], axis=1)
    x, s, seen = landmark_state(n, lm)
    zk = polar(x, lm[4]) + np.array([0.01, -0.005])
    zfar = np.array([6.0, 0.3])
    tw = np.tile([0.01, 0.02, 0.0], (2, 1))
    eng = engine(cuda_lib, np.zeros((2, 3)), n, JC | WRAP, CHI2, mode="strict")
    set_states(eng, [(x, s, seen)] * 2)
    ids0 = eng.step(tw, np.array([[zk, zfar], [zk, zk]]), None, return_ids=True)
    assert ids0.tolist() == [[5, ID_EXCEPTION], [5, -1]], "a landmark pairs with one measurement at most"
    x1, s1, sn, st = eng.get_state()
    assert list(st) == [MAP_FULL, 0] and list(sn) == [n, n]
    ref = JcbbEkf(n, x[:3], synth.Q_DEFAULT, synth.R_DEFAULT, options=JC | WRAP, amin=CHI2[0], amax=CHI2[1])
    ref.x, ref.S, ref.seen = x.copy(), s.copy(), seen
    assert ref.step(tw[0], [zk, zfar]) == [5, ID_EXCEPTION]
    assert rel(x1[0], ref.x) < TOL and rel(s1[0], ref.S) < TOL, "the match before the exception was applied"
    eng.close()
    eng = engine(cuda_lib, np.zeros((1, 3)), n, JC | WRAP, CHI2, mode="strict")
    set_states(eng, [(x, s, seen)])
    assert eng.step(tw[:1], np.array([[zk]]), None, return_ids=True).tolist() == [[5]]
    assert not eng.getStatus().any()
    eng.close()


def test_jcbb_scan_step_bit_identical_and_async(cuda_lib):
    """JOINT | WRAP, STRICT, n = 40: the fused scan step equals step(ids = None) fed with its own z_out bit for bit at ragged marker
    counts (one filter sees 26 tubes, of which it keeps 16); step_async_packed with IDS_NONE equals the synchronous step."""
    counts = [(0, 0), (5, 0), (10, 8), (13, 13)]
    B, T, m, n = len(counts), 4, 16, 40
    tubes = ring_tubes(counts, [0.05, 0.05, 0.05, 0.3])
    poses, tw = ring_run(T, B)
    Q = 1e-4 * np.eye(3)
    fused = engine(cuda_lib, poses[0], n, JC | WRAP, CHI2, mode="strict", Q=Q, prior=None)
    plain = [engine(cuda_lib, poses[0][b:b + 1], n, JC | WRAP, CHI2, mode="strict", Q=Q, prior=None) for b in range(B)]
    matched = 0
    zs = []
    for t in range(T):
        ranges = ranges_of(poses[t], tubes)
        seen0 = fused.getSeenLandmarks()
        nm, z, ids = fused.scan_step(tw[t], ranges, tube_world.MIN_RANGE, tube_world.MAX_RANGE, m, return_all=True)
        zs.append(z)
        mv = np.clip(nm, 0, m)
        for b in range(B):
            if mv[b] == 0:
                plain[b].predict(tw[t][b:b + 1])
                assert not ids[b].any(), (t, b)
            else:
                ids2 = plain[b].step(tw[t][b:b + 1], np.ascontiguousarray(z[b:b + 1, :mv[b]]), None, return_ids=True)
                assert np.array_equal(ids[b, :mv[b]], ids2[0]) and not ids[b, mv[b]:].any(), (t, b)
        for b in range(B):
            for u, v in zip(fused.get_state(), plain[b].get_state()):
                assert np.array_equal(u[b], v[0]), (t, b)
        matched += int(((ids > 0) & (ids <= seen0[:, None])).sum())
    print(f"[JCBB scan step] seen {fused.getSeenLandmarks().tolist()}, status {fused.getStatus().tolist()}, matched {matched}")
    assert matched > 0
    for e in [fused] + plain:
        e.close()
    # the pipelined packed step, unknown ids, against the synchronous step (filters 2 and 3 have 16 markers every scan)
    sync = engine(cuda_lib, poses[0][2:], n, JC | WRAP, CHI2, mode="strict", Q=Q, prior=None)
    pipe = engine(cuda_lib, poses[0][2:], n, JC | WRAP, CHI2, mode="strict", Q=Q, prior=None)
    total, off_z, _ = pipe.packed_layout(m, False)
    bufs, outs = [], [np.zeros((2, 3 + 2 * n)) for _ in range(T)]
    for t in range(T):
        pk = np.zeros(total, dtype=np.uint8)
        pk[:off_z].view(np.float64)[:] = tw[t][2:].ravel()
        pk[off_z:].view(np.float64)[:] = zs[t][2:].ravel()
        bufs.append(pk)
    for t in range(T):
        pipe.step_async_packed(bufs[t], m, pipe.IDS_NONE, outs[t])
    pipe.wait_async()
    for t in range(T):
        sync.step(np.ascontiguousarray(tw[t][2:]), np.ascontiguousarray(zs[t][2:]), None)
        assert np.array_equal(outs[t], sync.getStateVector(), equal_nan=True), t
    for u, v in zip(pipe.get_state(), sync.get_state()):
        assert np.array_equal(u, v, equal_nan=True)
    sync.close()
    pipe.close()


def test_jcbb_refusals_and_default_handles_unaffected(cuda_lib):
    """JOINT with NEAREST_NEIGHBOUR or a bad gate: INVALID; JOINT on a large-map handle (asked for, or chosen for a long map):
    UNSUPPORTED; more than 16 measurements with unknown ids: UNSUPPORTED (known ids are fine). Default FAST, STRICT and large-map
    handles compute the same bits before and after JOINT handles ran in the process."""
    from shermbot_navigation_b200 import nuslam
    B, T = 4, 6
    sc12 = synth.ekf_scenario(B, T, n=12, seed=9, geometry="adversarial", shuffle_order=True)
    sc96 = synth.ekf_scenario(B, T, n=96, seed=9, geometry="adversarial", shuffle_order=True)
    z96, _ = picked(sc96, np.linspace(1, 96, 20).astype(np.int32))

    def run(options, modes):
        out = []
        for mode, sc, z in modes:
            kw = {} if mode is None else {"mode": mode}
            eng = cuda_lib.BatchedExtendedKalman(sc["robot0"], n_landmarks=sc["n"], Q=sc["Q"], R=sc["R"], options=options,
                                                 assoc_min=9.21, assoc_max=60.0, **kw)
            ids = [eng.step(sc["twists"][t], z[t], None, return_ids=True) for t in range(T)]
            out.append((np.stack(ids),) + eng.get_state())
            eng.close()
        return out

    default_modes = (("fast", sc12, sc12["z"]), ("strict", sc12, sc12["z"]), (None, sc96, z96))
    before = run(0, default_modes)
    for options in (JC | WRAP, JC | WRAP | JOSEPH | PRE_MOTION):
        run(options, (("fast", sc12, sc12["z"]), ("strict", sc12, sc12["z"])))
    after = run(0, default_modes)
    for a, b in zip(before, after):
        for u, v in zip(a, b):
            assert np.array_equal(u, v)

    invalid, unsupported = r"code 1\)", r"code 4\)"
    for kw in ({"options": JC | NN}, {"options": JC, "assoc_min": 0.0}, {"options": JC, "assoc_min": -1.0},
               {"options": JC, "assoc_min": math.inf}, {"options": JC, "assoc_min": math.nan}):
        with pytest.raises(nuslam.NuslamError, match=invalid):
            cuda_lib.BatchedExtendedKalman(np.zeros((1, 3)), n_landmarks=12, **kw)
    with pytest.raises(nuslam.NuslamError, match=unsupported):
        cuda_lib.BatchedExtendedKalman(np.zeros((1, 3)), n_landmarks=12, mode="large", options=JC)
    with pytest.raises(nuslam.NuslamError, match=unsupported):
        cuda_lib.BatchedExtendedKalman(np.zeros((1, 3)), n_landmarks=4096, options=JC)
    eng = engine(cuda_lib, np.zeros((2, 3)), 40, JC | WRAP, CHI2, mode="strict")
    z17 = np.tile(np.array([1.0, 0.1]), (2, 17, 1))
    with pytest.raises(nuslam.NuslamError, match=unsupported):
        eng.step(np.zeros((2, 3)), z17, None)
    poses, tw = ring_run(1, 2)
    with pytest.raises(nuslam.NuslamError, match=unsupported):
        eng.scan_step(tw[0], ranges_of(poses[0], ring_tubes([(5, 0), (5, 0)], [0.05, 0.05])), tube_world.MIN_RANGE, tube_world.MAX_RANGE, 17)
    assert not eng.getSeenLandmarks().any(), "a refused step changes nothing"
    eng.step(np.zeros((2, 3)), z17, np.tile(np.arange(1, 18, dtype=np.int32), (2, 1)))
    assert list(eng.getSeenLandmarks()) == [17, 17]
    eng.close()
    assert nuslam.OPT_JOINT_COMPATIBILITY == JC and nuslam.FILTER_ASSOC_TRUNCATED == TRUNCATED
