"""GPU tests of the large-map mode's fused scan step (nuslam_ekf_scan_step: per-filter marker counts in the delayed passes) and of its
single associateLandmark call (nuslam_ekf_associate), against the oracle, against the on-chip STRICT kernels and against the
unfused call sequence; and the C++ facade running slam.cpp:262-319 at 100 landmarks.

Tolerances as in test_world_gpu.py / test_large_gpu.py: integer outputs (marker counts, ids, `seen`, status) exact; fp64 state
1e-9 relative under teacher forcing on scans that open no landmark, 1e-4 on scans that do (the <= 2 ulp between CUDA's and glibc's
sin / cos in predict / initializeLandmark, amplified by the INT_MAX first touch -- the same for the STRICT kernel)."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

from shermbot_navigation_b200 import synth, tube_world

pytestmark = pytest.mark.gpu
TOL = 1e-9
FIRST_TOUCH_TOL = 1e-4
ROOT = Path(__file__).resolve().parent.parent
ID_EXCEPTION, MAP_FULL, SINGULAR = -1000, 1, 2


def rel_max(a, b):
    return np.abs(a - b).max() / max(np.abs(a).max(), np.abs(b).max(), 1e-300)


def oracle_scan_step(orc, n, Q, R, state, twists, z, mv):
    """One slam.cpp:262-319 iteration per filter with unknown association, filter b using its first mv[b] measurements."""
    x, s, seen = state
    B, m = z.shape[0], z.shape[1]
    xo, so, no = x.copy(), s.copy(), seen.copy()
    ids = np.zeros((B, m), dtype=np.int32)
    status = np.zeros(B, dtype=np.int32)
    for k in np.unique(mv):
        sel = np.nonzero(mv == k)[0]
        zz = z[sel][None, :, :max(k, 1)] if k > 0 else np.zeros((1, sel.size, 0, 2))
        r = orc.ekf_run(n, np.zeros((sel.size, 3)), np.zeros((sel.size, 2 * n)), Q, R, twists[sel][None], zz, None,
                        init=(x[sel], s[sel], seen[sel]))
        xo[sel], so[sel], no[sel], status[sel] = r["x"], r["sigma"], r["seen"], r["status"]
        if k > 0:
            ids[sel, :k] = r["ids_out"][0]
    return xo, so, no, ids, status


def touched(seen):
    """State indices of the robot and of landmarks 1..seen (the others keep their INT_MAX prior, which would dominate a max-norm)."""
    return np.concatenate([[0, 1, 2]] + [[3 + 2 * k, 4 + 2 * k] for k in range(int(seen))]).astype(int)


def check_step(eng_state, want, state0, ids, ido, tag, first_touch_tol=FIRST_TOUCH_TOL):
    """The engine's scan step against the oracle's, both from state0."""
    xg, sg, seeng, stg = eng_state
    xo, so, no, sto = want
    assert np.array_equal(ids, ido), f"{tag}: association ids differ"
    assert np.array_equal(seeng, no) and np.array_equal(stg != 0, sto != 0), tag
    tol = TOL if np.array_equal(no, state0[2]) else first_touch_tol
    assert rel_max(xg, xo) < tol, tag
    for b in range(xg.shape[0]):
        sel = touched(max(no[b], seeng[b]))
        assert rel_max(sg[b][np.ix_(sel, sel)], so[b][np.ix_(sel, sel)]) < tol, (tag, b)


def check_padding(nm, z, ids, m):
    mv = np.clip(nm, 0, m)
    for b in range(z.shape[0]):
        assert not z[b, mv[b]:].any() and not ids[b, mv[b]:].any(), b
    return mv


# ---- a tube field for the simulator: 8 x 5 tubes 0.6 m apart, robots start between them ----
def grid_world(B, seed):
    gx, gy = np.meshgrid(np.arange(8) * 0.6 - 2.1, np.arange(5) * 0.6 - 1.2)
    tubes = np.ascontiguousarray(np.stack([gx.ravel(), gy.ravel()], axis=1))
    g = np.random.default_rng(seed)
    cell = g.integers(0, 7, B) * 0.6 - 1.8, g.integers(0, 4, B) * 0.6 - 0.9
    cfg = np.stack([cell[0] + g.uniform(-0.05, 0.05, B), cell[1] + g.uniform(-0.05, 0.05, B), g.uniform(-3.1, 3.1, B)], axis=1)
    world = np.zeros((B, 9))
    world[:, 0], world[:, 1], world[:, 2:5] = tube_world.WHEEL_BASE, tube_world.WHEEL_RAD, cfg
    return tubes, cfg, world


def world_scans(orc, world, odom, tubes, t):
    """One simulator step (tube_world.cpp:512-537) and the odometry twists of slam.cpp:264-265, both through the oracle."""
    B = world.shape[0]
    cmd = np.tile(np.array([0.2, 0.07, 0.0]), (B, 1))
    ranges = orc.world_step(world, cmd, None, 0.1, tubes, tube_world.TUBE_RADIUS, tube_world.ROBOT_RADIUS, 1.0)
    if t == 3:
        ranges[::5] = 2.0      # scans without any marker: predict only
        ranges[1, :] = 0.5     # one all-equal scan (NUSLAM_SCAN_UB)
    tw = np.zeros((B, 3))
    for b in range(B):
        odom[b], tw[b] = orc.diffdrive_step(odom[b], world[b, 7], world[b, 8])
    return ranges, tw


def test_scan_step_auto_large_matches_oracle(cuda_lib, orc):
    """n = 96 does not fit the oracle-order kernel's shared-memory image: the handle is in large-map mode without asking for it."""
    B, T, n, m = 16, 10, 96, 12
    length = 3 + 2 * n
    assert 8 * (length * length + 17 * length + 8) > 227 * 1024
    tubes, cfg, world = grid_world(B, 23)
    Q, R = 0.1 * np.eye(3), 0.001 * np.eye(2)
    eng = cuda_lib.BatchedExtendedKalman(cfg, n_landmarks=n, Q=Q, R=R)
    odom = world[:, :7].copy()
    opened, used = np.zeros(B, int), np.zeros(B, int)
    ub = 0
    for t in range(T):
        ranges, tw = world_scans(orc, world, odom, tubes, t)
        x0, s0, seen0, _ = eng.get_state()
        nm, z, ids = eng.scan_step(tw, ranges, tube_world.MIN_RANGE, tube_world.MAX_RANGE, m, return_all=True)
        got = eng.get_state()
        det = orc.scan_detect_batch(ranges, tube_world.MIN_RANGE, tube_world.MAX_RANGE, kmax=m)
        assert np.array_equal(nm, det["n_circles"]), t
        ub += int((nm == cuda_lib.SCAN_UB).sum())
        mv = check_padding(nm, z, ids, m)
        for b in range(B):
            for i in range(mv[b]):
                zo = orc.cartesian2polar(det["circles"][b, i, 0], det["circles"][b, i, 1])
                assert np.abs(z[b, i] - zo).max() <= 1e-9 * max(1.0, np.abs(zo).max())
        xo, so, no, ido, sto = oracle_scan_step(orc, n, Q, R, (x0, s0, seen0), tw, z, mv)
        check_step(got, (xo, so, no, sto), (x0, s0, seen0), ids, ido, f"step {t}")
        opened += no - seen0
        used += mv
    print(f"[large scan step n={n}] measurements used {used.sum()}, landmarks opened {opened.sum()}, seen per filter {got[2].mean():.1f}")
    assert ub >= 1 and (opened > 0).all() and (used > 0).all()


def test_scan_step_large_equals_strict(cuda_lib, orc):
    """n = 40 runs on chip too: the same scan-step sequence on a large-map handle and a STRICT handle, teacher-forced on STRICT's state."""
    B, T, n, m = 16, 8, 40, 12
    tubes, cfg, world = grid_world(B, 22)
    Q, R = 0.1 * np.eye(3), 0.001 * np.eye(2)
    large = cuda_lib.BatchedExtendedKalman(cfg, n_landmarks=n, Q=Q, R=R, mode="large")
    strict = cuda_lib.BatchedExtendedKalman(cfg, n_landmarks=n, Q=Q, R=R, mode="strict")
    odom = world[:, :7].copy()
    opened = 0
    for t in range(T):
        ranges, tw = world_scans(orc, world, odom, tubes, t)
        x0, s0, seen0, st0 = strict.get_state()
        large.set_state(x0, s0, seen0, st0)
        a = large.scan_step(tw, ranges, tube_world.MIN_RANGE, tube_world.MAX_RANGE, m, return_all=True)
        b = strict.scan_step(tw, ranges, tube_world.MIN_RANGE, tube_world.MAX_RANGE, m, return_all=True)
        for u, v in zip(a, b):
            assert np.array_equal(u, v), t
        xl, sl, seenl, stl = large.get_state()
        xs, ss, seens, sts = strict.get_state()
        assert np.array_equal(seenl, seens) and np.array_equal(stl, sts), t
        assert rel_max(xl, xs) < TOL and rel_max(sl, ss) < TOL, t
        # the touched block: 1e-9 on scans without a first touch. A scan that opens a landmark after delayed updates of the same pass
        # (FMA order) amplifies their last-bit differences in the INT_MAX first touch that follows (measured 2.5e-6 here)
        tol = TOL if np.array_equal(seens, seen0) else FIRST_TOUCH_TOL
        for f in range(B):
            sel = touched(seens[f])
            assert rel_max(sl[f][np.ix_(sel, sel)], ss[f][np.ix_(sel, sel)]) < tol, (t, f)
        opened += int((seens - seen0).sum())
    print(f"[large == strict n={n}] {T} scan steps, {opened} landmarks opened, status bits {np.bitwise_or.reduce(sts)}")
    assert opened > B


# ---- ragged marker counts: rings of tubes around each robot (0.4 m: 1 marker per tube; 0.8 m, offset half a step) ----
def rings(k_in, k_out, phase):
    a = phase + 2 * np.pi * np.arange(k_in) / max(k_in, 1)
    b = phase + np.pi / max(k_out, 1) + 2 * np.pi * np.arange(k_out) / max(k_out, 1)
    return np.concatenate([0.4 * np.stack([np.cos(a), np.sin(a)], axis=1), 0.8 * np.stack([np.cos(b), np.sin(b)], axis=1)])


def ring_tubes(counts, phases):
    tubes = np.full((len(counts), 2 * max(sum(c) for c in counts) + 1, 2), np.nan)   # NaN rows: no tube
    for f, (c, ph) in enumerate(zip(counts, phases)):
        r = rings(c[0], c[1], ph)
        tubes[f, :len(r)] = r
    return tubes


def ring_run(T, B):
    """Poses (th, x, y) and twists of robots creeping forward: the same tubes are seen again on every scan."""
    tw = np.tile(np.array([0.01, 0.005, 0.0]), (T, B, 1))
    tw[0] = 0.0
    poses = [np.tile(np.array([0.3, 0.02, -0.01]), (B, 1))]
    for t in range(1, T):
        p = poses[-1].copy()
        p[:, 1] += tw[t, :, 1] * np.cos(p[:, 0])
        p[:, 2] += tw[t, :, 1] * np.sin(p[:, 0])
        p[:, 0] += tw[t, :, 0]
        poses.append(p)
    return poses, tw


def ranges_of(poses, tubes):
    return synth.simulate_scans(poses, tubes)


@pytest.mark.parametrize("n,counts,m", [
    (96, [(0, 0), (5, 0), (10, 8), (13, 13)], 20),   # 0, some, two passes' worth, more than m markers (m = 20 > 16: two passes)
    (6, [(3, 0), (5, 4)], 12),                       # the second filter's map fills up on its seventh marker
])
def test_scan_step_ragged_counts(cuda_lib, orc, n, counts, m):
    B, T = len(counts), 4
    Q, R = 1e-4 * np.eye(3), 0.001 * np.eye(2)
    tubes = ring_tubes(counts, [0.05] * B)
    poses, tw = ring_run(T, B)
    eng = cuda_lib.BatchedExtendedKalman(poses[0], n_landmarks=n, Q=Q, R=R, mode="large")
    strict = cuda_lib.BatchedExtendedKalman(poses[0], n_landmarks=n, Q=Q, R=R, mode="strict") if n < 70 else None
    late_matches = 0
    for t in range(T):
        ranges = ranges_of(poses[t], tubes)
        x0, s0, seen0, st0 = eng.get_state()
        nm, z, ids = eng.scan_step(tw[t], ranges, tube_world.MIN_RANGE, tube_world.MAX_RANGE, m, return_all=True)
        got = eng.get_state()
        det = orc.scan_detect_batch(ranges, tube_world.MIN_RANGE, tube_world.MAX_RANGE, kmax=m)
        assert np.array_equal(nm, det["n_circles"]), t
        mv = check_padding(nm, z, ids, m)
        # a filter whose map filled up on an earlier scan stays frozen (the reference process would have died): no step, ids 0
        live = st0 == 0
        assert not ids[~live].any() and np.array_equal(got[0][~live], x0[~live]) and np.array_equal(got[1][~live], s0[~live])
        xo, so, no, ido, sto = oracle_scan_step(orc, n, Q, R, (x0[live], s0[live], seen0[live]), tw[t][live], z[live], mv[live])
        # up to 20 first touches in one scan with a small process noise (Q = 1e-4 I): the <= 2 ulp of CUDA's sin / cos against glibc's
        # reach 9e-4 of the touched block after them (measured); scans without a first touch are held to 1e-9
        check_step(tuple(a[live] for a in got), (xo, so, no, sto), (x0[live], s0[live], seen0[live]), ids[live], ido, f"step {t}",
                   first_touch_tol=1e-2)
        if strict is not None:
            strict.set_state(x0, s0, seen0, st0)
            ns, zs, idss = strict.scan_step(tw[t], ranges, tube_world.MIN_RANGE, tube_world.MAX_RANGE, m, return_all=True)
            xs, ss, seens, sts = strict.get_state()
            assert np.array_equal(ids, idss) and np.array_equal(got[2], seens) and np.array_equal(got[3], sts), t
        if t == 0:
            first_ids, first_mv = ids, mv
        late_matches += int((ids[:, 16:] > 0).sum())
    x, s, seen, status = eng.get_state()
    print(f"[large ragged n={n}] counts {first_mv.tolist()}, seen {seen.tolist()}, status {status.tolist()}, matched ids in pass 2: {late_matches}")
    if n == 96:
        assert first_mv[0] == 0 and 0 < first_mv[1] < first_mv[2] < m and first_mv[3] == m and (nm > m).any()
        assert late_matches > 0 and not status.any()
    else:
        # the marker that finds the map full gets the exception id, every later slot 0; the filter stays frozen
        assert status[1] & MAP_FULL and not status[0] and seen[1] == n and first_mv[1] > n
        assert first_ids[1, n] == ID_EXCEPTION and not first_ids[1, n + 1:].any() and not ids[1].any()


def detect_then_step(cuda_lib, eng, tw, ranges, m):
    """The unfused sequence: nuslam_scan_detect -> cartesian2polar -> nuslam_ekf_step(ids = NULL)."""
    from shermbot_navigation_b200 import circle_fit
    det = circle_fit.scan_detect(ranges, tube_world.MIN_RANGE, tube_world.MAX_RANGE, max_circles=m, want_cluster_of_beam=False)
    B = ranges.shape[0]
    z = cuda_lib.cartesian2polar(np.ascontiguousarray(det["circles"][:, :m, :2]).reshape(-1, 2)).reshape(B, m, 2)
    return det["n_circles"], z, eng.step(tw, z, None, return_ids=True)


def test_scan_step_uniform_counts_bit_identical(cuda_lib, orc):
    """Every filter with m markers: the fused step equals the unfused call sequence on a second handle, bit for bit."""
    B, T, n, m = 3, 4, 96, 20
    tubes = ring_tubes([(13, 13)] * B, [0.05, 0.3, 1.1])
    poses, tw = ring_run(T, B)
    Q, R = 1e-4 * np.eye(3), 0.001 * np.eye(2)
    fused = cuda_lib.BatchedExtendedKalman(poses[0], n_landmarks=n, Q=Q, R=R)
    plain = cuda_lib.BatchedExtendedKalman(poses[0], n_landmarks=n, Q=Q, R=R)
    for t in range(T):
        ranges = ranges_of(poses[t], tubes)
        nm, z, ids = fused.scan_step(tw[t], ranges, tube_world.MIN_RANGE, tube_world.MAX_RANGE, m, return_all=True)
        nm2, z2, ids2 = detect_then_step(cuda_lib, plain, tw[t], ranges, m)
        assert (nm >= m).all() and np.array_equal(nm, nm2)
        assert np.array_equal(z, z2) and np.array_equal(ids, ids2), t
        for u, v in zip(fused.get_state(), plain.get_state()):
            assert np.array_equal(u, v), t
    assert (ids > 0).any()


def built_map(cuda_lib, n, seen, pose, Q, R, seed, dev):
    """A map that is already built: landmarks at the tube positions plus noise, small diagonal Sigma (as after many scans), the robot
    at its true pose; one filter."""
    import torch
    g = np.random.default_rng(seed)
    side = int(np.ceil(np.sqrt(seen)))
    gx, gy = np.meshgrid(np.arange(side) * 0.3, np.arange(side) * 0.3)
    lm = np.stack([gx.ravel(), gy.ravel()], axis=1)[:seen] - 0.3 * (side - 1) / 2 + 0.15
    length = 3 + 2 * n
    B = 1
    robot = np.asarray(pose, dtype=np.float64).reshape(1, 3)
    eng = cuda_lib.BatchedExtendedKalman(robot, n_landmarks=n, Q=Q, R=R, stream=torch.cuda.current_stream(dev).cuda_stream)
    x = torch.zeros((B, length), dtype=torch.float64, device=dev)
    x[:, :3] = torch.tensor(robot, device=dev)
    x[:, 3:3 + 2 * seen] = torch.tensor((lm + g.normal(0, 1e-4, lm.shape)).ravel(), device=dev)
    sig = torch.zeros((B, length, length), dtype=torch.float64, device=dev)
    d = torch.full((length,), 1e-4, dtype=torch.float64, device=dev)
    d[:3] = 1e-6
    for b in range(B):
        sig[b].diagonal().copy_(d)
    sn = torch.full((B,), seen, dtype=torch.int32, device=dev)
    st = torch.zeros(B, dtype=torch.int32, device=dev)
    eng.bind_state(x, sig, sn, st)
    return eng, (x, sig, sn, st), lm, robot


def test_scan_step_4096_bit_identical(cuda_lib):
    """n = 4096 (len 8195, Sigma 537 MB) from a built map: fused scan step against the unfused sequence, bit for bit."""
    import torch
    dev = torch.device("cuda")
    n, seen, T = 4096, 4000, 2
    Q, R = 1e-8 * np.eye(3), 0.001 * np.eye(2)
    poses, tw = ring_run(T, 1)
    a, sa, lm, _ = built_map(cuda_lib, n, seen, poses[0], Q, R, 3, dev)
    b, sb, _, _ = built_map(cuda_lib, n, seen, poses[0], Q, R, 3, dev)
    for t in range(T):
        near = lm[np.hypot(lm[:, 0] - poses[t][0, 1], lm[:, 1] - poses[t][0, 2]) < 1.2]
        ranges = synth.simulate_scans(poses[t], near)
        torch.cuda.synchronize()
        from shermbot_navigation_b200 import circle_fit
        k = int(circle_fit.scan_detect(ranges, tube_world.MIN_RANGE, tube_world.MAX_RANGE, max_circles=32, want_cluster_of_beam=False)["n_circles"][0])
        m = min(k, 16)
        assert m >= 8
        nm, z, ids = a.scan_step(tw[t], ranges, tube_world.MIN_RANGE, tube_world.MAX_RANGE, m, return_all=True)
        nm2, z2, ids2 = detect_then_step(cuda_lib, b, tw[t], ranges, m)
        torch.cuda.synchronize()
        assert np.array_equal(z, z2) and np.array_equal(ids, ids2), t
        assert (ids > 0).sum() >= m // 2, ids
        for u, v in zip(sa, sb):
            assert torch.equal(u, v), t
    assert int(sa[3][0]) == 0
    for e in (a, b):
        e.close()


# ---- the single associateLandmark call ----
def oracle_ring_states(orc, n, counts, steps=2):
    """Oracle filters after `steps` scans of the ring fields (scan protocol of slam.cpp:262-319): x, Sigma, seen per filter."""
    B = len(counts)
    Q, R = 1e-4 * np.eye(3), 0.001 * np.eye(2)
    tubes = ring_tubes(counts, [0.05] * B)
    poses, tw = ring_run(steps, B)
    filt = [orc.ekf(n, poses[0][b], np.zeros(2 * n), Q, R) for b in range(B)]
    for t in range(steps):
        det = orc.scan_detect_batch(ranges_of(poses[t], tubes), tube_world.MIN_RANGE, tube_world.MAX_RANGE, kmax=16)
        for b, f in enumerate(filt):
            snap = f.get()[2]
            f.predict(*tw[t, b])
            for i in range(min(max(int(det["n_circles"][b]), 0), 16)):
                z = orc.cartesian2polar(det["circles"][b, i, 0], det["circles"][b, i, 1])
                j = f.associate(z)
                if j > snap:
                    f.init_landmark(z, j)
                elif j < 0:
                    continue
                f.update(z, j)
    got = [f.get() for f in filt]
    return np.stack([g[0] for g in got]), np.stack([g[1] for g in got]), np.array([g[2] for g in got], dtype=np.int32), Q, R


def polar_of(x, px, py):
    return np.array([np.hypot(px - x[1], py - x[2]), np.arctan2(py - x[2], px - x[1]) - x[0]])


def assoc_measurements(x, seen):
    """Per filter: (kind, z) -- at landmark 1 (match), 5 cm behind it (ambiguous), far away (new)."""
    out = {}
    for kind in ("match", "near", "far"):
        z = np.zeros((x.shape[0], 2))
        for b in range(x.shape[0]):
            if seen[b] == 0:
                z[b] = [0.5, 0.2]
                continue
            z[b] = polar_of(x[b], x[b, 3], x[b, 4])
            if kind == "near":
                z[b, 0] += 0.05
            elif kind == "far":
                z[b] = [30.0, 0.5]
        out[kind] = z
    return out


def test_associate_single_call_matches_oracle(cuda_lib, orc):
    import torch
    n = 96
    x, s, seen, Q, R = oracle_ring_states(orc, n, [(0, 0), (5, 0), (10, 8), (13, 13)])
    # a fifth filter with a full map: associateLandmark throws before any candidate (slam_library.cpp:204-207)
    x, s, seen = np.concatenate([x, x[3:]]), np.concatenate([s, s[3:]]), np.concatenate([seen, [n]]).astype(np.int32)
    B = x.shape[0]
    eng = cuda_lib.BatchedExtendedKalman(x[:, :3], n_landmarks=n, Q=Q, R=R)
    outcomes = set()
    for kind, z in assoc_measurements(x, seen).items():
        for mem in ("host", "device"):
            eng.set_state(x, s, seen, np.zeros(B, np.int32))
            if mem == "host":
                got = eng.associateLandmark(z)
            else:
                got = eng.associateLandmark(torch.tensor(z, device="cuda")).cpu().numpy()
            xg, sg, seeng, stg = eng.get_state()
            want, want_seen = [], []
            for b in range(B):
                f = orc.ekf(n, x[b, :3], np.zeros(2 * n), Q, R)
                f.set(x[b], s[b], int(seen[b]))
                want.append(f.associate(z[b]))
                want_seen.append(f.get()[2])
            assert np.array_equal(got, want), (kind, mem, got, want)
            assert np.array_equal(seeng, want_seen), (kind, mem)
            assert np.array_equal(stg, np.where(np.array(want) == ID_EXCEPTION, MAP_FULL, 0)), (kind, mem, stg)
            assert np.array_equal(xg, x) and np.array_equal(sg, s), (kind, mem)   # x and Sigma untouched
        for b in range(B):
            w = want[b]
            outcomes.add("exception" if w == ID_EXCEPTION else "empty" if seen[b] == 0 else "new" if w == seen[b] + 1 else
                         "ambiguous" if w == -1 else "match")
    print(f"[large associate n={n}] outcomes {sorted(outcomes)}")
    assert outcomes == {"exception", "empty", "new", "ambiguous", "match"}


def test_associate_single_call_large_equals_strict(cuda_lib, orc):
    """n = 40: the large-map single call against the STRICT kernel's kOpAssociate, sticky status bits included (a filter already
    flagged SINGULAR still associates, and its status keeps the bit)."""
    n = 40
    x, s, seen, Q, R = oracle_ring_states(orc, n, [(0, 0), (5, 0), (10, 8), (13, 13)])
    x, s, seen = np.concatenate([x, x[3:]]), np.concatenate([s, s[3:]]), np.concatenate([seen, [n]]).astype(np.int32)
    B = x.shape[0]
    status = np.array([0, 0, SINGULAR, SINGULAR, 0], dtype=np.int32)
    large = cuda_lib.BatchedExtendedKalman(x[:, :3], n_landmarks=n, Q=Q, R=R, mode="large")
    strict = cuda_lib.BatchedExtendedKalman(x[:, :3], n_landmarks=n, Q=Q, R=R, mode="strict")
    for kind, z in assoc_measurements(x, seen).items():
        res = []
        for e in (large, strict):
            e.set_state(x, s, seen, status)
            got = e.associateLandmark(z)
            res.append((got,) + e.get_state())
        (gl, xl, sl, nl, stl), (gs, xs, ss, ns, sts) = res
        assert np.array_equal(gl, gs) and np.array_equal(nl, ns) and np.array_equal(stl, sts), (kind, gl, gs, stl, sts)
        assert np.array_equal(xl, x) and np.array_equal(sl, s)
        assert (stl[2:4] & SINGULAR).all() and gl[3] != 0


# ---- the C++ facade at 100 landmarks (large-map mode, chosen by the engine) ----
def test_facade_loop_at_100_landmarks(cuda_lib, orc, tmp_path):
    exe = tmp_path / "facade_large_main"
    libdir = cuda_lib.LIB_PATH.parent
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-Werror", f"-I{ROOT / 'include'}", "-o", str(exe), str(ROOT / "tests" / "facade_large_main.cpp"),
           f"-L{libdir}", "-lnuslam_b200", f"-Wl,-rpath,{libdir}"]
    out = subprocess.run(cmd, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    lines, ids = {}, []
    for ln in out.stdout.splitlines():
        tok = ln.split()
        if tok[0] == "ID":
            ids.append(int(tok[3]))
        else:
            lines.setdefault(tok[0], []).append(tok[1:])
    assert "EXC" not in lines
    # the same loop on the oracle (slam.cpp:262-319); keep in step with tests/facade_large_main.cpp
    n, steps = 100, 20
    f = orc.ekf(n, np.array([0.1, -0.2, 0.3]), np.zeros(2 * n), 0.1 * np.eye(3), 0.001 * np.eye(2))
    zs = [np.array([1.0 + 0.25 * k, -1.5 + 0.5 * k]) for k in range(7)]
    want = []
    for step in range(steps):
        f.predict(0.02, 0.007)
        seen0 = f.get()[2]
        for z in zs:
            i = f.associate(z)
            want.append(i)
            if i > seen0:
                f.init_landmark(z, i)
            elif i < 0:
                continue
            f.update(z, i)
    x, S, seen = f.get()
    assert ids == want
    assert int(lines["SEEN"][0][0]) == seen
    gx = np.array([float(v) for v in lines["X"][0]])
    gS = np.array([float(v) for v in lines["S"][0]]).reshape(3 + 2 * n, 3 + 2 * n).T   # printed column-major
    sel = touched(seen)
    print(f"[facade n={n}] {len(ids)} associations, seen {seen}: x rel {rel_max(gx, x):.2e}, Sigma (touched) rel "
          f"{rel_max(gS[np.ix_(sel, sel)], S[np.ix_(sel, sel)]):.2e}")
    assert seen >= 2 and any(i > 0 and i <= 2 for i in want[len(zs):])
    assert rel_max(gx, x) < FIRST_TOUCH_TOL and rel_max(gS[np.ix_(sel, sel)], S[np.ix_(sel, sel)]) < FIRST_TOUCH_TOL
