"""The opt-in variants (NUSLAM_OPT_WRAP_INNOVATION, _JOSEPH, _PRE_MOTION_JACOBIAN) in large-map mode: the delayed passes, the
symmetric JOSEPH pass (Sigma_bar_0 - [K | A][A | K]^T), association, the oracle-order tail and the fused scan step. Checked against the
dense numpy restatement (tests/sane_reference.py), against the on-chip STRICT kernels, against the unfused call sequence and against
the sequential single-update form. Tolerance 1e-9 relative, as in test_options_gpu.py."""
import numpy as np
import pytest

from sane_reference import JOSEPH, PRE_MOTION, WRAP, SaneEkf
from shermbot_navigation_b200 import synth, tube_world
from test_large_scan_gpu import grid_world, ring_run, ring_tubes, ranges_of, touched, world_scans

pytestmark = pytest.mark.gpu
TOL = 1e-9
ALL = WRAP | JOSEPH | PRE_MOTION
SINGULAR = 2


def rel(a, b):
    return np.abs(a - b).max() / max(np.abs(a).max(), np.abs(b).max(), 1e-300)


def picked(sc, pick_ids):
    """Every step measures the same landmarks (ids in pick_ids), in the scenario's shuffled order."""
    T, B = sc["ids"].shape[:2]
    m = len(pick_ids)
    z = np.zeros((T, B, m, 2))
    ids = np.zeros((T, B, m), dtype=np.int32)
    for t in range(T):
        for b in range(B):
            sel = np.isin(sc["ids"][t, b], pick_ids)
            z[t, b], ids[t, b] = sc["z"][t, b][sel], sc["ids"][t, b][sel]
    return z, ids


def check_joseph(s, tag, filters=None):
    for b in (range(s.shape[0]) if filters is None else filters):
        assert np.array_equal(s[b], s[b].T), f"{tag}: Joseph form returns an exactly symmetric Sigma (filter {b})"
        assert np.linalg.eigvalsh(s[b]).min() > -1e-12 * np.abs(s[b]).max(), (tag, b)


def run_numpy(cuda_lib, sc, z, ids, options, prior, known=True, mode="large"):
    """mode None: the engine chooses the mode from the map size."""
    B, T = z.shape[1], z.shape[0]
    n = sc["n"]
    kw = {} if mode is None else {"mode": mode}
    eng = cuda_lib.BatchedExtendedKalman(sc["robot0"][:B], n_landmarks=n, Q=sc["Q"], R=sc["R"], options=options, landmark_prior=prior, **kw)
    refs = [SaneEkf(n, sc["robot0"][b], sc["Q"], sc["R"], prior=prior, options=options) for b in range(B)]
    ids_ok = True
    for t in range(T):
        got = eng.step(sc["twists"][t, :B], z[t], ids[t] if known else None, return_ids=True)
        for b, f in enumerate(refs):
            want = f.step(sc["twists"][t, b], z[t, b], ids[t, b] if known else None)
            ids_ok &= list(got[b]) == want
    return eng, refs, ids_ok


@pytest.mark.parametrize("options", [WRAP, JOSEPH, PRE_MOTION, ALL])
@pytest.mark.parametrize("geometry", ["benign", "adversarial"])
def test_large_options_match_numpy(cuda_lib, options, geometry):
    """n = 96 (large-map mode chosen by the engine), 20 measured landmarks per step: two passes (16 + 4) per step. The handle that
    chose its own mode computes the same bits as one created with mode="large" (the on-chip kernels round differently)."""
    B, T, n = 3, 10, 96
    sc = synth.ekf_scenario(B, T, n=n, seed=41, geometry=geometry, shuffle_order=True)
    z, ids = picked(sc, np.linspace(1, n, 20).astype(np.int32))
    eng, refs, ids_ok = run_numpy(cuda_lib, sc, z, ids, options, 100.0, mode=None)
    x, s, seen, status = eng.get_state()
    explicit, _, _ = run_numpy(cuda_lib, sc, z, ids, options, 100.0, mode="large")
    for u, v in zip((x, s, seen, status), explicit.get_state()):
        assert np.array_equal(u, v), "the engine did not choose large-map mode at 96 landmarks"
    explicit.close()
    assert ids_ok and not status.any()
    ex = max(rel(x[b], refs[b].x) for b in range(B))
    es = max(rel(s[b], refs[b].S) for b in range(B))
    print(f"[large options {options} {geometry}] x rel {ex:.2e}, Sigma rel {es:.2e}")
    assert ex < TOL and es < TOL
    if options & JOSEPH:
        check_joseph(s, f"options {options} {geometry}")
    eng.close()


def test_large_options_unknown_association_matches_numpy(cuda_lib):
    """WRAP | JOSEPH with associateLandmark in the delayed passes (the adversarial geometry's bearings cross +-pi, so the wrap decides
    matches), then the single associateLandmark call against SaneEkf.associate on the same state."""
    import copy
    B, T, n = 3, 8, 96
    opts = WRAP | JOSEPH
    sc = synth.ekf_scenario(B, T, n=n, seed=7, geometry="adversarial", shuffle_order=True)
    z, ids = picked(sc, np.arange(1, n + 1, 8, dtype=np.int32))   # 12 landmarks 0.31 m apart
    eng, refs, ids_ok = run_numpy(cuda_lib, sc, z, ids, opts, 50.0, known=False)
    x, s, seen, status = eng.get_state()
    assert ids_ok and not status.any()
    assert np.array_equal(seen, [f.seen for f in refs])
    ex, es = max(rel(x[b], refs[b].x) for b in range(B)), max(rel(s[b], refs[b].S) for b in range(B))
    print(f"[large association WRAP|JOSEPH] seen {seen.tolist()}: x rel {ex:.2e}, Sigma rel {es:.2e}")
    assert ex < TOL and es < TOL
    check_joseph(s, "association")
    # the single call: a measurement of landmark 1 with its bearing off by 2 pi matches only when the innovation is wrapped
    zz = np.zeros((B, 2))
    for b in range(B):
        zhat, _ = refs[b].model(1)
        zz[b] = [zhat[0], zhat[1] + (2 * np.pi if zhat[1] < 0 else -2 * np.pi)]
    got = eng.associateLandmark(zz)
    want = [copy.deepcopy(f).associate(zz[b]) for b, f in enumerate(refs)]
    assert list(got) == want and all(w == 1 for w in want), (got, want)
    xg, sg, seeng, _ = eng.get_state()
    assert np.array_equal(xg, x) and np.array_equal(sg, s) and np.array_equal(seeng, seen)
    eng.close()


def run_pair(cuda_lib, sc, z, ids, options, known):
    out = {}
    n = sc["n"]
    for mode in ("large", "strict"):
        eng = cuda_lib.BatchedExtendedKalman(sc["robot0"], n_landmarks=n, Q=sc["Q"], R=sc["R"], mode=mode, options=options)
        got = [eng.step(sc["twists"][t], z[t], ids[t] if known else None, return_ids=True) for t in range(z.shape[0])]
        out[mode] = (np.stack(got),) + eng.get_state()
        eng.close()
    return out["large"], out["strict"]


@pytest.mark.parametrize("known", [True, False])
def test_large_options_equal_strict_from_scratch(cuda_lib, known):
    """n = 40 on a large-map handle and on a STRICT handle, options = 7, INT_MAX prior, from scratch: the first touches of the first
    scan go through the oracle-order tail with the options set (bit for bit what STRICT does), the later scans through the delayed
    passes and the symmetric JOSEPH pass. 40 measurements per step: three passes (16 + 16 + 8)."""
    B, T, n = 4, 5, 40
    sc = synth.ekf_scenario(B, T, n=n, seed=62, geometry="adversarial", shuffle_order=True)
    (il, xl, sl, nl, stl), (is_, xs, ss, ns, sts) = run_pair(cuda_lib, sc, sc["z"], sc["ids"], ALL, known)
    assert np.array_equal(il, is_) and np.array_equal(nl, ns) and np.array_equal(stl, sts)
    assert not sts.any() and (ns > 0).all()
    ex = rel(xl, xs)
    es = max(rel(sl[b][np.ix_(touched(ns[b]), touched(ns[b]))], ss[b][np.ix_(touched(ns[b]), touched(ns[b]))]) for b in range(B))
    print(f"[large == strict, options 7, known={known}] seen {ns.tolist()}: x rel {ex:.2e}, Sigma (touched) rel {es:.2e}")
    assert ex < TOL and es < TOL
    check_joseph(sl, "large")


def test_large_options_scan_step_equals_strict(cuda_lib, orc):
    """The fused scan step at n = 40 with options = 7, large-map handle against STRICT handle, from scratch (INT_MAX prior)."""
    B, T, n, m = 8, 6, 40, 12
    tubes, cfg, world = grid_world(B, 22)
    Q, R = 0.1 * np.eye(3), 0.001 * np.eye(2)
    large = cuda_lib.BatchedExtendedKalman(cfg, n_landmarks=n, Q=Q, R=R, mode="large", options=ALL)
    strict = cuda_lib.BatchedExtendedKalman(cfg, n_landmarks=n, Q=Q, R=R, mode="strict", options=ALL)
    odom = world[:, :7].copy()
    worst = (0.0, 0.0)
    for t in range(T):
        ranges, tw = world_scans(orc, world, odom, tubes, t)
        a = large.scan_step(tw, ranges, tube_world.MIN_RANGE, tube_world.MAX_RANGE, m, return_all=True)
        b = strict.scan_step(tw, ranges, tube_world.MIN_RANGE, tube_world.MAX_RANGE, m, return_all=True)
        for u, v in zip(a, b):
            assert np.array_equal(u, v), t
        xl, sl, nl, stl = large.get_state()
        xs, ss, ns, sts = strict.get_state()
        assert np.array_equal(nl, ns) and np.array_equal(stl, sts), t
        es = max(rel(sl[f][np.ix_(touched(ns[f]), touched(ns[f]))], ss[f][np.ix_(touched(ns[f]), touched(ns[f]))]) for f in range(B))
        worst = (max(worst[0], rel(xl, xs)), max(worst[1], es))
        # exactly symmetric after any Joseph update; a filter whose scan applied none keeps predict's Sigma (STRICT's as well)
        check_joseph(sl, f"scan {t}", np.nonzero((a[2] > 0).any(axis=1))[0])
    print(f"[large == strict scan step, options 7] {T} scans, seen {ns.tolist()}: x rel {worst[0]:.2e}, Sigma (touched) rel {worst[1]:.2e}")
    assert worst[0] < TOL and worst[1] < TOL


def test_large_options_scan_step_bit_identical(cuda_lib):
    """The fused scan step with options = 7 equals detect -> cartesian2polar -> step(ids = None) bit for bit, at ragged marker
    counts (0, some, two passes' worth, more than m): filter b's unfused step runs on a one-filter handle of its own with its own
    count (nuslam_ekf_step has no per-filter counts; the large-map kernels treat the filters of a batch independently). A filter
    flagged SINGULAR keeps its x and Sigma bit for bit."""
    from shermbot_navigation_b200 import circle_fit
    counts = [(0, 0), (5, 0), (10, 8), (13, 13), (10, 8)]
    B, T, n, m = len(counts), 4, 96, 20
    tubes = ring_tubes(counts, [0.05, 0.05, 0.05, 0.05, 0.3])
    poses, tw = ring_run(T, B)
    Q, R = 1e-4 * np.eye(3), 0.001 * np.eye(2)
    fused = cuda_lib.BatchedExtendedKalman(poses[0], n_landmarks=n, Q=Q, R=R, mode="large", options=ALL)
    plain = [cuda_lib.BatchedExtendedKalman(poses[0][b:b + 1], n_landmarks=n, Q=Q, R=R, mode="large", options=ALL) for b in range(B)]
    frozen = None
    late_matches = 0
    for t in range(T):
        if t == 2:
            # filter 4 is flagged SINGULAR (its reference process would have died): from here on nothing may touch it
            x, s, seen, st = fused.get_state()
            st[4] |= SINGULAR
            fused.set_state(x, s, seen, st)
            plain[4].set_state(x[4:], s[4:], seen[4:], st[4:])
            frozen = (x[4].copy(), s[4].copy())
        ranges = ranges_of(poses[t], tubes)
        nm, z, ids = fused.scan_step(tw[t], ranges, tube_world.MIN_RANGE, tube_world.MAX_RANGE, m, return_all=True)
        det = circle_fit.scan_detect(ranges, tube_world.MIN_RANGE, tube_world.MAX_RANGE, max_circles=m, want_cluster_of_beam=False)
        assert np.array_equal(nm, det["n_circles"]), t
        mv = np.clip(nm, 0, m)
        for b in range(B):
            if mv[b] == 0:
                plain[b].predict(tw[t][b:b + 1])
                assert not ids[b].any() and not z[b].any(), (t, b)
            else:
                z2 = cuda_lib.cartesian2polar(np.ascontiguousarray(det["circles"][b, :mv[b], :2])).reshape(1, mv[b], 2)
                ids2 = plain[b].step(tw[t][b:b + 1], z2, None, return_ids=True)
                assert np.array_equal(z[b, :mv[b]], z2[0]) and not z[b, mv[b]:].any(), (t, b)
                assert np.array_equal(ids[b, :mv[b]], ids2[0]) and not ids[b, mv[b]:].any(), (t, b)
        x, s, seen, st = fused.get_state()
        for b in range(B):
            for u, v in zip((x, s, seen, st), plain[b].get_state()):
                assert np.array_equal(u[b], v[0]), (t, b)
        if frozen is not None:
            assert np.array_equal(x[4], frozen[0]) and np.array_equal(s[4], frozen[1]) and not ids[4].any(), t
        assert not st[:4].any(), t
        check_joseph(s, f"scan {t}", [b for b in range(4) if (ids[b] > 0).any()])
        late_matches += int((ids[:, 16:] > 0).sum())
    assert nm[0] == 0 and 0 < nm[1] < m and nm[3] > m and late_matches > 0
    for e in [fused] + plain:
        e.close()


def test_4096_landmarks_joseph_delayed_equals_sequential(cuda_lib):
    """len 8195, Sigma 537 MB, JOSEPH: one delayed rank-48 symmetric pass per scan (12 measurements) against twelve single-measurement
    update calls (twelve rank-4 passes); Sigma exactly symmetric after every scan."""
    import torch
    n, m = 4096, 12
    length = 3 + 2 * n
    rng = np.random.default_rng(7)
    lm = rng.uniform(-3, 3, size=(n, 2))
    robot = np.array([[0.05, -0.02, 0.01]])
    Q, R = synth.Q_DEFAULT, synth.R_DEFAULT
    pick = rng.choice(n, size=m, replace=False)
    dev = torch.device("cuda")
    x0 = torch.tensor(np.concatenate([robot[0], lm.ravel()])[None], device=dev)
    d = torch.full((length,), 1e-3, dtype=torch.float64, device=dev)
    d[:3] = 1e-2
    engs, states = [], []
    for _ in range(2):
        e = cuda_lib.BatchedExtendedKalman(robot, lm.reshape(1, -1), Q, R, mode="large", options=JOSEPH)
        xs = x0.clone()
        sig = torch.zeros((1, length, length), dtype=torch.float64, device=dev)
        sig[0].diagonal().copy_(d)
        seen = torch.full((1,), n, dtype=torch.int32, device=dev)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        e.bind_state(xs, sig, seen, status)
        engs.append(e)
        states.append((xs, sig, seen, status))
    ids = torch.tensor((pick + 1)[None].astype(np.int32), device=dev)
    for t in range(3):
        torch.cuda.synchronize()
        tw = torch.tensor([[0.02, 0.007, 0.0]], device=dev, dtype=torch.float64)
        px, py, th = float(states[0][0][0, 1]), float(states[0][0][0, 2]), float(states[0][0][0, 0])
        dl = lm[pick] - np.array([px, py])
        z = np.stack([np.hypot(dl[:, 0], dl[:, 1]) + rng.normal(0, 0.01, m),
                      synth.wrap_pi(np.arctan2(dl[:, 1], dl[:, 0]) - th + rng.normal(0, 0.01, m))], axis=1)
        zt = torch.tensor(z[None], device=dev)
        engs[0].step(tw, zt, ids)                                  # delayed: one rank-48 symmetric pass
        engs[1].predict(tw)
        for i in range(m):                                         # sequential: twelve rank-4 symmetric passes
            engs[1].update(zt[:, i].contiguous(), ids[:, i].contiguous())
        torch.cuda.synchronize()
        for xs, sig, seen, status in states:
            assert torch.equal(sig[0], sig[0].T), t
            assert int(status[0]) == 0 and bool(torch.isfinite(sig).all()), t
    ex = float((states[0][0] - states[1][0]).abs().max() / states[1][0].abs().max())
    es = float((states[0][1] - states[1][1]).abs().max() / states[1][1].abs().max())
    moved_s = float((states[0][1][0].diagonal() - d).abs().max() / d.max())
    print(f"[large n=4096 JOSEPH] delayed vs sequential after 3 scans: x rel {ex:.2e}, Sigma rel {es:.2e}; diagonal moved {moved_s:.2e}")
    assert moved_s > 1e-2
    assert ex < 1e-12 and es < 1e-11
    for e in engs:
        e.close()


def test_default_large_handle_unchanged_by_option_handles(cuda_lib):
    """options = 0 after option handles ran in the same process: the per-device launch state (cooperative occupancy, function
    attributes) is per kernel variant, so a default handle computes the same bits as one created before any option handle."""
    B, T, n = 3, 4, 96
    sc = synth.ekf_scenario(B, T, n=n, seed=5, geometry="adversarial", shuffle_order=True)
    z, ids = picked(sc, np.linspace(1, n, 20).astype(np.int32))

    def run(options):
        eng = cuda_lib.BatchedExtendedKalman(sc["robot0"], n_landmarks=n, Q=sc["Q"], R=sc["R"], mode="large", options=options,
                                             landmark_prior=100.0)
        for t in range(T):
            eng.step(sc["twists"][t], z[t], ids[t] if t % 2 == 0 else None)
        out = eng.get_state()
        eng.close()
        return out

    before = run(0)
    for options in (ALL, JOSEPH, WRAP, PRE_MOTION):
        run(options)
    after = run(0)
    for u, v in zip(before, after):
        assert np.array_equal(u, v)
