"""The FAST EKF kernels with a different twist and heading for every filter.

synth.ekf_scenario gives every filter and every step the same body twist, and its only dth == 0 step is the first-touch step, which
the FAST kernels hand to the strict kernel. So without these tests neither FAST kernel ever ran its dth == 0 branch, a negative or
zero dth / dx, a |dth| > 0.25 step (sincos_small's fall-back to sincos_fast) or a heading far outside [-pi, pi] at step entry; and
a kernel that read its partner filter's twist, or a twist prefetched for the wrong pair, gave the right answer. Here:
  * every filter gets its own twist at every step, drawn from dth in {0, +-1e-3, +-0.02, +-0.26, +-0.9}, dx in {0.007, -0.007, 0};
  * per-filter headings at step entry just inside +-pi (predict carries them across), exactly +-pi, 7.0 and -20.0 (a filter that
    had no measurement for a few steps: predict does not wrap the heading);
  * the adversarial ring (bearings cross +-pi), plus a landmark straight behind the robot (dy == 0 exactly, atan2 == pi) and one
    beside it (dx == 0 exactly) in the first updates of a step whose twist leaves the position unchanged (dx == 0);
  * measurements are generated from each filter's own motion and map estimate, so innovations stay small.
Each scenario runs through the resident pair kernel (ekf_res2.cuh, the default for known ids), the register kernel
(ekf_fast.cuh, NUSLAM_KERNEL=fast) and the association path (ids = None, ekf_fast.cuh), against the oracle's ekf_run from the same
warm-start state (the oracle's state after a full first-touch step)."""
import numpy as np
import pytest

from shermbot_navigation_b200 import synth

pytestmark = pytest.mark.gpu

TOL = 1e-9
N = 12
DTH = np.array([0.0, 1e-3, -1e-3, 0.02, -0.02, 0.26, -0.26, 0.9, -0.9])
DX = np.array([0.007, -0.007, 0.0])
CUT = 1e-9   # a predicted bearing closer than this to +-pi makes the reference ill-posed (see cut_filters)


def rel_max(a, b):
    scale = max(np.abs(a).max(), np.abs(b).max(), 1e-300)
    return np.abs(a - b).max() / scale


def twist_scenario(orc, B, T, seed, special=True, assoc=False):
    """B filters, T steps (step 0 is the first-touch step). Returns the engine's inputs, the warm-start state after step 0 (with
    per-filter headings and the two axis-aligned landmarks written into it), and the per-filter twists. assoc: the warm start is
    the oracle's state after three steps of association from scratch (ids = None), as in the other association tests: a map built
    from known ids is full, and the reference's associateLandmark then throws at once."""
    rng = np.random.default_rng(seed)
    sc = synth.ekf_scenario(B, 3 if assoc else 1, n=N, geometry="adversarial", seed=seed, shuffle_order=assoc)
    if assoc:
        first = orc.ekf_run(N, sc["robot0"], sc["map0"], sc["Q"], sc["R"], sc["twists"], sc["z"], None)
    else:
        first = orc.ekf_run(N, sc["robot0"], sc["map0"], sc["Q"], sc["R"], sc["twists"][:1], sc["z"][:1], sc["ids"][:1])
    x0, s0, seen0 = first["x"].copy(), first["sigma"], first["seen"]
    tw = np.zeros((T, B, 3))
    tw[:, :, 0] = rng.choice(DTH, (T, B))
    tw[:, :, 1] = rng.choice(DX, (T, B))
    tw[2, :, 0] = np.where(np.arange(B) % 3 == 0, 0.0, tw[2, :, 0])   # a step where only some filters have dth == 0
    tw[3, :, 0] = 0.0
    tw[3, B // 2, 0] = 0.02                                          # ... and one where all but one have
    ids = np.stack([np.stack([rng.permutation(N) + 1 for _ in range(B)]) for _ in range(T)]).astype(np.int32)
    if special:
        # headings at step entry: just inside +-pi, exactly +-pi, far outside [-pi, pi]
        head = {0: np.pi - 0.004, 1: -np.pi + 0.004, 2: np.pi, 3: -np.pi, 4: 7.0, 5: -20.0, 6: np.pi - 1e-6, 7: -np.pi + 1e-6}
        for b, th in head.items():
            if b < B:
                x0[b, 0] = th
        for b in range(min(B, 8)):
            tw[1, b, 0] = 0.02 if x0[b, 0] > 0 else -0.02   # carry the near-cut headings across +-pi
        for b in (4, 5):   # 7.0 and -20.0: no measurement in the first steps, then measurements
            if b < B:
                ids[1:3, b] = 0
        # straight behind (dy == 0, dx < 0: atan2 = pi) and beside (dx == 0) the robot, measured first in a step with dx == 0
        for b in range(8, min(B, 24)):
            px, py = x0[b, 1], x0[b, 2]
            x0[b, 3 + 2 * 10], x0[b, 4 + 2 * 10] = px - 0.4, py
            x0[b, 3 + 2 * 11], x0[b, 4 + 2 * 11] = px, (py + 0.3 if b % 2 else py - 0.3)
            tw[1, b, 1] = 0.0
            rest = [j for j in ids[1, b] if j not in (11, 12)]
            ids[1, b] = [11, 12] + rest
    # measurements from each filter's own motion (its twists from its warm-start pose) of its own map estimate
    pose = x0[:, :3].copy()
    lm = x0[:, 3:].reshape(B, N, 2)
    z = np.zeros((T, B, N, 2))
    g = np.random.default_rng(seed + 1)
    for t in range(1, T):
        dth, dx = tw[t, :, 0], tw[t, :, 1]
        th = pose[:, 0]
        straight = dth == 0.0
        q = np.where(straight, 0.0, dx / np.where(straight, 1.0, dth))
        pose = pose + np.stack([dth,
                                np.where(straight, dx * np.cos(th), -q * np.sin(th) + q * np.sin(th + dth)),
                                np.where(straight, dx * np.sin(th), q * np.cos(th) - q * np.cos(th + dth))], axis=1)
        d = lm[np.arange(B)[:, None], np.maximum(ids[t], 1) - 1] - pose[:, None, 1:]   # an empty slot (id 0) still gets a real measurement
        rng_ = np.hypot(d[..., 0], d[..., 1]) + g.normal(0, 0.002, (B, N))
        brg = synth.wrap_pi(np.arctan2(d[..., 1], d[..., 0]) - pose[:, None, 0] + g.normal(0, 0.002, (B, N)))
        brg = np.where(np.abs(np.abs(brg) - np.pi) < CUT, np.sign(brg) * (np.pi - 2 * CUT), brg)   # measured bearings off the cut
        z[t, :, :, 0], z[t, :, :, 1] = rng_, brg
    return dict(sc=sc, init=(x0, s0, seen0), status0=(first["status"] != 0).astype(np.int32), tw=tw, z=np.ascontiguousarray(z),
                ids=ids)


def cut_filters(orc, case, filters):
    """Filters whose run meets a predicted bearing within CUT of +-pi: the reference innovation z - zhat is not wrapped, so a 1-ulp
    difference in the predicted bearing there flips it by 2 pi and no tolerance separates a correct kernel from a wrong one. Found by
    stepping the oracle's filters through the scenario and reading zhat before every update."""
    x0, s0, seen0 = case["init"]
    sc = case["sc"]
    bad = []
    for b in filters:
        f = orc.ekf(N, sc["robot0"][b], sc["map0"][b], sc["Q"], sc["R"])
        f.set(x0[b], s0[b], seen0[b])
        hit = False
        for t in range(1, case["tw"].shape[0]):
            f.predict(*case["tw"][t, b])
            for i in range(N):
                j = int(case["ids"][t, b, i])
                if j > 0:
                    hit |= abs(abs(f.zhat(j)[1]) - np.pi) < CUT
                    f.update(case["z"][t, b, i], j)
        if hit:
            bad.append(b)
    return bad


def run_engine(cuda_lib, case, ids=True, order=None):
    sc = case["sc"]
    x0, s0, seen0 = case["init"]
    B = x0.shape[0]
    o = np.arange(B) if order is None else order
    eng = cuda_lib.BatchedExtendedKalman(sc["robot0"][o], sc["map0"][o], sc["Q"], sc["R"], mode="fast")
    eng.set_state(np.ascontiguousarray(x0[o]), np.ascontiguousarray(s0[o]), np.ascontiguousarray(seen0[o]))
    got_ids = []
    for t in range(1, case["tw"].shape[0]):
        r = eng.step(np.ascontiguousarray(case["tw"][t][o]), np.ascontiguousarray(case["z"][t][o]),
                     np.ascontiguousarray(case["ids"][t][o]) if ids else None, return_ids=True)
        got_ids.append(np.asarray(r).copy())
    x, s, seen, status = eng.get_state()
    eng.close()
    inv = np.argsort(o)
    return x[inv], s[inv], seen[inv], status[inv], np.stack(got_ids)[:, inv]


def oracle_run(orc, case, filters=None, ids=True):
    sc = case["sc"]
    x0, s0, seen0 = case["init"]
    f = np.arange(x0.shape[0]) if filters is None else filters
    return orc.ekf_run(N, sc["robot0"][f], sc["map0"][f], sc["Q"], sc["R"], case["tw"][1:, f], case["z"][1:, f],
                       case["ids"][1:, f] if ids else None, init=(x0[f], s0[f], seen0[f]))


@pytest.mark.parametrize("B,seed", [(61, 1), (64, 2), (33, 3)])
def test_per_filter_twists_and_headings(cuda_lib, orc, monkeypatch, B, seed):
    """Known ids, T = 10 (9 fused steps): both known-id kernels within 1e-9 of the oracle per filter (state and Sigma), and within
    1e-11 of each other; odd B leaves one filter alone in the last pair of the pair kernel."""
    T = 10
    case = twist_scenario(orc, B, T, seed)
    bad = cut_filters(orc, case, range(B))
    ok = np.setdiff1d(np.arange(B), bad)
    want = oracle_run(orc, case)
    out = {}
    for kern in ("res2", "fast"):
        monkeypatch.setenv("NUSLAM_KERNEL", kern)
        x, s, seen, status, _ = run_engine(cuda_lib, case)
        out[kern] = (x, s)
        assert not status.any() and np.array_equal(seen, want["seen"]), kern
        ex = max(rel_max(x[b], want["x"][b]) for b in ok)
        es = max(rel_max(s[b], want["sigma"][b]) for b in ok)
        print(f"[twists B={B} {kern}] worst per-filter rel vs oracle: x {ex:.2e}, Sigma {es:.2e}; filters set aside at the +-pi cut: {bad}")
        assert ex < TOL and es < TOL, kern
    (x0, s0), (x1, s1) = out["fast"], out["res2"]
    ex, es = rel_max(x1[ok], x0[ok]), max(rel_max(s1[b], s0[b]) for b in ok)
    print(f"[twists B={B}] res2 vs fast: x {ex:.2e}, Sigma {es:.2e}")
    assert ex < 1e-11 and es < 1e-11
    assert len(bad) <= 2, f"the generator met the cut too often: {bad}"


@pytest.mark.parametrize("B,seed", [(61, 4), (32, 5)])
def test_per_filter_twists_association(cuda_lib, orc, B, seed):
    """Association on the device (ids = None, ekf_fast.cuh) with per-filter twists and headings, teacher-forced per step from the
    oracle's state: ids bit-exact, state within 1e-9. A filter-step that opens a landmark (first touch at the INT_MAX prior, whose
    cancellation amplifies the CUDA-vs-glibc ulp of sin / cos / atan2, the L2 situation of tests/test_ekf_gpu.py) is held to 1e-4,
    as in test_config4_subsample_4096_filters."""
    T = 10
    case = twist_scenario(orc, B, T, seed, assoc=True)
    sc = case["sc"]
    state = case["init"] + (case["status0"],)
    eng = cuda_lib.BatchedExtendedKalman(sc["robot0"], sc["map0"], sc["Q"], sc["R"], mode="fast")
    mism, worst, worst_late, matched = 0, 0.0, 0.0, 0
    for t in range(1, T):
        o = orc.ekf_run(N, sc["robot0"], sc["map0"], sc["Q"], sc["R"], case["tw"][t:t + 1], case["z"][t:t + 1], None, init=state[:3])
        frozen = state[3] != 0   # a filter the reference process left (map full) stays frozen: the oracle's run is fresh, so skip it
        eng.set_state(state[0], state[1], state[2], state[3])
        ids = eng.step(np.ascontiguousarray(case["tw"][t]), case["z"][t], None, return_ids=True)
        x, s, seen, status = eng.get_state()
        for b in range(B):
            if frozen[b]:
                continue
            mism += int((ids[b] != o["ids_out"][0, b]).sum())
            if o["seen"][b] != state[2][b]:
                worst_late = max(worst_late, rel_max(x[b], o["x"][b]))
            else:
                worst = max(worst, rel_max(x[b], o["x"][b]))
            assert seen[b] == o["seen"][b] and (status[b] != 0) == (o["status"][b] != 0), (t, b)
        state = (o["x"], o["sigma"], o["seen"], np.where(frozen, 1, (o["status"] != 0).astype(np.int32)))
        matched += int((o["ids_out"][0][~frozen] > 0).sum())
    print(f"[twists association B={B}] id mismatches {mism}, {matched} matches applied, worst x rel {worst:.2e} (steps that open a landmark: {worst_late:.2e}); "
          f"frozen (map full) at the end {int((state[3] != 0).sum())}")
    assert mism == 0 and worst < TOL and worst_late < 1e-4 and matched > 0


def test_pair_position_invariance(cuda_lib, orc, monkeypatch):
    """B = 8 193 distinct filters (odd: the last pair holds one; more pairs than the grid's kRes2CtasPerSm x SMs warps, so the pair
    kernel runs its grid-stride loop and its one-pair-ahead prefetch) in three batch orders -- identity, reversed, a random
    permutation: every filter's state and Sigma must be bit-identical across the orders, in both known-id kernels (each filter's
    arithmetic, the in-place DMMA pass included, is its own: half 0, half 1 and a later grid stride change no bit). This caught the
    pair kernel wrapping the heading of a filter without a measurement in a slot whenever its partner had one (the 7.0 / -20.0
    filters: in the identity order they are each other's partner). A seeded sample of 256 filters is compared with the oracle."""
    B, T = 8193, 10
    case = twist_scenario(orc, B, T, seed=9)
    orders = {"identity": np.arange(B), "reversed": np.arange(B)[::-1].copy(), "random": np.random.default_rng(10).permutation(B)}
    sample = np.sort(np.random.default_rng(11).choice(B, 256, replace=False))
    sample = np.union1d(sample, np.arange(24))   # the special headings and geometries
    bad = cut_filters(orc, case, sample)
    sample = np.setdiff1d(sample, bad)
    want = oracle_run(orc, case, sample)
    for kern in ("res2", "fast"):
        monkeypatch.setenv("NUSLAM_KERNEL", kern)
        res = {name: run_engine(cuda_lib, case, order=o) for name, o in orders.items()}
        x, s, seen, status, _ = res["identity"]
        assert not status.any()
        for name in ("reversed", "random"):
            xr, sr, seenr, str_, _ = res[name]
            diff = np.flatnonzero((x != xr).any(axis=1) | (s != sr).reshape(B, -1).any(axis=1))
            assert diff.size == 0, f"{kern}: {diff.size} filters change bits with the batch order ({name}), first {diff[:8]}"
            assert np.array_equal(seen, seenr) and np.array_equal(status, str_)
        ex = max(rel_max(x[b], want["x"][k]) for k, b in enumerate(sample))
        es = max(rel_max(s[b], want["sigma"][k]) for k, b in enumerate(sample))
        print(f"[pair position {kern}] 3 orders bit-identical; {sample.size} sampled filters vs oracle: x {ex:.2e}, Sigma {es:.2e}; "
              f"set aside at the cut: {bad}")
        assert np.array_equal(seen[sample], want["seen"])
        assert ex < TOL and es < TOL
