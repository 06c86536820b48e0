"""Generate the committed fixtures under tests/golden/.

  NUSLAM_REFERENCE=<checkout> python tests/golden/make_golden.py          ekf_golden.npz from oracle/_ref (the unmodified reference)
  [NUSLAM_REFERENCE=<checkout>] python tests/golden/make_golden.py parity  parity_golden.npz from oracle.best()

ekf_golden.npz: the tests check the oracle restatement and the CUDA path against it without needing the reference.
parity_golden.npz: the inputs and outputs of the bitwise parity tests of tests/test_oracle.py (EKF runs of both geometries with and
without known ids, single calls, a sample of the scan batches, the edge scans, the simulator's lidar and main loop). It records which
oracle flavour wrote it (`flavour`); the tests hold every flavour present to it bit for bit, so the restatement keeps being checked
where the reference is absent, and the reference, where present, confirms the stored arrays.
"""
import hashlib
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent.parent
sys.path.insert(0, str(ROOT))

import oracle  # noqa: E402
from shermbot_navigation_b200 import synth  # noqa: E402


def main():
    oracle.build()
    ref = oracle.load("ref")
    assert ref.flavour == "reference"
    sc = synth.ekf_scenario(4, 25, n=12, seed=2024)
    out = dict(n=12, robot0=sc["robot0"], map0=sc["map0"], Q=sc["Q"], R=sc["R"], twists=sc["twists"], z=sc["z"], ids=sc["ids"])
    for tag, ids in (("known", sc["ids"]), ("unknown", None)):
        r = ref.ekf_run(12, sc["robot0"], sc["map0"], sc["Q"], sc["R"], sc["twists"], sc["z"], ids, trace=True)
        for k in ("x", "sigma", "seen", "ids_out", "trace"):
            out[f"{tag}_{k}"] = r[k]
        # the state after the first step (every landmark's first touch lies behind it): the warm start from which a GPU path can be
        # held to 1e-9 without sharing the reference's libm (SURVEY.md 7.3, gate L1)
        r1 = ref.ekf_run(12, sc["robot0"], sc["map0"], sc["Q"], sc["R"], sc["twists"][:1], sc["z"][:1], None if ids is None else ids[:1])
        for k in ("x", "sigma", "seen"):
            out[f"{tag}_{k}1"] = r1[k]
    s = synth.scan_scenario(64, seed=4242, noise_sigma=0.001)
    sd = ref.scan_detect_batch(s["ranges"], s["min_range"], s["max_range"])
    out["ranges"] = s["ranges"]
    out["scan_cluster_of_beam"] = sd["cluster_of_beam"]
    out["scan_n_clusters"] = sd["n_clusters"]
    out["scan_n_circles"] = sd["n_circles"]
    out["scan_circles"] = sd["circles"]
    p = Path(__file__).parent / "ekf_golden.npz"
    np.savez_compressed(p, **out)
    print("wrote", p, p.stat().st_size, "bytes")


# the inputs of the parity tests (tests/test_oracle.py uses the same constants)
EKF_VARIANTS = (("benign", True), ("adversarial", True), ("benign", False), ("adversarial", False))
SCAN_SAMPLE = 256          # of the 1 500 scans of each noise level
LIDAR_POSES = 400
WORLD_T = 300
WORLD_DT = 1e-9 * 20000000.0   # the node's loop period at 50 Hz as its clock returns it (oracle/shim_ros ros::Duration::toSec)


def sha256(a):
    """Digest of an array's bytes: the 40-step state traces are held bit for bit without storing them (they do not compress)."""
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def ekf_tag(geometry, ids_known):
    return f"ekf_{geometry}_{'known' if ids_known else 'unknown'}"


def scan_sample(noise):
    return np.sort(np.random.default_rng(31).choice(1500, SCAN_SAMPLE, replace=False)), synth.scan_scenario(1500, seed=31, noise_sigma=noise)


def lidar_poses(tubes):
    """Robot configurations around the six reference tubes, none inside a tube (check_collision would move the robot first)."""
    rng = np.random.default_rng(5)
    out = []
    while len(out) < LIDAR_POSES:
        x, y = rng.uniform(-1.2, 1.2, 2)
        th = rng.uniform(-7.0, 7.0)
        if np.hypot(*(tubes - [x, y]).T).min() > 0.0381 + 1e-6:
            out.append((x, y, th))
    return np.array(out)


def world_drive(tubes):
    """Commanded twists of the main-loop drive: turn towards tube 1, run into it, slide, keep turning."""
    cmd = np.zeros((WORLD_T, 3))
    cmd[:, 1] = 0.22
    cmd[:, 0] = 0.3 * np.sin(np.arange(WORLD_T) / 17.0)
    cmd[:40, 0] = np.arctan2(tubes[0, 1], tubes[0, 0]) / (40 * 0.02)
    cmd[:40, 1] = 0.0
    return cmd


def single_calls(L):
    """associate / init_landmark / zhat / H / update one call at a time on one filter (n = 6): every intermediate output."""
    sc = synth.ekf_scenario(1, 6, n=6, seed=5)
    f = L.ekf(6, sc["robot0"][0], sc["map0"][0], sc["Q"], sc["R"])
    ids, zhat, H = np.zeros((6, 6)), np.full((6, 6, 2), np.nan), np.full((6, 6, 2, 15), np.nan)
    x, s, seen = np.zeros((6, 6, 15)), np.zeros((6, 6, 15, 15)), np.zeros((6, 6))
    for t in range(6):
        f.predict(*sc["twists"][t, 0])
        for i in range(6):
            z = sc["z"][t, 0, i]
            ids[t, i] = j = f.associate(z)
            if j > 0:
                if t == 0:
                    f.init_landmark(z, j)
                zhat[t, i], H[t, i] = f.zhat(j), f.H(j)
                f.update(z, j)
            x[t, i], s[t, i], seen[t, i] = f.get()
    return dict(ids=ids, zhat=zhat, H=H, x=x, sigma=s, seen=seen)


def world_outputs(o, tubes):
    poses = lidar_poses(tubes)
    lidar = np.stack([o.world_step(np.array([[0.16, 0.033, x, y, th, 0.0, 0.0, 0.0, 0.0]]), np.zeros(3), None, 0.0, tubes, 0.0381, 1e-9, 1.0)[0]
                      for x, y, th in poses])
    cmd = world_drive(tubes)
    w = np.array([[0.16, 0.033, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0]])
    run_poses, run_joints, run_scans = np.empty((WORLD_T, 3)), np.empty((WORLD_T, 2)), np.empty((WORLD_T, 360), dtype=np.float32)
    for t in range(WORLD_T):
        run_scans[t] = o.world_step(w, cmd[t], np.array([0.0, 0.0, 0.02, 0.02]), WORLD_DT, tubes, 0.0381, 0.08, 1.0)[0]
        run_poses[t], run_joints[t] = w[0, 2:5], w[0, 7:9]
    return dict(lidar_poses=poses, lidar=lidar, run_poses=run_poses, run_joints=run_joints, run_scans=run_scans)


def parity():
    oracle.build()
    L = oracle.best()
    out = dict(flavour=np.array(L.flavour))
    for geometry, ids_known in EKF_VARIANTS:
        sc = synth.ekf_scenario(6, 40, geometry=geometry, seed=99)
        r = L.ekf_run(12, sc["robot0"], sc["map0"], sc["Q"], sc["R"], sc["twists"], sc["z"], sc["ids"] if ids_known else None, trace=True)
        for k in ("x", "sigma", "seen", "status", "ids_out"):
            out[f"{ekf_tag(geometry, ids_known)}_{k}"] = r[k]
        out[f"{ekf_tag(geometry, ids_known)}_trace_sha256"] = np.array(sha256(r["trace"]))
    for k, v in single_calls(L).items():
        out[f"calls_{k}"] = v
    for noise in (0.0, 0.002):
        idx, s = scan_sample(noise)
        sd = L.scan_detect_batch(s["ranges"][idx], s["min_range"], s["max_range"])
        for k, v in sd.items():
            out[f"scan{noise}_{k}"] = v
    for k, v in L.scan_detect_batch(synth.edge_scans(), 0.05, 1.0).items():
        out[f"edge_{k}"] = v
    out.update(world_outputs(L, np.ascontiguousarray(synth.TUBES[:6], dtype=np.float64)))
    p = Path(__file__).parent / "parity_golden.npz"
    np.savez_compressed(p, **out)
    print("wrote", p, p.stat().st_size, "bytes from", L.flavour)


if __name__ == "__main__":
    parity() if sys.argv[1:] == ["parity"] else main()
