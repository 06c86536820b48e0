#!/usr/bin/env python
"""Large-map fused scan step (nuslam_ekf_scan_step in large-map mode): lidar scan -> markers -> associateLandmark against 4 000
landmarks -> delayed updates, one 4 096-landmark map per filter (len 8195, Sigma 537 MB, far more than the 126 MB L2).

The map is already built (landmarks at the tube positions plus 0.1 mm noise, small diagonal Sigma, `seen` = 4 000 of 4 096 slots:
a full map would make associateLandmark throw on every new candidate, as the reference does), so the steady state is timed: no
first touches, hence no oracle-order tails. The tubes stand on a 0.6 m grid; the robot creeps through it and every scan is
generated on the host beforehand (synth.simulate_scans, only the tubes within lidar range). Reported, per batch size:
  fused_ms      nuslam_ekf_scan_step with m = the largest marker count of the scans
  unfused_ms    nuslam_ekf_step(ids = NULL) on the same markers' z, m = each scan's own marker count (detection not included)
  fused_m16_ms  nuslam_ekf_scan_step with m = 16: the slots past a filter's count still cost their launches and rank columns
plus the association outcomes of the fused step against the true tubes, and the card's name and power limit. Prints one JSON line."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from shermbot_navigation_b200 import synth, tube_world  # noqa: E402

N, SEEN, SPACING = 4096, 4000, 0.6


def trajectory(T, start):
    """Poses (th, x, y) under predictEstimate's own motion model (slam_library.cpp:71-94) and the twists that produce them."""
    tw = np.tile(np.array([0.002, 0.005, 0.0]), (T, 1))
    tw[0] = 0.0   # twist t moves pose t - 1 to pose t: the first scan is taken where the filter starts
    poses = [np.array(start, dtype=np.float64)]
    for t in range(1, T):
        th, x, y = poses[-1]
        q = tw[t, 1] / tw[t, 0]
        th1 = th + tw[t, 0]
        poses.append(np.array([th1, x - q * np.sin(th) + q * np.sin(th1), y + q * np.cos(th) - q * np.cos(th1)]))
    return np.stack(poses), tw


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30)
        out["power_limit_and_max_sm_clock"] = q.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        out["power_limit_and_max_sm_clock"] = None
    return out


def run(B, steps, warmup, seed=5):
    import torch
    from shermbot_navigation_b200 import circle_fit, nuslam
    dev = torch.device("cuda")
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    side = int(np.ceil(np.sqrt(SEEN)))
    gx, gy = np.meshgrid(np.arange(side) * SPACING, np.arange(side) * SPACING)
    lm = (np.stack([gx.ravel(), gy.ravel()], axis=1)[:SEEN] - SPACING * (side - 1) / 2).copy()
    T = warmup + steps
    poses, tw = trajectory(T, (0.3, 0.01, -0.02))   # between four tubes (they stand at odd multiples of SPACING / 2)
    ranges = np.stack([synth.simulate_scans(p[None], lm[np.hypot(lm[:, 0] - p[1], lm[:, 1] - p[2]) < 1.2])[0] for p in poses])
    # the markers of every scan, through the engine's own detection (the same kernels the fused step runs)
    det = circle_fit.scan_detect(ranges, tube_world.MIN_RANGE, tube_world.MAX_RANGE, max_circles=32, want_cluster_of_beam=False)
    counts = det["n_circles"].clip(0)
    m_max = int(counts.max())
    assert 1 <= m_max <= 16, counts
    length = 3 + 2 * N
    g = np.random.default_rng(seed)
    Q, R = 1e-8 * np.eye(3), 1e-3 * np.eye(2)   # R: the node's; Q small -- with Q = 0.1 I every landmark within 2 m is ambiguous
    eng = nuslam.BatchedExtendedKalman(np.tile(poses[0], (B, 1)), n_landmarks=N, Q=Q, R=R, stream=stream.cuda_stream)
    x0 = torch.zeros((B, length), dtype=torch.float64, device=dev)
    x0[:, :3] = torch.tensor(poses[0], device=dev)
    x0[:, 3:3 + 2 * SEEN] = torch.tensor((lm + g.normal(0, 1e-4, lm.shape)).ravel(), device=dev)
    d = torch.full((length,), 1e-4, dtype=torch.float64, device=dev)
    d[:3] = 1e-6
    x = x0.clone()
    sig = torch.zeros((B, length, length), dtype=torch.float64, device=dev)
    seen = torch.empty(B, dtype=torch.int32, device=dev)
    status = torch.empty(B, dtype=torch.int32, device=dev)
    eng.bind_state(x, sig, seen, status)

    def reset():
        x.copy_(x0)
        sig.zero_()
        for b in range(B):
            sig[b].diagonal().copy_(d)
        seen.fill_(SEEN)
        status.zero_()
        torch.cuda.synchronize()

    rg = torch.tensor(np.repeat(ranges[:, None], B, axis=1), device=dev)                 # T x B x 360
    tws = torch.tensor(np.repeat(tw[:, None], B, axis=1), device=dev)                   # T x B x 3
    zs = []
    for t in range(T):
        z = nuslam.cartesian2polar(np.ascontiguousarray(det["circles"][t, :counts[t], :2]))
        zs.append(torch.tensor(np.repeat(z[None], B, axis=0), device=dev))

    def timed(call):
        reset()
        for t in range(warmup):
            call(t)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for t in range(warmup, T):
            call(t)
        e1.record(stream)
        torch.cuda.synchronize()
        assert int(status.max()) == 0
        return e0.elapsed_time(e1) / steps

    lo, hi = tube_world.MIN_RANGE, tube_world.MAX_RANGE
    res = {"B": B}
    # association outcomes of the fused step over every scan, against the tube each marker came from
    reset()
    matched = ambiguous = new = other = 0
    for t in range(T):
        _, _, ids = eng.scan_step(tws[t], rg[t], lo, hi, m_max, return_all=True)
        ids = ids.cpu().numpy()
        th, px, py = poses[t]
        for i in range(counts[t]):
            cx, cy = det["circles"][t, i, 0], det["circles"][t, i, 1]
            wx, wy = px + np.cos(th) * cx - np.sin(th) * cy, py + np.sin(th) * cx + np.cos(th) * cy
            truth = int(np.argmin(np.hypot(lm[:, 0] - wx, lm[:, 1] - wy))) + 1
            for b in range(B):
                k = int(ids[b, i])
                matched += k == truth
                ambiguous += k == -1
                new += k > SEEN
                other += k not in (truth, -1) and k <= SEEN
    res["ids"] = {"matched_true_tube": matched, "ambiguous_-1": ambiguous, "new": new, "other": other}
    res["fused_ms"] = timed(lambda t: eng.scan_step(tws[t], rg[t], lo, hi, m_max))
    res["unfused_ms"] = timed(lambda t: eng.step(tws[t], zs[t], None))
    res["fused_m16_ms"] = timed(lambda t: eng.scan_step(tws[t], rg[t], lo, hi, 16))
    res["fused_scans_per_s"] = 1e3 / res["fused_ms"]
    eng.close()
    del sig
    torch.cuda.empty_cache()
    return res, counts, m_max


def main():
    import argparse
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    a = ap.parse_args()
    out = {"workload": f"large-map fused scan step: {N} landmarks per filter (len {3 + 2 * N}, Sigma {8 * (3 + 2 * N) ** 2 / 1e6:.0f} MB), built map "
                       f"(seen {SEEN}), tubes on a {SPACING} m grid, host-generated scans, CUDA events over {a.steps} steps after {a.warmup}",
           "card": card(), "per_batch": []}
    for B in (1, 4):
        res, counts, m_max = run(B, a.steps, a.warmup)
        out["per_batch"].append(res)
    out["markers_per_scan"] = {"min": int(counts.min()), "mean": float(counts.mean()), "max": int(counts.max()), "fused_m": m_max}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
