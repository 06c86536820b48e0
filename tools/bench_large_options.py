#!/usr/bin/env python
"""What the opt-in variants cost in large-map mode: options = 0 against JOSEPH alone and against WRAP | JOSEPH | PRE_MOTION_JACOBIAN on a
built 4 096-landmark map (len 8195, Sigma 537 MB, far more than the 126 MB L2), one filter.

The map is already built (landmarks on a 0.6 m grid plus 0.1 mm noise, small diagonal Sigma, `seen` = 4 000 of 4 096 slots), so the
steady state is timed: no first touches, hence no oracle-order tails. The robot creeps through the grid; every scan measures the 12
landmarks nearest to it (z from the filter's own map estimate plus 0.1 mm / 0.1 mrad of noise, generated on the host beforehand).
Each option setting has its own handle and its own Sigma; they are timed alternately in the same process, with CUDA events:
  known_ms     nuslam_ekf_step with the 12 ids given: one delayed pass of 12 updates (rank 24; JOSEPH: symmetric, rank 48)
  unknown_ms   nuslam_ekf_step(ids = NULL): associateLandmark over 4 000 candidates per measurement inside the delayed pass
Then, in a separate profiled run (torch.profiler, CUDA activities only), the rank pass on its own in both forms: the plain pass
(k_large_rank_update_pipe) for options 0 and the symmetric pass (k_large_rank_update_sym) under JOSEPH, at rank 24 / 48, with the
bytes the pass has to move (one read and one write of Sigma, 16 len^2). The card's name and power limit are read in the same run.
Prints one JSON line; --out also writes it to a file."""
import json
import statistics
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
from bench_large_scan import card, trajectory  # noqa: E402

N, SEEN, SPACING, M = 4096, 4000, 0.6, 12
WRAP, JOSEPH, PRE_MOTION = 1, 2, 4
VARIANTS = {"options_0": 0, "options_2": JOSEPH, "options_7": WRAP | JOSEPH | PRE_MOTION}


def scans(T, g):
    """Landmark map, poses, twists, and per scan the ids and polar z of the M landmarks nearest to the robot."""
    side = int(np.ceil(np.sqrt(SEEN)))
    gx, gy = np.meshgrid(np.arange(side) * SPACING, np.arange(side) * SPACING)
    lm = (np.stack([gx.ravel(), gy.ravel()], axis=1)[:SEEN] - SPACING * (side - 1) / 2).copy()
    est = lm + g.normal(0, 1e-4, lm.shape)   # the filter's map
    poses, tw = trajectory(T, (0.3, 0.01, -0.02))
    ids = np.zeros((T, M), dtype=np.int32)
    z = np.zeros((T, M, 2))
    for t, (th, px, py) in enumerate(poses):
        near = np.argsort(np.hypot(est[:, 0] - px, est[:, 1] - py))[:M]
        ids[t] = near + 1
        dx, dy = est[near, 0] - px, est[near, 1] - py
        z[t, :, 0] = np.hypot(dx, dy) + g.normal(0, 1e-4, M)
        z[t, :, 1] = np.arctan2(np.sin(np.arctan2(dy, dx) - th), np.cos(np.arctan2(dy, dx) - th)) + g.normal(0, 1e-4, M)
    return est, poses, tw, ids, z


def main():
    import argparse
    import torch
    from shermbot_navigation_b200 import nuslam
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5, help="alternations of the option settings; the median is reported")
    ap.add_argument("--out", help="also write the JSON line to this file")
    a = ap.parse_args()
    dev = torch.device("cuda")
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    g = np.random.default_rng(5)
    T = a.warmup + a.steps
    est, poses, tw, ids_np, z_np = scans(T, g)
    length = 3 + 2 * N
    Q, R = 1e-8 * np.eye(3), 1e-3 * np.eye(2)
    x0 = torch.zeros((1, length), dtype=torch.float64, device=dev)
    x0[0, :3] = torch.tensor(poses[0], device=dev)
    x0[0, 3:3 + 2 * SEEN] = torch.tensor(est.ravel(), device=dev)
    d = torch.full((length,), 1e-4, dtype=torch.float64, device=dev)
    d[:3] = 1e-6
    tws = torch.tensor(tw[:, None], device=dev)
    zs = torch.tensor(z_np[:, None], device=dev)
    ids = torch.tensor(ids_np[:, None], device=dev)
    handles = {}
    for name, opt in VARIANTS.items():
        eng = nuslam.BatchedExtendedKalman(poses[0][None], n_landmarks=N, Q=Q, R=R, options=opt, stream=stream.cuda_stream)
        st = (x0.clone(), torch.zeros((1, length, length), dtype=torch.float64, device=dev), torch.empty(1, dtype=torch.int32, device=dev),
              torch.empty(1, dtype=torch.int32, device=dev))
        eng.bind_state(*st)
        handles[name] = (eng, st)

    def reset(st):
        x, sig, seen, status = st
        x.copy_(x0)
        sig.zero_()
        sig[0].diagonal().copy_(d)
        seen.fill_(SEEN)
        status.zero_()
        torch.cuda.synchronize()

    def timed(name, known):
        eng, st = handles[name]
        reset(st)
        call = (lambda t: eng.step(tws[t], zs[t], ids[t])) if known else (lambda t: eng.step(tws[t], zs[t], None))
        for t in range(a.warmup):
            call(t)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for t in range(a.warmup, T):
            call(t)
        e1.record(stream)
        torch.cuda.synchronize()
        assert int(st[3][0]) == 0, (name, known, int(st[3][0]))
        return e0.elapsed_time(e1) / a.steps

    # association outcomes of the unknown-correspondence step, per variant (every measurement should find its landmark)
    outcomes = {}
    for name in VARIANTS:
        eng, st = handles[name]
        reset(st)
        got = np.stack([eng.step(tws[t], zs[t], None, return_ids=True)[0].cpu().numpy() for t in range(T)])
        outcomes[name] = {"matched": int((got == ids_np).sum()), "of": int(got.size)}
        if VARIANTS[name] & JOSEPH:
            s = st[1][0]
            outcomes[name]["sigma_exactly_symmetric"] = bool(torch.equal(s, s.T))
    samples = {name: {"known_ms": [], "unknown_ms": []} for name in VARIANTS}
    for _ in range(a.rounds):
        for known in (True, False):
            for name in VARIANTS:
                samples[name]["known_ms" if known else "unknown_ms"].append(timed(name, known))
    res = {name: {k: statistics.median(v) for k, v in s.items()} for name, s in samples.items()}
    for name in VARIANTS:
        res[name]["samples"] = samples[name]
    # the rank pass on its own, from a profiled run of the known-id step
    from torch.profiler import ProfilerActivity, profile
    passes = {}
    for name in VARIANTS:
        eng, st = handles[name]
        reset(st)
        for t in range(a.warmup):
            eng.step(tws[t], zs[t], ids[t])
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for t in range(a.warmup, min(T, a.warmup + 30)):
                eng.step(tws[t], zs[t], ids[t])
            torch.cuda.synchronize()
        for ev in prof.key_averages():
            if "k_large_rank_update" in ev.key:
                total = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
                us = total / ev.count
                passes[name] = {"kernel": ev.key.split("(")[0], "launches": ev.count, "us_per_pass": us,
                                "GB_per_s_of_16_len2": 16 * length * length / (us * 1e-6) / 1e9}
    out = {"workload": f"large-map step, built map: {N} landmarks (len {length}, Sigma {8 * length * length / 1e6:.0f} MB), seen {SEEN}, B = 1, "
                       f"m = {M} per scan (known ids, or associateLandmark over {SEEN} candidates), options 0, 2 and 7 alternated over "
                       f"{a.rounds} rounds, CUDA events over {a.steps} steps after {a.warmup}; rank-pass times from torch.profiler",
           "card": card(), "per_variant": res, "rank_pass": passes, "association": outcomes}
    for name in ("options_2", "options_7"):
        for k in ("known_ms", "unknown_ms"):
            out[f"{name}_over_default_{k}"] = res[name][k] / res["options_0"][k]
    line = json.dumps(out)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")
    for eng, _ in handles.values():
        eng.close()


if __name__ == "__main__":
    main()
