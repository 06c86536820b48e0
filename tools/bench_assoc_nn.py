#!/usr/bin/env python
"""Nearest-neighbour association (NUSLAM_OPT_NEAREST_NEIGHBOUR) against the reference's first-deciding-candidate rule.

(a) Quality: the config-4 scenario (synth.ekf_scenario, 12 landmarks, 12 markers per step, unknown ids, landmark_prior 100) in both
    geometries, FILTERS filters x STEPS steps on the oracle-order kernels: the reference's rule at its defaults (0.01 / 60) against
    NN | WRAP at 9.21 / 60. Reported: matched / ambiguous (-1) / new / exception ids over all steps, filters flagged MAP_FULL, and the
    pose RMSE and mean pose NEES of the last step (nuslam_ekf_error_stats [0], [2] over [3] filters; [6] flagged filters).
(b) Cost, variants alternated in one process on one card (CUDA events, steady state):
    - an oracle-order step at 131 072 filters x 12 landmarks (11 seen and measured, where both rules return the same ids) with
      unknown ids, options WRAP against WRAP | NN, both at 9.21 / 60;
    - a large-map association step (nuslam_ekf_step, ids = NULL, m = 12) on a built 4 096-landmark map (tools/bench_large_scan.py's
      map: tubes on a 0.6 m grid, 4 000 seen, small diagonal Sigma), options 0 against NN, both at 9.21 / 60.
Prints one JSON line; --out also writes it to a file."""
import argparse
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
from shermbot_navigation_b200 import nuslam, synth  # noqa: E402
from bench_large_scan import N as N_LARGE, SEEN, SPACING, card, trajectory  # noqa: E402

WRAP, NN = nuslam.OPT_WRAP_INNOVATION, nuslam.OPT_NEAREST_NEIGHBOUR
RULES = {"reference_0.01_60": (0, (0.01, 60.0)), "nn_wrap_9.21_60": (NN | WRAP, (9.21, 60.0))}


def classify(ids, seen_before):
    """ids [B, m] of one step in measurement order -> counts of matched / ambiguous / new / exception."""
    running = seen_before.copy()
    out = dict(matched=0, ambiguous=0, new=0, exception=0)
    for i in range(ids.shape[1]):
        k = ids[:, i]
        new = k > running
        out["new"] += int(new.sum())
        out["matched"] += int(((k > 0) & ~new).sum())
        out["ambiguous"] += int((k == -1).sum())
        out["exception"] += int((k == nuslam.ID_EXCEPTION).sum())
        running = np.where(new, k, running)
    return out


def quality(filters, steps, rules=RULES):
    import torch
    dev = torch.device("cuda")
    res = {}
    for geometry in ("benign", "adversarial"):
        sc = synth.ekf_scenario(filters, steps, n=12, seed=7, geometry=geometry, shuffle_order=True)
        for name, (opts, (amin, amax)) in rules.items():
            eng = nuslam.BatchedExtendedKalman(sc["robot0"], n_landmarks=12, Q=sc["Q"], R=sc["R"], mode="strict", options=opts,
                                               assoc_min=amin, assoc_max=amax, landmark_prior=100.0)
            counts = dict(matched=0, ambiguous=0, new=0, exception=0)
            for t in range(steps):
                seen = eng.getSeenLandmarks()
                ids = eng.step(sc["twists"][t], sc["z"][t], None, return_ids=True)
                for k, v in classify(ids, seen).items():
                    counts[k] += v
            pose = torch.tensor(np.ascontiguousarray(np.broadcast_to(sc["poses"][steps - 1], (filters, 3))), device=dev)
            st = eng.error_stats(truth_pose=pose).cpu().numpy()
            x, s, _, status = eng.get_state()
            nf = max(st[3], 1.0)
            # the same pose statistics over the filters still running (a filter frozen by MAP_FULL or SINGULAR keeps the pose of the scan
            # that froze it)
            live = (status & (nuslam.FILTER_MAP_FULL | nuslam.FILTER_SINGULAR)) == 0
            e = x[live, :3] - sc["poses"][steps - 1]
            e[:, 0] = synth.wrap_pi(e[:, 0])
            nees = np.einsum("bi,bi->b", e, np.linalg.solve(s[live][:, :3, :3], e[:, :, None])[:, :, 0])
            res[f"{geometry}/{name}"] = dict(counts, measurements=filters * steps * 12, map_full_filters=int(((status & nuslam.FILTER_MAP_FULL) != 0).sum()),
                                             singular_filters=int(((status & nuslam.FILTER_SINGULAR) != 0).sum()),
                                             truncated_filters=int(((status & nuslam.FILTER_ASSOC_TRUNCATED) != 0).sum()),
                                             rmse_position_m=float((st[0] / nf) ** 0.5), mean_pose_nees=float(st[2] / nf),
                                             stats_filters=float(st[3]), stats_bad_status=float(st[6]), live_filters=int(live.sum()),
                                             live_rmse_position_m=float(np.sqrt((e[:, 1:] ** 2).sum(axis=1).mean())) if live.any() else None,
                                             live_mean_pose_nees=float(nees.mean()) if live.any() else None)
            eng.close()
    return res


def timed(stream, reset, call, warmup, steps):
    import torch
    reset()
    for t in range(warmup):
        call(t)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    for t in range(warmup, warmup + steps):
        call(t)
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def cost_small(B, steps, warmup, rounds, n=12, seen=11, seed=9, variants=None):
    """Oracle-order step, 12 landmark slots, unknown ids, on a built map of 11 landmarks (a full map makes the reference's rule throw
    before it looks at a candidate) measured every step: they stand 0.86 m apart on a 1.5 m ring about the driven circle, Sigma small
    and diagonal. Every measurement lies well inside the gate of its own landmark and far beyond the new-landmark
    threshold of every other, so both rules return the same ids and apply the same updates (checked): the difference is the
    association alone. (On the config-4 scenario the reference's rule at 9.21 / 60 freezes most filters with MAP_FULL, and a frozen
    filter's step does no work.) D distinct filters tiled to B."""
    import torch
    dev = torch.device("cuda")
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    D, T = 256, warmup + steps
    g = np.random.default_rng(seed)
    a = 0.1 + 2 * np.pi * np.arange(seen) / seen
    lm = np.stack([1.5 * np.cos(a), 0.35 + 1.5 * np.sin(a)], axis=1)
    tw1 = synth.wheel_twists(T)
    poses = synth.true_trajectory(tw1)
    z = np.empty((T, D, seen, 2))
    for t in range(T):
        d = lm - poses[t, 1:3]
        zt = np.stack([np.hypot(d[:, 0], d[:, 1]), synth.wrap_pi(np.arctan2(d[:, 1], d[:, 0]) - poses[t, 0])], axis=1)
        for b in range(D):
            z[t, b] = zt[g.permutation(seen)] + g.normal(0, 1e-3, (seen, 2))
    z = [torch.tensor(z[t], device=dev).repeat(B // D, 1, 1) for t in range(T)]
    tw = [torch.tensor(np.tile(tw1[t], (B, 1)), device=dev) for t in range(T)]
    length = 3 + 2 * n
    x0 = torch.zeros((B, length), dtype=torch.float64, device=dev)
    x0[:, 3:3 + 2 * seen] = torch.tensor((lm + g.normal(0, 1e-4, lm.shape)).ravel(), device=dev)
    dg = torch.full((length,), 1e-4, dtype=torch.float64, device=dev)
    dg[:3] = 1e-6
    s0 = torch.diag_embed(dg).expand(B, length, length).contiguous()
    seen0 = torch.full((B,), seen, dtype=torch.int32, device=dev)
    status0 = torch.zeros(B, dtype=torch.int32, device=dev)
    variants = variants or {"wrap": WRAP, "wrap_nn": WRAP | NN}   # the first is the baseline of the ratios
    engs = {name: nuslam.BatchedExtendedKalman(np.zeros((B, 3)), n_landmarks=n, Q=1e-8 * np.eye(3), R=1e-3 * np.eye(2), mode="strict", options=opts,
                                               assoc_min=9.21, assoc_max=60.0, stream=stream.cuda_stream) for name, opts in variants.items()}
    ids = {}
    for name, e in engs.items():
        e.set_state(x0, s0, seen0, status0)
        ids[name] = [e.step(tw[t], z[t], None, return_ids=True) for t in range(T)]
        assert int(e.getStatus().max()) == 0
    base = next(iter(variants))
    same = all(torch.equal(u, v) for name in variants for u, v in zip(ids[base], ids[name]))
    matched = int(sum(int((u > 0).sum()) for u in ids[base]))
    out = {k: [] for k in variants}
    for _ in range(rounds):
        for name, e in engs.items():
            out[name].append(timed(stream, lambda: e.set_state(x0, s0, seen0, status0), lambda t: e.step(tw[t], z[t], None), warmup, steps))
    for e in engs.values():
        e.close()
    torch.cuda.set_stream(torch.cuda.default_stream(dev))
    return {"filters": B, "landmark_slots": n, "seen": seen, "m": seen, "ids_identical_between_rules": same, "matched": matched,
            "measurements": B * seen * T,
            "ms_per_step": {k: float(np.median(v)) for k, v in out.items()}, "ms_all_rounds": out,
            **{f"{k}_over_{base}": float(np.median(out[k]) / np.median(out[base])) for k in variants if k != base}}


def cost_large(steps, warmup, rounds, m=12, seed=5):
    """Large-map association step on a built 4 096-landmark map: m markers of the nearest tubes per step, ids = NULL."""
    import torch
    dev = torch.device("cuda")
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    side = int(np.ceil(np.sqrt(SEEN)))
    gx, gy = np.meshgrid(np.arange(side) * SPACING, np.arange(side) * SPACING)
    lm = (np.stack([gx.ravel(), gy.ravel()], axis=1)[:SEEN] - SPACING * (side - 1) / 2).copy()
    T = warmup + steps
    poses, tw = trajectory(T, (0.3, 0.01, -0.02))
    g = np.random.default_rng(seed)
    zs = []
    for p in poses:
        near = np.argsort(np.hypot(lm[:, 0] - p[1], lm[:, 1] - p[2]))[:m]
        d = lm[near] - p[1:3]
        z = np.stack([np.hypot(d[:, 0], d[:, 1]), synth.wrap_pi(np.arctan2(d[:, 1], d[:, 0]) - p[0])], axis=1) + g.normal(0, 1e-3, (m, 2))
        zs.append(torch.tensor(z[None], device=dev))
    tws = torch.tensor(tw[:, None], device=dev)
    length = 3 + 2 * N_LARGE
    x0 = torch.zeros((1, length), dtype=torch.float64, device=dev)
    x0[0, :3] = torch.tensor(poses[0], device=dev)
    x0[0, 3:3 + 2 * SEEN] = torch.tensor((lm + g.normal(0, 1e-4, lm.shape)).ravel(), device=dev)
    dg = torch.full((length,), 1e-4, dtype=torch.float64, device=dev)
    dg[:3] = 1e-6
    x = x0.clone()
    sig = torch.zeros((1, length, length), dtype=torch.float64, device=dev)
    seen = torch.empty(1, dtype=torch.int32, device=dev)
    status = torch.empty(1, dtype=torch.int32, device=dev)

    def reset():
        x.copy_(x0)
        sig.zero_()
        sig[0].diagonal().copy_(dg)
        seen.fill_(SEEN)
        status.zero_()
        torch.cuda.synchronize()

    variants = {"options_0": 0, "nn": NN}
    engs = {}
    for name, opts in variants.items():
        e = nuslam.BatchedExtendedKalman(poses[0][None], n_landmarks=N_LARGE, Q=1e-8 * np.eye(3), R=1e-3 * np.eye(2), options=opts, assoc_min=9.21,
                                         assoc_max=60.0, stream=stream.cuda_stream)
        e.bind_state(x, sig, seen, status)
        engs[name] = e
    outcomes = {}
    for name, e in engs.items():
        reset()
        ids = np.concatenate([e.step(tws[t], zs[t], None, return_ids=True).cpu().numpy() for t in range(T)])
        outcomes[name] = {"matched": int((ids > 0).sum()), "ambiguous": int((ids == -1).sum()), "other": int((ids <= -2).sum())}
        assert int(status[0]) == 0
    out = {k: [] for k in variants}
    for _ in range(rounds):
        for name, e in engs.items():
            out[name].append(timed(stream, reset, lambda t: e.step(tws[t], zs[t], None), warmup, steps))
    for e in engs.values():
        e.close()
    torch.cuda.set_stream(torch.cuda.default_stream(dev))
    return {"landmarks": N_LARGE, "seen": SEEN, "m": m, "batch": 1, "ms_per_step": {k: float(np.median(v)) for k, v in out.items()},
            "ms_all_rounds": out, "nn_over_options_0": float(np.median(out["nn"]) / np.median(out["options_0"])), "ids": outcomes}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--filters", type=int, default=4096)
    ap.add_argument("--quality-steps", type=int, default=60)
    ap.add_argument("--batch", type=int, default=131072)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", type=Path, default=None)
    a = ap.parse_args()
    out = {"workload": f"(a) config-4 scenario, {a.filters} filters x {a.quality_steps} steps, 12 landmarks, 12 markers per step, unknown ids, "
                       f"landmark_prior 100, oracle-order kernels; (b) cost, variants alternated over {a.rounds} rounds of {a.steps} steps after "
                       f"{a.warmup} (CUDA events)",
           "card": card(), "quality": quality(a.filters, a.quality_steps),
           "cost_oracle_order_step": cost_small(a.batch, a.steps, a.warmup, a.rounds),
           "cost_large_map_step": cost_large(a.steps, a.warmup, a.rounds)}
    line = json.dumps(out)
    print(line)
    if a.out is not None:
        a.out.parent.mkdir(parents=True, exist_ok=True)
        a.out.write_text(line + "\n")


if __name__ == "__main__":
    main()
