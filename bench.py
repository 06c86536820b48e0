#!/usr/bin/env python
"""bench.py -- headline benchmark of the batched EKF-SLAM hot path (BASELINE.json metric).

Metric: EKF predict+update steps/sec at 64K filters x 12 landmarks (fp64, known correspondence), reported
as filter-steps/s (one filter-step = 1 predict + 12 sequential updates = one iteration of
nuslam/src/slam.cpp:262-319 with 12 markers) and as a fraction of the measured HBM roofline.

  python bench.py --gpus N --steps K --warmup W          # our arm (one rank per GPU under torchrun)
  python bench.py --impl reference --steps K --warmup W  # the reference's CPU implementation, host cores

One JSON line on stdout (rank 0). See DESIGN.md "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

N_LANDMARKS = 12
FILTERS_PER_GPU = 65536
LEN = 3 + 2 * N_LANDMARKS
# algorithmic bytes per filter-step (SURVEY.md 8d): read x 216 + Sigma 5832 + u 16 + z 192 + ids 48, write x 216 + Sigma 5832
# known-correspondence kernels at 12 landmarks (NUSLAM_KERNEL selects; default: the resident pair kernel, csrc/ekf_static.cuh)
KERNEL_NAMES = {"res2": "k_ekf_res2_step<12, 3> (two filters per warp, both Sigma images resident in shared memory, ekf_res2.cuh)",
                "res": "k_ekf_res_step<12, 2> (one filter per warp, Sigma resident in shared memory, ekf_res.cuh)",
                "fas": "k_ekf_fast_step<12, BULK> (register fragments, ekf_fast.cuh)", "pair": "k_ekf_pair_step<12> (ekf_pair.cuh)",
                "sta": "k_ekf_static_step<12> (ekf_static.cuh)"}
BYTES_PER_FILTER_STEP = 2 * 8 * (LEN + LEN * LEN) + 16 + 20 * N_LANDMARKS
# filters sampled by --dump-outputs: x, Sigma, seen and status of 8192 filters come to 50 MB of float64
DUMP_FILTERS = 8192
METRIC = "EKF predict+update filter-steps/s (64K filters x 12 landmarks per GPU, fp64, known correspondence)"
UNIT = "filter-steps/s"


def hbm_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock, power and throttle reasons sampled DURING the timed region (NVML every ~4 ms in a thread; nvidia-smi as fallback)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap", 0x80: "hw_power_brake"}

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.stop_flag = threading.Event()
        self.thread = None
        self.nvml = None
        self.handle = None
        self.max_sm = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _read_nvml(self):
        n = self.nvml
        sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
        try:
            pw = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
        except Exception:
            pw = float("nan")
        try:
            rs = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
        except Exception:
            try:
                rs = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            except Exception:
                rs = 0
        return sm, pw, rs

    def _read_smi(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active"
        out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip().split(",")
        self.max_sm = float(out[1])
        return float(out[0]), float(out[2]), int(out[3].strip(), 16)

    def _run(self):
        while not self.stop_flag.is_set():
            try:
                self.samples.append(self._read_nvml() if self.nvml else self._read_smi())
            except Exception:
                pass
            time.sleep(0.004)

    def stop(self):
        self.stop_flag.set()
        if self.thread:
            self.thread.join(timeout=5)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_sm, "reasons": ["no samples"]}
        sm = [v[0] for v in self.samples]
        pw = [v[1] for v in self.samples if v[1] == v[1]]
        bits = 0
        for v in self.samples:
            bits |= v[2]
        reasons = sorted(nm for b, nm in self.REASONS.items() if bits & b)
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": self.max_sm, "power_w_max": float(max(pw)) if pw else None,
                "samples": len(sm), "reasons": reasons, "source": "nvml" if self.nvml else "nvidia-smi"}


def make_inputs_device(torch, dev, B, steps_total, seed, radius=0.20):
    """Synthetic config-2 inputs generated on the device (data: synthetic): robot on the reference circle
    (d_theta 0.02, dx 0.007 per step), 12 landmarks on the benign ring, exact range/bearing + N(0, 0.01^2)."""
    from shermbot_navigation_b200 import synth
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    tw1 = synth.wheel_twists(steps_total + 1, first_step_straight=True)
    poses = synth.true_trajectory(tw1)
    lm = synth.landmark_ring(N_LANDMARKS, radius)
    dxl = lm[None, :, 0] - poses[:, None, 1]
    dyl = lm[None, :, 1] - poses[:, None, 2]
    rng_true = torch.tensor(np.sqrt(dxl * dxl + dyl * dyl), device=dev)                      # (T, n)
    brg_true = torch.tensor(synth.wrap_pi(np.arctan2(dyl, dxl) - poses[:, None, 0]), device=dev)
    robot0 = (torch.randn((B, 3), generator=g, device=dev, dtype=torch.float64) * 0.01).cpu().numpy()
    twists = torch.tensor(tw1, device=dev)[:, None, :].expand(-1, B, -1).contiguous()           # (T, B, 3)
    ids = torch.arange(1, N_LANDMARKS + 1, device=dev, dtype=torch.int32)[None, :].expand(B, -1).contiguous()

    def z_of(t):
        noise = torch.randn((B, N_LANDMARKS, 2), generator=g, device=dev, dtype=torch.float64) * 0.01
        z = torch.empty((B, N_LANDMARKS, 2), device=dev, dtype=torch.float64)
        z[..., 0] = rng_true[t][None, :] + noise[..., 0]
        b = brg_true[t][None, :] + noise[..., 1]
        z[..., 1] = torch.atan2(torch.sin(b), torch.cos(b))
        return z

    return robot0, twists, ids, z_of


def bind_to_gpu_numa_node(index: int):
    """Run this rank's host threads on the CPUs next to its GPU (NVML's ideal affinity), so that the page-locked staging buffers of
    the end-to-end leg are allocated on that NUMA node and their DMA does not cross the socket link. Best effort; returns a note."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        before = len(os.sched_getaffinity(0))
        pynvml.nvmlDeviceSetCpuAffinity(h)
        after = len(os.sched_getaffinity(0))
        return f"nvml ideal affinity: {after} of {before} cpus"
    except Exception as e:   # containers often forbid it: not an error
        return f"unchanged ({type(e).__name__})"


def adversarial_leg(torch, nuslam, dev, local, stream, B, mode, seed, steps=12):
    """The same kernel on the ADVERSARIAL ring (landmarks on a 0.60 m ring around the robot's circle: bearings all around the robot, so the
    innovation's atan2 - theta leaves (-pi, pi] for half of the measurements and the conditional wraps of the update are taken). A separate
    engine, first-touch step + 3 warm-up steps untimed, `steps` steps between two CUDA events. Returns ms per step."""
    robot0, twists, ids, z_of = make_inputs_device(torch, dev, B, steps + 6, seed=seed, radius=0.60)
    eng = nuslam.BatchedExtendedKalman(robot0, None, n_landmarks=N_LANDMARKS, mode=mode, device=local, stream=stream.cuda_stream)
    zs = [z_of(t) for t in range(steps + 4)]
    for t in range(4):
        eng.step(twists[t], zs[t], ids)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for t in range(4, 4 + steps):
        eng.step(twists[t], zs[t], ids)
    e1.record(stream)
    torch.cuda.synchronize(dev)
    x, _, _, status = eng.get_state()
    bad = int((status != 0).sum()) + int((~np.isfinite(x)).any(axis=1).sum())
    eng.close()
    return e0.elapsed_time(e1) / steps, bad


def config_dict(world):
    """The workload description shared verbatim by both arms (the driver compares them)."""
    return {"workload": "BASELINE.json configs[1]: batched 64K independent EKF filters x 12 landmarks, known correspondence, fp64",
            "filters_per_gpu": FILTERS_PER_GPU, "landmarks": N_LANDMARKS, "state_len": LEN,
            "l2": f"inputs larger than L2: filter state {FILTERS_PER_GPU * (LEN + LEN * LEN) * 8 / 1e6:.0f} MB per GPU is streamed every step (L2 126 MB)",
            "parallelism": f"filters sharded {world}x, no data-path collective; final NCCL all_gather of states + all_reduce of error statistics"}


def dump_outputs(out_dir, state):
    """--dump-outputs: the state the last timed step left (x, Sigma [row, col], seen, status, as BatchedExtendedKalman.get_state
    returns it) for a fixed, seeded sample of DUMP_FILTERS filters, whose indices go to filters.npy; all as float64 .npy files."""
    x, sigma, seen, status = state
    B = x.shape[0]
    idx = np.sort(np.random.default_rng(0).choice(B, size=min(B, DUMP_FILTERS), replace=False))
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in (("filters", idx), ("x", x[idx]), ("sigma", sigma[idx]), ("seen", seen[idx]), ("status", status[idx])):
        np.save(out_dir / f"{name}.npy", np.ascontiguousarray(a, dtype=np.float64))


def e2e_leg(eng, torch, dist, world, dev, B, twists, zs, ids, t, K, dry, packed):
    """The same metric through the public host-buffer API: pinned host buffers, every step copies its inputs host -> device and its
    resulting state vector device -> host inside the timed region, three steps in flight.
      packed = True : BatchedExtendedKalman.step_async_packed (nuslam_ekf_step_async_packed): ONE packed buffer [twists | z] per step,
                      the known-correspondence ids kept on the device by set_ids (they are the same every step)
      packed = False: BatchedExtendedKalman.step_async (nuslam_ekf_step_async): three buffers (twists, z, ids) per step
    dry = True: the same calls with the kernels left out -- the ceiling the host side allows for that path."""
    nbuf = 3
    h_x = [torch.empty((B, LEN), dtype=torch.float64).pin_memory() for _ in range(nbuf)]
    if packed:
        total, off_z, _ = eng.packed_layout(N_LANDMARKS, False)
        h_p = [torch.empty(total, dtype=torch.uint8).pin_memory() for _ in range(nbuf)]
        for k in range(nbuf):
            h_p[k][:off_z].view(torch.float64).view(B, 3).copy_(twists[t + k])
            h_p[k][off_z:].view(torch.float64).view(B, N_LANDMARKS, 2).copy_(zs[t + k])
        eng.set_ids(ids)
        step = lambda k: eng.step_async_packed(h_p[k % nbuf].numpy(), N_LANDMARKS, eng.IDS_CACHED, h_x[k % nbuf].numpy())
    else:
        h_tw = [torch.empty((B, 3), dtype=torch.float64).pin_memory() for _ in range(nbuf)]
        h_z = [torch.empty((B, N_LANDMARKS, 2), dtype=torch.float64).pin_memory() for _ in range(nbuf)]
        h_ids = ids.cpu().pin_memory()
        for k in range(nbuf):
            h_tw[k].copy_(twists[t + k])
            h_z[k].copy_(zs[t + k])
        step = lambda k: eng.step_async(h_tw[k % nbuf].numpy(), h_z[k % nbuf].numpy(), h_ids.numpy(), h_x[k % nbuf].numpy())
    torch.cuda.synchronize(dev)
    eng.async_dry_run(dry)
    for k in range(6):   # warm the host path (staging buffers, streams, events)
        step(k)
    eng.wait_async()
    if world > 1:
        dist.barrier()
    checksum = 0.0
    t0 = time.perf_counter()
    for k in range(K):
        step(k)
        # the host consumes the result of the step that has just left the pipeline (three calls back): robot pose of filter 0
        if k >= nbuf:
            checksum += float(h_x[k % nbuf][0, 1])
    eng.wait_async()
    secs = time.perf_counter() - t0
    eng.async_dry_run(False)
    tt = torch.tensor([secs], device=dev, dtype=torch.float64)
    if world > 1:
        dist.barrier()
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    return world * B * K / float(tt.item())


def run_ours(args):
    import torch
    import torch.distributed as dist
    from shermbot_navigation_b200 import nuslam

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the engine has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, K, W = args.filters, args.steps, args.warmup
    total_steps = W + K + 6
    robot0, twists, ids, z_of = make_inputs_device(torch, dev, B, total_steps, seed=1234 + rank)
    stream = torch.cuda.Stream(dev)          # a real (non-NULL) stream shared by torch events and the engine's launches
    torch.cuda.set_stream(stream)
    eng = nuslam.BatchedExtendedKalman(robot0, None, n_landmarks=N_LANDMARKS, mode=args.mode, device=local, stream=stream.cuda_stream)
    # state lives in torch tensors so that the final gather is a plain NCCL collective on them
    xs = torch.zeros((B, LEN), device=dev, dtype=torch.float64)
    sig = torch.zeros((B, LEN, LEN), device=dev, dtype=torch.float64)
    seen = torch.zeros(B, device=dev, dtype=torch.int32)
    status = torch.zeros(B, device=dev, dtype=torch.int32)
    x0, s0, n0, st0 = eng.get_state()
    xs.copy_(torch.from_numpy(x0))
    sig.copy_(torch.from_numpy(np.ascontiguousarray(np.transpose(s0, (0, 2, 1)))))
    torch.cuda.synchronize(dev)
    eng.bind_state(xs, sig, seen, status)
    zs = [z_of(t) for t in range(total_steps)]          # resident in HBM before the timed region
    torch.cuda.synchronize(dev)

    # step 0 touches every landmark for the first time (strict arithmetic inside the kernel); then W warm-up steps
    t = 0
    eng.step(twists[t], zs[t], ids)
    t += 1
    for _ in range(W):
        eng.step(twists[t], zs[t], ids)
        t += 1
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # the K timed steps go through the C ABI directly (nuslam_ekf_step on device pointers resolved beforehand; the engine runs on this
    # stream, so no event ordering is needed): the Python wrapper's ~40 us per call would otherwise sit between the start event and the
    # first kernel -- 0.7 % of a 20-step timed region -- without being part of any step
    step_fn = nuslam.lib().nuslam_ekf_step
    handle, ids_ptr, m_meas = eng._h, ids.data_ptr(), int(zs[0].shape[1])
    arg_ptrs = [(twists[t + k].data_ptr(), zs[t + k].data_ptr()) for k in range(K)]
    rc_sum = 0
    torch.cuda.synchronize(dev)
    ev0.record(stream)
    for pt, pz in arg_ptrs:
        rc_sum |= step_fn(handle, pt, pz, ids_ptr, m_meas, None, nuslam.NUSLAM_DEVICE)
    ev1.record(stream)
    torch.cuda.synchronize(dev)
    t += K
    if rc_sum:
        raise RuntimeError(f"nuslam_ekf_step failed inside the timed region: {nuslam.lib().nuslam_last_error().decode()}")
    if world > 1:
        dist.barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    ms_t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
    ms_max = float(ms_t.item())
    if args.dump_outputs and rank == 0:   # after the clock sampler has stopped: the copy and the writes are not part of the timed region
        dump_outputs(Path(args.dump_outputs), eng.get_state())
    # K6: the shard's error statistics, reduced on the device (truth: the trajectory the measurements were generated from)
    from shermbot_navigation_b200 import synth
    poses = synth.true_trajectory(synth.wheel_twists(total_steps + 1, first_step_straight=True))
    truth_pose = torch.tensor(np.ascontiguousarray(np.broadcast_to(poses[t - 1], (B, 3))), device=dev)
    truth_map = torch.tensor(np.ascontiguousarray(synth.landmark_ring(N_LANDMARKS, 0.20)), device=dev)
    stats = eng.error_stats(truth_pose=truth_pose, truth_map=truth_map)
    bad_nonfinite = (~torch.isfinite(xs)).any(dim=1).sum().to(torch.float64)

    # ---- the adversarial ring, timed once beside the benign number (rank 0's shard) ----
    adv_ms, adv_bad = (None, 0)
    if not args.no_extras:
        adv_ms, adv_bad = adversarial_leg(torch, nuslam, dev, local, stream, B, args.mode, seed=99 + rank)

    # ---- end to end through the public API with HOST buffers, and the copy-only ceiling of the same path ----
    Ke = max(3, min(K, args.e2e_steps))
    leg = lambda dry, packed: e2e_leg(eng, torch, dist, world, dev, B, twists, zs, ids, t, Ke, dry=dry, packed=packed)
    e2e_runs = [leg(False, True) for _ in range(max(1, args.e2e_repeats))]
    e2e_value = float(np.median(e2e_runs))
    ceiling = leg(True, True)
    sep_value, sep_ceiling = leg(False, False), leg(True, False)
    h2d = B * (3 * 8 + N_LANDMARKS * 2 * 8)
    h2d_sep = h2d + B * N_LANDMARKS * 4
    d2h = B * LEN * 8

    # ---- the only communication of the whole run: gather final states + error statistics (NCCL over NVLink) ----
    if world > 1:
        from shermbot_navigation_b200 import shard
        gathered = shard.gather_states(xs, world * B)
        assert gathered.shape == (world * B, LEN)
        stats = shard.allreduce_stats(stats)
        bad_nonfinite = shard.allreduce_stats(bad_nonfinite.reshape(1)).reshape(())
    st = dict(zip(nuslam.BatchedExtendedKalman.STATS, [float(v) for v in stats.cpu().numpy()]))
    bad = int(st["bad_status"]) + int(bad_nonfinite.item())

    out = None
    if rank == 0:
        peak, peak_src = hbm_peak()
        per_launch_s = ms_max / 1e3 / K
        achieved = B * BYTES_PER_FILTER_STEP / per_launch_s / 1e9
        traffic = None
        prof = ROOT / "profiles" / "ncu_summary.json"
        if prof.exists():
            try:
                traffic = json.loads(prof.read_text()).get("ekf_step_traffic_bytes_per_launch")
            except Exception:
                pass
        value = world * B * K / (ms_max / 1e3)
        nf = max(st["filters"], 1.0)
        # FAST mode: the step kernel + the oracle-order list kernel, which the step kernel tail-launches itself only when a filter was
        # handed over (first touches: none in the timed steady state) when the library is built with device-side launches
        launches = 2 if (args.mode == "fast" and not nuslam.lib().nuslam_tail_launch()) else 1
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": config_dict(world),
            "details": {"mode": args.mode, "filters_this_run": B, "batched_steps_per_s": value / (world * B) if B else None,
                        "adversarial_ring": {"ms_per_step": adv_ms, "bad_filters": adv_bad,
                                             "note": "same kernel, landmarks on a 0.60 m ring around the robot's path (bearings wrap for half of the "
                                                     "measurements), rank 0's shard, 12 steps"}},
            "clocks": clocks, "gpu_launches": launches * K, "bad_filters": bad,
            "stats": {"reduced": "k_error_stats per rank" + (" + NCCL all_reduce(sum)" if world > 1 else ""), "filters": st["filters"],
                      "rmse_position_m": (st["sq_position_error"] / nf) ** 0.5, "rmse_heading_rad": (st["sq_heading_error"] / nf) ** 0.5,
                      "mean_nees_3dof": st["nees"] / nf, "rmse_landmark_m": (st["sq_landmark_error"] / max(st["landmarks"], 1.0)) ** 0.5,
                      "bad_status": st["bad_status"]},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": Ke,
                    "runs": e2e_runs, "copy_ceiling": ceiling, "frac_of_copy_ceiling": e2e_value / ceiling if ceiling else None,
                    "copy_ceiling_note": "the same calls with the kernels left out (nuslam_ekf_async_dry_run): identical copies, streams and events",
                    "api": "BatchedExtendedKalman.step_async_packed (nuslam_ekf_step_async_packed): one pinned packed buffer [twists | z] per step "
                           "(one H2D copy), known-correspondence ids kept on the device by set_ids, fused step, D2H of the FULL state vector per step, "
                           "3 steps in flight",
                    "separate_buffers": {"value": sep_value, "copy_ceiling": sep_ceiling, "h2d_bytes_per_step": h2d_sep, "d2h_bytes_per_step": d2h,
                                         "api": "BatchedExtendedKalman.step_async (nuslam_ekf_step_async): twists, z and ids as three host buffers per step"},
                    "host_affinity": numa},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "peak_source": peak_src, "algorithmic_bytes_per_filter_step": BYTES_PER_FILTER_STEP,
                         "kernel": (KERNEL_NAMES.get((os.environ.get("NUSLAM_KERNEL") or "res2")[:4].rstrip("t"), KERNEL_NAMES["res2"]) +
                                    (" (+ k_ekf_strict_list over the first-touch work list: launched by the step kernel itself, device-side, only when a filter was handed over -- never in the timed steady state)"
                                     if nuslam.lib().nuslam_tail_launch() else " (+ k_ekf_strict_list over the first-touch work list, empty in steady state)")) if args.mode == "fast" else "k_ekf_strict<kOpStep>",
                         "launch_us": per_launch_s * 1e6, "launches_per_step": launches},
        }
    eng.close()
    del xs, sig, zs, twists
    torch.cuda.empty_cache()
    torch.cuda.set_stream(torch.cuda.default_stream(dev))

    # ---- the other BASELINE configurations, each with its own roofline and the reference's CPU path timed beside it ----
    if not args.no_extras:
        sys.path.insert(0, str(ROOT / "tools"))
        import bench_assoc
        cpu_s = 0.0 if args.no_cpu_baseline else args.cpu_seconds / 2
        extra = {}
        # config 4: 1 Mi filters over the ranks of the job (strong scaling), unknown association, statistics all-reduced over NCCL
        a = bench_assoc.run(total=args.assoc_filters, steps=10, warmup=3, cpu_seconds=cpu_s if world == 1 else 0.0, world=world, rank=rank,
                            dist=dist if world > 1 else None)
        extra["assoc"] = a
        if world == 1:
            import bench_large
            import bench_scan
            extra["scan"] = bench_scan.run(cpu_seconds=cpu_s)
            extra["large"] = bench_large.run(steps=20, warmup=3, cpu_seconds=cpu_s, assoc=False)
        if out is not None:
            out["extra"] = extra
    if rank == 0 and world == 1 and not args.no_cpu_baseline and out is not None:
        out["cpu_baseline"] = cpu_baseline(args.cpu_seconds)
    if world > 1:
        dist.destroy_process_group()
    return out


class CpuArm:
    """The reference's own CPU implementation of the path (oracle/_ref: the unmodified sources; the C restatement only where that is
    absent) as a persistent batch of filters: the state stays inside the oracle library between steps, so a timed step is the
    reference's arithmetic on all host threads and nothing else. ONE protocol for `cpu_baseline` and `--impl reference`.
    Variants: the parity build (naive-loop Armadillo shim) and the timing build BASELINE.md 4.1 asks for (matrix products above 4 x 4
    through single-threaded OpenBLAS dgemm, as real Armadillo routes them); the faster one is the baseline, both are printed."""

    def __init__(self):
        import oracle
        self.oracle = oracle
        self.cores = os.cpu_count() or 1
        self.kinds = [k for k in ("ref_blas", "ref") if oracle.available(k)] or ["port"]

    def rate(self, kind, n_filters, n_steps, warmup=1):
        from shermbot_navigation_b200 import synth
        orc = self.oracle.load(kind)
        sc = synth.ekf_scenario(n_filters, 2, n=N_LANDMARKS, seed=4321)
        run = orc.ekf_stepper(N_LANDMARKS, sc["robot0"], sc["map0"], sc["Q"], sc["R"], nthreads=self.cores)
        tw = [np.ascontiguousarray(sc["twists"][t]) for t in range(2)]
        zz = [np.ascontiguousarray(sc["z"][t]) for t in range(2)]
        ii = [np.ascontiguousarray(sc["ids"][t], dtype=np.int32) for t in range(2)]
        run.step(tw[0], zz[0], ii[0])   # the first-touch step
        times = []
        for k in range(warmup + n_steps):
            t0 = time.perf_counter()
            run.step(tw[1], zz[1], ii[1])
            if k >= warmup:
                times.append(time.perf_counter() - t0)
        return n_filters * n_steps / float(np.sum(times)), float(np.sum(times)), orc.flavour

    def measure(self, n_steps, warmup, seconds_per_variant):
        """Each variant on a sample sized for ~seconds_per_variant of wall time; returns (best, all)."""
        results = []
        for kind in self.kinds:
            probe, _, _ = self.rate(kind, 64 * self.cores, 3, 1)
            nf = int(max(self.cores, min(FILTERS_PER_GPU, probe * seconds_per_variant / max(1, n_steps + warmup))))
            nf = max(self.cores, (nf // self.cores) * self.cores)
            value, secs, flavour = self.rate(kind, nf, n_steps, warmup)
            results.append({"value": value, "unit": UNIT, "cores": self.cores, "kind": "reference" if kind.startswith("ref") else "port",
                            "variant": flavour, "filters_per_step": nf, "seconds": secs,
                            "sample": f"{nf} of {FILTERS_PER_GPU} filters per step x {n_steps} steps on {self.cores} host threads, {secs:.1f} s "
                                      f"({flavour}: " + ("unmodified reference sources, " if kind.startswith("ref") else "C restatement, ") +
                                      ("matrix products above 4 x 4 through single-threaded OpenBLAS dgemm" if kind == "ref_blas" else "naive-loop Armadillo shim") + ", -O2)"})
        best = max(results, key=lambda r: r["value"])
        return best, results


def cpu_baseline(target_seconds=12.0):
    arm = CpuArm()
    best, allv = arm.measure(n_steps=20, warmup=1, seconds_per_variant=target_seconds / max(1, len(arm.kinds)))
    out = dict(best)
    out["variants"] = [{k: v[k] for k in ("variant", "value", "filters_per_step", "seconds")} for v in allv]
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return None
    K, W = args.steps, args.warmup
    arm = CpuArm()
    # each "step" = one batched fused step over a bounded sample of the 64K-filter workload; the whole run stays within minutes
    budget = min(150.0, max(20.0, 0.4 * (K + W)))
    best, allv = arm.measure(n_steps=K, warmup=W, seconds_per_variant=budget / max(1, len(arm.kinds)))
    value = best["value"]
    cb = dict(best)
    cb["variants"] = [{k: v[k] for k in ("variant", "value", "filters_per_step", "seconds")} for v in allv]
    return {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": best["seconds"] / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(world),
        "details": {"filters_this_run": best["filters_per_step"], "note": "the reference's CPU implementation timed on a bounded sample of the workload; value = filter-steps/s"},
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="fast", choices=["fast", "strict"])
    ap.add_argument("--filters", type=int, default=FILTERS_PER_GPU)
    ap.add_argument("--e2e-steps", type=int, default=100)
    ap.add_argument("--e2e-repeats", type=int, default=3, help="the end-to-end leg is repeated; the median is reported, all runs are listed")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the config 3 / 4 / 5 blocks (kernel A/B timing)")
    ap.add_argument("--assoc-filters", type=int, default=1 << 20, help="config 4: filters of the WHOLE job (sharded over the ranks)")
    ap.add_argument("--config", default="ekf", choices=["ekf", "scan", "assoc", "large", "closed_loop"],
                    help="ekf (default): the headline line of BASELINE.json configs[1] with the other configurations under `extra`; "
                         "the others run one per-config bench under tools/ on one GPU and print its own JSON line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the state of the last one (rank 0's filters, a fixed sample of "
                         f"{DUMP_FILTERS}) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.config != "ekf"):
        ap.error("--dump-outputs applies to the headline run (--impl ours, --config ekf)")
    if args.config != "ekf":
        import runpy
        tool = {"scan": "bench_scan.py", "assoc": "bench_assoc.py", "large": "bench_large.py", "closed_loop": "bench_closed_loop.py"}[args.config]
        sys.argv = [str(ROOT / "tools" / tool)]
        runpy.run_path(str(ROOT / "tools" / tool), run_name="__main__")
        return
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    out = run_reference(args) if args.impl == "reference" else run_ours(args)
    if out is not None:
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
