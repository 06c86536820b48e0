#!/usr/bin/env python
"""Per-phase clock64 breakdown of the FAST kernel (ekf_fast.cuh, block 0, warp 0). Needs a -DNUSLAM_TIMING build, and NUSLAM_KERNEL=fast:
   at 12 landmarks the default is the resident pair kernel (ekf_res2.cuh), which has no timing hooks.
   NUSLAM_KERNEL=fast NUSLAM_B200_LIB=build/variants/lib_timing.so python tools/fast_timing.py"""
import ctypes as C
import os, sys
from pathlib import Path
import numpy as np
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import torch
from shermbot_navigation_b200 import nuslam, synth

B, n, K = 65536, 12, 5
D = 64
sc = synth.ekf_scenario(D, K + 3, n=n, seed=5)
rep = lambda a: np.ascontiguousarray(np.tile(a, (B // D,) + (1,) * (a.ndim - 1)))
eng = nuslam.BatchedExtendedKalman(rep(sc["robot0"]), rep(sc["map0"]), sc["Q"], sc["R"], mode="fast")
dev = torch.device("cuda", 0)
tw = [torch.tensor(rep(sc["twists"][t]), device=dev) for t in range(K + 3)]
z = [torch.tensor(rep(sc["z"][t]), device=dev) for t in range(K + 3)]
ids = [torch.tensor(rep(sc["ids"][t]), device=dev) for t in range(K + 3)]
for t in range(3):
    eng.step(tw[t], z[t], ids[t])
eng.synchronize()
lib = nuslam.lib()
out = (C.c_longlong * 16)()
lib.nuslam_debug_fast_timing(out, 1)
for t in range(3, 3 + K):
    eng.step(tw[t], z[t], ids[t])
eng.synchronize()
lib.nuslam_debug_fast_timing(out, 0)
v = np.array(list(out), dtype=np.float64)
nblk = 148 * int(os.environ.get("NUSLAM_FAST_CTAS_PER_SM", "16"))
filters = K * ((B + nblk - 1) // nblk)   # filters processed by block 0 / warp 0
names = ["load", "predict", "publish", "pre (Pt,Wt)", "2x2 part + Kt", "post (x, robot)", "dmma", "store"]
tot = v[:8].sum()
print(f"block 0 / warp 0: {filters} filter-steps, {tot / filters:.0f} cycles per filter-step ({tot / filters / 12:.0f} per update)")
for k, nm in enumerate(names):
    print(f"  {nm:<24}{v[k] / filters:>10.0f} cycles/filter-step {100 * v[k] / tot:>6.1f} %")
