#!/usr/bin/env python
"""Joint-compatibility association (NUSLAM_OPT_JOINT_COMPATIBILITY) against nearest neighbour and the reference's rule.

(a) Quality: tools/bench_assoc_nn.py's study of the config-4 scenario (12 landmarks, 12 markers per step, unknown ids, landmark_prior 100,
    both geometries, FILTERS filters x STEPS steps, oracle-order kernels) with a third rule, JOINT | WRAP at 9.21 / 60, beside the
    reference's rule (0.01 / 60) and NN | WRAP (9.21 / 60). Reported: matched / ambiguous / new / exception ids, MAP_FULL, SINGULAR and
    ASSOC_TRUNCATED filters, pose RMSE and mean pose NEES over all filters and over live ones (neither MAP_FULL nor SINGULAR).
(b) Cost: tools/bench_assoc_nn.py's oracle-order step at 131 072 filters x 12 landmark slots (11 seen, well separated, measured every
    step, the same ids under every rule), WRAP against WRAP | NN and WRAP | JOINT, alternated in one process (CUDA events).
Prints one JSON line; --out also writes it to a file."""
import argparse
import json
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
from shermbot_navigation_b200 import nuslam  # noqa: E402
from bench_assoc_nn import RULES, cost_small, quality  # noqa: E402
from bench_large_scan import card  # noqa: E402

WRAP, NN, JC = nuslam.OPT_WRAP_INNOVATION, nuslam.OPT_NEAREST_NEIGHBOUR, nuslam.OPT_JOINT_COMPATIBILITY


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
    rules = dict(RULES, **{"jc_wrap_9.21_60": (JC | WRAP, (9.21, 60.0))})
    out = {"workload": f"(a) config-4 scenario, {a.filters} filters x {a.quality_steps} steps, 12 landmarks, 12 markers per step, unknown ids, "
                       f"landmark_prior 100, oracle-order kernels; (b) cost, variants alternated over {a.rounds} rounds of {a.steps} steps after "
                       f"{a.warmup} (CUDA events)",
           "card": card(), "quality": quality(a.filters, a.quality_steps, rules),
           "cost_oracle_order_step": cost_small(a.batch, a.steps, a.warmup, a.rounds,
                                                variants={"wrap": WRAP, "wrap_nn": WRAP | NN, "wrap_jc": WRAP | JC})}
    line = json.dumps(out)
    print(line)
    if a.out is not None:
        a.out.parent.mkdir(parents=True, exist_ok=True)
        a.out.write_text(line + "\n")


if __name__ == "__main__":
    main()
