"""Cost of Gaussian priors (rcc_ba_set_priors) on one GPU.

At the cfg2 geometry (1 camera, 500 tags, 5 000 views) and the cfg4 geometry (1 camera, 5 000 tags, 10 000 keyframes;
--scale4 multiplies the keyframes) one handle runs three prior sets, switched with rcc_ba_set_priors and alternated
over the rounds:
  - none:   no priors (the launches of a handle that never had any);
  - all:    a full 6 x 6 prior on every view and every marker;
  - shared: priors on the camera's intr and dist only.
For each: the linearisation (K2 E pass + F pass + finalize + the prior kernel) and one LM iteration (linearise, Schur
complement, step, candidate cost), CUDA events on the handle's stream, L2 flushed between timed iterations, and the
launches of one linearisation.

usage: python tools/prior_time.py [--steps 20] [--rounds 3] [--scale4 1.0]      (prints one JSON line)
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

from lens_time import time_handle  # noqa: E402
from robot_camera_calibration_b200.problem import BAProblem  # noqa: E402
from robot_camera_calibration_b200.scenes import config_scene  # noqa: E402

VARIANTS = ("none", "all", "shared")


def prior_sets(s, rng):
    """{variant: {kind: (index, mean, A)}}: full priors near the current parameters."""
    def full(values, sig):
        n, k = values.shape
        A = (np.eye(k) + 0.1 * rng.normal(size=(n, k, k))) / sig[None, None, :]
        return np.arange(n), values + rng.normal(0, 1, (n, k)) * sig, A
    pose = np.array([0.02] * 3 + [0.01] * 3)
    shared = {"intr": full(s.intr, np.array([3.0, 3.0, 2.0, 2.0])), "dist": full(s.dist, np.full(5, 0.01))}
    return {"none": {}, "all": {"view": full(s.views, pose), "marker": full(s.markers, pose)}, "shared": shared}


def use(gp, priors):
    gp.clear_priors()
    for kind, args in priors.items():
        gp.set_priors(kind, *args)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--scale4", type=float, default=1.0)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("prior_time.py needs a CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    threads = min(len(os.sched_getaffinity(0)), 16)
    rng = np.random.default_rng(7)
    out = {}
    for cfg, scale in ((2, 1.0), (4, args.scale4)):
        s = config_scene(cfg, scale, blocked=True, round_pixels=True, threads=threads)
        sets = prior_sets(s, rng)
        stream = torch.cuda.Stream()
        with BAProblem.from_scene(s, eliminate="views") as gp:
            gp._check(gp.lib.rcc_ba_set_stream(gp.h, stream.cuda_stream))
            per = {v: {"linearize_ms": [], "lm_iter_ms": []} for v in VARIANTS}
            for v in VARIANTS:
                use(gp, sets[v])
                gp.linearize(want_cost=False); gp.schur(1e4); gp.solve_step(); gp.candidate_cost()
                n0 = gp.launch_count()
                gp.linearize(want_cost=False)
                per[v]["launches_per_linearize"] = gp.launch_count() - n0
                per[v]["priors"] = int(sum(len(a[0]) for a in sets[v].values()))
            for _ in range(args.rounds):               # alternate the variants
                for v in VARIANTS:
                    use(gp, sets[v])
                    for _ in range(2):
                        gp.linearize(want_cost=False)
                    lin, lm = time_handle(torch, gp, stream, args.steps)
                    per[v]["linearize_ms"].append(round(lin, 4))
                    per[v]["lm_iter_ms"].append(round(lm, 4))
        out[f"cfg{cfg}" + (f"x{scale:g}" if scale != 1.0 else "")] = dict(
            views=len(s.views), markers=len(s.markers), observation_blocks=int(s.n_blocks), variants=per)
    print(json.dumps({"gpu": gpu[0] if gpu else torch.cuda.get_device_name(0), "steps": args.steps,
                      "rounds": args.rounds, **out}))


if __name__ == "__main__":
    main()
