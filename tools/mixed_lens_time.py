"""Cost of mixing lenses in one rig on one GPU.

The cfg3 geometry (4-camera rig, 2000 tags, ~25 tags per camera and body pose; --scale multiplies the body poses)
gets pixels synthesised per camera from the true poses: a radial-tangential camera keeps the workload's own pixels,
an equidistant camera gets the true poses projected through an equidistant camera with the same fx fy cx cy plus the
same pixel noise (tools/lens_time.py).  The lens sets RRRR, EEEE, RREE and RRRE (R radial-tangential, E equidistant;
camera 0 first) run on one handle each, alternating over the rounds:
  - the linearisation (K2 E pass + F pass + finalize): milliseconds and observations per second, L2 flushed between
    timed iterations;
  - one LM iteration (linearise, Schur complement, step, candidate cost).
A mixed set runs K2 once per lens and pass; its launches per linearisation are reported beside the times, and so
is the split of an LM iteration over the pipeline stages (rcc_ba_profile_*, in a run of its own after the timed ones).

usage: python tools/mixed_lens_time.py [--steps 20] [--rounds 3] [--scale 1.0]      (prints one JSON line)
"""
import argparse
import copy
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

from lens_time import FISHEYE_K, time_handle  # noqa: E402
from robot_camera_calibration_b200.problem import BAProblem  # noqa: E402
from robot_camera_calibration_b200.scenes import config_scene, project  # noqa: E402

LENS_SETS = ("RRRR", "EEEE", "RREE", "RRRE")


def with_lenses(s, code, rng):
    """The scene with camera c under lens code[c]: the equidistant cameras' pixels re-synthesised."""
    e = copy.copy(s)
    e.lens = tuple("equidistant" if k == "E" else "radtan" for k in code)
    e.pixels = s.pixels.copy()
    e.dist = s.dist.copy()
    t = s.truth
    for c, k in enumerate(code):
        if k != "E":
            continue
        sel = np.nonzero(s.cam_idx == c)[0]
        n = len(sel)
        uv, _ = project(s.model, np.broadcast_to(t["intr"][c], (n, 4)), np.broadcast_to(FISHEYE_K, (n, 5)),
                        np.broadcast_to(t["ext"][c], (n, 6)), t["views"][s.view_idx[sel]],
                        t["markers"][s.marker_idx[sel]], s.sizes[s.marker_idx[sel]], lens="equidistant")
        px = uv.reshape(-1, 8)
        e.pixels[sel] = np.trunc(px + rng.normal(0, 0.3, px.shape))
        e.dist[c] = FISHEYE_K + rng.normal(0, 1e-3, 5) * np.array([1, 1, 1, 1, 0])
    return e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("mixed_lens_time.py needs a CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    s = config_scene(3, args.scale, blocked=True, chunk_views=250, round_pixels=True,
                     threads=min(len(os.sched_getaffinity(0)), 16))
    rng = np.random.default_rng(7)
    scenes = {code: with_lenses(s, code, rng) for code in LENS_SETS}
    handles = {k: BAProblem.from_scene(v, eliminate="views") for k, v in scenes.items()}
    streams = {k: torch.cuda.Stream() for k in handles}
    launches = {}
    for k, gp in handles.items():
        gp._check(gp.lib.rcc_ba_set_stream(gp.h, streams[k].cuda_stream))
        for _ in range(3):
            gp.linearize(want_cost=False)
        gp.schur(1e4); gp.solve_step(); gp.candidate_cost()
        n0 = gp.launch_count()
        gp.linearize(want_cost=False)
        launches[k] = gp.launch_count() - n0
    per = {k: {"linearize_ms": [], "lm_iter_ms": [], "launches_per_linearize": launches[k]} for k in handles}
    for _ in range(args.rounds):                       # alternate the lens sets
        for k, gp in handles.items():
            lin, lm = time_handle(torch, gp, streams[k], args.steps)
            per[k]["linearize_ms"].append(round(lin, 4))
            per[k]["lm_iter_ms"].append(round(lm, 4))
    obs = 4 * s.n_blocks
    for k in per:
        per[k]["obs_per_s"] = [obs / (t * 1e-3) for t in per[k]["linearize_ms"]]
    for k, gp in handles.items():                      # where an LM iteration goes: stage events, a run of its own
        gp.profile_enable(True)
        gp.profile_reset()
        for _ in range(3):
            gp.flush_l2()
            gp.linearize(want_cost=False); gp.schur(1e4); gp.solve_step(); gp.candidate_cost()
        gp.synchronize()
        per[k]["lm_stage_ms"] = {st: round(ms / 3, 4) for st, (ms, n) in gp.profile().items() if n}
        gp.profile_enable(False)
    for gp in handles.values():
        gp.close()
    print(json.dumps({"gpu": gpu[0] if gpu else torch.cuda.get_device_name(0), "steps": args.steps,
                      "rounds": args.rounds, "workload": f"cfg3 x{args.scale:g} body poses: 4-camera rig, 2000 tags",
                      "observation_blocks": int(s.n_blocks), "blocks_per_camera": np.bincount(s.cam_idx).tolist(),
                      "observations": obs, "lens_sets": per}))


if __name__ == "__main__":
    main()
