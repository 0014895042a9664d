"""Cost of the equidistant lens against the radial-tangential one on one GPU.

For each workload the same geometry (tags, views, observation blocks) gets pixels synthesised per lens from the true
poses (radial-tangential: the workload's own pixels; equidistant: the true poses projected through an equidistant
camera with the same fx fy cx cy, plus the same pixel noise), and one handle per lens times, alternating the lenses:
  - the linearisation (K2 E pass + F pass + finalize, bench.py's `value`): observations per second, L2 flushed
    between timed iterations;
  - one LM iteration (linearise, Schur complement, step, candidate cost).
The registers, stack and spills of every kernel instantiation come from the -Xptxas -v build logs.

usage: python tools/lens_time.py [--steps 20] [--rounds 3] [--cfg4-scale 0.2]      (prints one JSON line)
"""
import argparse
import glob
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from bench import workload  # noqa: E402
from robot_camera_calibration_b200.problem import BAProblem  # noqa: E402
from robot_camera_calibration_b200.scenes import project  # noqa: E402

CUFILT = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cu++filt")
FISHEYE_K = np.array([-0.013, 0.004, -8e-4, 1.2e-4, 0.0])    # k1 k2 k3 k4, reserved slot


def equidistant_copy(s, rng):
    """The scene with pixels of an equidistant camera of the same fx fy cx cy at the true poses."""
    import copy
    e = copy.copy(s)
    e.lens = "equidistant"
    t = s.truth
    intr = np.broadcast_to(t["intr"][0], (s.n_blocks, 4))
    dist = np.broadcast_to(FISHEYE_K, (s.n_blocks, 5))
    px = np.empty((s.n_blocks, 8))
    step = 1 << 20
    for a in range(0, s.n_blocks, step):
        b = min(s.n_blocks, a + step)
        uv, _ = project(s.model, intr[a:b], dist[a:b], t["ext"][s.cam_idx[a:b]], t["views"][s.view_idx[a:b]],
                        t["markers"][s.marker_idx[a:b]], s.sizes[s.marker_idx[a:b]], lens="equidistant")
        px[a:b] = uv.reshape(-1, 8)
    e.pixels = np.trunc(px + rng.normal(0, 0.3, px.shape))      # the workload's integer corners
    e.dist = FISHEYE_K[None] + rng.normal(0, 1e-3, (len(s.intr), 5)) * np.array([1, 1, 1, 1, 0])
    return e


def time_handle(torch, gp, stream, steps):
    """Device time of the linearisation and of one LM iteration: CUDA events on the handle's stream."""
    ev = lambda: torch.cuda.Event(enable_timing=True)
    pairs = []
    for _ in range(steps):
        gp.flush_l2()
        a, b = ev(), ev()
        a.record(stream)
        gp.linearize(want_cost=False)
        b.record(stream)
        pairs.append((a, b))
    torch.cuda.synchronize()
    lin_ms = sum(a.elapsed_time(b) for a, b in pairs) / steps
    pairs = []
    for _ in range(max(2, steps // 4)):
        gp.flush_l2()
        a, b = ev(), ev()
        a.record(stream)
        gp.linearize(want_cost=False)
        gp.schur(1e4)
        gp.solve_step()
        gp.candidate_cost()
        b.record(stream)
        pairs.append((a, b))
    torch.cuda.synchronize()
    lm_ms = sum(a.elapsed_time(b) for a, b in pairs) / len(pairs)
    return lin_ms, lm_ms


def ptxas_table():
    """kernel instantiation -> registers, stack, spill stores, spill loads (the -Xptxas -v build logs).  A stack /
    spill line belongs to the function named by the 'Function properties for' line just above it, which is either the
    entry itself or a device function it calls (such as the slow path of a trigonometric argument reduction)."""
    out = {}
    for log in sorted(glob.glob(os.path.join(ROOT, "robot_camera_calibration_b200", "build", "*.log"))):
        entry = props = None
        for line in open(log):
            m = re.search(r"Compiling entry function '(\S+)'", line)
            if m:
                entry = m.group(1)
                continue
            m = re.search(r"Function properties for (\S+)", line)
            if m:
                props = m.group(1)
                continue
            if entry is None or not re.search(r"assemble_kernel|materialise_kernel|evaluate_kernel|pnp_kernel", entry):
                continue
            m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
            if m and props == entry:
                out.setdefault(entry, {})["stack_spill_st_ld"] = [int(g) for g in m.groups()]
            m = re.search(r"Used (\d+) registers", line)
            if m:
                out.setdefault(entry, {})["registers"] = int(m.group(1))
    named = {}
    for k, v in out.items():
        try:
            k = subprocess.run([CUFILT, k], capture_output=True, text=True).stdout.strip() or k
        except OSError:                     # no demangler: keep the mangled name
            pass
        named[k] = v
    return named


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--cfg4-scale", type=float, default=0.2)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("lens_time.py needs a CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": gpu[0] if gpu else torch.cuda.get_device_name(0), "steps": args.steps, "rounds": args.rounds,
           "workloads": {}}
    rng = np.random.default_rng(7)
    for name, cfg, scale in (("cfg2", 2, 1.0), (f"cfg4 x{args.cfg4_scale:g} views", 4, args.cfg4_scale)):
        s, desc, _ = workload(cfg, 0, 1, scale)
        scenes = {"radtan": s, "equidistant": equidistant_copy(s, rng)}
        handles = {k: BAProblem.from_scene(v, eliminate="views") for k, v in scenes.items()}
        streams = {k: torch.cuda.Stream() for k in handles}
        for k, gp in handles.items():
            gp._check(gp.lib.rcc_ba_set_stream(gp.h, streams[k].cuda_stream))
            for _ in range(3):
                gp.linearize(want_cost=False)
            gp.schur(1e4); gp.solve_step(); gp.candidate_cost()
        per = {k: {"linearize_ms": [], "lm_iter_ms": []} for k in handles}
        for _ in range(args.rounds):                       # alternate the lenses
            for k, gp in handles.items():
                lin, lm = time_handle(torch, gp, streams[k], args.steps)
                per[k]["linearize_ms"].append(round(lin, 4))
                per[k]["lm_iter_ms"].append(round(lm, 4))
        obs = 4 * s.n_blocks
        for k in per:
            per[k]["obs_per_s"] = [obs / (t * 1e-3) for t in per[k]["linearize_ms"]]
        med = lambda k, f: float(np.median(per[k][f]))
        res["workloads"][name] = {
            "workload": desc, "observations": obs, "lenses": per,
            "linearize_ratio_equidistant_over_radtan": med("equidistant", "linearize_ms") / med("radtan", "linearize_ms"),
            "lm_iter_ratio_equidistant_over_radtan": med("equidistant", "lm_iter_ms") / med("radtan", "lm_iter_ms")}
        for gp in handles.values():
            gp.close()
    res["ptxas"] = ptxas_table()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
