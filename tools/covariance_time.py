#!/usr/bin/env python
"""Time one rcc_ba_covariance call on the benchmark workloads (cfg2 in full, cfg4 on one GPU) and set it against one
LM iteration of the same problem.  One JSON line per configuration on stdout (and in --out).

  python tools/covariance_time.py [--configs 2 4] [--out covariance_time.jsonl]

Per-stage device times come from the library's CUDA-event stage timers (rcc_ba_profile_*):
  linearize = expand + assemble_e + assemble_f + finalize, schur = schur_prep + schur_syrk, cholesky (mask + dense
  factorisation + pivot check), inverse (cusolverDnDpotri), covariance (cov_eliminated_kernel), cov_extract.
The FP64 rate of cov_eliminated_kernel counts, per eliminated block with K partners (kept blocks + border blocks),
the 6 x 6 x 6 products it issues: K (K + 1) / 2 for U_l and K for T, 432 flop each (multiply + add).
The card's name, power limit and SM clock limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

LINEARIZE = ("expand", "assemble_e", "assemble_f", "finalize")
SCHUR = ("schur_prep", "schur_syrk", "schur_shared")


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = (x.strip() for x in q.split(","))
        return {"gpu": name, "power_limit": power, "sm_clock_max": clock}
    except Exception as e:
        return {"gpu": None, "error": repr(e)}


def kernel_flops(scene, n_bb, n_e):
    """Products of cov_eliminated_kernel from the pair structure (views eliminated)."""
    pairs = np.unique(scene.view_idx.astype(np.int64) * len(scene.markers) + scene.marker_idx)
    m = np.bincount(pairs // len(scene.markers), minlength=n_e)
    K = m.astype(np.float64) + n_bb
    return float(np.sum(K * (K + 1) / 2 + K) * 432.0), int(m.max()), float(m.mean())


def stages(gp):
    p = gp.profile()
    return {k: v[0] for k, v in p.items() if v[0] > 0}


def run(cfg, fp64_peak):
    from bench import workload
    from robot_camera_calibration_b200.problem import BAProblem
    s, desc, _ = workload(cfg, 0, 1)
    out = {"config": desc, "observation_blocks": int(s.n_blocks)}
    with BAProblem.from_scene(s, eliminate="views") as gp:
        d = gp.dims
        out["reduced_system_n"] = int(d.n_reduced)
        flops, m_max, m_mean = kernel_flops(s, (d.n_shared + 6) // 6, d.n_e)
        out.update(kernel_flop=flops, partners_max=m_max, partners_mean=m_mean)
        gp.covariance()                                  # warm-up: module load, library workspace, buffers
        gp.synchronize()
        gp.profile_reset()
        gp.profile_enable(True)
        t0 = time.perf_counter()
        gp.covariance()                                  # returns after the host copies (synchronised)
        wall = time.perf_counter() - t0
        st = stages(gp)
        gp.profile_enable(False)
        cov_ms = {"linearize": sum(st.get(k, 0.0) for k in LINEARIZE), "schur": sum(st.get(k, 0.0) for k in SCHUR),
                  "cholesky": st.get("mask", 0.0) + st.get("cholesky", 0.0), "inverse": st.get("inverse", 0.0),
                  "eliminated_kernel": st.get("covariance", 0.0), "extraction": st.get("cov_extract", 0.0)}
        out["covariance_stage_ms"] = cov_ms
        out["covariance_device_ms"] = sum(cov_ms.values())
        out["covariance_wall_ms"] = 1e3 * wall
        k_s = cov_ms["eliminated_kernel"] * 1e-3
        out["eliminated_kernel_tflops"] = flops / k_s / 1e12 if k_s > 0 else None
        out["fp64_peak_tflops_measured"] = fp64_peak
        out["potri_gflops"] = (d.n_reduced ** 3 / 1.5) / (cov_ms["inverse"] * 1e-3) / 1e9 if cov_ms["inverse"] else None

        def lm_iteration():
            gp.linearize(want_cost=False)
            gp.schur(1e4)
            gp.solve_step()
            gp.candidate_cost()
        lm_iteration()
        gp.synchronize()
        gp.profile_reset()
        gp.profile_enable(True)
        t0 = time.perf_counter()
        lm_iteration()
        gp.synchronize()
        out["lm_iteration_wall_ms"] = 1e3 * (time.perf_counter() - t0)
        lm = stages(gp)
        gp.profile_enable(False)
        out["lm_iteration_stage_ms"] = lm
        out["lm_iteration_device_ms"] = sum(lm.values())
        out["covariance_over_lm_iteration"] = out["covariance_device_ms"] / out["lm_iteration_device_ms"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", type=int, nargs="+", default=[2, 4])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("covariance_time.py needs a CUDA device")
    from robot_camera_calibration_b200.problem import fp64_peak_tflops
    info = gpu_info()
    peak = fp64_peak_tflops(0)
    lines = []
    for cfg in args.configs:
        r = run(cfg, peak)
        r.update(info)
        line = json.dumps(r)
        print(line, flush=True)
        lines.append(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
