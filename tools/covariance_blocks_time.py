#!/usr/bin/env python
"""Time rcc_ba_covariance_blocks on the benchmark workloads (cfg2 in full, cfg4 on one GPU, views eliminated) and set
its pair kernels against cov_eliminated_kernel of one rcc_ba_covariance call on the same problem.  One JSON line per
configuration on stdout (and in --out).

  python tools/covariance_blocks_time.py [--configs 2 4] [--out covariance_blocks_time.jsonl]

Requests, each timed after a warm-up call of the same request:
  (a) consecutive   every consecutive eliminated pair (view e, view e + 1)
      consecutive_shuffled: the pairs of (a) in a random order
  (b) view_camera   every (view, intr 0) and (view, dist 0) pair
  (c) lone          the single pair (view e, view e + 1) of the median-length row: the latency case
The pair kernels (cov_pairs_kernel + cov_pairs_combine_kernel) are the library's "covariance" stage of the call, read
from its CUDA-event stage timers (rcc_ba_profile_*); the rest of the call (linearise, reduced system, potrf, potri) is
reported beside it.  Block products are counted on the host from the partner lists: a pair whose canonical sides have
K_a <= K_b items (K = kept partners + border blocks for an eliminated block, 1 for a kept or shared one) issues
K_a K_b products for U and K_b more for X when side b is eliminated; cov_eliminated_kernel issues K (K + 1) / 2 + K per
eliminated block.  432 flop (multiply + add) per 6 x 6 x 6 product.  The card's name, power limit and SM clock limit
are read in the same run.
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

FLOP = 432.0


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = (x.strip() for x in q.split(","))
        return {"gpu": name, "power_limit": power, "sm_clock_max": clock}
    except Exception as e:
        return {"gpu": None, "error": repr(e)}


def partner_counts(scene):
    """Kept partners (distinct markers) of every view."""
    nm = len(scene.markers)
    pairs = np.unique(scene.view_idx.astype(np.int64) * nm + scene.marker_idx)
    return np.bincount(pairs // nm, minlength=len(scene.views)).astype(np.float64)


def pair_products(Ka, Kb, b_eliminated):
    """Block products of the pairs with canonical sides Ka <= Kb (arrays)."""
    lo, hi = np.minimum(Ka, Kb), np.maximum(Ka, Kb)
    return float(np.sum(lo * hi + np.where(b_eliminated, hi, 0.0)))


def timed_call(gp, fn):
    fn()                                                 # warm-up: same shapes, module load, library buffers
    gp.synchronize()
    gp.profile_reset()
    gp.profile_enable(True)
    t0 = time.perf_counter()
    fn()                                                 # returns after the host copies (synchronised)
    wall = time.perf_counter() - t0
    st = {k: v[0] for k, v in gp.profile().items() if v[0] > 0}
    gp.profile_enable(False)
    return st, wall


def run(cfg):
    from bench import workload
    from robot_camera_calibration_b200.problem import BAProblem
    s, desc, _ = workload(cfg, 0, 1)
    out = {"config": desc, "observation_blocks": int(s.n_blocks)}
    nv = len(s.views)
    with BAProblem.from_scene(s, eliminate="views") as gp:
        d = gp.dims
        n_bb = (d.n_shared + 6) // 6
        K = partner_counts(s) + n_bb
        out.update(reduced_system_n=int(d.n_reduced), partners_mean=float(K.mean() - n_bb), partners_max=int(K.max() - n_bb))
        mid = int(np.argsort(K[:-1])[(nv - 1) // 2])
        requests = {
            "consecutive": ([(("view", e), ("view", e + 1)) for e in range(nv - 1)],
                            pair_products(K[:-1], K[1:], True)),
            "view_camera": ([(("view", e), (k, 0)) for e in range(nv) for k in ("intr", "dist")],
                            2 * pair_products(np.ones(nv), K, True)),
            # (a) again in a random request order: items of neighbouring rows no longer run side by side, which
            # shows what the ordering by eliminated block is worth (L2 reuse of S^-1 blocks)
            "consecutive_shuffled": ([(("view", int(e)), ("view", int(e) + 1))
                                      for e in np.random.default_rng(0).permutation(nv - 1)],
                                     pair_products(K[:-1], K[1:], True)),
            "lone": ([(("view", mid), ("view", mid + 1))], pair_products(K[mid:mid + 1], K[mid + 1:mid + 2], True)),
        }
        res = {}
        for name, (pairs, products) in requests.items():
            st, wall = timed_call(gp, lambda: gp.covariance_blocks(pairs))
            k_ms = st.get("covariance", 0.0)
            res[name] = {"pairs": len(pairs), "block_products": products, "pair_kernels_ms": k_ms,
                         "pair_kernels_tflops": products * FLOP / (k_ms * 1e-3) / 1e12 if k_ms > 0 else None,
                         "inverse_ms": st.get("inverse", 0.0), "call_device_ms": sum(st.values()),
                         "call_wall_ms": 1e3 * wall}
        out["requests"] = res
        st, wall = timed_call(gp, gp.covariance)
        products = float(np.sum(K * (K + 1) / 2 + K))
        k_ms = st.get("covariance", 0.0)
        out["marginal"] = {"block_products": products, "eliminated_kernel_ms": k_ms,
                           "eliminated_kernel_tflops": products * FLOP / (k_ms * 1e-3) / 1e12 if k_ms > 0 else None,
                           "call_device_ms": sum(st.values()), "call_wall_ms": 1e3 * wall}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", type=int, nargs="+", default=[2, 4])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("covariance_blocks_time.py needs a CUDA device")
    info = gpu_info()
    lines = []
    for cfg in args.configs:
        r = run(cfg)
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
