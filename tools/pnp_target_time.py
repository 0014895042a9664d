"""Time of the batched rigid-target PnP (rcc_pnp_target_batch, pnp_target_kernel) on one GPU against OpenCV's
cv2.solvePnP on the host cores, over the same problems.

Workloads (seeded, radial-tangential lens, 0.3 px pixel noise, homography start):
  a: 10 000 frames of one 6 x 6 AprilGrid (tags 0.1 m, spacing 0.3), each tag detected with probability 0.8;
  b: 20 000 frames of four 8 x 8 boards, every tag detected: 80 000 problems of 64 tags.
Each board of each frame sits 1.5 - 4 m in front of the camera, tilted up to ~35 degrees.

Reported per workload:
  gpu_ms_per_call  device time of one whole call (host arrays in and out: uploads, kernel, downloads), CUDA events
                   on the legacy default stream, with which the library's stream synchronises; after one warm-up
                   call, over at least 1 s of calls;
  kernel_ms        pnp_target_kernel alone, from torch.profiler CUDA activities in a separate pass;
  cv2_ms           cv2.solvePnP(SOLVEPNP_ITERATIVE) over a random subset of the problems, one problem per task on a
                   thread pool of every host core (OpenCV releases the GIL; cv2.setNumThreads(1)), scaled to all
                   problems;
plus the card name and power limit, read in the same run.

usage: python tools/pnp_target_time.py [--out pnp_target_time.json] [--cv2-sample 4000]   (one JSON line on stdout,
       and in --out)
"""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from robot_camera_calibration_b200 import initialiser  # noqa: E402
from robot_camera_calibration_b200.scenes import board_layout, project_points, rodrigues_np  # noqa: E402


def workload(n_frames, rows, cols, n_boards, p_detect, seed):
    """-> (intr, dist, corners, start, slot, pixels) of n_frames * n_boards problems."""
    rng = np.random.default_rng(seed)
    intr = np.array([600.0, 600.0, 640.0, 512.0])
    dist = np.array([-0.1, 0.02, 1e-3, -1e-3, 0.0])
    corners = board_layout(rows, cols, 0.1, 0.3)
    n_tags = rows * cols
    n = n_frames * n_boards
    ctr = corners.reshape(-1, 2).mean(0)
    rvec = rng.normal(0, 0.35, (n, 3))
    rvec[:, 0] += np.pi                                          # board facing the camera
    poses = np.concatenate([rvec, np.zeros((n, 3))], 1)
    # centre of the board on the optical axis +- a little, at 1.5 - 4 m
    R = rodrigues_np(poses[:, :3])
    depth = rng.uniform(1.5, 4.0, n)
    c_cam = np.stack([rng.uniform(-0.15, 0.15, n) * depth, rng.uniform(-0.1, 0.1, n) * depth, depth], 1)
    poses[:, 3:] = c_cam - np.einsum('nij,j->ni', R[:, :, :2], ctr)
    keep = rng.random((n, n_tags)) < p_detect
    keep[keep.sum(1) == 0, 0] = True
    obj = np.concatenate([corners, np.zeros((n_tags, 4, 1))], -1)
    start, slot, pix = [0], [], []
    for p0 in range(0, n, 4096):
        p1 = min(n, p0 + 4096)
        pp = np.repeat(np.arange(p0, p1), n_tags)
        tt = np.tile(np.arange(n_tags), p1 - p0)
        uv, _ = project_points("single", np.broadcast_to(intr, (len(pp), 4)), np.broadcast_to(dist, (len(pp), 5)),
                               np.zeros((len(pp), 6)), np.zeros((len(pp), 6)), poses[pp], obj[tt])
        uv = uv.reshape(p1 - p0, n_tags, 8) + rng.normal(0, 0.3, (p1 - p0, n_tags, 8))
        for p in range(p1 - p0):
            k = np.nonzero(keep[p0 + p])[0]
            slot.append(k)
            pix.append(uv[p, k])
            start.append(start[-1] + len(k))
    return intr, dist, corners, np.array(start), np.concatenate(slot).astype(np.int32), np.concatenate(pix)


def gpu_time(args, min_seconds=1.0):
    import torch
    intr, dist, corners, start, slot, pix = args
    initialiser.pnp_targets(intr, dist, corners, start, slot, pix)           # warm-up
    times, t_end = [], time.perf_counter() + min_seconds
    while time.perf_counter() < t_end or len(times) < 5:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        poses, cost = initialiser.pnp_targets(intr, dist, corners, start, slot, pix)
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    return float(np.median(times)), len(times), poses, cost


def kernel_time(args):
    import torch
    from torch.profiler import ProfilerActivity, profile
    intr, dist, corners, start, slot, pix = args
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            initialiser.pnp_targets(intr, dist, corners, start, slot, pix)
        torch.cuda.synchronize()
    ks = [e for e in prof.events() if "pnp_target_kernel" in e.name]
    if not ks:
        raise RuntimeError("pnp_target_kernel not seen by the profiler")
    return float(np.median([e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
                            for e in ks])) / 1e3


def cv2_time(args, sample, seed=0):
    import cv2
    cv2.setNumThreads(1)
    intr, dist, corners, start, slot, pix = args
    K = np.array([[intr[0], 0, intr[2]], [0, intr[1], intr[3]], [0, 0, 1.0]])
    n = len(start) - 1
    idx = np.random.default_rng(seed).choice(n, min(sample, n), replace=False)
    jobs = []
    for p in idx:
        o = corners[slot[start[p]:start[p + 1]]].reshape(-1, 2)
        jobs.append((np.concatenate([o, np.zeros((len(o), 1))], 1), pix[start[p]:start[p + 1]].reshape(-1, 2)))

    def one(j):
        return cv2.solvePnP(j[0], j[1], K, dist, flags=cv2.SOLVEPNP_ITERATIVE)[0]

    workers = os.cpu_count() or 1
    with ThreadPoolExecutor(workers) as ex:
        list(ex.map(one, jobs[:64]))                                         # warm-up
        t0 = time.perf_counter()
        ok = list(ex.map(one, jobs))
        dt = time.perf_counter() - t0
    assert all(ok)
    return dt / len(jobs) * n * 1e3, workers, len(jobs)


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:          # noqa: BLE001 -- reported, not fatal
        q = f"unavailable ({e})"
    return name, q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--cv2-sample", type=int, default=4000)
    a = ap.parse_args()
    name, power = card()
    res = {"card": name, "power_limit": power, "workloads": {}}
    for key, spec in (("a_10000x_6x6_80pct", (10000, 6, 6, 1, 0.8, 1)), ("b_20000x_4_boards_8x8", (20000, 8, 8, 4, 1.0, 2))):
        w = workload(*spec)
        ms, calls, poses, cost = gpu_time(w)
        kms = kernel_time(w)
        cms, workers, sample = cv2_time(w, a.cv2_sample)
        n = len(w[3]) - 1
        res["workloads"][key] = {
            "problems": n, "tags": int(w[3][-1]), "corners_per_problem_mean": 4 * w[3][-1] / n,
            "gpu_ms_per_call": ms, "timed_calls": calls, "kernel_ms": kms,
            "cv2_ms_all_problems": cms, "cv2_threads": workers, "cv2_sampled_problems": sample,
            "speedup_call_vs_cv2": cms / ms, "failed_problems": int((cost < 0).sum())}
        print(key, json.dumps(res["workloads"][key]), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
