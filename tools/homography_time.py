"""Time of the batched plane homographies (rcc_homography_target_batch, homography_target_kernel) on one GPU against
OpenCV's cv2.findHomography on the host cores, over the same problems, and the wall clock of a calibration from
detections alone (--initialise --target --image-size) on workload a.

Workloads: those of tools/pnp_target_time.py (seeded, radial-tangential lens, 0.3 px pixel noise):
  a: 10 000 frames of one 6 x 6 AprilGrid, each tag detected with probability 0.8;
  b: 20 000 frames of four 8 x 8 boards, every tag detected: 80 000 problems of 64 tags.

Reported per workload:
  gpu_ms_per_call  device time of one whole call (host arrays in and out: uploads, kernel, downloads), CUDA events
                   on the legacy default stream, with which the library's stream synchronises; after one warm-up
                   call, over at least 1 s of calls;
  kernel_ms        homography_target_kernel alone, from torch.profiler CUDA activities in a separate pass;
  cv2_ms           cv2.findHomography(method 0) over a random subset of the problems, one problem per task on a
                   thread pool of every host core (OpenCV releases the GIL; cv2.setNumThreads(1)), scaled to all
                   problems.
For workload a also:
  e2e_s            wall clock of `python -m robot_camera_calibration_b200 DIR --initialise --target GRID
                   --image-size 1280 1024` on a directory of its 10 000 frames with integer corners and no
                   camera.yaml (reading the detections, the homographies, the closed form, the board PnP, the
                   bundle adjustment with free intrinsics, writing the results), and the intrinsics it found.
plus the card name and power limit, read in the same run.

usage: python tools/homography_time.py [--out homography_time.json] [--cv2-sample 20000]   (one JSON line on stdout,
       and in --out)
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

from pnp_target_time import card, workload  # noqa: E402
from robot_camera_calibration_b200 import initialiser, io_yaml  # noqa: E402


def gpu_time(args, min_seconds=1.0):
    import torch
    intr, dist, corners, start, slot, pix = args
    initialiser.homographies(corners, start, slot, pix)                    # warm-up
    times, t_end = [], time.perf_counter() + min_seconds
    while time.perf_counter() < t_end or len(times) < 5:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        H, cost = initialiser.homographies(corners, start, slot, pix)
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    return float(np.median(times)), len(times), H, cost


def kernel_time(args):
    import torch
    from torch.profiler import ProfilerActivity, profile
    intr, dist, corners, start, slot, pix = args
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            initialiser.homographies(corners, start, slot, pix)
        torch.cuda.synchronize()
    ks = [e for e in prof.events() if "homography_target_kernel" in e.name]
    if not ks:
        raise RuntimeError("homography_target_kernel not seen by the profiler")
    return float(np.median([e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
                            for e in ks])) / 1e3


def cv2_time(args, sample, seed=0):
    import cv2
    cv2.setNumThreads(1)
    intr, dist, corners, start, slot, pix = args
    n = len(start) - 1
    idx = np.random.default_rng(seed).choice(n, min(sample, n), replace=False)
    jobs = [(corners[slot[start[p]:start[p + 1]]].reshape(-1, 2), pix[start[p]:start[p + 1]].reshape(-1, 2))
            for p in idx if start[p + 1] - start[p] >= 1]

    def one(j):
        return cv2.findHomography(j[0], j[1], 0)[0] is not None

    workers = os.cpu_count() or 1
    with ThreadPoolExecutor(workers) as ex:
        list(ex.map(one, jobs[:64]))                                         # warm-up
        t0 = time.perf_counter()
        ok = list(ex.map(one, jobs))
        dt = time.perf_counter() - t0
    assert all(ok)
    return dt / len(jobs) * n * 1e3, workers, len(jobs)


def end_to_end(args, rows=6, cols=6, image_size=(1280, 1024)):
    """--initialise --target --image-size on a temporary directory of the workload's frames (integer corners)."""
    intr, dist, corners, start, slot, pix = args
    d = tempfile.mkdtemp(prefix="rcc_homography_e2e_")
    try:
        c = np.round(pix).astype(np.int64).reshape(-1, 4, 2)
        for p in range(len(start) - 1):
            sl = slice(start[p], start[p + 1])
            with open(os.path.join(d, f"detections_{p}.yaml"), "w") as f:
                f.write(io_yaml.detections_text(slot[sl], [0.1] * (start[p + 1] - start[p]), c[sl]))
        grid = os.path.join(d, "grid.yaml")
        with open(grid, "w") as f:
            f.write(f"target_type: aprilgrid\ntagRows: {rows}\ntagCols: {cols}\ntagSize: 0.1\ntagSpacing: 0.3\n")
        cmd = [sys.executable, "-m", "robot_camera_calibration_b200", d, "--initialise", "--target", grid,
               "--image-size", str(image_size[0]), str(image_size[1])]
        t0 = time.perf_counter()
        r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True)
        dt = time.perf_counter() - t0
        if r.returncode != 0:
            raise RuntimeError(f"{' '.join(cmd)} exited {r.returncode}:\n{r.stderr[-2000:]}")
        summary = json.loads(r.stdout.strip().splitlines()[-1])
        intr_out = io_yaml.read_camera(os.path.join(d, "camera_refined.yaml"))[0]
    finally:
        shutil.rmtree(d, ignore_errors=True)
    return {"e2e_s": dt, "initial_intrinsics": summary["initial_intrinsics"], "final_intr": intr_out.tolist(),
            "true_intr": list(map(float, intr)), "iterations": summary["iterations"],
            "termination": summary["termination_name"], "final_cost": summary["final_cost"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--cv2-sample", type=int, default=20000)
    ap.add_argument("--no-e2e", action="store_true")
    a = ap.parse_args()
    name, power = card()
    res = {"card": name, "power_limit": power, "workloads": {}}
    for key, spec in (("a_10000x_6x6_80pct", (10000, 6, 6, 1, 0.8, 1)), ("b_20000x_4_boards_8x8", (20000, 8, 8, 4, 1.0, 2))):
        w = workload(*spec)
        ms, calls, H, cost = gpu_time(w)
        kms = kernel_time(w)
        cms, workers, sample = cv2_time(w, a.cv2_sample)
        n = len(w[3]) - 1
        res["workloads"][key] = {
            "problems": n, "tags": int(w[3][-1]), "corners_per_problem_mean": 4 * w[3][-1] / n,
            "gpu_ms_per_call": ms, "timed_calls": calls, "kernel_ms": kms,
            "cv2_ms_all_problems": cms, "cv2_threads": workers, "cv2_sampled_problems": sample,
            "speedup_call_vs_cv2": cms / ms, "failed_problems": int((cost < 0).sum())}
        if key.startswith("a_") and not a.no_e2e:
            res["workloads"][key].update(end_to_end(w))
        print(key, json.dumps(res["workloads"][key]), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
