#!/usr/bin/env python
"""Benchmark of the BA hot path (BASELINE.json metric) -- one JSON line on stdout.

  python bench.py --gpus N --steps K --warmup W          (our CUDA path; N>1 under torchrun)
  python bench.py --impl reference ...                   (the Ceres-equivalent CPU restatement)

step      = one pass of the hot path over the batch: batched reprojection residual
            + analytic Jacobian + Gauss-Newton normal-equation assembly
            (rcc_ba_linearize: expand, assemble E pass, assemble F pass, finalize).
workload  = BASELINE.json configs[3], the largest configuration that fits one GPU: 1 camera, 5 000 tags,
            10 000 keyframes, 25 % visibility (~11.9 M observation blocks = ~47.5 M corner observations),
            integer pixel corners as the reference writes them (corner_detections.cpp:53-54).
            N>1 is STRONG scaling of that one fixed problem: rank r owns keyframes [10000 r / N, 10000 (r+1) / N)
            (observations shard by eliminated-block owner, SURVEY 8e); --config 2 selects configs[1].
value     = corner observations / s, whole job, inputs resident in HBM, L2 flushed
            between timed iterations, device time (CUDA events), max over ranks.
e2e       = same metric through the C ABI with HOST buffers: per step H2D of the pixel
            batch (int16, rcc_ba_update_pixels_i16) + all parameter blocks, linearize, D2H of cost + gradient.
lm_iter   = seconds per full LM iteration (linearize + Schur + reduction over ranks + Cholesky solve +
            back-substitution + candidate cost), max over ranks -- the strong-scaling curve.  lm_iter.cpu (N = 1) = the
            same iteration on the host cores (C++/OpenMP restatement + LAPACK), see cpu_lm_iter().
multi_gpu_parity (N>1) = N-rank vs 1-rank reduced system S, b and LM step on a small scene, run in this process;
            lm_iter.step_check = cost, model decrease, step norm and candidate cost of one LM step of the benchmarked
            problem: the problem is the same for every N, so these numbers must be too.

  python bench.py --dump-outputs bench_outputs/    (N = 1) also writes what the last timed step computed, see
                                                   dump_outputs(); the seeded workload makes two builds comparable
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True        # the benchmark writes nothing into the tree (it may be read-only)

METRIC = "BA corner observations/s (residual+Jacobian+normal equations)"
UNIT = "observations/s"
# algorithmic work per observation block (DESIGN.md section 4)
BYTES_PER_BLOCK_E = 64 + 4 + 288          # pixels + other index in, cross block W out
BYTES_PER_BLOCK_F = 64 + 4
# exact FP64 operation counts: tests/host_harness/flop_count.cpp compiles csrc/model.cuh with a counting scalar
# (profiles/r2_flop_count.json; tests/test_flop_count.py keeps these constants equal to the instrumented run)
FLOP_EVAL_PER_BLOCK = 1084                # block geometry (108) + 4 corners x (residual + analytic Jacobian) (976)
FLOP_PRODUCTS_ALL = 2 * 8 * 253           # J^T J / J^T r: 253 distinct entries x 8 residual rows x (mul + add)
FLOP_PRODUCTS_E = 2 * 8 * 172             # E pass alone: OO, OT, O x [S r], [S r] x [S r]
FLOP_PER_BLOCK = FLOP_PRODUCTS_ALL + FLOP_EVAL_PER_BLOCK
FLOP_PER_BLOCK_E = FLOP_PRODUCTS_E + FLOP_EVAL_PER_BLOCK
# dram__bytes_read.sum + dram__bytes_write.sum of one E-pass launch, measured once under `ncu --set full`:
NCU_DRAM_BYTES_E_PASS = {2: 32313856 + 89391616,       # cfg2, 454 996 blocks  (profiles/r1_ncu_full_summary.txt)
                         4: 819874048 + 3662994000}    # cfg4, 11 880 665 blocks (profiles/r2_ncu_k2_cfg4_summary.txt)

CONFIGS = {
    # cfg: (tags, views, visibility, seed, views per generator chunk, description)
    2: (500, 5000, 0.20, 20242, 125, "cfg2: 1 camera, 500 tags, 5000 views, 20% visibility"),
    4: (5000, 10000, 0.25, 20244, 250, "cfg4: 1 camera, 5000 tags, 10000 keyframes, 25% visibility"),
}


def view_ranges(cfg, world, scale=1.0):
    """Strong-scaling shards: contiguous keyframe ranges, cut at generator-chunk boundaries."""
    tags, views, vis, seed, chunk, desc = CONFIGS[cfg]
    views = max(chunk, int(views * scale) // chunk * chunk)
    n_chunks = views // chunk
    cuts = [n_chunks * r // world * chunk for r in range(world + 1)]
    return views, [(cuts[r], cuts[r + 1]) for r in range(world)]


def workload(cfg, rank, world, scale=1.0, view_range=None, threads=None):
    """The shard of the fixed problem this rank owns (the whole problem when world == 1).  Every shard comes
    from the same generator streams (scenes.make_scene(blocked=True)): the union over ranks is the N=1 scene."""
    from robot_camera_calibration_b200.scenes import make_scene
    if cfg not in CONFIGS:
        raise SystemExit(f"unsupported --config {cfg}")
    tags, _, vis, seed, chunk, desc = CONFIGS[cfg]
    views, ranges = view_ranges(cfg, world, scale)
    lo, hi = ranges[rank] if view_range is None else view_range
    if threads is None:
        threads = max(1, len(os.sched_getaffinity(0)) // max(1, world))
    s = make_scene(tags, views, vis, seed=seed, name=f"cfg{cfg}", blocked=True, chunk_views=chunk,
                   view_range=(lo, hi), round_pixels=True, threads=threads)
    if scale != 1.0:
        desc += f" (scaled to {views} views)"
    return s, desc, views


def config_dict(cfg, desc, views, n_blocks_total):
    """Identical in both arms (the driver compares them)."""
    return {"workload": desc, "tags": CONFIGS[cfg][0], "views": views, "observation_blocks": int(n_blocks_total),
            "observations": int(4 * n_blocks_total), "eliminated": "views",
            "pixels": "integer corners (corner_detections.cpp:53-54)",
            "l2": "GPU arm: flushed (256 MiB write) between timed iterations, untimed; inputs 0.9 GB > L2 anyway"}


def bind_near_gpu(torch, local):
    """Best effort: run this rank on the CPUs NVML calls ideal for its GPU, so that first-touch puts the
    pinned host buffers of the end-to-end path on the GPU's NUMA node (a remote node halves H2D bandwidth)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(local).uuid)
        h = pynvml.nvmlDeviceGetHandleByUUID(uuid if uuid.startswith("GPU-") else "GPU-" + uuid)
        before = len(os.sched_getaffinity(0))
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return {"cpus_before": before, "cpus_after": len(os.sched_getaffinity(0))}
    except Exception as e:  # not permitted in this cgroup, NVML missing, ...
        return {"unchanged": str(e)[:100]}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# CPU arm: the Ceres-equivalent C++/OpenMP restatement (oracle/), on every host thread
# ------------------------------------------------------------------------------------------------
class CpuWorkload:
    """The workload as a list of view slices, each a CpuBA problem of its own.  A slice holds its block-sparse
    Jacobian the way Ceres does (212 doubles per tag observation: 2.5 GB per 1 250 keyframes of cfg4), so the
    47.5 M observations of cfg4 are processed slice after slice; one pass = every slice linearised once.
    (The kept-block sums of the slices are not merged: 5 000 x 81 additions, nothing beside the pass.)"""

    def __init__(self, cfg, scale, ranges, threads):
        os.environ["OMP_NUM_THREADS"] = str(threads)           # before libgomp is loaded
        os.environ["OPENBLAS_NUM_THREADS"] = str(threads)
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import cpu_baseline
        from cpu_baseline import CpuBA
        cpu_baseline.set_num_threads(threads)                  # torchrun's OMP_NUM_THREADS=1 was read at load time
        self.slices, self.n_blocks = [], 0
        self.desc = self.views = None
        for lo, hi in ranges:
            s, self.desc, self.views = workload(cfg, 0, 1, scale, view_range=(lo, hi), threads=threads)
            self.slices.append(CpuBA(s, eliminate="views"))
            self.n_blocks += s.n_blocks
        self.threads = self.slices[0].threads

    def one_pass(self):
        for c in self.slices:
            c.linearize()

    def timed(self, passes):
        t0 = time.perf_counter()
        for _ in range(passes):
            self.one_pass()
        return time.perf_counter() - t0


def slice_ranges(cfg, scale, max_views=1250):
    views, _ = view_ranges(cfg, 1, scale)
    chunk = CONFIGS[cfg][4]
    step = max(chunk, max_views // chunk * chunk)
    return [(lo, min(views, lo + step)) for lo in range(0, views, step)]


def cpu_baseline(cfg, scale, ranges, what, seconds=10.0):
    """Throughput of the CPU restatement on the view ranges `ranges` of the workload, >= `seconds` of timed passes."""
    threads = len(os.sched_getaffinity(0))
    w = CpuWorkload(cfg, scale, ranges, threads)
    w.one_pass()                                       # warm-up: OpenMP pool, page faults
    t1 = w.timed(1)
    passes = max(2, int(np.ceil(seconds / max(t1, 1e-3))))
    el = w.timed(passes)
    obs = 4 * w.n_blocks
    return {"value": obs * passes / el, "unit": UNIT, "cores": w.threads, "kind": "port",
            "sample": f"{what} ({obs} observations per pass), {passes} passes in {el:.1f} s; C++/OpenMP Jet-autodiff "
                      "restatement of the Ceres evaluation + block normal equations (Ceres itself is not available), "
                      f"processed in {len(ranges)} view slice(s)",
            "s_per_pass": el / passes}


def cpu_lm_iter(cfg, scale, radius=1e4, max_views=None, min_free_gb=48.0):
    """Seconds per LM iteration of the CPU restatement (linearise -> block Schur complement -> dense Cholesky
    [LAPACK through SciPy] -> back-substitution), the figure that stands beside `lm_iter`.  A workload of one view
    slice (cfg2) is measured whole, second iteration of two.  A larger one (cfg4: a Schur complement of ~3 TFLOP,
    minutes on the host, and a 30 009-unknown Cholesky) is measured on its FIRST slice of 250 keyframes -- whose
    reduced system has the full size, so the dense solve is timed complete -- and the stages whose work is
    proportional to the keyframes are scaled by the number of slices; the line says so."""
    threads = len(os.sched_getaffinity(0))
    if max_views is None:
        max_views = {2: CONFIGS[2][1]}.get(cfg, CONFIGS[cfg][4])      # cfg2: the whole problem; else one generator chunk
    ranges = slice_ranges(cfg, scale, max_views)
    if len(ranges) > 1:
        try:
            import psutil
            free = psutil.virtual_memory().available / 2 ** 30
        except Exception:
            free = None
        if free is not None and free < min_free_gb:
            return {"skipped": f"{free:.0f} GiB of host memory free, {min_free_gb:.0f} wanted for the dense reduced system"}
    w = CpuWorkload(cfg, scale, ranges[:1], threads)
    try:
        from threadpoolctl import threadpool_limits
        limit = threadpool_limits(limits=threads)            # LAPACK's pool may have read torchrun's OMP_NUM_THREADS=1
    except Exception:
        limit = None
    c = w.slices[0]
    tm = {}
    if len(ranges) == 1:
        c.lm_iteration(radius)                                # warm-up: thread pools, page faults
    else:
        c.linearize()
    t0 = time.perf_counter()
    c.lm_iteration(radius, timings=tm)
    measured = time.perf_counter() - t0
    if limit is not None:
        limit.restore_original_limits()
    k = len(ranges)
    est = k * (tm["linearize"] + tm["schur"] + tm["backsub"]) + tm["solve"]
    what = ("the whole problem, one iteration after a warm-up iteration" if k == 1 else
            f"keyframes {ranges[0][0]}..{ranges[0][1] - 1} of the workload ({4 * c.n} observations; its reduced "
            f"system has the full size, so the dense solve is complete); linearise, Schur complement and "
            f"back-substitution scaled by the {k} slices of the workload")
    return {"s_per_iter": est, "measured_s": measured, "slices": k, "cores": w.threads, "kind": "port",
            "stages_s": {kk: (k if kk != "solve" else 1) * v for kk, v in tm.items()},
            "reduced_system_n": int(6 * c.n_f + c.ns), "sample": what,
            "what": "C++/OpenMP restatement: Jet-autodiff linearisation, block Schur complement, LAPACK dpotrf/dpotrs "
                    "(SciPy), back-substitution; same trust-region radius as lm_iter"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # torchrun pins OMP_NUM_THREADS=1; the reference arm may use every host thread it can get
    threads = len(os.sched_getaffinity(0))
    ranges = slice_ranges(args.config, args.scale)
    w = CpuWorkload(args.config, args.scale, ranges, threads)      # the FULL workload, whatever N is
    warm = max(3, args.warmup)
    for _ in range(warm):
        w.one_pass()
    el = w.timed(args.steps)
    obs = 4 * w.n_blocks
    v = obs * args.steps / el
    sample = (f"the full workload ({obs} observations) per step, in {len(ranges)} view slices; Ceres-equivalent "
              "C++/OpenMP restatement (Ceres and the reference optimiser do not exist here)")
    out = {"metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": warm,
           "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f64", "data": "synthetic", "impl": "reference",
           "config": config_dict(args.config, w.desc, w.views, w.n_blocks),
           "cpu_baseline": {"value": v, "unit": UNIT, "cores": w.threads, "kind": "port", "sample": sample},
           "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _emit(out)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def multi_gpu_parity(torch, dist, rank, world, local):
    """N-rank vs 1-rank on a small scene, through the library's NCCL path: the reduced system S, b as the library
    leaves it on every rank after its band-wise all-reduce, the LM step (solve_step) and a converged solve.
    Relative Frobenius errors; bar 1e-9 (FP64 sums in a different order)."""
    from robot_camera_calibration_b200.dist import shard_scene
    from robot_camera_calibration_b200.problem import BAProblem
    from robot_camera_calibration_b200.scenes import make_scene
    out = {}
    rel = lambda a, b: float(np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(np.asarray(b)), 1e-300))
    # "dist": the hand-written Cholesky with its block columns distributed over the ranks and the panels broadcast
    # (what cfg4 uses; forced here because these scenes are far below the size where it is chosen automatically);
    # "replicated": every rank factors the all-reduced system itself
    cases = (("single_dist", "dist", dict(n_markers=60, n_views=max(96, 12 * world), visibility=0.5, seed=77)),
             ("single_replicated", "cusolver", dict(n_markers=60, n_views=max(96, 12 * world), visibility=0.5, seed=77)),
             ("rig_dist", "dist", dict(n_markers=40, n_views=max(64, 8 * world), visibility=0.5, n_cam=2, model="rig",
                                       seed=78)))
    saved = os.environ.get("RCC_CHOLESKY")
    for name, chol, kw in cases:
        kw = dict(kw)
        os.environ["RCC_CHOLESKY"] = chol
        os.environ["RCC_SYRK_GROUPS"] = "3" if chol == "dist" else "1"         # several reduction bands, like cfg4
        scene = make_scene(kw.pop("n_markers"), kw.pop("n_views"), kw.pop("visibility"), **kw)
        local_scene, (lo, hi) = shard_scene(scene, rank, world, "views")
        gp = BAProblem.from_scene(local_scene, device=local, eliminate="views")
        ids = [BAProblem.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        gp.comm_init(ids[0], rank, world)
        gp.linearize()
        gp.schur(1e4)                                    # collective: the library sums S over the ranks behind the SYRK
        S, b = gp.reduced_system()                       # ... so every rank holds the whole reduced system here
        Sb = np.concatenate([S.ravel(), b])
        gp.solve_step()                                  # factorisation (distributed or replicated) + back-substitution
        st = gp.step()
        parts = [None] * world
        dist.all_gather_object(parts, (lo, hi, st["d_e"][lo:hi], st["d_f"], st["d_shared"]))
        opts = dict(max_iterations=30, function_tolerance=1e-14, gradient_tolerance=1e-12, parameter_tolerance=1e-13)
        gp.set_view_poses(scene.views); gp.set_marker_poses(scene.markers)
        summ = gp.solve(**opts)
        views_n, markers_n = gp.get_view_poses(), gp.get_marker_poses()
        vparts = [None] * world
        dist.all_gather_object(vparts, (lo, hi, views_n[lo:hi]))
        gp.close()
        if rank == 0:
            os.environ["RCC_CHOLESKY"] = "cusolver"      # the 1-rank comparator factors with the library routine
            with BAProblem.from_scene(scene, device=local, eliminate="views") as g1:
                g1.linearize()
                g1.schur(1e4)
                S1, b1 = g1.reduced_system()
                g1.solve_step()
                s1 = g1.step()
                g1.set_view_poses(scene.views); g1.set_marker_poses(scene.markers)
                summ1 = g1.solve(**opts)
                v1, m1 = g1.get_view_poses(), g1.get_marker_poses()
            n = len(b1)
            d_e = np.concatenate([p[2] for p in parts])
            views_all = np.concatenate([p[2] for p in vparts])
            same_everywhere = all(np.array_equal(p[3], parts[0][3]) and np.array_equal(p[4], parts[0][4]) for p in parts)
            out[name] = {"S": rel(Sb[:n * n].reshape(n, n), S1), "b": rel(Sb[n * n:], b1),
                         "delta_F": rel(np.concatenate([st["d_f"].ravel(), st["d_shared"]]),
                                        np.concatenate([s1["d_f"].ravel(), s1["d_shared"]])),
                         "delta_E": rel(d_e, s1["d_e"]), "delta_F_identical_on_all_ranks": bool(same_everywhere),
                         "lm_iterations": [summ["iterations"], summ1["iterations"]],
                         "final_cost_rel": abs(summ["final_cost"] - summ1["final_cost"]) / summ1["final_cost"],
                         "converged_views_max_abs": float(np.abs(views_all - v1).max()),
                         "converged_markers_max_abs": float(np.abs(markers_n - m1).max())}
        dist.barrier()
    os.environ.pop("RCC_SYRK_GROUPS", None)
    if saved is None:
        os.environ.pop("RCC_CHOLESKY", None)
    else:
        os.environ["RCC_CHOLESKY"] = saved
    if rank == 0:
        out["tolerance"] = 1e-9
        out["ok"] = bool(all(v["S"] < 1e-9 and v["b"] < 1e-9 and v["delta_F"] < 1e-9 and v["delta_E"] < 1e-9 and
                             v["delta_F_identical_on_all_ranks"] and v["converged_views_max_abs"] < 1e-6 and
                             v["converged_markers_max_abs"] < 1e-6 for k, v in out.items() if isinstance(v, dict)))
        out["ranks"] = world
    return out


DUMP_BUDGET_BYTES = 60_000_000           # array data; the .npy headers stay well inside 64 MB on top


def dump_outputs(gp, out_dir, seed=0):
    """What a caller of the timed step (rcc_ba_linearize) reads back, left on the device by the last timed step: the
    normal-equation blocks of rcc_ba_get_normal_blocks, FP64, as out_dir/<name>.npy.  W holds one 6 x 6 block per
    observation (3.4 GB on cfg4), so it is written as W_sample: the blocks of a fixed sorted sample of observations,
    drawn with default_rng(seed), as many as fit in DUMP_BUDGET_BYTES beside the other arrays."""
    nb = gp.normal_blocks(want_W=True)
    W = nb.pop("W")
    used = sum(a.nbytes for a in nb.values())
    if used > DUMP_BUDGET_BYTES:
        raise SystemExit(f"--dump-outputs: the normal-equation blocks alone take {used} bytes")
    n = min(len(W), (DUMP_BUDGET_BYTES - used) // (36 * 8))
    nb["W_sample"] = W[np.sort(np.random.default_rng(seed).choice(len(W), n, replace=False))]
    del W
    os.makedirs(out_dir, exist_ok=True)
    for k, a in nb.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def measure(torch, dist, gp, scene, stream, args, rank, world, local, full=True, dump_dir=None):
    """All device-side and end-to-end measurements of one resident problem.  Returns a dict of per-rank numbers
    (not yet reduced over ranks).  With dump_dir, the outputs of the last timed step are written there (untimed)."""
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def ev():
        return torch.cuda.Event(enable_timing=True)

    steps = args.steps
    r = {}
    # ---------------- device-resident steps (value) -------------------------------------
    for _ in range(max(3, args.warmup)):
        gp.linearize(want_cost=False)
    barrier()
    gp.profile_reset()
    gp.profile_enable(True)
    l0 = gp.launch_count()
    pairs = []
    barrier()
    for _ in range(steps):
        gp.flush_l2()                                     # evict L2 between timed iterations (untimed)
        a, b = ev(), ev()
        a.record(stream)
        gp.linearize(want_cost=False)
        b.record(stream)
        pairs.append((a, b))
    barrier()
    r["launches"] = gp.launch_count() - l0               # E pass + F pass + finalize per step (the untimed L2 flush
                                                         # between steps is not counted by rcc_ba_launch_count)
    r["total_ms"] = float(sum(a.elapsed_time(b) for a, b in pairs))
    r["prof"] = gp.profile()
    gp.profile_enable(False)
    if dump_dir is not None:
        dump_outputs(gp, dump_dir)

    # ---------------- materialised evaluation K1 (HBM-write-bound kernel) ----------------
    if full:
        for _ in range(2):
            gp.evaluate_device(want_jacobians=True)
        barrier()
        gp.profile_reset()
        gp.profile_enable(True)
        mat_steps = max(3, min(steps, 10))
        for _ in range(mat_steps):
            gp.flush_l2()
            gp.evaluate_device(want_jacobians=True)
        barrier()
        r["mat_ms"] = gp.profile()["evaluate"][0] / mat_steps
        gp.profile_enable(False)

    # ---------------- full LM iterations (lm_iter) --------------------------------------
    def lm_iteration():
        gp.linearize(want_cost=False)
        gp.schur(1e4)
        gp.solve_step()
        gp.candidate_cost()

    lm_iteration()
    barrier()
    gp.profile_reset()
    gp.profile_enable(True)
    lm_n = max(2, min(steps, 5))
    a, b = ev(), ev()
    a.record(stream)
    for _ in range(lm_n):
        lm_iteration()
    b.record(stream)
    barrier()
    r["lm_ms"] = a.elapsed_time(b) / lm_n
    r["lm_prof"] = {k: v[0] / lm_n for k, v in gp.profile().items() if v[0] > 0}
    gp.profile_enable(False)
    # the same LM step once more, untimed, for its numbers: the problem is fixed, so cost, model decrease, step norm
    # and candidate cost must come out the same for every N (an end-to-end N-rank check at full size)
    c_local = gp.linearize(want_cost=True)
    gp.schur(1e4)
    mcc, step_norm, x_norm = gp.solve_step()
    r["lm_check"] = {"cost_local": c_local, "model_cost_change": mcc, "step_norm": step_norm, "x_norm": x_norm,
                     "candidate_cost": gp.candidate_cost()}

    # ---------------- end-to-end steps through the C ABI with host buffers --------------
    pin = lambda x: torch.from_numpy(np.ascontiguousarray(x)).pin_memory().numpy()
    h_views, h_markers = pin(scene.views), pin(scene.markers)
    h_intr, h_dist = pin(scene.intr), pin(scene.dist)
    d = gp.dims
    h_ge, h_gf, h_gs = pin(np.zeros((d.n_e, 6))), pin(np.zeros((d.n_f, 6))), pin(np.zeros(d.n_shared))
    from robot_camera_calibration_b200.problem import _dp

    def e2e_loop(h_pix, n):
        def step():
            # parameters first: the pixel upload (99 % of the bytes) then overlaps with the E pass piece by piece
            gp.set_view_poses(h_views)
            gp.set_marker_poses(h_markers)
            gp.set_intrinsics(h_intr, h_dist)
            gp.update_pixels(h_pix)
            cost = gp.linearize(want_cost=True)
            gp._check(gp.lib.rcc_ba_get_normal_blocks(gp.h, None, _dp(h_ge), None, None, _dp(h_gf), None, None,
                                                      _dp(h_gs), None))
            return cost
        for _ in range(2):
            step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(n):
            step()
        barrier()
        return time.perf_counter() - t0

    param_bytes = h_views.nbytes + h_markers.nbytes + h_intr.nbytes + h_dist.nbytes
    r["d2h"] = 8 + h_ge.nbytes + h_gf.nbytes + h_gs.nbytes
    h_pix16 = pin(scene.pixels.astype(np.int16))                     # the reference's integer corners
    assert np.array_equal(h_pix16.astype(np.float64), scene.pixels)
    r["e2e_s"] = e2e_loop(h_pix16, steps)
    r["h2d"] = h_pix16.nbytes + param_bytes
    n64 = max(2, min(steps, 5))
    h_pix64 = pin(np.asarray(scene.pixels, dtype=np.float64))
    r["e2e64_s"] = e2e_loop(h_pix64, n64) * steps / n64              # normalised to `steps` steps
    r["h2d64"] = h_pix64.nbytes + param_bytes
    d_probe = torch.empty(h_pix64.size, dtype=torch.float64, device="cuda")
    t_probe = torch.from_numpy(h_pix64)
    h2d_ms = []
    for _ in range(3):
        a, b = ev(), ev()
        a.record(); d_probe.view(t_probe.shape).copy_(t_probe, non_blocking=True); b.record()
        torch.cuda.synchronize()
        h2d_ms.append(a.elapsed_time(b))
    r["h2d_gbs"] = h_pix64.nbytes / (min(h2d_ms) * 1e-3) / 1e9
    del d_probe
    return r


def run_ours(args):
    import torch
    import torch.distributed as dist
    from robot_camera_calibration_b200.problem import BAProblem, fp64_peak_tflops

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local)
    cpus_all = os.sched_getaffinity(0)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def rmax(x):
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def rsum(x):
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def problem_for(cfg):
        scene, desc, views = workload(cfg, rank, world, args.scale)
        gp = BAProblem.from_scene(scene, device=local, eliminate="views")
        stream = torch.cuda.Stream(device=local)
        gp._check(gp.lib.rcc_ba_set_stream(gp.h, stream.cuda_stream))
        if world > 1:
            ids = [BAProblem.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(ids, src=0)
            gp.comm_init(ids[0], rank, world)
        return scene, desc, views, gp, stream

    scene, desc, views, gp, stream = problem_for(args.config)
    placement = bind_near_gpu(torch, local)      # pinned host buffers must sit on the GPU's NUMA node
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    m = measure(torch, dist, gp, scene, stream, args, rank, world, local, dump_dir=args.dump_outputs)
    clocks = sampler.stop() if rank == 0 else None
    d = gp.dims
    n_red, n_pairs_local = int(d.n_reduced), int(d.n_pairs)
    gp.close()

    # ---------------- reduce over ranks --------------------------------------------------
    n_blocks_all = rsum(scene.n_blocks)
    obs_all = 4 * n_blocks_all
    total_ms_max = rmax(m["total_ms"])
    lm_ms_max = rmax(m["lm_ms"])
    e2e_s_max, e2e64_s_max = rmax(m["e2e_s"]), rmax(m["e2e64_s"])
    launches_all = int(rsum(m["launches"]))
    h2d_all, h2d64_all, d2h_all = int(rsum(m["h2d"])), int(rsum(m["h2d64"])), int(rsum(m["d2h"]))
    n_pairs_all = int(rsum(n_pairs_local))

    lm_check = dict(m["lm_check"])
    lm_check["cost"] = rsum(lm_check.pop("cost_local"))
    lm_check["gain_ratio"] = (lm_check["cost"] - lm_check["candidate_cost"]) / lm_check["model_cost_change"]
    parity = multi_gpu_parity(torch, dist, rank, world, local) if world > 1 else None

    # ---------------- the cfg2 line beside it (N = 1 only: round-1's headline configuration) ---------------
    cfg2 = None
    if world == 1 and args.config != 2 and not args.no_cfg2:
        s2, desc2, _, g2, st2 = problem_for(2)
        m2 = measure(torch, dist, g2, s2, st2, args, rank, world, local, full=False)
        o2 = 4 * s2.n_blocks
        cfg2 = {"workload": desc2, "observations": o2, "value": o2 * args.steps / (m2["total_ms"] * 1e-3),
                "ms_per_step": m2["total_ms"] / args.steps,
                "e2e": {"value": o2 * args.steps / m2["e2e_s"], "ms_per_step": 1e3 * m2["e2e_s"] / args.steps,
                        "h2d_bytes_per_step": int(m2["h2d"]), "d2h_bytes_per_step": int(m2["d2h"])},
                "e2e_f64_pixels": {"value": o2 * args.steps / m2["e2e64_s"], "h2d_bytes_per_step": int(m2["h2d64"])},
                "lm_iter": {"s_per_iter": m2["lm_ms"] * 1e-3, "stage_ms": m2["lm_prof"],
                            "reduced_system_n": int(g2.dims.n_reduced), "step_check": m2["lm_check"]}}
        g2.close()

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return

    # ---------------- rank 0: the CPU figure beside it (the other ranks have left: every host core is free) ---
    os.sched_setaffinity(0, cpus_all)
    if world == 1:
        base = cpu_baseline(args.config, args.scale, slice_ranges(args.config, args.scale), "the full workload",
                            seconds=args.cpu_seconds)
    else:
        _, ranges = view_ranges(args.config, world, args.scale)
        base = cpu_baseline(args.config, args.scale, [ranges[0]],
                            f"rank 0's shard of the workload (keyframes {ranges[0][0]}..{ranges[0][1] - 1})",
                            seconds=args.cpu_seconds)

    # ... and the CPU seconds per LM iteration beside lm_iter (N = 1: LAPACK's thread pool is not pinned by torchrun)
    lm_cpu = None
    if world == 1 and not args.no_cpu_lm:
        def guarded(cfg, scale):
            try:
                return cpu_lm_iter(cfg, scale)
            except Exception as e:                       # the GPU line must not die with the CPU comparison
                return {"error": repr(e)}
        lm_cpu = guarded(args.config, args.scale)
        if cfg2 is not None:
            cfg2["lm_iter"]["cpu"] = guarded(2, 1.0)

    hbm_peak, peak_src = measured_peaks()
    fp64_peak = fp64_peak_tflops(local)
    prof, n_blocks = m["prof"], scene.n_blocks
    k_ms = prof["assemble_e"][0] / max(1, prof["assemble_e"][1])
    kf_ms = prof["assemble_f"][0] / max(1, prof["assemble_f"][1])
    ach = BYTES_PER_BLOCK_E * n_blocks / (k_ms * 1e-3) / 1e9
    value = obs_all * args.steps / (total_ms_max * 1e-3)
    step_flops = FLOP_PER_BLOCK * n_blocks
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": total_ms_max / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(args.config, desc, views, n_blocks_all),
        "timing": "CUDA events per step on the library's stream, summed; max over ranks",
        "shard": {"keyframes_rank0": len(scene.views), "observation_blocks_rank0": n_blocks,
                  "rule": "contiguous keyframe ranges by eliminated-block owner; no data-path collective in `value`"},
        "roofline": {"bound": "hbm", "kernel": "assemble_kernel<E pass> (fused residual+Jacobian+J^T J tiles), rank 0",
                     "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                     "traffic": NCU_DRAM_BYTES_E_PASS.get(args.config) if (world == 1 and args.scale == 1.0) else None,
                     "traffic_source": "ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum of one E-pass launch "
                                       "on this workload (profiles/r2_ncu_k2_cfg4_summary.txt; cfg2: "
                                       "profiles/r1_ncu_full_summary.txt); N = 1 only",
                     "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": BYTES_PER_BLOCK_E * n_blocks,
                     "kernel_ms": k_ms, "f_pass_kernel_ms": kf_ms,
                     "note": "fused assembly is FP64-pipe-bound, not HBM-bound: see roofline_fp64"},
        "roofline_fp64_e_pass": {"bound": "fp64 (DFMA + DMMA.8x8x4 share one pipe; same peak either way)",
                                 "kernel": "assemble_kernel<E pass>",
                                 "achieved": FLOP_PER_BLOCK_E * n_blocks / (k_ms * 1e-3) / 1e12, "peak": fp64_peak,
                                 "unit": "TFLOP/s", "frac": FLOP_PER_BLOCK_E * n_blocks / (k_ms * 1e-3) / 1e12 / fp64_peak,
                                 "algorithmic_flop_per_launch": FLOP_PER_BLOCK_E * n_blocks,
                                 "flop_source": "instrumented count (tests/host_harness/flop_count.cpp, "
                                                "profiles/r2_flop_count.json): 1084 evaluation + 2752 products per block",
                                 "note": "executed work is larger: 8 DMMA x 512 flop + 4 corner evaluations per block"},
        "roofline_fp64": {"bound": "fp64", "achieved": step_flops / (m["total_ms"] / args.steps * 1e-3) / 1e12,
                          "peak": fp64_peak, "unit": "TFLOP/s",
                          "frac": step_flops / (m["total_ms"] / args.steps * 1e-3) / 1e12 / fp64_peak,
                          "peak_source": "measured here: DFMA microbenchmark (rcc_fp64_peak_tflops)",
                          "algorithmic_flop_per_step": step_flops, "scope": "rank 0"},
        "roofline_materialise": {"bound": "hbm", "kernel": "materialise_kernel (K1: residuals + Ceres-layout Jacobians to HBM)",
                                 "achieved": 1480 * n_blocks / (m["mat_ms"] * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                 "frac": 1480 * n_blocks / (m["mat_ms"] * 1e-3) / 1e9 / hbm_peak,
                                 "algorithmic_bytes_per_launch": 1480 * n_blocks, "kernel_ms": m["mat_ms"],
                                 "observations_per_s": 4 * n_blocks / (m["mat_ms"] * 1e-3),
                                 "note": "includes the 1-CTA cost reduction launched behind it; rank 0"},
        "cpu_baseline": base,
        "e2e": {"value": obs_all * args.steps / e2e_s_max, "unit": UNIT, "h2d_bytes_per_step": h2d_all,
                "d2h_bytes_per_step": d2h_all, "ms_per_step": 1e3 * e2e_s_max / args.steps,
                "h2d_gb_per_s_this_box": m["h2d_gbs"], "cpu_placement": placement,
                "what": "set_view/marker_poses + set_intrinsics + update_pixels_i16 (pinned host -> device; the "
                        "reference's integer corners, 16 B per tag, widened to FP64 on the device), linearize, read "
                        "back cost and gradient; wall clock, max over ranks"},
        "e2e_f64_pixels": {"value": obs_all * args.steps / e2e64_s_max, "unit": UNIT, "h2d_bytes_per_step": h2d64_all,
                           "what": "same step with FP64 pixel buffers (rcc_ba_update_pixels): 64 B per tag over PCIe"},
        "gpu_launches": launches_all,
        "clocks": clocks,
        "lm_iter": {"s_per_iter": lm_ms_max * 1e-3, "obs_per_s": obs_all / (lm_ms_max * 1e-3),
                    "stage_ms_rank0": m["lm_prof"], "reduced_system_n": n_red, "n_pairs": n_pairs_all,
                    "step_check": lm_check, "cpu": lm_cpu,
                    "what": "linearize + Schur + reduction over ranks + reduced solve + back-substitution + candidate "
                            "cost of the whole fixed problem; the strong-scaling curve is s_per_iter over N"},
        "stage_ms_per_step": {k: v[0] / args.steps for k, v in prof.items() if v[0] > 0},
    }
    if parity is not None:
        out["multi_gpu_parity"] = parity
    if cfg2 is not None:
        out["cfg2"] = cfg2
    _emit(out)


def _emit(obj):
    """The one JSON line goes to the process's ORIGINAL stdout; everything else any
    library prints (NCCL banners, warnings) was re-routed to stderr in main()."""
    os.write(_REAL_STDOUT, (json.dumps(obj) + "\n").encode())


_REAL_STDOUT = 1


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)                      # fd 1 -> stderr for the rest of the run
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=4, help="BASELINE.json configuration: 4 (default) or 2")
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the config's views (debug)")
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="timed CPU work of the cpu_baseline leg")
    ap.add_argument("--no-cfg2", action="store_true", help="skip the cfg2 line at N=1")
    ap.add_argument("--no-cpu-lm", action="store_true", help="skip the CPU seconds per LM iteration (lm_iter.cpu, N=1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy "
                                                          "(N=1, --impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.impl != "ours" or args.gpus != 1):
        ap.error("--dump-outputs needs --impl ours and --gpus 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
