"""Under torchrun (N ranks, one GPU each): DistributedBA with priors on views, markers, intr and dist must match the
1-rank solve of the whole problem: the summed reduced system S, b to 1e-12 relative and the converged parameters to
1e-9.  Each prior is added on exactly one rank (dist.shard_priors).  Rank 0 prints a JSON line."""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist
from robot_camera_calibration_b200.dist import DistributedBA
from robot_camera_calibration_b200.problem import BAProblem
from robot_camera_calibration_b200.scenes import make_scene


def priors_of(scene, seed):
    """Full priors on every third view and marker and on every camera's intr and dist."""
    rng = np.random.default_rng(seed)
    sig = {"view": np.array([0.02] * 3 + [0.01] * 3), "marker": np.array([0.02] * 3 + [0.01] * 3),
           "intr": np.array([3.0, 3.0, 2.0, 2.0]), "dist": np.full(5, 0.01)}
    value = {"view": scene.views, "marker": scene.markers, "intr": scene.intr, "dist": scene.dist}
    out = {}
    for kind, s in sig.items():
        idx = np.arange(0, len(value[kind]), 3 if kind in ("view", "marker") else 1)
        k = len(s)
        out[kind] = (idx, value[kind][idx] + rng.normal(0, 1, (len(idx), k)) * s,
                     np.stack([(np.eye(k) + 0.3 * rng.normal(size=(k, k))) / s[None, :] for _ in idx]))
    return out


rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
out = {}
opts = dict(max_iterations=30, function_tolerance=1e-14, gradient_tolerance=1e-12, parameter_tolerance=1e-13)
for name, kw, elim in (("single", dict(n_markers=40, n_views=120, visibility=0.5, seed=41), "views"),
                       ("single_markers", dict(n_markers=40, n_views=120, visibility=0.5, seed=45), "markers"),
                       ("rig", dict(n_markers=30, n_views=60, visibility=0.5, n_cam=2, model="rig", seed=42), "views")):
    kw = dict(kw)
    scene = make_scene(kw.pop("n_markers"), kw.pop("n_views"), kw.pop("visibility"), **kw)
    pri = priors_of(scene, 7)
    dba = DistributedBA(scene, device=local, eliminate=elim, priors=pri)
    p = dba.problem
    p.linearize()
    p.schur(1e4)
    S, b = p.reduced_system()
    summ = dba.solve(**opts)
    views, markers, intr, dst = dba.gather_parameters()
    dba.close()
    if rank == 0:
        with BAProblem.from_scene(scene, device=local, eliminate=elim) as gp:
            for kind, args in pri.items():
                gp.set_priors(kind, *args)
            gp.linearize()
            gp.schur(1e4)
            S1, b1 = gp.reduced_system()
            s1 = gp.solve(**opts)
            v1, m1 = gp.get_view_poses(), gp.get_marker_poses()
            i1, d1 = gp.get_intrinsics()
        out[name] = dict(dS=float(np.linalg.norm(S - S1) / np.linalg.norm(S1)),
                         db=float(np.linalg.norm(b - b1) / np.linalg.norm(b1)),
                         cost=(summ["final_cost"], s1["final_cost"]),
                         dviews=float(np.abs(views - v1).max()), dmarkers=float(np.abs(markers - m1).max()),
                         dintr=float(np.abs(intr - i1).max()), ddist=float(np.abs(dst - d1).max()))
    dist.barrier()
if rank == 0:
    ok = all(v["dS"] <= 1e-12 and v["db"] <= 1e-12 and v["dviews"] < 1e-9 and v["dmarkers"] < 1e-9 and
             v["ddist"] < 1e-9 and v["dintr"] < 1e-9 * 1e3 for v in out.values())
    print(json.dumps({"world": world, "ok": ok, **out}))
    if not ok:
        sys.exit(1)
dist.destroy_process_group()
