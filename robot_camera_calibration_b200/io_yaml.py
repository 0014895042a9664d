"""The reference's on-disk formats, read *and* write (SURVEY.md 8f-1).

  detections_N.yaml   corner_detections.cpp:18-39 (+ trailing "\\n" :59), and the
                      `world_T_camera:` stanza camera_pose.cpp:95-99 appends
  targets.yaml        camera_pose.cpp:103-129
  camera.yaml         ROS camera_calibration output that `rosparam load` feeds to
                      camera_pose.cpp:59-64 (/camera_matrix/data, /distortion_coefficients/data);
                      distortion_model plumb_bob (k1 k2 p1 p2 k3) or equidistant / fisheye (k1 k2 k3 k4)

Writers reproduce the reference's `fout <<` statements byte for byte
(`std::to_string(double)` == "%f", 6 decimals).  `optimise_directory` is the
missing Milestone 3: read what camera_pose_node wrote, refine on the GPU, write
the same files back so that opt_vis_node (opt_visualization.cpp:46-66,118-138)
displays the refined map.
"""
from __future__ import annotations

import glob
import os
import re

import numpy as np
import yaml

from .scenes import Scene


def _ts(x, precision=None):
    """std::to_string(double) (precision None) or a lossless/explicit variant."""
    if precision is None:
        return "%f" % float(x)
    if precision == "repr":
        return repr(float(x))
    return f"%.{int(precision)}f" % float(x)


# ------------------------------------------------------------------ writers
def detections_text(tag_ids, sizes, corners):
    """corner_detections.cpp:18-39,59.  corners: (n,4,2) integer pixels."""
    out = ["detections:"]
    for tid, sz, c in zip(tag_ids, sizes, corners):
        out.append("\n - targetID: " + str(int(tid)))
        out.append("\n   size: [ " + _ts(sz) + ", " + _ts(sz) + " ]")
        out.append("\n   corners:")
        for i in range(4):
            out.append("\n    " + str(i) + ": [ " + str(int(c[i][0])) + ", " + str(int(c[i][1])) + " ]")
    out.append("\n")
    return "".join(out)


def world_T_camera_text(rvec, t, precision=None):
    """camera_pose.cpp:95-99 (appended to detections_N.yaml, no trailing newline)."""
    s = "world_T_camera:"
    s += "\n rotation: [ " + _ts(rvec[0], precision) + " , " + _ts(rvec[1], precision) + " , " + _ts(rvec[2], precision) + " ]"
    s += "\n translation: [ " + _ts(t[0], precision) + " , " + _ts(t[1], precision) + " , " + _ts(t[2], precision) + " ]"
    return s


def targets_text(tag_ids, sizes, poses, precision=None):
    """camera_pose.cpp:103-129."""
    out = ["targets:"]
    for tid, sz, p in zip(tag_ids, sizes, poses):
        h = float(sz) / 2
        out.append("\n - targetID: " + str(int(tid)))
        out.append("\n   world_T_target:")
        out.append("\n    rotation: [ " + _ts(p[0], precision) + " , " + _ts(p[1], precision) + " , " + _ts(p[2], precision) + " ]")
        out.append("\n    translation: [ " + _ts(p[3], precision) + " , " + _ts(p[4], precision) + " , " + _ts(p[5], precision) + " ]")
        out.append("\n   obj_points_in_target:")
        out.append("\n    0: [ " + _ts(-h) + ", " + _ts(-h) + ", 0 ]")      # bl
        out.append("\n    1: [ " + _ts(h) + ", " + _ts(-h) + ", 0 ]")       # br
        out.append("\n    2: [ " + _ts(h) + ", " + _ts(h) + ", 0 ]")        # tr
        out.append("\n    3: [ " + _ts(-h) + ", " + _ts(h) + ", 0 ]")       # tl
    return "".join(out)


def camera_yaml_text(intr, dist, image_size=(640, 480), name="camera", lens="radtan"):
    """ROS camera_info YAML: distortion_model plumb_bob with 5 coefficients, or equidistant with k1 k2 k3 k4 (the
    reserved fifth slot of the library's dist[5] is not written)."""
    fx, fy, cx, cy = (float(v) for v in intr)
    if lens not in _LENS_MODEL:
        raise ValueError(f"unknown lens {lens!r}")
    coeffs = list(dist)[:4] if lens == "equidistant" else list(dist)
    d = ", ".join(repr(float(v)) for v in coeffs)
    return (f"image_width: {int(image_size[0])}\nimage_height: {int(image_size[1])}\ncamera_name: {name}\n"
            "camera_matrix:\n  rows: 3\n  cols: 3\n"
            f"  data: [{fx!r}, 0.0, {cx!r}, 0.0, {fy!r}, {cy!r}, 0.0, 0.0, 1.0]\n"
            f"distortion_model: {_LENS_MODEL[lens]}\ndistortion_coefficients:\n  rows: 1\n  cols: {len(coeffs)}\n"
            f"  data: [{d}]\n")


_LENS_MODEL = {"radtan": "plumb_bob", "equidistant": "equidistant"}     # library lens -> ROS distortion_model


def write_dataset(directory, scene, tag_ids=None, with_poses=True, precision=None):
    """Emit a scene as the reference pipeline would have left it on disk: one
    detections_N.yaml per view (integer pixels, corner_detections.cpp:53-54),
    targets.yaml and camera.yaml.  Single-camera model only (the reference has one
    camera, camera_pose.cpp:38)."""
    if scene.model != "single" or len(scene.intr) != 1:
        raise ValueError("the reference formats describe one camera")
    os.makedirs(directory, exist_ok=True)
    tag_ids = np.arange(len(scene.markers)) if tag_ids is None else np.asarray(tag_ids)
    order = np.argsort(scene.view_idx, kind="stable")
    vi = scene.view_idx[order]
    starts = np.searchsorted(vi, np.arange(len(scene.views) + 1))
    for v in range(len(scene.views)):
        sel = order[starts[v]:starts[v + 1]]
        m = scene.marker_idx[sel]
        if v == 0 and len(m) and 0 in m:
            # the world tag must be the first entry of frame 0 (camera_pose.cpp:74)
            k = int(np.nonzero(m == 0)[0][0])
            sel = np.concatenate([sel[k:k + 1], sel[:k], sel[k + 1:]])
            m = scene.marker_idx[sel]
        txt = detections_text(tag_ids[m], scene.sizes[m], np.trunc(scene.pixels[sel]).reshape(-1, 4, 2))
        if with_poses:
            txt += world_T_camera_text(scene.views[v, 0:3], scene.views[v, 3:6], precision)
        with open(os.path.join(directory, f"detections_{v}.yaml"), "w") as f:
            f.write(txt)
    with open(os.path.join(directory, "targets.yaml"), "w") as f:
        f.write(targets_text(tag_ids, scene.sizes, scene.markers, precision))
    with open(os.path.join(directory, "camera.yaml"), "w") as f:
        f.write(camera_yaml_text(scene.intr[0], scene.dist[0], scene.image_size, lens=scene.lens))


# ------------------------------------------------------------------ readers
def read_camera(path):
    """-> (intr[4], dist[5], lens) with fx=K[0] fy=K[4] cx=K[2] cy=K[5] (camera_pose.cpp:61-64).
    distortion_model equidistant or fisheye (ROS camera_info, Kalibr, cv::fisheye): lens "equidistant", dist =
    k1 k2 k3 k4 and the reserved slot 0.  Any other model (plumb_bob, or none given): lens "radtan", dist = the first
    five coefficients k1 k2 p1 p2 k3 (missing trailing ones 0)."""
    with open(path) as f:
        y = yaml.safe_load(f)
    K = [float(v) for v in y["camera_matrix"]["data"]]
    model = str(y.get("distortion_model", "plumb_bob")).strip().lower()
    lens = "equidistant" if model in ("equidistant", "fisheye") else "radtan"
    d = [float(v) for v in y["distortion_coefficients"]["data"]]
    if lens == "equidistant":
        if len(d) != 4:
            raise ValueError(f"{path}: an equidistant camera has 4 distortion coefficients, found {len(d)}")
    else:
        d = d[:5]
    d += [0.0] * (5 - len(d))
    return np.array([K[0], K[4], K[2], K[5]]), np.array(d), lens


def read_camera_yaml(path):
    """-> (intr[4], dist[5]) of a radial-tangential camera (camera_pose.cpp:61-64).  An equidistant (fisheye) file
    raises ValueError: its k1 k2 k3 k4 are not k1 k2 p1 p2, so read it with read_camera, which returns the lens."""
    intr, dist, lens = read_camera(path)
    if lens != "radtan":
        raise ValueError(f"{path} describes an {lens} lens: read it with io_yaml.read_camera, which returns "
                         "(intr, dist, lens)")
    return intr, dist


def read_dataset(directory, intr=None, dist=None, lens=None):
    """Read targets.yaml + detections_*.yaml (+ camera.yaml) into a Scene.
    The intrinsics come from camera.yaml unless `intr` (fx fy cx cy) and `dist` (k1 k2 p1 p2 k3, or k1 k2 k3 k4 with
    lens="equidistant") are given.  The lens is camera.yaml's distortion_model whenever camera.yaml exists, also with
    explicit intrinsics, so that a fisheye directory is never optimised as a radial-tangential camera; `lens` overrides
    it only for explicit intrinsics (with intrinsics from camera.yaml it must agree); "radtan" when there is neither;
    a dataset with neither is an error (the reference logs ROS_ERROR when the intrinsics are not loaded,
    camera_pose.cpp:66-67 -- optimising from made-up intrinsics would silently overwrite good files).
    Frames without a `world_T_camera` stanza (never referenced by
    camera_pose_node, camera_pose.cpp:278-281) and tags missing from targets.yaml
    are skipped.  Returns (scene, tag_ids, frame_numbers)."""
    with open(os.path.join(directory, "targets.yaml")) as f:
        targets = (yaml.safe_load(f) or {}).get("targets") or []
    if lens is not None and lens not in _LENS_MODEL:
        raise ValueError(f"unknown lens {lens!r}: expected one of {sorted(_LENS_MODEL)}")
    if not targets:
        raise ValueError(f"{directory}/targets.yaml lists no targets: nothing defines the world frame "
                         "(camera_pose.cpp:71-80 makes the first tag of frame 0 the world tag)")
    tag_ids = np.array([int(t["targetID"]) for t in targets])
    index_of = {int(t): i for i, t in enumerate(tag_ids)}
    markers = np.array([list(t["world_T_target"]["rotation"]) + list(t["world_T_target"]["translation"])
                        for t in targets], dtype=np.float64).reshape(-1, 6)
    # tag size: 2 * obj_points_in_target[2][0]  (opt_visualization.cpp:81)
    sizes = np.array([2.0 * float(t["obj_points_in_target"][2][0]) for t in targets])
    files = glob.glob(os.path.join(directory, "detections_*.yaml"))
    numbered = sorted((int(re.search(r"detections_(\d+)\.yaml$", p).group(1)), p) for p in files)
    views, frames, vi, mi, px = [], [], [], [], []
    for n, path in numbered:
        with open(path) as f:
            y = yaml.safe_load(f)
        if not y or "world_T_camera" not in y:
            continue
        v = len(views)
        views.append(list(y["world_T_camera"]["rotation"]) + list(y["world_T_camera"]["translation"]))
        frames.append(n)
        for det in y.get("detections") or []:
            tid = int(det["targetID"])
            if tid not in index_of:
                continue
            c = det["corners"]
            vi.append(v)
            mi.append(index_of[tid])
            px.append([c[k][a] for k in range(4) for a in range(2)])
    cam = os.path.join(directory, "camera.yaml")
    if intr is not None and dist is not None:
        intr, dist = np.asarray(intr, dtype=np.float64), np.asarray(dist, dtype=np.float64).ravel()
        dist = np.concatenate([dist, np.zeros(5 - len(dist))])
        if lens is None:
            lens = read_camera(cam)[2] if os.path.exists(cam) else "radtan"
    elif os.path.exists(cam):
        intr, dist, cam_lens = read_camera(cam)
        if lens is not None and lens != cam_lens:
            raise ValueError(f"{cam} describes an {cam_lens} lens, not {lens}: its coefficients are that model's")
        lens = cam_lens
    else:
        raise FileNotFoundError(f"{cam} not found and no intr/dist given: the camera intrinsics are required "
                                "(camera_pose.cpp:59-67)")
    scene = Scene(model="single", intr=intr.reshape(1, 4), dist=dist.reshape(1, 5), ext=np.zeros((1, 6)),
                  views=np.array(views, dtype=np.float64).reshape(-1, 6), markers=markers, sizes=sizes,
                  view_idx=np.array(vi, dtype=np.int32), marker_idx=np.array(mi, dtype=np.int32),
                  cam_idx=np.zeros(len(vi), dtype=np.int32), pixels=_pixel_array(px), lens=lens)
    return scene, tag_ids, np.array(frames)


def _pixel_array(px):
    """Corner lists -> (N,8) array.  corner_detections.cpp:53-54 writes integer corners: those stay integers
    (int16 when they fit) so that BAProblem ships 16 bytes per tag to the GPU; anything else is FP64."""
    if px and all(isinstance(v, int) for row in px for v in row):
        a = np.array(px, dtype=np.int64).reshape(-1, 8)
        if a.min() >= -32768 and a.max() <= 32767:
            return a.astype(np.int16)
        return a.astype(np.int32)
    return np.array(px, dtype=np.float64).reshape(-1, 8)


def write_results(directory, scene, tag_ids, frames, precision=None):
    """Write refined poses back: targets.yaml is rewritten (camera_pose.cpp:103-129)
    and the world_T_camera stanza of every frame is replaced (:95-99)."""
    with open(os.path.join(directory, "targets.yaml"), "w") as f:
        f.write(targets_text(tag_ids, scene.sizes, scene.markers, precision))
    for v, n in enumerate(frames):
        path = os.path.join(directory, f"detections_{int(n)}.yaml")
        with open(path) as f:
            txt = f.read()
        k = txt.find("world_T_camera:")
        head = txt[:k] if k >= 0 else txt
        with open(path, "w") as f:
            f.write(head + world_T_camera_text(scene.views[v, 0:3], scene.views[v, 3:6], precision))


def intrinsics_priors(intr, dist, sigma):
    """Diagonal priors that keep every camera's intr and dist near (intr, dist): sigma = (focal px, principal point
    px, distortion coefficient), the standard deviations of fx fy, of cx cy and of every distortion entry.  Returns
    {kind: (index, mean, sqrt_information)} for BAProblem.set_priors."""
    f, c, d = (float(x) for x in sigma)
    if not (f > 0 and c > 0 and d > 0 and np.isfinite([f, c, d]).all()):
        raise ValueError(f"intrinsics sigmas must be positive and finite, got {sigma}")
    intr, dist = np.asarray(intr, dtype=np.float64), np.asarray(dist, dtype=np.float64)
    n = len(intr)
    a_intr = np.diag([1 / f, 1 / f, 1 / c, 1 / c])
    a_dist = np.eye(5) / d
    return {"intr": (np.arange(n), intr, np.broadcast_to(a_intr, (n, 4, 4))),
            "dist": (np.arange(n), dist, np.broadcast_to(a_dist, (n, 5, 5)))}


def optimise_directory(directory, device=0, refine_intrinsics=True, precision=None, intr=None, dist=None,
                       lens=None, intrinsics_sigma=None, **lm_options):
    """Milestone 3: detections/ -> GPU bundle adjustment -> detections/ (same formats).  The lens is camera.yaml's
    distortion_model (plumb_bob, or equidistant / fisheye), and camera_refined.yaml is written in the same model.
    intrinsics_sigma = (focal px, principal point px, distortion): refine the intrinsics under a diagonal Gaussian
    prior centred on camera.yaml (intrinsics_priors) instead of freely; it needs refine_intrinsics."""
    from .problem import BAProblem
    if intrinsics_sigma is not None and not refine_intrinsics:
        raise ValueError("intrinsics_sigma puts a prior on refined intrinsics: it cannot be combined with fixed ones")
    scene, tag_ids, frames = read_dataset(directory, intr=intr, dist=dist, lens=lens)
    scene.const_intr[:] = not refine_intrinsics
    scene.const_dist[:] = not refine_intrinsics
    with BAProblem.from_scene(scene, device=device) as p:
        if intrinsics_sigma is not None:
            for kind, args in intrinsics_priors(scene.intr, scene.dist, intrinsics_sigma).items():
                p.set_priors(kind, *args)
        summary = p.solve(**lm_options)
        scene.views, scene.markers = p.get_view_poses(), p.get_marker_poses()
        intr, dist = p.get_intrinsics()
        scene.intr, scene.dist = intr, dist
    write_results(directory, scene, tag_ids, frames, precision)
    if refine_intrinsics:
        with open(os.path.join(directory, "camera_refined.yaml"), "w") as f:
            f.write(camera_yaml_text(intr[0], dist[0], scene.image_size, lens=scene.lens))
    return summary
