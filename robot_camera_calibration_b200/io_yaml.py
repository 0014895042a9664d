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

from .scenes import Scene, board_layout, compose, invert


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
    intr, dist, lens = _dataset_camera(directory, intr, dist, lens)
    scene = Scene(model="single", intr=intr.reshape(1, 4), dist=dist.reshape(1, 5), ext=np.zeros((1, 6)),
                  views=np.array(views, dtype=np.float64).reshape(-1, 6), markers=markers, sizes=sizes,
                  view_idx=np.array(vi, dtype=np.int32), marker_idx=np.array(mi, dtype=np.int32),
                  cam_idx=np.zeros(len(vi), dtype=np.int32), pixels=_pixel_array(px), lens=lens)
    return scene, tag_ids, np.array(frames)


def read_detections(directory):
    """detections_N.yaml of a directory in numeric order of N -> (frame numbers, frames_pixels), frames_pixels in the
    format initialiser.initialise takes: per frame [(tag_id, size, pixels8)], the size from the file's `size` entry
    (corner_detections.cpp:18-39) and the pixels as the corners' own numbers (integers stay integers, so that the
    scene keeps the int16 pixel path).  Any world_T_camera stanza is ignored."""
    files = glob.glob(os.path.join(directory, "detections_*.yaml"))
    numbered = sorted((int(re.search(r"detections_(\d+)\.yaml$", p).group(1)), p) for p in files)
    frames, out = [], []
    for n, path in numbered:
        with open(path) as f:
            y = yaml.safe_load(f) or {}
        fr = []
        for det in y.get("detections") or []:
            c = det["corners"]
            px = [c[k][a] for k in range(4) for a in range(2)]
            px = np.array(px, dtype=np.int64 if all(isinstance(v, int) for v in px) else np.float64)
            fr.append((int(det["targetID"]), float(det["size"][0]), px))
        frames.append(n)
        out.append(fr)
    return np.array(frames, dtype=np.int64), out


def _dataset_camera(directory, intr, dist, lens):
    """The camera of a dataset as read_dataset documents it -> (intr, dist[5], lens)."""
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
    return intr, dist, lens


def read_target(path):
    """A rigid tag board in Kalibr's AprilGrid format -> (tag ids (n,), corners (n, 4, 2)): keys target_type:
    aprilgrid, tagCols, tagRows, tagSize (m), tagSpacing (the gap between tags over tagSize), and firstTagId (ours,
    default 0).  Convention: tag (r, c) has id firstTagId + r tagCols + c; the board origin is the bottom-left corner
    of tag firstTagId, the tag axes are the board axes, and tag (r, c) is centred at (c (1 + spacing) s + s/2,
    r (1 + spacing) s + s/2) for s = tagSize (scenes.board_layout); the corners are bl br tr tl in the board frame.
    Agreement with Kalibr's own id numbering and board origin has not been verified against Kalibr."""
    with open(path) as f:
        y = yaml.safe_load(f) or {}
    if str(y.get("target_type", "")).strip().lower() != "aprilgrid":
        raise ValueError(f"{path}: target_type must be aprilgrid, got {y.get('target_type')!r}")
    try:
        rows, cols = int(y["tagRows"]), int(y["tagCols"])
        size, spacing = float(y["tagSize"]), float(y["tagSpacing"])
    except KeyError as e:
        raise ValueError(f"{path}: missing key {e.args[0]}") from None
    first = int(y.get("firstTagId", 0))
    if rows < 1 or cols < 1 or not 0 < size < np.inf or not 0 <= spacing < np.inf or first < 0:
        raise ValueError(f"{path}: tagRows and tagCols must be positive, tagSize positive, tagSpacing and firstTagId "
                         "not negative")
    return first + np.arange(rows * cols), board_layout(rows, cols, size, spacing)


def read_targets(paths):
    """read_target of every file; a tag id on two targets is an error."""
    out, owner = [], {}
    for k, path in enumerate(paths):
        ids, corners = read_target(path)
        for i in ids.tolist():
            if owner.setdefault(i, k) != k:
                raise ValueError(f"tag id {i} is on two targets: {paths[owner[i]]} and {path}")
        out.append((ids, corners))
    return out


def board_scene(scene, tag_ids, targets):
    """Map the tags of a per-tag scene (read_dataset) onto rigid boards: targets = read_targets(...).  Every board
    with a detected tag becomes one marker block, first the boards in target order, then the tags on no board (free,
    slot -1).  A board's initial pose is world_T_tag o (board_T_tag)^-1 of its most-detected tag; a board carrying
    the world tag (marker 0 of the scene, camera_pose.cpp:71-80) is the gauge and held constant.  Returns
    (board_scene, tag_pose) with tag_pose(markers) -> the world_T_tag of every tag of `scene` (tag_ids order) from
    the board scene's markers."""
    where = {}                                                  # tag id -> (target, slot)
    for b, (ids, _) in enumerate(targets):
        for k, i in enumerate(ids.tolist()):
            where[i] = (b, k)
    n_tags = len(tag_ids)
    counts = np.bincount(scene.marker_idx, minlength=n_tags)
    on = [where.get(int(t)) for t in tag_ids]
    used = sorted({w[0] for w, c in zip(on, counts) if w is not None and c > 0})
    new_of_board = {b: j for j, b in enumerate(used)}
    free = [m for m in range(n_tags) if on[m] is None or on[m][0] not in new_of_board]
    new_of_tag = np.empty(n_tags, dtype=np.int64)
    slot_of_tag = np.full(n_tags, -1, dtype=np.int32)
    offset = np.zeros(len(targets) + 1, dtype=np.int64)         # slots of target b: [offset[b], offset[b + 1])
    offset[1:] = np.cumsum([len(ids) for ids, _ in targets])
    for m in range(n_tags):
        if on[m] is not None and on[m][0] in new_of_board:
            new_of_tag[m] = new_of_board[on[m][0]]
            slot_of_tag[m] = offset[on[m][0]] + on[m][1]
    for j, m in enumerate(free):
        new_of_tag[m] = len(used) + j
    corners = np.concatenate([c for _, c in targets]).reshape(-1, 4, 2)

    def board_T_tag(slot):                                      # the tag frame: centred on the tag, board axes
        ctr = corners[slot].mean(0)
        return np.array([0.0, 0.0, 0.0, ctr[0], ctr[1], 0.0])

    markers = np.zeros((len(used) + len(free), 6))
    sizes = np.zeros(len(markers))
    const = np.zeros(len(markers), bool)
    for b in used:
        tags = [m for m in range(n_tags) if on[m] is not None and on[m][0] == b]
        best = max(tags, key=lambda m: counts[m])
        markers[new_of_board[b]] = compose(scene.markers[best], invert(board_T_tag(slot_of_tag[best])))
        sizes[new_of_board[b]] = scene.sizes[best]
        const[new_of_board[b]] = any(scene.const_markers[m] for m in tags)
    for j, m in enumerate(free):
        markers[len(used) + j] = scene.markers[m]
        sizes[len(used) + j] = scene.sizes[m]
        const[len(used) + j] = scene.const_markers[m]
    s = Scene(model=scene.model, intr=scene.intr, dist=scene.dist, ext=scene.ext, views=scene.views, markers=markers,
              sizes=sizes, view_idx=scene.view_idx, marker_idx=new_of_tag[scene.marker_idx].astype(np.int32),
              cam_idx=scene.cam_idx, pixels=scene.pixels, const_views=scene.const_views, const_markers=const,
              const_intr=scene.const_intr, const_dist=scene.const_dist, image_size=scene.image_size,
              lens=scene.lens, corners=corners, corner_slot=slot_of_tag[scene.marker_idx])

    def tag_pose(new_markers):
        out = np.empty((n_tags, 6))
        for m in range(n_tags):
            j = new_of_tag[m]
            out[m] = new_markers[j] if slot_of_tag[m] < 0 else compose(new_markers[j], board_T_tag(slot_of_tag[m]))
        return out

    boards = [(int(targets[b][0][0]), new_of_board[b]) for b in used]   # (first tag id, marker block)
    return s, tag_pose, boards


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
    _write_poses(directory, tag_ids, scene.sizes, scene.markers, scene.views, frames, precision)


def _write_poses(directory, tag_ids, sizes, markers, views, frames, precision=None):
    with open(os.path.join(directory, "targets.yaml"), "w") as f:
        f.write(targets_text(tag_ids, sizes, markers, precision))
    for v, n in enumerate(frames):
        path = os.path.join(directory, f"detections_{int(n)}.yaml")
        with open(path) as f:
            txt = f.read()
        k = txt.find("world_T_camera:")
        head = txt[:k] if k >= 0 else txt
        with open(path, "w") as f:
            f.write(head + world_T_camera_text(views[v, 0:3], views[v, 3:6], precision))


def _remove_stanza(path):
    """Drop the world_T_camera stanza of a detections file, if it has one."""
    with open(path) as f:
        txt = f.read()
    k = txt.find("world_T_camera:")
    if k >= 0:
        with open(path, "w") as f:
            f.write(txt[:k])


def _initialise_directory(directory, intr, dist, lens, targets, image_size=None, device=0):
    """The start of optimise_directory(initialise=True): the camera as read_dataset reads it, or, with image_size,
    initialiser.initialise_intrinsics from the board detections and zero distortion; the poses from the detections
    alone.  Returns (scene, tag_ids, kept frame numbers, (all frame numbers, frames_pixels), tag_pose, boards,
    initial intrinsics summary or None); tag_pose and boards as board_scene's (per tag and empty without targets)."""
    from . import initialiser
    if lens is not None and lens not in _LENS_MODEL:
        raise ValueError(f"unknown lens {lens!r}: expected one of {sorted(_LENS_MODEL)}")
    if image_size is None:
        intr, dist, lens = _dataset_camera(directory, intr, dist, lens)
    numbers, frames_pixels = read_detections(directory)
    if not frames_pixels or not frames_pixels[0]:
        raise ValueError(f"{directory}: the first detections file has no detection: nothing defines the world frame "
                         "(camera_pose.cpp:71-80 makes the first tag of frame 0 the world tag)")
    boards_read = read_targets(list(targets)) if targets else None
    initial = None
    if image_size is not None:
        lens = lens or "radtan"
        intr, used = initialiser.initialise_intrinsics(frames_pixels, boards_read, image_size, device=device)
        dist = np.zeros(5)
        initial = {"intr": intr.tolist(), "problems_used": used}
    if targets:
        scene, tag_ids, keep, tag_pose, boards = initialiser.initialise_targets(
            frames_pixels, intr, dist, boards_read, lens=lens)
        if image_size is not None:
            scene.image_size = (int(image_size[0]), int(image_size[1]))
    else:
        scene, tag_ids, keep = initialiser.initialise(frames_pixels, intr, dist, lens=lens)
        scene.pixels = _integer_pixels(scene.pixels, frames_pixels)
        tag_pose, boards = (lambda markers: markers), []
    return scene, tag_ids, numbers[keep], (numbers, frames_pixels), tag_pose, boards, initial


def _integer_pixels(pixels, frames_pixels):
    """initialiser.initialise returns FP64 pixels: give integer detections their integer type back (_pixel_array)."""
    if all(np.issubdtype(np.asarray(p).dtype, np.integer) for fr in frames_pixels for (_, _, p) in fr):
        return _pixel_array(np.asarray(pixels).astype(np.int64).tolist())
    return pixels


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
                       lens=None, intrinsics_sigma=None, targets=None, initialise=False, image_size=None,
                       **lm_options):
    """Milestone 3: detections/ -> GPU bundle adjustment -> detections/ (same formats).  The lens is camera.yaml's
    distortion_model (plumb_bob, or equidistant / fisheye), and camera_refined.yaml is written in the same model.
    intrinsics_sigma = (focal px, principal point px, distortion): refine the intrinsics under a diagonal Gaussian
    prior centred on camera.yaml (intrinsics_priors) instead of freely; it needs refine_intrinsics.
    targets: AprilGrid target files (read_target).  Their detected tags are solved as rigid boards, one pose each
    (board_scene); targets.yaml is still written per tag (world_T_board o board_T_tag), and the summary gains
    "boards": [{"first_tag_id", "world_T_board": rvec + t}] per board.
    initialise: start from the detections alone instead of camera_pose_node's output.  targets.yaml and any
    world_T_camera stanzas are ignored; the camera comes from camera.yaml or intr / dist as in read_dataset; the
    poses come from initialiser.initialise_targets (with targets) or initialiser.initialise (without).  After the
    solve targets.yaml is written per tag, every chained frame gets a world_T_camera stanza, and the stanza of a frame
    that could not be chained is removed, so that no stale pose is left behind.
    image_size = (width, height): calibrate the camera from the detections alone (needs initialise and targets, and
    excludes intr / dist, fixed intrinsics and intrinsics_sigma).  camera.yaml is neither read nor written; the start
    is initialiser.initialise_intrinsics with zero distortion, lens (default "radtan") is the model calibrated, and
    camera_refined.yaml carries image_size.  The summary gains "initial_intrinsics": {"intr", "problems_used"}."""
    from .problem import BAProblem
    if intrinsics_sigma is not None and not refine_intrinsics:
        raise ValueError("intrinsics_sigma puts a prior on refined intrinsics: it cannot be combined with fixed ones")
    if image_size is not None and (not initialise or not targets or intr is not None or dist is not None
                                   or not refine_intrinsics or intrinsics_sigma is not None):
        raise ValueError("image_size estimates the intrinsics from board detections: it needs initialise and targets "
                         "and excludes intr, dist, fixed intrinsics and intrinsics_sigma")
    initial = None
    if initialise:
        scene, tag_ids, frames, all_frames, tag_pose, boards, initial = _initialise_directory(
            directory, intr, dist, lens, targets, image_size, device)
    else:
        scene, tag_ids, frames = read_dataset(directory, intr=intr, dist=dist, lens=lens)
    scene.const_intr[:] = not refine_intrinsics
    scene.const_dist[:] = not refine_intrinsics
    tags = scene
    if targets and not initialise:
        scene, tag_pose, boards = board_scene(tags, tag_ids, read_targets(list(targets)))
    with BAProblem.from_scene(scene, device=device) as p:
        if intrinsics_sigma is not None:
            for kind, args in intrinsics_priors(scene.intr, scene.dist, intrinsics_sigma).items():
                p.set_priors(kind, *args)
        summary = p.solve(**lm_options)
        scene.views, scene.markers = p.get_view_poses(), p.get_marker_poses()
        intr, dist = p.get_intrinsics()
        scene.intr, scene.dist = intr, dist
    if targets:
        summary["boards"] = [{"first_tag_id": i, "world_T_board": scene.markers[j].tolist()} for i, j in boards]
    if initial is not None:
        summary["initial_intrinsics"] = initial
    if initialise:
        size_of = {int(t): float(sz) for fr in all_frames[1] for (t, sz, _) in fr}
        _write_poses(directory, tag_ids, [size_of[int(t)] for t in tag_ids], tag_pose(scene.markers), scene.views,
                     frames, precision)
        kept = set(frames.tolist())
        for n in all_frames[0].tolist():
            if n not in kept:
                _remove_stanza(os.path.join(directory, f"detections_{n}.yaml"))
    else:
        if targets:
            tags.views, tags.markers = scene.views, tag_pose(scene.markers)
            scene = tags
        write_results(directory, scene, tag_ids, frames, precision)
    if refine_intrinsics:
        with open(os.path.join(directory, "camera_refined.yaml"), "w") as f:
            f.write(camera_yaml_text(intr[0], dist[0], scene.image_size, lens=scene.lens))
    return summary
