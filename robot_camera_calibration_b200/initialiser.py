"""Pose initialisation (the reference's camera_pose_node, SURVEY.md 8f-2) with the
per-tag PnP batched on the GPU.

Mirrors PoseSystem in /root/reference/real_preprocessing/src/camera_pose.cpp:
  tagTcam   :132-173  per-tag cv::solvePnP            -> rcc_pnp_batch (all tags of all frames at once)
  worldLoad :71-80    first tag of frame 0 = world tag, pose identity
  fileReader:207-246  frame status: world tag present > known tag present > unknown
  tagCalc   :176-203  w_T_cam = w_T_tag * tag_T_cam ; new tags: w_T_tag = w_T_cam * cam_T_tag
  unknownFilepoll :249-263 / fileStream :267-285  deferred frames are retried, last first
The pose chaining itself is a few 4x4 products per frame and stays on the host.

initialise_targets does the same for rigid tag boards (io_yaml.read_targets): one PnP per (frame, board) over all
of the board's detected corners (rcc_pnp_target_batch), as cv::calibrateCamera and Kalibr start a board, and the
same chaining with a board or a free tag in place of each tag.

initialise_intrinsics gives a camera without known intrinsics its start, as cv::initCameraMatrix2D does for
cv::calibrateCamera: one plane homography per (frame, board) on the GPU (rcc_homography_target_batch) and
OpenCV's closed form for fx and fy with the principal point at the image centre.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib as L
from .scenes import Scene, compose, invert


def pnp_batch(intr, dist, sizes, pixels, guess=None, device=0, max_iterations=100, lens="radtan"):
    """cam_T_tag (n,6) and final cost (n,) for n tags (4 corners each) on the GPU.  lens "radtan" (dist = k1 k2 p1 p2
    k3) or "equidistant" (dist = k1 k2 k3 k4); missing trailing coefficients are zero."""
    lib = L.load()
    if lens not in L.LENSES:
        raise ValueError(f"unknown lens {lens!r}: expected one of {sorted(L.LENSES)}")
    sizes = np.ascontiguousarray(sizes, np.float64)
    pixels = np.ascontiguousarray(pixels, np.float64).reshape(-1, 8)
    n = len(sizes)
    d = np.asarray(dist, float).ravel()[:5]
    sh = np.ascontiguousarray(np.concatenate([np.asarray(intr, float).ravel()[:4], d, np.zeros(5 - len(d))]))
    poses = np.zeros((n, 6)) if guess is None else np.ascontiguousarray(guess, np.float64).reshape(n, 6).copy()
    cost = np.empty(n)
    dp = lambda a: a.ctypes.data_as(L.c_double_p)
    rc = lib.rcc_pnp_batch_lens(int(device), L.LENSES[lens], n, dp(sh), dp(sizes), dp(pixels), dp(poses), dp(cost),
                                int(max_iterations))
    if rc != L.RCC_OK:
        raise L.RccError(rc, "rcc_pnp_batch failed (no CPU fallback)")
    return poses, cost


def pnp_targets(intr, dist, corners, start, slot, pixels, guess=None, device=0, max_iterations=100, lens="radtan"):
    """cam_T_target (n,6) and final cost (n,) of n rigid-target problems on the GPU.  corners (n_slots,4,2): the
    corners bl br tr tl of each layout slot in the target frame; problem p owns the tags [start[p], start[p + 1]) of
    slot (tag's layout slot) and pixels (tag's 8 pixels).  A zero guess row starts from the DLT homography of the
    problem's corners.  Cost -1: a corner behind the camera or a non-finite residual.  lens and dist as in
    pnp_batch."""
    lib = L.load()
    if lens not in L.LENSES:
        raise ValueError(f"unknown lens {lens!r}: expected one of {sorted(L.LENSES)}")
    corners = np.ascontiguousarray(corners, np.float64).reshape(-1, 8)
    start = np.ascontiguousarray(start, np.int64).ravel()
    slot = np.ascontiguousarray(slot, np.int32).ravel()
    pixels = np.ascontiguousarray(pixels, np.float64).reshape(-1, 8)
    n = max(len(start) - 1, 0)
    if len(start) == 0 or len(slot) != start[-1] or len(pixels) != len(slot):
        raise ValueError(f"start ({len(start)}) must end at the number of tags: slot has {len(slot)}, "
                         f"pixels {len(pixels)}")
    d = np.asarray(dist, float).ravel()[:5]
    sh = np.ascontiguousarray(np.concatenate([np.asarray(intr, float).ravel()[:4], d, np.zeros(5 - len(d))]))
    poses = np.zeros((n, 6)) if guess is None else np.ascontiguousarray(guess, np.float64).reshape(n, 6).copy()
    cost = np.empty(n)
    dp = lambda a: a.ctypes.data_as(L.c_double_p)
    rc = lib.rcc_pnp_target_batch(int(device), L.LENSES[lens], dp(sh), len(corners), dp(corners), n,
                                  start.ctypes.data_as(L.c_int64_p), slot.ctypes.data_as(L.c_int32_p), dp(pixels),
                                  dp(poses), dp(cost), int(max_iterations))
    if rc != L.RCC_OK:
        raise L.RccError(rc, "rcc_pnp_target_batch failed (no CPU fallback)")
    return poses, cost


WORLD_PRES, KNOWN_TAG, UNKNOWN = 0, 1, 2      # camera_pose.cpp:11-13


def chain_poses(frames, cam_T_tag):
    """frames: list of lists of (tag_id, size); cam_T_tag: matching list of (k,6)
    arrays.  Returns (tag_ids, tag_sizes, w_T_tag (m,6), w_T_cam list (6,) or None)
    following the reference's processing order exactly."""
    ids, sizes, poses = [], [], []
    w_T_cam = [None] * len(frames)
    if not frames or not frames[0]:
        return ids, sizes, np.zeros((0, 6)), w_T_cam
    world = frames[0][0][0]                                   # worldLoad, :74
    ids.append(world); sizes.append(frames[0][0][1]); poses.append(np.zeros(6))

    def status(n):                                            # fileReader, :207-246
        if n == 0:
            return WORLD_PRES, 0
        st, known = UNKNOWN, -1
        for k, (tid, _) in enumerate(frames[n]):
            if tid == world:
                return WORLD_PRES, k
            if tid in ids:
                known, st = k, KNOWN_TAG                      # the LAST known tag wins (:236-240)
        return st, known

    def tag_calc(n, known):                                   # tagCalc, :176-203
        tid = frames[n][known][0]
        wTc = compose(poses[ids.index(tid)], invert(cam_T_tag[n][known]))
        w_T_cam[n] = wTc
        for k, (t, sz) in enumerate(frames[n]):
            if k != known and t not in ids:
                poses.append(compose(wTc, cam_T_tag[n][k]))
                ids.append(t); sizes.append(sz)

    deferred = []
    for n in range(len(frames)):                              # fileStream, :267-285
        if not frames[n]:
            continue
        st, known = status(n)
        if st in (WORLD_PRES, KNOWN_TAG):
            tag_calc(n, known)
            for j in range(len(deferred) - 1, -1, -1):        # unknownFilepoll, :249-263
                st2, k2 = status(deferred[j])
                if st2 == KNOWN_TAG:
                    tag_calc(deferred[j], k2)
                    deferred.pop(j)
        else:
            deferred.append(n)
    return ids, sizes, np.array(poses).reshape(-1, 6), w_T_cam


def initialise(frames_pixels, intr, dist, device=0, lens="radtan"):
    """frames_pixels: list (per frame) of lists of (tag_id, size, pixels8).
    Returns a Scene holding the initial guesses (frames never referenced are dropped,
    like the reference leaves them without a world_T_camera stanza), the tag ids and
    the frame numbers kept."""
    flat_sizes = [sz for fr in frames_pixels for (_, sz, _) in fr]
    flat_pix = [px for fr in frames_pixels for (_, _, px) in fr]
    poses, _ = pnp_batch(intr, dist, flat_sizes, np.array(flat_pix).reshape(-1, 8), device=device, lens=lens)
    per_frame, o = [], 0
    for fr in frames_pixels:
        per_frame.append(poses[o:o + len(fr)])
        o += len(fr)
    frames = [[(t, s) for (t, s, _) in fr] for fr in frames_pixels]
    ids, sizes, w_T_tag, w_T_cam = chain_poses(frames, per_frame)
    keep = [n for n in range(len(frames)) if w_T_cam[n] is not None]
    index_of = {t: i for i, t in enumerate(ids)}
    vi, mi, px = [], [], []
    for v, n in enumerate(keep):
        for (t, _, p) in frames_pixels[n]:
            if t in index_of:
                vi.append(v); mi.append(index_of[t]); px.append(p)
    d = np.asarray(dist, float).ravel()
    scene = Scene(model="single", intr=np.asarray(intr, float).reshape(1, 4),
                  dist=np.concatenate([d, np.zeros(5 - len(d))]).reshape(1, 5), lens=lens,
                  ext=np.zeros((1, 6)), views=np.array([w_T_cam[n] for n in keep]).reshape(-1, 6), markers=w_T_tag,
                  sizes=np.array(sizes, float), view_idx=np.array(vi, np.int32), marker_idx=np.array(mi, np.int32),
                  cam_idx=np.zeros(len(vi), np.int32), pixels=np.array(px, float).reshape(-1, 8))
    return scene, np.array(ids), np.array(keep)


def board_T_tag(corners):
    """The frame of a tag on a board: centred on its corners (4,2), with the board's axes."""
    ctr = np.asarray(corners, float).reshape(4, 2).mean(0)
    return np.array([0.0, 0.0, 0.0, ctr[0], ctr[1], 0.0])


def group_entities(frame, where):
    """The entities of one frame's detections [(tag_id, size, pixels8)]: one per target with a detected tag, keyed
    ("target", b), and one per free tag, keyed ("tag", id), in the order of their first detection.  where: tag id ->
    (target, slot).  Returns [(key, [detection index, ..])]."""
    order, members = [], {}
    for k, (t, _, _) in enumerate(frame):
        w = where.get(int(t))
        key = ("target", w[0]) if w is not None else ("tag", int(t))
        if key not in members:
            members[key] = []
            order.append(key)
        members[key].append(k)
    return [(key, members[key]) for key in order]


def _entity_problems(frames_pixels, targets):
    """The problems of initialise_targets: where (tag id -> (target, slot)), the corner layout (n_slots,4,2), each
    frame's group_entities, the target problems (start, slot, pixels) in the order of the frames and their entities,
    and the free tags (sizes, pixels) in the same order."""
    where, offset = {}, 0
    for b, (ids, _) in enumerate(targets):
        for k, i in enumerate(np.asarray(ids).tolist()):
            where[int(i)] = (b, offset + k)
        offset += len(ids)
    corners = (np.concatenate([np.asarray(c, float).reshape(-1, 4, 2) for _, c in targets]) if targets
               else np.zeros((0, 4, 2)))
    grouped = [group_entities(fr, where) for fr in frames_pixels]
    # one target problem per (frame, target entity), one pnp_batch row per free tag
    t_start, t_slot, t_pix, f_size, f_pix = [0], [], [], [], []
    for fr, ents in zip(frames_pixels, grouped):
        for key, ks in ents:
            if key[0] == "target":
                t_slot += [where[int(fr[k][0])][1] for k in ks]
                t_pix += [fr[k][2] for k in ks]
                t_start.append(len(t_slot))
            else:
                f_size.append(fr[ks[0]][1])
                f_pix.append(fr[ks[0]][2])
    return where, corners, grouped, (t_start, t_slot, t_pix), (f_size, f_pix)


def homographies(corners, start, slot, pixels, device=0, max_iterations=100):
    """H (n,3,3) and final cost (n,) of n rigid-target problems on the GPU (rcc_homography_target_batch): the plane
    homography (X, Y, 1) in the target frame -> (u, v, 1) in raw pixels, scaled to H[2,2] = 1, that minimises the
    pixel reprojection error of the problem's corners (cv2.findHomography, method 0, refined to convergence).
    corners, start, slot and pixels as in pnp_targets.  Cost -1 (and H zero): a singular DLT, a non-finite residual
    or a corner on or behind the horizon of the plane (w <= 0)."""
    lib = L.load()
    corners = np.ascontiguousarray(corners, np.float64).reshape(-1, 8)
    start = np.ascontiguousarray(start, np.int64).ravel()
    slot = np.ascontiguousarray(slot, np.int32).ravel()
    pixels = np.ascontiguousarray(pixels, np.float64).reshape(-1, 8)
    n = max(len(start) - 1, 0)
    if len(start) == 0 or len(slot) != start[-1] or len(pixels) != len(slot):
        raise ValueError(f"start ({len(start)}) must end at the number of tags: slot has {len(slot)}, "
                         f"pixels {len(pixels)}")
    H = np.zeros((n, 9))
    cost = np.empty(n)
    dp = lambda a: a.ctypes.data_as(L.c_double_p)
    rc = lib.rcc_homography_target_batch(int(device), len(corners), dp(corners), n, start.ctypes.data_as(L.c_int64_p),
                                         slot.ctypes.data_as(L.c_int32_p), dp(pixels), dp(H), dp(cost),
                                         int(max_iterations))
    if rc != L.RCC_OK:
        raise L.RccError(rc, "rcc_homography_target_batch failed (no CPU fallback)")
    return H.reshape(n, 3, 3), cost


_UNCONSTRAINED = "the views do not constrain the focal length -- tilt the board"


def intrinsics_from_homographies(H, image_size):
    """intr = (fx, fy, cx, cy) from plane homographies H (n,3,3) of views of a plane and the image size (W, H): the
    closed form of OpenCV's initIntrinsicParams2D (cv2.initCameraMatrix2D with aspectRatio = 0), restated.  The
    principal point is the image centre ((W - 1)/2, (H - 1)/2); with it subtracted, each homography's columns h, v
    and d1 = (h + v)/2, d2 = (h - v)/2 (of the columns before normalisation, each then normalised) give Zhang's two
    orthogonality rows in (1/fx^2, 1/fy^2), solved by least squares over all views.
    One intended difference from OpenCV: where OpenCV takes the absolute value of a solution that is not positive,
    this raises ValueError, as it does when the 2x2 normal matrix is singular or has a condition number above 1e12 --
    views that do not constrain the focal length (all fronto-parallel, say) give no start at all rather than a wrong
    one."""
    H = np.asarray(H, np.float64).reshape(-1, 3, 3)
    cx, cy = (float(image_size[0]) - 1) * 0.5, (float(image_size[1]) - 1) * 0.5
    A, b = np.empty((2 * len(H), 2)), np.empty(2 * len(H))
    for i, h in enumerate(H):
        h = h.copy()
        h[0] -= h[2] * cx
        h[1] -= h[2] * cy
        t0, t1 = h[:, 0], h[:, 1]
        d1, d2 = (t0 + t1) * 0.5, (t0 - t1) * 0.5
        t0, t1, d1, d2 = (x / np.sqrt(x @ x) for x in (t0, t1, d1, d2))
        A[2 * i] = t0[0] * t1[0], t0[1] * t1[1]
        A[2 * i + 1] = d1[0] * d2[0], d1[1] * d2[1]
        b[2 * i], b[2 * i + 1] = -t0[2] * t1[2], -d1[2] * d2[2]
    N = A.T @ A
    if not len(H) or not np.isfinite(N).all() or not np.linalg.cond(N) <= 1e12:
        raise ValueError(_UNCONSTRAINED)
    f = np.linalg.solve(N, A.T @ b)
    if not (f > 0).all():
        raise ValueError(_UNCONSTRAINED)
    return np.array([np.sqrt(1.0 / f[0]), np.sqrt(1.0 / f[1]), cx, cy])


def initialise_intrinsics(frames_pixels, targets, image_size, device=0, min_tags=4):
    """A pinhole start (fx, fy, cx, cy) for a camera from board detections alone, as cv2.initCameraMatrix2D gives
    cv2.calibrateCamera's: one homography per (frame, target) problem of initialise_targets with at least min_tags
    detected tags of the target (homographies, on the GPU), then intrinsics_from_homographies.  Free tags never
    contribute: the homography of one small tag's 4 corners is too noisy to constrain the focal length.  Returns
    (intr, number of problems used).  ValueError when no problem qualifies or the views do not constrain the focal
    length.
    The start is meant for initialise_targets(frames_pixels, intr, zeros(5), targets, lens=...) with either lens,
    distortion starting at zero as in OpenCV.  For the equidistant lens the pinhole start is an approximation that
    holds for boards seen within a moderate field of view; boards seen near 90 degrees off the optical axis have not
    been verified."""
    where, corners, grouped, (t_start, t_slot, t_pix), _ = _entity_problems(frames_pixels, targets)
    n_tags = np.diff(t_start)
    use = np.nonzero(n_tags >= min_tags)[0]
    if len(use) == 0:
        raise ValueError(f"no (frame, board) problem has {min_tags} or more detected tags of a board: the intrinsics "
                         "are estimated from board views only (free tags are too small to constrain them)")
    start = np.concatenate([[0], np.cumsum(n_tags[use])])
    sel = np.concatenate([np.arange(t_start[p], t_start[p + 1]) for p in use])
    H, cost = homographies(corners, start, np.asarray(t_slot, np.int32)[sel],
                           np.array(t_pix, float).reshape(-1, 8)[sel], device=device)
    good = cost >= 0
    if not good.any():
        raise ValueError("no board view gave a homography")
    return intrinsics_from_homographies(H[good], image_size), int(good.sum())


def initialise_targets(frames_pixels, intr, dist, targets, device=0, lens="radtan"):
    """initialise() with rigid targets: targets = io_yaml.read_targets(...) [(tag ids, corners (n,4,2))].
    Each frame's detections are grouped into entities (group_entities): a target's cam_T_target comes from one
    pnp_targets problem over all its detected corners in the frame, a free tag's from pnp_batch.  The entities are
    chained by chain_poses exactly as tags are (camera_pose.cpp: the world entity first, the last known entity wins,
    deferred frames retried).  The world is the frame of the first tag of frame 0 (camera_pose.cpp:71-80): when
    that tag is on a target, the target's pose is invert(board_T_tag) of it, and the target is held constant.
    Returns (scene, tag_ids, kept_frames, tag_pose, boards) as io_yaml.board_scene: the scene (marker 0 the world
    entity, then the entities in the order they were chained) carries the corner layout; tag_ids are the detected
    tags of the chained entities, the world tag first; tag_pose(markers) -> world_T_tag of every tag of tag_ids;
    boards = [(first tag id of the target, marker block)] in target order."""
    where, corners, grouped, (t_start, t_slot, t_pix), (f_size, f_pix) = _entity_problems(frames_pixels, targets)
    t_pose = (pnp_targets(intr, dist, corners, t_start, t_slot, np.array(t_pix, float).reshape(-1, 8),
                          device=device, lens=lens)[0] if len(t_start) > 1 else np.zeros((0, 6)))
    f_pose = (pnp_batch(intr, dist, f_size, np.array(f_pix, float).reshape(-1, 8), device=device, lens=lens)[0]
              if f_size else np.zeros((0, 6)))
    frames, cTe, it, jf = [], [], 0, 0
    for fr, ents in zip(frames_pixels, grouped):
        poses = []
        for key, ks in ents:
            if key[0] == "target":
                poses.append(t_pose[it]); it += 1
            else:
                poses.append(f_pose[jf]); jf += 1
        frames.append([(key, fr[ks[0]][1]) for key, ks in ents])
        cTe.append(np.array(poses).reshape(-1, 6))
    keys, _, w_T_e, w_T_cam = chain_poses(frames, cTe)
    if keys and keys[0][0] == "target":
        # the chain's world is the target's frame: move it to the world tag's, world_T_target = invert(board_T_tag)
        w_T_b = invert(board_T_tag(corners[where[int(frames_pixels[0][0][0])][1]]))
        w_T_e = compose(np.broadcast_to(w_T_b, w_T_e.shape), w_T_e)
        w_T_cam = [None if x is None else compose(w_T_b, x) for x in w_T_cam]
    keep = [n for n in range(len(frames)) if w_T_cam[n] is not None]
    marker_of = {key: m for m, key in enumerate(keys)}
    vi, mi, sl, px, tags, sizes = [], [], [], [], {}, np.zeros(len(keys))
    for v, n in enumerate(keep):
        for key, ks in grouped[n]:
            for k in ks:
                t, sz, p = frames_pixels[n][k]
                vi.append(v); mi.append(marker_of[key]); px.append(p)
                sl.append(where[int(t)][1] if key[0] == "target" else -1)
                tags.setdefault(int(t), (marker_of[key], sl[-1]))
                if sizes[marker_of[key]] == 0:
                    sizes[marker_of[key]] = sz
    world_tag = int(frames_pixels[0][0][0]) if keys else None
    tag_ids = sorted(tags, key=lambda t: (t != world_tag, tags[t][0], tags[t][1]))
    pix = np.array(px).reshape(-1, 8)
    if not np.issubdtype(pix.dtype, np.integer):
        pix = pix.astype(np.float64)
    elif pix.size and pix.min() >= -32768 and pix.max() <= 32767:
        pix = pix.astype(np.int16)
    d = np.asarray(dist, float).ravel()
    scene = Scene(model="single", intr=np.asarray(intr, float).reshape(1, 4),
                  dist=np.concatenate([d, np.zeros(5 - len(d))]).reshape(1, 5), lens=lens,
                  ext=np.zeros((1, 6)), views=np.array([w_T_cam[n] for n in keep]).reshape(-1, 6),
                  markers=np.asarray(w_T_e, float).reshape(-1, 6), sizes=sizes, view_idx=np.array(vi, np.int32),
                  marker_idx=np.array(mi, np.int32), cam_idx=np.zeros(len(vi), np.int32), pixels=pix,
                  corners=corners, corner_slot=np.array(sl, np.int32))

    def tag_pose(markers):
        out = np.empty((len(tag_ids), 6))
        for j, t in enumerate(tag_ids):
            m, s = tags[t]
            out[j] = markers[m] if s < 0 else compose(markers[m], board_T_tag(corners[s]))
        return out

    boards = [(int(targets[key[1]][0][0]), marker_of[key]) for key in sorted(k for k in keys if k[0] == "target")]
    return scene, np.array(tag_ids, dtype=np.int64), np.array(keep, dtype=np.int64), tag_pose, boards
