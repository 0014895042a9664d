"""Pose initialisation (the reference's camera_pose_node, SURVEY.md 8f-2) with the
per-tag PnP batched on the GPU.

Mirrors PoseSystem in /root/reference/real_preprocessing/src/camera_pose.cpp:
  tagTcam   :132-173  per-tag cv::solvePnP            -> rcc_pnp_batch (all tags of all frames at once)
  worldLoad :71-80    first tag of frame 0 = world tag, pose identity
  fileReader:207-246  frame status: world tag present > known tag present > unknown
  tagCalc   :176-203  w_T_cam = w_T_tag * tag_T_cam ; new tags: w_T_tag = w_T_cam * cam_T_tag
  unknownFilepoll :249-263 / fileStream :267-285  deferred frames are retried, last first
The pose chaining itself is a few 4x4 products per frame and stays on the host.
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
