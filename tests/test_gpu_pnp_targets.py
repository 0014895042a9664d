"""GPU: rigid-target PnP (rcc_pnp_target_batch, initialiser.pnp_targets / initialise_targets) against OpenCV on
make_target_scene data for both lenses, and the --initialise command line end to end."""
import copy
import os

import numpy as np
import pytest
import yaml

from robot_camera_calibration_b200 import initialiser, io_yaml
from robot_camera_calibration_b200.__main__ import main
from robot_camera_calibration_b200.scenes import (compose, invert, make_scene, make_target_scene, obj_points,
                                                  project_points, rodrigues_np)

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")


def _K(intr):
    return np.array([[intr[0], 0, intr[2]], [0, intr[1], intr[3]], [0, 0, 1.0]])


def _problems(s, sizes, rng):
    """(frame, board) problems of a one-board scene: for every view, one problem of each tag count in `sizes` that
    the view can fill (a random subset of its detected tags, shuffled), plus one shuffled partial subset of random
    size.  Returns (start, slot, pixels, truth cam_T_board, per problem the block indices)."""
    start, slot, pix, truth, blocks = [0], [], [], [], []
    for v in range(len(s.views)):
        sel = np.nonzero((s.view_idx == v) & (s.marker_idx == 0))[0]
        if len(sel) == 0:
            continue
        counts = [k for k in sizes if k <= len(sel)] + [int(rng.integers(1, len(sel) + 1))]
        for k in counts:
            b = rng.permutation(sel)[:k]
            slot += s.corner_slot[b].tolist()
            pix.append(s.pixels[b])
            start.append(len(slot))
            truth.append(compose(invert(s.truth["views"][v]), s.truth["markers"][0]))
            blocks.append(b)
    return (np.array(start), np.array(slot, np.int32), np.concatenate(pix).reshape(-1, 8), np.array(truth),
            blocks)


def _gn_polish(obj, img, K, dist, lens, x):
    """Gauss-Newton on OpenCV's own projection and Jacobian (cv2.projectPoints / cv2.fisheye.projectPoints) from x,
    with step halving, down to rounding."""
    r = img.reshape(-1)

    def proj(x):
        if lens == "radtan":
            uv, J = cv2.projectPoints(obj, x[:3].copy(), x[3:].copy(), K, dist[:5])
            return uv.reshape(-1) - r, J[:, :6]
        uv, J = cv2.fisheye.projectPoints(obj.reshape(-1, 1, 3), x[:3].copy(), x[3:].copy(), K, dist[:4])
        return uv.reshape(-1) - r, J[:, 8:14]
    res, J = proj(x)
    for _ in range(60):
        dx = np.linalg.lstsq(J, -res, rcond=None)[0]
        step = 1.0
        while True:
            x2 = x + step * dx
            res2, J2 = proj(x2)
            if res2 @ res2 <= res @ res * (1 + 1e-15) or step < 1e-6:
                break
            step *= 0.5
        x, res, J = x2, res2, J2
        if np.abs(step * dx).max() < 1e-15:
            break
    return x


def _cv2_pose(obj, img, K, dist, lens):
    """The pose OpenCV finds, polished to convergence: solvePnP(SOLVEPNP_ITERATIVE) + solvePnPRefineLM with a tight
    TermCriteria (radtan) or cv2.fisheye.solvePnP (equidistant), then Gauss-Newton on OpenCV's Jacobian."""
    if lens == "radtan":
        ok, rv, tv = cv2.solvePnP(obj, img, K, dist[:5], flags=cv2.SOLVEPNP_ITERATIVE)
        rv, tv = cv2.solvePnPRefineLM(obj, img, K, dist[:5], rv, tv,
                                      criteria=(cv2.TERM_CRITERIA_EPS + cv2.TERM_CRITERIA_COUNT, 1000, 1e-16))
    else:
        ok, rv, tv = cv2.fisheye.solvePnP(obj.reshape(1, -1, 3), img.reshape(1, -1, 2), K, dist[:4].reshape(4, 1))
    assert ok
    return _gn_polish(obj, img, K, dist, lens, np.concatenate([rv.ravel(), tv.ravel()]))


def _ippe_poses(obj, img, K, dist, lens):
    """Both poses of the planar ambiguity from OpenCV's IPPE, polished as _cv2_pose."""
    if lens == "radtan":
        n, rvs, tvs, _ = cv2.solvePnPGeneric(obj, img, K, dist[:5], flags=cv2.SOLVEPNP_IPPE)
    else:
        und = cv2.fisheye.undistortPoints(img.reshape(1, -1, 2), K, dist[:4].reshape(4, 1))
        n, rvs, tvs, _ = cv2.solvePnPGeneric(obj, und.reshape(-1, 2), np.eye(3), None, flags=cv2.SOLVEPNP_IPPE)
    return [_gn_polish(obj, img, K, dist, lens, np.concatenate([r.ravel(), t.ravel()])) for r, t in zip(rvs, tvs)]


def _obj(corners, slots):
    o = corners[slots].reshape(-1, 2)
    return np.concatenate([o, np.zeros((len(o), 1))], 1)


@pytest.fixture(scope="module", params=["radtan", "equidistant"])
def board_problems(request):
    lens = request.param
    s = make_target_scene(10, 10, 24, seed=5, lens=lens, distance=3.0)
    rng = np.random.default_rng(7)
    start, slot, pix, truth, blocks = _problems(s, (1, 8, 9, 36, 100), rng)
    return lens, s, start, slot, pix, truth


def test_pnp_targets_matches_polished_opencv(board_problems):
    lens, s, start, slot, pix, truth = board_problems
    tags = np.diff(start)
    for k in (1, 8, 9, 36, 100):              # 4, 32, 36, 144 and 400 corners
        assert (tags == k).sum() >= 3, k
    assert len(set(tags.tolist())) > 8       # and the random partial subsets
    intr, dist = s.truth["intr"][0], s.truth["dist"][0]
    poses, cost = initialiser.pnp_targets(intr, dist, s.corners, start, slot, pix, lens=lens)
    assert (cost >= 0).all()
    K = _K(intr)
    other_minimum = 0
    for p in range(len(tags)):
        sl = slice(start[p], start[p + 1])
        obj, img = _obj(s.corners, slot[sl]), pix[sl].reshape(-1, 2)
        ref = _cv2_pose(obj, img, K, dist, lens)
        err = np.abs(poses[p] - ref).max()
        if err > 1e-8 and tags[p] == 1:
            # one small tag: the planar pose ambiguity has two minima, and starts that differ in the last bits can
            # fall into either.  The pose must then be OpenCV's other minimum (IPPE's two solutions, polished).
            err = min(np.abs(poses[p] - r).max() for r in _ippe_poses(obj, img, K, dist, lens))
            other_minimum += 1
        assert err <= 1e-8, (p, tags[p], poses[p], ref)
    assert other_minimum <= 0.25 * (tags == 1).sum(), other_minimum
    # sanity against the truth: 0.3 px noise
    assert np.median(np.abs(poses[tags >= 8, 3:] - truth[tags >= 8, 3:])) < 0.01


def test_one_tag_problems_match_the_per_tag_pnp(board_problems):
    lens, s, start, slot, pix, truth = board_problems
    one = np.nonzero(np.diff(start) == 1)[0]
    px = pix[start[one]]
    sq = obj_points(np.array([s.sizes[0]]))[:, :, :2]          # the tag's own square as its slot
    poses, cost = initialiser.pnp_targets(s.truth["intr"][0], s.truth["dist"][0], sq, np.arange(len(one) + 1),
                                          np.zeros(len(one), np.int32), px, lens=lens)
    ref, ref_cost = initialiser.pnp_batch(s.truth["intr"][0], s.truth["dist"][0], np.full(len(one), s.sizes[0]), px,
                                          lens=lens)
    assert (cost >= 0).all() and (ref_cost >= 0).all()
    err = np.abs(poses - ref).max(1)
    # where the two starts fell into different minima of the planar ambiguity, both must be OpenCV's minima
    K = _K(s.truth["intr"][0])
    for j in np.nonzero(err > 1e-8)[0]:
        minima = _ippe_poses(obj_points(np.array([s.sizes[0]]))[0], px[j].reshape(4, 2), K, s.truth["dist"][0], lens)
        for x in (poses[j], ref[j]):
            assert min(np.abs(x - m).max() for m in minima) <= 1e-8, (j, x, minima)
    assert (err > 1e-8).sum() <= 0.25 * len(one), err


def test_guess_converges_to_the_same_minimiser(board_problems):
    lens, s, start, slot, pix, truth = board_problems
    intr, dist = s.truth["intr"][0], s.truth["dist"][0]
    big = np.diff(start) >= 8
    poses, _ = initialiser.pnp_targets(intr, dist, s.corners, start, slot, pix, lens=lens)
    guess = truth + np.random.default_rng(3).normal(0, [0.05] * 3 + [0.05] * 3, truth.shape)
    poses_g, cost_g = initialiser.pnp_targets(intr, dist, s.corners, start, slot, pix, guess=guess, lens=lens)
    assert (cost_g >= 0).all()
    assert np.abs(poses_g[big] - poses[big]).max() <= 1e-8


def test_target_behind_the_camera_fails_alone(board_problems):
    lens, s, start, slot, pix, truth = board_problems
    intr, dist = s.truth["intr"][0], s.truth["dist"][0]
    poses, cost = initialiser.pnp_targets(intr, dist, s.corners, start, slot, pix, lens=lens)
    # problem 3 moved behind the camera (t_z negated: every corner at negative depth), with the pixels that pose
    # projects to and the pose itself as the guess
    p = 3
    sl = slice(start[p], start[p + 1])
    behind = truth[p].copy()
    behind[5] = -behind[5]
    n = start[p + 1] - start[p]
    uv, Z = project_points("single", np.broadcast_to(intr, (n, 4)), np.broadcast_to(dist, (n, 5)), np.zeros((n, 6)),
                           np.zeros((n, 6)), np.broadcast_to(behind, (n, 6)),
                           np.concatenate([s.corners[slot[sl]], np.zeros((n, 4, 1))], -1), lens)
    assert (Z < 0).all()
    pix2 = pix.copy()
    pix2[sl] = uv.reshape(-1, 8)
    guess = np.zeros_like(truth)
    guess[p] = behind
    poses2, cost2 = initialiser.pnp_targets(intr, dist, s.corners, start, slot, pix2, guess=guess, lens=lens)
    assert cost2[p] == -1.0
    others = np.arange(len(cost)) != p
    assert np.array_equal(poses2[others], poses[others]) and np.array_equal(cost2[others], cost[others])


def test_results_are_bitwise_the_same_alone_in_any_batch_and_twice(board_problems):
    import torch
    from torch.profiler import ProfilerActivity, profile
    from test_pnp_targets_host import PNP_TARGET_LENSES
    lens, s, start, slot, pix, truth = board_problems
    intr, dist = s.truth["intr"][0], s.truth["dist"][0]
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        a, ca = initialiser.pnp_targets(intr, dist, s.corners, start, slot, pix, lens=lens)
        torch.cuda.synchronize()
    # the instantiation of this lens ran (test_pnp_targets_host.py checks that these are all there are)
    import re
    from test_gpu_kernel_matrix import _template_arg
    ran = {_template_arg(m.group(1).strip()) for m in (re.search(r"\bpnp_target_kernel<([^<>]*)>", e.name)
                                                       for e in prof.events()) if m}
    assert ran == {k for k, v in PNP_TARGET_LENSES.items() if v == lens}, ran
    b, cb = initialiser.pnp_targets(intr, dist, s.corners, start, slot, pix, lens=lens)
    assert np.array_equal(a, b) and np.array_equal(ca, cb)
    order = np.random.default_rng(11).permutation(len(a))
    st, sl, px = [0], [], []
    for p in order:
        sl.append(slot[start[p]:start[p + 1]]); px.append(pix[start[p]:start[p + 1]])
        st.append(st[-1] + start[p + 1] - start[p])
    c, cc = initialiser.pnp_targets(intr, dist, s.corners, st, np.concatenate(sl), np.concatenate(px), lens=lens)
    assert np.array_equal(c, a[order]) and np.array_equal(cc, ca[order])
    for p in range(0, len(a), 7):
        d, cd = initialiser.pnp_targets(intr, dist, s.corners, [0, start[p + 1] - start[p]],
                                        slot[start[p]:start[p + 1]], pix[start[p]:start[p + 1]], lens=lens)
        assert np.array_equal(d[0], a[p]) and cd[0] == ca[p]


# ------------------------------------------------------------------ initialise_targets
def _frames(s, first_ids, rng):
    """frames_pixels of a target scene: board b's tag in slot k has id first_ids[b] + k, free tag j id 1000 + j;
    detections shuffled, with board 0's slot-0 tag first in frame 0 when it is seen (the world tag)."""
    n_boards = len(first_ids)
    frames = []
    for v in range(len(s.views)):
        sel = rng.permutation(np.nonzero(s.view_idx == v)[0])
        fr = []
        for b in sel:
            m = int(s.marker_idx[b])
            tid = first_ids[m] + int(s.corner_slot[b]) if m < n_boards else 1000 + m - n_boards
            fr.append((tid, float(s.sizes[m]), s.pixels[b].copy()))
        if v == 0:
            fr.sort(key=lambda t: t[0] != first_ids[0])
        frames.append(fr)
    return frames


def _targets(s, first_ids):
    n = len(s.corners)
    return [(f + np.arange(n), s.corners) for f in first_ids]


def _restatement(frames, intr, dist, targets, lens):
    """initialise_targets restated with OpenCV: polished solvePnP per (frame, target) (free tags: one pnp_batch call
    each), then chain_poses over the entities and the move to the world tag's frame."""
    K = _K(intr)
    where = {int(i): (b, b * len(targets[0][0]) + k) for b, (ids, _) in enumerate(targets) for k, i in enumerate(ids)}
    corners = np.concatenate([c for _, c in targets])
    ent_frames, cTe = [], []
    for fr in frames:
        ents = initialiser.group_entities(fr, where)
        poses = []
        for key, ks in ents:
            if key[0] == "target":
                img = np.concatenate([fr[k][2] for k in ks]).reshape(-1, 2)
                poses.append(_cv2_pose(_obj(corners, [where[fr[k][0]][1] for k in ks]), img, K, dist, lens))
            else:   # free tags keep the per-tag PnP (compared with cv2.solvePnP in test_initialiser.py)
                poses.append(initialiser.pnp_batch(intr, dist, [fr[ks[0]][1]], fr[ks[0]][2], lens=lens)[0][0])
        ent_frames.append([(key, 0.0) for key, _ in ents])
        cTe.append(np.array(poses).reshape(-1, 6))
    keys, _, w_T_e, w_T_cam = initialiser.chain_poses(ent_frames, cTe)
    if keys[0][0] == "target":
        w_T_b = invert(initialiser.board_T_tag(corners[where[frames[0][0][0]][1]]))
        w_T_e = compose(np.broadcast_to(w_T_b, w_T_e.shape), w_T_e)
        w_T_cam = [None if x is None else compose(w_T_b, x) for x in w_T_cam]
    return keys, w_T_e, w_T_cam


def _rot_err(a, b):
    R = np.einsum('nji,njk->nik', rodrigues_np(a[:, :3]), rodrigues_np(b[:, :3]))
    return np.arccos(np.clip((np.trace(R, axis1=1, axis2=2) - 1) / 2, -1, 1))


@pytest.mark.parametrize("lens,n_free", [("radtan", 3), ("equidistant", 0)])
def test_initialise_targets_matches_the_cv2_restatement(lens, n_free):
    s = make_target_scene(6, 6, 30, n_boards=2, n_free=n_free, seed=21, lens=lens)
    first = [0, 100]
    frames = _frames(s, first, np.random.default_rng(2))
    intr, dist = s.truth["intr"][0], s.truth["dist"][0]
    targets = _targets(s, first)
    scene, ids, keep, tag_pose, boards = initialiser.initialise_targets(frames, intr, dist, targets, lens=lens)
    keys, w_T_e, w_T_cam = _restatement(frames, intr, dist, targets, lens)
    assert list(keep) == [n for n, t in enumerate(w_T_cam) if t is not None]
    assert scene.markers.shape == w_T_e.shape
    assert np.abs(rodrigues_np(scene.markers[:, :3]) - rodrigues_np(w_T_e[:, :3])).max() < 1e-6
    assert np.abs(scene.markers[:, 3:] - w_T_e[:, 3:]).max() < 1e-6
    ref_views = np.array([w_T_cam[n] for n in keep])
    assert np.abs(rodrigues_np(scene.views[:, :3]) - rodrigues_np(ref_views[:, :3])).max() < 1e-6
    assert np.abs(scene.views[:, 3:] - ref_views[:, 3:]).max() < 1e-6
    assert [b for b, _ in boards] == first and ids[0] == 0


@pytest.mark.parametrize("lens", ["radtan", "equidistant"])
def test_board_pnp_beats_per_tag_pnp_and_feeds_the_bundle_adjustment(lens):
    from robot_camera_calibration_b200.problem import BAProblem
    s = make_target_scene(6, 6, 40, n_boards=2, seed=31, lens=lens, tag_size=0.06, distance=3.0)
    first = [0, 100]
    frames = _frames(s, first, np.random.default_rng(4))
    intr, dist = s.truth["intr"][0], s.truth["dist"][0]
    targets = _targets(s, first)
    scene, ids, keep, tag_pose, boards = initialiser.initialise_targets(frames, intr, dist, targets, lens=lens)
    tags, tag_ids, keep_t = initialiser.initialise(frames, intr, dist, lens=lens)
    per_tag, _, _ = io_yaml.board_scene(tags, tag_ids, targets)
    # truth in the world tag's frame (board 0's slot 0)
    w_T_g = invert(compose(s.truth["markers"][0], initialiser.board_T_tag(s.corners[0])))
    true_views = compose(np.broadcast_to(w_T_g, s.truth["views"].shape), s.truth["views"])
    err = lambda v, k: (np.median(_rot_err(v, true_views[k])), np.median(np.linalg.norm(v[:, 3:] - true_views[k, 3:],
                                                                                          axis=1)))
    r_board, t_board = err(scene.views, keep)
    r_tag, t_tag = err(per_tag.views, keep_t)
    assert r_board < r_tag and t_board < t_tag, (r_board, r_tag, t_board, t_tag)
    # the bundle adjustment converges from it to the minimum it reaches from the truth
    scene.const_intr[:] = True
    scene.const_dist[:] = True
    from_truth = copy.deepcopy(scene)
    from_truth.views = true_views[keep]
    for first_id, m in boards:
        from_truth.markers[m] = compose(w_T_g, s.truth["markers"][first.index(first_id)])
    assert len(boards) == len(scene.markers)
    out = []
    for sc in (scene, from_truth):
        with BAProblem.from_scene(sc) as p:
            summ = p.solve(max_iterations=50)
            out.append((summ, p.get_view_poses()))
    (summ, views), (_, views_t) = out
    assert summ["termination"] in (1, 2, 3), summ
    assert summ["final_cost"] < 0.5 * scene.n_blocks          # 0.3 px noise: 0.36 per block
    assert np.abs(views - views_t).max() < 1e-4


# ------------------------------------------------------------------ the command line, end to end
def _write_grid(path, rows, cols, size, spacing, first):
    with open(path, "w") as f:
        f.write(f"target_type: aprilgrid\ntagRows: {rows}\ntagCols: {cols}\ntagSize: {size}\ntagSpacing: {spacing}\n"
                f"firstTagId: {first}\n")


def _stanza_views(d, numbers):
    out = []
    for n in numbers:
        with open(os.path.join(d, f"detections_{n}.yaml")) as f:
            y = yaml.safe_load(f)
        out.append(list(y["world_T_camera"]["rotation"]) + list(y["world_T_camera"]["translation"]))
    return np.array(out)


def test_command_line_initialises_boards_from_detections_alone(tmp_path):
    d = str(tmp_path)
    s = make_target_scene(5, 6, 20, n_boards=2, seed=41, pixel_noise=0.0)
    first = [0, 100]
    frames = _frames(s, first, np.random.default_rng(5))
    for n, fr in enumerate(frames):
        c = np.round(np.array([p for _, _, p in fr])).astype(np.int64).reshape(-1, 4, 2)
        with open(os.path.join(d, f"detections_{n}.yaml"), "w") as f:
            f.write(io_yaml.detections_text([t for t, _, _ in fr], [sz for _, sz, _ in fr], c))
    with open(os.path.join(d, "camera.yaml"), "w") as f:
        f.write(io_yaml.camera_yaml_text(s.truth["intr"][0], s.truth["dist"][0]))
    g = [os.path.join(d, "grid0.yaml"), os.path.join(d, "grid1.yaml")]
    for path, f0 in zip(g, first):
        _write_grid(path, 5, 6, 0.1, 0.3, f0)
    assert main([d, "--initialise", "--target", g[0], "--target", g[1], "--fix-intrinsics"]) == 0
    assert os.path.exists(os.path.join(d, "targets.yaml"))
    views = _stanza_views(d, range(len(frames)))
    w_T_g = invert(compose(s.truth["markers"][0], initialiser.board_T_tag(s.corners[0])))
    true_views = compose(np.broadcast_to(w_T_g, s.truth["views"].shape), s.truth["views"])
    # rounding to whole pixels is ~0.3 px of noise
    assert np.median(_rot_err(views, true_views)) < 2e-3
    assert np.median(np.linalg.norm(views[:, 3:] - true_views[:, 3:], axis=1)) < 5e-3
    # targets.yaml holds every detected tag; the world tag at the identity
    scene, tag_ids, numbers = io_yaml.read_dataset(d)
    assert tag_ids[0] == 0 and np.abs(scene.markers[0]).max() < 1e-6
    assert set(tag_ids.tolist()) == {t for fr in frames for t, _, _ in fr}


def test_command_line_initialises_free_tags_and_drops_stale_stanzas(tmp_path):
    d = str(tmp_path)
    s = make_scene(12, 16, 0.7, seed=43, pixel_noise=0.0)
    io_yaml.write_dataset(d, s, with_poses=False)
    os.remove(os.path.join(d, "targets.yaml"))
    with open(os.path.join(d, "camera.yaml"), "w") as f:
        f.write(io_yaml.camera_yaml_text(s.truth["intr"][0], s.truth["dist"][0]))
    # a frame that cannot be chained (an unknown tag), with an old stanza
    n_stale = len(s.views)
    with open(os.path.join(d, f"detections_{n_stale}.yaml"), "w") as f:
        f.write(io_yaml.detections_text([999], [0.1], np.full((1, 4, 2), 50) + np.array([[0, 0], [9, 0], [9, 9], [0, 9]]))
                + io_yaml.world_T_camera_text([0, 0, 0], [1, 2, 3]))
    assert main([d, "--initialise", "--fix-intrinsics"]) == 0
    with open(os.path.join(d, f"detections_{n_stale}.yaml")) as f:
        assert "world_T_camera" not in f.read()
    views = _stanza_views(d, range(len(s.views)))
    # the world is one small tag, whose orientation is known to ~1e-2: compare camera poses relative to frame 0
    rel = lambda v: compose(np.broadcast_to(invert(v[0]), v.shape), v)
    got, want = rel(views), rel(s.truth["views"])
    assert np.median(_rot_err(got, want)) < 5e-3
    assert np.median(np.linalg.norm(got[:, 3:] - want[:, 3:], axis=1)) < 2e-2
