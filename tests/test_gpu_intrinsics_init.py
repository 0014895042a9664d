"""GPU: camera intrinsics from board detections alone -- rcc_homography_target_batch (initialiser.homographies)
against polished cv2.findHomography, initialiser.initialise_intrinsics against cv2.initCameraMatrix2D, calibrations
started from it against the same solves started from the truth and against cv2.calibrateCamera /
cv2.fisheye.calibrate, and --initialise --target --image-size end to end."""
import copy
import os

import numpy as np
import pytest
import yaml

from robot_camera_calibration_b200 import initialiser, io_yaml
from robot_camera_calibration_b200.__main__ import main
from robot_camera_calibration_b200.problem import BAProblem
from robot_camera_calibration_b200.scenes import compose, invert, make_target_scene
from test_gpu_pnp_targets import _frames, _problems, _stanza_views, _targets, _write_grid

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")


def _apply(H, obj):
    w = H[2, 0] * obj[:, 0] + H[2, 1] * obj[:, 1] + H[2, 2]
    return np.stack([(H[0, 0] * obj[:, 0] + H[0, 1] * obj[:, 1] + H[0, 2]) / w,
                     (H[1, 0] * obj[:, 0] + H[1, 1] * obj[:, 1] + H[1, 2]) / w], 1)


def _gn_polish(obj, img, H):
    """Gauss-Newton on the 8 entries of H (H[2,2] = 1) over the pixel residual H(X) - u, down to rounding: the cost
    cv2.findHomography's refinement minimises, run to convergence.  The columns of J are scaled to unit norm (the
    entries differ by ~1e5 in size); a step is halved while it raises the cost, except below 1e-8 relative, where the
    cost comparison is rounding noise and the Gauss-Newton step is taken."""
    h = (H / H[2, 2]).reshape(-1)[:8].copy()

    def res_jac(h):
        Hm = np.append(h, 1.0).reshape(3, 3)
        X, Y = obj[:, 0], obj[:, 1]
        w = Hm[2, 0] * X + Hm[2, 1] * Y + 1.0
        uv = _apply(Hm, obj)
        J = np.zeros((2 * len(X), 8))
        J[0::2, 0], J[0::2, 1], J[0::2, 2] = X / w, Y / w, 1 / w
        J[1::2, 3], J[1::2, 4], J[1::2, 5] = X / w, Y / w, 1 / w
        J[0::2, 6], J[0::2, 7] = -uv[:, 0] * X / w, -uv[:, 0] * Y / w
        J[1::2, 6], J[1::2, 7] = -uv[:, 1] * X / w, -uv[:, 1] * Y / w
        return (uv - img).reshape(-1), J
    r, J = res_jac(h)
    for _ in range(100):
        sc = np.linalg.norm(J, axis=0)
        dx = np.linalg.lstsq(J / sc, -r, rcond=None)[0] / sc
        small = np.abs(dx).max() <= 1e-8 * np.abs(h).max()
        step = 1.0
        while True:
            h2 = h + step * dx
            r2, J2 = res_jac(h2)
            if small or r2 @ r2 <= r @ r or step < 1e-6:
                break
            step *= 0.5
        h, r, J = h2, r2, J2
        if np.abs(step * dx).max() <= 1e-15 * np.abs(h).max():
            break
    return np.append(h, 1.0).reshape(3, 3), 0.5 * r @ r


@pytest.fixture(scope="module")
def board_problems():
    s = make_target_scene(6, 6, 24, seed=5)
    start, slot, pix, truth, blocks = _problems(s, (1, 2, 8, 36), np.random.default_rng(9))
    return s, start, slot, pix


def test_homographies_match_polished_opencv(board_problems):
    s, start, slot, pix = board_problems
    tags = np.diff(start)
    for k in (1, 2, 8, 36):
        assert (tags == k).sum() >= 3, k
    H, cost = initialiser.homographies(s.corners, start, slot, pix)
    assert (cost >= 0).all() and np.array_equal(H[:, 2, 2], np.ones(len(H)))
    for p in range(len(tags)):
        sl = slice(start[p], start[p + 1])
        obj, img = s.corners[slot[sl]].reshape(-1, 2), pix[sl].reshape(-1, 2)
        ref, ref_cost = _gn_polish(obj, img, cv2.findHomography(obj, img, 0)[0])
        assert np.linalg.norm(H[p] - ref) <= 1e-9 * np.linalg.norm(ref), (p, tags[p], H[p], ref)
        assert abs(cost[p] - ref_cost) <= 1e-9 * ref_cost + 1e-18, (p, tags[p], cost[p], ref_cost)
        w = H[p][2, 0] * obj[:, 0] + H[p][2, 1] * obj[:, 1] + 1.0
        assert (w > 0).all()


def test_results_are_bitwise_the_same_alone_in_any_batch_and_twice(board_problems):
    import torch
    from torch.profiler import ProfilerActivity, profile
    s, start, slot, pix = board_problems
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        a, ca = initialiser.homographies(s.corners, start, slot, pix)
        torch.cuda.synchronize()
    assert any("homography_target_kernel" in e.name for e in prof.events())
    b, cb = initialiser.homographies(s.corners, start, slot, pix)
    assert np.array_equal(a, b) and np.array_equal(ca, cb)
    order = np.random.default_rng(11).permutation(len(a))
    st, sl, px = [0], [], []
    for p in order:
        sl.append(slot[start[p]:start[p + 1]]); px.append(pix[start[p]:start[p + 1]])
        st.append(st[-1] + start[p + 1] - start[p])
    c, cc = initialiser.homographies(s.corners, st, np.concatenate(sl), np.concatenate(px))
    assert np.array_equal(c, a[order]) and np.array_equal(cc, ca[order])
    for p in range(0, len(a), 5):
        d, cd = initialiser.homographies(s.corners, [0, start[p + 1] - start[p]], slot[start[p]:start[p + 1]],
                                         pix[start[p]:start[p + 1]])
        assert np.array_equal(d[0], a[p]) and cd[0] == ca[p]


def test_a_degenerate_problem_fails_alone(board_problems):
    s, start, slot, pix = board_problems
    H, cost = initialiser.homographies(s.corners, start, slot, pix)
    p = int(np.nonzero(np.diff(start) >= 8)[0][1])
    pix2 = pix.copy()
    pix2[start[p]:start[p + 1]] = 123.0                     # every corner on one pixel: the DLT is singular
    H2, cost2 = initialiser.homographies(s.corners, start, slot, pix2)
    assert cost2[p] == -1.0 and not H2[p].any()
    others = np.arange(len(cost)) != p
    assert np.array_equal(H2[others], H[others]) and np.array_equal(cost2[others], cost[others])


# ------------------------------------------------------------------ the closed form and calibrations from it
def _float32_frames(s, first_ids, seed):
    """_frames with float32-exact pixels and targets with float32-exact corners: OpenCV's calibration functions
    compute with float32 points, so both sides then solve the same problem."""
    frames = [[(t, sz, px.astype(np.float32).astype(np.float64)) for t, sz, px in fr]
              for fr in _frames(s, first_ids, np.random.default_rng(seed))]
    targets = [(ids, c.astype(np.float32).astype(np.float64)) for ids, c in _targets(s, first_ids)]
    return frames, targets


def _board_views(frames, targets, min_tags=4):
    """Per frame with min_tags tags of board 0: its (n,3) float32 board points and (n,2) float32 pixels."""
    ids, corners = targets[0]
    slot_of = {int(i): k for k, i in enumerate(ids)}
    objs, imgs = [], []
    for fr in frames:
        on = [(slot_of[t], px) for t, _, px in fr if t in slot_of]
        if len(on) < min_tags:
            continue
        o = corners[[k for k, _ in on]].reshape(-1, 2)
        objs.append(np.concatenate([o, np.zeros((len(o), 1))], 1).astype(np.float32))
        imgs.append(np.array([px for _, px in on]).reshape(-1, 2).astype(np.float32))
    return objs, imgs


@pytest.mark.parametrize("lens", ["radtan", "equidistant"])
def test_initialise_intrinsics_matches_opencv_init_camera_matrix(lens):
    s = make_target_scene(6, 6, 60, seed=3, lens=lens)
    frames, targets = _float32_frames(s, [0], 1)
    intr, used = initialiser.initialise_intrinsics(frames, targets, s.image_size)
    objs, imgs = _board_views(frames, targets)
    assert used == len(objs) == 60
    K = cv2.initCameraMatrix2D(objs, imgs, s.image_size, 0)
    # OpenCV refines each homography by 10 LM iterations, the kernel to convergence
    assert np.abs(intr[:2] / [K[0, 0], K[1, 1]] - 1).max() <= 1e-7, (intr, K)
    assert intr[2] == K[0, 2] and intr[3] == K[1, 2]


def _solve(scene):
    with BAProblem.from_scene(scene) as p:
        summ = p.solve(max_iterations=500, function_tolerance=1e-16, gradient_tolerance=1e-16,
                       parameter_tolerance=1e-16)
        intr, dist = p.get_intrinsics()
        return summ, intr[0], dist[0], p.get_view_poses()


def _from_estimate_and_truth(s, frames, targets, first_ids, lens):
    """The calibration started from initialise_intrinsics and initialise_targets, and the same problem started from
    the true intrinsics, distortion and poses.  Returns (estimated start, both solves, the scene)."""
    intr0, _ = initialiser.initialise_intrinsics(frames, targets, s.image_size)
    scene, ids, keep, tag_pose, boards = initialiser.initialise_targets(frames, intr0, np.zeros(5), targets,
                                                                        lens=lens)
    truth = copy.deepcopy(scene)
    # the truth's entity of a tag id (_frames: board b's slot k is first_ids[b] + k, free tag j is 1000 + j)
    entity_of = lambda t: first_ids.index(t - t % 100) if t < 1000 else len(first_ids) + t - 1000
    # the world is the frame of the first tag of frame 0
    t0 = frames[0][0][0]
    g_T_w = s.truth["markers"][entity_of(t0)]
    if t0 < 1000:
        g_T_w = compose(g_T_w, initialiser.board_T_tag(targets[entity_of(t0)][1][t0 % 100]))
    w_T_g = invert(g_T_w)
    truth.views = compose(np.broadcast_to(w_T_g, s.truth["views"].shape), s.truth["views"])[keep]
    truth.intr, truth.dist = s.truth["intr"][:1].copy(), s.truth["dist"][:1].copy()
    entity = {px.tobytes(): entity_of(t) for fr in frames for t, _, px in fr}
    for b in range(scene.n_blocks):
        truth.markers[scene.marker_idx[b]] = compose(w_T_g, s.truth["markers"][entity[scene.pixels[b].tobytes()]])
    return intr0, _solve(scene), _solve(truth), scene


def _check_same_minimum(est, tru):
    (summ, intr, _, _), (summ_t, intr_t, _, _) = est, tru
    assert summ["termination"] != 4 and summ_t["termination"] != 4
    assert abs(summ["final_cost"] - summ_t["final_cost"]) <= 1e-9 * summ_t["final_cost"], (summ, summ_t)
    assert np.abs(intr / intr_t - 1).max() <= 1e-6, (intr, intr_t)


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_radtan_calibration_from_the_estimate_reaches_the_minimum(seed):
    s = make_target_scene(6, 6, 60, seed=seed)
    frames, targets = _float32_frames(s, [0], seed)
    intr0, est, tru, scene = _from_estimate_and_truth(s, frames, targets, [0], "radtan")
    assert np.abs(intr0[:2] / s.truth["intr"][0][:2] - 1).max() < 0.03
    _check_same_minimum(est, tru)
    objs, imgs = _board_views(frames, targets, min_tags=1)
    assert len(objs) == len(scene.views)
    crit = (cv2.TERM_CRITERIA_COUNT + cv2.TERM_CRITERIA_EPS, 300, 1e-16)
    rms, K, D, _, _ = cv2.calibrateCamera(objs, imgs, s.image_size, None, None, criteria=crit)
    cv_cost = 0.5 * rms ** 2 * sum(len(o) for o in objs)
    assert est[0]["final_cost"] <= cv_cost * (1 + 1e-9), (est[0]["final_cost"], cv_cost)


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_equidistant_calibration_from_the_estimate_reaches_the_minimum(seed):
    s = make_target_scene(6, 6, 60, seed=seed, lens="equidistant")
    frames, targets = _float32_frames(s, [0], seed)
    intr0, est, tru, scene = _from_estimate_and_truth(s, frames, targets, [0], "equidistant")
    assert np.abs(intr0[:2] / s.truth["intr"][0][:2] - 1).max() < 0.03
    _check_same_minimum(est, tru)
    objs, imgs = _board_views(frames, targets, min_tags=1)
    # cv2.fisheye.calibrate from the same closed-form start (its own start fails its InitExtrinsics on these views)
    K0 = cv2.initCameraMatrix2D(objs, imgs, s.image_size, 0)
    flags = cv2.fisheye.CALIB_RECOMPUTE_EXTRINSIC | cv2.fisheye.CALIB_FIX_SKEW | cv2.fisheye.CALIB_USE_INTRINSIC_GUESS
    crit = (cv2.TERM_CRITERIA_COUNT + cv2.TERM_CRITERIA_EPS, 300, 1e-16)
    o64 = [o.reshape(1, -1, 3).astype(np.float64) for o in objs]
    i64 = [i.reshape(1, -1, 2).astype(np.float64) for i in imgs]
    _, K, D, rv, tv = cv2.fisheye.calibrate(o64, i64, s.image_size, K0, np.zeros(4), flags=flags, criteria=crit)
    cv_cost = 0.5 * sum(((cv2.fisheye.projectPoints(o, r, t, K, D)[0] - i) ** 2).sum()
                        for o, i, r, t in zip(o64, i64, rv, tv))
    assert est[0]["final_cost"] <= cv_cost * (1 + 1e-9), (est[0]["final_cost"], cv_cost)


def test_boards_and_free_tags_from_the_estimate_reach_the_minimum():
    s = make_target_scene(6, 6, 60, n_boards=2, n_free=3, seed=7)
    frames, targets = _float32_frames(s, [0, 100], 7)
    _, est, tru, scene = _from_estimate_and_truth(s, frames, targets, [0, 100], "radtan")
    assert (scene.corner_slot < 0).any() and len(scene.markers) == 5
    _check_same_minimum(est, tru)


# ------------------------------------------------------------------ the command line, end to end
@pytest.mark.parametrize("lens", ["radtan", "equidistant"])
def test_command_line_calibrates_from_detections_alone(tmp_path, lens):
    d = str(tmp_path)
    s = make_target_scene(6, 6, 60, seed=41, lens=lens, pixel_noise=0.0)
    frames = _frames(s, [0], np.random.default_rng(5))
    for n, fr in enumerate(frames):
        c = np.round(np.array([p for _, _, p in fr])).astype(np.int64).reshape(-1, 4, 2)
        with open(os.path.join(d, f"detections_{n}.yaml"), "w") as f:
            f.write(io_yaml.detections_text([t for t, _, _ in fr], [sz for _, sz, _ in fr], c))
    g = os.path.join(d, "grid.yaml")
    _write_grid(g, 6, 6, 0.1, 0.3, 0)
    W, H = s.image_size
    assert main([d, "--initialise", "--target", g, "--image-size", str(W), str(H), "--lens", lens]) == 0
    assert not os.path.exists(os.path.join(d, "camera.yaml"))
    assert os.path.exists(os.path.join(d, "targets.yaml"))
    assert _stanza_views(d, range(len(frames))).shape == (len(frames), 6)
    with open(os.path.join(d, "camera_refined.yaml")) as f:
        y = yaml.safe_load(f)
    assert (y["image_width"], y["image_height"]) == (W, H)
    assert y["distortion_model"] == {"radtan": "plumb_bob", "equidistant": "equidistant"}[lens]
    intr, dist, got_lens = io_yaml.read_camera(os.path.join(d, "camera_refined.yaml"))
    assert got_lens == lens
    # the Python API on the same detections
    numbers, fp = io_yaml.read_detections(d)
    tg = io_yaml.read_targets([g])
    intr0, _ = initialiser.initialise_intrinsics(fp, tg, (W, H))
    scene = initialiser.initialise_targets(fp, intr0, np.zeros(5), tg, lens=lens)[0]
    with BAProblem.from_scene(scene) as p:
        p.solve(max_iterations=50)
        api_intr, api_dist = p.get_intrinsics()
    assert np.abs(intr - api_intr[0]).max() <= 1e-9 * np.abs(api_intr[0]).max()
    n = 4 if lens == "equidistant" else 5
    assert np.abs(dist[:n] - api_dist[0][:n]).max() <= 1e-9 * max(np.abs(api_dist[0]).max(), 1e-3)
    # rounding to whole pixels is ~0.3 px of noise
    assert np.abs(intr / s.truth["intr"][0] - 1).max() < 0.01, (intr, s.truth["intr"][0])
