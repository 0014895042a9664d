"""Intrinsics from board detections without a GPU: the argument checks of rcc_homography_target_batch, the closed form
(initialiser.intrinsics_from_homographies) against cv2.initCameraMatrix2D, the views it refuses, and the
--image-size command line combinations it refuses."""
import os

import numpy as np
import pytest

from robot_camera_calibration_b200 import _lib as L
from robot_camera_calibration_b200 import initialiser, io_yaml
from robot_camera_calibration_b200.__main__ import main
from robot_camera_calibration_b200.scenes import board_layout, make_target_scene, rodrigues_np


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


# ------------------------------------------------------------------ rcc_homography_target_batch argument checks
def _call(n_slots=4, corners=None, n=2, start=None, slot=None, pixels=True, H=True, cost=True, null_start=False,
          null_slot=False):
    lib = L.load()
    corners = board_layout(2, 2, 0.1, 0.3).reshape(-1) if corners is None else np.asarray(corners, float)
    start = np.array([0, 2, 3], np.int64) if start is None else np.asarray(start, np.int64)
    slot = np.array([0, 1, 3], np.int32) if slot is None else np.asarray(slot, np.int32)
    px = np.zeros(8 * 3)
    out = np.zeros(9 * max(n, 1))
    fc = np.zeros(max(n, 1))
    dp = lambda a, keep: a.ctypes.data_as(L.c_double_p) if keep else None
    return lib.rcc_homography_target_batch(0, n_slots, dp(corners, corners is not None), n,
                                           None if null_start else start.ctypes.data_as(L.c_int64_p),
                                           None if null_slot else slot.ctypes.data_as(L.c_int32_p),
                                           dp(px, pixels), dp(out, H), dp(fc, cost), 30)


@pytest.mark.parametrize("case", [
    dict(n=-1), dict(pixels=False), dict(H=False), dict(null_start=True), dict(null_slot=True),
    dict(start=[1, 2, 3]), dict(start=[0, 2, 2]), dict(start=[0, 3, 2]),
    dict(n_slots=0), dict(n_slots=-3),
    dict(slot=[0, 4, 1]), dict(slot=[0, -1, 1]),
    dict(corners=np.where(np.arange(32) == 5, np.nan, board_layout(2, 2, 0.1, 0.3).reshape(-1))),
    dict(corners=np.where(np.arange(32) == 31, np.inf, board_layout(2, 2, 0.1, 0.3).reshape(-1))),
])
def test_bad_arguments_are_rejected_before_any_device_query(case):
    assert _call(**case) == L.RCC_BAD_ARG


def test_null_corners_are_rejected_and_no_problems_is_ok():
    lib = L.load()
    assert lib.rcc_homography_target_batch(0, 4, None, 1, None, None, None, None, None, 0) == L.RCC_BAD_ARG
    assert lib.rcc_homography_target_batch(0, 4, None, 0, None, None, None, None, None, 0) == L.RCC_OK
    # the final cost may be NULL; without a device valid arguments fail with RCC_CUDA_ERROR, not RCC_BAD_ARG
    assert _call(cost=False) == (L.RCC_OK if _has_gpu() else L.RCC_CUDA_ERROR)


# ------------------------------------------------------------------ the closed form against OpenCV
def _float32_views(s, min_tags=4):
    """Per view of board 0 with at least min_tags tags: float32-exact board points (n,3) and pixels (n,2), what
    OpenCV's calibration functions compute with (they convert their points to float32)."""
    c32 = s.corners.astype(np.float32)
    objs, imgs = [], []
    for v in range(len(s.views)):
        b = np.nonzero((s.view_idx == v) & (s.marker_idx == 0))[0]
        if len(b) < min_tags:
            continue
        o = c32[s.corner_slot[b]].reshape(-1, 2)
        objs.append(np.concatenate([o, np.zeros((len(o), 1), np.float32)], 1))
        imgs.append(s.pixels[b].astype(np.float32).reshape(-1, 2))
    return objs, imgs


@pytest.mark.parametrize("lens", ["radtan", "equidistant"])
def test_closed_form_matches_opencv_init_camera_matrix(lens):
    cv2 = pytest.importorskip("cv2")
    s = make_target_scene(6, 6, 60, seed=3, lens=lens)
    objs, imgs = _float32_views(s)
    assert len(objs) >= 40
    H = np.array([cv2.findHomography(o[:, :2], i, 0)[0] for o, i in zip(objs, imgs)])
    intr = initialiser.intrinsics_from_homographies(H, s.image_size)
    K = cv2.initCameraMatrix2D(objs, imgs, s.image_size, 0)
    ref = np.array([K[0, 0], K[1, 1], K[0, 2], K[1, 2]])
    assert np.abs(intr / ref - 1).max() <= 1e-12, (intr, ref)
    assert intr[2] == (s.image_size[0] - 1) / 2 and intr[3] == (s.image_size[1] - 1) / 2
    # and it is a start the bundle adjustment converges from: within 3 % of the truth
    assert np.abs(intr[:2] / s.truth["intr"][0][:2] - 1).max() < 0.03


def _plane_homography(fx, fy, cx, cy, rvec, t):
    R = rodrigues_np(np.asarray(rvec, float).reshape(1, 3))[0]
    H = np.array([[fx, 0, cx], [0, fy, cy], [0, 0, 1.0]]) @ np.stack([R[:, 0], R[:, 1], t], 1)
    return H / H[2, 2]


def test_fronto_parallel_views_do_not_constrain_the_focal_length():
    # rotations about the optical axis only: both of Zhang's rows of every view are proportional to (fx^2, -fy^2)
    # with a zero right-hand side, so the normal matrix is singular
    views = [_plane_homography(600, 620, 319.5, 239.5, [0, 0, a], [x, y, 2.0])
             for a, x, y in ((0.0, -0.2, 0.1), (0.4, 0.1, -0.3), (-1.1, 0.3, 0.2), (2.5, 0.0, 0.0))]
    with pytest.raises(ValueError, match="tilt the board"):
        initialiser.intrinsics_from_homographies(views, (640, 480))
    # tilted views of the same camera give it back exactly
    tilted = [_plane_homography(600, 620, 319.5, 239.5, r, [0.1, -0.1, 2.0])
              for r in ([0.3, 0.1, 0.2], [-0.2, 0.35, -0.1], [0.1, -0.3, 1.0])]
    assert np.abs(initialiser.intrinsics_from_homographies(tilted, (640, 480)) - [600, 620, 319.5, 239.5]).max() < 1e-9


def test_a_negative_solution_is_refused_where_opencv_takes_its_absolute_value():
    # columns h = (1, 0, 1), v = (1, 1, 1) and h = (0, 1, 1), v = (1, 1, 1) with the principal point at 0 (a 1 x 1
    # image): Zhang's rows ask for 1/fx^2 and 1/fy^2 < 0, from a well-conditioned normal matrix
    bad = np.array([[[1, 1, 0], [0, 1, 0], [1, 1, 1]], [[0, 1, 0], [1, 1, 0], [1, 1, 1]]], float)
    with pytest.raises(ValueError, match="tilt the board"):
        initialiser.intrinsics_from_homographies(bad, (1, 1))
    # the same rows restated here: the refusal is the sign, not the conditioning
    rows, rhs = [], []
    for h in bad:
        t0, t1 = h[:, 0], h[:, 1]
        d1, d2 = (t0 + t1) / 2, (t0 - t1) / 2
        t0, t1, d1, d2 = (x / np.linalg.norm(x) for x in (t0, t1, d1, d2))
        rows += [[t0[0] * t1[0], t0[1] * t1[1]], [d1[0] * d2[0], d1[1] * d2[1]]]
        rhs += [-t0[2] * t1[2], -d1[2] * d2[2]]
    A, b = np.array(rows), np.array(rhs)
    assert np.linalg.cond(A.T @ A) < 1e3
    assert (np.linalg.solve(A.T @ A, A.T @ b) < 0).any()


def _frames_of(s, first_ids, free_only=False):
    frames = []
    for v in range(len(s.views)):
        fr = []
        for b in np.nonzero(s.view_idx == v)[0]:
            m = int(s.marker_idx[b])
            if m < len(first_ids):
                if free_only:
                    continue
                tid = first_ids[m] + int(s.corner_slot[b])
            else:
                tid = 1000 + m
            fr.append((tid, float(s.sizes[m]), s.pixels[b].copy()))
        frames.append(fr)
    return frames


def test_free_tags_and_small_board_views_are_refused():
    s = make_target_scene(3, 3, 6, n_free=4, seed=2)
    targets = [(np.arange(9), s.corners)]
    with pytest.raises(ValueError, match="free tags"):
        initialiser.initialise_intrinsics(_frames_of(s, [0], free_only=True), targets, s.image_size)
    with pytest.raises(ValueError, match="10 or more"):
        initialiser.initialise_intrinsics(_frames_of(s, [0]), targets, s.image_size, min_tags=10)


# ------------------------------------------------------------------ the command line
def _grid(d):
    path = os.path.join(d, "grid.yaml")
    with open(path, "w") as f:
        f.write("target_type: aprilgrid\ntagRows: 2\ntagCols: 2\ntagSize: 0.1\ntagSpacing: 0.3\n")
    return path


@pytest.mark.parametrize("extra", [
    ["--image-size", "640", "480"],                                    # without --initialise and --target
    ["--image-size", "640", "480", "--initialise"],                    # without --target
    ["--image-size", "640", "480", "--target", "GRID"],                # without --initialise
    ["--image-size", "640", "480", "--initialise", "--target", "GRID", "--fix-intrinsics"],
    ["--image-size", "640", "480", "--initialise", "--target", "GRID", "--intrinsics-sigma", "1", "1", "1"],
    ["--image-size", "0", "480", "--initialise", "--target", "GRID"],
    ["--lens", "equidistant", "--initialise", "--target", "GRID"],     # --lens alone
    ["--lens", "pinhole", "--image-size", "640", "480", "--initialise", "--target", "GRID"],
])
def test_rejected_combinations_exit_with_status_2(tmp_path, extra):
    d = str(tmp_path)
    g = _grid(d)
    with pytest.raises(SystemExit) as e:
        main([d] + [g if a == "GRID" else a for a in extra])
    assert e.value.code == 2


def test_a_dataset_without_a_qualifying_board_view_exits_with_status_2(tmp_path, capsys):
    d = str(tmp_path)
    g = _grid(d)
    # frame 0: three tags of the 2 x 2 board and a free tag -- fewer than 4 tags of a board in every frame
    with open(os.path.join(d, "detections_0.yaml"), "w") as f:
        f.write(io_yaml.detections_text([0, 1, 2, 50], [0.1] * 4, 10 * np.arange(32).reshape(4, 4, 2)))
    assert main([d, "--initialise", "--target", g, "--image-size", "640", "480"]) == 2
    err = capsys.readouterr().err
    assert "4 or more" in err
    assert not os.path.exists(os.path.join(d, "camera.yaml"))
    assert not os.path.exists(os.path.join(d, "camera_refined.yaml"))
    # without --image-size a missing camera.yaml is still the error it was
    assert main([d, "--initialise", "--target", g]) == 2
    assert "camera.yaml" in capsys.readouterr().err


def test_image_size_and_lens_are_passed_to_optimise_directory(monkeypatch, tmp_path):
    seen = {}

    def fake(directory, **kw):
        seen.update(kw)
        return {"termination": 1}
    monkeypatch.setattr(io_yaml, "optimise_directory", fake)
    g = _grid(str(tmp_path))
    assert main(["d", "--initialise", "--target", g, "--image-size", "1280", "1024", "--lens", "equidistant"]) == 0
    assert seen["image_size"] == [1280, 1024] and seen["lens"] == "equidistant" and seen["refine_intrinsics"]
    assert main(["d", "--initialise", "--target", g]) == 0
    assert seen["image_size"] is None and seen["lens"] is None


def test_optimise_directory_refuses_image_size_with_given_intrinsics(tmp_path):
    with pytest.raises(ValueError, match="image_size"):
        io_yaml.optimise_directory(str(tmp_path), initialise=True, targets=["g.yaml"], image_size=(640, 480),
                                   intr=[500, 500, 320, 240], dist=np.zeros(5))
    with pytest.raises(ValueError, match="image_size"):
        io_yaml.optimise_directory(str(tmp_path), initialise=False, targets=["g.yaml"], image_size=(640, 480))
