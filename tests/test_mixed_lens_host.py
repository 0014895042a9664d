"""CPU: cameras of different lenses in one problem -- the argument checks of rcc_ba_set_camera_lenses that need no
device, the mixed-lens oracle of tests/mixed_lens_oracle.py against the single-lens oracles camera by camera, the
mixed scenes of make_scene, and the ceres_like checks that run before any device is touched."""
import numpy as np
import pytest

import ba_oracle as O
import lens_oracle as LO
import mixed_lens_oracle as MO
from robot_camera_calibration_b200 import _lib as L
from robot_camera_calibration_b200 import ceres_like
from robot_camera_calibration_b200.scenes import _corners_in_camera, make_scene

MIXED = {
    "rig4": dict(n_markers=16, n_views=10, visibility=0.6, n_cam=4, model="rig", seed=13,
                 lens=("radtan", "equidistant", "radtan", "equidistant")),
    "rig3": dict(n_markers=16, n_views=10, visibility=0.6, n_cam=3, model="rig", seed=17,
                 lens=("radtan", "radtan", "equidistant")),
    "single2": dict(n_markers=12, n_views=20, visibility=0.7, n_cam=2, seed=11, lens=("radtan", "equidistant")),
}


def _scene(name, **kw):
    args = dict(MIXED[name])
    args.update(kw)
    return make_scene(args.pop("n_markers"), args.pop("n_views"), args.pop("visibility"), **args)


def test_set_camera_lenses_rejects_a_null_handle():
    lib = L.load()
    lenses = np.zeros(4, np.int32)
    assert lib.rcc_ba_set_camera_lenses(None, lenses.ctypes.data_as(L.c_int32_p)) == L.RCC_BAD_ARG
    assert lib.rcc_ba_set_camera_lenses(None, None) == L.RCC_BAD_ARG


@pytest.mark.parametrize("name", list(MIXED))
def test_mixed_oracle_is_the_single_lens_oracles_camera_by_camera(name):
    s = _scene(name)
    p = MO.oracle_problem(s)
    r, Jb = MO.residuals(p), MO.jacobian_blocks_cs(p)
    for lens in ("radtan", "equidistant"):
        # the whole problem through one lens: its rows of the cameras with that lens are the mixed oracle's
        whole = LO.oracle_problem(s)
        whole.lens = lens
        rows = np.asarray(p.lens)[s.cam_idx] == lens
        assert rows.any()
        assert np.array_equal(LO.residuals(whole)[rows], r[rows])
        Jw = LO.jacobian_blocks_cs(whole)
        for k in Jb:
            assert np.array_equal(Jw[k][rows], Jb[k][rows]), (lens, k)
    # and an independent check of each half: ba_oracle (radial-tangential) and OpenCV's cv2.fisheye (equidistant)
    rt = np.asarray(p.lens)[s.cam_idx] == "radtan"
    Jo = O.jacobian_blocks_cs(p)
    assert np.abs(O.residuals(p)[rt] - r[rt]).max() < 1e-9
    for k in Jb:
        assert np.abs(Jo[k][rt] - Jb[k][rt]).max() <= 1e-9 * np.abs(Jb[k][rt]).max(), k
    for b in np.nonzero(~rt)[0][::5]:
        c, v, m = s.cam_idx[b], s.view_idx[b], s.marker_idx[b]
        pts, J = LO.jacobian_block_cv2(s.model, s.intr[c], s.dist[c], s.ext[c], s.views[v], s.markers[m], s.sizes[m])
        assert np.abs(r[b] + s.pixels[b] - pts).max() < 1e-9
        for k in J:
            assert np.linalg.norm(Jb[k][b] - J[k]) <= 1e-8 * np.linalg.norm(J[k]), (b, k)
    # the distortion column 4: zero on the equidistant blocks only (k3 of a radial-tangential camera is live)
    assert np.all(Jb["dist"][~rt][..., 4] == 0.0) and np.any(Jb["dist"][rt][..., 4] != 0.0)
    # the reserved slot is held constant for the equidistant cameras only
    cm = p.const_mask()
    slot = p.offsets()[2] + p.shared_per_cam * np.arange(p.n_cam) + 8
    assert np.array_equal(cm[slot], [lens == "equidistant" for lens in p.lens])
    assert abs(MO.cost(p) - 0.5 * float((r * r).sum())) <= 1e-12 * MO.cost(p)


def test_mixed_oracle_normal_equations_add_up_per_lens():
    """H = J^T J over all blocks is the sum of the per-lens halves."""
    s = _scene("rig3", n_views=6)
    p = MO.oracle_problem(s)
    H, g, c = MO.normal_equations(p)
    Hs, gs, cs = 0.0, 0.0, 0.0
    for lens in ("radtan", "equidistant"):
        q, _ = p.of_lens(lens)
        Hq, gq, cq = LO.normal_equations(q)
        Hs, gs, cs = Hs + Hq, gs + gq, cs + cq
    assert np.abs(H - Hs).max() <= 1e-12 * np.abs(H).max()
    assert np.abs(g - gs).max() <= 1e-12 * np.abs(g).max() and abs(c - cs) <= 1e-12 * c


@pytest.mark.parametrize("name", list(MIXED))
def test_mixed_scenes_are_deterministic_and_every_camera_sees_tags(name):
    s, t = _scene(name), _scene(name)
    for k in ("intr", "dist", "ext", "views", "markers", "view_idx", "marker_idx", "cam_idx", "pixels"):
        assert np.array_equal(getattr(s, k), getattr(t, k)), k
    lenses = MIXED[name]["lens"]
    assert s.lens == lenses and len(s.image_size) == len(lenses)
    assert np.all(np.bincount(s.cam_idx, minlength=len(lenses)) > 0)
    for c, lens in enumerate(lenses):
        m = s.cam_idx == c
        W, H = s.image_size[c]
        assert (W, H) == ((1280, 1024) if lens == "equidistant" else (640, 480))
        f = s.truth["intr"][c, 0]
        assert (320 <= f <= 340) if lens == "equidistant" else (550 <= f <= 650)
        uv = s.pixels[m].reshape(-1, 4, 2)
        assert uv[..., 0].max() < W + 5 and uv[..., 1].max() < H + 5
        q = _corners_in_camera(s.model, s.truth["ext"][c], s.truth["views"][s.view_idx[m]],
                               s.truth["markers"][s.marker_idx[m]], s.sizes[s.marker_idx[m]])
        off_axis = np.degrees(np.arctan2(np.hypot(q[..., 0], q[..., 1]), q[..., 2]))
        if lens == "equidistant":
            assert off_axis.max() > 60 and off_axis.max() < 85 and s.dist[c, 4] == 0.0
        else:
            assert off_axis.max() < 45


def test_one_lens_given_per_camera_is_the_named_scene():
    a = make_scene(12, 10, 0.7, n_cam=2, seed=4, lens=("equidistant", "equidistant"))
    b = make_scene(12, 10, 0.7, n_cam=2, seed=4, lens="equidistant")
    assert a.lens == "equidistant"
    for k in ("intr", "dist", "views", "pixels", "view_idx", "cam_idx"):
        assert np.array_equal(getattr(a, k), getattr(b, k)), k
    with pytest.raises(ValueError):
        make_scene(12, 10, 0.7, n_cam=2, lens=("radtan",))
    with pytest.raises(ValueError):
        make_scene(12, 10, 0.7, n_cam=2, lens=("radtan", "fisheye"))


def test_ceres_like_refuses_one_camera_under_two_lenses():
    intr, dist = np.array([600.0, 600, 320, 240]), np.zeros(5)
    view, marker = np.zeros(6), np.array([0, 0, 0, 0, 0, 2.0])
    prob = ceres_like.Problem()
    prob.AddResidualBlock(ceres_like.TagReprojectionCost(np.zeros(8), 0.1), None, intr, dist, view, marker)
    prob.AddResidualBlock(ceres_like.TagReprojectionCost(np.zeros(8), 0.1, lens="equidistant"), None, intr, dist,
                          view, marker)
    with pytest.raises(ValueError, match="different lenses"):
        prob._build()
