"""CPU checks of the equidistant (fisheye) lens: the model.cuh arithmetic the kernels run (compiled with g++ through
tests/host_harness/lens_harness.cpp) against the complex-step oracle, oracle A against OpenCV's cv2.fisheye, the
camera YAML reader and writer, the argument checks of the new C entry points, and the unchanged default scenes."""
import ctypes
import hashlib
import os
import subprocess

import numpy as np
import pytest

import lens_oracle as LO
from robot_camera_calibration_b200 import _lib, io_yaml
from robot_camera_calibration_b200.scenes import _corners_in_camera, make_scene, rodrigues_np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DP = ctypes.POINTER(ctypes.c_double)


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    so = tmp_path_factory.mktemp("harness") / "lens_harness.so"
    subprocess.run(["/usr/bin/g++", "-O2", "-shared", "-fPIC", "-x", "c++", "-o", str(so),
                    os.path.join(ROOT, "tests", "host_harness", "lens_harness.cpp")], check=True)
    return ctypes.CDLL(str(so))


def _add_view_with_corner_at(s, b, k, pc):
    """Append a view (a copy of block b's view, moved) from which corner k of block b's tag lies at pc in the camera
    frame, and a block that observes the tag from it."""
    v, m, c = s.view_idx[b], s.marker_idx[b], s.cam_idx[b]
    o = np.array([[-1, -1], [1, -1], [1, 1], [-1, 1]])[k] * s.sizes[m] / 2
    Pw = rodrigues_np(s.markers[m, 0:3]) @ np.array([o[0], o[1], 0.0]) + s.markers[m, 3:6]
    Rv = rodrigues_np(s.views[v, 0:3])
    if s.model == "rig":
        want = s.ext[c, 3:6] + rodrigues_np(s.ext[c, 0:3]) @ pc      # the corner in the body frame
    else:
        want = pc
    view = np.concatenate([s.views[v, 0:3], Pw - Rv @ want])
    s.views = np.vstack([s.views, view])
    s.const_views = np.append(s.const_views, False)
    s.view_idx = np.append(s.view_idx, len(s.views) - 1).astype(np.int32)
    for a in ("marker_idx", "cam_idx"):
        setattr(s, a, np.append(getattr(s, a), getattr(s, a)[b]).astype(np.int32))
    s.pixels = np.vstack([s.pixels, s.pixels[b]])


def _add_block_on_the_axis(s, d=0.8):
    """Append a tag of zero rotation and a view at the origin (identity pose) seen through camera 0 (whose rig
    extrinsics are the identity: the gauge), with the tag's corner 0 at exactly (0, 0, d) in the camera frame."""
    h = s.sizes[0] / 2
    s.markers = np.vstack([s.markers, [0.0, 0.0, 0.0, h, h, d]])
    s.sizes = np.append(s.sizes, s.sizes[0])
    s.const_markers = np.append(s.const_markers, False)
    s.views = np.vstack([s.views, np.zeros(6)])
    s.const_views = np.append(s.const_views, False)
    s.view_idx = np.append(s.view_idx, len(s.views) - 1).astype(np.int32)
    s.marker_idx = np.append(s.marker_idx, len(s.markers) - 1).astype(np.int32)
    s.cam_idx = np.append(s.cam_idx, 0).astype(np.int32)
    s.pixels = np.vstack([s.pixels, s.pixels[0]])
    pc = _corners_in_camera(s.model, s.ext[0], s.views[-1:], s.markers[-1:], s.sizes[-1:])
    assert s.model == "single" or not s.ext[0].any()
    assert pc[0, 0, 0] == 0.0 and pc[0, 0, 1] == 0.0 and pc[0, 0, 2] == d


def _hard_scene(model, ncam):
    s = make_scene(20, 14, 0.5, n_cam=ncam, model=model, seed=5, lens="equidistant")
    s.views[3, 0:3] = [1e-9, -2e-9, 3e-10]          # series branches of the Rodrigues coefficients
    s.markers[5, 0:3] = [1e-4, 2e-4, -1e-4]
    s.views[7, 0:3] *= 0.01
    b0 = int(np.nonzero(s.cam_idx == ncam - 1)[0][0])
    d = 0.8
    _add_block_on_the_axis(s)                                           # exactly on the optical axis: rho = 0
    for k, pc in [(0, [0.0, 0.0, d]),                                   # on the axis up to rounding (rho ~ 1e-17)
                  (2, [1e-8, -3e-9, d]),                                # within 1e-8 of it
                  (1, [2e-5, 1e-5, d]),                                 # inside the series branch of th / rho
                  (3, [3 * np.sin(np.deg2rad(85)), 0.0, 3 * np.cos(np.deg2rad(85))]),   # 85 degrees off axis
                  (1, [0.0, -3 * np.sin(np.deg2rad(84)), 3 * np.cos(np.deg2rad(84))])]:
        _add_view_with_corner_at(s, b0, k, np.array(pc, float))
    return s


@pytest.mark.parametrize("model,ncam", [("single", 1), ("rig", 3)])
def test_equidistant_jacobian_matches_complex_step(harness, model, ncam):
    s = _hard_scene(model, ncam)
    p = LO.oracle_problem(s)
    z = LO.depths(p)
    assert (z > 0).all()
    r, Jb = LO.residuals(p), LO.jacobian_blocks_cs(p)
    P = lambda a: np.ascontiguousarray(a, np.float64).ctypes.data_as(DP)
    worst = 0.0
    rel = lambda a, ref: np.linalg.norm(a - ref) / max(np.linalg.norm(ref), 1e-300)
    for b in range(s.n_blocks):
        c = s.cam_idx[b]
        sh = np.concatenate([s.intr[c], s.dist[c]])
        r8, jv, jm, js, jx, d4 = np.zeros(8), np.zeros(48), np.zeros(48), np.zeros(72), np.zeros(48), np.zeros(4)
        harness.model_eval_block_lens(1, int(model == "rig"), P(s.views[s.view_idx[b]]), P(s.markers[s.marker_idx[b]]),
                                      P(s.ext[c]), P(sh), ctypes.c_double(s.sizes[s.marker_idx[b]]), P(s.pixels[b]),
                                      r8.ctypes.data_as(DP), jv.ctypes.data_as(DP), jm.ctypes.data_as(DP),
                                      js.ctypes.data_as(DP), jx.ctypes.data_as(DP), d4.ctypes.data_as(DP))
        assert np.all(np.isfinite(r8)) and np.all(np.isfinite(js)), b
        assert np.abs(r8 - r[b]).max() <= 1e-9 * max(1.0, np.abs(r[b]).max())
        assert np.all(js.reshape(8, 9)[:, 8] == 0.0)                       # the reserved slot
        errs = [rel(jv.reshape(8, 6), Jb["view"][b]), rel(jm.reshape(8, 6), Jb["marker"][b]),
                rel(js.reshape(8, 9)[:, :4], Jb["intr"][b]), rel(js.reshape(8, 9)[:, 4:], Jb["dist"][b])]
        if model == "rig":
            errs.append(rel(jx.reshape(8, 6), Jb["ext"][b]))
        worst = max(worst, max(errs))
    assert worst < 1e-12


def test_radtan_instantiation_of_the_lens_harness_is_the_existing_model(harness):
    """LENS_RADTAN through the lens template parameter is the radial-tangential model of ba_oracle."""
    import ba_oracle as O
    from helpers import to_oracle
    s = make_scene(10, 8, 0.6, n_cam=2, model="rig", seed=9)
    p = to_oracle(s)
    r, Jb = O.residuals(p), O.jacobian_blocks_cs(p)
    P = lambda a: np.ascontiguousarray(a, np.float64).ctypes.data_as(DP)
    for b in range(s.n_blocks):
        c = s.cam_idx[b]
        r8, jv, jm, js, jx, d4 = np.zeros(8), np.zeros(48), np.zeros(48), np.zeros(72), np.zeros(48), np.zeros(4)
        harness.model_eval_block_lens(0, 1, P(s.views[s.view_idx[b]]), P(s.markers[s.marker_idx[b]]), P(s.ext[c]),
                                      P(np.concatenate([s.intr[c], s.dist[c]])),
                                      ctypes.c_double(s.sizes[s.marker_idx[b]]), P(s.pixels[b]),
                                      r8.ctypes.data_as(DP), jv.ctypes.data_as(DP), jm.ctypes.data_as(DP),
                                      js.ctypes.data_as(DP), jx.ctypes.data_as(DP), d4.ctypes.data_as(DP))
        assert np.abs(r8 - r[b]).max() <= 1e-9
        assert np.linalg.norm(js.reshape(8, 9)[:, 4:] - Jb["dist"][b]) <= 1e-12 * np.linalg.norm(Jb["dist"][b])


@pytest.mark.parametrize("model,ncam", [("single", 1), ("rig", 3)])
def test_oracle_a_matches_cv2_fisheye(model, ncam):
    s = make_scene(12, 16, 0.7, n_cam=ncam, model=model, seed=21, lens="equidistant")
    p = LO.oracle_problem(s)
    uv, _ = LO.project_blocks(p.model, p.lens, *LO.O._gather(p))
    Jb = LO.jacobian_blocks_cs(p)
    worst_v, worst_j = 0.0, 0.0
    for b in range(s.n_blocks):
        c, v, m = s.cam_idx[b], s.view_idx[b], s.marker_idx[b]
        pts, J = LO.jacobian_block_cv2(s.model, s.intr[c], s.dist[c], s.ext[c], s.views[v], s.markers[m], s.sizes[m])
        worst_v = max(worst_v, np.abs(pts - uv[b].reshape(8)).max())
        for k in J:
            worst_j = max(worst_j, np.linalg.norm(J[k] - Jb[k][b]) / np.linalg.norm(Jb[k][b]))
    assert worst_v < 1e-9          # pixels (measured: 3.4e-13)
    assert worst_j < 1e-12         # per-block relative (measured: 5.8e-15)


def test_camera_yaml_round_trip(tmp_path):
    intr, dist = np.array([331.5, 329.25, 641.0, 513.5]), np.array([-0.012, 0.0031, -7e-4, 1.5e-4, 0.0])
    path = tmp_path / "camera.yaml"
    path.write_text(io_yaml.camera_yaml_text(intr, dist, (1280, 1024), lens="equidistant"))
    assert "distortion_model: equidistant" in path.read_text()
    i2, d2, lens = io_yaml.read_camera(str(path))
    assert lens == "equidistant" and np.array_equal(i2, intr) and np.array_equal(d2, dist)
    with pytest.raises(ValueError, match="read_camera"):
        io_yaml.read_camera_yaml(str(path))
    # the fisheye alias, and the radial-tangential file read both ways
    path.write_text(path.read_text().replace("distortion_model: equidistant", "distortion_model: fisheye"))
    assert io_yaml.read_camera(str(path))[2] == "equidistant"
    rt = np.array([0.1, -0.05, 1e-3, -2e-3, 0.01])
    path.write_text(io_yaml.camera_yaml_text(intr, rt))
    i3, d3, lens = io_yaml.read_camera(str(path))
    assert lens == "radtan" and np.array_equal(d3, rt)
    assert all(np.array_equal(a, b) for a, b in zip(io_yaml.read_camera_yaml(str(path)), (i3, d3)))
    # an equidistant file must carry exactly 4 coefficients
    path.write_text(io_yaml.camera_yaml_text(intr, rt).replace("plumb_bob", "equidistant"))
    with pytest.raises(ValueError, match="4 distortion coefficients"):
        io_yaml.read_camera(str(path))


def test_read_dataset_takes_the_lens_from_camera_yaml(tmp_path):
    s = make_scene(6, 8, 0.8, seed=3, lens="equidistant")
    io_yaml.write_dataset(str(tmp_path), s)
    r, _, _ = io_yaml.read_dataset(str(tmp_path))
    assert r.lens == "equidistant"
    assert np.array_equal(r.dist[0, :4], s.dist[0, :4]) and r.dist[0, 4] == 0.0
    # explicit intrinsics keep camera.yaml's lens unless a lens is given with them
    assert io_yaml.read_dataset(str(tmp_path), intr=s.intr[0], dist=s.dist[0, :4])[0].lens == "equidistant"
    assert io_yaml.read_dataset(str(tmp_path), intr=s.intr[0], dist=s.dist[0], lens="radtan")[0].lens == "radtan"
    with pytest.raises(ValueError, match="equidistant lens"):
        io_yaml.read_dataset(str(tmp_path), lens="radtan")
    with pytest.raises(ValueError, match="unknown lens"):
        io_yaml.read_dataset(str(tmp_path), lens="fisheye")
    os.remove(tmp_path / "camera.yaml")
    assert io_yaml.read_dataset(str(tmp_path), intr=s.intr[0], dist=s.dist[0])[0].lens == "radtan"


def test_new_entry_points_check_their_arguments_without_a_device():
    lib = _lib.load()
    assert lib.rcc_ba_set_lens(None, _lib.LENS_EQUIDISTANT) == _lib.RCC_BAD_ARG
    sh = np.zeros(9)
    dp = sh.ctypes.data_as(_lib.c_double_p)
    assert lib.rcc_pnp_batch_lens(0, 2, 0, dp, None, None, None, None, 10) == _lib.RCC_BAD_ARG
    assert lib.rcc_pnp_batch_lens(0, -1, 0, dp, None, None, None, None, 10) == _lib.RCC_BAD_ARG
    assert lib.rcc_pnp_batch_lens(0, _lib.LENS_EQUIDISTANT, 0, dp, None, None, None, None, 10) == _lib.RCC_OK
    assert lib.rcc_pnp_batch_lens(0, _lib.LENS_EQUIDISTANT, -1, dp, None, None, None, None, 10) == _lib.RCC_BAD_ARG


# sha256 of every array of these scenes, computed with the scene generator before the lens existed: the default
# (radial-tangential) path must draw the same random numbers in the same order
_SCENES = [
    (dict(n_markers=12, n_views=30, visibility=0.7, seed=11),
     "5d8a8c1d66b6a521f5ab00d4afbf2750b4eb270738881e7ac003dcef96fc1fcf"),
    (dict(n_markers=16, n_views=20, visibility=0.6, n_cam=3, model="rig", seed=13),
     "7b20e52620fa52f30e3b604361cfef28515526020d0a5838bc5e0e537dd3dc9a"),
    (dict(n_markers=40, n_views=600, visibility=0.3, seed=7, blocked=True, chunk_views=256, threads=1),
     "15ed7d72951a1b77357dfaaf1bc8a932a5fec3875383c7b21eee7883a7e82b7a"),
    (dict(n_markers=12, n_views=30, visibility=0.7, seed=11, round_pixels=True, view_seed=3),
     "b6e1234c346d342b967cb0d9a546db2763215b2f202036c106e33c048d6e3bed"),
]


@pytest.mark.parametrize("kw,digest", _SCENES)
def test_default_scenes_are_bitwise_unchanged(kw, digest):
    s = make_scene(**kw)
    h = hashlib.sha256()
    for k in ("intr", "dist", "ext", "views", "markers", "sizes", "view_idx", "marker_idx", "cam_idx", "pixels",
              "const_views", "const_markers", "const_intr", "const_dist", "const_ext"):
        a = np.ascontiguousarray(getattr(s, k))
        h.update(k.encode())
        h.update(str(a.dtype).encode())
        h.update(a.tobytes())
    for k in sorted(s.truth):
        h.update(np.ascontiguousarray(s.truth[k]).tobytes())
    assert h.hexdigest() == digest
    assert s.lens == "radtan" and s.image_size == (640, 480)
