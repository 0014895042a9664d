"""GPU: rigid multi-tag targets (rcc_ba_set_corner_layout) and the target instantiations of K1, K2 and K6
(materialise_target_kernel, assemble_target_kernel, evaluate_target_kernel).

- Same corners, same results: a layout whose slot for each block holds the square of its own marker's size (the same
  doubles) gives results bitwise equal to the plain handle, in every cell of model x elimination x lens set x loss of
  test_gpu_kernel_matrix.py, whose plain kernels are checked there against the oracle.  The markers get distinct
  sizes, so a block that read another block's slot would differ.  The profiler proves that the layout handle ran
  exactly the target instantiations of its cell and no plain K1, K2 or K6 kernel.
- Real boards: residuals against the numpy projection of the layout corners, the normal blocks, S and b against dense
  products of K1's Jacobians on a 9 x 9 board seen whole in one image (pairs of 81 observation blocks), convergence
  to the truth, clearing, piecewise pixel uploads and the argument checks."""
import contextlib
import re

import numpy as np
import pytest
from torch.profiler import ProfilerActivity, profile

from helpers import max_block_rel, rel_fro
from robot_camera_calibration_b200 import _lib as L
from robot_camera_calibration_b200.problem import BAProblem
from robot_camera_calibration_b200.scenes import make_target_scene, project_points
from test_gpu_kernel_matrix import _scene, _template_arg
from test_targets_host import TARGET_CELLS, expected_target_kernels, square_layout

RADIUS = 1e4
_K = re.compile(r"\brcc::(assemble_kernel|materialise_kernel|evaluate_kernel|assemble_target_kernel|"
                r"materialise_target_kernel|evaluate_target_kernel)<([^<>]*)>")


@contextlib.contextmanager
def kernels_launched():
    """`with kernels_launched() as got:` -- on exit `got` holds (kernel, template arguments) of every plain or target
    K1, K2 and K6 kernel launched inside the block (torch.profiler, the library's own streams included)."""
    got = set()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        yield got
    for e in prof.events():
        m = _K.search(e.name)
        if m:
            got.add((m.group(1), tuple(_template_arg(a.strip()) for a in m.group(2).split(","))))


def _run(s, elim, loss, scale, layout=None):
    """Every product the cells compare, from one handle."""
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        if layout is not None:
            gp.set_corner_layout(*layout)
        if loss != "trivial":
            gp.set_loss(loss, scale)
        out = {"k1": gp.evaluate(), "k6": gp.evaluate(want_jacobians=False)}
        out["cost"] = gp.linearize()
        out["nb"] = gp.normal_blocks()
        gp.schur(RADIUS)
        out["S"], out["b"] = gp.reduced_system()
        out["mcc"] = gp.solve_step()
        out["step"] = gp.step()
        out["cand"] = gp.candidate_cost()
    return out


def _flat(out):
    """name -> array of every result, for bitwise comparisons."""
    f = {"k1 residuals": out["k1"]["residuals"], "k1 cost": out["k1"]["cost"], "k6 residuals": out["k6"]["residuals"],
         "k6 cost": out["k6"]["cost"], "cost": out["cost"], "S": out["S"], "b": out["b"], "mcc": out["mcc"],
         "cand": out["cand"]}
    f.update({"J " + k: v for k, v in out["k1"]["jacobians"].items()})
    f.update({"nb " + k: v for k, v in out["nb"].items()})
    f.update({"step " + k: v for k, v in out["step"].items()})
    return f


@pytest.mark.gpu
@pytest.mark.parametrize("model,elim,lens_set,loss", TARGET_CELLS)
def test_same_corners_same_results(model, elim, lens_set, loss):
    s, scale = _scene(model, lens_set)
    s = s.__class__(**{**s.__dict__})
    s.sizes = np.random.default_rng(3).uniform(0.08, 0.12, len(s.markers))
    plain = _flat(_run(s, elim, loss, scale))
    with kernels_launched() as launched:
        target = _flat(_run(s, elim, loss, scale, square_layout(s)))
    assert launched == expected_target_kernels(model, elim, lens_set, loss)
    for k, v in plain.items():
        assert np.array_equal(np.asarray(target[k]), np.asarray(v)), k


def _board(model="single", **kw):
    if model == "rig":
        return make_target_scene(4, 5, 24, n_boards=2, n_free=6, n_cam=3, model="rig", seed=7,
                                 lens=("equidistant", "radtan", "equidistant"), **kw)
    return make_target_scene(9, 9, 24, n_free=4, seed=3, distance=3.0, **kw)


def _numpy_residuals(s, which="views"):
    """pixels - projection of the layout corners (slot -1: the marker's square) at the scene's parameters."""
    obj = np.zeros((s.n_blocks, 4, 3))
    on = s.corner_slot >= 0
    obj[on, :, :2] = s.corners[s.corner_slot[on]]
    h = s.sizes[s.marker_idx[~on]] / 2
    obj[~on, :, :2] = np.stack([np.stack([-h, -h], -1), np.stack([h, -h], -1), np.stack([h, h], -1),
                                np.stack([-h, h], -1)], 1)
    lens = s.lens if not isinstance(s.lens, str) else (s.lens,) * len(s.intr)
    r = np.empty((s.n_blocks, 8))
    for c in range(len(s.intr)):
        m = s.cam_idx == c
        uv, _ = project_points(s.model, np.broadcast_to(s.intr[c], (m.sum(), 4)), np.broadcast_to(s.dist[c], (m.sum(), 5)),
                               np.broadcast_to(s.ext[c], (m.sum(), 6)), s.views[s.view_idx[m]],
                               s.markers[s.marker_idx[m]], obj[m], lens[c])
        r[m] = uv.reshape(-1, 8) - s.pixels[m]
    return r


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["single", "rig"])
def test_board_residuals_match_numpy(model):
    s = _board(model)
    r = _numpy_residuals(s)
    with BAProblem.from_scene(s) as gp:
        k1, k6 = gp.evaluate(), gp.evaluate(want_jacobians=False)
    assert max_block_rel(k1["residuals"], r, floor=1e-6) < 1e-9
    assert max_block_rel(k6["residuals"], r, floor=1e-6) < 1e-9
    assert abs(k1["cost"] - 0.5 * (r ** 2).sum()) <= 1e-9 * k1["cost"]
    assert k1["cost"] == pytest.approx(k6["cost"], rel=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("elim", ["views", "markers"])
def test_board_normal_equations_match_dense_products(elim):
    """A 9 x 9 board seen whole: every (view, board) pair has 81 observation blocks, more than one E-pass chunk of
    64.  H, g, W, S and b against dense products of K1's Jacobian blocks (trivial loss)."""
    s = _board("single")
    ev = elim == "views"
    pair = s.view_idx.astype(np.int64) * len(s.markers) + s.marker_idx
    assert np.bincount(pair).max() > 64
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        k1 = gp.evaluate()
        gp.linearize()
        nb = gp.normal_blocks()
        gp.schur(RADIUS)
        S, b = gp.reduced_system()
    nv, nm, n = len(s.views), len(s.markers), s.n_blocks
    J = np.zeros((8 * n, 6 * nv + 6 * nm + 9))
    rows = np.arange(8 * n).reshape(n, 8)
    for i in range(n):
        v, m = s.view_idx[i], s.marker_idx[i]
        J[rows[i], 6 * v:6 * v + 6] = k1["jacobians"]["view"][i]
        J[rows[i], 6 * nv + 6 * m:6 * nv + 6 * m + 6] = k1["jacobians"]["marker"][i]
        J[rows[i], 6 * (nv + nm):6 * (nv + nm) + 4] = k1["jacobians"]["intr"][i]
        J[rows[i], 6 * (nv + nm) + 4:] = k1["jacobians"]["dist"][i]
    H, g = J.T @ J, J.T @ k1["residuals"].ravel()
    e_off, n_e, f_off, n_f = (0, nv, 6 * nv, nm) if ev else (6 * nv, nm, 0, nv)
    blk = lambda off, i: slice(off + 6 * i, off + 6 * i + 6)
    ref = {"Hee": np.stack([H[blk(e_off, i), blk(e_off, i)] for i in range(n_e)]),
           "Hff": np.stack([H[blk(f_off, i), blk(f_off, i)] for i in range(n_f)]),
           "ge": g[e_off:e_off + 6 * n_e].reshape(-1, 6), "gf": g[f_off:f_off + 6 * n_f].reshape(-1, 6)}
    Je, Jf = (k1["jacobians"]["view"], k1["jacobians"]["marker"]) if ev else (k1["jacobians"]["marker"], k1["jacobians"]["view"])
    ref["W"] = np.einsum('nri,nrj->nij', Je, Jf)
    for k, v in ref.items():
        assert max_block_rel(nb[k], v, floor=1e-6 * np.abs(v).max()) < 1e-9, k
    e_idx = np.arange(e_off, e_off + 6 * n_e)
    Hd = H.copy()
    Hd[e_idx, e_idx] += np.clip(np.diag(H)[e_idx], 1e-6, 1e32) / RADIUS
    gd = g.copy()
    const = np.concatenate([np.repeat(s.const_views, 6), np.repeat(s.const_markers, 6), np.zeros(9, bool)])
    ce = e_idx[const[e_idx]]            # constant eliminated blocks are decoupled (the board is the gauge)
    Hd[ce, :] = 0
    Hd[:, ce] = 0
    Hd[ce, ce] = 1
    gd[ce] = 0
    f_idx = np.concatenate([np.arange(f_off, f_off + 6 * n_f), np.arange(6 * (nv + nm), H.shape[0])])
    X = np.linalg.solve(Hd[np.ix_(e_idx, e_idx)], np.concatenate([Hd[np.ix_(e_idx, f_idx)], gd[e_idx, None]], 1))
    S_ref = Hd[np.ix_(f_idx, f_idx)] - Hd[np.ix_(e_idx, f_idx)].T @ X[:, :-1]
    b_ref = gd[f_idx] - Hd[np.ix_(e_idx, f_idx)].T @ X[:, -1]
    assert rel_fro(S, S_ref) < 1e-9
    assert rel_fro(b, b_ref) < 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["single", "rig"])
def test_board_converges_to_the_truth(model):
    """From the perturbed start the solve reaches the truth to the noise level, and the board solve's intrinsics are
    at least as close to the truth as the solve of the same blocks as free tags would need a pose per tag for."""
    s = _board(model, pixel_noise=0.05)
    with BAProblem.from_scene(s, eliminate="views") as gp:
        summ = gp.solve(max_iterations=50)
        intr, _ = gp.get_intrinsics()
        markers = gp.get_marker_poses()
    assert summ["termination"] in (1, 2, 3)
    assert np.abs(intr - s.truth["intr"]).max() < 1.0
    assert np.abs(markers - s.truth["markers"]).max() < 2e-3
    assert summ["final_cost"] < 0.05 ** 2 * s.n_blocks * 8


@pytest.mark.gpu
def test_clearing_the_layout():
    """set_corner_layout(0) returns the handle to the plain launches and to results bitwise equal to a fresh plain
    handle; set_observations clears the layout too."""
    s, scale = _scene("rig", "mixed")
    plain = _flat(_run(s, "views", "huber", scale))
    layout = square_layout(s)
    layout[0][:, :, :] *= 1.01
    for how in ("clear", "observations"):
        with kernels_launched() as launched:
            with BAProblem.from_scene(s, eliminate="views") as gp:
                gp.set_corner_layout(*layout)
                gp.linearize()
                if how == "clear":
                    gp.clear_corner_layout()
                else:
                    gp.set_observations(s.view_idx, s.marker_idx, s.cam_idx, s.pixels)
                gp.set_loss("huber", scale)
                got = {"k1": gp.evaluate(), "k6": gp.evaluate(want_jacobians=False), "cost": gp.linearize(),
                       "nb": gp.normal_blocks()}
                gp.schur(RADIUS)
                got["S"], got["b"] = gp.reduced_system()
                got["mcc"] = gp.solve_step()
                got["step"] = gp.step()
                got["cand"] = gp.candidate_cost()
        got = _flat(got)
        for k, v in plain.items():
            assert np.array_equal(np.asarray(got[k]), np.asarray(v)), (how, k)
        names = {k for k, _ in launched}
        assert {"evaluate_kernel", "assemble_kernel", "materialise_kernel"} <= names
        assert "assemble_target_kernel" in names   # the linearisation before the layout was cleared


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["f64", "i16"])
def test_piecewise_update_keeps_the_layout(dtype):
    """update_pixels in the sorted order (the piecewise path) with a layout: bitwise the one-shot setup."""
    s = _board("rig")
    order = np.lexsort((s.marker_idx, s.cam_idx, s.view_idx))
    for k in ("view_idx", "marker_idx", "cam_idx", "pixels", "corner_slot"):
        setattr(s, k, getattr(s, k)[order])
    if dtype == "i16":
        s.pixels = np.trunc(s.pixels).astype(np.int16)
    with BAProblem.from_scene(s, eliminate="views") as gp:
        c0 = gp.linearize()
        nb0 = gp.normal_blocks()
        gp.update_pixels(s.pixels)
        c1 = gp.linearize()
        nb1 = gp.normal_blocks()
    assert c1 == c0
    for k in nb0:
        assert np.array_equal(nb0[k], nb1[k]), k


@pytest.mark.gpu
def test_bad_arguments_change_nothing():
    s = _board("single")
    n = s.n_blocks
    good = (s.corners, s.corner_slot)
    with BAProblem(len(s.views), len(s.markers), 1, n) as gp:
        rc = gp.lib.rcc_ba_set_corner_layout(gp.h, 0, None, None)
        assert rc == L.RCC_NOT_READY
    with BAProblem.from_scene(s) as gp:
        ref = gp.linearize()
        c = np.ascontiguousarray(s.corners)
        bad_c = c.copy()
        bad_c[3, 2, 1] = np.nan
        sl = np.ascontiguousarray(s.corner_slot)
        cases = [(-1, c, sl), (len(c), None, sl), (len(c), c, None), (len(c), bad_c, sl)]
        for v in (len(c), -2):
            b = sl.copy()
            b[n // 2] = v
            cases.append((len(c), c, b))
        dp = lambda a: None if a is None else a.ctypes.data_as(L.c_double_p)
        ip = lambda a: None if a is None else a.ctypes.data_as(L.c_int32_p)
        for k, (ns, cc, ss) in enumerate(cases):
            assert gp.lib.rcc_ba_set_corner_layout(gp.h, ns, dp(cc), ip(ss)) == L.RCC_BAD_ARG, k
            assert gp.linearize() == ref, k
        gp.set_corner_layout(*good)
        assert gp.linearize() == ref


@pytest.mark.gpu
def test_ceres_like_board_is_the_corner_layout():
    """TagReprojectionCost(corners=) residual blocks sharing one marker array: the same cost, gradient and solve as
    BAProblem with the layout."""
    from robot_camera_calibration_b200 import ceres_like as CL
    s = make_target_scene(3, 4, 8, n_free=2, seed=5)
    intr, dist = s.intr[0].copy(), s.dist[0].copy()
    views = [v.copy() for v in s.views]
    markers = [m.copy() for m in s.markers]
    pb = CL.Problem()
    for i in range(s.n_blocks):
        k = s.corner_slot[i]
        cost = (CL.TagReprojectionCost(s.pixels[i], corners=s.corners[k]) if k >= 0 else
                CL.TagReprojectionCost(s.pixels[i], tag_size=s.sizes[s.marker_idx[i]]))
        pb.AddResidualBlock(cost, None, intr, dist, views[s.view_idx[i]], markers[s.marker_idx[i]])
    pb.SetParameterBlockConstant(markers[0])
    o = CL.SolverOptions()
    with BAProblem.from_scene(s) as gp:
        ref = gp.evaluate()
        gp.solve(max_iterations=o.max_num_iterations, initial_radius=o.initial_trust_region_radius,
                 max_radius=o.max_trust_region_radius, min_relative_decrease=o.min_relative_decrease,
                 function_tolerance=o.function_tolerance, gradient_tolerance=o.gradient_tolerance,
                 parameter_tolerance=o.parameter_tolerance, min_diagonal=o.min_lm_diagonal,
                 max_diagonal=o.max_lm_diagonal, jacobi_scaling=int(o.jacobi_scaling))
        ref_views, ref_markers = gp.get_view_poses(), gp.get_marker_poses()
    cost, res, _ = pb.Evaluate()
    assert abs(cost - ref["cost"]) <= 1e-12 * ref["cost"]
    assert np.array_equal(res, ref["residuals"].ravel())
    CL.Solve(o, pb)
    # the Problem numbers blocks by first use: the same solve up to the order of its sums
    np.testing.assert_allclose(np.stack(views), ref_views, atol=1e-9)
    np.testing.assert_allclose(np.stack(markers), ref_markers, atol=1e-9)


@pytest.mark.gpu
def test_command_line_target(tmp_path, capsys):
    """A board dataset written per tag plus an AprilGrid file through the command line: the tags of the grid in the
    refined targets.yaml are rigid (board_T_tag between any two equals the layout), the JSON carries the board pose,
    and a tag id on two targets exits with status 2."""
    import json
    import shutil
    from robot_camera_calibration_b200 import io_yaml
    from robot_camera_calibration_b200.__main__ import main
    from robot_camera_calibration_b200.scenes import compose, invert
    from test_targets_host import scene_as_tags
    s = make_target_scene(3, 4, 20, n_free=3, seed=6)
    tags, ids = scene_as_tags(s)
    d = str(tmp_path / "data")
    io_yaml.write_dataset(d, tags, tag_ids=ids)
    grid = tmp_path / "grid.yaml"
    grid.write_text("target_type: aprilgrid\ntagCols: 4\ntagRows: 3\ntagSize: 0.1\ntagSpacing: 0.3\n")
    capsys.readouterr()
    assert main([d, "--precision", "repr", "--target", str(grid)]) == 0
    out = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert len(out["boards"]) == 1 and out["boards"][0]["first_tag_id"] == 0
    r, got_ids, _ = io_yaml.read_dataset(d)
    on = got_ids < 12
    pose = {int(i): r.markers[k] for k, i in enumerate(got_ids)}
    ctr = s.corners.mean(1)
    for i in range(12):
        rel = compose(invert(pose[0]), pose[i])
        np.testing.assert_allclose(rel, [0, 0, 0, *(ctr[i] - ctr[0]), 0], atol=1e-12)
    np.testing.assert_allclose(out["boards"][0]["world_T_board"], compose(pose[0], invert(
        np.array([0, 0, 0, *ctr[0], 0.0]))), atol=1e-12)
    assert on.sum() == 12
    other = tmp_path / "other.yaml"
    other.write_text("target_type: aprilgrid\ntagCols: 2\ntagRows: 2\ntagSize: 0.1\ntagSpacing: 0.3\nfirstTagId: 11\n")
    d2 = str(tmp_path / "data2")
    shutil.copytree(d, d2)
    assert main([d2, "--target", str(grid), "--target", str(other)]) == 2
    capsys.readouterr()
