"""GPU: the equidistant (fisheye) lens through the C ABI against the CPU oracles of tests/lens_oracle.py (oracle A:
closed form + complex step, oracle B: cv2.fisheye), with the tolerances of test_gpu_parity.py.  The scenes are wide-
angle cameras (1280 x 1024, f ~ 330 px) whose tags reach 85 degrees off the optical axis."""
import os
import subprocess
import sys

import numpy as np
import pytest

import lens_oracle as LO
from helpers import max_block_rel, rel_fro
from robot_camera_calibration_b200 import _lib as L
from robot_camera_calibration_b200 import io_yaml
from robot_camera_calibration_b200.initialiser import pnp_batch
from robot_camera_calibration_b200.problem import BAProblem
from robot_camera_calibration_b200.scenes import compose, invert, make_scene

pytestmark = pytest.mark.gpu
TOL = 1e-9
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SCENES = {
    "single": dict(n_markers=12, n_views=30, visibility=0.7, seed=11),
    "rig": dict(n_markers=16, n_views=20, visibility=0.6, n_cam=3, model="rig", seed=13),
}


def _compact(s):
    """Drop views and markers that no block observes (the scenes turn some cameras away from the wall)."""
    for kind, idx in (("views", "view_idx"), ("markers", "marker_idx")):
        used = np.unique(getattr(s, idx))
        remap = np.full(len(getattr(s, kind)), -1)
        remap[used] = np.arange(len(used))
        setattr(s, kind, getattr(s, kind)[used])
        setattr(s, "const_" + kind, getattr(s, "const_" + kind)[used])
        setattr(s, idx, remap[getattr(s, idx)].astype(np.int32))
        s.truth[kind] = s.truth[kind][used]
    if not s.const_markers.any():
        s.const_markers[0] = True
    return s


def _scene(name, **kw):
    args = dict(SCENES[name])
    args.update(kw)
    return _compact(make_scene(args.pop("n_markers"), args.pop("n_views"), args.pop("visibility"),
                               lens="equidistant", **args))


@pytest.mark.parametrize("name", list(SCENES))
def test_evaluate_matches_both_oracles(name):
    s = _scene(name)
    p = LO.oracle_problem(s)
    r, Jb = LO.residuals(p), LO.jacobian_blocks_cs(p)
    with BAProblem.from_scene(s) as gp:
        out = gp.evaluate()
    assert abs(out["cost"] - LO.cost(p)) <= TOL * LO.cost(p)
    assert max_block_rel(out["residuals"], r) < TOL
    for k in Jb:
        assert max_block_rel(out["jacobians"][k], Jb[k]) < TOL, k
    assert np.all(out["jacobians"]["dist"][..., 4] == 0.0)          # the reserved slot
    for b in range(0, s.n_blocks, 7):                                  # oracle B: OpenCV's analytic chain
        c, v, m = s.cam_idx[b], s.view_idx[b], s.marker_idx[b]
        pts, J = LO.jacobian_block_cv2(s.model, s.intr[c], s.dist[c], s.ext[c], s.views[v], s.markers[m], s.sizes[m])
        assert np.abs(out["residuals"][b] + s.pixels[b] - pts).max() < 1e-9
        for k in J:
            assert rel_fro(out["jacobians"][k][b], J[k]) < 1e-8, (b, k)


@pytest.mark.parametrize("elim", ["views", "markers"])
@pytest.mark.parametrize("name", list(SCENES))
def test_normal_equations_schur_and_step_match_oracle(name, elim):
    s = _scene(name)
    s.dist[:, 4] = 0.125              # the reserved slot: ignored by the projection, never stepped
    p = LO.oracle_problem(s)
    ob = LO.blocks(p, elim == "views")
    radius = 1e4
    S, b = LO.reduced(p, elim == "views", radius)
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        cost = gp.linearize()
        nb = gp.normal_blocks()
        gp.schur(radius)
        Sg, bg = gp.reduced_system()
        mcc, step_norm, _ = gp.solve_step()
        st = gp.step()
        c_new = gp.candidate_cost()
        gp.accept_step()
        intr, dist = gp.get_intrinsics()
    assert abs(cost - ob["cost"]) <= TOL * ob["cost"]
    for k in ("Hee", "Hff", "W", "ge", "gf", "Hes", "Hfs"):
        assert max_block_rel(nb[k], ob[k], floor=1e-6 * np.abs(ob[k]).max()) < TOL, k
    assert rel_fro(nb["Hss"], ob["Hss"]) < TOL and rel_fro(nb["gs"], ob["gs"]) < TOL
    assert rel_fro(Sg, S) < TOL and rel_fro(bg, b) < TOL
    delta, mcc_o, _, _ = LO.lm_step(p, radius)
    o_view, o_marker, o_shared, n = p.offsets()
    dv, dm, ds = (delta[o_view:o_marker].reshape(-1, 6), delta[o_marker:o_shared].reshape(-1, 6), delta[o_shared:])
    de, df = (dv, dm) if elim == "views" else (dm, dv)
    assert rel_fro(st["d_e"], de) < 1e-6 and rel_fro(st["d_f"], df) < 1e-6 and rel_fro(st["d_shared"], ds) < 1e-6
    assert abs(mcc - mcc_o) <= 1e-6 * abs(mcc_o)
    assert abs(step_norm - np.linalg.norm(delta)) <= 1e-6 * np.linalg.norm(delta)
    sp = p.shared_per_cam
    assert np.all(st["d_shared"][sp * np.arange(p.n_cam) + 8] == 0.0)
    assert np.all(dist[:, 4] == 0.125)
    cand = p.copy()
    cand.unpack(p.pack() + delta)
    assert abs(c_new - LO.cost(cand)) <= 1e-6 * LO.cost(cand)


@pytest.mark.parametrize("name", list(SCENES))
def test_huber_and_jacobi_scaling(name):
    s = _scene(name)
    rng = np.random.default_rng(5)
    bad = rng.choice(s.n_blocks, 12, replace=False)
    s.pixels[bad] += rng.normal(0, 25.0, (12, 8))
    p = LO.oracle_problem(s)
    p.loss, p.loss_scale = "huber", 2.0
    ob = LO.blocks(p, True)
    S, b = LO.reduced(p, True, 1e4)
    steps = {}
    for jac in (False, True):
        with BAProblem.from_scene(s, eliminate="views") as gp:
            gp.set_loss("huber", 2.0)
            gp.set_lm_diagonal(1e-6, 1e32, jac)
            cost = gp.linearize()
            nb = gp.normal_blocks()
            gp.schur(1e4)
            Sg, bg = gp.reduced_system()
            gp.solve_step()
            st = gp.step()
            steps[jac] = np.concatenate([st["d_e"].ravel(), st["d_f"].ravel(), st["d_shared"]])
        assert abs(cost - ob["cost"]) <= TOL * ob["cost"]
        for k in ("Hee", "Hff", "W", "ge", "gf", "Hes", "Hfs"):
            assert max_block_rel(nb[k], ob[k], floor=1e-6 * np.abs(ob[k]).max()) < TOL, k
        assert rel_fro(nb["Hss"], ob["Hss"]) < TOL and rel_fro(Sg, S) < TOL and rel_fro(bg, b) < TOL
    # the clamp of the scaled diagonal is inactive on every free parameter here: the same step
    assert rel_fro(steps[True], steps[False]) < 1e-9
    delta, _, _, _ = LO.lm_step(p, 1e4)
    o_shared = p.offsets()[2]
    assert rel_fro(steps[False][-len(s.intr) * p.shared_per_cam:], delta[o_shared:]) < 1e-6


@pytest.mark.parametrize("elim", ["views", "markers"])
@pytest.mark.parametrize("name", list(SCENES))
def test_reserved_slot_covariance(name, elim):
    s = _scene(name)
    p = LO.oracle_problem(s)
    H, _, _ = LO.normal_equations(p)
    free = np.nonzero(~p.const_mask())[0]
    C = np.zeros_like(H)
    C[np.ix_(free, free)] = np.linalg.inv(H[np.ix_(free, free)])
    o_shared = p.offsets()[2]
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        cov = gp.covariance()
        pair = gp.covariance_blocks([(("dist", 0), ("dist", 0)), (("dist", 0), ("view", 1))])
    sp = p.shared_per_cam
    slot = sp * np.arange(p.n_cam) + 8
    assert np.all(cov["shared"][slot, :] == 0.0) and np.all(cov["shared"][:, slot] == 0.0)
    assert np.all(pair[0][4, :] == 0.0) and np.all(pair[0][:, 4] == 0.0) and np.all(pair[1][4, :] == 0.0)
    Cs = C[o_shared:, o_shared:]
    assert rel_fro(cov["shared"], Cs) < 1e-6
    k14 = slice(4, 8)
    for c in range(p.n_cam):
        blk = cov["shared"][sp * c:sp * c + 9, sp * c:sp * c + 9]
        assert rel_fro(blk[k14, k14], Cs[sp * c:sp * c + 9, sp * c:sp * c + 9][k14, k14]) < 1e-6


def test_converged_parameters_match_an_independent_solver():
    from scipy.optimize import least_squares
    s = _scene("single", n_markers=8, n_views=14, visibility=0.9, seed=61)
    p = LO.oracle_problem(s)
    free = ~p.const_mask()
    x0 = p.pack()

    def with_x(xf):
        q = p.copy()
        x = x0.copy()
        x[free] = xf
        q.unpack(x)
        return q

    sol = least_squares(lambda xf: LO.residuals(with_x(xf)).ravel(), x0[free],
                        jac=lambda xf: LO.O.dense_jacobian(with_x(xf), LO.jacobian_blocks_cs(with_x(xf)))[:, free],
                        method="trf", x_scale="jac", ftol=1e-15, xtol=1e-15, gtol=1e-13, max_nfev=200)
    ref = with_x(sol.x)
    with BAProblem.from_scene(s) as gp:
        summ = gp.solve(max_iterations=100, function_tolerance=1e-16, gradient_tolerance=1e-13,
                        parameter_tolerance=1e-15)
        views, markers = gp.get_view_poses(), gp.get_marker_poses()
        intr, dist = gp.get_intrinsics()
    assert abs(summ["final_cost"] - LO.cost(ref)) <= 1e-9 * LO.cost(ref)
    assert np.abs(views - ref.views).max() < 1e-6
    assert np.abs(markers - ref.markers).max() < 1e-6
    assert np.abs(dist - ref.dist).max() < 1e-6
    assert np.abs(intr - ref.intr).max() < 1e-4


@pytest.mark.parametrize("name", list(SCENES))
def test_wide_angle_solve_recovers_the_truth(name):
    s = _scene(name, pixel_noise=0.0)
    with BAProblem.from_scene(s) as gp:
        summ = gp.solve(max_iterations=100, function_tolerance=1e-16, gradient_tolerance=1e-14,
                        parameter_tolerance=1e-15)
        views, markers = gp.get_view_poses(), gp.get_marker_poses()
        intr, dist = gp.get_intrinsics()
    assert summ["final_cost"] < 1e-14 * summ["initial_cost"]
    assert np.abs(views - s.truth["views"]).max() < 1e-6
    assert np.abs(markers - s.truth["markers"]).max() < 1e-6
    assert np.abs(intr - s.truth["intr"]).max() < 1e-4
    assert np.abs(dist[:, :4] - s.truth["dist"][:, :4]).max() < 1e-6


def _pnp_problem(noise, seed=3):
    """Tags of a wide-angle scene with their true cam_T_tag = inv(world_T_camera) * world_T_target."""
    s = _compact(make_scene(10, 12, 0.8, seed=seed, pixel_noise=noise, lens="equidistant"))
    return s, compose(invert(s.truth["views"][s.view_idx]), s.truth["markers"][s.marker_idx])


def _pnp_least_squares(intr, dist, size, pix, x0):
    """The same pixel cost (view = identity, marker = cam_T_tag) converged tightly by SciPy."""
    from scipy.optimize import least_squares

    def res(x):
        uv, _ = LO.project_blocks("single", "equidistant", intr[None], dist[None], np.zeros((1, 6)), np.zeros((1, 6)),
                                  x[None], np.array([size]))
        return uv.reshape(8) - pix
    return least_squares(res, x0, method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15, max_nfev=2000).x


def _ippe_starts(intr, dist, size, pix):
    """Both poses of the planar ambiguity, from OpenCV alone: cv2.fisheye.undistortPoints, then IPPE."""
    import cv2
    K = np.array([[intr[0], 0, intr[2]], [0, intr[1], intr[3]], [0, 0, 1.0]])
    und = cv2.fisheye.undistortPoints(pix.reshape(1, 4, 2), K, dist[:4].reshape(4, 1))
    n, rvs, tvs, _ = cv2.solvePnPGeneric(LO.O.obj_points(size).reshape(4, 1, 3), und.reshape(4, 1, 2), np.eye(3),
                                        None, flags=cv2.SOLVEPNP_IPPE)
    return [np.concatenate([r.ravel(), t.ravel()]) for r, t in zip(rvs, tvs)]


def test_pnp_matches_least_squares_and_cv2_fisheye():
    import cv2
    s, truth = _pnp_problem(0.3)
    intr, dist = s.truth["intr"][0], s.truth["dist"][0]
    sizes = s.sizes[s.marker_idx]
    guess = truth + np.random.default_rng(1).normal(0, [0.05] * 3 + [0.02] * 3, truth.shape)
    for start in (None, guess):
        poses, cost = pnp_batch(intr, dist, sizes, s.pixels, guess=start, lens="equidistant")
        assert np.all(cost >= 0)
        for b in range(0, s.n_blocks, 5):
            if start is not None:        # from a guess: the minimum SciPy reaches from the same guess
                refs = [_pnp_least_squares(intr, dist, sizes[b], s.pixels[b], start[b])]
            else:                        # from zeros: either minimum of the planar pose ambiguity (IPPE's two)
                refs = [_pnp_least_squares(intr, dist, sizes[b], s.pixels[b], x0)
                        for x0 in _ippe_starts(intr, dist, sizes[b], s.pixels[b])]
            err = min(np.abs(poses[b] - ref).max() for ref in refs)
            assert err < 1e-6, (b, poses[b], refs)
    # noise-free pixels: OpenCV's fisheye PnP finds the same pose
    s0, truth0 = _pnp_problem(0.0)
    poses0, _ = pnp_batch(intr, dist, s0.sizes[s0.marker_idx], s0.pixels, lens="equidistant")
    K = np.array([[intr[0], 0, intr[2]], [0, intr[1], intr[3]], [0, 0, 1.0]])
    for b in range(0, s0.n_blocks, 5):
        o = LO.O.obj_points(s0.sizes[s0.marker_idx[b]]).reshape(1, 4, 3)
        ok, rv, tv = cv2.fisheye.solvePnP(o, s0.pixels[b].reshape(1, 4, 2), K, dist[:4].reshape(4, 1))
        assert ok
        assert np.abs(poses0[b] - truth0[b]).max() < 1e-6
        assert np.abs(np.concatenate([rv.ravel(), tv.ravel()]) - poses0[b]).max() < 1e-4


def test_corner_behind_the_camera_fails_the_evaluation():
    s = _scene("single")
    s.views[3] = compose(s.views[3], np.array([0.0, np.pi, 0.0, 0.0, 0.0, 0.0]))
    assert (LO.depths(LO.oracle_problem(s)) <= 0).any()
    with BAProblem.from_scene(s) as gp:
        out = gp.evaluate(allow_failure=True)
        assert out["failed"]
        with pytest.raises(L.RccError) as e:
            gp.linearize()
        assert e.value.status == L.RCC_EVAL_FAILED


def test_switching_the_lens_back_is_bitwise_a_fresh_handle():
    s = make_scene(12, 30, 0.7, seed=11)
    outs = []
    for switch in (False, True):
        with BAProblem.from_scene(s) as gp:
            if switch:
                gp.set_lens("equidistant")
                gp.linearize()
                gp.set_lens("radtan")
            ev = gp.evaluate()
            cost = gp.linearize()
            nb = gp.normal_blocks()
            summ = gp.solve(max_iterations=5)
            outs.append((ev, cost, nb, summ, gp.get_view_poses(), gp.get_intrinsics()))
    (e0, c0, n0, s0, v0, i0), (e1, c1, n1, s1, v1, i1) = outs
    assert c0 == c1 and np.array_equal(e0["residuals"], e1["residuals"])
    assert all(np.array_equal(e0["jacobians"][k], e1["jacobians"][k]) for k in e0["jacobians"])
    assert all(np.array_equal(n0[k], n1[k]) for k in n0)
    assert s0["final_cost"] == s1["final_cost"] and np.array_equal(v0, v1)
    assert np.array_equal(i0[0], i1[0]) and np.array_equal(i0[1], i1[1])
    with BAProblem.from_scene(s) as gp:
        assert gp.lib.rcc_ba_set_lens(gp.h, 7) == L.RCC_BAD_ARG
        with pytest.raises(ValueError):
            gp.set_lens("fisheye")


def test_cli_on_an_equidistant_detections_directory(tmp_path):
    s = make_scene(10, 25, 0.8, seed=8, pixel_noise=0.0, perturb=(0.01, 0.01, 0.0), lens="equidistant")
    io_yaml.write_dataset(str(tmp_path), s)
    r = subprocess.run([sys.executable, "-m", "robot_camera_calibration_b200", str(tmp_path), "--max-iterations", "60"],
                       cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    import json
    summ = json.loads(r.stdout.strip().splitlines()[-1])
    assert summ["termination"] in (1, 2, 3), summ
    assert summ["final_cost"] < 0.2 * summ["initial_cost"]
    intr, dist, lens = io_yaml.read_camera(str(tmp_path / "camera_refined.yaml"))
    assert lens == "equidistant"
    assert "distortion_model: equidistant" in (tmp_path / "camera_refined.yaml").read_text()
