"""Parameter covariance (rcc_ba_covariance, BAProblem.covariance, ceres_like.Covariance) against dense host inverses.

C = (J^T J)^-1 of the undamped system restricted to the free parameters, zero at the constants.  The scenes' J^T J
have condition numbers of about 3e9 (single) and 3e10 (rig), so two correct FP64 inversions may differ by far more
than rounding: 1e-6 relative per block is the conditioning allowance, as for the LM step.
"""
import numpy as np
import pytest

import ba_oracle as O
from helpers import max_block_rel, to_oracle
from robot_camera_calibration_b200 import _lib as L
from robot_camera_calibration_b200 import ceres_like as CL
from robot_camera_calibration_b200.problem import BAProblem
from robot_camera_calibration_b200.scenes import config_scene, make_scene
from test_gpu_parity import SCENES, _scene

pytestmark = pytest.mark.gpu
TOL = 1e-6
TILE = 32          # partners per tile of cov_eliminated_kernel


def oracle_covariance(p):
    """(C_views, C_markers, C_shared) from the dense oracle's J^T J."""
    H, _, _ = O.normal_equations(p)
    free = np.nonzero(~p.const_mask())[0]
    C = np.zeros_like(H)
    C[np.ix_(free, free)] = np.linalg.inv(H[np.ix_(free, free)])
    o_view, o_marker, o_shared, _ = p.offsets()
    blocks = lambda off, k: np.stack([C[off + 6 * i:off + 6 * i + 6, off + 6 * i:off + 6 * i + 6] for i in range(k)])
    return blocks(o_view, len(p.views)), blocks(o_marker, len(p.markers)), C[o_shared:, o_shared:]


def compare(cov, ref_views, ref_markers, ref_shared):
    """Largest per-block relative Frobenius error over the view, marker and shared blocks."""
    err = {}
    for k, ref in (("views", ref_views), ("markers", ref_markers)):
        floor = 1e-6 * np.linalg.norm(ref.reshape(len(ref), -1), axis=1).max()
        err[k] = max_block_rel(cov[k], ref, floor=floor)
    err["shared"] = max_block_rel(cov["shared"][None], ref_shared[None])
    return err


@pytest.mark.parametrize("elim", ["views", "markers"])
@pytest.mark.parametrize("name", list(SCENES))
def test_covariance_matches_dense_inverse(name, elim):
    s = _scene(name)
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        cov = gp.covariance()
    err = compare(cov, *oracle_covariance(to_oracle(s)))
    print(f"{name}/{elim}: largest block error {max(err.values()):.2e} {err}")
    assert max(err.values()) < TOL, err


def test_covariance_with_huber_loss():
    s = _scene("single")
    rng = np.random.default_rng(5)
    bad = rng.choice(s.n_blocks, 12, replace=False)
    s.pixels[bad] += rng.normal(0, 25.0, (12, 8))
    p = to_oracle(s)
    p.loss, p.loss_scale = "huber", 2.0
    with BAProblem.from_scene(s, eliminate="views") as gp:
        gp.set_loss("huber", 2.0)
        cov = gp.covariance()
    err = compare(cov, *oracle_covariance(p))
    print(f"huber: largest block error {max(err.values()):.2e}")
    assert max(err.values()) < TOL, err


@pytest.mark.parametrize("elim", ["views", "markers"])
def test_constant_blocks_give_exact_zeros(elim):
    s = _scene("single_2cam")
    s.const_intr[1] = True
    s.const_views[3] = True
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        cov = gp.covariance()
    sh = cov["shared"]
    assert np.all(cov["views"][3] == 0)
    assert np.all(cov["markers"][0] == 0)                  # the gauge
    assert np.all(sh[9:13, :] == 0) and np.all(sh[:, 9:13] == 0)
    err = compare(cov, *oracle_covariance(to_oracle(s)))
    assert max(err.values()) < TOL, err


def _unobserved_marker_scene():
    s = _scene("single")
    keep = s.marker_idx != 5
    s.view_idx, s.marker_idx, s.cam_idx, s.pixels = s.view_idx[keep], s.marker_idx[keep], s.cam_idx[keep], s.pixels[keep]
    return s


@pytest.mark.parametrize("elim", ["markers", "views"])
def test_unobserved_block_is_not_spd(elim):
    with BAProblem.from_scene(_unobserved_marker_scene(), eliminate=elim) as gp:
        with pytest.raises(L.RccError) as ei:
            gp.covariance()
    assert ei.value.status == L.RCC_NOT_SPD


@pytest.mark.parametrize("elim", ["markers", "views"])
def test_problem_without_gauge_is_not_spd(elim):
    s = _scene("single")
    s.const_markers[:] = False
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        with pytest.raises(L.RccError) as ei:
            gp.covariance()
    assert ei.value.status == L.RCC_NOT_SPD


def test_solve_after_covariance_is_unchanged():
    s = _scene("rig")
    opts = dict(max_iterations=30, function_tolerance=1e-14, gradient_tolerance=1e-12, parameter_tolerance=1e-13)
    res = []
    for with_cov in (False, True):
        with BAProblem.from_scene(s, eliminate="views") as gp:
            if with_cov:
                gp.covariance()
            summ = gp.solve(**opts)
            res.append((summ["final_cost"], gp.get_view_poses(), gp.get_marker_poses(), gp.get_intrinsics()[0]))
    assert abs(res[0][0] - res[1][0]) <= 1e-12 * res[0][0]
    for a, b in zip(res[0][1:], res[1][1:]):
        assert np.abs(a - b).max() < 1e-10


def test_two_calls_are_bitwise_equal():
    s = config_scene(2, scale=0.2)
    with BAProblem.from_scene(s, eliminate="views") as gp:
        a = gp.covariance()
        b = gp.covariance()
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def _host_eliminated_covariance(gp, scene, sample):
    """Cov(e) rebuilt on the host from the undamped reduced system and the normal-equation blocks."""
    d = gp.dims
    gp.linearize()
    gp.schur(float("inf"))
    S, _ = gp.reduced_system()
    nb = gp.normal_blocks()
    const = np.zeros(d.n_reduced, bool)
    elim_view = bool(d.eliminated_is_view)
    cf = scene.const_markers if elim_view else scene.const_views
    const[:6 * d.n_f] = np.repeat(cf, 6)
    sp = 15 if scene.model == "rig" else 9
    for c in range(len(scene.intr)):
        const[6 * d.n_f + sp * c:6 * d.n_f + sp * c + 4] = scene.const_intr[c]
        const[6 * d.n_f + sp * c + 4:6 * d.n_f + sp * c + 9] = scene.const_dist[c]
    free = np.nonzero(~const)[0]
    Si = np.zeros_like(S)
    Si[np.ix_(free, free)] = np.linalg.inv(S[np.ix_(free, free)])
    e_of = scene.view_idx if elim_view else scene.marker_idx
    f_of = scene.marker_idx if elim_view else scene.view_idx
    out = {}
    for e in sample:
        B = np.zeros((6, d.n_reduced))
        for o in np.nonzero(e_of == e)[0]:
            B[:, 6 * f_of[o]:6 * f_of[o] + 6] += nb["W"][o]          # W summed per (e, f) over cameras
        B[:, 6 * d.n_f:] = nb["Hes"][e]
        Hi = np.linalg.inv(nb["Hee"][e])
        out[e] = Hi + Hi @ B @ Si @ B.T @ Hi
    return out


@pytest.mark.parametrize("case", ["cfg2", "long_rows"])
def test_long_rows_match_host_rebuild(case):
    if case == "cfg2":
        s = config_scene(2)
    else:
        # cfg4-shaped: a few hundred keyframes that each see 500+ tags (the generator's nearer views see fewer: drop them)
        s = make_scene(1500, 300, 0.7, seed=41)
        seen = np.bincount(s.view_idx, minlength=len(s.views))
        keep_v = np.nonzero(seen >= 500)[0]
        new_id = np.full(len(s.views), -1)
        new_id[keep_v] = np.arange(len(keep_v))
        keep = new_id[s.view_idx] >= 0
        s.views, s.const_views = s.views[keep_v], s.const_views[keep_v]
        s.view_idx, s.marker_idx, s.cam_idx, s.pixels = (new_id[s.view_idx[keep]], s.marker_idx[keep], s.cam_idx[keep],
                                                         s.pixels[keep])
    rows = [len(np.unique(s.marker_idx[s.view_idx == v])) for v in range(len(s.views))]
    if case == "long_rows":
        assert min(rows) >= 500 and max(rows) > 3 * TILE
    sample = np.random.default_rng(0).choice(len(s.views), 12, replace=False)
    with BAProblem.from_scene(s, eliminate="views") as gp:
        ref = _host_eliminated_covariance(gp, s, sample)
        cov = gp.covariance()
    got = np.stack([cov["views"][e] for e in sample])
    want = np.stack([ref[e] for e in sample])
    err = max_block_rel(got, want)
    print(f"{case}: longest row {max(rows)} partners, largest block error {err:.2e}")
    assert err < TOL


def test_covariance_covers_the_estimation_error():
    """Over 30 seeded scenes with sigma = 0.3 px, e^T (sigma^2 C_ss)^-1 e of the converged intrinsics + distortion
    must average like 30 draws of chi^2(9): inside [6.4, 11.6], the 99.9 % band of that mean."""
    sigma, stats = 0.3, []
    for seed in range(100, 130):
        s = make_scene(8, 20, 0.7, seed=seed, pixel_noise=sigma)
        with BAProblem.from_scene(s) as gp:
            gp.solve(max_iterations=50, function_tolerance=1e-14, gradient_tolerance=1e-12, parameter_tolerance=1e-13)
            intr, dist = gp.get_intrinsics()
            C = sigma ** 2 * gp.covariance()["shared"]
        e = np.concatenate([intr[0], dist[0]]) - np.concatenate([s.truth["intr"][0], s.truth["dist"][0]])
        stats.append(float(e @ np.linalg.solve(C, e)))
    print(f"mean chi^2(9) statistic {np.mean(stats):.2f}")
    assert 6.4 <= np.mean(stats) <= 11.6


def _ceres_problem(s, loss=None):
    """The scene as a ceres_like.Problem, one residual block per tag observation."""
    intr = [np.ascontiguousarray(s.intr[c], dtype=np.float64) for c in range(len(s.intr))]
    dist = [np.ascontiguousarray(s.dist[c], dtype=np.float64) for c in range(len(s.dist))]
    views = [np.ascontiguousarray(v, dtype=np.float64) for v in s.views]
    markers = [np.ascontiguousarray(m, dtype=np.float64) for m in s.markers]
    pr = CL.Problem()
    for o in range(s.n_blocks):
        c = int(s.cam_idx[o])
        pr.AddResidualBlock(CL.TagReprojectionCost(s.pixels[o], s.sizes[s.marker_idx[o]]), loss, intr[c], dist[c],
                            views[s.view_idx[o]], markers[s.marker_idx[o]])
    pr.SetParameterBlockConstant(markers[0])
    return pr, intr, dist, views, markers


def test_ceres_like_covariance_matches_the_library():
    s = _scene("single_2cam")
    pr, intr, dist, views, markers = _ceres_problem(s, CL.HuberLoss(2.0))
    CL.Solve(CL.SolverOptions(max_num_iterations=20), pr)
    pr.SetParameterBlockConstant(intr[1])
    blocks = [(intr[0], intr[0]), (intr[0], dist[1]), (dist[1], intr[1]), (views[2], views[2]),
              (markers[3], markers[3]), (markers[0], markers[0]), (intr[1], intr[1])]
    for apply_loss in (True, False):
        cv = CL.Covariance(CL.CovarianceOptions(apply_loss_function=apply_loss))
        assert cv.Compute(blocks, pr)
        gp, (vlist, mlist, clist, _) = pr._build()
        with gp:
            if not apply_loss:
                gp.set_loss("trivial")
            ref = gp.covariance()
        vi = [id(a) for a in vlist].index(id(views[2]))
        mi = [id(a) for a in mlist].index(id(markers[3]))
        ci = [id(c[1]) for c in clist]
        c0, c1 = ci.index(id(intr[0])), ci.index(id(intr[1]))
        out = np.empty((4, 5))
        assert cv.GetCovarianceBlock(intr[0], dist[1], out)
        assert np.array_equal(out, ref["shared"][9 * c0:9 * c0 + 4, 9 * c1 + 4:9 * c1 + 9])
        out = np.empty((4, 4))
        assert cv.GetCovarianceBlock(intr[0], intr[0], out)
        assert np.array_equal(out, ref["shared"][9 * c0:9 * c0 + 4, 9 * c0:9 * c0 + 4])
        out = np.empty((5, 4))
        assert cv.GetCovarianceBlock(dist[1], intr[1], out) and np.all(out == 0)     # intr[1] is constant
        out = np.empty((6, 6))
        assert cv.GetCovarianceBlock(views[2], views[2], out) and np.array_equal(out, ref["views"][vi])
        assert cv.GetCovarianceBlock(markers[3], markers[3], out) and np.array_equal(out, ref["markers"][mi])
        assert cv.GetCovarianceBlock(markers[0], markers[0], out) and np.all(out == 0)
        assert not cv.GetCovarianceBlock(views[2], views[3], out)                     # not requested
    with pytest.raises(NotImplementedError):
        CL.Covariance().Compute([(views[2], markers[3])], pr)
    with pytest.raises(NotImplementedError):
        CL.Covariance().Compute([(views[2], views[3])], pr)
