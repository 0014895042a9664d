"""GPU: cameras of different lenses in one problem (rcc_ba_set_camera_lenses) against the mixed-lens oracle of
tests/mixed_lens_oracle.py, and camera by camera against single-lens handles on the same data, with the tolerances of
test_gpu_equidistant.py.  A rig of 4 cameras (radtan, equidistant, radtan, equidistant), one of 3 (radtan, radtan,
equidistant) and a single-model problem of 2 cameras (radtan, equidistant)."""
import numpy as np
import pytest

import mixed_lens_oracle as MO
from helpers import max_block_rel, rel_fro
from robot_camera_calibration_b200 import _lib as L
from robot_camera_calibration_b200 import ceres_like
from robot_camera_calibration_b200.problem import BAProblem
from robot_camera_calibration_b200.scenes import make_scene

pytestmark = pytest.mark.gpu
TOL = 1e-9
NB_KEYS = ("Hee", "Hff", "W", "ge", "gf", "Hes", "Hfs", "Hss", "gs")

SCENES = {
    "rig4": dict(n_markers=16, n_views=16, visibility=0.6, n_cam=4, model="rig", seed=13,
                 lens=("radtan", "equidistant", "radtan", "equidistant")),
    "rig3": dict(n_markers=16, n_views=16, visibility=0.6, n_cam=3, model="rig", seed=17,
                 lens=("radtan", "radtan", "equidistant")),
    "single2": dict(n_markers=12, n_views=24, visibility=0.7, n_cam=2, seed=11, lens=("radtan", "equidistant")),
}


def _compact(s):
    """Drop views and markers that no block observes (turned views may see nothing)."""
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
    return _compact(make_scene(args.pop("n_markers"), args.pop("n_views"), args.pop("visibility"), **args))


def _fish(s):
    return np.array([lens == "equidistant" for lens in s.lens])


def _with_lens(s, lens):
    """The same data as a handle whose every camera has `lens`."""
    import copy
    t = copy.copy(s)
    t.lens = lens
    return t


@pytest.mark.parametrize("name", list(SCENES))
def test_evaluate_matches_mixed_oracle(name):
    s = _scene(name)
    p = MO.oracle_problem(s)
    r, Jb = MO.residuals(p), MO.jacobian_blocks_cs(p)
    with BAProblem.from_scene(s) as gp:
        assert gp.lens == s.lens
        out = gp.evaluate()
        res_only = gp.evaluate(want_jacobians=False)
    assert abs(out["cost"] - MO.cost(p)) <= TOL * MO.cost(p)
    assert abs(res_only["cost"] - MO.cost(p)) <= TOL * MO.cost(p)
    assert max_block_rel(out["residuals"], r) < TOL
    assert np.array_equal(res_only["residuals"], out["residuals"])
    for k in Jb:
        assert max_block_rel(out["jacobians"][k], Jb[k]) < TOL, k
    eq = _fish(s)[s.cam_idx]
    assert np.all(out["jacobians"]["dist"][eq][..., 4] == 0.0)        # the reserved slot of the equidistant cameras
    assert np.all(np.any(out["jacobians"]["dist"][~eq][..., 4] != 0.0, axis=1))   # k3 of the radtan cameras


@pytest.mark.parametrize("elim", ["views", "markers"])
@pytest.mark.parametrize("name", list(SCENES))
def test_each_camera_is_bitwise_its_single_lens_handle(name, elim):
    """K1 outputs and W of every observation, and the H_ss block of every camera, are those of a handle whose every
    camera has that camera's lens: the same kernels run on the same chunks."""
    s = _scene(name)
    sp = 15 if s.model == "rig" else 9
    outs, nbs = {}, {}
    for key, sc in (("mixed", s), ("radtan", _with_lens(s, "radtan")), ("equidistant", _with_lens(s, "equidistant"))):
        with BAProblem.from_scene(sc, eliminate=elim) as gp:
            outs[key] = gp.evaluate()
            gp.linearize()
            nbs[key] = gp.normal_blocks()
    for c, lens in enumerate(s.lens):
        m = s.cam_idx == c
        assert np.array_equal(outs["mixed"]["residuals"][m], outs[lens]["residuals"][m])
        for k in outs["mixed"]["jacobians"]:
            assert np.array_equal(outs["mixed"]["jacobians"][k][m], outs[lens]["jacobians"][k][m]), (c, k)
        assert np.array_equal(nbs["mixed"]["W"][m], nbs[lens]["W"][m])
        blk = slice(sp * c, sp * c + sp)
        assert np.array_equal(nbs["mixed"]["Hss"][blk, blk], nbs[lens]["Hss"][blk, blk])
        assert np.array_equal(nbs["mixed"]["gs"][blk], nbs[lens]["gs"][blk])


@pytest.mark.parametrize("elim", ["views", "markers"])
@pytest.mark.parametrize("name", list(SCENES))
def test_normal_equations_schur_and_step_match_oracle(name, elim):
    s = _scene(name)
    fish = _fish(s)
    s.dist[fish, 4] = 0.125           # the reserved slot: ignored by the projection, never stepped
    p = MO.oracle_problem(s)
    ob = MO.blocks(p, elim == "views")
    radius = 1e4
    S, b = MO.reduced(p, elim == "views", radius)
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
    delta, mcc_o, _, _ = MO.lm_step(p, radius)
    o_view, o_marker, o_shared, n = p.offsets()
    dv, dm, ds = (delta[o_view:o_marker].reshape(-1, 6), delta[o_marker:o_shared].reshape(-1, 6), delta[o_shared:])
    de, df = (dv, dm) if elim == "views" else (dm, dv)
    assert rel_fro(st["d_e"], de) < 1e-6 and rel_fro(st["d_f"], df) < 1e-6 and rel_fro(st["d_shared"], ds) < 1e-6
    assert abs(mcc - mcc_o) <= 1e-6 * abs(mcc_o)
    assert abs(step_norm - np.linalg.norm(delta)) <= 1e-6 * np.linalg.norm(delta)
    slot = st["d_shared"][p.shared_per_cam * np.arange(p.n_cam) + 8]
    assert np.all(slot[fish] == 0.0) and np.all(slot[~fish] != 0.0)
    assert np.all(dist[fish, 4] == 0.125)
    cand = p.copy()
    cand.unpack(p.pack() + delta)
    assert abs(c_new - MO.cost(cand)) <= 1e-6 * MO.cost(cand)


@pytest.mark.parametrize("name", list(SCENES))
def test_huber_and_jacobi_scaling(name):
    s = _scene(name)
    rng = np.random.default_rng(5)
    bad = rng.choice(s.n_blocks, 12, replace=False)
    s.pixels[bad] += rng.normal(0, 25.0, (12, 8))
    p = MO.oracle_problem(s)
    p.loss, p.loss_scale = "huber", 2.0
    ob = MO.blocks(p, True)
    S, b = MO.reduced(p, True, 1e4)
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
            c_new = gp.candidate_cost()
            steps[jac] = np.concatenate([st["d_e"].ravel(), st["d_f"].ravel(), st["d_shared"]])
        assert abs(cost - ob["cost"]) <= TOL * ob["cost"]
        for k in ("Hee", "Hff", "W", "ge", "gf", "Hes", "Hfs"):
            assert max_block_rel(nb[k], ob[k], floor=1e-6 * np.abs(ob[k]).max()) < TOL, k
        assert rel_fro(nb["Hss"], ob["Hss"]) < TOL and rel_fro(Sg, S) < TOL and rel_fro(bg, b) < TOL
    assert rel_fro(steps[True], steps[False]) < 1e-9
    delta, _, _, _ = MO.lm_step(p, 1e4)
    o_shared = p.offsets()[2]
    assert rel_fro(steps[False][-len(s.intr) * p.shared_per_cam:], delta[o_shared:]) < 1e-6
    cand = p.copy()
    cand.unpack(p.pack() + delta)
    assert abs(c_new - MO.cost(cand)) <= 1e-6 * MO.cost(cand)


def _sorted_by_view(s):
    """Observations in the E-sorted order of eliminate="views" (view, camera, marker): update_pixels then uploads in
    pieces."""
    o = np.lexsort((s.marker_idx, s.cam_idx, s.view_idx))
    s.view_idx, s.marker_idx, s.cam_idx, s.pixels = s.view_idx[o], s.marker_idx[o], s.cam_idx[o], s.pixels[o]
    return s


def _lenses_per_piece(s, n_pieces):
    """How many lenses the blocks of each upload piece of a view-sorted scene have.  Piece k ends at the first view
    that starts at or after k / n_pieces of the blocks (problem.cu: build_indices)."""
    starts = np.append(np.flatnonzero(np.diff(s.view_idx, prepend=-1)), s.n_blocks)
    ends = starts[np.searchsorted(starts, s.n_blocks * np.arange(1, n_pieces + 1) // n_pieces)]
    fish = _fish(s)[s.cam_idx]
    return np.array([len(np.unique(fish[a:b])) for a, b in zip(np.append(0, ends[:-1]), ends)])


@pytest.mark.parametrize("name", list(SCENES))
def test_piecewise_update_pixels_is_bitwise_set_observations(name):
    s = _sorted_by_view(_scene(name))
    pix2 = np.ascontiguousarray(s.pixels + np.random.default_rng(7).normal(0.0, 0.5, s.pixels.shape))
    # K2's E pass once per lens of each of the 4 pieces, the F pass once per lens, finalize
    want = _lenses_per_piece(s, 4).sum() + len(np.unique(_fish(s)[s.cam_idx])) + 1
    runs = []
    for _ in range(2):
        with BAProblem.from_scene(s, eliminate="views") as gp:
            gp.linearize()
            gp.update_pixels(pix2)
            n0 = gp.launch_count()
            c = gp.linearize()
            assert gp.launch_count() - n0 == want
            runs.append((c, gp.normal_blocks(), gp.evaluate(want_jacobians=False)["residuals"]))
    s.pixels = pix2
    with BAProblem.from_scene(s, eliminate="views") as gq:
        c_ref = gq.linearize()
        nb_ref = gq.normal_blocks()
    for c, nb, res in runs:
        assert c == c_ref
        for k in NB_KEYS:
            assert np.array_equal(nb[k], nb_ref[k]), k
        assert np.array_equal(res, runs[0][2])


def test_piecewise_update_pixels_in_pieces_at_size_is_bitwise_set_observations():
    """From LARGE_UPLOAD_BLOCKS (problem.h) on, linearize runs the E and the F pass of each upload piece as the piece
    lands: with mixed lenses each of them once per lens."""
    s = make_scene(5000, 2000, 0.25, n_cam=2, lens=("radtan", "equidistant"), blocked=True, chunk_views=250,
                   round_pixels=True, seed=65)
    assert s.n_blocks >= 4_000_000
    s = _sorted_by_view(s)
    pix = s.pixels + np.random.default_rng(10).integers(-2, 3, s.pixels.shape)
    with BAProblem.from_scene(s, eliminate="views") as gp:
        gp.linearize()
        gp.update_pixels(pix)
        n0 = gp.launch_count()
        cost = gp.linearize()
        assert gp.launch_count() - n0 == 2 * _lenses_per_piece(s, 8).sum() + 1    # E and F of each piece, finalize
        nb = gp.normal_blocks(want_W=False)
    s.pixels = pix
    with BAProblem.from_scene(s, eliminate="views") as gq:
        assert gq.linearize() == cost
        nq = gq.normal_blocks(want_W=False)
    for k in NB_KEYS:
        if k != "W":
            assert np.array_equal(nq[k], nb[k]), k


@pytest.mark.parametrize("elim", ["views", "markers"])
@pytest.mark.parametrize("name", list(SCENES))
def test_reserved_slot_covariance(name, elim):
    s = _scene(name)
    fish = _fish(s)
    p = MO.oracle_problem(s)
    H, _, _ = MO.normal_equations(p)
    free = np.nonzero(~p.const_mask())[0]
    C = np.zeros_like(H)
    C[np.ix_(free, free)] = np.linalg.inv(H[np.ix_(free, free)])
    o_shared = p.offsets()[2]
    ce, cr = int(np.nonzero(fish)[0][0]), int(np.nonzero(~fish)[0][0])
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        cov = gp.covariance()
        pair = gp.covariance_blocks([(("dist", ce), ("dist", ce)), (("dist", cr), ("dist", cr)),
                                     (("dist", ce), ("dist", cr))])
    slot = p.shared_per_cam * np.arange(p.n_cam) + 8
    assert np.all(cov["shared"][slot[fish], :] == 0.0) and np.all(cov["shared"][:, slot[fish]] == 0.0)
    assert np.all(np.diag(cov["shared"])[slot[~fish]] > 0.0)
    assert np.all(pair[0][4, :] == 0.0) and np.all(pair[0][:, 4] == 0.0) and np.all(pair[2][4, :] == 0.0)
    assert pair[1][4, 4] > 0.0
    Cs = C[o_shared:, o_shared:]
    assert rel_fro(cov["shared"], Cs) < 1e-6
    sp = p.shared_per_cam
    for c in range(p.n_cam):
        k = slice(4, 8) if fish[c] else slice(4, 9)
        blk = cov["shared"][sp * c:sp * c + 9, sp * c:sp * c + 9]
        assert rel_fro(blk[k, k], Cs[sp * c:sp * c + 9, sp * c:sp * c + 9][k, k]) < 1e-6


@pytest.mark.parametrize("name", ["rig4", "single2"])
def test_noise_free_mixed_rig_recovers_the_truth(name):
    s = _scene(name, pixel_noise=0.0)
    fish = _fish(s)
    with BAProblem.from_scene(s) as gp:
        summ = gp.solve(max_iterations=100, function_tolerance=1e-16, gradient_tolerance=1e-14,
                        parameter_tolerance=1e-15)
        views, markers = gp.get_view_poses(), gp.get_marker_poses()
        intr, dist = gp.get_intrinsics()
        ext = gp.get_rig_extrinsics() if s.model == "rig" else None
    assert summ["final_cost"] < 1e-14 * summ["initial_cost"]
    assert np.abs(views - s.truth["views"]).max() < 1e-6
    assert np.abs(markers - s.truth["markers"]).max() < 1e-6
    assert np.abs(intr - s.truth["intr"]).max() < 1e-4
    assert np.abs(dist[fish, :4] - s.truth["dist"][fish, :4]).max() < 1e-6
    assert np.abs(dist[~fish] - s.truth["dist"][~fish]).max() < 1e-6
    if ext is not None:
        assert np.abs(ext - s.truth["ext"]).max() < 1e-6


def _linearised(gp):
    """Linearise and evaluate: (cost, normal blocks, K1 outputs, launches these took)."""
    n0 = gp.launch_count()
    c = gp.linearize()
    return c, gp.normal_blocks(), gp.evaluate(), gp.launch_count() - n0


@pytest.mark.parametrize("lens", ["radtan", "equidistant"])
def test_uniform_lenses_are_a_single_lens_handle(lens):
    s = _scene("rig4")
    n = len(s.intr)
    with BAProblem.from_scene(_with_lens(s, lens)) as gp:
        ref = _linearised(gp)
        gp.set_lens(lens)
        again = _linearised(gp)                            # the poses stay expanded: one launch less
    codes = np.full(n, L.LENSES[lens], np.int32)
    with BAProblem.from_scene(_with_lens(s, "radtan")) as gp:
        gp._check(gp.lib.rcc_ba_set_camera_lenses(gp.h, codes.ctypes.data_as(L.c_int32_p)))
        uniform = _linearised(gp)
    with BAProblem.from_scene(s) as gp:                    # mixed, then every camera set to one lens
        mixed = _linearised(gp)
        gp.set_lens(lens)
        assert gp.lens == lens
        after = _linearised(gp)
    for got in (uniform, after):
        assert got[0] == ref[0]
        for k in NB_KEYS:
            assert np.array_equal(got[1][k], ref[1][k]), k
        assert np.array_equal(got[2]["residuals"], ref[2]["residuals"])
        for k in ref[2]["jacobians"]:
            assert np.array_equal(got[2]["jacobians"][k], ref[2]["jacobians"][k]), k
    assert uniform[3] == ref[3] and after[3] == again[3]
    # mixed: one more K2 launch per pass and one more K1 launch
    assert mixed[3] == ref[3] + 3


def test_set_camera_lenses_checks_every_camera_first():
    s = _scene("rig3")
    with BAProblem.from_scene(s) as gp:
        c0, nb0, _, _ = _linearised(gp)
        bad = np.array([0, 1, 7], np.int32)
        assert gp.lib.rcc_ba_set_camera_lenses(gp.h, bad.ctypes.data_as(L.c_int32_p)) == L.RCC_BAD_ARG
        assert gp.lib.rcc_ba_set_camera_lenses(gp.h, None) == L.RCC_BAD_ARG
        c1, nb1, _, _ = _linearised(gp)
        with pytest.raises(ValueError):
            gp.set_lens(("radtan", "equidistant"))          # one lens per camera
        with pytest.raises(ValueError):
            gp.set_lens(("radtan", "fisheye", "radtan"))
        assert gp.lens == s.lens
    assert c0 == c1 and all(np.array_equal(nb0[k], nb1[k]) for k in NB_KEYS)


def test_ceres_like_mixed_lenses_match_baproblem():
    s = _scene("rig3")
    cams = [(s.intr[c].copy(), s.dist[c].copy(), s.ext[c].copy()) for c in range(len(s.intr))]
    views = [v.copy() for v in s.views]
    markers = [m.copy() for m in s.markers]
    prob = ceres_like.Problem(eliminate="views")
    for b in range(s.n_blocks):
        c = s.cam_idx[b]
        cost = ceres_like.TagReprojectionCost(s.pixels[b], s.sizes[s.marker_idx[b]], rig=True, lens=s.lens[c])
        prob.AddResidualBlock(cost, None, cams[c][0], cams[c][1], views[s.view_idx[b]], markers[s.marker_idx[b]],
                              cams[c][2])
    prob.SetParameterBlockConstant(markers[0])
    prob.SetParameterBlockConstant(cams[0][2])
    cost, res, jac = prob.Evaluate()
    with BAProblem.from_scene(s, eliminate="views") as gp:
        out = gp.evaluate()
    # per block the same arithmetic; the parameter blocks are numbered in first-use order, so sums may differ in order
    assert abs(cost - out["cost"]) <= 1e-12 * out["cost"]
    assert np.array_equal(res, out["residuals"].reshape(-1))
    for k in out["jacobians"]:
        assert np.array_equal(jac[k], out["jacobians"][k]), k
    summ = ceres_like.Solve(ceres_like.SolverOptions(max_num_iterations=5), prob)
    with BAProblem.from_scene(s, eliminate="views") as gp:
        ref = gp.solve(max_iterations=5, initial_radius=1e4, max_radius=1e16, min_relative_decrease=1e-3,
                       function_tolerance=1e-6, gradient_tolerance=1e-10, parameter_tolerance=1e-8, min_diagonal=1e-6,
                       max_diagonal=1e32, jacobi_scaling=1)       # ceres_like.SolverOptions' defaults
        intr, dist = gp.get_intrinsics()
        v, m = gp.get_view_poses(), gp.get_marker_poses()
    assert abs(summ.final_cost - ref["final_cost"]) <= 1e-9 * ref["final_cost"]
    assert np.abs(np.stack([c[0] for c in cams]) - intr).max() < 1e-6
    assert np.abs(np.stack([c[1] for c in cams]) - dist).max() < 1e-9
    assert np.abs(np.stack(views) - v).max() < 1e-9 and np.abs(np.stack(markers) - m).max() < 1e-9
