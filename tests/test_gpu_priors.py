"""GPU: Gaussian priors on parameter blocks (rcc_ba_set_priors, BAProblem.set_priors, ceres_like.NormalPrior, the
--intrinsics-sigma command line) against the stacked (tag + prior) oracle of tests/prior_oracle.py.

Scenes: one camera, a 3-camera rig, a 4-camera rig that mixes radial-tangential and equidistant cameras, and a scene
whose eliminated blocks span several chunks.  Priors sit on every kind with full, non-diagonal A, including the
constant gauge marker and an equidistant camera's distortion (A's column 4 is nonzero there)."""
import json
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

import mixed_lens_oracle as MO
import prior_oracle as PO
from helpers import max_block_rel, rel_fro
from robot_camera_calibration_b200 import _lib as L
from robot_camera_calibration_b200 import ceres_like as CL
from robot_camera_calibration_b200 import io_yaml
from robot_camera_calibration_b200.problem import BAProblem, sqrt_information
from robot_camera_calibration_b200.scenes import make_scene
from test_gpu_mixed_lens import _scene as mixed_scene

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 1e-9          # normal equations and reduced system, per block
COST_TOL = 1e-12
STEP_TOL = 1e-6
SIGMA = {"view": [0.02] * 3 + [0.01] * 3, "marker": [0.02] * 3 + [0.01] * 3, "intr": [3.0, 3.0, 2.0, 2.0],
         "dist": [0.01] * 5, "ext": [0.01] * 3 + [0.002] * 3}


def _scene(name):
    if name == "single":
        return make_scene(12, 30, 0.7, seed=11)
    if name == "rig":
        return make_scene(16, 20, 0.6, n_cam=3, model="rig", seed=13)
    if name == "mixed_rig":
        return mixed_scene("rig4")
    if name == "multichunk":          # about 90 tags per view: two or more chunks per eliminated view
        return make_scene(100, 8, 0.9, seed=21)
    raise KeyError(name)


def make_priors(s, seed=3, kinds=None, every=2):
    """Full, non-diagonal priors on every `every`-th block of each kind (marker 0, the gauge, included), centred near
    the current value: {kind: (index, mean, A)}."""
    rng = np.random.default_rng(seed)
    count = {"view": len(s.views), "marker": len(s.markers), "intr": len(s.intr), "dist": len(s.intr),
             "ext": len(s.intr) if s.model == "rig" else 0}
    value = {"view": s.views, "marker": s.markers, "intr": s.intr, "dist": s.dist, "ext": s.ext}
    out = {}
    for kind in kinds or count:
        if count[kind] == 0:
            continue
        idx = np.arange(0, count[kind], every if kind in ("view", "marker") else 1)
        sig = np.asarray(SIGMA[kind])
        k = len(sig)
        mean = value[kind][idx] + rng.normal(0, 1, (len(idx), k)) * sig
        A = np.stack([(np.eye(k) + 0.3 * rng.normal(size=(k, k))) / sig[None, :] for _ in idx])
        out[kind] = (idx, mean, A)
    return out


def _with_priors(gp, priors):
    for kind, (idx, mean, A) in priors.items():
        gp.set_priors(kind, idx, mean, A)
    return gp


def _dense_step(st, elim_view):
    """The library's step in the dense layout [views | markers | shared]."""
    dv, dm = (st["d_e"], st["d_f"]) if elim_view else (st["d_f"], st["d_e"])
    return np.concatenate([dv.ravel(), dm.ravel(), st["d_shared"]])


def _canonical(s):
    """Views and markers renumbered in order of first use by the observation blocks: the order in which
    ceres_like.Problem numbers them, so that both front ends build the same handle."""
    for kind, idx, sizes in (("views", "view_idx", None), ("markers", "marker_idx", "sizes")):
        order = list(dict.fromkeys(getattr(s, idx).tolist()))
        remap = np.empty(len(order), np.int64)
        remap[order] = np.arange(len(order))
        setattr(s, kind, getattr(s, kind)[order])
        setattr(s, "const_" + kind, getattr(s, "const_" + kind)[order])
        if sizes:
            s.sizes = s.sizes[order]
        setattr(s, idx, remap[getattr(s, idx)].astype(np.int32))
    return s


def _split(p, delta, elim_view):
    o_view, o_marker, o_shared, _ = p.offsets()
    dv, dm = delta[o_view:o_marker].reshape(-1, 6), delta[o_marker:o_shared].reshape(-1, 6)
    return (dv, dm, delta[o_shared:]) if elim_view else (dm, dv, delta[o_shared:])


@pytest.mark.parametrize("elim", ["views", "markers"])
@pytest.mark.parametrize("name", ["single", "rig", "mixed_rig", "multichunk"])
def test_normal_equations_schur_and_step_match_oracle(name, elim):
    s = _scene(name)
    ev = elim == "views"
    fish = np.array([lens == "equidistant" for lens in ((s.lens,) * len(s.intr) if isinstance(s.lens, str) else s.lens)])
    s.dist[fish, 4] = 0.125
    pri = make_priors(s)
    p = MO.oracle_problem(s)
    ob = PO.blocks(p, pri, ev)
    radius = 1e4
    S, b = PO.reduced(p, pri, ev, radius)
    with BAProblem.from_scene(s, eliminate=elim) as plain:
        plain.linearize()
        nb0 = plain.normal_blocks()
    with _with_priors(BAProblem.from_scene(s, eliminate=elim), pri) as gp:
        cost = gp.linearize()
        nb = gp.normal_blocks()
        gp.schur(radius)
        Sg, bg = gp.reduced_system()
        mcc, step_norm, _ = gp.solve_step()
        st = gp.step()
        c_new = gp.candidate_cost()
        gp.accept_step()
        _, dist = gp.get_intrinsics()
    assert abs(cost - ob["cost"]) <= COST_TOL * ob["cost"]
    for k in ("Hee", "Hff", "ge", "gf"):
        assert max_block_rel(nb[k], ob[k], floor=1e-6 * np.abs(ob[k]).max()) < TOL, k
    assert rel_fro(nb["Hss"], ob["Hss"]) < TOL and rel_fro(nb["gs"], ob["gs"]) < TOL
    for k in ("W", "Hes", "Hfs"):           # the priors never touch the cross blocks
        assert np.array_equal(nb[k], nb0[k]), k
    assert rel_fro(Sg, S) < TOL and rel_fro(bg, b) < TOL
    delta, mcc_o, _, _ = PO.lm_step(p, pri, radius)
    de, df, ds = _split(p, delta, ev)
    assert rel_fro(st["d_e"], de) < STEP_TOL and rel_fro(st["d_f"], df) < STEP_TOL
    assert rel_fro(st["d_shared"], ds) < STEP_TOL
    assert abs(mcc - mcc_o) <= STEP_TOL * abs(mcc_o)
    # the constant gauge marker carries a prior: cost only, a zero step; so does the reserved slot
    assert np.all((st["d_f"] if ev else st["d_e"])[0] == 0.0)
    slot = st["d_shared"][p.shared_per_cam * np.arange(p.n_cam) + 8]
    assert np.all(slot[fish] == 0.0) and np.all(dist[fish, 4] == 0.125)
    cand = p.copy()
    cand.unpack(p.pack() + _dense_step(st, ev))
    assert abs(c_new - PO.cost(cand, pri)) <= COST_TOL * PO.cost(cand, pri)


@pytest.mark.parametrize("loss", [None, ("huber", 2.0), ("cauchy", 3.0)])
def test_every_reported_cost_includes_the_priors(loss):
    s = make_scene(12, 30, 0.7, seed=11)
    rng = np.random.default_rng(5)
    bad = rng.choice(s.n_blocks, 12, replace=False)
    s.pixels[bad] += rng.normal(0, 25.0, (12, 8))
    pri = make_priors(s, seed=7)
    p = MO.oracle_problem(s)
    if loss:
        p.loss, p.loss_scale = loss
    ref = PO.cost(p, pri)
    with _with_priors(BAProblem.from_scene(s, eliminate="views"), pri) as gp:
        if loss:
            gp.set_loss(*loss)
        costs = {"linearize": gp.linearize(), "evaluate": gp.evaluate()["cost"],
                 "evaluate_nojac": gp.evaluate(want_jacobians=False)["cost"],
                 "evaluate_device": gp.evaluate_device(want_jacobians=True, want_cost=True),
                 "evaluate_device_nojac": gp.evaluate_device(want_jacobians=False, want_cost=True)}
        out = gp.evaluate()
        assert out["residuals"].shape == (s.n_blocks, 8)           # tag blocks only
        gp.schur(1e4)
        gp.solve_step()
        st = gp.step()
        cand_cost = gp.candidate_cost()
        summ = gp.solve(max_iterations=5)
        views, markers = gp.get_view_poses(), gp.get_marker_poses()
        intr, dist = gp.get_intrinsics()
    for k, c in costs.items():
        assert abs(c - ref) <= COST_TOL * ref, (k, c, ref)
    assert abs(summ["initial_cost"] - ref) <= COST_TOL * ref
    cand = p.copy()
    cand.unpack(p.pack() + _dense_step(st, True))
    assert abs(cand_cost - PO.cost(cand, pri)) <= COST_TOL * PO.cost(cand, pri)
    fin = p.copy()
    fin.views, fin.markers, fin.intr, fin.dist = views, markers, intr, dist
    assert abs(summ["final_cost"] - PO.cost(fin, pri)) <= COST_TOL * summ["final_cost"]


@pytest.mark.parametrize("name", ["single", "rig"])
def test_jacobi_scaled_step_matches_oracle(name):
    s = _scene(name)
    pri = make_priors(s, seed=9)
    p = MO.oracle_problem(s)
    for jac in (False, True):
        with _with_priors(BAProblem.from_scene(s, eliminate="views"), pri) as gp:
            gp.set_lm_diagonal(1e-6, 1e32, jac)
            gp.linearize()
            gp.schur(1e2)
            Sg, bg = gp.reduced_system()
            gp.solve_step()
            st = gp.step()
        S, b = PO.reduced(p, pri, True, 1e2, jacobi=jac)
        assert rel_fro(Sg, S) < TOL and rel_fro(bg, b) < TOL
        de, df, ds = _split(p, PO.lm_step(p, pri, 1e2, jacobi=jac)[0], True)
        assert rel_fro(st["d_e"], de) < STEP_TOL and rel_fro(st["d_f"], df) < STEP_TOL
        assert rel_fro(st["d_shared"], ds) < STEP_TOL


OPTS = dict(max_iterations=100, function_tolerance=1e-15, gradient_tolerance=1e-14, parameter_tolerance=1e-15)


@pytest.mark.parametrize("name", ["single", "rig"])
def test_solve_reaches_the_least_squares_minimiser(name):
    s = _scene(name)
    pri = make_priors(s, seed=11)
    p = MO.oracle_problem(s)
    x = PO.minimise(p, pri)
    q = p.copy()
    q.unpack(x)
    with _with_priors(BAProblem.from_scene(s), pri) as gp:
        summ = gp.solve(**OPTS)
        views, markers = gp.get_view_poses(), gp.get_marker_poses()
        intr, dist = gp.get_intrinsics()
        ext = gp.get_rig_extrinsics() if s.model == "rig" else None
    assert summ["termination"] in (1, 2, 3)
    for a, r in ((views, q.views), (markers, q.markers)):
        assert np.abs(a[:, :3] - r[:, :3]).max() < 1e-6 and np.abs(a[:, 3:] - r[:, 3:]).max() < 1e-6
    if ext is not None:
        assert np.abs(ext - q.ext).max() < 1e-6
    assert np.abs(dist - q.dist).max() < 1e-6 and np.abs(intr - q.intr).max() < 1e-4   # pixels
    assert abs(summ["final_cost"] - PO.cost(q, pri)) <= 1e-9 * summ["final_cost"]


def test_tight_prior_pulls_block_to_its_mean():
    s = make_scene(12, 30, 0.7, seed=11)
    mu = s.views[5] + np.array([0.01, -0.02, 0.015, 0.03, -0.01, 0.02])
    with BAProblem.from_scene(s) as gp:
        gp.set_priors("view", [5], mu[None], 1e9 * np.eye(6)[None])
        gp.solve(**OPTS)
        v = gp.get_view_poses()
    assert np.abs(v[5] - mu).max() < 1e-7


def test_prior_on_a_constant_block_adds_cost_only():
    s = make_scene(12, 30, 0.7, seed=11)
    assert s.const_markers[0]
    mu = s.markers[0] + 0.05
    A = np.diag([10.0, 20.0, 30.0, 40.0, 50.0, 60.0])
    with BAProblem.from_scene(s, eliminate="views") as g0:
        c0 = g0.linearize()
        g0.schur(1e4)
        g0.solve_step()
        st0 = g0.step()
    with BAProblem.from_scene(s, eliminate="views") as gp:
        gp.set_priors("marker", [0], mu[None], A[None])
        c1 = gp.linearize()
        gp.schur(1e4)
        gp.solve_step()
        st = gp.step()
        summ = gp.solve(**OPTS)
        m = gp.get_marker_poses()
    prior = 0.5 * float(np.sum((A @ (s.markers[0] - mu)) ** 2))
    assert abs(c1 - (c0 + prior)) <= COST_TOL * c1
    assert np.all(st["d_f"][0] == 0.0) and np.array_equal(m[0], s.markers[0])
    # the step of every free block is the plain handle's: the prior adds to a masked block only
    assert np.array_equal(st["d_e"], st0["d_e"]) and np.array_equal(st["d_shared"], st0["d_shared"])
    assert summ["final_cost"] >= prior


def _no_gauge(name):
    s = _scene(name)
    s.const_markers[:] = False
    return s


@pytest.mark.parametrize("elim", ["views", "markers"])
@pytest.mark.parametrize("name", ["single", "rig"])
def test_covariance_with_a_prior_gauge(name, elim):
    s = _no_gauge(name)
    pri = {"marker": ([0], s.markers[:1], sqrt_information(np.diag([1e-4] * 3 + [1e-6] * 3))[None])}
    if s.model == "rig":
        pri["ext"] = ([0], s.ext[:1], sqrt_information(np.diag([1e-4] * 3 + [1e-6] * 3))[None])
    with BAProblem.from_scene(s, eliminate=elim) as g0:
        with pytest.raises(L.RccError) as e:
            g0.covariance()
        assert e.value.status == L.RCC_NOT_SPD
    p = MO.oracle_problem(s)
    C = PO.covariance(p, pri)
    o_view, o_marker, o_shared, n = p.offsets()
    with _with_priors(BAProblem.from_scene(s, eliminate=elim), pri) as gp:
        cov = gp.covariance()
        pairs = [(("view", 1), ("marker", 2)), (("marker", 0), ("intr", 0)), (("dist", 0), ("view", 3)),
                 (("view", 2), ("view", 2))]
        blocks = gp.covariance_blocks(pairs)
    blk = lambda off, i: C[off + 6 * i:off + 6 * i + 6, off + 6 * i:off + 6 * i + 6]
    ref_v = np.stack([blk(o_view, i) for i in range(len(s.views))])
    ref_m = np.stack([blk(o_marker, i) for i in range(len(s.markers))])
    assert max_block_rel(cov["views"], ref_v, floor=1e-6 * np.abs(ref_v).max()) < STEP_TOL
    assert max_block_rel(cov["markers"], ref_m, floor=1e-6 * np.abs(ref_m).max()) < STEP_TOL
    assert rel_fro(cov["shared"], C[o_shared:, o_shared:]) < STEP_TOL
    for ((ka, ia), (kb, ib)), got in zip(pairs, blocks):
        ca, cb = PO.columns(p, ka, ia), PO.columns(p, kb, ib)
        # relative to the two marginal blocks: the prior pins marker 0 so tightly that its cross terms are ~1e-13
        scale = np.sqrt(np.linalg.norm(C[np.ix_(ca, ca)]) * np.linalg.norm(C[np.ix_(cb, cb)]))
        assert np.linalg.norm(got - C[np.ix_(ca, cb)]) < STEP_TOL * scale, (ka, ia, kb, ib)


def _run(gp, solve=True):
    n0 = gp.launch_count()
    gp.linearize()
    nb = gp.normal_blocks()
    gp.schur(1e4)
    S, b = gp.reduced_system()
    gp.solve_step()
    st = gp.step()
    c = gp.candidate_cost()
    ev = gp.evaluate()["cost"]
    out = dict(nb=nb, S=S, b=b, st=st, c=c, ev=ev, launches=gp.launch_count() - n0)
    if solve:
        n1 = gp.launch_count()
        summ = gp.solve(max_iterations=10)
        out["summ"] = [summ[k] for k in ("iterations", "accepted", "termination", "initial_cost", "final_cost")]
        out["solve_launches"] = gp.launch_count() - n1
        out["x"] = (gp.get_view_poses(), gp.get_marker_poses(), *gp.get_intrinsics())
    return out


def _bitwise(a, b):
    if isinstance(a, dict):
        return a.keys() == b.keys() and all(_bitwise(a[k], b[k]) for k in a)
    if isinstance(a, (tuple, list)):
        return len(a) == len(b) and all(_bitwise(x, y) for x, y in zip(a, b))
    if a is None:
        return b is None
    return np.array_equal(np.asarray(a), np.asarray(b))


@pytest.mark.parametrize("name", ["single", "mixed_rig"])
def test_nothing_changes_without_priors(name):
    s = _scene(name)
    pri = make_priors(s)
    with BAProblem.from_scene(s, eliminate="views") as gp:
        plain = _run(gp)
    with BAProblem.from_scene(s, eliminate="views") as gp:
        _with_priors(gp, pri)
        with_p = _run(gp, solve=False)
        gp.set_view_poses(s.views)
        gp.set_marker_poses(s.markers)
        gp.set_intrinsics(s.intr, s.dist)
        if s.model == "rig":
            gp.set_rig_extrinsics(s.ext)
        gp.clear_priors()
        cleared = _run(gp)
    assert _bitwise(plain, cleared)
    assert with_p["launches"] == plain["launches"] + 3      # one prior launch in linearize, candidate cost, evaluate


def test_set_priors_rejects_bad_arguments_and_changes_nothing():
    s = make_scene(12, 30, 0.7, seed=11)
    pri = make_priors(s, kinds=["view", "intr"])
    lib = L.load()
    with _with_priors(BAProblem.from_scene(s, eliminate="views"), pri) as gp:
        before = _run(gp, solve=False)
        idx = np.array([0, 1], dtype=np.int32)
        mean = np.zeros((2, 6))
        A = np.stack([np.eye(6)] * 2)
        dp = lambda a: a.ctypes.data_as(L.c_double_p)
        ip = lambda a: a.ctypes.data_as(L.c_int32_p)
        bad = [
            (None, L.BLOCK_VIEW, 2, ip(idx), dp(mean), dp(A)),
            (gp.h, 7, 2, ip(idx), dp(mean), dp(A)),
            (gp.h, -1, 2, ip(idx), dp(mean), dp(A)),
            (gp.h, L.BLOCK_EXT, 1, ip(idx), dp(mean), dp(A)),                 # single model
            (gp.h, L.BLOCK_VIEW, -1, ip(idx), dp(mean), dp(A)),
            (gp.h, L.BLOCK_VIEW, 2, None, dp(mean), dp(A)),
            (gp.h, L.BLOCK_VIEW, 2, ip(idx), None, dp(A)),
            (gp.h, L.BLOCK_VIEW, 2, ip(idx), dp(mean), None),
            (gp.h, L.BLOCK_VIEW, 2, ip(np.array([0, len(s.views)], np.int32)), dp(mean), dp(A)),
            (gp.h, L.BLOCK_VIEW, 2, ip(np.array([-1, 0], np.int32)), dp(mean), dp(A)),
            (gp.h, L.BLOCK_VIEW, 2, ip(np.array([3, 3], np.int32)), dp(mean), dp(A)),
            (gp.h, L.BLOCK_VIEW, 2, ip(idx), dp(np.array([[0.0] * 5 + [np.nan]] * 2)), dp(A)),
            (gp.h, L.BLOCK_VIEW, 2, ip(idx), dp(mean), dp(np.stack([np.eye(6), np.eye(6) * np.inf]))),
            (gp.h, L.BLOCK_MARKER, len(s.markers) + 1, ip(np.arange(len(s.markers) + 1, dtype=np.int32)),
             dp(np.zeros((len(s.markers) + 1, 6))), dp(np.zeros((len(s.markers) + 1, 6, 6)))),
        ]
        for args in bad:
            assert lib.rcc_ba_set_priors(*args) == L.RCC_BAD_ARG
        gp.set_view_poses(s.views)          # expand the poses again, as the first run did
        after = _run(gp, solve=False)
        with pytest.raises(ValueError):
            gp.set_priors("intr", [0], np.zeros((1, 4)), np.zeros((1, 5, 5)))    # wrong A shape, refused in Python
    assert _bitwise(before, after)


def _ceres(s, priors, stacked=False, rect=False):
    """ceres_like problem of scene s with the priors as NormalPrior blocks."""
    views = [np.array(v) for v in s.views]
    markers = [np.array(m) for m in s.markers]
    intr = [np.array(i) for i in s.intr]
    dist = [np.array(d) for d in s.dist]
    pb = CL.Problem(eliminate="views")
    for b in range(s.n_blocks):
        c = s.cam_idx[b]
        pb.AddResidualBlock(CL.TagReprojectionCost(s.pixels[b], s.sizes[s.marker_idx[b]]), None, intr[c], dist[c],
                            views[s.view_idx[b]], markers[s.marker_idx[b]])
    pb.SetParameterBlockConstant(markers[0])
    blocks = {"view": views, "marker": markers, "intr": intr, "dist": dist}
    for kind, (idx, mean, A) in priors.items():
        for i, mu, a in zip(idx, mean, A):
            pb.AddResidualBlock(CL.NormalPrior(a, mu), None, blocks[kind][i])
    return pb, blocks


def test_ceres_like_normal_prior_is_bitwise_set_priors():
    s = _canonical(make_scene(10, 16, 0.8, seed=31))
    pri = make_priors(s, seed=13)
    pb, blocks = _ceres(s, pri)
    n_prior = sum(len(v[0]) for v in pri.values())
    assert pb.NumResidualBlocks() == s.n_blocks + n_prior
    assert pb.NumResiduals() == 8 * s.n_blocks + sum(len(v[0]) * v[2].shape[1] for v in pri.values())
    cost, res, _ = pb.Evaluate()
    with _with_priors(BAProblem.from_scene(s, eliminate="views"), pri) as gp:
        ref_cost = gp.evaluate()["cost"]
        summ = gp.solve()
        views, markers = gp.get_view_poses(), gp.get_marker_poses()
        intr, dist = gp.get_intrinsics()
    assert abs(cost - ref_cost) <= COST_TOL * ref_cost and abs(0.5 * res @ res - ref_cost) <= 1e-10 * ref_cost
    with pytest.raises(NotImplementedError):
        pb.AddResidualBlock(CL.NormalPrior(np.eye(6), np.zeros(6)), CL.HuberLoss(1.0), blocks["view"][0])
    cs = CL.Solve(CL.SolverOptions(), pb)
    assert cs.final_cost == summ["final_cost"]
    assert np.array_equal(np.stack(blocks["view"]), views) and np.array_equal(np.stack(blocks["marker"]), markers)
    assert np.array_equal(np.stack(blocks["intr"]), intr) and np.array_equal(np.stack(blocks["dist"]), dist)


def test_ceres_like_rectangular_and_stacked_priors_are_their_qr_form():
    s = _canonical(make_scene(10, 16, 0.8, seed=31))
    rng = np.random.default_rng(17)
    A1 = rng.normal(size=(9, 6)) * 50                    # m > k
    A2, A3 = rng.normal(size=(6, 6)) * 30, rng.normal(size=(4, 6)) * 30   # two priors, one with m < k, same mean
    mu = s.views[2] + 0.01
    pb, blocks = _ceres(s, {})
    pb.AddResidualBlock(CL.NormalPrior(A1, s.views[1]), None, blocks["view"][1])
    pb.AddResidualBlock(CL.NormalPrior(A2, mu), None, blocks["view"][2])
    pb.AddResidualBlock(CL.NormalPrior(A3, mu), None, blocks["view"][2])
    cost, res, _ = pb.Evaluate()
    R1 = np.linalg.qr(A1, mode="r")
    R23 = np.linalg.qr(np.vstack([A2, A3]), mode="r")
    with BAProblem.from_scene(s, eliminate="views") as gp:
        gp.set_priors("view", [1, 2], np.stack([s.views[1], mu]), np.stack([R1, R23]))
        ref_cost = gp.evaluate()["cost"]
        gp.solve()
        views = gp.get_view_poses()
    assert abs(cost - ref_cost) <= 1e-10 * ref_cost and abs(0.5 * res @ res - cost) <= 1e-10 * cost
    CL.Solve(CL.SolverOptions(), pb)
    assert np.array_equal(np.stack(blocks["view"]), views)


def _cli(tmp, name, s, *flags):
    d = os.path.join(tmp, name)
    shutil.rmtree(d, ignore_errors=True)
    io_yaml.write_dataset(d, s)
    from robot_camera_calibration_b200.__main__ import main
    assert main([d, "--precision", "repr", "--max-iterations", "100", "--function-tolerance", "1e-15",
                 "--gradient-tolerance", "1e-14", "--parameter-tolerance", "1e-15", *flags]) == 0
    r, _, _ = io_yaml.read_dataset(d)
    cam = os.path.join(d, "camera_refined.yaml")
    return r, (io_yaml.read_camera(cam)[0] if os.path.exists(cam) else None), io_yaml.read_camera(
        os.path.join(d, "camera.yaml"))[0]


def test_command_line_intrinsics_sigma(tmp_path, capsys):
    s = make_scene(10, 25, 0.8, seed=8, pixel_noise=0.0, perturb=(0.01, 0.01, 0.0))
    tmp = str(tmp_path)
    fixed, _, _ = _cli(tmp, "fixed", s, "--fix-intrinsics")
    tight, cam_t, yaml_intr = _cli(tmp, "tight", s, "--intrinsics-sigma", "1e-7", "1e-7", "1e-10")
    free, cam_f, _ = _cli(tmp, "free", s)
    loose, cam_l, _ = _cli(tmp, "loose", s, "--intrinsics-sigma", "1e8", "1e8", "1e8")
    for a, b, tol in ((tight, fixed, 1e-9), (loose, free, 1e-6)):
        assert np.abs(a.views - b.views).max() < tol and np.abs(a.markers - b.markers).max() < tol
    assert cam_t is not None and np.abs(cam_t - yaml_intr).max() < 1e-9 * np.abs(yaml_intr).max()
    assert np.abs(cam_l - cam_f).max() < 1e-6 * np.abs(cam_f).max()
    capsys.readouterr()


def test_two_gpu_priors_match_single_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", "29613", os.path.join(ROOT, "tools", "prior_multi_gpu_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    assert json.loads(line)["ok"]
