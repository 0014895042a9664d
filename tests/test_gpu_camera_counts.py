"""Every camera count the library accepts, against the oracle: 1-8 rig cameras and 1-13 single-model cameras.

The shared parameters (fx fy cx cy k1 k2 p1 p2 k3 per camera, plus body_T_cam in the rig) form the dense border of the
reduced system, 6 n_bb columns wide with n_bb = ceil((n_shared + 1) / 6).  Several kernels change their path with that
width or with the camera count:
  * schur_border_kernel runs ceil(cols / 32) passes over the border columns (1-4), with 32 / min(32, cols) pair slots
    per warp;
  * finalize_fused_kernel reduces the shared blocks in fin_slices = max(64, ceil(2 SMs / n_cam)) CTAs per camera;
  * backsub_kernel, the schur_prep border fill and schur_shared stride over the border 32 columns per lane round;
  * finalize_side_body splits a block's chunk list into per-camera segments.
test_gpu_parity.py and test_gpu_full_size.py run 1 and 2 single-model cameras and 2, 3 and 4 rig cameras; the counts
here reach every other path: 3 and 4 border passes, the exact 96-column edge, the fin_slices floor, 3 and 4 border
strides per lane, up to 13 per-camera segments, and a camera without any observation.

Tolerances are the suite's: 1e-9 relative per block for K1, K2 and K3, 1e-6 for the LM step and the covariance (the
conditioning allowance of test_gpu_parity.py and test_gpu_covariance.py), 1e-6 rad / 1e-6 m / 1e-4 px / 1e-6 for
converged parameters.
"""
import ctypes
import functools

import numpy as np
import pytest
import torch

import ba_oracle as O
from helpers import SparseSchurOracle, max_block_rel, oracle_blocks, oracle_blocks_sparse, oracle_reduced, rel_fro, to_oracle
from robot_camera_calibration_b200 import _lib as L
from robot_camera_calibration_b200.problem import BAProblem
from robot_camera_calibration_b200.scenes import make_scene
from test_gpu_covariance import compare, oracle_covariance
from test_gpu_covariance_blocks import block_errors, dense_covariance

TOL = 1e-9
STEP_TOL = 1e-6
SP = {"single": 9, "rig": 15}
MAX_CAM = {"single": 13, "rig": 8}
CHUNK = 64                      # observation blocks per chunk: one (eliminated block, camera) run of at most 64

# border columns 6 n_bb per camera count
COLS = {"single": {1: 12, 2: 24, 3: 30, 4: 42, 5: 48, 6: 60, 7: 66, 8: 78, 9: 84, 10: 96, 11: 102, 12: 114, 13: 120},
        "rig": {1: 18, 2: 36, 3: 48, 4: 66, 5: 78, 6: 96, 7: 108, 8: 126}}

# camera counts the other GPU tests run (test_gpu_parity.py, test_gpu_edge_cases.py, test_k2_groups.py,
# test_gpu_full_size.py), and the ones this file adds
COVERED_ELSEWHERE = {"single": (1, 2), "rig": (2, 3, 4)}
COUNTS = {"single": (3, 4, 5, 10, 11, 13), "rig": (1, 5, 6, 7, 8)}


def border_passes(cols):
    return -(-cols // 32)


def pair_slots(cols):
    return 32 // min(32, cols)


def fin_slices(n_sm, n_cam):
    """First-stage CTAs per camera of the shared-parameter finalize (kernels.h)."""
    return max(64, -(-2 * n_sm // n_cam))


def _all_counts():
    return [(m, n) for m in ("single", "rig") for n in COUNTS[m] + COVERED_ELSEWHERE[m]]


assert all(cols == 6 * -(-(n * SP[m] + 1) // 6) for m in COLS for n, cols in COLS[m].items())
assert {border_passes(COLS[m][n]) for m, n in _all_counts()} == {1, 2, 3, 4}
assert {pair_slots(COLS[m][n]) for m, n in _all_counts()} == {1, 2}
assert any(COLS[m][n] == 96 for m, n in _all_counts())          # the last 3-pass width, exactly full
assert any(n * SP[m] >= 96 for m, n in _all_counts())           # 4 border strides per lane in backsub_kernel


def _device_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


if torch.cuda.is_available():                                   # the floor of fin_slices depends on the SM count
    assert any(fin_slices(_device_sms(), n) == 64 for _, n in _all_counts())
    assert any(fin_slices(_device_sms(), n) > 64 for _, n in _all_counts())


# ---------------------------------------------------------------------------------------------------------------
# scenes
# ---------------------------------------------------------------------------------------------------------------
def _select(s, keep):
    s.view_idx, s.marker_idx, s.cam_idx, s.pixels = s.view_idx[keep], s.marker_idx[keep], s.cam_idx[keep], s.pixels[keep]
    return s


def _keep_views(s, views):
    new = np.full(len(s.views), -1)
    new[views] = np.arange(len(views))
    keep = new[s.view_idx] >= 0
    s.views, s.const_views = s.views[views], s.const_views[views]
    _select(s, keep)
    s.view_idx = new[s.view_idx].astype(np.int32)
    return s


# name -> (model, n_cam, one camera per view).  "single" with one camera per view: view v belongs to camera v mod n_cam,
# as test_gpu_parity's single_2cam; "single5_all_views" keeps the generator's raw output, every view seen through
# every camera, so that an eliminated view's chunk list spans several cameras.  Rig body poses see through every camera.
CASES = {f"single{n}": ("single", n, True) for n in COUNTS["single"]}
CASES["single5_all_views"] = ("single", 5, False)
CASES.update({f"rig{n}": ("rig", n, False) for n in COUNTS["rig"]})


def make_case(name):
    model, n, split = CASES[name]
    if model == "rig":
        return make_scene(16, 20, 0.6, n_cam=n, model="rig", seed=200 + n)
    if not split:
        return make_scene(16, 20, 0.7, n_cam=n, seed=125)
    s = make_scene(16, 8 * n, 0.7, n_cam=n, seed=100 + n)
    return _select(s, s.cam_idx == (np.arange(len(s.views)) % n)[s.view_idx])


@functools.lru_cache(maxsize=None)
def _case(name):
    s = make_case(name)
    return s, to_oracle(s)


@functools.lru_cache(maxsize=None)
def _blocks(name, elim_view):
    return oracle_blocks(_case(name)[1], elim_view)


def check_dims(gp, model, n_cam):
    """The handle runs the border width this case is listed for."""
    d = gp.dims
    assert d.n_shared == n_cam * SP[model]
    assert d.ld_reduced - 6 * d.n_f == COLS[model][n_cam]


def free_condition(p):
    H, _, _ = O.normal_equations(p)
    free = ~p.const_mask()
    return np.linalg.cond(H[np.ix_(free, free)])


@pytest.mark.parametrize("name", list(CASES))
def test_scenes_determine_every_camera(name):
    """Every camera has enough observations for its 9 (or 15) parameters, and the free J^T J is conditioned like the
    scenes the covariance tests use."""
    s, p = _case(name)
    model, n, _ = CASES[name]
    per_cam = np.bincount(s.cam_idx, minlength=n)
    assert per_cam.min() >= 40, per_cam
    assert free_condition(p) <= 1e11


# ---------------------------------------------------------------------------------------------------------------
# K1, K2, K3 and the step at every count, both elimination directions
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("elim", ["views", "markers"])
@pytest.mark.parametrize("name", list(CASES))
def test_evaluate_matches_oracle(name, elim):
    s, p = _case(name)
    model, n, _ = CASES[name]
    r, Jb = O.residuals(p), O.jacobian_blocks_cs(p)
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        check_dims(gp, model, n)
        out = gp.evaluate()
    err = {k: max_block_rel(out["jacobians"][k], Jb[k]) for k in Jb}
    err["residuals"] = max_block_rel(out["residuals"], r)
    print(f"{name}/{elim}: K1 largest block error {max(err.values()):.1e}")
    assert abs(out["cost"] - O.cost(p)) <= TOL * O.cost(p)
    assert set(out["jacobians"]) == set(Jb)
    assert max(err.values()) < TOL, err


def off_diagonal_camera_blocks(Hss, sp):
    n = len(Hss) // sp
    mask = np.kron(1 - np.eye(n), np.ones((sp, sp))).astype(bool)
    return Hss[mask]


@pytest.mark.gpu
@pytest.mark.parametrize("elim", ["views", "markers"])
@pytest.mark.parametrize("name", list(CASES))
def test_normal_blocks_match_oracle(name, elim):
    s, p = _case(name)
    model, n, _ = CASES[name]
    ob = _blocks(name, elim == "views")
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        check_dims(gp, model, n)
        cost = gp.linearize()
        nb = gp.normal_blocks()
    err = {k: max_block_rel(nb[k], ob[k], floor=1e-6 * np.abs(ob[k]).max())
           for k in ("Hee", "ge", "Hes", "Hff", "gf", "Hfs", "W")}
    err.update(Hss=rel_fro(nb["Hss"], ob["Hss"]), gs=rel_fro(nb["gs"], ob["gs"]))
    print(f"{name}/{elim}: normal blocks largest error {max(err.values()):.1e}")
    assert abs(cost - ob["cost"]) <= TOL * ob["cost"]
    assert max(err.values()) < TOL, err
    assert np.all(off_diagonal_camera_blocks(nb["Hss"], SP[model]) == 0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("elim", ["views", "markers"])
@pytest.mark.parametrize("name", list(CASES))
def test_reduced_system_matches_oracle(name, elim):
    """S and b, region by region: kept x kept, the border strip (kept x shared), and the shared corner, which carries
    the cross-camera terms of schur_shared."""
    s, p = _case(name)
    model, n, _ = CASES[name]
    S, b, *_ = oracle_reduced(p, elim == "views", 1e4)
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        check_dims(gp, model, n)
        gp.linearize()
        gp.schur(1e4)
        Sg, bg = gp.reduced_system()
        k = 6 * gp.dims.n_f
    err = {"S": rel_fro(Sg, S), "b": rel_fro(bg, b), "kept": rel_fro(Sg[:k, :k], S[:k, :k]),
           "border": rel_fro(Sg[:k, k:], S[:k, k:]), "corner": rel_fro(Sg[k:, k:], S[k:, k:]),
           "b_kept": rel_fro(bg[:k], b[:k]), "b_shared": rel_fro(bg[k:], b[k:])}
    print(f"{name}/{elim}: reduced system largest error {max(err.values()):.1e}")
    assert max(err.values()) < TOL, err


def check_step(gp, p, elim, radius):
    mcc, step_norm, _ = gp.solve_step()
    st = gp.step()
    c_new = gp.candidate_cost()
    delta, mcc_o, _, _ = O.lm_step(p, radius)
    o_view, o_marker, o_shared, _ = p.offsets()
    dv = delta[o_view:o_marker].reshape(-1, 6)
    dm = delta[o_marker:o_shared].reshape(-1, 6)
    de, df = (dv, dm) if elim == "views" else (dm, dv)
    print(f"step error d_e {rel_fro(st['d_e'], de):.1e} d_f {rel_fro(st['d_f'], df):.1e} "
          f"d_shared {rel_fro(st['d_shared'], delta[o_shared:]):.1e}")
    assert rel_fro(st["d_e"], de) < STEP_TOL
    assert rel_fro(st["d_f"], df) < STEP_TOL
    assert rel_fro(st["d_shared"], delta[o_shared:]) < STEP_TOL
    assert abs(mcc - mcc_o) <= STEP_TOL * abs(mcc_o)
    assert abs(step_norm - np.linalg.norm(delta)) <= STEP_TOL * np.linalg.norm(delta)
    cand = p.copy()
    cand.unpack(p.pack() + delta)
    assert abs(c_new - O.cost(cand)) <= STEP_TOL * O.cost(cand)
    return st


@pytest.mark.gpu
@pytest.mark.parametrize("elim", ["views", "markers"])
@pytest.mark.parametrize("name", list(CASES))
def test_step_matches_oracle(name, elim):
    s, p = _case(name)
    model, n, _ = CASES[name]
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        check_dims(gp, model, n)
        gp.linearize()
        gp.schur(1e4)
        check_step(gp, p, elim, 1e4)


# ---------------------------------------------------------------------------------------------------------------
# every slice of the shared-parameter finalize holds chunks
# ---------------------------------------------------------------------------------------------------------------
def every_camera_scene(model, n_cam):
    """128 views (body poses) that each see between 1 and 64 tags through every camera: with the views eliminated,
    every camera has exactly 128 E-pass chunks, so each of 64 finalize slices sums two of them."""
    if model == "rig":
        s = make_scene(60, 200, 0.5, n_cam=n_cam, model="rig", seed=302)
    else:
        s = make_scene(40, 200, 0.7, n_cam=n_cam, seed=301)
    per = np.zeros((len(s.views), n_cam), int)
    np.add.at(per, (s.view_idx, s.cam_idx), 1)
    ok = np.nonzero((per >= 1).all(1) & (per <= CHUNK).all(1))[0]
    assert len(ok) >= 128
    return _keep_views(s, ok[:128])


def e_chunks_per_camera(s, n_cam):
    """E-pass chunks of each camera with the views eliminated: ceil(run / 64) per (view, camera) run."""
    per = np.zeros((len(s.views), n_cam), int)
    np.add.at(per, (s.view_idx, s.cam_idx), 1)
    return (-(-per // CHUNK)).sum(0)


@pytest.mark.gpu
@pytest.mark.parametrize("model,n_cam", [("single", 11), ("rig", 8)])
def test_every_finalize_slice_holds_chunks(model, n_cam):
    s = every_camera_scene(model, n_cam)
    n = e_chunks_per_camera(s, n_cam)
    S = fin_slices(_device_sms(), n_cam)
    per = -(-n // S)
    assert np.all((S - 1) * per < n), (S, n)              # the last slice of every camera sums real partials
    p = to_oracle(s)
    radius = 1e4
    ob = oracle_blocks_sparse(p, True)
    so = SparseSchurOracle(p, ob, True, radius)
    with BAProblem.from_scene(s, eliminate="views") as gp:
        check_dims(gp, model, n_cam)
        n_f, ns = gp.dims.n_f, gp.dims.n_shared
        cost = gp.linearize()
        nb = gp.normal_blocks()
        assert abs(cost - ob["cost"]) <= TOL * ob["cost"]
        assert rel_fro(nb["Hss"], ob["Hss"]) < TOL and rel_fro(nb["gs"], ob["gs"]) < TOL
        for k in ("Hes", "Hfs"):
            assert max_block_rel(nb[k], ob[k], floor=1e-6 * np.abs(ob[k]).max()) < TOL, k
        gp.schur(radius)
        sample = sorted({0, n_f - 1, *np.random.default_rng(n_cam).choice(n_f, 10).tolist()})
        for f in sample:
            want = so.border(f)
            got = gp.reduced_block(6 * f, 6, 6 * n_f, ns + 1)
            assert np.linalg.norm(got - want) <= TOL * np.linalg.norm(want), f
        want = so.corner()
        got = gp.reduced_block(6 * n_f, ns, 6 * n_f, ns + 1)
        assert np.linalg.norm(got - want) <= TOL * np.linalg.norm(want)
        # the per-camera completion counters are back at zero after each launch: the same sums again
        for _ in range(2):
            assert gp.linearize() == cost
            again = gp.normal_blocks()
            for k in nb:
                assert np.array_equal(again[k], nb[k]), k


# ---------------------------------------------------------------------------------------------------------------
# robust loss, covariance and the converged solve at the largest counts
# ---------------------------------------------------------------------------------------------------------------
MAX_CASES = ["rig8", "single13"]


@pytest.mark.gpu
@pytest.mark.parametrize("loss,scale", [("huber", 2.0), ("cauchy", 3.0)])
@pytest.mark.parametrize("name", MAX_CASES)
def test_robust_loss_matches_oracle(name, loss, scale):
    s = make_case(name)
    rng = np.random.default_rng(5)
    bad = rng.choice(s.n_blocks, 12, replace=False)
    s.pixels[bad] += rng.normal(0, 25.0, (12, 8))            # gross outliers
    p = to_oracle(s)
    p.loss, p.loss_scale = loss, scale
    ob = oracle_blocks(p, True)
    S, b, *_ = oracle_reduced(p, True, 1e4)
    with BAProblem.from_scene(s, eliminate="views") as gp:
        gp.set_loss(loss, scale)
        out = gp.evaluate(want_jacobians=False)
        cost = gp.linearize()
        nb = gp.normal_blocks()
        gp.schur(1e4)
        Sg, bg = gp.reduced_system()
    assert abs(out["cost"] - ob["cost"]) <= TOL * ob["cost"]
    assert abs(cost - ob["cost"]) <= TOL * ob["cost"]
    for k in ("Hee", "Hff", "W", "ge", "gf", "Hes", "Hfs"):
        assert max_block_rel(nb[k], ob[k], floor=1e-6 * np.abs(ob[k]).max()) < TOL, k
    assert rel_fro(nb["Hss"], ob["Hss"]) < TOL and rel_fro(nb["gs"], ob["gs"]) < TOL
    assert rel_fro(Sg, S) < TOL and rel_fro(bg, b) < TOL


def shared_block_errors(got, ref, sp):
    """Relative error of every (camera, camera) block of cov_shared, floored by the scale of its diagonal blocks."""
    n = len(ref) // sp
    blk = lambda A, a, b: A[sp * a:sp * a + sp, sp * b:sp * b + sp]
    err = np.zeros((n, n))
    for a in range(n):
        for b in range(n):
            scale = np.sqrt(np.linalg.norm(blk(ref, a, a)) * np.linalg.norm(blk(ref, b, b)))
            err[a, b] = np.linalg.norm(blk(got, a, b) - blk(ref, a, b)) / max(np.linalg.norm(blk(ref, a, b)), 1e-6 * scale)
    return err


@pytest.mark.gpu
@pytest.mark.parametrize("elim", ["views", "markers"])
@pytest.mark.parametrize("name", MAX_CASES)
def test_covariance_matches_dense_inverse(name, elim):
    s, p = _case(name)
    model, n, _ = CASES[name]
    ref = oracle_covariance(p)
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        check_dims(gp, model, n)
        cov = gp.covariance()
    assert cov["shared"].shape == (n * SP[model],) * 2
    err = compare(cov, *ref)
    err["shared_blocks"] = shared_block_errors(cov["shared"], ref[2], SP[model]).max()
    print(f"{name}/{elim}: covariance largest block error {max(err.values()):.1e}")
    assert max(err.values()) < STEP_TOL, err


@pytest.mark.gpu
@pytest.mark.parametrize("name", MAX_CASES)
def test_covariance_blocks_for_every_camera(name):
    s, _ = _case(name)
    model, n, _ = CASES[name]
    nv, nm = len(s.views), len(s.markers)
    pairs = [(("intr", c), ("dist", c2)) for c in range(n) for c2 in range(n)]
    pairs += [(("intr", c), ("marker", m)) for c in range(n) for m in (0, 1, nm - 1)]
    if model == "rig":
        pairs += [(("ext", c), ("view", v)) for c in range(n) for v in (0, nv - 1)]
    C, cols = dense_covariance(s)
    with BAProblem.from_scene(s, eliminate="views") as gp:
        got = gp.covariance_blocks(pairs)
    const = {("marker", 0)} | ({("ext", 0)} if model == "rig" else set())
    var = [k for k, (a, b) in enumerate(pairs) if a not in const and b not in const]
    for k, (a, b) in enumerate(pairs):
        if a in const or b in const:
            assert np.all(got[k] == 0.0), (a, b)
    err = block_errors([got[k] for k in var], [pairs[k] for k in var], C, cols)
    print(f"{name}: covariance blocks largest error {err.max():.1e}")
    assert err.max() < STEP_TOL, pairs[var[int(err.argmax())]]


def check_converged(gp, p, model, skip_cam=None):
    """Parameters of the GPU solve against the oracle's minimiser (test_gpu_parity tolerances)."""
    views, markers = gp.get_view_poses(), gp.get_marker_poses()
    intr, dist = gp.get_intrinsics()
    cams = [c for c in range(len(intr)) if c != skip_cam]
    assert np.abs(views - p.views).max() < 1e-6
    assert np.abs(markers - p.markers).max() < 1e-6
    assert np.abs(intr[cams] - p.intr[cams]).max() < 1e-4      # pixels
    assert np.abs(dist[cams] - p.dist[cams]).max() < 1e-6
    if model == "rig":
        assert np.abs(gp.get_rig_extrinsics()[cams] - p.ext[cams]).max() < 1e-6


SOLVE = dict(max_iterations=60, function_tolerance=1e-15, gradient_tolerance=1e-12, parameter_tolerance=1e-14)


@pytest.mark.gpu
@pytest.mark.parametrize("name", MAX_CASES)
def test_converged_parameters_match_oracle(name):
    s, _ = _case(name)
    model, n, _ = CASES[name]
    p = to_oracle(s)
    O.lm_solve(p, max_iters=60)
    with BAProblem.from_scene(s, eliminate="views") as gp:
        summ = gp.solve(**SOLVE)
        assert summ["final_cost"] <= summ["initial_cost"]
        assert abs(summ["final_cost"] - O.cost(p)) <= 1e-9 * O.cost(p)
        check_converged(gp, p, model)


# ---------------------------------------------------------------------------------------------------------------
# a camera without a single observation
# ---------------------------------------------------------------------------------------------------------------
BLIND = {"rig6": 2, "single5_all_views": 2}


def blind_scene(name, hold):
    s = make_case(name)
    c = BLIND[name]
    _select(s, s.cam_idx != c)
    if hold:
        s.const_intr[c] = s.const_dist[c] = True
        if s.model == "rig":
            s.const_ext[c] = True
    return s


def camera_columns(name):
    model, _, _ = CASES[name]
    c = BLIND[name]
    return slice(SP[model] * c, SP[model] * (c + 1))


@pytest.mark.gpu
@pytest.mark.parametrize("elim", ["views", "markers"])
@pytest.mark.parametrize("name", list(BLIND))
def test_blind_camera_has_exactly_zero_blocks(name, elim):
    s = blind_scene(name, hold=False)
    model, n, _ = CASES[name]
    cc = camera_columns(name)
    ob = oracle_blocks(to_oracle(s), elim == "views")
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        check_dims(gp, model, n)
        cost = gp.linearize()
        nb = gp.normal_blocks()
    assert np.all(nb["Hes"][:, :, cc] == 0.0) and np.all(nb["Hfs"][:, :, cc] == 0.0)
    assert np.all(nb["Hss"][cc, :] == 0.0) and np.all(nb["Hss"][:, cc] == 0.0)
    assert np.all(nb["gs"][cc] == 0.0)
    assert abs(cost - ob["cost"]) <= TOL * ob["cost"]
    for k in ("Hee", "ge", "Hes", "Hff", "gf", "Hfs", "W"):
        assert max_block_rel(nb[k], ob[k], floor=1e-6 * np.abs(ob[k]).max()) < TOL, k
    assert rel_fro(nb["Hss"], ob["Hss"]) < TOL and rel_fro(nb["gs"], ob["gs"]) < TOL


def camera_parameters(gp, c):
    intr, dist = gp.get_intrinsics()
    out = [intr[c], dist[c]]
    if gp.model == "rig":
        out.append(gp.get_rig_extrinsics()[c])
    return np.concatenate(out)


@pytest.mark.gpu
@pytest.mark.parametrize("hold", [True, False], ids=["held_constant", "free"])
@pytest.mark.parametrize("name", list(BLIND))
def test_blind_camera_stays_put_in_the_solve(name, hold):
    """Held constant or not, the camera's gradient is zero, so its step is exactly zero: its parameters come back
    bitwise unchanged, and every other parameter reaches the oracle's minimiser."""
    s = blind_scene(name, hold)
    model, _, _ = CASES[name]
    c = BLIND[name]
    p = to_oracle(s)
    O.lm_solve(p, max_iters=60)
    with BAProblem.from_scene(s, eliminate="views") as gp:
        before = camera_parameters(gp, c)
        summ = gp.solve(**SOLVE)
        assert summ["final_cost"] <= summ["initial_cost"]
        assert np.array_equal(camera_parameters(gp, c), before)
        check_converged(gp, p, model, skip_cam=c)


@pytest.mark.gpu
@pytest.mark.parametrize("elim", ["views", "markers"])
@pytest.mark.parametrize("name", list(BLIND))
def test_blind_camera_held_constant_covariance(name, elim):
    s = blind_scene(name, hold=True)
    cc = camera_columns(name)
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        cov = gp.covariance()
    assert np.all(cov["shared"][cc, :] == 0.0) and np.all(cov["shared"][:, cc] == 0.0)
    err = compare(cov, *oracle_covariance(to_oracle(s)))
    assert max(err.values()) < STEP_TOL, err


@pytest.mark.gpu
@pytest.mark.parametrize("elim", ["views", "markers"])
@pytest.mark.parametrize("name", list(BLIND))
def test_blind_free_camera_covariance_is_not_spd(name, elim):
    with BAProblem.from_scene(blind_scene(name, hold=False), eliminate=elim) as gp:
        with pytest.raises(L.RccError) as ei:
            gp.covariance()
    assert ei.value.status == L.RCC_NOT_SPD


# ---------------------------------------------------------------------------------------------------------------
# the limit
# ---------------------------------------------------------------------------------------------------------------
def test_camera_limit_is_an_argument_error_without_a_device():
    """One camera past the limit is refused by the argument check, before any device is looked for."""
    lib = L.load()
    h = ctypes.c_void_p()
    for model, n in ((L.MODEL_RIG, MAX_CAM["rig"] + 1), (L.MODEL_SINGLE, MAX_CAM["single"] + 1)):
        opt = L.Options(model=model, n_views=4, n_markers=4, n_cameras=n, n_obs_blocks=0, device=0, eliminate=0)
        assert lib.rcc_ba_create(ctypes.byref(opt), ctypes.byref(h)) == L.RCC_BAD_ARG
        assert not h.value
        msg = lib.rcc_ba_last_error(None).decode()
        assert "too many cameras" in msg and "8 rig or 13 single-model cameras" in msg, msg


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["rig", "single"])
def test_largest_camera_count_is_accepted(model):
    n = MAX_CAM[model]
    with BAProblem(4, 4, n, 0, model) as gp:
        check_dims(gp, model, n)
    with pytest.raises(L.RccError) as ei:
        BAProblem(4, 4, n + 1, 0, model)
    assert ei.value.status == L.RCC_BAD_ARG
