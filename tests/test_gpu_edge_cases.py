"""GPU: edge cases of the domain -- empty / ragged inputs, unobserved blocks, duplicate
observations, argument and call-order errors."""
import numpy as np
import pytest

import ba_oracle as O
from helpers import max_block_rel, oracle_blocks, oracle_reduced, rel_fro, to_oracle
from robot_camera_calibration_b200 import _lib as L
from robot_camera_calibration_b200.problem import BAProblem
from robot_camera_calibration_b200.scenes import make_scene

pytestmark = pytest.mark.gpu
TOL = 1e-9


def _keep(s, mask):
    s.view_idx, s.marker_idx, s.cam_idx, s.pixels = s.view_idx[mask], s.marker_idx[mask], s.cam_idx[mask], s.pixels[mask]
    return s


def _check_against_oracle(s, elim="views"):
    p = to_oracle(s)
    ob = oracle_blocks(p, elim == "views")
    S, b, *_ = oracle_reduced(p, elim == "views", 1e4)
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        cost = gp.linearize()
        nb = gp.normal_blocks()
        gp.schur(1e4)
        Sg, bg = gp.reduced_system()
        gp.solve_step()
        st = gp.step()
    assert abs(cost - ob["cost"]) <= TOL * max(ob["cost"], 1e-300)
    for k in ("Hee", "Hff", "W", "ge", "gf", "Hes", "Hfs"):
        assert max_block_rel(nb[k], ob[k], floor=1e-6 * np.abs(ob[k]).max()) < TOL, k
    assert rel_fro(Sg, S) < TOL and rel_fro(bg, b) < TOL
    return st


@pytest.mark.parametrize("elim", ["views", "markers"])
def test_unobserved_view_and_marker_stay_put(elim):
    s = make_scene(9, 12, 0.9, seed=51)
    _keep(s, (s.view_idx != 4) & (s.marker_idx != 6))          # view 4 and tag 6 are never observed
    st = _check_against_oracle(s, elim)
    dv, dm = (st["d_e"], st["d_f"]) if elim == "views" else (st["d_f"], st["d_e"])
    assert np.all(dv[4] == 0.0) and np.all(dm[6] == 0.0)
    assert np.all(dm[0] == 0.0)                                 # gauge


def test_ragged_segments_cross_every_chunk_boundary():
    """views with 1, 5, 6, 7, 12, 13, 47, 48, 49, 97 ... tags: partial thread-groups, exact
    multiples of the 6-block warp iteration, and segments split into several chunks."""
    s = make_scene(130, 30, 1.0, seed=52, image_size=(2000, 1500))
    want = sorted([1, 5, 6, 7, 12, 13, 47, 48, 49, 97, 61, 60, 120, 2], reverse=True)
    counts = np.bincount(s.view_idx, minlength=len(s.views))
    order = np.argsort(-counts)                       # views with the most visible tags first
    keep = np.zeros(s.n_blocks, bool)
    for v, n in zip(order, want):
        idx = np.nonzero(s.view_idx == v)[0]
        assert len(idx) >= n, (v, len(idx), n)
        keep[idx[:n]] = True
    _keep(s, keep)                                    # the other 16 views end up unobserved
    got = np.bincount(s.view_idx, minlength=len(s.views))
    assert sorted(got[got > 0].tolist(), reverse=True) == want
    _check_against_oracle(s, "views")
    _check_against_oracle(s, "markers")


def test_duplicate_observations_are_summed():
    """the same tag reported twice in one frame (and, in a rig, by two cameras)."""
    s = make_scene(8, 10, 0.9, seed=53)
    dup = np.arange(0, s.n_blocks, 5)
    s.view_idx = np.concatenate([s.view_idx, s.view_idx[dup]])
    s.marker_idx = np.concatenate([s.marker_idx, s.marker_idx[dup]])
    s.cam_idx = np.concatenate([s.cam_idx, s.cam_idx[dup]])
    s.pixels = np.concatenate([s.pixels, s.pixels[dup] + 0.5])
    _check_against_oracle(s, "views")
    r = make_scene(10, 8, 0.9, n_cam=3, model="rig", seed=54)      # overlapping cameras see the same tag
    _check_against_oracle(r, "views")
    _check_against_oracle(r, "markers")


def test_single_observation_and_empty_problem():
    s = make_scene(4, 3, 1.0, seed=55)
    _keep(s, np.arange(s.n_blocks) == 0)
    _check_against_oracle(s)
    with BAProblem(3, 4, 1, 0) as gp:                              # no observations at all
        gp.set_intrinsics(s.intr, s.dist)
        gp.set_view_poses(s.views); gp.set_marker_poses(s.markers); gp.set_marker_sizes(s.sizes)
        gp.set_observations(np.zeros(0, np.int32), np.zeros(0, np.int32), None, np.zeros((0, 8)))
        assert gp.linearize() == 0.0
        out = gp.evaluate()
        assert out["cost"] == 0.0 and out["residuals"].shape == (0, 8)
        nb = gp.normal_blocks()
        assert not nb["Hee"].any() and not nb["Hss"].any()
        summ = gp.solve(max_iterations=3)
        assert summ["final_cost"] == 0.0
        assert np.array_equal(gp.get_view_poses(), s.views)


def test_argument_and_call_order_errors():
    s = make_scene(5, 6, 0.9, seed=56)
    with BAProblem(len(s.views), len(s.markers), 1, s.n_blocks) as gp:
        with pytest.raises(L.RccError) as e:
            gp.linearize()
        assert e.value.status == L.RCC_NOT_READY
        bad = s.view_idx.copy(); bad[3] = len(s.views)
        with pytest.raises(L.RccError) as e:
            gp.set_observations(bad, s.marker_idx, s.cam_idx, s.pixels)
        assert e.value.status == L.RCC_BAD_ARG and "view index" in str(e.value)
        bad = s.cam_idx.copy(); bad[0] = 1
        with pytest.raises(L.RccError) as e:
            gp.set_observations(s.view_idx, s.marker_idx, bad, s.pixels)
        assert e.value.status == L.RCC_BAD_ARG
        gp.set_observations(s.view_idx, s.marker_idx, s.cam_idx, s.pixels)
        with pytest.raises(L.RccError) as e:
            gp.schur(1e4)
        assert e.value.status == L.RCC_NOT_READY
        with pytest.raises(L.RccError) as e:
            gp.set_constant("marker", 99)
        assert e.value.status == L.RCC_BAD_ARG
        with pytest.raises(L.RccError) as e:
            gp.set_rig_extrinsics(np.zeros((1, 6)))
        assert e.value.status == L.RCC_BAD_ARG
        gp.set_intrinsics(s.intr, s.dist); gp.set_view_poses(s.views)
        gp.set_marker_poses(s.markers); gp.set_marker_sizes(s.sizes)
        gp.linearize()
        with pytest.raises(L.RccError) as e:
            gp.schur(-1.0)
        assert e.value.status == L.RCC_BAD_ARG
        with pytest.raises(L.RccError) as e:
            gp.solve_step()
        assert e.value.status == L.RCC_NOT_READY
        with pytest.raises(L.RccError) as e:
            gp.reduced_system()
        assert e.value.status == L.RCC_NOT_READY
    with pytest.raises(L.RccError) as e:            # 14 single-model cameras = 126 shared parameters: over the border limit
        BAProblem(4, 4, 14, 8)
    assert e.value.status == L.RCC_BAD_ARG and "cameras" in str(e.value)


def test_constant_intrinsics_and_all_views_constant():
    s = make_scene(8, 9, 0.9, seed=57)
    s.const_intr[:] = True
    s.const_dist[:] = True
    st = _check_against_oracle(s)
    assert np.all(st["d_shared"] == 0.0)
    s.const_views[:] = True                                     # only the tags move
    p = to_oracle(s)
    delta, *_ = O.lm_step(p, 1e4)
    st = _check_against_oracle(s, "views")
    assert np.all(st["d_e"] == 0.0)
    o_view, o_marker, o_shared, n = p.offsets()
    assert rel_fro(st["d_f"].ravel(), delta[o_marker:o_shared]) < 1e-6


def test_deterministic_bitwise_repeatability():
    s = make_scene(20, 40, 0.6, seed=58)
    res = []
    for _ in range(2):
        with BAProblem.from_scene(s) as gp:
            gp.linearize(); gp.schur(1e4)
            S, b = gp.reduced_system()
            nb = gp.normal_blocks()
        res.append((S, b, nb["Hee"], nb["Hss"]))
    for a, b in zip(*res):
        assert np.array_equal(a, b)                             # fixed summation order, no atomics


@pytest.mark.parametrize("model", ["single", "rig"])
@pytest.mark.parametrize("elim", ["views", "markers"])
def test_evaluate_in_shuffled_caller_order(model, elim):
    """Evaluate() must return residual blocks in the caller's order whatever the internal sort is:
    a random caller order exercises the per-(block, array) copy-out of the materialising kernel,
    the view-major order of make_scene its one-copy-per-array path."""
    kw = dict(n_cam=2, model="rig") if model == "rig" else {}
    s = make_scene(14, 23, 0.8, seed=57, **kw)
    perm = np.random.default_rng(5).permutation(s.n_blocks)
    s.view_idx, s.marker_idx, s.cam_idx, s.pixels = s.view_idx[perm], s.marker_idx[perm], s.cam_idx[perm], s.pixels[perm]
    p = to_oracle(s)
    r, Jb = O.residuals(p), O.jacobian_blocks_cs(p)
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        out = gp.evaluate()
        res_only = gp.evaluate(want_jacobians=False)
    assert abs(out["cost"] - O.cost(p)) <= TOL * O.cost(p)
    assert abs(res_only["cost"] - O.cost(p)) <= TOL * O.cost(p)
    assert max_block_rel(out["residuals"], r) < TOL
    assert max_block_rel(res_only["residuals"], r) < TOL
    for k in Jb:
        assert max_block_rel(out["jacobians"][k], Jb[k]) < TOL, k


@pytest.mark.parametrize("shuffled", [False, True])
def test_update_pixels_matches_a_fresh_problem(shuffled):
    """rcc_ba_update_pixels: new pixel coordinates on the same indices must give exactly what a problem
    built from those pixels gives -- in the caller order == sorted order case (piecewise upload on the side
    stream, overlapped with the E pass) and in the general case (staging buffer + device permutation),
    followed by linearize, by evaluate, and twice in a row."""
    s = make_scene(60, 40, 0.7, seed=58)
    if shuffled:
        perm = np.random.default_rng(6).permutation(s.n_blocks)
        s.view_idx, s.marker_idx, s.cam_idx, s.pixels = s.view_idx[perm], s.marker_idx[perm], s.cam_idx[perm], s.pixels[perm]
    rng = np.random.default_rng(7)
    pix2 = np.ascontiguousarray(s.pixels + rng.normal(0.0, 0.5, s.pixels.shape))
    pix3 = np.ascontiguousarray(s.pixels + rng.normal(0.0, 0.5, s.pixels.shape))
    with BAProblem.from_scene(s) as gp:
        gp.linearize()
        gp.update_pixels(pix2)
        c2 = gp.linearize()
        nb2 = gp.normal_blocks()
        gp.update_pixels(pix3)
        gp.update_pixels(pix2)                       # overwritten before anything consumed it
        e2 = gp.evaluate(want_jacobians=False)
        gp.update_pixels(pix3)
        c3 = gp.linearize()
    ref = make_scene(60, 40, 0.7, seed=58)
    ref.view_idx, ref.marker_idx, ref.cam_idx = s.view_idx, s.marker_idx, s.cam_idx
    for pix, cost, nb in ((pix2, c2, nb2), (pix3, c3, None)):
        ref.pixels = pix
        with BAProblem.from_scene(ref) as gq:
            assert gq.linearize() == cost
            if nb is not None:
                nq = gq.normal_blocks()
                for k in ("Hee", "Hff", "W", "ge", "gf", "Hes", "Hfs", "Hss", "gs"):
                    assert np.array_equal(nq[k], nb[k]), k
                assert np.array_equal(gq.evaluate(want_jacobians=False)["residuals"], e2["residuals"])


def test_update_pixels_in_pieces_at_size_matches_a_fresh_problem():
    """From LARGE_UPLOAD_BLOCKS (problem.h) on, a piecewise update_pixels is cut into 8 pieces and linearize runs the
    F pass of each piece as soon as it has landed.  FP64 and int16 updates on such a scene must give exactly what a
    problem built from those pixels gives: the F chunks are cut at the same piece boundaries in both."""
    s = make_scene(5000, 4000, 0.25, blocked=True, chunk_views=250, round_pixels=True, seed=65)
    assert s.n_blocks >= 4_000_000
    key = s.view_idx.astype(np.int64) * len(s.markers) + s.marker_idx
    assert np.all(np.diff(key) >= 0)                 # caller order == E-sorted order: the piecewise path
    rng = np.random.default_rng(10)
    new_pixels = [s.pixels + rng.integers(-2, 3, s.pixels.shape) for _ in range(2)]
    with BAProblem.from_scene(s, eliminate="views") as gp:
        gp.linearize()
        for pix, dt in zip(new_pixels, (np.float64, np.int16)):
            gp.update_pixels(pix.astype(dt))
            cost = gp.linearize()
            nb = gp.normal_blocks()
            s.pixels = pix
            with BAProblem.from_scene(s, eliminate="views") as gq:
                assert gq.linearize() == cost
                nq = gq.normal_blocks()
            for k in ("Hee", "Hff", "W", "ge", "gf", "Hes", "Hfs", "Hss", "gs"):
                assert np.array_equal(nq[k], nb[k]), k
            del nb, nq


@pytest.mark.parametrize("model", ["single", "rig"])
def test_bitwise_repeatability_stress(model):
    """compute-sanitizer's racecheck is closed on the pool, so the hand-rolled last-CTA protocol of the
    finalize kernel and the __syncwarp-ordered shared-memory read-modify-write of the Schur SYRK are
    exercised the slow way: 60 runs of linearize + Schur + solve_step on one handle (timing differs from
    run to run) and 4 fresh handles, on a scene whose rows span several chunks and (rig) several cameras;
    every output must be bit-identical to the first run."""
    kw = dict(n_cam=3, model="rig") if model == "rig" else {}
    s = make_scene(150, 60, 1.0, seed=61, image_size=(2000, 1500), **kw)      # ~150 tags per view: 3 chunks per row
    assert np.bincount(s.view_idx).max() > 64

    def run(gp):
        gp.set_view_poses(s.views)            # invalidates everything: the whole pipeline runs again
        gp.linearize()
        nb = gp.normal_blocks()
        gp.schur(1e4)
        S, b = gp.reduced_system()
        gp.solve_step()
        st = gp.step()
        return [nb[k] for k in ("Hee", "Hff", "W", "ge", "gf", "Hes", "Hfs", "Hss", "gs")] + [S, b, st["d_e"], st["d_f"], st["d_shared"]]

    first = None
    for fresh in range(4):
        with BAProblem.from_scene(s) as gp:
            for rep in range(15):
                out = run(gp)
                if first is None:
                    first = out
                    continue
                for i, (a, b) in enumerate(zip(first, out)):
                    assert np.array_equal(a, b), (fresh, rep, i)


def test_two_handles_on_two_devices_in_one_process():
    """include/rcc_ba.h: "distinct handles are independent".  The > 48 KB dynamic shared-memory opt-in of the
    assemble / materialise / SYRK kernels is a per-device attribute: a second handle on another device of the
    same process must work, interleaved with the first, and give bit-identical results."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs in one process")
    s = make_scene(40, 50, 0.8, seed=62)
    with BAProblem.from_scene(s, device=0) as g0, BAProblem.from_scene(s, device=1) as g1:
        outs = []
        for gp in (g0, g1, g0, g1):
            gp.set_view_poses(s.views)
            c = gp.linearize()
            ev = gp.evaluate()
            gp.schur(1e4)
            S, b = gp.reduced_system()
            gp.solve_step()
            outs.append((c, ev["residuals"], ev["jacobians"]["view"], S, b, gp.step()["d_f"]))
        for o in outs[1:]:
            for a, b in zip(outs[0], o):
                assert np.array_equal(np.asarray(a), np.asarray(b))


def test_solve_reports_failure_when_the_starting_point_cannot_be_evaluated():
    """A corner behind the camera at the INITIAL point: Ceres returns FAILURE from the first evaluation;
    the LM driver must stop with termination 4 instead of iterating on a garbage linearisation."""
    s = make_scene(8, 9, 0.9, seed=63)
    s.views[3, 0:3] += np.array([0.0, np.pi, 0.0])                      # view 3 now looks away from the wall
    with BAProblem.from_scene(s) as gp:
        assert gp.evaluate(allow_failure=True)["failed"]
        summ = gp.solve(max_iterations=10)
    assert summ["termination"] == 4 and summ["iterations"] == 0 and summ["accepted"] == 0


@pytest.mark.parametrize("shuffled", [False, True])
def test_integer_pixel_entry_points_are_bit_identical_to_fp64(shuffled):
    """rcc_ba_set_observations_i16 / _i32 / rcc_ba_update_pixels_i16 (the reference's integer corners,
    corner_detections.cpp:53-54, camera_pose.cpp:135-142) widen on the device: every result must be bit-identical
    to the FP64 entry points fed the same integers -- on the golden integer-pixel fixture and on a larger scene,
    in caller order == sorted order (piecewise overlapped upload) and in a shuffled order."""
    from helpers import load_golden
    for s in (load_golden("single_intpix")[0], make_scene(60, 40, 0.7, seed=64, round_pixels=True)):
        if shuffled:
            perm = np.random.default_rng(8).permutation(s.n_blocks)
            s.view_idx, s.marker_idx, s.cam_idx, s.pixels = s.view_idx[perm], s.marker_idx[perm], s.cam_idx[perm], s.pixels[perm]
        assert np.array_equal(s.pixels, np.trunc(s.pixels))
        pix2 = np.trunc(s.pixels + np.random.default_rng(9).integers(-2, 3, s.pixels.shape))

        def run(gp):
            c = gp.linearize()
            nb = gp.normal_blocks()
            ev = gp.evaluate(want_jacobians=False)
            return [c, ev["residuals"]] + [nb[k] for k in ("Hee", "Hff", "W", "ge", "gf", "Hes", "Hfs", "Hss", "gs")]

        with BAProblem.from_scene(s) as gp:
            ref1 = run(gp)
            gp.update_pixels(pix2)
            ref2 = run(gp)
        for dt in (np.int16, np.int32):
            si = make_scene(3, 3, 1.0, seed=1)          # container only
            import copy
            si = copy.copy(s)
            si.pixels = s.pixels.astype(dt)
            with BAProblem.from_scene(si) as gp:
                got1 = run(gp)
                gp.update_pixels(pix2.astype(np.int16))
                got2 = run(gp)
                gp.update_pixels(s.pixels.astype(np.int16))
                gp.update_pixels(pix2.astype(np.int16))       # overwritten before anything consumed it
                got3 = run(gp)
            for want, got in ((ref1, got1), (ref2, got2), (ref2, got3)):
                for a, b in zip(want, got):
                    assert np.array_equal(np.asarray(a), np.asarray(b))


@pytest.mark.parametrize("model,elim", [("single", "views"), ("single", "markers"), ("rig", "views")])
def test_syrk_ragged_rows_over_several_subtiles_match_the_oracle(model, elim):
    """The block-sparse Schur SYRK on ragged rows that span several 32-block column sub-tiles, in both elimination
    directions and for the rig model."""
    s = make_scene(70, 90, 0.35, n_cam=2 if model == "rig" else 1, model=model, seed=77, round_pixels=True)
    rng = np.random.default_rng(5)
    _keep(s, rng.random(s.n_blocks) < 0.8)               # ragged rows
    _check_against_oracle(s, elim)
