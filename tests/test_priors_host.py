"""CPU: the prior oracle (tests/prior_oracle.py), the host side of the prior front ends (QR reduction of NormalPrior
blocks, sqrt_information, the multi-rank split, the --intrinsics-sigma command line) and the argument checks of
rcc_ba_set_priors that need no device."""
import numpy as np
import pytest

import mixed_lens_oracle as MO
import prior_oracle as PO
from robot_camera_calibration_b200 import _lib as L
from robot_camera_calibration_b200 import io_yaml
from robot_camera_calibration_b200.ceres_like import NormalPrior, reduce_normal_priors
from robot_camera_calibration_b200.dist import owner_ranges, shard_priors
from robot_camera_calibration_b200.problem import sqrt_information
from robot_camera_calibration_b200.scenes import make_scene


def _priors(s, rng):
    out = {}
    for kind, vals in (("view", s.views), ("marker", s.markers), ("intr", s.intr), ("dist", s.dist), ("ext", s.ext)):
        idx = np.arange(0, len(vals), 2)
        k = vals.shape[1]
        out[kind] = (idx, vals[idx] + 0.01 * rng.normal(size=(len(idx), k)), rng.normal(size=(len(idx), k, k)))
    return out


def test_oracle_appends_prior_rows_to_the_tag_system():
    s = make_scene(5, 6, 0.8, n_cam=2, model="rig", seed=3)
    rng = np.random.default_rng(1)
    pri = _priors(s, rng)
    p = MO.oracle_problem(s)
    H0, g0, c0 = MO.normal_equations(p)
    H, g, c = PO.normal_equations(p, pri)
    x = p.pack()
    dH, dg, dc = np.zeros_like(H), np.zeros_like(g), 0.0
    for kind, (idx, mean, A) in pri.items():
        for i, mu, a in zip(idx, mean, A):
            cols = PO.columns(p, kind, i)
            r = a @ (x[cols] - mu)
            dH[np.ix_(cols, cols)] += a.T @ a
            dg[cols] += a.T @ r
            dc += 0.5 * r @ r
    assert np.allclose(H - H0, dH, rtol=1e-12, atol=1e-14 * np.abs(H).max())
    assert np.allclose(g - g0, dg, rtol=1e-12, atol=1e-14 * np.abs(g).max())
    assert abs(c - c0 - dc) <= 1e-12 * c
    # the prior rows are exactly linear: the cost at x + d is the model's
    d = 1e-3 * rng.normal(size=len(x))
    Jp, rp = PO.prior_rows(p, pri)
    _, rp2 = PO.prior_rows(p, pri, x + d)
    assert np.allclose(rp2, rp + Jp @ d, rtol=1e-12, atol=1e-12)


def test_qr_reduction_keeps_the_normal_equations_and_the_cost():
    rng = np.random.default_rng(2)
    x = rng.normal(size=6)
    b = rng.normal(size=6)
    for m in (9, 6, 3):
        A = rng.normal(size=(m, 6))
        R, mu, c = reduce_normal_priors([(A, b)])
        assert R.shape == (6, 6) and c == 0.0 and np.array_equal(mu, b)
        assert np.allclose(R.T @ R, A.T @ A, rtol=1e-12, atol=1e-12)
        assert np.isclose(np.sum((R @ (x - mu)) ** 2), np.sum((A @ (x - b)) ** 2), rtol=1e-12)
    A6 = rng.normal(size=(6, 6))
    R, mu, c = reduce_normal_priors([(A6, b)])
    assert R is A6 and mu is b and c == 0.0                 # one square prior goes through unchanged
    A1, A2, b2 = rng.normal(size=(6, 6)), rng.normal(size=(4, 6)), rng.normal(size=6)
    R, mu, c = reduce_normal_priors([(A1, b), (A2, b2)])
    ref = np.sum((A1 @ (x - b)) ** 2) + np.sum((A2 @ (x - b2)) ** 2)
    assert c > 0 and np.isclose(np.sum((R @ (x - mu)) ** 2) + c, ref, rtol=1e-11)
    assert np.allclose(R.T @ R, A1.T @ A1 + A2.T @ A2, rtol=1e-12, atol=1e-12)
    pr = NormalPrior(A2, b2)
    assert pr.num_residuals() == 4 and pr.parameter_block_sizes() == [6]
    res, jac = np.empty(4), np.empty((4, 6))
    assert pr.Evaluate([x], res, [jac]) and np.allclose(res, A2 @ (x - b2)) and np.array_equal(jac, A2)


def test_sqrt_information_whitens_the_covariance():
    rng = np.random.default_rng(3)
    M = rng.normal(size=(3, 5, 5))
    cov = M @ np.swapaxes(M, 1, 2) + 0.1 * np.eye(5)
    A = sqrt_information(cov)
    assert np.allclose(A @ cov @ np.swapaxes(A, 1, 2), np.eye(5), atol=1e-10)
    assert np.allclose(sqrt_information(cov[0]), A[0])


@pytest.mark.parametrize("elim_view", [True, False])
def test_each_prior_goes_to_exactly_one_rank(elim_view):
    s = make_scene(10, 20, 0.7, seed=4)
    pri = _priors(s, np.random.default_rng(4))
    del pri["ext"]
    e_idx = s.view_idx if elim_view else s.marker_idx
    world = 3
    ranges = owner_ranges(np.bincount(e_idx, minlength=len(s.views) if elim_view else len(s.markers)), world)
    parts = [shard_priors(pri, elim_view, r, ranges[r]) for r in range(world)]
    for kind, (idx, mean, A) in pri.items():
        got = np.concatenate([parts[r][kind][0] for r in range(world)])
        assert sorted(got.tolist()) == sorted(idx.tolist())
        eliminated = kind == ("view" if elim_view else "marker")
        for r in range(world):
            ir, mr, ar = parts[r][kind]
            pos = np.searchsorted(idx, ir)
            assert np.array_equal(mean[pos], mr) and np.array_equal(A[pos], ar)
            if eliminated:
                assert np.all((ir >= ranges[r][0]) & (ir < ranges[r][1]))
            elif r > 0:
                assert len(ir) == 0


def test_command_line_intrinsics_sigma_arguments(tmp_path, capsys):
    from robot_camera_calibration_b200.__main__ import main, parser
    a = parser().parse_args([str(tmp_path), "--intrinsics-sigma", "2", "1.5", "0.01"])
    assert a.intrinsics_sigma == [2.0, 1.5, 0.01] and not a.fix_intrinsics
    assert parser().parse_args([str(tmp_path)]).intrinsics_sigma is None
    for bad in (["--fix-intrinsics", "--intrinsics-sigma", "1", "1", "1"], ["--intrinsics-sigma", "1", "1"],
                ["--intrinsics-sigma", "1", "0", "1"], ["--intrinsics-sigma", "1", "-1", "1"]):
        with pytest.raises(SystemExit) as e:
            main([str(tmp_path), *bad])
        assert e.value.code == 2
    capsys.readouterr()
    with pytest.raises(ValueError):
        io_yaml.optimise_directory(str(tmp_path), refine_intrinsics=False, intrinsics_sigma=(1, 1, 1))
    pri = io_yaml.intrinsics_priors([[500, 510, 320, 240]] * 2, [[0.1, 0.01, 0, 0, 0]] * 2, (2.0, 4.0, 0.5))
    assert np.array_equal(pri["intr"][0], [0, 1]) and np.array_equal(pri["dist"][1][1], [0.1, 0.01, 0, 0, 0])
    assert np.array_equal(pri["intr"][2][1], np.diag([0.5, 0.5, 0.25, 0.25]))
    assert np.array_equal(pri["dist"][2][0], 2.0 * np.eye(5))


def test_set_priors_without_a_handle_is_a_bad_argument():
    lib = L.load()
    idx = np.zeros(1, np.int32)
    mean, A = np.zeros(6), np.eye(6)
    assert lib.rcc_ba_set_priors(None, L.BLOCK_VIEW, 1, idx.ctypes.data_as(L.c_int32_p),
                                 mean.ctypes.data_as(L.c_double_p), A.ctypes.data_as(L.c_double_p)) == L.RCC_BAD_ARG
