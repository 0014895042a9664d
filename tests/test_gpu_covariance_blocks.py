"""Cross-covariance blocks (rcc_ba_covariance_blocks, BAProblem.covariance_blocks) against the dense inverse of the
oracle's J^T J over the free parameters, against host rebuilds from the reduced system, and against the marginal
blocks of rcc_ba_covariance.

The scenes' J^T J have condition numbers of about 3e9 (single) and 3e10 (rig): 1e-6 relative per block is the
conditioning allowance, as in test_gpu_covariance.py.  A cross block can be far smaller than the marginal blocks of
its two sides, so its error is taken relative to max(|ref|, 1e-6 sqrt(|C_aa| |C_bb|)) (Frobenius norms).
"""
import numpy as np
import pytest

import ba_oracle as O
from helpers import to_oracle
from robot_camera_calibration_b200 import _lib as L
from robot_camera_calibration_b200.problem import BAProblem
from robot_camera_calibration_b200.scenes import config_scene, make_scene
from test_gpu_parity import SCENES, _scene

pytestmark = pytest.mark.gpu
TOL = 1e-6
SIZE = {"view": 6, "marker": 6, "intr": 4, "dist": 5, "ext": 6}


def dense_covariance(s, loss=None):
    """C = (J^T J)^-1 over the free parameters (zero at the constants) and the block -> columns map."""
    p = to_oracle(s)
    if loss:
        p.loss, p.loss_scale = loss
    H, _, _ = O.normal_equations(p)
    free = np.nonzero(~p.const_mask())[0]
    C = np.zeros_like(H)
    C[np.ix_(free, free)] = np.linalg.inv(H[np.ix_(free, free)])
    o_view, o_marker, o_shared, _ = p.offsets()
    sp = p.shared_per_cam

    def cols(block):
        kind, i = block
        start = {"view": o_view + 6 * i, "marker": o_marker + 6 * i, "intr": o_shared + sp * i,
                 "dist": o_shared + sp * i + 4, "ext": o_shared + sp * i + 9}[kind]
        return slice(start, start + SIZE[kind])
    return C, cols


def block_errors(got, pairs, C, cols):
    """Per-pair relative error against the dense inverse (floored by the Cauchy-Schwarz scale of the block)."""
    err = []
    for g, (a, b) in zip(got, pairs):
        ref = C[cols(a), cols(b)]
        assert g.shape == ref.shape, (a, b)
        scale = np.sqrt(np.linalg.norm(C[cols(a), cols(a)]) * np.linalg.norm(C[cols(b), cols(b)]))
        err.append(np.linalg.norm(g - ref) / max(np.linalg.norm(ref), 1e-6 * scale, 1e-300))
    return np.array(err)


def covisible(s, first, second):
    """Boolean matrix: pose i of `first` ("view" / "marker") shares an observation partner with pose j."""
    idx = {"view": s.view_idx, "marker": s.marker_idx}
    n = {"view": len(s.views), "marker": len(s.markers)}
    V = np.zeros((n[first], n[second]), bool)
    V[idx[first], idx[second]] = True
    return (V.astype(int) @ V.T.astype(int)) > 0


def pair_list(s):
    """Every kind of pair, both orders of each, and (a, a) for every block kind."""
    n_cam = len(s.intr)
    rig = s.model == "rig"
    cov_v, cov_m = covisible(s, "view", "marker"), covisible(s, "marker", "view")
    pairs = []
    for cv in (cov_v, cov_m):
        kind = "view" if cv is cov_v else "marker"
        i, j = np.nonzero(np.triu(cv, 1))
        pairs += [((kind, int(i[k])), (kind, int(j[k]))) for k in (0, len(i) // 2, len(i) - 1)]
        i, j = np.nonzero(np.triu(~cv, 1))
        pairs += [((kind, int(i[k])), (kind, int(j[k]))) for k in range(min(2, len(i)))]
    pairs += [(("view", 1), ("marker", 2)), (("view", 7), ("marker", 0)), (("view", 4), ("marker", 5))]
    shared = ["intr", "dist"] + (["ext"] if rig else [])
    for pose in (("view", 2), ("view", 5), ("marker", 3), ("marker", 0)):
        own = int(s.cam_idx[(s.view_idx if pose[0] == "view" else s.marker_idx) == pose[1]][0])
        for c in sorted({own, (own + 1) % n_cam}):
            pairs += [(pose, (k, c)) for k in shared]
    for c in range(n_cam):
        for c2 in range(n_cam):
            pairs += [(("intr", c), ("dist", c2)), (("intr", c), ("intr", c2))]
            if rig:
                pairs.append((("ext", c), ("intr", c2)))
    pairs += [(b, b) for b in (("view", 3), ("marker", 4), ("intr", 0), ("dist", n_cam - 1))]
    if rig:
        pairs.append((("ext", n_cam - 1), ("ext", n_cam - 1)))
    return pairs + [(b, a) for a, b in pairs]


@pytest.mark.parametrize("elim", ["views", "markers"])
@pytest.mark.parametrize("name", list(SCENES))
def test_pairs_match_dense_inverse(name, elim):
    s = _scene(name)
    pairs = pair_list(s)
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        got = gp.covariance_blocks(pairs)
    err = block_errors(got, pairs, *dense_covariance(s))
    print(f"{name}/{elim}: {len(pairs)} pairs, largest block error {err.max():.2e}")
    assert err.max() < TOL, [(pairs[i], err[i]) for i in np.argsort(err)[-5:]]
    if name == "single":
        assert not covisible(s, "view", "marker").all()      # the list has never co-visible view pairs


def test_pairs_with_huber_loss():
    s = _scene("single")
    rng = np.random.default_rng(5)
    bad = rng.choice(s.n_blocks, 12, replace=False)
    s.pixels[bad] += rng.normal(0, 25.0, (12, 8))
    pairs = pair_list(s)
    with BAProblem.from_scene(s, eliminate="views") as gp:
        gp.set_loss("huber", 2.0)
        got = gp.covariance_blocks(pairs)
    err = block_errors(got, pairs, *dense_covariance(s, ("huber", 2.0)))
    print(f"huber: largest block error {err.max():.2e}")
    assert err.max() < TOL


@pytest.mark.parametrize("elim", ["views", "markers"])
def test_constant_blocks_give_exact_zeros(elim):
    s = _scene("single_2cam")
    s.const_intr[1] = True
    s.const_views[3] = True
    const = [("intr", 1), ("view", 3), ("marker", 0)]
    others = [("view", 0), ("view", 3), ("view", 8), ("marker", 0), ("marker", 2), ("intr", 0), ("intr", 1),
              ("dist", 0), ("dist", 1)]
    pairs = [(a, b) for a in const for b in others] + [(b, a) for a in const for b in others]
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        got = gp.covariance_blocks(pairs)
        free = gp.covariance_blocks([(("view", 0), ("dist", 1)), (("view", 8), ("marker", 2))])
    for g, pr in zip(got, pairs):
        assert np.all(g == 0), pr
    err = block_errors(free, [(("view", 0), ("dist", 1)), (("view", 8), ("marker", 2))], *dense_covariance(s))
    assert err.max() < TOL and all(np.abs(f).max() > 0 for f in free)


@pytest.mark.parametrize("elim", ["views", "markers"])
@pytest.mark.parametrize("name", ["single_2cam", "rig"])
def test_consistent_with_marginal_covariance(name, elim):
    s = _scene(name)
    n_cam = len(s.intr)
    sp = 15 if s.model == "rig" else 9
    kept, elim_kind = ("marker", "view") if elim == "views" else ("view", "marker")
    n_kept = len(s.markers) if elim == "views" else len(s.views)
    n_elim = len(s.views) if elim == "views" else len(s.markers)
    shared = [("intr", c) for c in range(n_cam)] + [("dist", c) for c in range(n_cam)]
    shared += [("ext", c) for c in range(n_cam)] if s.model == "rig" else []
    start = {"intr": 0, "dist": 4, "ext": 9}
    kept_pairs = [((kept, i), (kept, i)) for i in range(n_kept)] + [(a, b) for a in shared for b in shared]
    elim_pairs = [((elim_kind, i), (elim_kind, i)) for i in range(n_elim)]
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        marg = gp.covariance()
        got = gp.covariance_blocks(kept_pairs + elim_pairs)
    for g, (a, b) in zip(got, kept_pairs):
        if a[0] == kept:
            want = marg[kept + "s"][a[1]]
        else:
            ra, rb = sp * a[1] + start[a[0]], sp * b[1] + start[b[0]]
            want = marg["shared"][ra:ra + SIZE[a[0]], rb:rb + SIZE[b[0]]]
        assert np.array_equal(g, want), (a, b)
    ref = marg[elim_kind + "s"]
    rel = [np.linalg.norm(g - ref[i]) / np.linalg.norm(ref[i]) for i, g in enumerate(got[len(kept_pairs):])
           if np.linalg.norm(ref[i]) > 0]
    print(f"{name}/{elim}: (e, e) against the marginal blocks: largest relative difference {max(rel):.2e}")
    assert max(rel) <= 1e-10
    for g in got[len(kept_pairs):]:
        assert np.array_equal(g, g.T)


def test_transposes_and_request_independence():
    s = config_scene(2, scale=0.2)
    rng = np.random.default_rng(3)
    nv, nm = len(s.views), len(s.markers)
    blocks = ([("view", int(i)) for i in rng.choice(nv, 6, replace=False)] +
              [("marker", int(i)) for i in rng.choice(nm, 4, replace=False)] + [("intr", 0), ("dist", 0)])
    pairs = [(a, b) for a in blocks for b in blocks]
    order = rng.permutation(len(pairs))
    lone = rng.choice(len(pairs), 8, replace=False)
    with BAProblem.from_scene(s, eliminate="views") as gp:
        first = gp.covariance_blocks(pairs)
        again = gp.covariance_blocks(pairs)
        shuffled = gp.covariance_blocks([pairs[i] for i in order])
        alone = [gp.covariance_blocks([pairs[i]])[0] for i in lone]
    index = {pr: i for i, pr in enumerate(pairs)}
    for i, (a, b) in enumerate(pairs):
        assert np.array_equal(first[i], again[i])
        assert np.array_equal(first[index[(b, a)]], first[i].T), (a, b)
    for k, i in enumerate(order):
        assert np.array_equal(shuffled[k], first[i])
    for g, i in zip(alone, lone):
        assert np.array_equal(g, first[i]), pairs[i]


def _long_row_scene():
    """cfg4-shaped: a few hundred keyframes that each see 500+ tags (as in test_gpu_covariance.py)."""
    s = make_scene(1500, 300, 0.7, seed=41)
    seen = np.bincount(s.view_idx, minlength=len(s.views))
    keep_v = np.nonzero(seen >= 500)[0]
    new_id = np.full(len(s.views), -1)
    new_id[keep_v] = np.arange(len(keep_v))
    keep = new_id[s.view_idx] >= 0
    s.views, s.const_views = s.views[keep_v], s.const_views[keep_v]
    s.view_idx, s.marker_idx, s.cam_idx, s.pixels = (new_id[s.view_idx[keep]], s.marker_idx[keep], s.cam_idx[keep],
                                                     s.pixels[keep])
    return s


def test_long_rows_match_host_rebuild():
    s = _long_row_scene()
    rows = [len(np.unique(s.marker_idx[s.view_idx == v])) for v in range(len(s.views))]
    assert min(rows) >= 500 and max(rows) > 3 * 32
    rng = np.random.default_rng(0)
    ev = rng.choice(len(s.views), 8, replace=False)
    pairs = [(("view", int(ev[i])), ("view", int(ev[i + 1]))) for i in range(0, 8, 2)]
    pairs += [(("view", int(ev[i])), ("view", int(ev[i]))) for i in range(2)]
    pairs += [(("view", int(e)), ("marker", int(m))) for e, m in zip(ev[:4], rng.choice(len(s.markers), 4))]
    pairs += [(("view", int(e)), ("intr", 0)) for e in ev[4:6]] + [(("dist", 0), ("view", int(ev[6])))]
    with BAProblem.from_scene(s, eliminate="views") as gp:
        d = gp.dims
        gp.linearize()
        gp.schur(float("inf"))
        S, _ = gp.reduced_system()
        nb = gp.normal_blocks()
        got = gp.covariance_blocks(pairs)
    const = np.zeros(d.n_reduced, bool)
    const[:6 * d.n_f] = np.repeat(s.const_markers, 6)
    free = np.nonzero(~const)[0]
    Si = np.zeros_like(S)
    Si[np.ix_(free, free)] = np.linalg.inv(S[np.ix_(free, free)])

    def HB(e):
        B = np.zeros((6, d.n_reduced))
        for o in np.nonzero(s.view_idx == e)[0]:
            B[:, 6 * s.marker_idx[o]:6 * s.marker_idx[o] + 6] += nb["W"][o]
        B[:, 6 * d.n_f:] = nb["Hes"][e]
        Hi = np.linalg.inv(nb["Hee"][e])
        return Hi, Hi @ B

    col = {"marker": lambda i: slice(6 * i, 6 * i + 6), "intr": lambda c: slice(6 * d.n_f + 9 * c, 6 * d.n_f + 9 * c + 4),
           "dist": lambda c: slice(6 * d.n_f + 9 * c + 4, 6 * d.n_f + 9 * c + 9)}
    err = 0.0
    for g, (a, b) in zip(got, pairs):
        if a[0] != "view":
            a, b, g = b, a, g.T
        Hi, HiB = HB(a[1])
        if b[0] == "view":
            Hj, HjB = HB(b[1])
            want = HiB @ Si @ HjB.T + (Hi if a == b else 0)
        else:
            want = -HiB @ Si[:, col[b[0]](b[1])]
        err = max(err, np.linalg.norm(g - want) / np.linalg.norm(want))
    print(f"long rows: longest row {max(rows)} partners, largest block error {err:.2e}")
    assert err < TOL


def _call(gp, n_pairs, pairs, out):
    return gp.lib.rcc_ba_covariance_blocks(gp.h, n_pairs, pairs, out)


def test_bad_arguments():
    s = _scene("single")
    out = np.zeros(36)
    dp = out.ctypes.data_as(L.c_double_p)

    def req(*row):
        a = np.array(row, np.int32)
        return a, a.ctypes.data_as(L.c_int32_p)
    with BAProblem.from_scene(s, eliminate="views") as gp:
        bad = [(L.BLOCK_VIEW, 0, 7, 0), (L.BLOCK_VIEW, len(s.views), L.BLOCK_VIEW, 0), (L.BLOCK_MARKER, -1, L.BLOCK_VIEW, 0),
               (L.BLOCK_INTR, 1, L.BLOCK_VIEW, 0), (L.BLOCK_DIST, 0, L.BLOCK_MARKER, len(s.markers)),
               (L.BLOCK_EXT, 0, L.BLOCK_VIEW, 0)]
        for row in bad:
            a, ip = req(*row)
            assert _call(gp, 1, ip, dp) == L.RCC_BAD_ARG, row
        a, ip = req(L.BLOCK_VIEW, 0, L.BLOCK_VIEW, 1)
        assert _call(gp, -1, ip, dp) == L.RCC_BAD_ARG
        assert _call(gp, 1, None, dp) == L.RCC_BAD_ARG
        assert _call(gp, 1, ip, None) == L.RCC_BAD_ARG
        assert _call(gp, 0, None, None) == L.RCC_OK
        assert gp.covariance_blocks([]) == []
        assert _call(gp, 1, ip, dp) == L.RCC_OK


def _unobserved_marker_scene():
    s = _scene("single")
    keep = s.marker_idx != 5
    s.view_idx, s.marker_idx, s.cam_idx, s.pixels = s.view_idx[keep], s.marker_idx[keep], s.cam_idx[keep], s.pixels[keep]
    return s


def _no_gauge_scene():
    s = _scene("single")
    s.const_markers[:] = False
    return s


@pytest.mark.parametrize("elim", ["markers", "views"])
@pytest.mark.parametrize("make", [_unobserved_marker_scene, _no_gauge_scene])
def test_singular_problem_is_not_spd(make, elim):
    with BAProblem.from_scene(make(), eliminate=elim) as gp:
        with pytest.raises(L.RccError) as ei:
            gp.covariance_blocks([(("view", 0), ("marker", 1))])
    assert ei.value.status == L.RCC_NOT_SPD


def test_solve_after_pairs_is_unchanged():
    s = _scene("rig")
    opts = dict(max_iterations=30, function_tolerance=1e-14, gradient_tolerance=1e-12, parameter_tolerance=1e-13)
    res = []
    for with_cov in (False, True):
        with BAProblem.from_scene(s, eliminate="views") as gp:
            if with_cov:
                gp.covariance_blocks([(("view", 0), ("marker", 1)), (("view", 2), ("ext", 1))])
            summ = gp.solve(**opts)
            res.append((summ["final_cost"], gp.get_view_poses(), gp.get_marker_poses(), gp.get_intrinsics()[0]))
    assert abs(res[0][0] - res[1][0]) <= 1e-12 * res[0][0]
    for a, b in zip(res[0][1:], res[1][1:]):
        assert np.abs(a - b).max() < 1e-10


def test_joint_covariance_covers_the_estimation_error():
    """Over 30 seeded scenes with sigma = 0.3 px, e^T (sigma^2 C)^-1 e of the converged (intrinsics + distortion of
    camera 0, view 3, marker 2), C their joint 21 x 21 covariance assembled from pairs, must average like 30 draws of
    chi^2(21): inside [17.3, 25.1], the 99.9 % band of that mean.  Marker 0, the gauge, is held at its true pose
    (scenes.make_scene), so the estimate and the truth share one frame."""
    sigma, stats = 0.3, []
    blocks = [("intr", 0), ("dist", 0), ("view", 3), ("marker", 2)]
    for seed in range(100, 130):
        s = make_scene(8, 20, 0.7, seed=seed, pixel_noise=sigma)
        with BAProblem.from_scene(s) as gp:
            gp.solve(max_iterations=50, function_tolerance=1e-14, gradient_tolerance=1e-12, parameter_tolerance=1e-13)
            intr, dist = gp.get_intrinsics()
            est = np.concatenate([intr[0], dist[0], gp.get_view_poses()[3], gp.get_marker_poses()[2]])
            cb = gp.covariance_blocks([(a, b) for a in blocks for b in blocks])
        C = sigma ** 2 * np.block([[cb[4 * i + j] for j in range(4)] for i in range(4)])
        t = s.truth
        e = est - np.concatenate([t["intr"][0], t["dist"][0], t["views"][3], t["markers"][2]])
        stats.append(float(e @ np.linalg.solve(C, e)))
    print(f"mean chi^2(21) statistic {np.mean(stats):.2f}")
    assert 17.3 <= np.mean(stats) <= 25.1
