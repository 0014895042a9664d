"""GPU: the linearisation kernel walks a chunk 8 observation blocks at a time and runs a full group of 8 and the
last, partial group of a chunk on different code paths.  Every chunk length from 1 to 15 and two longer ones is
checked against the oracle, for both passes, the single-camera and the rig model, with and without a robust loss."""
import numpy as np
import pytest

from helpers import max_block_rel, oracle_blocks, rel_fro, to_oracle
from robot_camera_calibration_b200.problem import BAProblem
from robot_camera_calibration_b200.scenes import make_scene

pytestmark = pytest.mark.gpu
TOL = 1e-9
# observation blocks per (view, camera): chunks shorter than one group, one full group, and a full group followed by
# a last group of every size from 1 to 7
COUNTS = [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 19, 23]


def _scene(model):
    n_cam = 2 if model == "rig" else 1
    s = make_scene(60, 20, 1.0, n_cam=n_cam, model=model, seed=91, image_size=(2000, 1500))
    key = s.view_idx.astype(np.int64) * n_cam + s.cam_idx
    order = np.argsort(-np.bincount(key))
    keep = np.zeros(s.n_blocks, bool)
    for k, n in zip(order, COUNTS):
        idx = np.nonzero(key == k)[0]
        assert len(idx) >= n, (k, len(idx), n)
        keep[idx[:n]] = True
    s.view_idx, s.marker_idx, s.cam_idx, s.pixels = s.view_idx[keep], s.marker_idx[keep], s.cam_idx[keep], s.pixels[keep]
    got = np.bincount(s.view_idx.astype(np.int64) * n_cam + s.cam_idx)
    assert sorted(got[got > 0].tolist()) == COUNTS
    return s


@pytest.mark.parametrize("elim", ["views", "markers"])
@pytest.mark.parametrize("loss", [None, "huber"])
@pytest.mark.parametrize("model", ["single", "rig"])
def test_every_last_group_size_matches_the_oracle(model, loss, elim):
    s = _scene(model)
    p = to_oracle(s)
    if loss:
        p.loss, p.loss_scale = loss, 2.0
    ob = oracle_blocks(p, elim == "views")
    with BAProblem.from_scene(s, eliminate=elim) as gp:
        if loss:
            gp.set_loss(loss, 2.0)
        cost = gp.linearize()
        nb = gp.normal_blocks()
    assert abs(cost - ob["cost"]) <= TOL * ob["cost"]
    for k in ("Hee", "Hff", "W", "ge", "gf", "Hes", "Hfs"):
        assert max_block_rel(nb[k], ob[k], floor=1e-6 * np.abs(ob[k]).max()) < TOL, k
    assert rel_fro(nb["Hss"], ob["Hss"]) < TOL and rel_fro(nb["gs"], ob["gs"]) < TOL
