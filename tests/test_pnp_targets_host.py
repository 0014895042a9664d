"""Rigid-target PnP without a GPU: the argument checks of rcc_pnp_target_batch, the grouping of detections into
targets and free tags and their chaining (initialiser.initialise_targets with the PnP calls replaced by exact
hand-made poses), io_yaml.read_detections and the --initialise command line."""
import os

import numpy as np
import pytest

from robot_camera_calibration_b200 import _lib as L
from robot_camera_calibration_b200 import initialiser, io_yaml
from robot_camera_calibration_b200.__main__ import main, parser
from robot_camera_calibration_b200.scenes import board_layout, compose, invert


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


# ------------------------------------------------------------------ rcc_pnp_target_batch argument checks
def _call(lens=0, shared9=True, n_slots=4, corners=None, n=2, start=None, slot=None, pixels=True, poses=True,
          cost=True):
    lib = L.load()
    corners = board_layout(2, 2, 0.1, 0.3).reshape(-1) if corners is None else np.asarray(corners, float)
    start = np.array([0, 2, 3], np.int64) if start is None else np.asarray(start, np.int64)
    slot = np.array([0, 1, 3], np.int32) if slot is None else np.asarray(slot, np.int32)
    sh = np.array([500.0, 500, 320, 240, 0, 0, 0, 0, 0])
    px = np.zeros(8 * 3)
    out = np.zeros(6 * max(n, 1))
    fc = np.zeros(max(n, 1))
    dp = lambda a, keep: a.ctypes.data_as(L.c_double_p) if keep else None
    return lib.rcc_pnp_target_batch(0, lens, dp(sh, shared9), n_slots, dp(corners, corners is not None), n,
                                    start.ctypes.data_as(L.c_int64_p) if start is not None else None,
                                    slot.ctypes.data_as(L.c_int32_p) if slot is not None else None,
                                    dp(px, pixels), dp(out, poses), dp(fc, cost), 30)


def _null_start():
    lib = L.load()
    sh, cr, px, out = np.zeros(9), np.zeros(32), np.zeros(8), np.zeros(6)
    slot = np.zeros(1, np.int32)
    dp = lambda a: a.ctypes.data_as(L.c_double_p)
    return lib.rcc_pnp_target_batch(0, 0, dp(sh), 4, dp(cr), 1, None, slot.ctypes.data_as(L.c_int32_p), dp(px),
                                    dp(out), None, 0)


def _null_slot():
    lib = L.load()
    sh, cr, px, out = np.zeros(9), np.zeros(32), np.zeros(8), np.zeros(6)
    start = np.array([0, 1], np.int64)
    dp = lambda a: a.ctypes.data_as(L.c_double_p)
    return lib.rcc_pnp_target_batch(0, 0, dp(sh), 4, dp(cr), 1, start.ctypes.data_as(L.c_int64_p), None, dp(px),
                                    dp(out), None, 0)


@pytest.mark.parametrize("case", [
    dict(lens=2), dict(lens=-1), dict(n=-1),
    dict(shared9=False), dict(pixels=False), dict(poses=False),
    dict(start=[1, 2, 3]), dict(start=[0, 2, 2]), dict(start=[0, 3, 2]),
    dict(n_slots=0), dict(n_slots=-3),
    dict(slot=[0, 4, 1]), dict(slot=[0, -1, 1]),
    dict(corners=np.where(np.arange(32) == 5, np.nan, board_layout(2, 2, 0.1, 0.3).reshape(-1))),
    dict(corners=np.where(np.arange(32) == 31, np.inf, board_layout(2, 2, 0.1, 0.3).reshape(-1))),
])
def test_bad_arguments_are_rejected_before_any_device_query(case):
    assert _call(**case) == L.RCC_BAD_ARG


def test_null_index_arrays_are_rejected():
    assert _null_start() == L.RCC_BAD_ARG
    assert _null_slot() == L.RCC_BAD_ARG
    lib = L.load()
    sh = np.zeros(9)
    assert lib.rcc_pnp_target_batch(0, 0, sh.ctypes.data_as(L.c_double_p), 4, None, 1, None, None, None, None, None,
                                    0) == L.RCC_BAD_ARG


def test_no_problems_is_ok_and_valid_arguments_reach_the_device():
    assert _call(n=0, shared9=False, pixels=False, poses=False, cost=False) == L.RCC_OK
    # the final cost may be NULL; without a device valid arguments fail with RCC_CUDA_ERROR, not RCC_BAD_ARG
    rc = _call(cost=False)
    assert rc == (L.RCC_OK if _has_gpu() else L.RCC_CUDA_ERROR)


# ------------------------------------------------------------------ grouping and chaining on hand-made poses
TARGETS = [(np.arange(4), board_layout(2, 2, 0.1, 0.3)), (10 + np.arange(4), board_layout(2, 2, 0.08, 0.25))]
SLOT = {int(i): (b, o + k) for b, o in ((0, 0), (1, 4)) for k, i in enumerate(TARGETS[b][0])}
CORNERS = np.concatenate([c for _, c in TARGETS])


def _truth(rng):
    """World poses in an arbitrary frame G of both boards, free tags 20, 21 and 6 cameras."""
    rt = lambda: np.concatenate([rng.normal(0, 0.3, 3), rng.normal(0, 1.0, 3)])
    return {("target", 0): rt(), ("target", 1): rt(), ("tag", 20): rt(), ("tag", 21): rt()}, [rt() for _ in range(6)]


def _key(t):
    return ("target", SLOT[t][0]) if t in SLOT else ("tag", t)


def _fake_pnp(monkeypatch, ents, views):
    """pnp_targets / pnp_batch returning the exact cam_T_entity; the pixels carry (frame, tag id)."""
    def exact(px):
        n, t = int(px[0]), int(px[1])
        return compose(invert(views[n]), ents[_key(t)])

    def pnp_targets(intr, dist, corners, start, slot, pixels, guess=None, device=0, max_iterations=100,
                    lens="radtan"):
        assert np.array_equal(corners, CORNERS)
        assert [SLOT[int(pixels[k][1])][1] for k in range(len(slot))] == list(slot)
        return np.array([exact(pixels[start[p]]) for p in range(len(start) - 1)]).reshape(-1, 6), np.zeros(len(start) - 1)

    def pnp_batch(intr, dist, sizes, pixels, guess=None, device=0, max_iterations=100, lens="radtan"):
        return np.array([exact(p) for p in pixels]).reshape(-1, 6), np.zeros(len(sizes))

    monkeypatch.setattr(initialiser, "pnp_targets", pnp_targets)
    monkeypatch.setattr(initialiser, "pnp_batch", pnp_batch)


def _frames(tag_lists):
    return [[(t, 0.1 if t >= 20 else 0.09, np.array([n, t, 0, 0, 0, 0, 0, 0], float)) for t in tags]
            for n, tags in enumerate(tag_lists)]


def test_group_entities_orders_by_first_detection():
    fr = _frames([[21, 2, 13, 0, 20, 11, 3]])[0]
    ents = initialiser.group_entities(fr, SLOT)
    assert ents == [(("tag", 21), [0]), (("target", 0), [1, 3, 6]), (("target", 1), [2, 5]), (("tag", 20), [4])]


def _expected(ents, views, world_tag):
    """Every pose re-expressed in the frame of the world tag."""
    g_T_w = ents[_key(world_tag)]
    if world_tag in SLOT:
        g_T_w = compose(g_T_w, initialiser.board_T_tag(CORNERS[SLOT[world_tag][1]]))
    w_T_g = invert(g_T_w)
    return {k: compose(w_T_g, v) for k, v in ents.items()}, [compose(w_T_g, v) for v in views]


def _check(scene, tag_ids, keep, tag_pose, boards, ents, views, world_tag, expect_keep):
    exp_e, exp_v = _expected(ents, views, world_tag)
    assert list(keep) == expect_keep
    assert tag_ids[0] == world_tag
    for v, n in enumerate(keep):
        assert np.abs(scene.views[v] - exp_v[n]).max() < 1e-12
    assert scene.const_markers[0] and not scene.const_markers[1:].any()
    per_tag = tag_pose(scene.markers)
    for j, t in enumerate(tag_ids):
        want = exp_e[_key(t)] if t not in SLOT else compose(exp_e[_key(t)], initialiser.board_T_tag(CORNERS[SLOT[t][1]]))
        assert np.abs(per_tag[j] - want).max() < 1e-12, t
    # the scene carries the layout: slot of each block, -1 for free tags, and the marker of its entity
    for b in range(scene.n_blocks):
        n, t = int(scene.pixels[b][0]), int(scene.pixels[b][1])
        assert n == keep[scene.view_idx[b]]
        assert scene.corner_slot[b] == (SLOT[t][1] if t in SLOT else -1)
        assert np.abs(scene.markers[scene.marker_idx[b]] - exp_e[_key(t)]).max() < 1e-12
    assert boards == sorted(boards)                         # in target order
    return per_tag


def test_board_as_world_entity(monkeypatch):
    ents, views = _truth(np.random.default_rng(1))
    _fake_pnp(monkeypatch, ents, views)
    tag_lists = [[2, 20, 0, 3], [21, 1], [11, 20], [12, 21, 10], [3, 13]]
    scene, ids, keep, tag_pose, boards = initialiser.initialise_targets(_frames(tag_lists), np.ones(4), np.zeros(5),
                                                                        TARGETS)
    per_tag = _check(scene, ids, keep, tag_pose, boards, ents, views, 2, [0, 1, 2, 3, 4])
    # the world board's pose is invert(board_T_tag) of the world tag, so the world tag sits at the identity
    assert np.abs(scene.markers[0] - invert(initialiser.board_T_tag(CORNERS[2]))).max() < 1e-15
    assert np.abs(per_tag[0]).max() < 1e-15
    assert boards == [(0, 0), (10, 3)]                     # chained as board 0, tag 20, tag 21, board 1
    assert scene.markers.shape == (4, 6) and scene.corners.shape == (8, 4, 2)


def test_free_tag_as_world_entity(monkeypatch):
    ents, views = _truth(np.random.default_rng(2))
    _fake_pnp(monkeypatch, ents, views)
    tag_lists = [[20, 1, 2], [0, 13, 21], [21, 12]]
    scene, ids, keep, tag_pose, boards = initialiser.initialise_targets(_frames(tag_lists), np.ones(4), np.zeros(5),
                                                                        TARGETS)
    _check(scene, ids, keep, tag_pose, boards, ents, views, 20, [0, 1, 2])
    assert np.abs(scene.markers[0]).max() == 0.0
    assert list(ids) == [20, 0, 1, 2, 12, 13, 21]          # by entity in chaining order, then by slot
    assert boards == [(0, 1), (10, 2)]


def test_deferred_frame_resolved_through_a_board(monkeypatch):
    ents, views = _truth(np.random.default_rng(3))
    _fake_pnp(monkeypatch, ents, views)
    # frame 1 sees board 1 and tag 21, both unknown: deferred.  Frame 2 links board 0 -> board 1 through two
    # different tags of board 1 than frame 1 saw, and frame 1 is then resolved through board 1.  Frame 3 never links.
    ents[("tag", 30)] = np.zeros(6)
    tag_lists = [[0, 3], [13, 21], [1, 10], [], [30]]
    scene, ids, keep, tag_pose, boards = initialiser.initialise_targets(_frames(tag_lists), np.ones(4), np.zeros(5),
                                                                        TARGETS)
    _check(scene, ids, keep, tag_pose, boards, ents, views, 0, [0, 1, 2])
    assert 30 not in ids and 21 in ids


def test_last_known_entity_wins(monkeypatch):
    # frame 2 knows board 0 and tag 20 (the world tag is absent): the last known entity is the reference; with exact
    # poses both give the same camera, so check that the chaining reaches everything through either
    ents, views = _truth(np.random.default_rng(4))
    _fake_pnp(monkeypatch, ents, views)
    tag_lists = [[21, 0], [20, 21], [1, 20, 12]]
    scene, ids, keep, tag_pose, boards = initialiser.initialise_targets(_frames(tag_lists), np.ones(4), np.zeros(5),
                                                                        TARGETS)
    _check(scene, ids, keep, tag_pose, boards, ents, views, 21, [0, 1, 2])


# ------------------------------------------------------------------ read_detections and the command line
def test_read_detections_numeric_order_sizes_and_integer_pixels(tmp_path):
    d = str(tmp_path)
    c = np.arange(8).reshape(1, 4, 2)
    with open(os.path.join(d, "detections_10.yaml"), "w") as f:
        f.write(io_yaml.detections_text([7], [0.05], c) + io_yaml.world_T_camera_text([1, 2, 3], [4, 5, 6]))
    with open(os.path.join(d, "detections_2.yaml"), "w") as f:
        f.write(io_yaml.detections_text([3, 4], [0.1, 0.2], np.concatenate([c, c + 100])))
    with open(os.path.join(d, "detections_3.yaml"), "w") as f:
        f.write("detections:\n - targetID: 5\n   size: [ 0.3, 0.3 ]\n   corners:\n"
                + "".join(f"    {k}: [ {k}.5, {k}.25 ]\n" for k in range(4)))
    with open(os.path.join(d, "detections_4.yaml"), "w") as f:
        f.write("detections:\n")
    numbers, frames = io_yaml.read_detections(d)
    assert list(numbers) == [2, 3, 4, 10]
    assert [[(t, s) for t, s, _ in fr] for fr in frames] == [[(3, 0.1), (4, 0.2)], [(5, 0.3)], [], [(7, 0.05)]]
    assert frames[0][1][2].dtype == np.int64 and list(frames[0][1][2]) == list(range(100, 108))
    assert frames[1][0][2].dtype == np.float64 and frames[1][0][2][0] == 0.5
    assert io_yaml._integer_pixels(np.array([[1.0] * 8]), [frames[0]]).dtype == np.int16
    assert io_yaml._integer_pixels(np.array([[1.0] * 8]), frames[:2]).dtype == np.float64


def test_initialise_flag_combines_with_targets_and_intrinsics_options():
    a = parser().parse_args(["d", "--initialise", "--target", "a.yaml", "--target", "b.yaml", "--fix-intrinsics"])
    assert a.initialise and a.target == ["a.yaml", "b.yaml"] and a.fix_intrinsics
    a = parser().parse_args(["d", "--initialise", "--intrinsics-sigma", "1", "2", "0.1"])
    assert a.initialise and a.intrinsics_sigma == [1.0, 2.0, 0.1]
    assert not parser().parse_args(["d"]).initialise


def test_initialise_is_passed_to_optimise_directory(monkeypatch):
    seen = {}

    def fake(directory, **kw):
        seen.update(kw, directory=directory)
        return {"termination": 1}
    monkeypatch.setattr(io_yaml, "optimise_directory", fake)
    assert main(["somewhere", "--initialise", "--target", "g.yaml", "--fix-intrinsics"]) == 0
    assert seen["initialise"] and seen["targets"] == ["g.yaml"] and not seen["refine_intrinsics"]
    assert main(["somewhere"]) == 0 and not seen["initialise"]


def _detections_only(d):
    with open(os.path.join(d, "detections_0.yaml"), "w") as f:
        f.write(io_yaml.detections_text([0, 1], [0.1, 0.1], np.arange(16).reshape(2, 4, 2)))


def test_initialise_exit_codes(tmp_path, capsys):
    d = str(tmp_path)
    _detections_only(d)
    # no camera.yaml (and no targets.yaml, which --initialise never needs): status 2
    assert main([d, "--initialise"]) == 2
    assert "camera.yaml" in capsys.readouterr().err
    with open(os.path.join(d, "camera.yaml"), "w") as f:
        f.write(io_yaml.camera_yaml_text([500, 500, 320, 240], [0, 0, 0, 0, 0]))
    bad = os.path.join(d, "bad.yaml")
    with open(bad, "w") as f:
        f.write("target_type: checkerboard\n")
    assert main([d, "--initialise", "--target", bad]) == 2
    assert "aprilgrid" in capsys.readouterr().err
    g1, g2 = os.path.join(d, "g1.yaml"), os.path.join(d, "g2.yaml")
    for g in (g1, g2):
        with open(g, "w") as f:
            f.write("target_type: aprilgrid\ntagRows: 2\ntagCols: 2\ntagSize: 0.1\ntagSpacing: 0.3\n")
    assert main([d, "--initialise", "--target", g1, "--target", g2]) == 2
    assert "two targets" in capsys.readouterr().err
    # an empty first frame defines no world: status 2
    with open(os.path.join(d, "detections_0.yaml"), "w") as f:
        f.write("detections:\n")
    assert main([d, "--initialise"]) == 2
    assert "world" in capsys.readouterr().err
    with pytest.raises(SystemExit) as e:
        main([d, "--initialise", "--fix-intrinsics", "--intrinsics-sigma", "1", "1", "1"])
    assert e.value.code == 2


# ------------------------------------------------------------------ coverage of the kernel's instantiations
PNP_TARGET_LENSES = {0: "radtan", 1: "equidistant"}      # what tests/test_gpu_pnp_targets.py launches, per lens


def compiled_pnp_target_lenses():
    """The Lens arguments of the pnp_target_kernel instantiations in the built library (cuobjdump -symbols, cu++filt:
    no GPU needed)."""
    import re
    import subprocess
    from robot_camera_calibration_b200 import _build
    bin_dir = os.path.dirname(_build.NVCC)
    syms = subprocess.run([os.path.join(bin_dir, "cuobjdump"), "-symbols", L.LIB_PATH], capture_output=True,
                          text=True, check=True).stdout
    mangled = [line.split()[-1] for line in syms.splitlines() if "STO_ENTRY" in line]
    names = subprocess.run([os.path.join(bin_dir, "cu++filt")], input="\n".join(mangled) + "\n", capture_output=True,
                           text=True, check=True).stdout.splitlines()
    pat = re.compile(r"\brcc::pnp_target_kernel<(?:\(rcc::Lens\))?(\d+)>")
    return sorted(int(m.group(1)) for m in map(pat.search, names) if m)


def test_every_pnp_target_instantiation_is_launched_by_a_gpu_test():
    assert compiled_pnp_target_lenses() == sorted(PNP_TARGET_LENSES)
