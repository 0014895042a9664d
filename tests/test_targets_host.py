"""CPU: the corner layout of rigid targets -- the board geometry, the target scene generator, and that the target
instantiations of K1, K2 and K6 in the built library are exactly the ones the cells of test_gpu_targets.py launch."""
import hashlib
import os
import subprocess

import numpy as np
import pytest

from robot_camera_calibration_b200 import _build
from robot_camera_calibration_b200 import _lib as L
from robot_camera_calibration_b200.scenes import board_layout, make_scene, make_target_scene
from test_gpu_kernel_matrix import CELLS, LENS_CODE, LENS_PER_CAMERA, lenses

# one cell per model x elimination x lens set, with the trivial loss and a robust one: the LOSS template parameter
# of K2 takes both values in every other combination
TARGET_CELLS = [c for c in CELLS if c[3] in ("trivial", "huber")]
_TARGET_KERNEL = {"assemble_kernel": "assemble_target_kernel", "materialise_kernel": "materialise_target_kernel",
                  "evaluate_kernel": "evaluate_target_kernel"}


def expected_target_kernels(model, elim, lens_set, loss):
    """The target instantiations a cell with a corner layout launches: those of test_gpu_kernel_matrix's
    expected_kernels under the target names, with the same template arguments."""
    from test_gpu_kernel_matrix import expected_kernels
    return {(_TARGET_KERNEL[k], args) for k, args in expected_kernels(model, elim, lens_set, loss)}


def square_layout(s):
    """A layout with one slot per marker holding the square of its size (the same doubles as the kernels' own
    corners), slot = the block's marker."""
    h = np.asarray(s.sizes, dtype=np.float64) / 2
    corners = np.stack([np.stack([-h, -h], -1), np.stack([h, -h], -1), np.stack([h, h], -1),
                        np.stack([-h, h], -1)], 1)
    return corners, np.asarray(s.marker_idx, dtype=np.int32)


def test_board_layout_geometry():
    c = board_layout(2, 3, 0.1, 0.3)
    assert c.shape == (6, 4, 2)
    np.testing.assert_allclose(c[0, 0], [0.0, 0.0], atol=1e-15)                 # bottom-left corner of tag 0
    np.testing.assert_allclose(c[0, 2], [0.1, 0.1])                             # its top-right
    np.testing.assert_allclose(c[1].mean(0), [1.3 * 0.1 + 0.05, 0.05])          # tag (0, 1)
    np.testing.assert_allclose(c[3].mean(0), [0.05, 1.3 * 0.1 + 0.05])          # tag (1, 0)
    side = np.linalg.norm(np.diff(c[:, [0, 1, 2, 3, 0]], axis=1), axis=-1)
    np.testing.assert_allclose(side, 0.1)


def test_target_scene_is_deterministic_and_consistent():
    kw = dict(rows=4, cols=5, n_views=12, n_boards=2, n_free=5, n_cam=3, model="rig", seed=4,
              lens=("equidistant", "radtan", "equidistant"))
    a, b = make_target_scene(**kw), make_target_scene(**kw)
    for k in ("views", "markers", "intr", "dist", "ext", "pixels", "view_idx", "marker_idx", "cam_idx", "corners",
              "corner_slot"):
        assert np.array_equal(getattr(a, k), getattr(b, k)), k
    assert a.corners.shape == (20, 4, 2)
    assert a.corner_slot.dtype == np.int32 and len(a.corner_slot) == a.n_blocks
    board = a.marker_idx < 2
    assert (a.corner_slot[board] >= 0).all() and (a.corner_slot[~board] == -1).all()
    assert (~board).any() and len(set(a.cam_idx)) == 3
    assert a.const_markers[0] and not a.const_markers[1:].any()


def test_make_scene_is_unchanged():
    """make_scene's random streams are untouched by the target generator: the same arrays as before it existed."""
    h = hashlib.sha256()
    for kw in (dict(n_markers=12, n_views=30, visibility=0.7, seed=11),
               dict(n_markers=30, n_views=40, visibility=0.5, n_cam=3, model="rig", seed=5,
                    lens=("equidistant", "radtan", "equidistant"))):
        s = make_scene(**kw)
        assert s.corners is None and s.corner_slot is None
        for a in (s.intr, s.dist, s.ext, s.views, s.markers, s.sizes, s.view_idx, s.marker_idx, s.cam_idx, s.pixels):
            h.update(np.ascontiguousarray(a).tobytes())
    assert h.hexdigest() == "6e6295764aecfc00fbd02d41f88df03725c33a054e82f9b1a56d6b8c5dfb3cc5"


def test_every_target_instantiation_has_a_cell():
    """The target kernels in the built library (cuobjdump -symbols, cu++filt) are exactly those the cells of
    test_gpu_targets.py launch, and there is one for every plain K1, K2 and K6 instantiation."""
    import re
    from test_gpu_kernel_matrix import _template_arg
    bin_dir = os.path.dirname(_build.NVCC)
    syms = subprocess.run([os.path.join(bin_dir, "cuobjdump"), "-symbols", L.LIB_PATH], capture_output=True,
                          text=True, check=True).stdout
    mangled = [line.split()[-1] for line in syms.splitlines() if "STO_ENTRY" in line]
    names = subprocess.run([os.path.join(bin_dir, "cu++filt")], input="\n".join(mangled) + "\n", capture_output=True,
                           text=True, check=True).stdout.splitlines()
    pat = re.compile(r"\brcc::(assemble_target_kernel|materialise_target_kernel|evaluate_target_kernel)<([^<>]*)>")
    compiled = set()
    for n in names:
        m = pat.search(n)
        if m:
            compiled.add((m.group(1), tuple(_template_arg(a.strip()) for a in m.group(2).split(","))))
    covered = set().union(*(expected_target_kernels(*cell) for cell in TARGET_CELLS))
    assert compiled == covered
    assert len(compiled) == 46


# ---------------------------------------------------------------------------------------------- front ends
def _write(path, text):
    with open(path, "w") as f:
        f.write(text)
    return str(path)


def test_aprilgrid_layout_and_ids(tmp_path):
    from robot_camera_calibration_b200 import io_yaml
    p = _write(tmp_path / "grid.yaml", "target_type: 'aprilgrid'\ntagCols: 3\ntagRows: 2\ntagSize: 0.088\n"
                                       "tagSpacing: 0.3\nfirstTagId: 10\n")
    ids, corners = io_yaml.read_target(p)
    assert ids.tolist() == list(range(10, 16))
    assert np.array_equal(corners, board_layout(2, 3, 0.088, 0.3))
    np.testing.assert_allclose(corners[0, 0], [0.0, 0.0], atol=1e-15)          # origin: bottom-left of the first tag
    np.testing.assert_allclose(corners[4].mean(0), [1.3 * 0.088 + 0.044, 1.3 * 0.088 + 0.044])   # id 14 = (1, 1)
    q = _write(tmp_path / "g0.yaml", "target_type: aprilgrid\ntagCols: 2\ntagRows: 2\ntagSize: 0.1\ntagSpacing: 0.2\n")
    assert io_yaml.read_target(q)[0].tolist() == [0, 1, 2, 3]                    # firstTagId defaults to 0


def test_bad_and_overlapping_targets(tmp_path):
    from robot_camera_calibration_b200 import io_yaml
    base = "tagCols: 2\ntagRows: 2\ntagSize: 0.1\ntagSpacing: 0.2\n"
    bad = {"type": "target_type: checkerboard\n" + base, "missing": "target_type: aprilgrid\ntagCols: 2\n",
           "rows": "target_type: aprilgrid\n" + base.replace("tagRows: 2", "tagRows: 0"),
           "size": "target_type: aprilgrid\n" + base.replace("tagSize: 0.1", "tagSize: -1"),
           "first": "target_type: aprilgrid\nfirstTagId: -3\n" + base}
    for k, txt in bad.items():
        with pytest.raises(ValueError):
            io_yaml.read_target(_write(tmp_path / f"{k}.yaml", txt))
    a = _write(tmp_path / "a.yaml", "target_type: aprilgrid\n" + base)                     # ids 0..3
    b = _write(tmp_path / "b.yaml", "target_type: aprilgrid\nfirstTagId: 3\n" + base)      # ids 3..6
    c = _write(tmp_path / "c.yaml", "target_type: aprilgrid\nfirstTagId: 4\n" + base)      # ids 4..7
    with pytest.raises(ValueError, match="tag id 3"):
        io_yaml.read_targets([a, b])
    assert [t[0].tolist() for t in io_yaml.read_targets([a, c])] == [[0, 1, 2, 3], [4, 5, 6, 7]]


def scene_as_tags(s, free_id0=100):
    """A single-board scene of make_target_scene as the reference's per-tag files see it: one marker per tag (board
    tags: world_T_board o board_T_tag, id = slot; free tags: id free_id0 + j), marker 0 the board's tag 0."""
    from robot_camera_calibration_b200.scenes import Scene, compose
    n_slots, n_free = len(s.corners), len(s.markers) - 1
    ctr = s.corners.mean(1)
    b_T_t = np.concatenate([np.zeros((n_slots, 3)), ctr, np.zeros((n_slots, 1))], 1)
    markers = np.concatenate([compose(np.broadcast_to(s.markers[0], (n_slots, 6)), b_T_t), s.markers[1:]])
    tag = np.where(s.corner_slot >= 0, s.corner_slot, n_slots + s.marker_idx - 1).astype(np.int32)
    t = Scene(model="single", intr=s.intr, dist=s.dist, ext=s.ext, views=s.views, markers=markers,
              sizes=np.full(n_slots + n_free, s.sizes[0]), view_idx=s.view_idx, marker_idx=tag, cam_idx=s.cam_idx,
              pixels=s.pixels, lens=s.lens, image_size=s.image_size)
    return t, np.concatenate([np.arange(n_slots), free_id0 + np.arange(n_free)])


def test_board_scene_maps_tags_onto_the_board():
    from robot_camera_calibration_b200 import io_yaml
    s = make_target_scene(3, 4, 10, n_free=3, seed=2)
    tags, ids = scene_as_tags(s)
    bs, tag_pose, boards = io_yaml.board_scene(tags, ids, [(np.arange(12), board_layout(3, 4, 0.1, 0.3))])
    assert boards == [(0, 0)] and len(bs.markers) == 1 + 3
    assert np.array_equal(bs.corner_slot, s.corner_slot) and np.array_equal(bs.marker_idx, s.marker_idx)
    assert bs.const_markers.tolist() == [True, False, False, False]     # the board carries the world tag
    np.testing.assert_allclose(bs.markers, s.markers, atol=1e-12)       # tag poses of one rigid board: exact pose
    np.testing.assert_allclose(tag_pose(bs.markers), tags.markers, atol=1e-12)


def test_ceres_like_deduplicates_corner_sets():
    from robot_camera_calibration_b200.ceres_like import corner_layout
    a, b = board_layout(1, 2, 0.1, 0.3)
    table, slot = corner_layout([a, None, b, a.copy(), None, b])
    assert slot.tolist() == [0, -1, 1, 0, -1, 1]
    assert np.array_equal(table, np.stack([a, b]))
    table, slot = corner_layout([None, None])
    assert table.shape == (0, 4, 2) and slot.tolist() == [-1, -1]


def _shard_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    from robot_camera_calibration_b200.dist import shard_scene
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    s = make_target_scene(3, 4, 16, n_free=4, seed=9)
    local, (lo, hi) = shard_scene(s, rank, world, eliminate="views")
    keep = (s.view_idx >= lo) & (s.view_idx < hi)
    ok = (len(local.corner_slot) == local.n_blocks and np.array_equal(local.corner_slot, s.corner_slot[keep])
          and local.corners is s.corners)
    t = torch.tensor([int(ok), local.n_blocks, int((local.corner_slot >= 0).sum())])
    dist.all_reduce(t)
    if rank == 0:
        q.put((t.tolist(), s.n_blocks, int((s.corner_slot >= 0).sum())))
    dist.destroy_process_group()


def test_shard_scene_carries_the_slots_under_gloo():
    """Two ranks over gloo: each shard keeps the slots of its own blocks and the whole corner table."""
    import torch.multiprocessing as mp
    from test_dist_gloo import _free_port
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_shard_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    (ok, n_sum, n_board), n_all, n_board_all = q.get(timeout=240)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert ok == 2 and n_sum == n_all and n_board == n_board_all
