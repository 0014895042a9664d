"""GPU: every compiled instantiation of the three kernels that evaluate the cost functor -- K2 assemble_kernel, K1
materialise_kernel and K6 evaluate_kernel -- against the oracle of tests/prior_oracle.py (no priors), one case per
cell of model x elimination x lens set x loss, with the tolerances of test_gpu_mixed_lens.py.

Each case runs under torch.profiler and checks that it launched exactly the instantiations its cell selects
(`expected_kernels`); test_every_compiled_instantiation_has_a_cell checks, without a GPU, that those cells together
select every instantiation in the built library.  So every instantiation runs in some oracle case, and a new lens or
template parameter fails that test until a cell covers it.

The scenes put the chunk boundaries where the kernels go wrong: in both elimination directions an eliminated block
with more than 64 observation blocks of one camera (its row spans several chunks of the E pass), last groups of every
size from 1 to 7, and blocks on both sides of the loss threshold in full and in partial last groups."""
import contextlib
import os
import re
import subprocess
from functools import lru_cache

import numpy as np
import pytest
from torch.profiler import ProfilerActivity, profile

import ba_oracle as O
import mixed_lens_oracle as MO
import prior_oracle as PO
from helpers import max_block_rel, rel_fro
from robot_camera_calibration_b200 import _build
from robot_camera_calibration_b200 import _lib as L
from robot_camera_calibration_b200.problem import BAProblem
from robot_camera_calibration_b200.scenes import make_scene
from test_gpu_mixed_lens import _compact

TOL = 1e-9          # K1, K2, K6, the costs and the reduced system
STEP_TOL = 1e-6     # the step, its model cost change and the candidate cost
RADIUS = 1e4
CHUNK = 64          # observation blocks per chunk at most (problem.cu: build_indices)
BPW = 8             # observation blocks per warp iteration (kernels.h: PassGeom::BPW)

N_CAM = {"single": 2, "rig": 3}
LENS_SETS = ("radtan", "equidistant", "mixed")
LOSSES = ("trivial", "huber", "cauchy")
CELLS = [(model, elim, lens_set, loss) for model in N_CAM for elim in ("views", "markers") for lens_set in LENS_SETS
         for loss in LOSSES]
LENS_CODE = {"radtan": 0, "equidistant": 1}     # model.cuh: Lens
LENS_PER_CAMERA = 2


def lenses(model, lens_set):
    if lens_set != "mixed":
        return (lens_set,) * N_CAM[model]
    return ("radtan", "equidistant") if model == "single" else ("equidistant", "radtan", "equidistant")


def expected_kernels(model, elim, lens_set, loss):
    """The K1, K2 and K6 instantiations a cell launches, as (kernel, template arguments):
    assemble_kernel<RIG, EPASS, OWN_IS_VIEW, LOSS, lens>: the E pass owns the eliminated blocks, the F pass the kept
    ones, once per lens among the cameras; materialise_kernel<RIG, OWN_IS_VIEW, lens> walks the E chunks, once per
    lens; evaluate_kernel<RIG, lens> takes the common lens, or LENS_PER_CAMERA when the cameras differ."""
    rig, ev, robust = int(model == "rig"), int(elim == "views"), int(loss != "trivial")
    codes = sorted({LENS_CODE[x] for x in lenses(model, lens_set)})
    out = {("evaluate_kernel", (rig, codes[0] if len(codes) == 1 else LENS_PER_CAMERA))}
    for lens in codes:
        out |= {("assemble_kernel", (rig, 1, ev, robust, lens)), ("assemble_kernel", (rig, 0, 1 - ev, robust, lens)),
                ("materialise_kernel", (rig, ev, lens))}
    return out


_KERNEL = re.compile(r"\brcc::(assemble_kernel|materialise_kernel|evaluate_kernel)<([^<>]*)>")
_NAMED = {"true": 1, "false": 0, "rcc::LENS_RADTAN": 0, "rcc::LENS_EQUIDISTANT": 1, "rcc::LENS_PER_CAMERA": 2}


def _template_arg(a):
    if a in _NAMED:
        return _NAMED[a]
    m = re.fullmatch(r"(?:\([\w:]+\))?(\d+)", a)         # cu++filt: (bool)1, (rcc::Lens)1
    if not m:
        raise ValueError(f"unrecognised template argument {a!r}")
    return int(m.group(1))


def instantiation(name):
    """Demangled kernel name -> (kernel, template arguments as ints) for K1, K2 and K6, None for any other name.  The
    profiler prints `true`, cu++filt `(bool)1`."""
    m = _KERNEL.search(name)
    if not m:
        return None
    return m.group(1), tuple(_template_arg(a.strip()) for a in m.group(2).split(","))


@pytest.fixture
def kernels_launched():
    """`with kernels_launched() as got:` runs the body under torch.profiler with CUDA activities; on exit `got` holds
    the instantiation of every K1, K2 and K6 kernel launched inside it, from the library's own streams included."""
    @contextlib.contextmanager
    def record():
        got = set()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            yield got
        got.update(k for k in (instantiation(e.name) for e in prof.events()) if k)
    return record


# ---------------------------------------------------------------------------------------------- scenes
def e_chunks(s, elim_view):
    """The E-pass chunks of problem.cu (sort_by_owner, make_chunks), each as the positions of its blocks in walk
    order: blocks sorted by (eliminated block, camera, other block), every (eliminated block, camera) run cut into
    the fewest chunks of at most CHUNK blocks, all but the last a multiple of BPW long."""
    own, oth = (s.view_idx, s.marker_idx) if elim_view else (s.marker_idx, s.view_idx)
    order = np.lexsort((np.arange(s.n_blocks), oth, s.cam_idx, own))
    key = own[order].astype(np.int64) * len(s.intr) + s.cam_idx[order]
    starts = np.flatnonzero(np.diff(key, prepend=-1))
    out = []
    for a, b in zip(starts, np.append(starts[1:], s.n_blocks)):
        n_chunks = -(-(b - a) // CHUNK)
        per = -(-(-(-(b - a) // n_chunks)) // BPW) * BPW
        out += [order[k:min(k + per, b)] for k in range(a, b, per)]
    return out


@lru_cache(maxsize=None)
def _scene(model, lens_set):
    """(scene, loss scale).  Every camera keeps every block of its busiest view and of its busiest marker (more than
    64 in one direction at least); of the other blocks a random 8 %.  4 % of the blocks get 25 px outliers.  The loss
    scale splits the blocks in half: s = ||r||^2 above and below a^2."""
    n_cam = N_CAM[model]
    s = make_scene(80, 90, 0.9, n_cam=n_cam, model=model, seed=29 + n_cam, lens=lenses(model, lens_set))
    rng = np.random.default_rng(41)
    keep = rng.random(s.n_blocks) < 0.08
    for own in (s.view_idx, s.marker_idx):
        key = own.astype(np.int64) * n_cam + s.cam_idx
        cnt = np.bincount(key, minlength=(own.max() + 1) * n_cam).reshape(-1, n_cam)
        for c in range(n_cam):
            keep |= key == cnt[:, c].argmax() * n_cam + c
    s.view_idx, s.marker_idx, s.cam_idx, s.pixels = s.view_idx[keep], s.marker_idx[keep], s.cam_idx[keep], s.pixels[keep]
    s = _compact(s)
    bad = rng.choice(s.n_blocks, s.n_blocks // 25, replace=False)
    s.pixels[bad] += rng.normal(0, 25.0, (len(bad), 8))
    fish = np.array([x == "equidistant" for x in lenses(model, lens_set)])
    s.dist[fish, 4] = 0.125           # the reserved slot: ignored by the projection, never stepped
    sq = (MO.residuals(MO.oracle_problem(s)) ** 2).sum(1)
    mid = np.sort(sq)[len(sq) // 2 - 1:len(sq) // 2 + 1]
    a2 = float(mid.mean())
    above = sq > a2
    for ev in (True, False):
        chunks = e_chunks(s, ev)
        lengths = np.array([len(c) for c in chunks])
        assert lengths.sum() == s.n_blocks
        own = s.view_idx if ev else s.marker_idx
        assert np.bincount(own.astype(np.int64) * n_cam + s.cam_idx).max() > CHUNK, (model, lens_set, ev)
        assert set(range(1, BPW)) <= set(lengths % BPW), (model, lens_set, ev)
        full = np.concatenate([c[:len(c) // BPW * BPW] for c in chunks])
        last = np.concatenate([c[len(c) // BPW * BPW:] for c in chunks])
        for part in (full, last):
            assert above[part].any() and (~above[part]).any(), (model, lens_set, ev)
    return s, float(np.sqrt(a2))


# ---------------------------------------------------------------------------------------------- the matrix
def _errors(model, elim, lens_set, loss, kernels_launched):
    """Run the cell on the GPU and against the oracle: (launched instantiations, {quantity: error}, reserved-slot
    checks)."""
    s, scale = _scene(model, lens_set)
    ev = elim == "views"
    fish = np.array([x == "equidistant" for x in lenses(model, lens_set)])
    p = MO.oracle_problem(s)
    if loss != "trivial":
        p.loss, p.loss_scale = loss, scale
    with kernels_launched() as launched:
        with BAProblem.from_scene(s, eliminate=elim) as gp:
            if loss != "trivial":
                gp.set_loss(loss, scale)
            k1 = gp.evaluate()
            k6 = gp.evaluate(want_jacobians=False)
            cost = gp.linearize()
            nb = gp.normal_blocks()
            gp.schur(RADIUS)
            Sg, bg = gp.reduced_system()
            mcc, _, _ = gp.solve_step()
            st = gp.step()
            c_new = gp.candidate_cost()

    r, Jb = MO.residuals(p), MO.jacobian_blocks_cs(p)
    c_ref = PO.cost(p, {})
    rel = lambda a, b: abs(a - b) / abs(b)
    err = {"K1 residuals": max_block_rel(k1["residuals"], r),
           "K1 jacobians": max(max_block_rel(k1["jacobians"][k], Jb[k]) for k in Jb),
           "K1 cost": rel(k1["cost"], c_ref),
           "K6 residuals": max_block_rel(k6["residuals"], r),
           "K6 cost": rel(k6["cost"], c_ref),
           "K2 cost": rel(cost, c_ref)}
    ob = PO.blocks(p, {}, ev)
    w, _ = O.robust(p, r)
    Je, Jf = (Jb["view"], Jb["marker"]) if ev else (Jb["marker"], Jb["view"])
    ob["W"] = np.einsum('nri,nrj->nij', Je, Jf) * (w * w)[:, None, None]
    for k in ("Hee", "ge", "Hes", "Hff", "gf", "Hfs", "W"):
        err["K2 " + k] = max_block_rel(nb[k], ob[k], floor=1e-6 * np.abs(ob[k]).max())
    err["K2 Hss"], err["K2 gs"] = rel_fro(nb["Hss"], ob["Hss"]), rel_fro(nb["gs"], ob["gs"])
    S, b = PO.reduced(p, {}, ev, RADIUS)
    err["S"], err["b"] = rel_fro(Sg, S), rel_fro(bg, b)
    delta, mcc_o, _, _ = PO.lm_step(p, {}, RADIUS)
    o_view, o_marker, o_shared, _ = p.offsets()
    dv, dm = delta[o_view:o_marker].reshape(-1, 6), delta[o_marker:o_shared].reshape(-1, 6)
    de, df = (dv, dm) if ev else (dm, dv)
    err["step"] = max(rel_fro(st["d_e"], de), rel_fro(st["d_f"], df), rel_fro(st["d_shared"], delta[o_shared:]))
    err["model cost change"] = rel(mcc, mcc_o)
    cand = p.copy()
    cand.unpack(p.pack() + delta)
    err["candidate cost"] = rel(c_new, PO.cost(cand, {}))
    eq = fish[s.cam_idx]
    slots = {"K1 reserved slot": k1["jacobians"]["dist"][eq][..., 4],
             "step reserved slot": st["d_shared"][p.shared_per_cam * np.flatnonzero(fish) + 8]}
    return launched, err, slots


@pytest.mark.gpu
@pytest.mark.parametrize("model,elim,lens_set,loss", CELLS)
def test_cell_matches_oracle(model, elim, lens_set, loss, kernels_launched):
    launched, err, slots = _errors(model, elim, lens_set, loss, kernels_launched)
    assert launched == expected_kernels(model, elim, lens_set, loss)
    for k, e in err.items():
        assert e < (STEP_TOL if k in ("step", "model cost change", "candidate cost") else TOL), (k, e)
    for k, v in slots.items():
        assert np.all(v == 0.0), k


def test_every_compiled_instantiation_has_a_cell():
    """The K1, K2 and K6 kernels in the built library (cuobjdump -symbols, demangled by cu++filt: no GPU needed) are
    exactly the instantiations the cells of test_cell_matches_oracle launch."""
    bin_dir = os.path.dirname(_build.NVCC)
    syms = subprocess.run([os.path.join(bin_dir, "cuobjdump"), "-symbols", L.LIB_PATH], capture_output=True,
                          text=True, check=True).stdout
    mangled = [line.split()[-1] for line in syms.splitlines() if "STO_ENTRY" in line]
    names = subprocess.run([os.path.join(bin_dir, "cu++filt")], input="\n".join(mangled) + "\n", capture_output=True,
                           text=True, check=True).stdout.splitlines()
    assert len(names) == len(mangled)
    compiled = {k for k in map(instantiation, names) if k}
    covered = set().union(*(expected_kernels(*cell) for cell in CELLS))
    assert {k for k, _ in compiled} == {"assemble_kernel", "materialise_kernel", "evaluate_kernel"}
    assert compiled - covered == set(), "instantiations no cell launches"
    assert covered - compiled == set(), "cells expect instantiations the library does not have"
