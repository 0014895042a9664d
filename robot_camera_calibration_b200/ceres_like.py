"""Python mirror of the Ceres interface the hot path stands behind (SURVEY 8b).

Same names, argument meaning and error behaviour as the published Ceres API
(external; the reference snapshot never calls it -- see DESIGN.md section 1):

    problem = Problem()
    problem.AddResidualBlock(TagReprojectionCost(pixels8, tag_size), None, intr, dist, view, marker)
    problem.SetParameterBlockConstant(marker0)              # gauge, camera_pose.cpp:71-80
    summary = Solve(SolverOptions(max_num_iterations=50), problem)   # refines the arrays in place

Parameter blocks are numpy float64 arrays that the caller owns (Ceres: `double*`);
a block is identified by the array object, and `Solve` writes the refined values
back into the same arrays.  All evaluation runs in librcc_ba.so on the GPU: the
residual blocks are batched into one `BAProblem` (the EvaluationCallback pattern
of INTEGRATION.md section 3); nothing is computed in Python.
"""
from __future__ import annotations

import numpy as np

from . import _lib as L
from .problem import BAProblem


class TagReprojectionCost:
    """CostFunction of one detected tag: 8 residuals (4 corners x (u,v)), parameter
    blocks intr[4], dist[5], view[6], marker[6] (+ ext[6] in a rig)."""

    def __init__(self, pixels, tag_size, rig=False):
        self.pixels = np.ascontiguousarray(pixels, dtype=np.float64).reshape(8)
        self.tag_size = float(tag_size)
        self.rig = bool(rig)

    def num_residuals(self):
        return 8

    def parameter_block_sizes(self):
        return [4, 5, 6, 6] + ([6] if self.rig else [])

    def Evaluate(self, parameters, residuals, jacobians):
        """bool Evaluate(double const* const* parameters, double* residuals, double** jacobians).
        `jacobians` may be None; `jacobians[i]` may be None; otherwise it is filled
        row-major (8 x block_size_i).  Returns False on evaluation failure."""
        intr, dist, view, marker = parameters[:4]
        ext = parameters[4] if self.rig else None
        with BAProblem(1, 1, 1, 1, model="rig" if self.rig else "single") as p:
            p.set_intrinsics(intr, dist)
            if self.rig:
                p.set_rig_extrinsics(ext)
            p.set_view_poses(view)
            p.set_marker_poses(marker)
            p.set_marker_sizes([self.tag_size])
            p.set_observations([0], [0], [0], self.pixels)
            out = p.evaluate(want_jacobians=jacobians is not None, allow_failure=True)
        residuals[:] = out["residuals"].reshape(8)
        if jacobians is not None:
            names = ["intr", "dist", "view", "marker"] + (["ext"] if self.rig else [])
            for j, n in zip(jacobians, names):
                if j is not None:
                    np.asarray(j).reshape(-1)[:] = out["jacobians"][n].reshape(-1)
        return not out["failed"]


class HuberLoss:
    """ceres::HuberLoss(a): rho(s) = s for s <= a^2, 2 a sqrt(s) - a^2 beyond."""
    kind = "huber"

    def __init__(self, a):
        self.a = float(a)


class CauchyLoss:
    """ceres::CauchyLoss(a): rho(s) = a^2 log(1 + s / a^2)."""
    kind = "cauchy"

    def __init__(self, a):
        self.a = float(a)


class SolverOptions:
    def __init__(self, max_num_iterations=50, initial_trust_region_radius=1e4, max_trust_region_radius=1e16,
                 min_relative_decrease=1e-3, function_tolerance=1e-6, gradient_tolerance=1e-10,
                 parameter_tolerance=1e-8, min_lm_diagonal=1e-6, max_lm_diagonal=1e32,
                 minimizer_progress_to_stdout=False, jacobi_scaling=True):
        self.__dict__.update(locals())
        del self.__dict__["self"]


class Summary:
    def __init__(self, d):
        self.__dict__.update(d)
        self.num_iterations = d["iterations"]
        self.num_successful_steps = d["accepted"]
        self.termination_type = ["NO_CONVERGENCE", "CONVERGENCE", "CONVERGENCE", "CONVERGENCE", "FAILURE"][d["termination"]]

    def BriefReport(self):
        return (f"rcc_ba report: iterations {self.num_iterations}, initial cost {self.initial_cost:.6e}, "
                f"final cost {self.final_cost:.6e}, termination {self.termination_type}")

    def IsSolutionUsable(self):
        return self.termination_type != "FAILURE"


class Problem:
    """ceres::Problem for tag-reprojection residual blocks."""

    def __init__(self, device=0, eliminate="auto"):
        self.device, self.eliminate = device, eliminate
        self._blocks = []            # (cost, intr, dist, view, marker, ext)
        self._const = set()
        self._known = {}
        self._loss = None

    # -- Ceres names --------------------------------------------------------
    def AddParameterBlock(self, values, size=None):
        a = self._check_block(values, size)
        self._known[id(a)] = a
        return a

    def AddResidualBlock(self, cost_function, loss_function, *parameter_blocks):
        key = None if loss_function is None else (loss_function.kind, loss_function.a)
        if self._blocks and key != self._loss:
            raise NotImplementedError("all residual blocks must share one loss function on this path")
        self._loss = key
        sizes = cost_function.parameter_block_sizes()
        if len(parameter_blocks) != len(sizes):
            raise ValueError(f"expected {len(sizes)} parameter blocks, got {len(parameter_blocks)}")
        blocks = [self._check_block(b, s) for b, s in zip(parameter_blocks, sizes)]
        for b in blocks:
            self._known[id(b)] = b
        self._blocks.append((cost_function, *blocks, *([None] if len(blocks) == 4 else [])))
        return len(self._blocks) - 1

    def SetParameterBlockConstant(self, values):
        if id(values) not in self._known:
            raise ValueError("parameter block not found in the problem")      # Ceres aborts here
        self._const.add(id(values))

    def SetParameterBlockVariable(self, values):
        self._const.discard(id(values))

    def NumResidualBlocks(self):
        return len(self._blocks)

    def NumResiduals(self):
        return 8 * len(self._blocks)

    def NumParameterBlocks(self):
        return len(self._known)

    def Evaluate(self):
        """-> (cost, residuals (8N,), jacobian blocks dict) like Problem::Evaluate."""
        gp, maps = self._build()
        with gp:
            out = gp.evaluate()
        return out["cost"], out["residuals"].reshape(-1), out["jacobians"]

    # -- batching -----------------------------------------------------------
    @staticmethod
    def _check_block(values, size):
        if not isinstance(values, np.ndarray) or values.dtype != np.float64 or not values.flags.c_contiguous:
            raise TypeError("parameter blocks must be C-contiguous float64 numpy arrays (Ceres: double*)")
        if size is not None and values.size != size:
            raise ValueError(f"parameter block has {values.size} values, expected {size}")
        return values

    def _build(self):
        if not self._blocks:
            raise ValueError("problem has no residual blocks")
        rig = self._blocks[0][0].rig
        views, markers, cams = {}, {}, {}
        vi, mi, ci, px, sizes = [], [], [], [], {}
        seen = {}     # id(array) -> camera key: one Ceres parameter block must belong to exactly one GPU camera
        for cost, intr, dist, view, marker, ext in self._blocks:
            if cost.rig != rig:
                raise NotImplementedError("rig and single-camera cost functions cannot be mixed in one problem")
            v = views.setdefault(id(view), (len(views), view))[0]
            m = markers.setdefault(id(marker), (len(markers), marker))[0]
            key = (id(intr), id(dist), id(ext) if ext is not None else 0)
            for arr in (intr, dist, ext):
                if arr is not None and seen.setdefault(id(arr), key) != key:
                    raise NotImplementedError(
                        "an intrinsics / distortion / extrinsics array is shared by residual blocks whose other "
                        "camera blocks differ: the GPU camera record is (intr, dist, ext) as a unit, so the shared "
                        "array would be optimised as several independent copies")
            c = cams.setdefault(key, (len(cams), intr, dist, ext))[0]
            if sizes.setdefault(m, cost.tag_size) != cost.tag_size:
                raise ValueError("one marker was given two different tag sizes")
            vi.append(v); mi.append(m); ci.append(c); px.append(cost.pixels)
        vlist = [a for _, a in sorted(views.values(), key=lambda t: t[0])]
        mlist = [a for _, a in sorted(markers.values(), key=lambda t: t[0])]
        clist = sorted(cams.values(), key=lambda t: t[0])
        gp = BAProblem(len(vlist), len(mlist), len(clist), len(vi), model="rig" if rig else "single",
                       device=self.device, eliminate=self.eliminate)
        gp.set_intrinsics(np.stack([c[1] for c in clist]), np.stack([c[2] for c in clist]))
        if rig:
            gp.set_rig_extrinsics(np.stack([c[3] for c in clist]))
        gp.set_view_poses(np.stack(vlist))
        gp.set_marker_poses(np.stack(mlist))
        gp.set_marker_sizes([sizes[m] for m in range(len(mlist))])
        gp.set_observations(vi, mi, ci, np.stack(px))
        if self._loss is not None:
            gp.set_loss(*self._loss)
        for i, a in enumerate(vlist):
            if id(a) in self._const:
                gp.set_constant("view", i)
        for i, a in enumerate(mlist):
            if id(a) in self._const:
                gp.set_constant("marker", i)
        for i, (_, intr, dist, ext) in enumerate(clist):
            if id(intr) in self._const:
                gp.set_constant("intr", i)
            if id(dist) in self._const:
                gp.set_constant("dist", i)
            if rig and id(ext) in self._const:
                gp.set_constant("ext", i)
        return gp, (vlist, mlist, clist, rig)


def Solve(options, problem):
    """ceres::Solve(options, &problem, &summary): refines the caller's arrays in place."""
    gp, (vlist, mlist, clist, rig) = problem._build()
    o = options
    with gp:
        s = gp.solve(max_iterations=o.max_num_iterations, initial_radius=o.initial_trust_region_radius,
                     max_radius=o.max_trust_region_radius, min_relative_decrease=o.min_relative_decrease,
                     function_tolerance=o.function_tolerance, gradient_tolerance=o.gradient_tolerance,
                     parameter_tolerance=o.parameter_tolerance, min_diagonal=o.min_lm_diagonal,
                     max_diagonal=o.max_lm_diagonal, verbose=int(o.minimizer_progress_to_stdout),
                     jacobi_scaling=int(o.jacobi_scaling))
        views, markers = gp.get_view_poses(), gp.get_marker_poses()
        intr, dist = gp.get_intrinsics()
        ext = gp.get_rig_extrinsics() if rig else None
    for a, v in zip(vlist, views):
        a[:] = v
    for a, v in zip(mlist, markers):
        a[:] = v
    for i, (_, ia, da, ea) in enumerate(clist):
        ia[:] = intr[i]
        da[:] = dist[i]
        if rig:
            ea[:] = ext[i]
    return Summary(s)


class CovarianceOptions:
    """ceres::Covariance::Options.  apply_loss_function=False evaluates J without the robust loss."""

    def __init__(self, apply_loss_function=True):
        self.apply_loss_function = bool(apply_loss_function)


class Covariance:
    """ceres::Covariance: blocks of (J^T J)^-1 at the problem's current parameters (rcc_ba_covariance; not scaled by
    a residual variance).  Supported pairs: (x, x) for any parameter block, and any pair of intrinsics, distortion
    or extrinsics arrays, of one camera or of two.  A constant block gives zeros."""

    def __init__(self, options=None):
        self.options = options if options is not None else CovarianceOptions()
        self._blocks = {}

    def Compute(self, covariance_blocks, problem):
        """bool Compute(covariance_blocks, problem): False when J^T J is not positive definite (rank deficient)."""
        pairs = [(a, b) for a, b in covariance_blocks]
        gp, (vlist, mlist, clist, rig) = problem._build()
        where = {}          # id(array) -> ("views" | "markers", index) or ("shared", first column)
        for i, a in enumerate(vlist):
            where[id(a)] = ("views", i)
        for i, a in enumerate(mlist):
            where[id(a)] = ("markers", i)
        sp = 15 if rig else 9
        for c, (_, intr, dist, ext) in enumerate(clist):
            where[id(intr)] = ("shared", sp * c)
            where[id(dist)] = ("shared", sp * c + 4)
            if rig:
                where[id(ext)] = ("shared", sp * c + 9)
        for a, b in pairs:
            for x in (a, b):
                if id(x) not in where:
                    raise ValueError("parameter block not found in the problem")      # Ceres aborts here
            if a is not b and (where[id(a)][0] != "shared" or where[id(b)][0] != "shared"):
                raise NotImplementedError("covariance between two different pose blocks, or a pose and a camera "
                                          "block, is not computed on this path")
        with gp:
            if not self.options.apply_loss_function:
                gp.set_loss("trivial")
            try:
                cov = gp.covariance()
            except L.RccError as e:
                if e.status == L.RCC_NOT_SPD:
                    return False
                raise
        self._blocks = {}
        for a, b in pairs:
            (ka, ia), (kb, ib) = where[id(a)], where[id(b)]
            if ka == "shared":
                blk = cov["shared"][ia:ia + a.size, ib:ib + b.size]
            else:
                blk = cov[ka][ia]
            self._blocks[(id(a), id(b))] = blk.copy()
            self._blocks[(id(b), id(a))] = blk.T.copy()
        return True

    def GetCovarianceBlock(self, a, b, out):
        """bool GetCovarianceBlock(a, b, out): out (row-major size(a) x size(b)); False for a pair Compute did not get."""
        blk = self._blocks.get((id(a), id(b)))
        if blk is None:
            return False
        np.asarray(out).reshape(-1)[:] = blk.reshape(-1)
        return True
