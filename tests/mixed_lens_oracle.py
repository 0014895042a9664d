"""CPU oracle for a problem whose cameras mix lenses.  TEST INFRASTRUCTURE ONLY.

``p.lens`` is a tuple of one lens name per camera.  The residuals and Jacobian blocks of the observation blocks of
each lens are tests/lens_oracle.py's for that lens (oracle A: closed form + complex step), evaluated on a
lens_oracle.LensProblem that holds those blocks only, so that camera by camera the mixed oracle is the single-lens
one.  The dense normal equations, the LM step and the Schur reduction are lens_oracle's functions evaluated with this
module's residuals and Jacobians.
"""
from __future__ import annotations

import types

import numpy as np

import ba_oracle as O
import lens_oracle as LO


class MixedProblem(LO.LensProblem):
    """LensProblem with one lens per camera.  Its constant mask holds the reserved distortion slot of the equidistant
    cameras only; the slot 4 (k3) of a radial-tangential camera stays free."""

    def _copy(self):
        return MixedProblem(self.lens, self.model, self.intr, self.dist, self.ext, self.views, self.markers,
                            self.sizes, self.view_idx, self.marker_idx, self.cam_idx, self.pixels, self.const_views,
                            self.const_markers, self.const_intr, self.const_dist,
                            self.const_ext if self.model == "rig" else None)

    def const_mask(self):
        m = O.OracleProblem.const_mask(self)
        eq = np.nonzero([lens == "equidistant" for lens in self.lens])[0]
        m[self.offsets()[2] + self.shared_per_cam * eq + 8] = True
        return m

    def of_lens(self, lens):
        """(LensProblem of the blocks whose camera has `lens`, the positions of those blocks)."""
        sel = np.nonzero(np.asarray(self.lens)[self.cam_idx] == lens)[0]
        q = LO.LensProblem(lens, self.model, self.intr, self.dist, self.ext, self.views, self.markers, self.sizes,
                           self.view_idx[sel], self.marker_idx[sel], self.cam_idx[sel], self.pixels[sel],
                           self.const_views, self.const_markers, self.const_intr, self.const_dist,
                           self.const_ext if self.model == "rig" else None)
        q.loss, q.loss_scale = self.loss, self.loss_scale
        return q, sel


def oracle_problem(s):
    """Scene with one lens per camera -> MixedProblem."""
    lens = (s.lens,) * len(s.intr) if isinstance(s.lens, str) else tuple(s.lens)
    return MixedProblem(lens, s.model, s.intr, s.dist, s.ext, s.views, s.markers, s.sizes, s.view_idx, s.marker_idx,
                        s.cam_idx, s.pixels, s.const_views, s.const_markers, s.const_intr, s.const_dist,
                        s.const_ext if s.model == "rig" else None)


def _per_lens(p, fn, shape):
    """out[positions of lens l] = fn(LensProblem of lens l), for every lens present."""
    out = np.empty((len(p.view_idx),) + shape)
    for lens in sorted(set(p.lens)):
        q, sel = p.of_lens(lens)
        if len(sel):
            out[sel] = fn(q)
    return out


def residuals(p):
    return _per_lens(p, LO.residuals, (8,))


def depths(p):
    return _per_lens(p, LO.depths, (4,))


def cost(p):
    return 0.5 * float(O.robust(p, residuals(p))[1].sum())


def jacobian_blocks_cs(p):
    """Per-block Jacobians, each block's from its camera's lens: dict name -> (N,8,k)."""
    return {name: _per_lens(p, lambda q: LO.jacobian_blocks_cs(q)[name], (8, k))
            for name, k in O.local_param_names(p.model)}


def _with_mixed_globals(f):
    """lens_oracle's function f with its global names (residuals, jacobian_blocks_cs, normal_equations, O) resolved in
    this module."""
    return types.FunctionType(f.__code__, globals(), f.__name__, f.__defaults__)


normal_equations = _with_mixed_globals(LO.normal_equations)
lm_step = _with_mixed_globals(LO.lm_step)
blocks = _with_mixed_globals(LO.blocks)
reduced = _with_mixed_globals(LO.reduced)
