"""CPU oracle for Gaussian priors on parameter blocks (rcc_ba_set_priors, ceres::NormalPrior).  TEST INFRASTRUCTURE ONLY.

A prior on block x_i is the residual block A_i (x_i - mu_i).  This module appends those rows to the dense Jacobian
and residual of the tag oracle (tests/mixed_lens_oracle.py, which is oracle/ba_oracle.py camera by camera for any
lens set) and forms the normal equations, the Schur reduction, the LM step and the costs of the stacked problem.
`priors` is {kind: (index, mean (n, k), sqrt_information (n, k, k))}, kind "view" | "marker" | "intr" | "dist" | "ext".
"""
from __future__ import annotations

import numpy as np

import ba_oracle as O
import mixed_lens_oracle as MO

SIZES = {"view": 6, "marker": 6, "intr": 4, "dist": 5, "ext": 6}


def columns(p, kind, i):
    """Columns of block (kind, i) in the dense layout of OracleProblem.offsets()."""
    o_view, o_marker, o_shared, _ = p.offsets()
    if kind == "view":
        s = o_view + 6 * i
    elif kind == "marker":
        s = o_marker + 6 * i
    else:
        s = o_shared + p.shared_per_cam * i + {"intr": 0, "dist": 4, "ext": 9}[kind]
    return np.arange(s, s + SIZES[kind])


def prior_rows(p, priors, x=None):
    """(J_p, r_p): the prior rows A_i and residuals A_i (x_i - mu_i), in the order of `priors`."""
    x = p.pack() if x is None else x
    J, r = [], []
    for kind, (index, mean, A) in priors.items():
        for i, mu, a in zip(index, mean, A):
            cols = columns(p, kind, int(i))
            row = np.zeros((len(cols), len(x)))
            row[:, cols] = a
            J.append(row)
            r.append(np.asarray(a) @ (x[cols] - mu))
    if not J:
        return np.zeros((0, len(x))), np.zeros(0)
    return np.vstack(J), np.concatenate(r)


def normal_equations(p, priors):
    """H = J^T J, g = J^T r and the cost of the stacked (tag + prior) problem; constants not masked."""
    H, g, c = MO.normal_equations(p)
    Jp, rp = prior_rows(p, priors)
    return H + Jp.T @ Jp, g + Jp.T @ rp, c + 0.5 * float(rp @ rp)


def cost(p, priors):
    return MO.cost(p) + 0.5 * float(np.sum(prior_rows(p, priors)[1] ** 2))


def lm_diagonal(H, radius, jacobi=False, min_diag=1e-6, max_diag=1e32):
    """kernels.h lm_diagonal on every parameter."""
    h = np.diag(H)
    if not jacobi:
        return np.clip(h, min_diag, max_diag) / radius
    s = 1.0 / (1.0 + np.sqrt(np.maximum(h, 0.0)))
    return np.clip(h * s * s, min_diag, max_diag) / (radius * s * s)


def _layout(p, elim_view):
    o_view, o_marker, o_shared, n = p.offsets()
    nv, nm = len(p.views), len(p.markers)
    e_off, n_e = (o_view, nv) if elim_view else (o_marker, nm)
    f_off, n_f = (o_marker, nm) if elim_view else (o_view, nv)
    return e_off, n_e, f_off, n_f, o_shared, n


def blocks(p, priors, elim_view):
    """The normal-equation blocks in the library's layout (W, which the priors leave alone, is not formed)."""
    H, g, c = normal_equations(p, priors)
    e_off, n_e, f_off, n_f, o_shared, _ = _layout(p, elim_view)
    blk = lambda off, i: slice(off + 6 * i, off + 6 * i + 6)
    return {
        "Hee": np.stack([H[blk(e_off, i), blk(e_off, i)] for i in range(n_e)]),
        "ge": g[e_off:e_off + 6 * n_e].reshape(n_e, 6),
        "Hes": np.stack([H[blk(e_off, i), o_shared:] for i in range(n_e)]),
        "Hff": np.stack([H[blk(f_off, i), blk(f_off, i)] for i in range(n_f)]),
        "gf": g[f_off:f_off + 6 * n_f].reshape(n_f, 6),
        "Hfs": np.stack([H[blk(f_off, i), o_shared:] for i in range(n_f)]),
        "Hss": H[o_shared:, o_shared:], "gs": g[o_shared:], "cost": c, "H": H, "g": g,
    }


def reduced(p, priors, elim_view, radius, jacobi=False):
    """(S, b) of rcc_ba_schur: damping on the eliminated blocks only, constant eliminated blocks decoupled."""
    H, g, _ = normal_equations(p, priors)
    e_off, n_e, f_off, n_f, o_shared, n = _layout(p, elim_view)
    d2 = lm_diagonal(H, radius, jacobi)
    Hd, gd = H.copy(), g.copy()
    e_idx = np.arange(e_off, e_off + 6 * n_e)
    Hd[e_idx, e_idx] += d2[e_idx]
    ce = e_idx[p.const_mask()[e_idx]]
    Hd[ce, :] = 0
    Hd[:, ce] = 0
    Hd[ce, ce] = 1
    gd[ce] = 0
    f_index = np.concatenate([np.arange(f_off, f_off + 6 * n_f), np.arange(o_shared, n)])
    return O.schur_reduce(Hd, gd, slice(e_off, e_off + 6 * n_e), f_index)


def lm_step(p, priors, radius, jacobi=False):
    """The damped, masked Gauss-Newton step of the stacked problem: (delta, model_cost_change, cost, gmax)."""
    H, g, c = normal_equations(p, priors)
    cm = p.const_mask()
    d2 = lm_diagonal(H, radius, jacobi)
    Hd, gm = O.masked_system(H + np.diag(d2), g, cm)
    delta = -np.linalg.solve(Hd, gm)
    delta[cm] = 0
    d2m = np.where(cm, 0.0, d2)
    mcc = -0.5 * float(gm @ delta) + 0.5 * float(delta @ (d2m * delta))
    return delta, mcc, c, float(np.abs(gm).max())


def covariance(p, priors):
    """(J^T J)^-1 of the stacked problem restricted to the free parameters, zero at the constants."""
    H, _, _ = normal_equations(p, priors)
    free = np.nonzero(~p.const_mask())[0]
    C = np.zeros_like(H)
    C[np.ix_(free, free)] = np.linalg.inv(H[np.ix_(free, free)])
    return C


def minimise(p, priors, **kw):
    """scipy.optimize.least_squares on the stacked (tag + prior) residuals over the free parameters; returns the
    minimiser in the dense layout."""
    from scipy.optimize import least_squares
    x0 = p.pack()
    free = np.nonzero(~p.const_mask())[0]

    def fun(z):
        x = x0.copy()
        x[free] = z
        q = p.copy()
        q.unpack(x)
        return np.concatenate([MO.residuals(q).ravel(), prior_rows(q, priors, x)[1]])

    opts = dict(method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15, max_nfev=4000)
    opts.update(kw)
    z = least_squares(fun, x0[free], **opts).x
    x = x0.copy()
    x[free] = z
    return x
