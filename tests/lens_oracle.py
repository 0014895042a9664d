"""CPU oracle for the equidistant (fisheye) lens.  TEST INFRASTRUCTURE ONLY.

The same problem container and dense machinery as ``ba_oracle`` (which stays the radial-tangential reference), with
the projection chosen by ``p.lens``:

  Oracle A  closed-form projection in NumPy, complex-step safe, + complex-step derivatives (h = 1e-30).
            th = arctan(rho / Z) for Z > 0 (numpy's arctan2 rejects complex input), and th / rho = arctan(w) / w / Z,
            w^2 = rho^2 / Z^2, by its series for small w, so nothing divides by rho on the optical axis.
  Oracle B  cv2.fisheye.projectPoints (OpenCV 4.13: a (2N, 15) Jacobian, columns fx fy | cx cy | k1..k4 | rvec |
            tvec | alpha) chained through cv2.composeRT exactly as ba_oracle.jacobian_block_cv2 does.
A and B agree on the wide-angle scenes of tests/test_equidistant_host.py (tags up to 85 degrees off the axis) to
3.4e-13 px in the projected corners and 5.8e-15 relative (per-block Frobenius) in every Jacobian block.
"""
from __future__ import annotations

import numpy as np

import ba_oracle as O


class LensProblem(O.OracleProblem):
    """ba_oracle.OracleProblem with a lens, "radtan" or "equidistant".  Its constant mask is what the library holds
    constant: the caller's constant blocks and, under the equidistant lens, the reserved distortion slot of every
    camera."""

    def __init__(self, lens, *args, **kw):
        super().__init__(*args, **kw)
        self.lens = lens

    def _copy(self):
        return LensProblem(self.lens, self.model, self.intr, self.dist, self.ext, self.views, self.markers, self.sizes,
                           self.view_idx, self.marker_idx, self.cam_idx, self.pixels, self.const_views,
                           self.const_markers, self.const_intr, self.const_dist,
                           self.const_ext if self.model == "rig" else None)

    def const_mask(self):
        m = super().const_mask()
        if self.lens == "equidistant":
            m[self.offsets()[2] + self.shared_per_cam * np.arange(self.n_cam) + 8] = True
        return m


def oracle_problem(s):
    """Scene -> LensProblem with the scene's lens."""
    return LensProblem(s.lens, s.model, s.intr, s.dist, s.ext, s.views, s.markers, s.sizes, s.view_idx, s.marker_idx,
                       s.cam_idx, s.pixels, s.const_views, s.const_markers, s.const_intr, s.const_dist,
                       s.const_ext if s.model == "rig" else None)


def _atan_over(w2):
    """arctan(w) / w as a function of w^2 (complex-step safe, exact at w = 0)."""
    w2 = np.asarray(w2)
    small = np.abs(w2) < 1e-3
    series = 1 - w2 * (1 / 3 - w2 * (1 / 5 - w2 * (1 / 7 - w2 * (1 / 9 - w2 / 11))))
    ws = np.sqrt(np.where(small, 1.0, w2))
    return np.where(small, series, np.arctan(ws) / ws)


def distort(lens, dist, X, Y, Z):
    """Normalised distorted coordinates (x', y') of camera-frame points; dist (N,1) columns broadcast over corners."""
    if lens == "equidistant":
        w2 = (X * X + Y * Y) / (Z * Z)
        c = _atan_over(w2) / Z                       # th / rho
        t2 = w2 * _atan_over(w2) ** 2                 # th^2
        k1, k2, k3, k4 = (dist[:, i:i + 1] for i in range(4))
        s = c * (1 + t2 * (k1 + t2 * (k2 + t2 * (k3 + t2 * k4))))
        return s * X, s * Y
    x, y = X / Z, Y / Z
    r2 = x * x + y * y
    k1, k2, p1, p2, k3 = (dist[:, i:i + 1] for i in range(5))
    rad = 1 + r2 * (k1 + r2 * (k2 + r2 * k3))
    return x * rad + 2 * p1 * x * y + p2 * (r2 + 2 * x * x), y * rad + p1 * (r2 + 2 * y * y) + 2 * p2 * x * y


def project_blocks(model, lens, intr, dist, ext, view, marker, size, dtype=np.float64):
    """ba_oracle.project_blocks with a lens: (uv (N,4,2), Z (N,4))."""
    intr, dist = np.asarray(intr, dtype=dtype), np.asarray(dist, dtype=dtype)
    view, marker = np.asarray(view, dtype=dtype), np.asarray(marker, dtype=dtype)
    o = O.obj_points(size).astype(dtype)
    Pw = np.einsum('nij,nkj->nki', O.rodrigues(marker[:, 0:3]), o) + marker[:, None, 3:6]
    q = np.einsum('nji,nkj->nki', O.rodrigues(view[:, 0:3]), Pw - view[:, None, 3:6])
    if model == "rig":
        ext = np.asarray(ext, dtype=dtype)
        q = np.einsum('nji,nkj->nki', O.rodrigues(ext[:, 0:3]), q - ext[:, None, 3:6])
    X, Y, Z = q[..., 0], q[..., 1], q[..., 2]
    xd, yd = distort(lens, dist, X, Y, Z)
    return np.stack([intr[:, 0:1] * xd + intr[:, 2:3], intr[:, 1:2] * yd + intr[:, 3:4]], -1), Z


def residuals(p):
    uv, _ = project_blocks(p.model, p.lens, *O._gather(p))
    return uv.reshape(-1, 8) - p.pixels


def depths(p):
    return project_blocks(p.model, p.lens, *O._gather(p))[1]


def cost(p):
    return 0.5 * float(O.robust(p, residuals(p))[1].sum())


def jacobian_blocks_cs(p):
    """Per-block Jacobians by complex step: dict name -> (N,8,k)."""
    intr, dist, ext, view, marker, size = O._gather(p)
    base = dict(intr=intr, dist=dist, ext=ext, view=view, marker=marker)
    out = {}
    for name, k in O.local_param_names(p.model):
        J = np.empty((len(size), 8, k))
        for c in range(k):
            args = {n: a.astype(np.complex128) for n, a in base.items()}
            args[name][:, c] += 1j * O.CS_H
            uv, _ = project_blocks(p.model, p.lens, args["intr"], args["dist"], args["ext"], args["view"],
                                   args["marker"], size, dtype=np.complex128)
            J[:, :, c] = uv.reshape(-1, 8).imag / O.CS_H
        out[name] = J
    return out


def jacobian_block_cv2(model, intr, dist, ext, view, marker, size):
    """Oracle B for one block of an equidistant camera: (uv (8,), dict name -> (8,k)), dist column 4 = 0."""
    import cv2
    K = np.array([[intr[0], 0, intr[2]], [0, intr[1], intr[3]], [0, 0, 1.0]])
    ct, dct = _chain(model, ext, view, marker)
    pts, J = cv2.fisheye.projectPoints(O.obj_points(size).reshape(1, 4, 3), ct[0:3].reshape(3, 1),
                                       ct[3:6].reshape(3, 1), K, np.asarray(dist[:4], float).reshape(4, 1))
    # J columns: fx fy 0:2 | cx cy 2:4 | k1..k4 4:8 | rvec 8:11 | tvec 11:14 | alpha 14
    Jrt = J[:, 8:14]
    out = {k: Jrt @ v for k, v in dct.items()}
    out["intr"] = J[:, 0:4]
    out["dist"] = np.concatenate([J[:, 4:8], np.zeros((8, 1))], 1)
    return pts.reshape(8), out


# cam_T_target = inv(body_T_cam) * inv(world_T_view) * world_T_target and its partials: the cv2.Rodrigues /
# cv2.composeRT chain of ba_oracle.jacobian_block_cv2
def _invert(rt):
    import cv2
    r, t = rt[0:3].reshape(3, 1), rt[3:6].reshape(3, 1)
    R, dRdr = cv2.Rodrigues(r)
    D = np.zeros((6, 6))
    D[0:3, 0:3] = -np.eye(3)
    dR = dRdr.reshape(3, 3, 3)
    for k in range(3):
        D[3:6, k] = -(dR[k].T @ t).ravel()
    D[3:6, 3:6] = -R.T
    return np.concatenate([-r.ravel(), (-R.T @ t).ravel()]), D


def _compose(rt1, rt2):
    import cv2
    r3, t3, dr3dr1, dr3dt1, dr3dr2, dr3dt2, dt3dr1, dt3dt1, dt3dr2, dt3dt2 = cv2.composeRT(
        rt1[0:3].reshape(3, 1), rt1[3:6].reshape(3, 1), rt2[0:3].reshape(3, 1), rt2[3:6].reshape(3, 1))
    return (np.concatenate([r3.ravel(), t3.ravel()]), np.block([[dr3dr1, dr3dt1], [dt3dr1, dt3dt1]]),
            np.block([[dr3dr2, dr3dt2], [dt3dr2, dt3dt2]]))


def _chain(model, ext, view, marker):
    vinv, Dv = _invert(np.asarray(view, float))
    ct, D_m, D_vi = _compose(np.asarray(marker, float), vinv)
    d = {"marker": D_m, "view": D_vi @ Dv}
    if model == "rig":
        xinv, Dx = _invert(np.asarray(ext, float))
        ct, D_prev, D_xi = _compose(ct, xinv)
        d = {k: D_prev @ v for k, v in d.items()}
        d["ext"] = D_xi @ Dx
    return ct, d


# ---------------------------------------------------------------------------------------------- dense system
def normal_equations(p):
    J = O.dense_jacobian(p, jacobian_blocks_cs(p))
    r = residuals(p)
    w, rho = O.robust(p, r)
    J = J * np.repeat(w, 8)[:, None]
    r = (r * w[:, None]).ravel()
    return J.T @ J, J.T @ r, 0.5 * float(rho.sum())


def lm_step(p, radius):
    """ba_oracle.lm_step with the lens's Jacobian and mask: (delta, model_cost_change, cost, gmax)."""
    H, g, c = normal_equations(p)
    cm = p.const_mask()
    d2 = O.lm_diagonal(H, radius)
    Hd, gm = O.masked_system(H + np.diag(d2), g, cm)
    delta = -np.linalg.solve(Hd, gm)
    delta[cm] = 0
    d2m = np.where(cm, 0.0, d2)
    mcc = -0.5 * float(gm @ delta) + 0.5 * float(delta @ (d2m * delta))
    return delta, mcc, c, float(np.abs(gm).max())


def blocks(p, elim_view):
    """helpers.oracle_blocks for the lens: the normal-equation blocks in the library's layout."""
    H, g, c = normal_equations(p)
    o_view, o_marker, o_shared, n = p.offsets()
    nv, nm = len(p.views), len(p.markers)
    e_off, n_e = (o_view, nv) if elim_view else (o_marker, nm)
    f_off, n_f = (o_marker, nm) if elim_view else (o_view, nv)
    blk = lambda off, i: slice(off + 6 * i, off + 6 * i + 6)
    Jb = jacobian_blocks_cs(p)
    Je, Jf = (Jb["view"], Jb["marker"]) if elim_view else (Jb["marker"], Jb["view"])
    w, _ = O.robust(p, residuals(p))
    return {
        "Hee": np.stack([H[blk(e_off, i), blk(e_off, i)] for i in range(n_e)]),
        "ge": g[e_off:e_off + 6 * n_e].reshape(n_e, 6),
        "Hes": np.stack([H[blk(e_off, i), o_shared:] for i in range(n_e)]),
        "Hff": np.stack([H[blk(f_off, i), blk(f_off, i)] for i in range(n_f)]),
        "gf": g[f_off:f_off + 6 * n_f].reshape(n_f, 6),
        "Hfs": np.stack([H[blk(f_off, i), o_shared:] for i in range(n_f)]),
        "Hss": H[o_shared:, o_shared:], "gs": g[o_shared:], "cost": c, "H": H, "g": g,
        "W": np.einsum('nri,nrj->nij', Je, Jf) * (w * w)[:, None, None],
    }


def reduced(p, elim_view, radius, min_diag=1e-6, max_diag=1e32):
    """helpers.oracle_reduced for the lens: (S, b) of rcc_ba_schur (damping on the eliminated blocks only)."""
    H, g, _ = normal_equations(p)
    o_view, o_marker, o_shared, n = p.offsets()
    nv, nm = len(p.views), len(p.markers)
    e_off, n_e = (o_view, nv) if elim_view else (o_marker, nm)
    f_off, n_f = (o_marker, nm) if elim_view else (o_view, nv)
    d2 = np.clip(np.diag(H), min_diag, max_diag) / radius
    Hd = H.copy()
    e_idx = np.arange(e_off, e_off + 6 * n_e)
    Hd[e_idx, e_idx] += d2[e_idx]
    ce = e_idx[p.const_mask()[e_idx]]
    gd = g.copy()
    Hd[ce, :] = 0
    Hd[:, ce] = 0
    Hd[ce, ce] = 1
    gd[ce] = 0
    f_index = np.concatenate([np.arange(f_off, f_off + 6 * n_f), np.arange(o_shared, n)])
    return O.schur_reduce(Hd, gd, slice(e_off, e_off + 6 * n_e), f_index)
