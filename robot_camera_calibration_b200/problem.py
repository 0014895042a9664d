"""Host-side mirror of the C ABI: one `BAProblem` per CUDA device.

The method names follow the C entry points of include/rcc_ba.h one-to-one;
array arguments are numpy (host) buffers, exactly what the C ABI takes.  All
arithmetic happens in librcc_ba.so on the GPU; nothing here computes.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib as L


def _dp(a):
    return a.ctypes.data_as(L.c_double_p) if a is not None else None


def _ip(a):
    return a.ctypes.data_as(L.c_int32_p) if a is not None else None


_BLOCK_KINDS = {"view": L.BLOCK_VIEW, "marker": L.BLOCK_MARKER, "intr": L.BLOCK_INTR, "dist": L.BLOCK_DIST,
                "ext": L.BLOCK_EXT}
_BLOCK_SIZES = {L.BLOCK_VIEW: 6, L.BLOCK_MARKER: 6, L.BLOCK_INTR: 4, L.BLOCK_DIST: 5, L.BLOCK_EXT: 6}


def sqrt_information(cov):
    """The sqrt_information A of a Gaussian prior whose covariance is cov: A = L^-1 for cov = L L^T (Cholesky), so
    that ||A (x - mu)||^2 = (x - mu)^T cov^-1 (x - mu).  cov is one k x k matrix or a stack (..., k, k)."""
    L_ = np.linalg.cholesky(np.asarray(cov, dtype=np.float64))
    return np.linalg.solve(L_, np.broadcast_to(np.eye(L_.shape[-1]), L_.shape))


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        a = a.reshape(shape)
    return a


class BAProblem:
    """Bundle-adjustment problem resident on one B200.

    model "single": views are world_T_camera (camera_pose.cpp:88-98);
    model "rig":    views are world_T_body and ext[c] is body_T_cam_c.
    lens "radtan" (dist = k1 k2 p1 p2 k3) or "equidistant" (dist = k1 k2 k3 k4 + a reserved slot held constant)
    for every camera (rcc_ba_set_lens), or a sequence of n_cameras such names, one per camera
    (rcc_ba_set_camera_lenses): a rig may mix pinhole and fisheye cameras.
    """

    def __init__(self, n_views, n_markers, n_cameras=1, n_obs_blocks=0, model="single", device=0,
                 eliminate="auto", lens="radtan"):
        self.lib = L.load()
        self.model = model
        self.n_views, self.n_markers, self.n_cameras = int(n_views), int(n_markers), int(n_cameras)
        self.n_obs = int(n_obs_blocks)
        opt = L.Options(model=L.MODEL_RIG if model == "rig" else L.MODEL_SINGLE, n_views=self.n_views,
                        n_markers=self.n_markers, n_cameras=self.n_cameras, n_obs_blocks=self.n_obs,
                        device=int(device),
                        eliminate={"auto": L.ELIM_AUTO, "views": L.ELIM_VIEWS, "markers": L.ELIM_MARKERS}[eliminate])
        h = C.c_void_p()
        rc = self.lib.rcc_ba_create(C.byref(opt), C.byref(h))
        if rc != L.RCC_OK:
            raise L.RccError(rc, self.lib.rcc_ba_last_error(None).decode())
        self.h = h
        d = L.Dims()
        self._check(self.lib.rcc_ba_get_dims(self.h, C.byref(d)))
        self.dims = d
        self.lens = "radtan"
        if lens != "radtan":
            self.set_lens(lens)

    # ------------------------------------------------------------------ plumbing
    def _check(self, rc):
        if rc != L.RCC_OK:
            raise L.RccError(rc, self.lib.rcc_ba_last_error(self.h).decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.rcc_ba_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ------------------------------------------------------------------ setup
    @classmethod
    def from_scene(cls, scene, device=0, eliminate="auto"):
        p = cls(len(scene.views), len(scene.markers), len(scene.intr), scene.n_blocks, scene.model,
                device=device, eliminate=eliminate, lens=scene.lens)
        p.set_intrinsics(scene.intr, scene.dist)
        if scene.model == "rig":
            p.set_rig_extrinsics(scene.ext)
        p.set_view_poses(scene.views)
        p.set_marker_poses(scene.markers)
        p.set_marker_sizes(scene.sizes)
        p.set_observations(scene.view_idx, scene.marker_idx, scene.cam_idx, scene.pixels)
        for kind, mask in ((L.BLOCK_VIEW, scene.const_views), (L.BLOCK_MARKER, scene.const_markers),
                           (L.BLOCK_INTR, scene.const_intr), (L.BLOCK_DIST, scene.const_dist)):
            for i in np.nonzero(mask)[0]:
                p.set_constant(kind, int(i), True)
        if scene.model == "rig":
            for i in np.nonzero(scene.const_ext)[0]:
                p.set_constant(L.BLOCK_EXT, int(i), True)
        if getattr(scene, "corners", None) is not None:
            p.set_corner_layout(scene.corners, scene.corner_slot)
        return p

    def set_intrinsics(self, intr, dist):
        intr, dist = _f64(intr, (self.n_cameras, 4)), _f64(dist, (self.n_cameras, 5))
        self._check(self.lib.rcc_ba_set_intrinsics(self.h, _dp(intr), _dp(dist)))

    def set_rig_extrinsics(self, ext):
        ext = _f64(ext, (self.n_cameras, 6))
        self._check(self.lib.rcc_ba_set_rig_extrinsics(self.h, _dp(ext)))

    def set_view_poses(self, views):
        views = _f64(views, (self.n_views, 6))
        self._check(self.lib.rcc_ba_set_view_poses(self.h, _dp(views)))

    def set_marker_poses(self, markers):
        markers = _f64(markers, (self.n_markers, 6))
        self._check(self.lib.rcc_ba_set_marker_poses(self.h, _dp(markers)))

    def set_marker_sizes(self, sizes):
        sizes = _f64(sizes, (self.n_markers,))
        self._check(self.lib.rcc_ba_set_marker_sizes(self.h, _dp(sizes)))

    def set_observations(self, view_idx, marker_idx, cam_idx, pixels):
        vi = np.ascontiguousarray(view_idx, dtype=np.int32)
        mi = np.ascontiguousarray(marker_idx, dtype=np.int32)
        ci = None if cam_idx is None else np.ascontiguousarray(cam_idx, dtype=np.int32)
        if len(vi) != self.n_obs or len(mi) != self.n_obs:
            raise ValueError("observation arrays do not match n_obs_blocks")
        pixels = np.asarray(pixels)
        if pixels.dtype == np.int16:        # the reference's integer corners (corner_detections.cpp:53-54)
            px = np.ascontiguousarray(pixels).reshape(self.n_obs, 8)
            rc = self.lib.rcc_ba_set_observations_i16(self.h, _ip(vi), _ip(mi), _ip(ci), px.ctypes.data_as(L.c_int16_p))
        elif np.issubdtype(pixels.dtype, np.integer):
            px = np.ascontiguousarray(pixels, dtype=np.int32).reshape(self.n_obs, 8)
            rc = self.lib.rcc_ba_set_observations_i32(self.h, _ip(vi), _ip(mi), _ip(ci), _ip(px))
        else:
            px = _f64(pixels, (self.n_obs, 8))
            rc = self.lib.rcc_ba_set_observations(self.h, _ip(vi), _ip(mi), _ip(ci), _dp(px))
        self._check(rc)
        self._check(self.lib.rcc_ba_get_dims(self.h, C.byref(self.dims)))

    def update_pixels(self, pixels):
        """FP64 pixels, or int16 (the reference's integer corners: a quarter of the bytes over PCIe)."""
        pixels = np.asarray(pixels)
        if pixels.dtype == np.int16:
            px = np.ascontiguousarray(pixels).reshape(self.n_obs, 8)
            self._check(self.lib.rcc_ba_update_pixels_i16(self.h, px.ctypes.data_as(L.c_int16_p)))
            return
        px = _f64(pixels, (self.n_obs, 8))
        self._check(self.lib.rcc_ba_update_pixels(self.h, _dp(px)))

    def set_corner_layout(self, corners, slot):
        """Rigid planar targets (rcc_ba_set_corner_layout): corners (n_slots, 4, 2) bl br tr tl in the frame of the
        block's marker, slot (n_obs_blocks,) in caller order, -1 for the square of the marker's size.  A marker whose
        blocks use different slots is one tag board with one pose.  An empty corners array clears the layout;
        set_observations clears it too, update_pixels keeps it."""
        c = _f64(corners).reshape(-1, 4, 2)
        if len(c) == 0:
            self.clear_corner_layout()
            return
        sl = np.ascontiguousarray(slot, dtype=np.int32).reshape(-1)
        if len(sl) != self.n_obs:
            raise ValueError(f"{len(sl)} slots for {self.n_obs} observation blocks")
        self._check(self.lib.rcc_ba_set_corner_layout(self.h, len(c), _dp(c), _ip(sl)))

    def clear_corner_layout(self):
        self._check(self.lib.rcc_ba_set_corner_layout(self.h, 0, None, None))

    def set_constant(self, kind, index, is_constant=True):
        kind = _BLOCK_KINDS[kind] if isinstance(kind, str) else kind
        self._check(self.lib.rcc_ba_set_constant(self.h, kind, index, int(bool(is_constant))))

    def set_loss(self, loss, scale=1.0):
        """loss: 'trivial' | 'huber' | 'cauchy' on each tag's 8-residual block (scale in pixels)."""
        code = {"trivial": 0, "huber": 1, "cauchy": 2}[loss] if isinstance(loss, str) else int(loss)
        self._check(self.lib.rcc_ba_set_loss(self.h, code, float(scale)))

    def set_lens(self, lens):
        """lens: 'radtan' | 'equidistant' for every camera, or a sequence of n_cameras such names (one per camera);
        invalidates the linearisation like set_loss.  Afterwards .lens is the name when every camera has the same
        lens and the tuple of names otherwise."""
        names = (lens,) if isinstance(lens, str) else tuple(lens)
        for n in names:
            if n not in L.LENSES:
                raise ValueError(f"unknown lens {n!r}: expected one of {sorted(L.LENSES)}")
        if isinstance(lens, str):
            self._check(self.lib.rcc_ba_set_lens(self.h, L.LENSES[lens]))
        else:
            if len(names) != self.n_cameras:
                raise ValueError(f"{len(names)} lenses for {self.n_cameras} cameras")
            codes = np.array([L.LENSES[n] for n in names], dtype=np.int32)
            self._check(self.lib.rcc_ba_set_camera_lenses(self.h, _ip(codes)))
        self.lens = names[0] if len(set(names)) == 1 else names

    def set_priors(self, kind, index, mean, sqrt_information):
        """Gaussian priors (ceres::NormalPrior) on the blocks of one kind: the residual block A_i (x_i - mu_i) on block
        index[i], mean (n, k), sqrt_information (n, k, k) with k the kind's block size (view / marker / ext 6, intr 4,
        dist 5).  Replaces every earlier prior of that kind; an empty index clears them (rcc_ba_set_priors).  For a
        covariance Sigma use sqrt_information(Sigma)."""
        kind = _BLOCK_KINDS[kind] if isinstance(kind, str) else int(kind)
        k = _BLOCK_SIZES.get(kind, 6)
        idx = np.ascontiguousarray(index, dtype=np.int32).reshape(-1)
        n = len(idx)
        mu = _f64(mean, (n, k))
        A = _f64(sqrt_information, (n, k, k))
        self._check(self.lib.rcc_ba_set_priors(self.h, kind, n, _ip(idx), _dp(mu), _dp(A)))

    def clear_priors(self, kind=None):
        """Remove the priors of one kind, or of every kind (kind=None)."""
        kinds = [kind] if kind is not None else ["view", "marker", "intr", "dist"] + (["ext"] if self.model == "rig" else [])
        for k in kinds:
            k = _BLOCK_KINDS[k] if isinstance(k, str) else int(k)
            self._check(self.lib.rcc_ba_set_priors(self.h, k, 0, None, None, None))

    # ------------------------------------------------------------------ getters
    def get_intrinsics(self):
        intr, dist = np.empty((self.n_cameras, 4)), np.empty((self.n_cameras, 5))
        self._check(self.lib.rcc_ba_get_intrinsics(self.h, _dp(intr), _dp(dist)))
        return intr, dist

    def get_rig_extrinsics(self):
        ext = np.empty((self.n_cameras, 6))
        self._check(self.lib.rcc_ba_get_rig_extrinsics(self.h, _dp(ext)))
        return ext

    def get_view_poses(self):
        v = np.empty((self.n_views, 6))
        self._check(self.lib.rcc_ba_get_view_poses(self.h, _dp(v)))
        return v

    def get_marker_poses(self):
        m = np.empty((self.n_markers, 6))
        self._check(self.lib.rcc_ba_get_marker_poses(self.h, _dp(m)))
        return m

    # ------------------------------------------------------------------ evaluation
    def evaluate(self, want_jacobians=True, want_residuals=True, allow_failure=False):
        """Materialised residuals and Ceres-layout Jacobians (host arrays)."""
        n = self.n_obs
        cost = C.c_double()
        res = np.empty((n, 8)) if want_residuals else None
        J = {}
        if want_jacobians:
            J = {"intr": np.empty((n, 8, 4)), "dist": np.empty((n, 8, 5)), "view": np.empty((n, 8, 6)),
                 "marker": np.empty((n, 8, 6))}
            if self.model == "rig":
                J["ext"] = np.empty((n, 8, 6))
        rc = self.lib.rcc_ba_evaluate(self.h, int(want_jacobians), C.byref(cost), _dp(res), _dp(J.get("intr")),
                                      _dp(J.get("dist")), _dp(J.get("view")), _dp(J.get("marker")),
                                      _dp(J.get("ext")))
        failed = rc == L.RCC_EVAL_FAILED
        if rc != L.RCC_OK and not (failed and allow_failure):
            self._check(rc)
        return {"cost": cost.value, "residuals": res, "jacobians": J, "failed": failed}

    def evaluate_device(self, want_jacobians=True, want_cost=False):
        cost = C.c_double()
        self._check(self.lib.rcc_ba_evaluate_device(self.h, int(want_jacobians), C.byref(cost) if want_cost else None))
        return cost.value if want_cost else None

    # ------------------------------------------------------------------ normal equations / LM
    def linearize(self, want_cost=True):
        cost = C.c_double()
        self._check(self.lib.rcc_ba_linearize(self.h, C.byref(cost) if want_cost else None))
        return cost.value if want_cost else None

    def normal_blocks(self, want_W=True):
        d = self.dims
        out = {"Hee": np.empty((d.n_e, 6, 6)), "ge": np.empty((d.n_e, 6)), "Hes": np.empty((d.n_e, 6, d.n_shared)),
               "Hff": np.empty((d.n_f, 6, 6)), "gf": np.empty((d.n_f, 6)), "Hfs": np.empty((d.n_f, 6, d.n_shared)),
               "Hss": np.empty((d.n_shared, d.n_shared)), "gs": np.empty(d.n_shared),
               "W": np.empty((self.n_obs, 6, 6)) if want_W else None}
        self._check(self.lib.rcc_ba_get_normal_blocks(self.h, *[_dp(out[k]) for k in
                                                                ("Hee", "ge", "Hes", "Hff", "gf", "Hfs", "Hss", "gs", "W")]))
        return out

    def set_lm_diagonal(self, min_diagonal=1e-6, max_diagonal=1e32, jacobi_scaling=False):
        self._check(self.lib.rcc_ba_set_lm_diagonal(self.h, float(min_diagonal), float(max_diagonal), int(jacobi_scaling)))

    def schur(self, radius):
        self._check(self.lib.rcc_ba_schur(self.h, float(radius)))

    def reduced_system(self):
        n = self.dims.n_reduced
        S, b = np.empty((n, n)), np.empty(n)
        self._check(self.lib.rcc_ba_get_reduced_system(self.h, _dp(S), _dp(b)))
        return S, b

    def reduced_block(self, row0, n_rows, col0, n_cols):
        """S[row0:row0+n_rows, col0:col0+n_cols] (column n_reduced = the right-hand side b)."""
        out = np.empty((n_rows, n_cols))
        self._check(self.lib.rcc_ba_get_reduced_block(self.h, int(row0), int(n_rows), int(col0), int(n_cols), _dp(out)))
        return out

    def solve_step(self):
        mcc, sn, xn = C.c_double(), C.c_double(), C.c_double()
        self._check(self.lib.rcc_ba_solve_step(self.h, C.byref(mcc), C.byref(sn), C.byref(xn)))
        return mcc.value, sn.value, xn.value

    def step(self):
        d = self.dims
        de, df, ds = np.empty((d.n_e, 6)), np.empty((d.n_f, 6)), np.empty(d.n_shared)
        self._check(self.lib.rcc_ba_get_step(self.h, _dp(de), _dp(df), _dp(ds)))
        return {"d_e": de, "d_f": df, "d_shared": ds}

    def candidate_cost(self):
        c = C.c_double()
        self._check(self.lib.rcc_ba_candidate_cost(self.h, C.byref(c)))
        return c.value

    def accept_step(self):
        self._check(self.lib.rcc_ba_accept_step(self.h))

    def solve(self, **kw):
        o = L.LMOptions()
        self.lib.rcc_lm_default_options(C.byref(o))
        for k, v in kw.items():
            if not hasattr(o, k):
                raise TypeError(f"unknown LM option {k}")
            setattr(o, k, v)
        s = L.LMSummary()
        self._check(self.lib.rcc_ba_solve(self.h, C.byref(o), C.byref(s)))
        return {f: getattr(s, f) for f, _ in L.LMSummary._fields_}

    def covariance(self):
        """Parameter covariance at the current parameters, ceres::Covariance semantics: the marginal blocks of
        (J^T J)^-1 of the undamped Gauss-Newton system, J the loss-weighted Jacobian the LM step uses.  Not scaled by
        a residual variance: with pixel noise of standard deviation sigma, multiply by sigma**2.  Rows and columns of
        constant blocks are exactly zero.  Returns {"shared": (n_shared, n_shared), "views": (n_views, 6, 6),
        "markers": (n_markers, 6, 6)}; raises RccError(RCC_NOT_SPD) when J^T J restricted to the free parameters is
        not positive definite.  Leaves the handle linearised at the current point (rcc_ba_covariance)."""
        out = {"shared": np.empty((self.dims.n_shared, self.dims.n_shared)), "views": np.empty((self.n_views, 6, 6)),
               "markers": np.empty((self.n_markers, 6, 6))}
        self._check(self.lib.rcc_ba_covariance(self.h, _dp(out["shared"]), _dp(out["views"]), _dp(out["markers"])))
        return out

    def covariance_blocks(self, pairs):
        """Cross-covariance blocks of (J^T J)^-1, the same semantics as covariance(): pairs is an iterable of
        ((kind, index), (kind, index)), kind "view" | "marker" | "intr" | "dist" | "ext" (or the integer codes) and
        index the view, marker or camera.  Returns one (size_a, size_b) array per pair, size 6 for a pose or rig
        extrinsic, 4 for intrinsics, 5 for distortion; Cov(b, a) is exactly Cov(a, b).T.  With pixel noise of
        standard deviation sigma, multiply by sigma**2 (rcc_ba_covariance_blocks)."""
        req = np.array([[_BLOCK_KINDS[k] if isinstance(k, str) else int(k), int(i)] for pair in pairs
                        for k, i in pair], dtype=np.int32).reshape(-1, 4)
        out = np.zeros((len(req), 36))
        self._check(self.lib.rcc_ba_covariance_blocks(self.h, len(req), _ip(req), _dp(out)))
        return [out[p, :_BLOCK_SIZES[ka] * _BLOCK_SIZES[kb]].reshape(_BLOCK_SIZES[ka], _BLOCK_SIZES[kb])
                for p, (ka, _, kb, _) in enumerate(req.tolist())]

    # ------------------------------------------------------------------ multi-GPU
    @staticmethod
    def comm_unique_id():
        buf = C.create_string_buffer(L.COMM_ID_BYTES)
        rc = L.load().rcc_comm_get_unique_id(buf)
        if rc != L.RCC_OK:
            raise L.RccError(rc, "ncclGetUniqueId failed")
        return bytes(buf.raw)

    def comm_init(self, unique_id, rank, n_ranks):
        self._check(self.lib.rcc_ba_comm_init(self.h, unique_id, int(rank), int(n_ranks)))

    # ------------------------------------------------------------------ measurement
    def profile_enable(self, on=True):
        self._check(self.lib.rcc_ba_profile_enable(self.h, int(on)))

    def profile_reset(self):
        self._check(self.lib.rcc_ba_profile_reset(self.h))

    def profile_get(self, stage):
        ms, n = C.c_double(), C.c_int64()
        self._check(self.lib.rcc_ba_profile_get(self.h, stage.encode(), C.byref(ms), C.byref(n)))
        return ms.value, n.value

    STAGES = ("expand", "assemble_e", "assemble_f", "finalize", "schur_prep", "schur_syrk", "schur_shared",
              "allreduce", "mask", "cholesky", "backsub", "cost", "evaluate", "h2d", "inverse", "covariance", "cov_extract")

    def profile(self):
        return {s: self.profile_get(s) for s in self.STAGES}

    def launch_count(self):
        return int(self.lib.rcc_ba_launch_count(self.h))

    def synchronize(self):
        self._check(self.lib.rcc_ba_synchronize(self.h))

    def flush_l2(self):
        self._check(self.lib.rcc_ba_flush_l2(self.h))


def fp64_peak_tflops(device=0):
    v = C.c_double()
    rc = L.load().rcc_fp64_peak_tflops(int(device), C.byref(v))
    if rc != L.RCC_OK:
        raise L.RccError(rc, "fp64 peak microbenchmark failed")
    return v.value
