"""Synthetic fiducial-marker scenes (the `Camera` data path the simulator
promises at rviz_simulator/include/rviz_simulator/target.h:40 but never ships).

A scene is: a wall-like cloud of square tags (world_T_target poses, tag 0 at
identity = the gauge, camera_pose.cpp:71-80), a set of camera views looking at
it (world_T_camera, or world_T_body + body_T_cam for a rig), and the projected
corner pixels of every tag whose four corners land inside the image with
positive depth -- exactly the content of the reference's detections_N.yaml
(corner_detections.cpp:18-39) plus the initial guesses camera_pose_node would
write (camera_pose.cpp:83-129).

Everything here is host-side numpy; it produces inputs for the GPU path, it
does not evaluate the cost (that is csrc/).
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np


# ---------------------------------------------------------------- small SO(3) helpers
def rodrigues_np(r):
    r = np.asarray(r, dtype=np.float64)
    t2 = (r * r).sum(-1)
    small = t2 < 1e-16
    t = np.sqrt(np.where(small, 1.0, t2))
    A = np.where(small, 1 - t2 / 6, np.sin(t) / t)
    B = np.where(small, 0.5 - t2 / 24, (1 - np.cos(t)) / np.where(small, 1.0, t2))
    x, y, z = r[..., 0], r[..., 1], r[..., 2]
    zero = np.zeros_like(x)
    K = np.stack([np.stack([zero, -z, y], -1), np.stack([z, zero, -x], -1),
                  np.stack([-y, x, zero], -1)], -2)
    return np.eye(3) + A[..., None, None] * K + B[..., None, None] * (K @ K)


def rotation_to_rvec(R):
    """Inverse of rodrigues_np for rotation angles < pi (batched)."""
    R = np.asarray(R, dtype=np.float64)
    w = np.stack([R[..., 2, 1] - R[..., 1, 2], R[..., 0, 2] - R[..., 2, 0],
                  R[..., 1, 0] - R[..., 0, 1]], -1) * 0.5          # sin(t) * axis
    s = np.linalg.norm(w, axis=-1)
    c = (np.trace(R, axis1=-2, axis2=-1) - 1) * 0.5
    t = np.arctan2(s, c)
    scale = np.where(s < 1e-12, 1.0, t / np.where(s < 1e-12, 1.0, s))
    return w * scale[..., None]


def compose(rt_a, rt_b):
    """T_a * T_b for (rvec,t) 6-vectors (batched)."""
    Ra, Rb = rodrigues_np(rt_a[..., 0:3]), rodrigues_np(rt_b[..., 0:3])
    R = Ra @ Rb
    t = np.einsum('...ij,...j->...i', Ra, rt_b[..., 3:6]) + rt_a[..., 3:6]
    return np.concatenate([rotation_to_rvec(R), t], -1)


def invert(rt):
    R = rodrigues_np(rt[..., 0:3])
    t = -np.einsum('...ji,...j->...i', R, rt[..., 3:6])
    return np.concatenate([-rt[..., 0:3], t], -1)


def obj_points(size):
    """Tag-frame corners, order bl br tr tl (camera_pose.cpp:123-126)."""
    s = np.asarray(size, dtype=np.float64) / 2
    z = np.zeros_like(s)
    return np.stack([np.stack([-s, -s, z], -1), np.stack([s, -s, z], -1),
                     np.stack([s, s, z], -1), np.stack([-s, s, z], -1)], -2)


def project(model, intr, dist, ext, view, marker, size, lens="radtan"):
    """Projection of the 4 tag corners through a pinhole + radial-tangential lens or an equidistant fisheye lens
    (numpy; used only to synthesise pixels).  Returns (uv (N,4,2), depth (N,4))."""
    return project_points(model, intr, dist, ext, view, marker, obj_points(size), lens)


def project_points(model, intr, dist, ext, view, marker, o, lens="radtan"):
    """project() of the object points o (N,4,3) in the marker frame instead of the square of a tag size."""
    Rm = rodrigues_np(marker[:, 0:3])
    Pw = np.einsum('nij,nkj->nki', Rm, o) + marker[:, None, 3:6]
    Rv = rodrigues_np(view[:, 0:3])
    q = np.einsum('nji,nkj->nki', Rv, Pw - view[:, None, 3:6])
    if model == "rig":
        Rx = rodrigues_np(ext[:, 0:3])
        q = np.einsum('nji,nkj->nki', Rx, q - ext[:, None, 3:6])
    Z = q[..., 2]
    if lens == "equidistant":
        # th = atan2(rho, Z), th_d = th (1 + k1 th^2 + k2 th^4 + k3 th^6 + k4 th^8), (xd, yd) = th_d (X, Y) / rho
        rho = np.hypot(q[..., 0], q[..., 1])
        th = np.arctan2(rho, Z)
        t2 = th * th
        k1, k2, k3, k4 = (dist[:, i:i + 1] for i in range(4))
        thd = th * (1 + t2 * (k1 + t2 * (k2 + t2 * (k3 + t2 * k4))))
        s = np.where(rho > 1e-12, thd / np.where(rho > 1e-12, rho, 1.0), 1.0 / np.where(Z > 1e-9, Z, 1e-9))
        xd, yd = s * q[..., 0], s * q[..., 1]
    else:
        Zs = np.where(np.abs(Z) < 1e-9, 1e-9, Z)
        x, y = q[..., 0] / Zs, q[..., 1] / Zs
        r2 = x * x + y * y
        k1, k2, p1, p2, k3 = (dist[:, i:i + 1] for i in range(5))
        rad = 1 + r2 * (k1 + r2 * (k2 + r2 * k3))
        xd = x * rad + 2 * p1 * x * y + p2 * (r2 + 2 * x * x)
        yd = y * rad + p1 * (r2 + 2 * y * y) + 2 * p2 * x * y
    u = intr[:, 0:1] * xd + intr[:, 2:3]
    v = intr[:, 1:2] * yd + intr[:, 3:4]
    return np.stack([u, v], -1), Z


# ---------------------------------------------------------------- scene container
@dataclass
class Scene:
    """Inputs of one bundle-adjustment problem (numpy, host)."""
    model: str                      # "single" | "rig"
    intr: np.ndarray                # (n_cam,4) fx fy cx cy         (initial guess)
    dist: np.ndarray                # (n_cam,5) k1 k2 p1 p2 k3 | equidistant: k1 k2 k3 k4 + reserved slot
    ext: np.ndarray                 # (n_cam,6) body_T_cam (rig) else zeros
    views: np.ndarray               # (n_views,6) world_T_camera | world_T_body
    markers: np.ndarray             # (n_markers,6) world_T_target
    sizes: np.ndarray               # (n_markers,)
    view_idx: np.ndarray            # (N,) int32
    marker_idx: np.ndarray          # (N,) int32
    cam_idx: np.ndarray             # (N,) int32
    pixels: np.ndarray              # (N,8) u0 v0 u1 v1 u2 v2 u3 v3
    const_views: np.ndarray = None
    const_markers: np.ndarray = None
    const_intr: np.ndarray = None
    const_dist: np.ndarray = None
    const_ext: np.ndarray = None
    truth: dict = field(default_factory=dict)   # ground-truth parameter arrays
    image_size: tuple = (640, 480)  # mixed lenses: one (width, height) per camera
    name: str = ""
    lens: str = "radtan"            # "radtan" | "equidistant" for every camera, or a tuple of one per camera
    corners: np.ndarray = None      # (n_slots,4,2) corner layout (rcc_ba_set_corner_layout) or None
    corner_slot: np.ndarray = None  # (N,) int32 layout slot of each block, -1: the square of the marker's size

    def __post_init__(self):
        nv, nm, nc = len(self.views), len(self.markers), len(self.intr)
        if self.const_views is None:
            self.const_views = np.zeros(nv, bool)
        if self.const_markers is None:
            self.const_markers = np.zeros(nm, bool)
            self.const_markers[0] = True          # gauge: world tag, camera_pose.cpp:71-80
        if self.const_intr is None:
            self.const_intr = np.zeros(nc, bool)
        if self.const_dist is None:
            self.const_dist = np.zeros(nc, bool)
        if self.const_ext is None:
            self.const_ext = np.zeros(nc, bool)
            if self.model == "rig":
                self.const_ext[0] = True          # gauge of the rig: body frame == camera 0

    @property
    def n_blocks(self):
        return len(self.view_idx)

    @property
    def n_observations(self):
        return 4 * len(self.view_idx)


# ---------------------------------------------------------------- generator
def _look_at(cam_pos, target, roll):
    """world_T_camera rotations with +z towards target, x right, y down."""
    z = target - cam_pos
    z /= np.linalg.norm(z, axis=-1, keepdims=True)
    up = np.array([0.0, -1.0, 0.0])
    x = np.cross(-up, z)                      # world "down" is +y_cam
    x /= np.linalg.norm(x, axis=-1, keepdims=True)
    y = np.cross(z, x)
    R = np.stack([x, y, z], -1)               # columns = camera axes in world
    cr, sr = np.cos(roll), np.sin(roll)
    Rz = np.zeros(roll.shape + (3, 3))
    Rz[..., 0, 0], Rz[..., 0, 1], Rz[..., 1, 0], Rz[..., 1, 1], Rz[..., 2, 2] = cr, -sr, sr, cr, 1
    return R @ Rz


def _wall_views(rng, n, wall_w, wall_h, d_mean, T0inv, tilt=0.0):
    """n views looking at random points of the wall from d in [0.7, 1.3] d_mean (tags face -z of the wall
    frame towards the cameras: wall normal is +z, the camera sits at negative z looking towards +z).
    tilt > 0 then turns each camera about its x and y axes by up to +-tilt rad (wide-angle lenses: the tags
    land far off the optical axis)."""
    tgt = np.stack([rng.uniform(-0.5, 0.5, n) * wall_w * 0.9,
                    rng.uniform(-0.5, 0.5, n) * wall_h * 0.9,
                    np.zeros(n)], -1)
    dist_cam = rng.uniform(0.7, 1.3, n) * d_mean
    off = rng.normal(0, 0.25, (n, 2))
    cam_pos = tgt + np.stack([off[:, 0] * dist_cam, off[:, 1] * dist_cam,
                              -dist_cam * np.sqrt(np.maximum(0.2, 1 - (off ** 2).sum(-1)))], -1)
    Rwc = _look_at(cam_pos, tgt, rng.normal(0, 0.2, n))
    views_wall = np.concatenate([rotation_to_rvec(Rwc), cam_pos], -1)
    if tilt > 0:
        turn = np.concatenate([rng.uniform(-tilt, tilt, (n, 2)), np.zeros((n, 4))], -1)
        views_wall = compose(views_wall, turn)
    return compose(np.broadcast_to(T0inv, views_wall.shape), views_wall)


def _chunk_observations(rng, v0, views_c, markers_t, sizes, intr_t, dist_t, ext_t, model, n_cam, visibility,
                        W, Himg, tag_size, dtype_idx, lens="radtan"):
    """Observation blocks of the views views_c (global view numbers v0, v0+1, ...): every tag whose 4 corners
    project inside the image with positive depth (equidistant: less than 85 degrees off the optical axis), thinned
    at random to the requested visibility."""
    n_markers = len(markers_t)
    nv = len(views_c)
    m_all = np.arange(n_markers)
    vi_l, mi_l, ci_l, px_l = [], [], [], []
    Rv = rodrigues_np(views_c[:, 0:3])                                       # (nv,3,3)
    # marker centres in the view/body frame: R^T (t_m - t_v)   (cheap conservative prefilter)
    ctr = np.einsum('vji,vmj->vmi', Rv, markers_t[None, :, 3:6] - views_c[:, None, 3:6])
    for c in range(n_cam):
        # mixed lenses: one lens and image size per camera
        lens_c = lens if isinstance(lens, str) else lens[c]
        W_c, H_c = (W, Himg) if np.ndim(W) == 0 else (W[c], Himg[c])
        pc = ctr
        if model == "rig":
            Rx = rodrigues_np(ext_t[c, 0:3])
            pc = (ctr - ext_t[c, 3:6]) @ Rx                                   # Rx^T (p - t_x)
        zc = np.maximum(pc[..., 2], 1e-9)
        if lens_c == "equidistant":
            cand = (pc[..., 2] > 0.05) & (np.arctan2(np.hypot(pc[..., 0], pc[..., 1]), pc[..., 2]) < np.deg2rad(88))
        else:
            margin = 0.35 * max(W_c, H_c) + intr_t[c, 0] * tag_size / zc          # distortion + tag extent
            cand = ((pc[..., 2] > 0.05)
                    & (np.abs(intr_t[c, 0] * pc[..., 0] / zc + intr_t[c, 2] - W_c / 2) < W_c / 2 + margin)
                    & (np.abs(intr_t[c, 1] * pc[..., 1] / zc + intr_t[c, 3] - H_c / 2) < H_c / 2 + margin))
        cv_, cm_ = np.nonzero(cand)
        uv_c, Z_c = project(model, np.broadcast_to(intr_t[c], (len(cv_), 4)),
                            np.broadcast_to(dist_t[c], (len(cv_), 5)),
                            np.broadcast_to(ext_t[c], (len(cv_), 6)),
                            views_c[cv_], markers_t[cm_], sizes[cm_], lens_c)
        ok_c = ((Z_c > 0.1).all(-1) & (uv_c[..., 0] >= 0).all(-1) & (uv_c[..., 0] < W_c).all(-1)
                & (uv_c[..., 1] >= 0).all(-1) & (uv_c[..., 1] < H_c).all(-1))
        if lens_c == "equidistant":
            # the corner itself, not only the tag centre, within 85 degrees of the optical axis
            Pq = _corners_in_camera(model, ext_t[c], views_c[cv_], markers_t[cm_], sizes[cm_])
            ok_c &= (np.arctan2(np.hypot(Pq[..., 0], Pq[..., 1]), Pq[..., 2]) < np.deg2rad(85)).all(-1)
        # scatter back to the dense (view, marker) grid the thinning below works on
        vv = np.repeat(np.arange(v0, v0 + nv), n_markers)
        mm = np.tile(m_all, nv)
        ok = np.zeros(nv * n_markers, bool)
        flat = cv_ * n_markers + cm_
        ok[flat[ok_c]] = True
        # thin to the requested visibility
        n_keep = int(round(visibility * n_markers))
        okm = ok.reshape(nv, n_markers)
        cnt = okm.sum(1)
        over = np.nonzero(cnt > n_keep)[0]
        if len(over):
            score = rng.random((nv, n_markers))
            score[~okm] = 2.0
            kth = np.partition(score[over], n_keep - 1, axis=1)[:, n_keep - 1]
            okm[over] &= score[over] <= kth[:, None]
        ok = okm.ravel()
        sel = np.nonzero(ok)[0]
        vi_l.append(vv[sel].astype(dtype_idx))
        mi_l.append(mm[sel].astype(dtype_idx))
        ci_l.append(np.full(len(sel), c, dtype_idx))
        pos = np.searchsorted(flat, sel)                      # flat is sorted (np.nonzero order)
        px_l.append(uv_c[pos].reshape(-1, 8))
    return np.concatenate(vi_l), np.concatenate(mi_l), np.concatenate(ci_l), np.concatenate(px_l)


def _corners_in_camera(model, ext, view, marker, size):
    """(N,4,3) tag corners in the camera frame."""
    o = obj_points(size)
    Pw = np.einsum('nij,nkj->nki', rodrigues_np(marker[:, 0:3]), o) + marker[:, None, 3:6]
    q = np.einsum('nji,nkj->nki', rodrigues_np(view[:, 0:3]), Pw - view[:, None, 3:6])
    if model == "rig":
        q = (q - ext[3:6]) @ rodrigues_np(ext[0:3])
    return q


def make_scene(n_markers, n_views, visibility, n_cam=1, model="single", seed=0,
               tag_size=0.1, pixel_noise=0.3, image_size=None,
               perturb=(0.02, 0.02, 0.01), round_pixels=False, chunk_views=256,
               name="", dtype_idx=np.int32, view_seed=None, blocked=False, view_range=None, threads=None,
               lens="radtan"):
    """Generate a synthetic marker scene.

    visibility : target fraction of tags seen per view (per camera); the wall
                 is sized so that the image footprint covers about that share.
    perturb    : (rad, m, relative-intrinsics) sigma of the initial guess.
    view_seed  : if given, views / observations / noise come from a second
                 generator seeded (seed, view_seed) while cameras and tags only
                 depend on `seed` -- weak-scaling shards share one tag cloud.
    round_pixels: truncate pixels to int like corner_detections.cpp:53-54.
    lens       : "radtan" (640 x 480, f ~ 600 px) or "equidistant": a wide-angle fisheye camera (1280 x 1024,
                 f ~ 330 px, k1..k4, reserved slot 0) whose views are turned by up to +-1.2 rad so that tags are
                 seen up to 85 degrees off the optical axis.  image_size overrides the default size.
                 A sequence of n_cam such names gives each camera its own lens, image size and intrinsics range
                 (Scene.image_size is then one size per camera).  In a rig the equidistant cameras other than
                 camera 0 are yawed a further 1 rad away from the body axis, so that they see the tags the body
                 looks at far off their own axis; the views are turned by up to +-0.6 rad when there is no such
                 camera to yaw (single model, or camera 0 equidistant).
    blocked    : every chunk of `chunk_views` views draws from its own random stream
                 (seed, chunk number): chunks are generated by `threads` host threads, and
                 `view_range=(lo, hi)` (multiples of chunk_views) yields exactly the views lo..hi-1 of the
                 full scene, renumbered from 0 -- the strong-scaling shards of one fixed problem.
                 The default (False) keeps the single sequential stream.
    """
    lenses = (lens,) if isinstance(lens, str) else tuple(lens)
    for name_ in lenses:
        if name_ not in ("radtan", "equidistant"):
            raise ValueError(f"unknown lens {name_!r}")
    if not isinstance(lens, str):
        if len(lenses) != n_cam:
            raise ValueError(f"{len(lenses)} lenses for {n_cam} cameras")
        if len(set(lenses)) == 1:
            lens = lenses[0]                    # one lens after all: the same scene as the name gives
    mixed = not isinstance(lens, str)
    fisheye = lens == "equidistant"
    rng = np.random.default_rng(seed)
    if not mixed:
        if image_size is None:
            image_size = (1280, 1024) if fisheye else (640, 480)
        W, Himg = image_size
        # ---- cameras (truth): SURVEY 8(d2)
        f_lo, f_hi = (320, 340) if fisheye else (550, 650)
        intr_t = np.stack([rng.uniform(f_lo, f_hi, n_cam), rng.uniform(f_lo, f_hi, n_cam),
                           W / 2 + rng.uniform(-10, 10, n_cam),
                           Himg / 2 + rng.uniform(-10, 10, n_cam)], -1)
        if fisheye:
            dist_t = np.stack([rng.normal(0, 0.02, n_cam), rng.normal(0, 0.01, n_cam),
                               rng.normal(0, 2e-3, n_cam), rng.normal(0, 5e-4, n_cam), np.zeros(n_cam)], -1)
        else:
            dist_t = np.stack([rng.normal(0, 0.1, n_cam), rng.normal(0, 0.05, n_cam),
                               rng.normal(0, 2e-3, n_cam), rng.normal(0, 2e-3, n_cam),
                               rng.normal(0, 0.01, n_cam)], -1)
    else:
        # each camera from its own lens's ranges; the wall below is sized for the radial-tangential default
        fish = np.array([name_ == "equidistant" for name_ in lenses])
        image_size = tuple(tuple(image_size) if image_size is not None else ((1280, 1024) if f_ else (640, 480))
                           for f_ in fish)
        W_cam = np.array([sz[0] for sz in image_size], dtype=np.float64)
        H_cam = np.array([sz[1] for sz in image_size], dtype=np.float64)
        f_lo, f_hi = np.where(fish, 320.0, 550.0), np.where(fish, 340.0, 650.0)
        intr_t = np.stack([rng.uniform(f_lo, f_hi), rng.uniform(f_lo, f_hi),
                           W_cam / 2 + rng.uniform(-10, 10, n_cam),
                           H_cam / 2 + rng.uniform(-10, 10, n_cam)], -1)
        dist_f = np.stack([rng.normal(0, 0.02, n_cam), rng.normal(0, 0.01, n_cam),
                           rng.normal(0, 2e-3, n_cam), rng.normal(0, 5e-4, n_cam), np.zeros(n_cam)], -1)
        dist_r = np.stack([rng.normal(0, 0.1, n_cam), rng.normal(0, 0.05, n_cam),
                           rng.normal(0, 2e-3, n_cam), rng.normal(0, 2e-3, n_cam),
                           rng.normal(0, 0.01, n_cam)], -1)
        dist_t = np.where(fish[:, None], dist_f, dist_r)
        W, Himg = (640, 480)
    ext_t = np.zeros((n_cam, 6))
    if model == "rig":
        # cameras fan out around the body's optical axis
        ang = np.linspace(-0.5, 0.5, n_cam) if n_cam > 1 else np.zeros(1)
        ext_t[:, 1] = ang                       # yaw
        ext_t[:, 3] = np.linspace(-0.1, 0.1, n_cam) if n_cam > 1 else 0.0
        ext_t[1:, 0:3] += rng.normal(0, 0.02, (n_cam - 1, 3))
        ext_t[1:, 3:6] += rng.normal(0, 0.01, (n_cam - 1, 3))
        ext_t[0] = 0.0                          # body frame == camera 0 (gauge)
        if mixed:
            # fisheye cameras look 1 rad further out: the tags the body looks at land far off their axis
            yaw_out = fish & (np.arange(n_cam) > 0)
            ext_t[yaw_out, 1] += np.where(ang[yaw_out] < 0, -1.0, 1.0)

    # ---- wall of tags: area so that footprint/area ~ visibility
    d_mean = 2.0
    f = 600.0
    foot = (W / f * d_mean) * (Himg / f * d_mean) * 0.6     # usable share (all 4 corners inside)
    area = max(foot / max(visibility, 1e-3), n_markers * (1.6 * tag_size) ** 2)
    d_mean = np.sqrt(area * max(visibility, 1e-3) / ((W / f) * (Himg / f) * 0.6))
    aspect = W / Himg
    wall_w, wall_h = np.sqrt(area * aspect), np.sqrt(area / aspect)
    # jittered grid so tags do not overlap pathologically
    gx = int(np.ceil(np.sqrt(n_markers * aspect)))
    gy = int(np.ceil(n_markers / gx))
    cells = rng.permutation(gx * gy)[:n_markers]
    cx_, cy_ = cells % gx, cells // gx
    mpos = np.stack([(cx_ + 0.5 + rng.uniform(-0.3, 0.3, n_markers)) / gx * wall_w - wall_w / 2,
                     (cy_ + 0.5 + rng.uniform(-0.3, 0.3, n_markers)) / gy * wall_h - wall_h / 2,
                     rng.uniform(-0.15, 0.15, n_markers) * d_mean / 2], -1)
    mrot = rng.normal(0, 0.25, (n_markers, 3))              # tilt up to ~ +-40 deg
    markers_t = np.concatenate([mrot, mpos], -1)
    # tag 0 defines the world frame (camera_pose.cpp:71-80): re-express everything in it
    T0inv = invert(markers_t[0:1])
    markers_t = compose(np.broadcast_to(T0inv, markers_t.shape), markers_t)
    markers_t[0] = 0.0
    sizes = np.full(n_markers, tag_size)
    s_r, s_t, s_i = perturb
    if mixed:
        obs_args = (markers_t, sizes, intr_t, dist_t, ext_t, model, n_cam, visibility, W_cam, H_cam, tag_size,
                    dtype_idx, lenses)
        tilt = 0.6 if (model != "rig" or fish[0]) else 0.0
    else:
        obs_args = (markers_t, sizes, intr_t, dist_t, ext_t, model, n_cam, visibility, W, Himg, tag_size, dtype_idx,
                    lens)
        tilt = 1.2 if fisheye else 0.0

    if blocked:
        # ---- one random stream per chunk of views: parallel, and any aligned view range on its own
        lo, hi = (0, n_views) if view_range is None else view_range
        if lo % chunk_views or not (0 <= lo <= hi <= n_views):
            raise ValueError("view_range must start on a multiple of chunk_views and lie inside 0..n_views")
        rng_shared = np.random.default_rng([seed, 7919])
        vs = [] if view_seed is None else [int(view_seed)]

        def one(v0):
            r = np.random.default_rng([seed, 104729, v0 // chunk_views] + vs)
            v1 = min(hi, v0 + chunk_views, n_views)
            vt = _wall_views(r, v1 - v0, wall_w, wall_h, d_mean, T0inv, tilt)
            vi, mi, ci, px = _chunk_observations(r, v0 - lo, vt, *obs_args)
            px = px + r.normal(0, pixel_noise, px.shape)
            v0g = vt + np.concatenate([r.normal(0, s_r, (v1 - v0, 3)), r.normal(0, s_t, (v1 - v0, 3))], -1)
            return vt, v0g, vi, mi, ci, px

        starts = list(range(lo, hi, chunk_views))
        if threads is None:
            import os
            threads = min(len(os.sched_getaffinity(0)), 16)
        if threads > 1 and len(starts) > 1:
            from concurrent.futures import ThreadPoolExecutor
            with ThreadPoolExecutor(max_workers=threads) as ex:
                parts = list(ex.map(one, starts))
        else:
            parts = [one(v0) for v0 in starts]
        views_t = np.concatenate([p[0] for p in parts]) if parts else np.zeros((0, 6))
        views0 = np.concatenate([p[1] for p in parts]) if parts else np.zeros((0, 6))
        view_idx, marker_idx, cam_idx, pixels = (np.concatenate([p[k] for p in parts]) for k in (2, 3, 4, 5))
        n_views = hi - lo
        rs = rng_shared
    else:
        if view_range is not None:
            raise ValueError("view_range needs blocked=True")
        if view_seed is not None:
            # initial guesses of the shared blocks must not depend on the shard either
            rng_shared = np.random.default_rng([seed, 7919])
            rng = np.random.default_rng([seed, int(view_seed)])
        else:
            rng_shared = None
        views_t = _wall_views(rng, n_views, wall_w, wall_h, d_mean, T0inv, tilt)
        # ---- observations (chunked over views so 10k x 5k scenes stay in memory)
        parts = [_chunk_observations(rng, v0, views_t[v0:min(n_views, v0 + chunk_views)], *obs_args)
                 for v0 in range(0, n_views, chunk_views)]
        view_idx, marker_idx, cam_idx, pixels = (np.concatenate([p[k] for p in parts]) for k in range(4))
        pixels = pixels + rng.normal(0, pixel_noise, pixels.shape)
        # ---- initial guess = truth perturbed
        views0 = views_t + np.concatenate([rng.normal(0, s_r, (n_views, 3)),
                                           rng.normal(0, s_t, (n_views, 3))], -1)
        rs = rng if rng_shared is None else rng_shared
    if round_pixels:
        pixels = np.trunc(pixels)               # int(...) truncation, corner_detections.cpp:53-54

    markers0 = markers_t + np.concatenate([rs.normal(0, s_r, (n_markers, 3)),
                                           rs.normal(0, s_t, (n_markers, 3))], -1)
    markers0[0] = 0.0
    intr0 = intr_t * (1 + rs.normal(0, s_i, intr_t.shape))
    dist0 = dist_t + rs.normal(0, s_i, dist_t.shape) * 0.1
    if fisheye:
        dist0[:, 4] = 0.0                       # the reserved slot
    elif mixed:
        dist0[fish, 4] = 0.0
    ext0 = ext_t.copy()
    if model == "rig" and n_cam > 1:
        ext0[1:] += np.concatenate([rs.normal(0, s_r, (n_cam - 1, 3)),
                                    rs.normal(0, s_t, (n_cam - 1, 3))], -1)
    return Scene(model=model, intr=intr0, dist=dist0, ext=ext0, views=views0,
                 markers=markers0, sizes=sizes, view_idx=view_idx, marker_idx=marker_idx,
                 cam_idx=cam_idx, pixels=pixels,
                 truth=dict(intr=intr_t, dist=dist_t, ext=ext_t, views=views_t,
                            markers=markers_t),
                 image_size=image_size, name=name, lens=lens)


# ---------------------------------------------------------------- rigid multi-tag targets
def board_layout(rows, cols, tag_size, spacing):
    """(rows*cols, 4, 2) corners bl br tr tl of the tags of a rows x cols board in the board frame, slot r*cols + c
    for tag (r, c): the origin is the bottom-left corner of tag 0, the tag axes are the board axes, and tag (r, c) is
    centred at (c (1 + spacing) s + s/2, r (1 + spacing) s + s/2) for s = tag_size (Kalibr AprilGrid: tagSpacing is
    the gap over the tag size)."""
    r, c = np.divmod(np.arange(rows * cols), cols)
    pitch = (1 + spacing) * tag_size
    ctr = np.stack([c * pitch + tag_size / 2, r * pitch + tag_size / 2], -1)
    h = tag_size / 2
    return ctr[:, None, :] + np.array([[-h, -h], [h, -h], [h, h], [-h, h]])


def make_target_scene(rows, cols, n_views, n_boards=1, n_free=0, n_cam=1, model="single", seed=0, tag_size=0.1,
                      spacing=0.3, distance=2.5, pixel_noise=0.3, perturb=(0.02, 0.02, 0.01), lens="radtan",
                      image_size=None, name=""):
    """A scene of rigid tag boards (Scene.corners / corner_slot): n_boards boards of rows x cols tags (board_layout,
    one marker block each, slot = tag number, shared by the boards) side by side on a wall, plus n_free free tags
    (slot -1) between them; marker 0 is board 0 at the world origin (the gauge).  Each of the n_views views (body
    poses of a rig) looks at a random point of the wall from about `distance` and sees every tag whose four corners
    project inside the image with positive depth (equidistant: within 85 degrees of the optical axis).  Cameras and
    lenses as make_scene, which this does not call and whose random streams it leaves alone."""
    lenses = (lens,) * n_cam if isinstance(lens, str) else tuple(lens)
    if len(lenses) != n_cam or any(x not in ("radtan", "equidistant") for x in lenses):
        raise ValueError(f"lens must be 'radtan', 'equidistant' or one of them per camera, got {lens!r}")
    rng = np.random.default_rng([seed, 52361])
    fish = np.array([x == "equidistant" for x in lenses])
    sizes_img = [tuple(image_size) if image_size is not None else ((1280, 1024) if f_ else (640, 480)) for f_ in fish]
    W = np.array([sz[0] for sz in sizes_img], dtype=np.float64)
    H = np.array([sz[1] for sz in sizes_img], dtype=np.float64)
    f_lo, f_hi = np.where(fish, 320.0, 550.0), np.where(fish, 340.0, 650.0)
    intr_t = np.stack([rng.uniform(f_lo, f_hi), rng.uniform(f_lo, f_hi), W / 2 + rng.uniform(-10, 10, n_cam),
                       H / 2 + rng.uniform(-10, 10, n_cam)], -1)
    dist_f = np.stack([rng.normal(0, 0.02, n_cam), rng.normal(0, 0.01, n_cam), rng.normal(0, 2e-3, n_cam),
                       rng.normal(0, 5e-4, n_cam), np.zeros(n_cam)], -1)
    dist_r = np.stack([rng.normal(0, 0.1, n_cam), rng.normal(0, 0.05, n_cam), rng.normal(0, 2e-3, n_cam),
                       rng.normal(0, 2e-3, n_cam), rng.normal(0, 0.01, n_cam)], -1)
    dist_t = np.where(fish[:, None], dist_f, dist_r)
    ext_t = np.zeros((n_cam, 6))
    if model == "rig" and n_cam > 1:
        ext_t[:, 1] = np.linspace(-0.3, 0.3, n_cam)
        ext_t[:, 3] = np.linspace(-0.1, 0.1, n_cam)
        ext_t[1:, 0:3] += rng.normal(0, 0.02, (n_cam - 1, 3))
        ext_t[1:, 3:6] += rng.normal(0, 0.01, (n_cam - 1, 3))
        ext_t[0] = 0.0
    # boards in a row along x with a gap of two tags, free tags in the gaps and below the boards
    layout = board_layout(rows, cols, tag_size, spacing)
    pitch = (1 + spacing) * tag_size
    bw, bh = cols * pitch, rows * pitch
    boards = np.zeros((n_boards, 6))
    boards[:, 3] = np.arange(n_boards) * (bw + 2 * pitch)
    boards[1:, 0:3] = rng.normal(0, 0.05, (n_boards - 1, 3))
    free = np.zeros((n_free, 6))
    free[:, 0:3] = rng.normal(0, 0.2, (n_free, 3))
    free[:, 3] = rng.uniform(-pitch, n_boards * (bw + 2 * pitch) - pitch, n_free)
    free[:, 4] = rng.uniform(-1.5 * pitch, bh + 0.5 * pitch, n_free)
    free[:, 5] = rng.uniform(-0.05, 0.05, n_free)
    markers_t = np.concatenate([boards, free])
    sizes = np.full(len(markers_t), tag_size)
    # every tag of the scene: (marker, slot, object points)
    tag_marker = np.concatenate([np.repeat(np.arange(n_boards), rows * cols), n_boards + np.arange(n_free)])
    tag_slot = np.concatenate([np.tile(np.arange(rows * cols), n_boards), np.full(n_free, -1)]).astype(np.int32)
    obj = np.concatenate([np.broadcast_to(np.concatenate([layout, np.zeros((rows * cols, 4, 1))], -1),
                                          (n_boards, rows * cols, 4, 3)).reshape(-1, 4, 3),
                          obj_points(np.full(n_free, tag_size))])
    # views: cameras at -z looking at random points of the wall (the tags face -z)
    wall_c = np.array([(n_boards * (bw + 2 * pitch) - 2 * pitch) / 2, bh / 2, 0.0])
    wall_w, wall_h = n_boards * (bw + 2 * pitch), bh
    tgt = wall_c + np.stack([rng.uniform(-0.4, 0.4, n_views) * wall_w, rng.uniform(-0.4, 0.4, n_views) * wall_h,
                             np.zeros(n_views)], -1)
    d = rng.uniform(0.8, 1.2, n_views) * distance
    off = rng.normal(0, 0.25, (n_views, 2))
    cam_pos = tgt + np.stack([off[:, 0] * d, off[:, 1] * d, -d * np.sqrt(np.maximum(0.2, 1 - (off ** 2).sum(-1)))], -1)
    Rwc = _look_at(cam_pos, tgt, rng.normal(0, 0.2, n_views))
    views_t = np.concatenate([rotation_to_rvec(Rwc), cam_pos], -1)
    vi_l, mi_l, ci_l, sl_l, px_l = [], [], [], [], []
    n_tags = len(tag_marker)
    for c in range(n_cam):
        vv, tt = np.repeat(np.arange(n_views), n_tags), np.tile(np.arange(n_tags), n_views)
        uv, Z = project_points(model, np.broadcast_to(intr_t[c], (len(vv), 4)), np.broadcast_to(dist_t[c], (len(vv), 5)),
                               np.broadcast_to(ext_t[c], (len(vv), 6)), views_t[vv], markers_t[tag_marker[tt]],
                               obj[tt], lenses[c])
        ok = ((Z > 0.1).all(-1) & (uv[..., 0] >= 0).all(-1) & (uv[..., 0] < W[c]).all(-1)
              & (uv[..., 1] >= 0).all(-1) & (uv[..., 1] < H[c]).all(-1))
        if fish[c]:
            Rm = rodrigues_np(markers_t[tag_marker[tt], 0:3])
            Pw = np.einsum('nij,nkj->nki', Rm, obj[tt]) + markers_t[tag_marker[tt], None, 3:6]
            q = np.einsum('nji,nkj->nki', rodrigues_np(views_t[vv, 0:3]), Pw - views_t[vv, None, 3:6])
            if model == "rig":
                q = (q - ext_t[c, 3:6]) @ rodrigues_np(ext_t[c, 0:3])
            ok &= (np.arctan2(np.hypot(q[..., 0], q[..., 1]), q[..., 2]) < np.deg2rad(85)).all(-1)
        vi_l.append(vv[ok]); mi_l.append(tag_marker[tt[ok]]); ci_l.append(np.full(ok.sum(), c))
        sl_l.append(tag_slot[tt[ok]]); px_l.append(uv[ok].reshape(-1, 8))
    view_idx, marker_idx, cam_idx, slot = (np.concatenate(x).astype(np.int32) for x in (vi_l, mi_l, ci_l, sl_l))
    pixels = np.concatenate(px_l) + rng.normal(0, pixel_noise, (len(view_idx), 8))
    s_r, s_t, s_i = perturb
    n_m = len(markers_t)
    views0 = views_t + np.concatenate([rng.normal(0, s_r, (n_views, 3)), rng.normal(0, s_t, (n_views, 3))], -1)
    markers0 = markers_t + np.concatenate([rng.normal(0, s_r, (n_m, 3)), rng.normal(0, s_t, (n_m, 3))], -1)
    markers0[0] = markers_t[0]
    intr0 = intr_t * (1 + rng.normal(0, s_i, intr_t.shape))
    dist0 = dist_t + rng.normal(0, s_i, dist_t.shape) * 0.1
    dist0[fish, 4] = 0.0
    ext0 = ext_t.copy()
    if model == "rig" and n_cam > 1:
        ext0[1:] += np.concatenate([rng.normal(0, s_r, (n_cam - 1, 3)), rng.normal(0, s_t, (n_cam - 1, 3))], -1)
    one = lenses[0] if len(set(lenses)) == 1 else lenses
    return Scene(model=model, intr=intr0, dist=dist0, ext=ext0, views=views0, markers=markers0, sizes=sizes,
                 view_idx=view_idx, marker_idx=marker_idx, cam_idx=cam_idx, pixels=pixels,
                 truth=dict(intr=intr_t, dist=dist_t, ext=ext_t, views=views_t, markers=markers_t),
                 image_size=sizes_img[0] if isinstance(one, str) else tuple(sizes_img), name=name, lens=one,
                 corners=layout, corner_slot=slot)


# ---------------------------------------------------------------- the BASELINE.json configs
def config_scene(cfg, scale=1.0, seed=None, **kw):
    """The five BASELINE.json configurations (SURVEY.md 8(d2)).

    cfg 1: 1 camera, 20 tags, 200 views, all visible        (<= 4k blocks / 16k obs)
    cfg 2: 1 camera, 500 tags, 5 000 views, 20 % visible     (~0.5 M blocks / 2 M obs)
    cfg 3: 4-camera rig, 2 000 tags, 20 000 body poses, ~25 tags/camera/pose
    cfg 4: 1 camera, 5 000 tags, 10 000 keyframes, 25 %      (~12.5 M blocks / 50 M obs)
    cfg 5: sweep -- n_obs given via scale (views scaled at fixed 5 000 tags)
    `scale` multiplies the number of views (weak-scaling shards, reduced tests).
    """
    seed = 20240 + cfg if seed is None else seed
    if cfg == 1:
        return make_scene(20, max(2, int(200 * scale)), 1.0, seed=seed, name="cfg1", **kw)
    if cfg == 2:
        return make_scene(500, max(2, int(5000 * scale)), 0.20, seed=seed, name="cfg2", **kw)
    if cfg == 3:
        return make_scene(2000, max(2, int(20000 * scale)), 25 / 2000, n_cam=4, model="rig",
                          seed=seed, name="cfg3", **kw)
    if cfg == 4:
        return make_scene(5000, max(2, int(10000 * scale)), 0.25, seed=seed, name="cfg4", **kw)
    if cfg == 5:
        # scale = millions of corner observations requested
        n_views = max(2, int(round(scale * 1e6 / 4 / (0.25 * 5000))))
        return make_scene(5000, n_views, 0.25, seed=seed, name=f"cfg5_{scale:g}M", **kw)
    raise ValueError(f"unknown config {cfg}")
