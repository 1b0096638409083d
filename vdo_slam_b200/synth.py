"""Seeded synthetic inputs shaped like the reference's workloads (SURVEY.md section 8(d)).

`make_batch_graph` emits the factor graph that `Optimizer::FullBatchOptimization` builds from a `Map`
(/root/reference/src/Optimizer.cc:1350-1755): camera-pose and per-frame object-motion SE(3) vertices,
static points (one vertex per track) and dynamic points (one vertex per observation), with
EdgeSE3Prior / EdgeSE3 (odometry, motion smoothness) / EdgeSE3PointXYZ / LandmarkMotionTernaryEdge factors and
the information / Huber constants of Optimizer.cc:1330-1335,1352 (full) or :190-195,213 (partial window).

No dataset is on disk (KITTI / OMD demo data are external downloads), so everything is procedural.
"""
from __future__ import annotations

import numpy as np

# float constants exactly as the reference declares them (`const float ...`), promoted to double on use
FULL_BATCH = dict(sigma2_cam=np.float32(0.001), sigma2_3d_sta=np.float32(80), sigma2_obj_smo=np.float32(0.001),
                  sigma2_obj=np.float32(100), sigma2_3d_dyn=np.float32(80), huber=np.float32(0.0001), prior_w=100000.0)
PARTIAL_BATCH = dict(sigma2_cam=np.float32(0.0001), sigma2_3d_sta=np.float32(16), sigma2_obj_smo=np.float32(0.1),
                     sigma2_obj=np.float32(20), sigma2_3d_dyn=np.float32(16), huber=np.float32(0.0001), prior_w=100000.0)


def _rot(axis: np.ndarray, ang: np.ndarray) -> np.ndarray:
    """Rodrigues; axis (...,3) unit, ang (...) -> (...,3,3)."""
    axis = np.asarray(axis, np.float64)
    ang = np.asarray(ang, np.float64)
    x, y, z = axis[..., 0], axis[..., 1], axis[..., 2]
    c, s = np.cos(ang), np.sin(ang)
    C = 1 - c
    R = np.stack([
        np.stack([c + x * x * C, x * y * C - z * s, x * z * C + y * s], -1),
        np.stack([y * x * C + z * s, c + y * y * C, y * z * C - x * s], -1),
        np.stack([z * x * C - y * s, z * y * C + x * s, c + z * z * C], -1)], -2)
    return R


def iso(R: np.ndarray, t: np.ndarray) -> np.ndarray:
    """(…,3,3),(…,3) -> (…,12) row-major R then t (the layout every C entry point uses)."""
    return np.concatenate([R.reshape(R.shape[:-2] + (9,)), t], -1)


def iso_R(T):
    return T[..., :9].reshape(T.shape[:-1] + (3, 3))


def iso_t(T):
    return T[..., 9:12]


def iso_mul(A, B):
    Ra, Rb = iso_R(A), iso_R(B)
    return iso(Ra @ Rb, (Ra @ iso_t(B)[..., None])[..., 0] + iso_t(A))


def iso_inv(A):
    Rt = np.swapaxes(iso_R(A), -1, -2)
    return iso(Rt, -(Rt @ iso_t(A)[..., None])[..., 0])


def iso_apply(A, p):
    return (iso_R(A) @ p[..., None])[..., 0] + iso_t(A)


def _small_iso(rng, n, sig_t, sig_r):
    ax = rng.normal(size=(n, 3))
    ax /= np.linalg.norm(ax, axis=1, keepdims=True)
    return iso(_rot(ax, rng.normal(scale=sig_r, size=n)), rng.normal(scale=sig_t, size=(n, 3)))


def make_batch_graph(n_frames=200, n_objects=5, n_static=40000, n_dynamic=10000, seed=4, consts=FULL_BATCH,
                     obj_span=None, geom_p=0.35, max_len=30, obs_sigma=0.05, odo_sigma_t=0.01,
                     odo_sigma_r=np.deg2rad(0.1)):
    """Config 4 (defaults) / config 5 (n_frames=1000, n_objects=50, n_static=800000, n_dynamic=200000,
    obj_span=(100, 400), seed=5) generator.  Returns a dict of C-contiguous arrays:

      se3 (C,12) f64 initial estimates [cameras 0..N-1, then motion vertices]; se3_gt
      pt (P,3) f64 initial estimates [static tracks, then dynamic observations in chain order]; pt_gt
      prior_v (1,) i32, prior_Z (1,12), prior_w (1,)
      se3e_ij (E,2) i32, se3e_Z (E,12), se3e_w (E,), se3e_delta (E,)      odometry then smoothness edges
      obs_cp (E,2) i32 [se3 idx, point idx], obs_z (E,3), obs_w, obs_delta
      ter_pph (E,3) i32 [p1, p2, motion se3 idx], ter_w, ter_delta
    """
    rng = np.random.default_rng(seed)
    N = int(n_frames)
    # ---- ground-truth camera trajectory: 1 m / frame along a gentle arc (0.3 deg / frame yaw) ----
    yaw = np.deg2rad(0.3) * np.arange(N)
    Rwc = _rot(np.tile([0.0, 1.0, 0.0], (N, 1)), yaw)
    fwd = (Rwc @ np.array([0.0, 0.0, 1.0]))
    twc = np.concatenate([np.zeros((1, 3)), np.cumsum(fwd[:-1], 0)], 0)
    cam_gt = iso(Rwc, twc)
    # odometry measurements Z_i = T_i^-1 T_{i+1} (+ noise); initial estimates = chained odometry from Identity
    Z = iso_mul(iso_mul(iso_inv(cam_gt[:-1]), cam_gt[1:]), _small_iso(rng, N - 1, odo_sigma_t, odo_sigma_r))
    cam_est = np.empty_like(cam_gt)
    cam_est[0] = cam_gt[0]
    for i in range(N - 1):
        cam_est[i + 1] = iso_mul(cam_est[i], Z[i])

    # ---- objects: constant world-frame rigid motion, visible over a frame span ----
    K = int(n_objects)
    if obj_span is None or K == 0:
        o_s = np.zeros(K, np.int64)
        o_e = np.full(K, N - 1, np.int64)
    else:
        lo, hi = obj_span
        span = rng.integers(min(lo, N - 1), min(hi, N - 1) + 1, size=K)
        o_s = np.array([rng.integers(0, N - s) for s in span], np.int64)
        o_e = o_s + span
    # pivot = object centre at its first frame, placed in front of the camera
    piv = iso_apply(cam_gt[o_s], np.stack([rng.uniform(-8, 8, K), rng.uniform(-1, 1, K), rng.uniform(8, 22, K)], -1)) if K else np.zeros((0, 3))
    Ro = _rot(np.tile([0.0, 1.0, 0.0], (K, 1)), rng.normal(scale=np.deg2rad(0.4), size=K)) if K else np.zeros((0, 3, 3))
    vel = (iso_R(cam_gt[o_s]) @ np.stack([rng.normal(scale=0.05, size=K), np.zeros(K), rng.uniform(0.7, 1.3, K)], -1)[..., None])[..., 0] if K else np.zeros((0, 3))
    Hobj = iso(Ro, piv - (Ro @ piv[..., None])[..., 0] + vel) if K else np.zeros((0, 12))
    # motion vertex index table: mot_idx[o, k] for transition k -> k+1, k in [o_s, o_e-1]
    mot_idx = -np.ones((K, max(N - 1, 1)), np.int64)
    nxt = N
    mot_obj, mot_k = [], []
    for k in range(N - 1):                       # frame-major like the reference's vertex creation order
        for o in range(K):
            if o_s[o] <= k < o_e[o]:
                mot_idx[o, k] = nxt
                nxt += 1
                mot_obj.append(o)
                mot_k.append(k)
    C = nxt
    mot_obj = np.asarray(mot_obj, np.int64)
    mot_k = np.asarray(mot_k, np.int64)
    se3_gt = np.concatenate([cam_gt, Hobj[mot_obj]], 0) if len(mot_obj) else cam_gt.copy()
    se3 = np.concatenate([cam_est, np.tile(iso(np.eye(3), np.zeros(3)), (len(mot_obj), 1))], 0)  # motions start at Identity (Optimizer.cc:1581)

    def track_lengths(n, cap):
        L = 3 + rng.geometric(geom_p, size=n) - 1
        return np.minimum(np.minimum(L, max_len), cap)

    # ---- static tracks ----
    Ns = int(n_static)
    Ls = track_lengths(Ns, N)
    s_start = (rng.random(Ns) * (N - Ls + 1)).astype(np.int64)
    s_pt_gt = iso_apply(cam_gt[s_start], np.stack([rng.uniform(-15, 15, Ns), rng.uniform(-2, 2, Ns), rng.uniform(5, 40, Ns)], -1))
    s_tid = np.repeat(np.arange(Ns), Ls)
    s_frame = s_start[s_tid] + (np.arange(Ls.sum()) - np.repeat(np.cumsum(Ls) - Ls, Ls))
    s_z = iso_apply(iso_inv(cam_gt[s_frame]), s_pt_gt[s_tid]) + rng.normal(scale=obs_sigma, size=(len(s_tid), 3))
    first = np.cumsum(Ls) - Ls
    s_pt_est = iso_apply(cam_est[s_frame[first]], s_z[first])          # Map::vp3DPointSta of the first sighting

    # ---- dynamic tracks ----
    Nd = int(n_dynamic) if K else 0
    d_obj = rng.integers(0, K, size=Nd) if Nd else np.zeros(0, np.int64)
    span_len = (o_e - o_s + 1)
    Ld = track_lengths(Nd, 10 ** 9)
    Ld = np.minimum(Ld, span_len[d_obj]) if Nd else Ld
    d_start = o_s[d_obj] + (rng.random(Nd) * (span_len[d_obj] - Ld + 1)).astype(np.int64) if Nd else np.zeros(0, np.int64)
    # object centre at frame k: apply H repeatedly to the pivot; tabulate per object
    centre = np.zeros((K, N, 3))
    for o in range(K):
        c = piv[o].copy()
        for k in range(o_s[o], o_e[o] + 1):
            centre[o, k] = c
            c = Ro[o] @ c + iso_t(Hobj[o])
    p0 = centre[d_obj, d_start] + rng.uniform(-1.0, 1.0, size=(Nd, 3)) if Nd else np.zeros((0, 3))
    nd_obs = int(Ld.sum()) if Nd else 0
    d_tid = np.repeat(np.arange(Nd), Ld)
    d_pos = np.arange(nd_obs) - np.repeat(np.cumsum(Ld) - Ld, Ld)
    d_frame = d_start[d_tid] + d_pos
    d_pt_gt = np.zeros((nd_obs, 3))
    cur = p0.copy()
    offs = np.cumsum(Ld) - Ld
    for j in range(int(Ld.max()) if Nd else 0):      # propagate p_{k+1} = H p_k for all tracks still alive
        alive = np.nonzero(Ld > j)[0]
        d_pt_gt[offs[alive] + j] = cur[alive]
        cur[alive] = (Ro[d_obj[alive]] @ cur[alive][..., None])[..., 0] + iso_t(Hobj[d_obj[alive]])
    d_z = iso_apply(iso_inv(cam_gt[d_frame]), d_pt_gt) + rng.normal(scale=obs_sigma, size=(nd_obs, 3))
    d_pt_est = iso_apply(cam_est[d_frame], d_z)

    pt_gt = np.concatenate([s_pt_gt, d_pt_gt], 0)
    pt = np.concatenate([s_pt_est, d_pt_est], 0)
    P = len(pt)

    # ---- edges ----
    f = lambda v: 1.0 / float(v)
    hub = float(consts["huber"])
    obs_cp = np.concatenate([np.stack([s_frame, s_tid], -1), np.stack([d_frame, Ns + np.arange(nd_obs)], -1)], 0).astype(np.int32)
    obs_z = np.concatenate([s_z, d_z], 0)
    obs_w = np.concatenate([np.full(len(s_tid), f(consts["sigma2_3d_sta"])), np.full(nd_obs, f(consts["sigma2_3d_dyn"]))])
    obs_delta = np.full(len(obs_w), hub)
    not_last = d_pos < (Ld[d_tid] - 1) if Nd else np.zeros(0, bool)
    t_p1 = Ns + np.nonzero(not_last)[0]
    ter_pph = np.stack([t_p1, t_p1 + 1, mot_idx[d_obj[d_tid[not_last]], d_frame[not_last]]], -1).astype(np.int32) if Nd else np.zeros((0, 3), np.int32)
    assert (ter_pph[:, 2] >= N).all() if len(ter_pph) else True
    ter_w = np.full(len(ter_pph), f(consts["sigma2_obj"]))
    ter_delta = np.full(len(ter_pph), hub)
    # odometry + smoothness (Optimizer.cc:1383-1399, :1596-1623; smoothness only for frame index i>2, i.e. k>=2)
    odo_ij = np.stack([np.arange(N - 1), np.arange(1, N)], -1)
    sm = [(mot_idx[o, k - 1], mot_idx[o, k]) for k in range(2, N - 1) for o in range(K) if mot_idx[o, k] >= 0 and mot_idx[o, k - 1] >= 0]
    sm_ij = np.asarray(sm, np.int64).reshape(-1, 2)
    se3e_ij = np.concatenate([odo_ij, sm_ij], 0).astype(np.int32)
    se3e_Z = np.concatenate([Z, np.tile(iso(np.eye(3), np.zeros(3)), (len(sm_ij), 1))], 0)
    se3e_w = np.concatenate([np.full(N - 1, f(consts["sigma2_cam"])), np.full(len(sm_ij), f(consts["sigma2_obj_smo"]))])
    se3e_delta = np.full(len(se3e_w), hub)

    g = dict(se3=se3, se3_gt=se3_gt, pt=pt, pt_gt=pt_gt, n_cam=N,
             prior_v=np.zeros(1, np.int32), prior_Z=cam_est[:1].copy(), prior_w=np.array([float(consts["prior_w"])]),
             se3e_ij=se3e_ij, se3e_Z=se3e_Z, se3e_w=se3e_w, se3e_delta=se3e_delta,
             obs_cp=obs_cp, obs_z=obs_z, obs_w=obs_w, obs_delta=obs_delta,
             ter_pph=ter_pph, ter_w=ter_w, ter_delta=ter_delta)
    for k, v in list(g.items()):
        if isinstance(v, np.ndarray):
            g[k] = np.ascontiguousarray(v, dtype=np.int32 if v.dtype.kind == "i" else np.float64)
    assert P == g["pt"].shape[0] and C == g["se3"].shape[0]
    return g


def graph_sizes(g) -> dict:
    return dict(C=len(g["se3"]), P=len(g["pt"]), E_p=len(g["obs_cp"]), E_t=len(g["ter_pph"]), E_o=len(g["se3e_ij"]), E_prior=len(g["prior_v"]))


def algorithmic_bytes_per_iter(g) -> int:
    """SURVEY.md section 8(d): bytes one LM linearisation must move in the explicit-block formulation."""
    s = graph_sizes(g)
    return 216 * s["E_p"] + 412 * s["E_t"] + 416 * s["E_o"] + 96 * s["P"] + 272 * s["C"]


# ---------------------------------------------------------------------------------------------------------------------
# Config 2: one Optimizer::PoseOptimizationFlow2 problem (SURVEY.md section 8(d))
# ---------------------------------------------------------------------------------------------------------------------
KITTI_K = np.array([721.5377, 721.5377, 609.5593, 172.8540], np.float32)   # example/kitti-0000-0013.yaml:8-11


def make_flow_problem(n=2000, seed=1234, outlier_frac=0.10, flow_sigma=0.3, width=1242, height=375,
                      rot_deg=2.0, trans=(0.3, 0.02, 1.0), init_sigma=(0.01, 0.05), depth_range=(4.0, 25.0)):
    """Returns float32 arrays shaped like the reference's inputs: pts (n,2) last-frame pixels, depth (n,), flow (n,2)
    measured optical flow, K (4,), Tcw_last (4,4) (= identity: Twl = I), T_init (4,4), plus T_true (4,4 f64)."""
    rng = np.random.default_rng(seed)
    fx, fy, cx, cy = [float(v) for v in KITTI_K]
    pts = np.stack([rng.uniform(50, width - 50, n), rng.uniform(25, height - 25, n)], -1)
    depth = rng.uniform(*depth_range, n)
    X = np.stack([(pts[:, 0] - cx) * depth / fx, (pts[:, 1] - cy) * depth / fy, depth], -1)
    R = _rot(np.array([0.0, 1.0, 0.0]), np.deg2rad(rot_deg))
    t = np.asarray(trans, np.float64)
    Xc = X @ R.T + t
    proj = np.stack([Xc[:, 0] / Xc[:, 2] * fx + cx, Xc[:, 1] / Xc[:, 2] * fy + cy], -1)
    flow = proj - pts + rng.normal(scale=flow_sigma, size=(n, 2))
    out = rng.random(n) < outlier_frac
    flow[out] += rng.uniform(-15, 15, size=(int(out.sum()), 2))
    T_true = np.eye(4); T_true[:3, :3] = R; T_true[:3, 3] = t
    ax = rng.normal(size=3); ax /= np.linalg.norm(ax)
    dT = np.eye(4); dT[:3, :3] = _rot(ax, rng.normal(scale=init_sigma[0])); dT[:3, 3] = rng.normal(scale=init_sigma[1], size=3)
    T_init = T_true @ dT
    return dict(pts=pts.astype(np.float32), depth=depth.astype(np.float32), flow=flow.astype(np.float32), K=KITTI_K.copy(),
                Tcw_last=np.eye(4, dtype=np.float32), T_init=T_init.astype(np.float32), T_true=T_true, outlier=out)


# ---------------------------------------------------------------------------------------------------------------------
# Config 3 building block: one synthetic KITTI-shaped RGB-D frame (gray, raw depth, optical flow, semantic mask)
# ---------------------------------------------------------------------------------------------------------------------
KITTI_BF, KITTI_DEPTH_FACTOR = np.float32(387.5744), np.float32(256.0)


def make_frame(seed=0, width=1242, height=375, n_rect=3500, n_obj=4):
    """gray u8 (H,W): blocky texture so FAST fires a few thousand times; depth_raw f32 (H,W): disparity*256 as
    example/vdo_slam.cc feeds it (negative = invalid); flow f32 (H,W,2); mask i32 (H,W) with objects labelled 1..n_obj."""
    rng = np.random.default_rng(seed)
    gray = np.full((height, width), 110, np.uint8)
    x0 = rng.integers(0, width - 8, n_rect); y0 = rng.integers(0, height - 8, n_rect)
    ww = rng.integers(6, 60, n_rect); hh = rng.integers(6, 40, n_rect); val = rng.integers(20, 236, n_rect)
    for i in range(n_rect):
        gray[y0[i]:y0[i] + hh[i], x0[i]:x0[i] + ww[i]] = val[i]
    gray = np.clip(gray.astype(np.int16) + rng.integers(-3, 4, gray.shape), 0, 255).astype(np.uint8)
    yy, xx = np.mgrid[0:height, 0:width].astype(np.float32)
    z = (6.0 + 50.0 * (1.0 - yy / height) + 2.0 * np.sin(xx / 90.0)).astype(np.float32)     # far at the top, near at the bottom
    mask = np.zeros((height, width), np.int32)
    flow = np.stack([-(xx - width / 2) * 0.01 - 0.3, (yy - height / 2) * 0.012 + 0.2], -1).astype(np.float32)
    for o in range(n_obj):
        ow, oh = int(rng.integers(60, 200)), int(rng.integers(40, 110))
        ox, oy = int(rng.integers(20, width - ow - 20)), int(rng.integers(height // 3, height - oh - 10))
        mask[oy:oy + oh, ox:ox + ow] = o + 1
        z[oy:oy + oh, ox:ox + ow] = np.float32(rng.uniform(6, 22))
        flow[oy:oy + oh, ox:ox + ow] = np.array([rng.uniform(-6, 6), rng.uniform(-1.5, 1.5)], np.float32)
    depth_raw = (KITTI_BF * KITTI_DEPTH_FACTOR / z).astype(np.float32)
    bad = rng.random((height, width)) < 0.01
    depth_raw[bad] = -1.0                                        # invalid disparities
    flow[rng.random((height, width)) < 0.01] = 0.0               # exact zeros exercise the flow != 0 test
    return dict(gray=gray, depth_raw=depth_raw, flow=flow, mask=mask)


# ---------------------------------------------------------------------------------------------------------------------
# Config 3: synthetic KITTI-shape RGB-D sequence with geometry-consistent depth / flow / masks (SURVEY.md 8d).
# A corridor (ground plane, two side walls, far wall) seen from a camera on a gentle arc, plus rigid fronto-parallel boxes that
# translate with constant velocity.  Depth is rendered by ray casting, flow is the exact projection of each pixel's world point
# (moved with its object) into the next camera plus N(0, flow_sigma^2); the gray image only has to make FAST fire (the pipeline
# never matches appearance, it follows the flow).
# ---------------------------------------------------------------------------------------------------------------------
def _cam_pose(t, speed=0.8, yaw_rate=0.002):
    """camera-to-world (Twc) at frame t: forward motion on a gentle arc (y down, z forward)."""
    yaw = yaw_rate * t
    c, s = np.cos(yaw), np.sin(yaw)
    R = np.array([[c, 0, s], [0, 1, 0], [-s, 0, c]])
    # integrate the arc in closed form for small yaw_rate
    pos = np.array([speed * (1 - np.cos(yaw)) / yaw_rate, 0.0, speed * np.sin(yaw) / yaw_rate]) if yaw_rate else np.array([0, 0, speed * t])
    T = np.eye(4); T[:3, :3] = R; T[:3, 3] = pos
    return T


def make_sequence_frame(t, seed=0, width=1242, height=375, n_obj=3, flow_sigma=0.2, K=None, cam_h=1.65, half_w=7.0, depth_factor=KITTI_DEPTH_FACTOR):
    """Frame t of the sequence `seed`.  Returns dict(gray, depth_raw (disparity*depth_factor, f32: 256 = KITTI's DepthMapFactor, 1000 =
    OMD's), flow (H,W,2 to frame t+1), mask, Twc (4x4 f64 ground truth), obj_ids (semantic ids visible), K)."""
    K = KITTI_K if K is None else K
    fx, fy, cx, cy = [float(v) for v in K]
    rng_o = np.random.default_rng(1000 + seed)
    objs = []
    for o in range(n_obj):
        objs.append(dict(id=o + 1, x=float(rng_o.uniform(-4.0, 4.0)), z0=float(rng_o.uniform(9.0, 18.0)) + 2.0 * o,
                         vz=float(rng_o.uniform(0.55, 1.0)), vx=float(rng_o.uniform(-0.02, 0.02)), w=float(rng_o.uniform(1.6, 2.4)), h=float(rng_o.uniform(1.3, 1.8))))
    T0, T1 = _cam_pose(t), _cam_pose(t + 1)
    vv, uu = np.mgrid[0:height, 0:width].astype(np.float64)
    d_cam = np.stack([(uu - cx) / fx, (vv - cy) / fy, np.ones_like(uu)], -1)
    d_w = d_cam @ T0[:3, :3].T
    c_w = T0[:3, 3]
    big = 1e9
    with np.errstate(divide="ignore", invalid="ignore"):
        lam = np.full(uu.shape, big)
        # ground y = cam_h, walls x = +-half_w, far wall z = c_z + 400
        for axis, val in ((1, cam_h), (0, half_w), (0, -half_w), (2, c_w[2] + 400.0)):
            l = (val - c_w[axis]) / d_w[..., axis]
            l = np.where((l > 0) & np.isfinite(l), l, big)
            lam = np.minimum(lam, l)
        mask = np.zeros(uu.shape, np.int32)
        vel = np.zeros(uu.shape + (3,))
        for ob in objs:
            zc = ob["z0"] + ob["vz"] * t; xc = ob["x"] + ob["vx"] * t
            l = (zc - c_w[2]) / d_w[..., 2]
            P = c_w + l[..., None] * d_w
            hit = (l > 0) & (l < lam) & (np.abs(P[..., 0] - xc) < ob["w"] / 2) & (P[..., 1] < cam_h) & (P[..., 1] > cam_h - ob["h"])
            lam = np.where(hit, l, lam); mask[hit] = ob["id"]; vel[hit] = [ob["vx"], 0.0, ob["vz"]]
    Pw = c_w + lam[..., None] * d_w
    z = lam.copy()                                  # d_cam has unit z: lambda is the camera-frame depth
    Pn = Pw + vel
    Pc1 = (Pn - T1[:3, 3]) @ T1[:3, :3]             # R^T (P - c)
    u1 = fx * Pc1[..., 0] / Pc1[..., 2] + cx; v1 = fy * Pc1[..., 1] / Pc1[..., 2] + cy
    rng = np.random.default_rng(7919 * seed + t)
    flow = np.stack([u1 - uu, v1 - vv], -1) + rng.normal(0, flow_sigma, uu.shape + (2,))
    flow = flow.astype(np.float32)
    flow[rng.random(uu.shape) < 0.005] = 0.0
    disp = np.round(KITTI_BF * np.float32(depth_factor) / np.maximum(z, 0.5))
    depth_raw = disp.astype(np.float32)
    depth_raw[rng.random(uu.shape) < 0.005] = -1.0
    gray = make_frame(seed=31 * seed + t, width=width, height=height, n_obj=0)["gray"]
    ids = [ob["id"] for ob in objs if (mask == ob["id"]).any()]
    return dict(gray=gray, depth_raw=depth_raw, flow=flow, mask=mask, Twc=T0, obj_ids=ids, K=np.asarray(K, np.float32))
