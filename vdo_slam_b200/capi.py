"""ctypes binding of libvdo_b200.so (C ABI in include/vdo_b200.h).

The library is built in-tree by `__graft_entry__.build()` (nvcc, sm_100a).  There is no CPU fallback: if the
shared object is missing or no CUDA device is usable, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvdo_b200.so")


class LMOptions(C.Structure):
    _fields_ = [("max_iterations", C.c_int), ("gain_threshold", C.c_double), ("max_trials", C.c_int),
                ("pcg_rel_tol", C.c_double), ("pcg_max_iterations", C.c_int), ("verbose", C.c_int),
                ("force_all_iterations", C.c_int), ("pcg_loose_tol", C.c_double), ("pcg_switch_gain", C.c_double)]


class LMStats(C.Structure):
    _fields_ = [("iterations", C.c_int), ("trials", C.c_int), ("pcg_iterations", C.c_int),
                ("initial_chi2", C.c_double), ("final_chi2", C.c_double), ("final_lambda", C.c_double),
                ("ms_linearize", C.c_double), ("ms_solve", C.c_double), ("ms_total", C.c_double),
                ("kernel_launches", C.c_int)]

    def asdict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class VdoError(RuntimeError):
    pass


_libs = {}


def load(path: str | None = None) -> C.CDLL:
    path = path or LIB_PATH
    if path in _libs:
        return _libs[path]
    if not os.path.exists(path):
        raise VdoError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). "
                       "There is no CPU fallback.")
    L = C.CDLL(path)
    L.vdo_last_error.restype = C.c_char_p
    L.vdo_ctx_stream.restype = C.c_uint64
    # the structs below are mirrored by hand: refuse a library whose layout differs (it would write past the ctypes buffers)
    for name, cls in (("vdo_lm_options", LMOptions), ("vdo_lm_stats", LMStats), ("vdo_tracker_params", globals().get("TrackerParams"))):
        if cls is not None and hasattr(L, "vdo_abi_struct_size"):
            n = L.vdo_abi_struct_size(name.encode())
            if n != C.sizeof(cls):
                raise VdoError(f"{path}: sizeof({name}) is {n} in the library but {C.sizeof(cls)} in capi.py -- rebuild the library or update the binding")
    _libs[path] = L
    return L


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int))


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


class Context:
    """vdo_ctx: one per System (device + stream)."""

    def __init__(self, device: int = 0, lib_path: str | None = None):
        self.L = load(lib_path)
        self.h = C.c_void_p()
        rc = self.L.vdo_ctx_create(C.c_int(device), C.byref(self.h))
        if rc != 0:
            raise VdoError(f"vdo_ctx_create(device={device}) failed with {rc}: no usable CUDA device (no CPU fallback)")

    def check(self, rc: int, what: str):
        if rc != 0:
            raise VdoError(f"{what} failed with {rc}: {self.L.vdo_last_error(self.h).decode()}")

    @property
    def stream(self) -> int:
        return int(self.L.vdo_ctx_stream(self.h))

    rank, world = 0, 1

    def init_comm(self, rank: int, world: int, dist=None):
        """Multi-GPU: create the NCCL communicator of this context (id from rank 0, broadcast through torch.distributed)."""
        self.rank, self.world = rank, world
        if world <= 1:
            return
        import torch
        dist = dist or torch.distributed
        buf = C.create_string_buffer(128)
        if rank == 0:
            self.check(self.L.vdo_nccl_unique_id(buf), "vdo_nccl_unique_id")
        dev = "cuda" if dist.get_backend() == "nccl" else "cpu"
        t = torch.frombuffer(bytearray(buf.raw), dtype=torch.uint8).clone().to(dev)
        dist.broadcast(t, src=0)
        idb = bytes(t.cpu().numpy().tobytes())
        self.check(self.L.vdo_ctx_init_comm(self.h, C.c_int(rank), C.c_int(world), C.c_char_p(idb)), "vdo_ctx_init_comm")

    def set_collective_emul(self, rank: int, world: int, dist):
        """TEST ONLY (tests/emul/libvdo_emul.so): all-reduce of the emulated backend through torch.distributed (gloo)."""
        import torch
        self.rank, self.world = rank, world
        CB = C.CFUNCTYPE(None, C.POINTER(C.c_double), C.c_size_t, C.c_int, C.c_void_p)

        def _cb(ptr, n, op, user):
            a = np.ctypeslib.as_array(ptr, shape=(n,))
            t = torch.from_numpy(a)
            dist.all_reduce(t, op=dist.ReduceOp.SUM if op == 0 else dist.ReduceOp.MAX)

        self._cb = CB(_cb)
        self.check(self.L.vdo_emul_set_collective(self.h, C.c_int(rank), C.c_int(world), self._cb, None), "vdo_emul_set_collective")

    def close(self):
        if self.h:
            self.L.vdo_ctx_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def g2o_read(ctx: "Context", path: str) -> dict:
    """Parse a .g2o file (the reference's optimizer.save() dumps) into the dict layout of synth.make_batch_graph plus the file
    ids (se3_id / pt_id / fixed_id) and the information matrices as written (prior_info / se3e_info: n x 21, obs_info /
    ter_info: n x 6, upper triangles)."""
    L = ctx.L
    h = C.c_void_p()
    rc = L.vdo_g2o_read(path.encode(), C.byref(h))
    if rc != 0:
        L.vdo_g2o_error.restype = C.c_char_p
        msg = L.vdo_g2o_error(h).decode() if h else "cannot open"
        if h:
            L.vdo_g2o_free(h)
        raise VdoError(f"vdo_g2o_read({path}) failed ({rc}): {msg}")
    try:
        cnt = (C.c_int64 * 8)()
        ctx.check(L.vdo_g2o_counts(h, cnt), "vdo_g2o_counts")
        n_se3, n_pt, n_pr, n_se, n_ob, n_te, n_fix, n_off = list(cnt)

        def geti(name, shape):
            a = np.zeros(shape, np.int32)
            ctx.check(L.vdo_g2o_get_i32(h, name.encode(), _ip(a), C.c_int64(a.size)), name)
            return a

        def getf(name, shape):
            a = np.zeros(shape, np.float64)
            ctx.check(L.vdo_g2o_get_f64(h, name.encode(), _dp(a), C.c_int64(a.size)), name)
            return a
        g = {"se3": getf("se3", (n_se3, 12)), "pt": getf("pt", (n_pt, 3)), "se3_id": geti("se3_id", (n_se3,)), "pt_id": geti("pt_id", (n_pt,)),
             "fixed_id": geti("fixed_id", (n_fix,)), "prior_v": geti("prior_v", (n_pr,)), "prior_Z": getf("prior_Z", (n_pr, 12)),
             "prior_info": getf("prior_info", (n_pr, 21)), "se3e_ij": geti("se3e_ij", (n_se, 2)), "se3e_Z": getf("se3e_Z", (n_se, 12)),
             "se3e_info": getf("se3e_info", (n_se, 21)), "obs_cp": geti("obs_cp", (n_ob, 2)), "obs_z": getf("obs_z", (n_ob, 3)),
             "obs_info": getf("obs_info", (n_ob, 6)), "ter_pph": geti("ter_pph", (n_te, 3)), "ter_meas": getf("ter_meas", (n_te, 3)),
             "ter_info": getf("ter_info", (n_te, 6)), "offset": getf("offset", (n_off, 13))}
        g["prior_w"] = g["prior_info"][:, 0].copy(); g["se3e_w"] = g["se3e_info"][:, 0].copy()
        g["obs_w"] = g["obs_info"][:, 0].copy(); g["ter_w"] = g["ter_info"][:, 0].copy()
        return g
    finally:
        L.vdo_g2o_free(h)


def g2o_write(ctx: "Context", path: str, g: dict, precision: int = 0):
    """Write a graph in the make_batch_graph layout as a .g2o file (ids from g['se3_id'] / g['pt_id'] when present)."""
    se3, pt = _f64(g["se3"]), _f64(g["pt"])
    sid = _i32(g["se3_id"]) if "se3_id" in g else None
    pid = _i32(g["pt_id"]) if "pt_id" in g else None
    fix = _i32(g.get("fixed_id", np.zeros(0, np.int32)))
    pv, pZ, pw = _i32(g["prior_v"]), _f64(g["prior_Z"]), _f64(g["prior_w"])
    ij, sZ, sw = _i32(g["se3e_ij"]), _f64(g["se3e_Z"]), _f64(g["se3e_w"])
    cp, oz, ow = _i32(g["obs_cp"]), _f64(g["obs_z"]), _f64(g["obs_w"])
    pph, tw = _i32(g["ter_pph"]), _f64(g["ter_w"])
    ctx.check(ctx.L.vdo_g2o_write(path.encode(), len(se3), _dp(se3), _ip(sid) if sid is not None else None, len(pt), _dp(pt),
                                  _ip(pid) if pid is not None else None, len(fix), _ip(fix), len(pv), _ip(pv), _dp(pZ), _dp(pw), len(sw), _ip(ij), _dp(sZ), _dp(sw),
                                  len(ow), _ip(cp), _dp(oz), _dp(ow), len(tw), _ip(pph), _dp(tw), int(precision)), "vdo_g2o_write")


class BatchGraph:
    """vdo_graph: the factor graph of Optimizer::FullBatchOptimization / PartialBatchOptimization."""

    @classmethod
    def from_g2o(cls, ctx: "Context", path: str, delta_se3: float, delta_pointxyz: float, delta_motion: float):
        """Load a .g2o file straight into a finalised graph (vdo_g2o_read + vdo_graph_from_g2o)."""
        L = ctx.L
        f = C.c_void_p()
        rc = L.vdo_g2o_read(path.encode(), C.byref(f))
        if rc != 0:
            if f:
                L.vdo_g2o_free(f)
            raise VdoError(f"vdo_g2o_read({path}) failed ({rc})")
        try:
            cnt = (C.c_int64 * 8)()
            ctx.check(L.vdo_g2o_counts(f, cnt), "vdo_g2o_counts")
            self = cls.__new__(cls)
            self.ctx, self.h = ctx, C.c_void_p()
            self.n_se3, self.n_pt = int(cnt[0]), int(cnt[1])
            ctx.check(L.vdo_graph_from_g2o(ctx.h, f, C.c_double(delta_se3), C.c_double(delta_pointxyz), C.c_double(delta_motion), C.byref(self.h)), "vdo_graph_from_g2o")
            return self
        finally:
            L.vdo_g2o_free(f)

    def __init__(self, ctx: Context, g: dict):
        """g: dict in the layout of vdo_slam_b200.synth.make_batch_graph."""
        self.ctx, L = ctx, ctx.L
        self.h = C.c_void_p()
        ctx.check(L.vdo_graph_create(ctx.h, C.byref(self.h)), "vdo_graph_create")
        se3, pt = _f64(g["se3"]), _f64(g["pt"])
        self.n_se3, self.n_pt = len(se3), len(pt)
        ctx.check(L.vdo_graph_set_vertices(self.h, len(se3), _dp(se3), len(pt), _dp(pt)), "vdo_graph_set_vertices")
        if len(g["prior_v"]):
            v, Z, w = _i32(g["prior_v"]), _f64(g["prior_Z"]), _f64(g["prior_w"])
            ctx.check(L.vdo_graph_add_edges_se3_prior(self.h, len(v), _ip(v), _dp(Z), _dp(w)), "add_edges_se3_prior")
        if len(g["se3e_ij"]):
            ij, Z, w, dl = _i32(g["se3e_ij"]), _f64(g["se3e_Z"]), _f64(g["se3e_w"]), _f64(g["se3e_delta"])
            ctx.check(L.vdo_graph_add_edges_se3(self.h, len(w), _ip(ij), _dp(Z), _dp(w), _dp(dl)), "add_edges_se3")
        if len(g["obs_cp"]):
            cp, z, w, dl = _i32(g["obs_cp"]), _f64(g["obs_z"]), _f64(g["obs_w"]), _f64(g["obs_delta"])
            ctx.check(L.vdo_graph_add_edges_se3_pointxyz(self.h, len(w), _ip(cp), _dp(z), _dp(w), _dp(dl)), "add_edges_se3_pointxyz")
        if len(g["ter_pph"]):
            pph, w, dl = _i32(g["ter_pph"]), _f64(g["ter_w"]), _f64(g["ter_delta"])
            ctx.check(L.vdo_graph_add_edges_landmark_motion(self.h, len(w), _ip(pph), _dp(w), _dp(dl)), "add_edges_landmark_motion")
        ctx.check(L.vdo_graph_finalize(self.h), "vdo_graph_finalize")

    def optimize(self, max_iterations=300, gain_threshold=1e-4, pcg_rel_tol=None, pcg_max_iterations=2000,
                 verbose=False, force_all_iterations=False, pcg_loose_tol=None, pcg_switch_gain=None):
        o = LMOptions()
        self.ctx.L.vdo_lm_options_default(C.byref(o))
        o.max_iterations, o.gain_threshold = int(max_iterations), float(gain_threshold)
        o.pcg_max_iterations = int(pcg_max_iterations)
        if pcg_rel_tol is not None:
            o.pcg_rel_tol = float(pcg_rel_tol)
        if pcg_loose_tol is not None:
            o.pcg_loose_tol = float(pcg_loose_tol)
        if pcg_switch_gain is not None:
            o.pcg_switch_gain = float(pcg_switch_gain)
        o.verbose, o.force_all_iterations = int(verbose), int(force_all_iterations)
        st = LMStats()
        hist = np.zeros(max_iterations + 1)
        self.ctx.check(self.ctx.L.vdo_graph_optimize(self.h, C.byref(o), C.byref(st), _dp(hist)), "vdo_graph_optimize")
        d = st.asdict()
        d["chi2"] = hist[: st.iterations + 1].copy()
        return d

    def vertices(self):
        se3 = np.zeros((self.n_se3, 12))
        pt = np.zeros((self.n_pt, 3))
        self.ctx.check(self.ctx.L.vdo_graph_get_vertices(self.h, _dp(se3), _dp(pt)), "vdo_graph_get_vertices")
        return se3, pt

    def vertices_gathered(self, dist):
        """Sharded graphs: every rank gets all landmark estimates (each rank holds only its own after optimize())."""
        import torch
        se3 = np.zeros((self.n_se3, 12))
        pt = np.full((self.n_pt, 3), np.nan)
        self.ctx.check(self.ctx.L.vdo_graph_get_vertices(self.h, _dp(se3), _dp(pt)), "vdo_graph_get_vertices")
        own = ~np.isnan(pt[:, 0])
        t = torch.from_numpy(np.where(own[:, None], pt, 0.0).copy())
        c = torch.from_numpy(own.astype(np.float64))
        if dist.get_backend() == "nccl":
            t, c = t.cuda(), c.cuda()
        dist.all_reduce(t); dist.all_reduce(c)
        assert bool((c.cpu() == 1).all()), "every landmark must be owned by exactly one rank"
        return se3, t.cpu().numpy()

    def reset(self):
        self.ctx.check(self.ctx.L.vdo_graph_reset_vertices(self.h), "vdo_graph_reset_vertices")

    def info(self):
        out = (C.c_int64 * 8)()
        self.ctx.check(self.ctx.L.vdo_graph_info(self.h, out), "vdo_graph_info")
        return dict(zip(["n_se3", "n_pt", "n_pointxyz_edges", "n_motion_edges", "n_se3_edges", "n_prior", "n_tracklets", "device_bytes"], list(out)))

    def solver_info(self):
        out = (C.c_int64 * 8)()
        self.ctx.check(self.ctx.L.vdo_graph_solver_info(self.h, out), "vdo_graph_solver_info")
        return dict(zip(["tiled", "n_tiles", "n_static_tiles", "band_width", "band_rows", "dense", "path_sharded", "n_paths"], list(out)))

    def time_kernel(self, name: str, reps: int = 20) -> float:
        ms = C.c_float(0)
        self.ctx.check(self.ctx.L.vdo_graph_time_kernel(self.h, name.encode(), C.c_int(reps), C.byref(ms)), f"vdo_graph_time_kernel({name})")
        return float(ms.value)

    def debug_linearize(self):
        Hpp = np.zeros((self.n_se3, 6, 6)); bp = np.zeros((self.n_se3, 6)); Hll = np.zeros(self.n_pt); bl = np.zeros((self.n_pt, 3))
        chi = C.c_double(0)
        self.ctx.check(self.ctx.L.vdo_graph_debug_linearize(self.h, _dp(Hpp), _dp(bp), _dp(Hll), _dp(bl), C.byref(chi)), "debug_linearize")
        return Hpp, bp, Hll, bl, chi.value

    def close(self):
        if self.h:
            self.ctx.L.vdo_graph_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def pose_opt_flow2(ctx: Context, problems, quirk: int = 1, modes=None):
    """Optimizer::PoseOptimizationFlow2 / Flow2Cam for a list of problems (dicts shaped like synth.make_flow_problem);
    all problems run in one kernel launch.  Returns a list of dict(T, flow, inlier, iters, trials, chi2, lam, n_inliers)."""
    L = ctx.L
    nprob = len(problems)
    modes = np.asarray(modes if modes is not None else [1] * nprob, np.int32)
    f32 = lambda a: np.ascontiguousarray(a, np.float32)
    off = np.zeros(nprob + 1, np.int32)
    off[1:] = np.cumsum([len(p["depth"]) for p in problems])
    cat = lambda k, shape: f32(np.concatenate([np.asarray(p[k], np.float32).reshape(shape) for p in problems], 0)) if off[-1] else np.zeros((0,) + shape[1:], np.float32)
    pts, depth, flow = cat("pts", (-1, 2)), cat("depth", (-1,)), cat("flow", (-1, 2))
    K = f32(np.stack([p["K"] for p in problems])); Tl = f32(np.stack([p["Tcw_last"] for p in problems])); Ti = f32(np.stack([p["T_init"] for p in problems]))
    T_out = np.zeros((nprob, 4, 4), np.float32); flow_out = np.zeros((int(off[-1]), 2)); inl = np.zeros(int(off[-1]), np.uint8); stats = np.zeros((nprob, 8))
    fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
    ctx.check(L.vdo_pose_opt_flow2_batch(ctx.h, C.c_int(quirk), C.c_int(nprob), _ip(modes), _ip(off), fp(pts), fp(depth), fp(flow), fp(K), fp(Tl), fp(Ti),
                                         fp(T_out), _dp(flow_out), inl.ctypes.data_as(C.POINTER(C.c_uint8)), _dp(stats)), "vdo_pose_opt_flow2_batch")
    out = []
    for i in range(nprob):
        a, b = off[i], off[i + 1]
        out.append(dict(T=T_out[i], flow=flow_out[a:b], inlier=inl[a:b].astype(bool), iters=int(stats[i, 0]), trials=int(stats[i, 1]),
                        chi2=stats[i, 2], lam=stats[i, 3], n_inliers=int(stats[i, 4])))
    return out


def pose_opt_flow2_time(ctx: Context, nprob: int, quirk: int = 1, reps: int = 20) -> float:
    ms = C.c_float(0)
    ctx.check(ctx.L.vdo_pose_opt_flow2_time(ctx.h, C.c_int(quirk), C.c_int(nprob), C.c_int(reps), C.byref(ms)), "vdo_pose_opt_flow2_time")
    return float(ms.value)


class Frame:
    """vdo_frame: one RGB-D frame resident on the device (gray u8, depth f32, flow f32x2, mask i32)."""

    def __init__(self, ctx: Context, width: int, height: int):
        self.ctx, self.w, self.h = ctx, width, height
        self.h_ = C.c_void_p()
        ctx.check(ctx.L.vdo_frame_create(ctx.h, C.c_int(width), C.c_int(height), C.byref(self.h_)), "vdo_frame_create")

    def upload(self, gray=None, depth=None, flow=None, mask=None):
        self._keep = [None if a is None else np.ascontiguousarray(a, dt) for a, dt in ((gray, np.uint8), (depth, np.float32), (flow, np.float32), (mask, np.int32))]
        ptr = lambda a, ty: None if a is None else a.ctypes.data_as(C.POINTER(ty))
        g, d, f, m = self._keep
        self.ctx.check(self.ctx.L.vdo_frame_upload(self.h_, ptr(g, C.c_ubyte), ptr(d, C.c_float), ptr(f, C.c_float), ptr(m, C.c_int)), "vdo_frame_upload")

    def orb_describe(self, n):
        """vdo_orb_describe: descriptors (n x 32 u8) of the keypoints of the last orb_extract()."""
        out = np.zeros((max(n, 1), 32), np.uint8)
        self.ctx.check(self.ctx.L.vdo_orb_describe(self.h_, C.c_int(n), out.ctypes.data_as(C.POINTER(C.c_ubyte))), "vdo_orb_describe")
        return out[:n]

    def debug_blur(self, level, shape):
        out = np.zeros(shape, np.uint8)
        self.ctx.check(self.ctx.L.vdo_frame_debug_blur(self.h_, C.c_int(level), out.ctypes.data_as(C.POINTER(C.c_ubyte))), "vdo_frame_debug_blur")
        return out

    def depth_prep(self, bf, factor):
        out = np.zeros((self.h, self.w), np.float32)
        self.ctx.check(self.ctx.L.vdo_frame_depth_prep(self.h_, C.c_float(bf), C.c_float(factor), out.ctypes.data_as(C.POINTER(C.c_float))), "vdo_frame_depth_prep")
        return out

    def orb_extract(self, nfeatures=2500, scale=1.2, nlevels=8, ini_th=20, min_th=7, max_out=20000):
        f32 = lambda n: np.zeros(n, np.float32); i32 = lambda n: np.zeros(n, np.int32)
        x, y, resp, ang = f32(max_out), f32(max_out), f32(max_out), f32(max_out)
        octv, size, ncand = i32(max_out), i32(max_out), i32(nlevels)
        n = C.c_int(0)
        fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float)); ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int))
        self.ctx.check(self.ctx.L.vdo_orb_extract(self.h_, C.c_int(nfeatures), C.c_float(scale), C.c_int(nlevels), C.c_int(ini_th), C.c_int(min_th), C.c_int(max_out),
                                                  fp(x), fp(y), ip(octv), fp(resp), fp(ang), ip(size), C.byref(n), ip(ncand)), "vdo_orb_extract")
        k = n.value
        return dict(x=x[:k], y=y[:k], octave=octv[:k], response=resp[:k], angle=ang[:k], size=size[:k], n_candidates=ncand.tolist())

    def filter_static(self, kx, ky, th_depth):
        n = len(kx)
        kx, ky = np.ascontiguousarray(kx, np.float32), np.ascontiguousarray(ky, np.float32)
        idx = np.zeros(n, np.int32); out = [np.zeros(n, np.float32) for _ in range(5)]
        m = C.c_int(0)
        fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
        self.ctx.check(self.ctx.L.vdo_frame_filter_static(self.h_, C.c_int(n), fp(kx), fp(ky), C.c_float(th_depth), idx.ctypes.data_as(C.POINTER(C.c_int)),
                                                          *[fp(a) for a in out], C.byref(m)), "vdo_frame_filter_static")
        k = m.value
        return (idx[:k],) + tuple(a[:k] for a in out)

    SAMPLE_KEYPOINTS = 3000      # VDO_SAMPLE_KEYPOINTS

    def sample_static(self, seed, th_depth):
        """vdo_frame_sample_static: Frame::SampleKeyPoints (cv::RNG(seed); seed 0 = stream of 0xffffffff) + the Option II filter.
        Returns dict(raw (3000, 2) unfiltered samples, x, y, cx, cy, fu, fv, depth of the kept ones, in order)."""
        n = self.SAMPLE_KEYPOINTS
        out = [np.zeros(n, np.float32) for _ in range(7)]
        raw = np.zeros((n, 2), np.float32)
        m = C.c_int(0)
        self.ctx.check(self.ctx.L.vdo_frame_sample_static(self.h_, C.c_uint32(seed), C.c_float(th_depth), C.c_int(n), *[_fp(a) for a in out], C.byref(m), _fp(raw)),
                       "vdo_frame_sample_static")
        k = m.value
        return dict(raw=raw, **{name: a[:k] for name, a in zip(("x", "y", "cx", "cy", "fu", "fv", "depth"), out)})

    def sample_objects(self, th_depth_obj, step=4, max_out=None):
        max_out = max_out or ((self.w + step - 1) // step) * ((self.h + step - 1) // step)
        x, y, lab = (np.zeros(max_out, np.int32) for _ in range(3))
        cx, cy, fx, fy, dep = (np.zeros(max_out, np.float32) for _ in range(5))
        n = C.c_int(0)
        fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float)); ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int))
        self.ctx.check(self.ctx.L.vdo_frame_sample_objects(self.h_, C.c_float(th_depth_obj), C.c_int(step), C.c_int(max_out), ip(x), ip(y), fp(cx), fp(cy), fp(fx), fp(fy),
                                                           fp(dep), ip(lab), C.byref(n)), "vdo_frame_sample_objects")
        k = n.value
        return dict(x=x[:k], y=y[:k], cx=cx[:k], cy=cy[:k], fx=fx[:k], fy=fy[:k], depth=dep[:k], label=lab[:k])

    def debug_level(self, level: int):
        w, h = C.c_int(0), C.c_int(0)
        self.ctx.check(self.ctx.L.vdo_frame_debug_level(self.h_, C.c_int(level), None, None, C.byref(w), C.byref(h)), "vdo_frame_debug_level")
        img = np.zeros((h.value, w.value), np.uint8); sc = np.zeros((h.value, w.value), np.uint8)
        up = lambda a: a.ctypes.data_as(C.POINTER(C.c_ubyte))
        self.ctx.check(self.ctx.L.vdo_frame_debug_level(self.h_, C.c_int(level), up(img), up(sc), None, None), "vdo_frame_debug_level")
        return img, sc

    def orb_time(self, reps=20):
        ms = C.c_float(0)
        self.ctx.check(self.ctx.L.vdo_orb_time(self.h_, C.c_int(reps), C.byref(ms)), "vdo_orb_time")
        return float(ms.value)

    def close(self):
        if self.h_:
            self.ctx.L.vdo_frame_destroy(self.h_)
            self.h_ = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def scene_flow(ctx: Context, u_prev, v_prev, z_prev, Tcw_prev, u_cur, v_cur, z_cur, Tcw_cur, K, lab_prev, lab_cur):
    n = len(u_prev)
    f32 = lambda a: np.ascontiguousarray(a, np.float32); i32 = lambda a: np.ascontiguousarray(a, np.int32)
    arrs = [f32(a) for a in (u_prev, v_prev, z_prev)] + [f32(Tcw_prev)] + [f32(a) for a in (u_cur, v_cur, z_cur)] + [f32(Tcw_cur), f32(K)]
    lp, lc = i32(lab_prev), i32(lab_cur)
    flow3d = np.zeros((n, 3), np.float32); Xp = np.zeros((n, 3), np.float32); valid = np.zeros(n, np.uint8)
    fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
    ctx.check(ctx.L.vdo_scene_flow(ctx.h, C.c_int(n), *[fp(a) for a in arrs], lp.ctypes.data_as(C.POINTER(C.c_int)), lc.ctypes.data_as(C.POINTER(C.c_int)),
                                   fp(flow3d), fp(Xp), valid.ctypes.data_as(C.POINTER(C.c_uint8))), "vdo_scene_flow")
    return flow3d, Xp, valid.astype(bool)


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def tracklets_build(assoc_rows, label_rows=None, lib_path: str | None = None):
    """vdo_tracklets_build (host-only): Tracking::GetStaticTrack / GetDynamicTrackNew.  Returns (tracklets, obj_ids)."""
    L = load(lib_path)
    rb = np.zeros(len(assoc_rows) + 1, np.int32)
    rb[1:] = np.cumsum([len(r) for r in assoc_rows])
    flat = _i32(np.concatenate([np.asarray(r, np.int32) for r in assoc_rows])) if len(assoc_rows) and rb[-1] else np.zeros(0, np.int32)
    lab = None
    if label_rows is not None:
        lab = _i32(np.concatenate([np.asarray(r, np.int32) for r in label_rows])) if rb[-1] else np.zeros(0, np.int32)
    max_t = int(np.count_nonzero(flat != -1)) + 1
    max_e = 2 * max_t
    tb, tf, tk, oid = np.zeros(max_t + 1, np.int32), np.zeros(max_e, np.int32), np.zeros(max_e, np.int32), np.zeros(max_t, np.int32)
    nt = C.c_int(0)
    rc = L.vdo_tracklets_build(C.c_int(len(assoc_rows)), _ip(rb), _ip(flat), None if lab is None else _ip(lab), C.c_int(max_t), C.c_int(max_e),
                               C.byref(nt), _ip(tb), _ip(tf), _ip(tk), _ip(oid))
    if rc != 0:
        raise VdoError(f"vdo_tracklets_build failed ({rc})")
    n = nt.value
    trk = [list(zip(tf[tb[t]:tb[t + 1]].tolist(), tk[tb[t]:tb[t + 1]].tolist())) for t in range(n)]
    return trk, (oid[:n].tolist() if label_rows is not None else [])


def update_mask(cur: "Frame", last: "Frame", sem_label_last, corres):
    """vdo_update_mask: Tracking::UpdateMask on two resident frames.  Returns (updated mask, recovered labels)."""
    ctx = cur.ctx
    sl = _i32(sem_label_last)
    n = len(sl)
    corres = np.asarray(corres, np.float32).reshape(-1, 2)
    cx, cy = np.ascontiguousarray(corres[:, 0]), np.ascontiguousarray(corres[:, 1])
    out = np.zeros((cur.h, cur.w), np.int32)
    wl = np.zeros(max(1, len(set(sl.tolist()))), np.int32)
    nw = C.c_int(0)
    ctx.check(ctx.L.vdo_update_mask(cur.h_, last.h_, C.c_int(n), _ip(sl), _fp(cx), _fp(cy), _ip(out), C.byref(nw), _ip(wl)), "vdo_update_mask")
    return out, wl[:nw.value].tolist()


def dyn_obj_tracking(ctx: Context, sem_label, obj_label, keys, depth, flow3d, sem_label_last, last_sem_position, last_obj_stat, last_mod_label,
                     rows, cols, shrink_row, shrink_col, sf_mg_thres, sf_ds_thres, th_depth_obj, f_id, max_id, max_objects=256):
    """vdo_dyn_obj_tracking: Tracking::DynObjTracking.  Returns (obj_label', objects, mod_label, sem_position, max_id')."""
    sl, ol, sll = _i32(sem_label), _i32(obj_label).copy(), _i32(sem_label_last)
    n = len(sl)
    keys = np.asarray(keys, np.float32).reshape(-1, 2)
    kx, ky = np.ascontiguousarray(keys[:, 0]), np.ascontiguousarray(keys[:, 1])
    dp, f3 = np.ascontiguousarray(depth, np.float32), np.ascontiguousarray(flow3d, np.float32)
    lsp, lml = _i32(last_sem_position), _i32(last_mod_label)
    los = np.ascontiguousarray(last_obj_stat, np.uint8)
    mid, no = C.c_int(max_id), C.c_int(0)
    ob, oi = np.zeros(max_objects + 1, np.int32), np.zeros(max(n, 1), np.int32)
    ml, sp = np.zeros(max_objects, np.int32), np.zeros(max_objects, np.int32)
    ctx.check(ctx.L.vdo_dyn_obj_tracking(ctx.h, C.c_int(n), _ip(sl), _ip(ol), _fp(kx), _fp(ky), _fp(dp), _fp(f3), _ip(sll), C.c_int(len(lsp)), _ip(lsp),
                                         los.ctypes.data_as(C.POINTER(C.c_ubyte)), _ip(lml), C.c_int(rows), C.c_int(cols), C.c_int(shrink_row), C.c_int(shrink_col),
                                         C.c_float(sf_mg_thres), C.c_float(sf_ds_thres), C.c_float(th_depth_obj), C.c_int(f_id), C.byref(mid), C.c_int(max_objects),
                                         C.byref(no), _ip(ob), _ip(oi), _ip(ml), _ip(sp)), "vdo_dyn_obj_tracking")
    k = no.value
    objs = [oi[ob[t]:ob[t + 1]].tolist() for t in range(k)]
    return ol, objs, ml[:k].tolist(), sp[:k].tolist(), mid.value


def init_model_batch(ctx: Context, problems, K4, iters=500, thr=0.4, conf=0.98):
    """vdo_init_model_batch: GetInitModelCam/Obj for a batch.  problems: list of dict(obj (n,3), img (n,2), T_mm (4,4) or None).
    Returns list of dict(T, sub (local indices), n_ransac, n_mm, used_mm, iters_run, best_it, n_valid, Rt, Rt_hyp)."""
    npb = len(problems)
    off = np.zeros(npb + 1, np.int32)
    off[1:] = np.cumsum([len(p["obj"]) for p in problems])
    tot = int(off[-1])
    obj = np.ascontiguousarray(np.concatenate([np.asarray(p["obj"], np.float32).reshape(-1, 3) for p in problems]) if tot else np.zeros((0, 3), np.float32))
    img = np.ascontiguousarray(np.concatenate([np.asarray(p["img"], np.float32).reshape(-1, 2) for p in problems]) if tot else np.zeros((0, 2), np.float32))
    Tmm = np.zeros((npb, 16), np.float32); has = np.zeros(npb, np.uint8)
    for i, p in enumerate(problems):
        if p.get("T_mm") is not None:
            Tmm[i] = np.asarray(p["T_mm"], np.float32).reshape(16); has[i] = 1
    K = np.ascontiguousarray(K4, np.float32)
    T = np.zeros((npb, 16), np.float32); nsub = np.zeros(npb, np.int32); sub = np.zeros(max(tot, 1), np.int32)
    info = np.zeros((npb, 8), np.int32); Rt = np.zeros((npb, 12)); Rh = np.zeros((npb, 12))
    ctx.check(ctx.L.vdo_init_model_batch(ctx.h, C.c_int(npb), _ip(off), _fp(obj), _fp(img), _fp(K), C.c_int(iters), C.c_double(thr), C.c_double(conf),
                                         _fp(Tmm), has.ctypes.data_as(C.POINTER(C.c_ubyte)), _fp(T), _ip(nsub), _ip(sub), _ip(info), _dp(Rt), _dp(Rh)), "vdo_init_model_batch")
    out = []
    for i in range(npb):
        out.append(dict(T=T[i].reshape(4, 4).copy(), sub=sub[off[i]:off[i] + nsub[i]].copy(), n_ransac=int(info[i, 0]), n_mm=int(info[i, 1]), used_mm=bool(info[i, 2]),
                        iters_run=int(info[i, 4]), best_it=int(info[i, 5]), n_valid=int(info[i, 6]), Rt=Rt[i].copy(), Rt_hyp=Rh[i].copy()))
    return out


def renew_frame_info(cur: "Frame", tm_sta, stat_keys, samp_keys, max_num_sta, obj_inliers, obj_stat, sem_position, mod_label, obj_keys, obj_label,
                     tmp_keys, tmp_depth, tmp_sem, tmp_flow, tmp_corres, max_num_obj, K4, Twc):
    """vdo_renew_frame_info: Tracking::RenewFrameInfo on a resident frame.  Returns (static dict, object dict)."""
    ctx = cur.ctx
    f2 = lambda a: np.ascontiguousarray(np.asarray(a, np.float32).reshape(-1, 2))
    tm = _i32(tm_sta); sk = f2(stat_keys); sp = f2(samp_keys); ok = f2(obj_keys); ol = _i32(obj_label)
    n_obj = len(obj_inliers)
    ib = np.zeros(n_obj + 1, np.int32); ib[1:] = np.cumsum([len(x) for x in obj_inliers])
    ii = _i32(np.concatenate([np.asarray(x, np.int32) for x in obj_inliers])) if n_obj and ib[-1] else np.zeros(0, np.int32)
    st = np.ascontiguousarray(obj_stat, np.uint8); sem = _i32(sem_position); ml = _i32(mod_label)
    tk = f2(tmp_keys); td = np.ascontiguousarray(tmp_depth, np.float32); ts = _i32(tmp_sem); tf = f2(tmp_flow); tc = f2(tmp_corres)
    K = np.ascontiguousarray(K4, np.float32); T = np.ascontiguousarray(Twc, np.float32).reshape(16)
    cap_s = len(tm) + len(sp) + 8; cap_o = int(ib[-1]) + (n_obj + 1) * len(tk) + 8
    z2 = lambda n: np.zeros((n, 2), np.float32)
    s_keys, s_cor, s_flow, s_id, s_dep, s_3d = z2(cap_s), z2(cap_s), z2(cap_s), np.zeros(cap_s, np.int32), np.zeros(cap_s, np.float32), np.zeros((cap_s, 3), np.float32)
    o_keys, o_dep, o_cor, o_flow = z2(cap_o), np.zeros(cap_o, np.float32), z2(cap_o), z2(cap_o)
    o_sem, o_id, o_lab, o_3d = np.zeros(cap_o, np.int32), np.zeros(cap_o, np.int32), np.zeros(cap_o, np.int32), np.zeros((cap_o, 3), np.float32)
    ns, no = C.c_int(0), C.c_int(0)
    ub = lambda a: a.ctypes.data_as(C.POINTER(C.c_ubyte))
    ctx.check(ctx.L.vdo_renew_frame_info(cur.h_, C.c_int(len(tm)), _ip(tm), C.c_int(len(sk)), _fp(sk), C.c_int(len(sp)), _fp(sp), C.c_int(max_num_sta),
                                         C.c_int(n_obj), _ip(ib), _ip(ii), ub(st), _ip(sem), _ip(ml), C.c_int(len(ok)), _fp(ok), _ip(ol), C.c_int(len(tk)),
                                         _fp(tk), _fp(td), _ip(ts), _fp(tf), _fp(tc), C.c_int(max_num_obj), _fp(K), _fp(T),
                                         C.c_int(cap_s), C.byref(ns), _fp(s_keys), _fp(s_cor), _fp(s_flow), _ip(s_id), _fp(s_dep), _fp(s_3d),
                                         C.c_int(cap_o), C.byref(no), _fp(o_keys), _fp(o_dep), _fp(o_cor), _fp(o_flow), _ip(o_sem), _ip(o_id), _ip(o_lab), _fp(o_3d)),
              "vdo_renew_frame_info")
    a, b = ns.value, no.value
    return (dict(keys=s_keys[:a], corres=s_cor[:a], flow=s_flow[:a], inlier_id=s_id[:a], depth=s_dep[:a], p3d=s_3d[:a]),
            dict(keys=o_keys[:b], depth=o_dep[:b], corres=o_cor[:b], flow=o_flow[:b], sem=o_sem[:b], inlier_id=o_id[:b], label=o_lab[:b], p3d=o_3d[:b]))


class TrackerParams(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float), ("cy", C.c_float), ("bf", C.c_float),
                ("depth_factor", C.c_float), ("th_depth_bg", C.c_float), ("th_depth_obj", C.c_float), ("max_track_bg", C.c_int), ("max_track_obj", C.c_int),
                ("sf_mg_thres", C.c_float), ("sf_ds_thres", C.c_float), ("n_features", C.c_int), ("scale_factor", C.c_float), ("n_levels", C.c_int),
                ("ini_th_fast", C.c_int), ("min_th_fast", C.c_int), ("is_kitti", C.c_int), ("quirk", C.c_int), ("window_size", C.c_int),
                ("overlap_size", C.c_int), ("local_batch", C.c_int), ("dataset", C.c_int), ("use_sample_feature", C.c_int),
                ("sample_seed", C.c_uint)]


class Tracker:
    """vdo_tracker: System::TrackRGBD -> Tracking::GrabImageRGBD -> Tracking::Track on the device stages."""
    _INT = {"nStaInlierID", "vSemObjLabel", "vObjLabel", "nDynInlierID", "nModLabel", "nSemPosition", "bObjStat", "TemperalMatch_subset", "max_id", "f_id", "local_ba",
            "sample_seed"}

    def __init__(self, ctx: Context, **overrides):
        self.ctx = ctx
        self.params = TrackerParams()
        ctx.L.vdo_tracker_params_default(C.byref(self.params))
        for k, v in overrides.items():
            setattr(self.params, k, v)
        self.h_ = C.c_void_p()
        ctx.check(ctx.L.vdo_tracker_create(ctx.h, C.byref(self.params), C.byref(self.h_)), "vdo_tracker_create")
        ctx.L.vdo_tracker_last_error.restype = C.c_char_p

    def track(self, gray, depth, flow, mask, gt_ids, writeback=True):
        """depth (f32 h x w) and mask (i32 h x w) must be C-contiguous arrays; with writeback they are mutated like the reference's cv::Mat."""
        assert depth.dtype == np.float32 and depth.flags.c_contiguous and mask.dtype == np.int32 and mask.flags.c_contiguous
        g = np.ascontiguousarray(gray, np.uint8); f = np.ascontiguousarray(flow, np.float32)
        ids = _i32(gt_ids)
        T = np.zeros((4, 4), np.float32)
        h, w = g.shape
        assert depth.shape == (h, w) and mask.shape == (h, w) and f.shape == (h, w, 2)
        rc = self.ctx.L.vdo_tracker_track(self.h_, C.c_int(w), C.c_int(h), g.ctypes.data_as(C.POINTER(C.c_ubyte)), _fp(depth), _fp(f), _ip(mask), C.c_int(len(ids)),
                                          _ip(ids), C.c_int(int(writeback)), _fp(T))
        if rc != 0:
            raise VdoError(f"vdo_tracker_track failed ({rc}): {self.ctx.L.vdo_tracker_last_error(self.h_).decode()}")
        return T

    def get(self, name: str):
        n = C.c_int(0)
        self.ctx.check(self.ctx.L.vdo_tracker_get(self.h_, name.encode(), None, C.c_int(0), C.byref(n)), "vdo_tracker_get")
        out = np.zeros(max(n.value, 1), np.int32 if name in self._INT else np.float32)
        self.ctx.check(self.ctx.L.vdo_tracker_get(self.h_, name.encode(), out.ctypes.data_as(C.c_void_p), C.c_int(len(out)), C.byref(n)), "vdo_tracker_get")
        return out[:n.value]

    _GI = {"prior_v", "se3e_ij", "obs_cp", "ter_pph"}

    def graph_export(self, mode: int):
        """arrays the Map->graph builder hands to vdo_graph_* (mode 0 partial window, 1 full batch), in make_batch_graph layout"""
        g = {}
        shapes = dict(se3=(-1, 12), pt=(-1, 3), prior_Z=(-1, 12), se3e_Z=(-1, 12), obs_z=(-1, 3), se3e_ij=(-1, 2), obs_cp=(-1, 2), ter_pph=(-1, 3))
        for name in ("se3", "pt", "prior_v", "prior_Z", "prior_w", "se3e_ij", "se3e_Z", "se3e_w", "se3e_delta", "obs_cp", "obs_z", "obs_w", "obs_delta", "ter_pph",
                     "ter_w", "ter_delta"):
            n = C.c_int(0)
            self.ctx.check(self.ctx.L.vdo_tracker_graph_export(self.h_, C.c_int(mode), name.encode(), None, C.c_int(0), C.byref(n)), "vdo_tracker_graph_export")
            out = np.zeros(max(n.value, 1), np.int32 if name in self._GI else np.float64)
            self.ctx.check(self.ctx.L.vdo_tracker_graph_export(self.h_, C.c_int(mode), name.encode(), out.ctypes.data_as(C.c_void_p), C.c_int(len(out)), C.byref(n)),
                           "vdo_tracker_graph_export")
            g[name] = out[:n.value].reshape(shapes.get(name, -1))
        return g

    def batch_optimize(self, mode: int, **opt):
        o = LMOptions(); self.ctx.L.vdo_lm_options_default(C.byref(o))
        st = LMStats(); info = np.zeros(6, np.int32)
        po = None
        if opt:
            for k, v in opt.items():
                setattr(o, k, v)
            po = C.byref(o)
        rc = self.ctx.L.vdo_tracker_batch_optimize(self.h_, C.c_int(mode), po, C.byref(st), _ip(info))
        if rc != 0:
            raise VdoError(f"vdo_tracker_batch_optimize failed ({rc}): {self.ctx.L.vdo_tracker_last_error(self.h_).decode()}")
        r = st.asdict(); r["sizes"] = dict(zip(["n_se3", "n_pt", "n_prior", "n_se3_edges", "n_obs", "n_ternary"], info.tolist()))
        return r

    def map_get(self, name: str):
        n = C.c_int(0)
        self.ctx.check(self.ctx.L.vdo_tracker_map_get(self.h_, name.encode(), None, C.c_int(0), C.byref(n)), "vdo_tracker_map_get")
        out = np.zeros(max(n.value, 1), np.int32 if name in ("vnRMLabel", "n_frames", "n_per_frame") else np.float32)
        self.ctx.check(self.ctx.L.vdo_tracker_map_get(self.h_, name.encode(), out.ctypes.data_as(C.c_void_p), C.c_int(len(out)), C.byref(n)), "vdo_tracker_map_get")
        return out[:n.value]

    def close(self):
        if getattr(self, "h_", None):
            self.ctx.L.vdo_tracker_destroy(self.h_)
            self.h_ = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- per-frame input files of the reference's driver (vdo_io_*, host-only; SURVEY 8(f) N3) ----
def io_read_png(ctx: "Context", path: str) -> np.ndarray:
    """cv::imread(path, UNCHANGED): uint8 / uint16, HxW or HxWxC in BGR[A] order."""
    w, h, ch, bd = C.c_int(), C.c_int(), C.c_int(), C.c_int()
    ctx.check(ctx.L.vdo_io_png_info(path.encode(), C.byref(w), C.byref(h), C.byref(ch), C.byref(bd)), f"vdo_io_png_info({path})")
    a = np.zeros((h.value, w.value, ch.value), np.uint8 if bd.value == 8 else np.uint16)
    ctx.check(ctx.L.vdo_io_read_png(path.encode(), a.ctypes.data_as(C.c_void_p), C.c_size_t(a.nbytes)), f"vdo_io_read_png({path})")
    return a[:, :, 0] if ch.value == 1 else a


def io_read_png_gray_f32(ctx: "Context", path: str, w: int, h: int) -> np.ndarray:
    a = np.zeros((h, w), np.float32)
    ctx.check(ctx.L.vdo_io_read_png_gray_f32(path.encode(), a.ctypes.data_as(C.POINTER(C.c_float)), C.c_int(w), C.c_int(h)), f"vdo_io_read_png_gray_f32({path})")
    return a


def io_read_flo(ctx: "Context", path: str) -> np.ndarray:
    w, h = C.c_int(), C.c_int()
    ctx.check(ctx.L.vdo_io_flo_info(path.encode(), C.byref(w), C.byref(h)), f"vdo_io_flo_info({path})")
    a = np.zeros((h.value, w.value, 2), np.float32)
    ctx.check(ctx.L.vdo_io_read_flo(path.encode(), a.ctypes.data_as(C.POINTER(C.c_float)), C.c_size_t(a.size)), f"vdo_io_read_flo({path})")
    return a


def io_read_mask_txt(ctx: "Context", path: str, w: int, h: int) -> np.ndarray:
    a = np.zeros((h, w), np.int32)
    ctx.check(ctx.L.vdo_io_read_mask_txt(path.encode(), _ip(a), C.c_int(w), C.c_int(h)), f"vdo_io_read_mask_txt({path})")
    return a


# ---- result files / metrics (vdo_results_*, vdo_metric_error; host-only; SURVEY 8(f) N4) ----
def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _flatten_frames(per_frame):
    """list (frames) of lists (entries) of arrays -> (counts i32, stacked f32 array)"""
    cnt = np.array([len(f) for f in per_frame], np.int32)
    flat = [np.asarray(m, np.float32) for f in per_frame for m in f]
    return cnt, (np.stack(flat) if flat else np.zeros((0, 4, 4), np.float32))


def results_write_poses(ctx: "Context", path: str, poses, start_frame: int = 0):
    P = np.ascontiguousarray(np.asarray(poses, np.float32).reshape(-1, 16))
    ctx.check(ctx.L.vdo_results_write_poses(path.encode(), C.c_int(start_frame), C.c_int(len(P)), _fp(P)), "vdo_results_write_poses")


def results_write_object_motions(ctx: "Context", path: str, motions, labels, pose_pre=None, start_frame: int = 0):
    cnt, H = _flatten_frames(motions)
    H = np.ascontiguousarray(H.reshape(-1, 16))
    lab = np.ascontiguousarray(np.concatenate([np.asarray(l, np.int32) for l in labels]) if len(labels) else np.zeros(0, np.int32))
    L = None
    if pose_pre is not None:
        L = np.ascontiguousarray(_flatten_frames(pose_pre)[1].reshape(-1, 16))
    ctx.check(ctx.L.vdo_results_write_object_motions(path.encode(), C.c_int(start_frame), C.c_int(len(cnt)), _ip(cnt), _ip(lab), _fp(H),
                                                     _fp(L) if L is not None else None), "vdo_results_write_object_motions")


def results_write_object_centres(ctx: "Context", path: str, centres, labels, start_frame: int = 0):
    cnt = np.array([len(f) for f in centres], np.int32)
    Cn = np.ascontiguousarray(np.concatenate([np.asarray(f, np.float32).reshape(-1, 3) for f in centres]) if len(centres) else np.zeros((0, 3), np.float32))
    lab = np.ascontiguousarray(np.concatenate([np.asarray(l, np.int32) for l in labels]) if len(labels) else np.zeros(0, np.int32))
    ctx.check(ctx.L.vdo_results_write_object_centres(path.encode(), C.c_int(start_frame), C.c_int(len(cnt)), _ip(cnt), _ip(lab), _fp(Cn)), "vdo_results_write_object_centres")


def metric_error(ctx: "Context", cam, cam_gt, motions, pose_pre, motions_gt, labels, obj_stat, max_id: int) -> dict:
    Cm = np.ascontiguousarray(np.asarray(cam, np.float32).reshape(-1, 16)); Cg = np.ascontiguousarray(np.asarray(cam_gt, np.float32).reshape(-1, 16))
    cnt, H = _flatten_frames(motions)
    H = np.ascontiguousarray(H.reshape(-1, 16)); L = np.ascontiguousarray(_flatten_frames(pose_pre)[1].reshape(-1, 16)); G = np.ascontiguousarray(_flatten_frames(motions_gt)[1].reshape(-1, 16))
    lab = np.ascontiguousarray(np.concatenate([np.asarray(l, np.int32) for l in labels]))
    st = np.ascontiguousarray(np.concatenate([np.asarray(s, np.uint8) for s in obj_stat]))
    out = np.zeros(4, np.float32); n = max(max_id - 1, 0)
    et, er, ec = np.zeros(n, np.float32), np.zeros(n, np.float32), np.zeros(n, np.int32)
    ctx.check(ctx.L.vdo_metric_error(C.c_int(len(Cm)), _fp(Cm), _fp(Cg), C.c_int(len(cnt)), _ip(cnt), _ip(lab), st.ctypes.data_as(C.POINTER(C.c_ubyte)), _fp(H), _fp(L), _fp(G),
                                     C.c_int(max_id), _fp(out), _fp(et), _fp(er), _ip(ec)), "vdo_metric_error")
    return {"cam_t": float(out[0]), "cam_r": float(out[1]), "obj_t": float(out[2]), "obj_r": float(out[3]), "each_t": et, "each_r": er, "each_count": ec}
