"""ctypes binding of libisdf_b200.so (include/isdf.h) used by tests/ and bench.py.

Thin by design: every method is one C-ABI call with host numpy buffers, or device pointers for the
`*_device` variants. There is NO fallback: if the shared library or a CUDA device is missing, loading /
`Evaluator()` raises.
"""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ISDF_B200_LIB") or os.path.join(os.path.dirname(_HERE), "libisdf_b200.so")  # env override: A/B builds

# isdf_shape_kind (include/isdf.h)
SHAPE_KINDS = dict(BALL=0, POINT=1, TORUS=2, CAPPED_TORUS=3, CAPPED_CONE=4, ROUNDED_CONE=5, WIREFRAME_BOX=6,
                   BEND_LINEAR=7, TWIST_BOX=8, BEND_BOX=9, TABLE=10, TREFOIL=11, SMOOTH_DIFFERENCE=12,
                   SMOOTH_INTERSECTION=13, CSG=14, BOX=15, MESH=16)
NAMED_SHAPES = ["Ball", "Point", "Torus", "Torus_big", "Cappedtorus", "CappedCone", "RoundedCone", "WireframeBox",
                "BendLinear", "BendLinear_big", "TwistBox", "BendBox", "Table", "Trefoil", "SmoothDifference",
                "SmoothIntersection", "SmoothIntersection_big", "CSG"]
WITH_DYNAMICS, WITH_COLLISION = 1, 2
QUERY_SDF, QUERY_GRAD, QUERY_SDF_GRAD = 0, 1, 2
MESH_SIGN_AUTO, MESH_SIGN_EXACT, MESH_SIGN_WINDING = 0, 1, 2

# every symbol include/isdf.h declares (tests assert the library exports all of them)
ABI_SYMBOLS = ["isdf_default_config", "isdf_create", "isdf_destroy", "isdf_last_error", "isdf_get_stats", "isdf_set_shard",
               "isdf_set_shape_analytic", "isdf_set_shape_named", "isdf_set_shape_mesh", "isdf_set_shape_mesh_ex", "isdf_shape_query",
               "isdf_set_map_u8", "isdf_set_map_f64", "isdf_points_in_aabb", "isdf_eval_discrete",
               "isdf_eval_discrete_device", "isdf_set_points", "isdf_eval_swept", "isdf_eval_swept_device",
               "isdf_get_swept_results", "isdf_eval_swept_given", "isdf_get_piece_costs",
               "isdf_gather_obstacle_points", "isdf_callback_batch", "isdf_callback_batch_device", "isdf_get_batch_trajectories",
               "isdf_lbfgs_default_params", "isdf_lbfgs_batch", "isdf_lbfgs_batch_device", "isdf_set_points_batch",
               "isdf_frontend_build_kernels", "isdf_frontend_get_kernels", "isdf_frontend_feasibility", "isdf_frontend_feasibility_device",
               "isdf_frontend_check_batch", "isdf_peer_export", "isdf_peer_connect", "isdf_peer_allreduce_device", "isdf_peer_status", "isdf_peer_disconnect",
               "isdf_check_collision", "isdf_check_collision_device"]


class KernelConfig(C.Structure):
    """isdf_kernel_config"""
    _fields_ = [(n, C.c_double) for n in ["kernel_max_roll", "kernel_max_pitch", "kernel_ang_res", "front_end_safeh"]]


class Config(C.Structure):
    """isdf_config — same field order as include/isdf.h."""
    _fields_ = [(n, C.c_double) for n in
                ["vehicle_mass", "grav_acc", "horiz_drag", "vert_drag", "paras_drag", "speed_eps", "vmax", "omgmax", "thetamax",
                 "weight_v", "weight_p", "weight_omg", "weight_theta", "smoothing_eps", "safety_hor", "occupancy_resolution"]] + \
               [(n, C.c_int32) for n in ["kernel_size", "integral_intervs", "threads_num", "flags"]]

    def copy(self):
        c = Config()
        C.memmove(C.byref(c), C.byref(self), C.sizeof(Config))
        return c


class LbfgsParams(C.Structure):
    """isdf_lbfgs_params"""
    _fields_ = [(n, C.c_int32) for n in ["mem_size", "past", "max_iterations", "max_linesearch", "max_rounds", "reserved_"]] + \
               [(n, C.c_double) for n in ["g_epsilon", "delta", "min_step", "max_step", "f_dec_coeff", "cautious_factor", "machine_prec"]]


class ClearanceReport(C.Structure):
    """isdf_clearance_report — one per trajectory checked by isdf_check_collision (96 bytes)."""
    _fields_ = [("min_clearance", C.c_double), ("t_min", C.c_double), ("p_min", C.c_double * 3), ("t_hit", C.c_double), ("p_hit", C.c_double * 3)] + \
               [(n, C.c_int32) for n in ["collides", "piece_min", "sample_min", "piece_hit", "sample_hit", "reserved_"]]

    def as_dict(self):
        return dict(min_clearance=self.min_clearance, t_min=self.t_min, p_min=np.array(self.p_min[:]), t_hit=self.t_hit, p_hit=np.array(self.p_hit[:]),
                    collides=bool(self.collides), piece_min=self.piece_min, sample_min=self.sample_min, piece_hit=self.piece_hit,
                    sample_hit=self.sample_hit)


class Stats(C.Structure):
    _fields_ = [("kernel_launches", C.c_int64), ("evals_discrete", C.c_int64), ("evals_swept", C.c_int64),
                ("last_pairs", C.c_int64), ("last_sdf_evals", C.c_int64), ("last_kernel_ms", C.c_double)]


def default_config_values():
    """plan_manager/config/config_CappedCone.yaml — pure python (no library needed)."""
    c = Config()
    c.vehicle_mass, c.grav_acc, c.horiz_drag, c.vert_drag, c.paras_drag, c.speed_eps = 0.61, 9.8, 0.10, 0.10, 0.01, 1e-4
    c.vmax, c.omgmax, c.thetamax = 10, 10, 100.0
    c.weight_v, c.weight_p, c.weight_omg, c.weight_theta = 1000.0, 4000.0, 1000.0, 1000.0
    c.smoothing_eps, c.safety_hor, c.occupancy_resolution = 1e-2, 0.866, 1.0
    c.kernel_size, c.integral_intervs, c.threads_num, c.flags = 13, 64, 30, WITH_DYNAMICS   # discrete collision term: opt-in
    return c


_lib = None


def load_library(path=None):
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise RuntimeError(f"{p} not found: build it with `python __graft_entry__.py build` (no CPU fallback exists)")
    lib = C.CDLL(p)
    dp, ip, vp = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.c_void_p
    lib.isdf_last_error.restype = C.c_char_p
    lib.isdf_default_config.argtypes = [C.POINTER(Config)]
    lib.isdf_create.argtypes = [C.POINTER(Config), C.c_int, C.POINTER(vp)]
    lib.isdf_destroy.argtypes = [vp]
    lib.isdf_get_stats.argtypes = [vp, C.POINTER(Stats)]
    lib.isdf_set_shard.argtypes = [vp, C.c_int, C.c_int]
    lib.isdf_set_shape_analytic.argtypes = [vp, C.c_int, dp, C.c_int, dp, dp]
    lib.isdf_set_shape_named.argtypes = [vp, C.c_char_p, dp, dp]
    lib.isdf_set_shape_mesh.argtypes = [vp, dp, C.c_int, ip, C.c_int, dp]
    lib.isdf_set_shape_mesh_ex.argtypes = [vp, dp, C.c_int, ip, C.c_int, dp, C.c_int]
    lib.isdf_shape_query.argtypes = [vp, dp, C.c_int, dp, dp, C.c_int]
    lib.isdf_set_map_u8.argtypes = [vp, C.POINTER(C.c_uint8), C.c_int, C.c_int, C.c_int, dp, C.c_double]
    lib.isdf_set_map_f64.argtypes = [vp, dp, C.c_int, C.c_int, C.c_int, dp, C.c_double]
    lib.isdf_points_in_aabb.argtypes = [vp, dp, C.c_double, dp, C.c_int, C.POINTER(C.c_int)]
    lib.isdf_eval_discrete.argtypes = [vp, C.c_int, dp, dp, dp, dp, dp]
    lib.isdf_eval_discrete_device.argtypes = [vp, C.c_int, vp, vp, vp, vp]
    lib.isdf_set_points.argtypes = [vp, dp, C.c_int]
    lib.isdf_eval_swept.argtypes = [vp, C.c_int, dp, dp, dp, dp, dp]
    lib.isdf_eval_swept_device.argtypes = [vp, C.c_int, vp, vp, vp, vp]
    lib.isdf_get_swept_results.argtypes = [vp, dp, dp, dp]
    lib.isdf_get_piece_costs.argtypes = [vp, dp, C.c_int]
    lib.isdf_gather_obstacle_points.argtypes = [vp, dp, C.c_int, C.c_double, dp, dp, C.c_int, C.POINTER(C.c_int), C.c_int]
    lib.isdf_callback_batch.argtypes = [vp, C.c_int, C.c_int, dp, dp, C.c_int, C.c_double, dp, dp, dp]
    lib.isdf_callback_batch_device.argtypes = [vp, C.c_int, C.c_int, vp, vp, C.c_int, C.c_double, vp, vp, vp, vp]
    lib.isdf_get_batch_trajectories.argtypes = [vp, dp, dp, dp]
    lib.isdf_set_points_batch.argtypes = [vp, C.c_int, ip, dp]
    lib.isdf_lbfgs_default_params.argtypes = [C.POINTER(LbfgsParams)]
    lib.isdf_lbfgs_batch.argtypes = [vp, C.c_int, C.c_int, dp, dp, C.c_int, C.c_double, C.POINTER(LbfgsParams), dp, dp, ip, ip, ip, ip]
    lib.isdf_lbfgs_batch_device.argtypes = [vp, C.c_int, C.c_int, vp, vp, C.c_int, C.c_double, C.POINTER(LbfgsParams), vp, vp, vp, vp, vp, ip, vp]
    lib.isdf_frontend_build_kernels.argtypes = [vp, C.POINTER(KernelConfig), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.isdf_frontend_get_kernels.argtypes = [vp, C.POINTER(C.c_uint8), C.c_int]
    lib.isdf_frontend_feasibility.argtypes = [vp, C.POINTER(C.c_uint32)]
    lib.isdf_frontend_feasibility_device.argtypes = [vp, vp, vp]
    lib.isdf_frontend_check_batch.argtypes = [vp, C.c_int, ip, dp, dp, C.POINTER(C.c_uint8)]
    lib.isdf_peer_export.argtypes = [vp, C.c_int, C.c_int, C.c_char_p]
    lib.isdf_peer_connect.argtypes = [vp, C.c_int, C.c_int, C.c_char_p, C.c_int]
    lib.isdf_peer_allreduce_device.argtypes = [vp, vp, C.c_int, vp]
    lib.isdf_peer_status.argtypes = [vp]
    lib.isdf_peer_disconnect.argtypes = [vp]
    lib.isdf_eval_swept_given.argtypes = [vp, C.c_int, dp, dp, dp, dp, dp, dp, dp, dp]
    lib.isdf_check_collision.argtypes = [vp, C.c_int, C.c_int, dp, dp, C.c_int, C.c_double, C.c_double, C.POINTER(ClearanceReport), dp]
    lib.isdf_check_collision_device.argtypes = [vp, C.c_int, C.c_int, vp, vp, C.c_int, C.c_double, C.c_double, vp, vp, vp]
    for s in ABI_SYMBOLS:
        if s != "isdf_last_error":
            getattr(lib, s).restype = C.c_int
    if path is None:
        _lib = lib
    return lib


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


class IsdfError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"isdf error {code}: {msg}")
        self.code = code


class Evaluator:
    """One isdf_ctx. Mirrors the call order of the reference: setParam -> setEnvironment(shape) / setGridMap(map) ->
    cost callbacks (back_end_optimizer.hpp:667-747)."""

    def __init__(self, cfg=None, device=0):
        self.lib = load_library()
        self.cfg = cfg.copy() if cfg is not None else default_config_values()
        h = C.c_void_p()
        self._check(self.lib.isdf_create(C.byref(self.cfg), device, C.byref(h)))
        self.h = h

    def _check(self, r):
        if r != 0:
            raise IsdfError(r, self.lib.isdf_last_error().decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.isdf_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- shape ----
    def set_shape_named(self, name, rotate=None, trans=None):
        r = _f64(rotate).reshape(9) if rotate is not None else None
        t = _f64(trans).reshape(3) if trans is not None else None
        self._check(self.lib.isdf_set_shape_named(self.h, name.encode(), _dp(r), _dp(t)))

    def set_shape_analytic(self, kind, params, rotate=None, trans=None):
        p = _f64(params).reshape(-1)
        r = _f64(rotate).reshape(9) if rotate is not None else None
        t = _f64(trans).reshape(3) if trans is not None else None
        self._check(self.lib.isdf_set_shape_analytic(self.h, int(kind), _dp(p) if p.size else None, p.size, _dp(r), _dp(t)))

    def set_shape_mesh(self, V, F, poly_params=None, sign_mode=MESH_SIGN_AUTO):
        V = _f64(V).reshape(-1, 3)
        F = np.ascontiguousarray(F, dtype=np.int32).reshape(-1, 3)
        pp = _f64(poly_params).reshape(6) if poly_params is not None else None
        self._check(self.lib.isdf_set_shape_mesh_ex(self.h, _dp(V), V.shape[0], F.ctypes.data_as(C.POINTER(C.c_int32)), F.shape[0], _dp(pp), int(sign_mode)))

    def shape_query(self, p, what=QUERY_SDF_GRAD):
        p = _f64(p).reshape(-1, 3)
        n = p.shape[0]
        sdf = np.zeros(n)
        grad = np.zeros((n, 3))
        self._check(self.lib.isdf_shape_query(self.h, _dp(p), n, _dp(sdf), _dp(grad), what))
        return sdf, grad

    # ---- map ----
    def set_map_u8(self, occ, bmin, res):
        occ = np.ascontiguousarray(occ, dtype=np.uint8)
        X, Y, Z = occ.shape
        b = _f64(bmin).reshape(3)
        self._check(self.lib.isdf_set_map_u8(self.h, occ.ctypes.data_as(C.POINTER(C.c_uint8)), X, Y, Z, _dp(b), float(res)))

    def set_map_f64(self, grid, bmin, res):
        grid = _f64(grid)
        X, Y, Z = grid.shape
        b = _f64(bmin).reshape(3)
        self._check(self.lib.isdf_set_map_f64(self.h, _dp(grid), X, Y, Z, _dp(b), float(res)))

    def points_in_aabb(self, centre, half, cap=100000):
        out = np.zeros((cap, 3))
        n = C.c_int(0)
        c = _f64(centre).reshape(3)
        self._check(self.lib.isdf_points_in_aabb(self.h, _dp(c), float(half), _dp(out), cap, C.byref(n)))
        return out[:min(n.value, cap)].copy(), n.value

    # ---- evaluation (host buffers; ACCUMULATES like the reference) ----
    def eval_discrete(self, T, coeffs, cost=0.0, gradC=None, gradT=None):
        T = _f64(T).reshape(-1)
        N = T.size
        Cc = _f64(coeffs).reshape(-1)
        assert Cc.size == 18 * N
        gC = np.zeros(18 * N) if gradC is None else _f64(gradC).reshape(-1)
        gT = np.zeros(N) if gradT is None else _f64(gradT).reshape(-1)
        c = C.c_double(cost)
        self._check(self.lib.isdf_eval_discrete(self.h, N, _dp(T), _dp(Cc), C.byref(c), _dp(gC), _dp(gT)))
        return c.value, gC, gT

    def gather_obstacle_points(self, waypoints, half, offset=(0.0, 0.0, 0.0), cap=1000000, set_as_points=False):
        wp = _f64(waypoints).reshape(-1, 3)
        off = _f64(offset).reshape(3)
        out = np.zeros((cap, 3))
        n = C.c_int(0)
        self._check(self.lib.isdf_gather_obstacle_points(self.h, _dp(wp), wp.shape[0], float(half), _dp(off), _dp(out), cap, C.byref(n), int(set_as_points)))
        if set_as_points:
            self.n_points = n.value
        return out[:min(n.value, cap)].copy(), n.value

    def callback_batch(self, head, tail, rho, X):
        """B decision vectors [tau (N0) | xi (3(N0-1))] -> (cost[B], grad[B, 4*N0-3]); head/tail 3x3 (columns p, v, a), shared (3,3)
        or per problem (B,3,3); passed to the library column-major."""
        X = _f64(X)
        B, dim = X.shape
        N0 = (dim + 3) // 4
        assert 4 * N0 - 3 == dim
        head, tail = np.asarray(head, dtype=np.float64), np.asarray(tail, dtype=np.float64)
        per = int(head.ndim == 3)
        colmajor = (lambda a: np.ascontiguousarray(np.swapaxes(a, -1, -2)).reshape(-1))
        h, t = colmajor(head), colmajor(tail)
        cost, grad = np.zeros(B), np.zeros((B, dim))
        Xf = np.ascontiguousarray(X).reshape(-1)
        self._check(self.lib.isdf_callback_batch(self.h, B, N0, _dp(h), _dp(t), per, float(rho), _dp(Xf), _dp(cost), _dp(grad.reshape(-1))))
        return cost, grad

    def callback_batch_device(self, B, N0, d_head, d_tail, per_problem_bc, rho, d_x, d_cost, d_grad, stream=None):
        self._check(self.lib.isdf_callback_batch_device(self.h, B, N0, d_head, d_tail, int(per_problem_bc), float(rho), d_x, d_cost, d_grad, stream))

    def set_points_batch(self, point_sets):
        """per-problem obstacle point sets for the batched callback (list of (P_b, 3) arrays); an empty list switches the batched swept term off"""
        B = len(point_sets)
        off = np.zeros(B + 1, dtype=np.int32)
        for b, p in enumerate(point_sets):
            off[b + 1] = off[b] + len(p)
        pts = _f64(np.concatenate([np.asarray(p, float).reshape(-1, 3) for p in point_sets])) if B and off[B] else np.zeros((0, 3))
        self._check(self.lib.isdf_set_points_batch(self.h, B, off.ctypes.data_as(C.POINTER(C.c_int32)), _dp(pts) if pts.size else None))

    def lbfgs_params(self, **kw):
        p = LbfgsParams()
        self._check(self.lib.isdf_lbfgs_default_params(C.byref(p)))
        for k, v in kw.items():
            setattr(p, k, v)
        return p

    def lbfgs_batch(self, head, tail, rho, X, params=None):
        """device-resident lock-step L-BFGS over the batched callback: X (B, 4*N0-3) starting points -> dict(x, f, ret, iterations, evaluations, rounds)"""
        X = _f64(X)
        B, dim = X.shape
        N0 = (dim + 3) // 4
        head, tail = np.asarray(head, dtype=np.float64), np.asarray(tail, dtype=np.float64)
        per = int(head.ndim == 3)
        colmajor = (lambda a: np.ascontiguousarray(np.swapaxes(a, -1, -2)).reshape(-1))
        h, t = colmajor(head), colmajor(tail)
        x = np.ascontiguousarray(X).copy().reshape(-1)
        f = np.zeros(B)
        ret, it, evs = (np.zeros(B, dtype=np.int32) for _ in range(3))
        rounds = C.c_int32(0)
        ip = C.POINTER(C.c_int32)
        p = params if params is not None else self.lbfgs_params()
        self._check(self.lib.isdf_lbfgs_batch(self.h, B, N0, _dp(h), _dp(t), per, float(rho), C.byref(p), _dp(x), _dp(f), ret.ctypes.data_as(ip), it.ctypes.data_as(ip),
                                              evs.ctypes.data_as(ip), C.byref(rounds)))
        return dict(x=x.reshape(B, dim), f=f, ret=ret, iterations=it, evaluations=evs, rounds=rounds.value)

    def batch_trajectories(self, B, N0):
        T, Cc, en = np.zeros(B * N0), np.zeros(18 * B * N0), np.zeros(B)
        self._check(self.lib.isdf_get_batch_trajectories(self.h, _dp(T), _dp(Cc), _dp(en)))
        return T, Cc, en

    # ---- whole-body collision check (see include/isdf.h) ----
    def check_collision(self, T, coeffs, samples_per_piece, margin, horizon, B=1, per_sample=False):
        """B trajectories of N0 = len(T) / B pieces (coefficient block as eval_discrete / batch_trajectories) -> list of B report dicts,
        plus the per-sample clearance (B, N0, M + 1) when per_sample. Raises IsdfError on failure (the library's reports are poisoned)."""
        T = _f64(T).reshape(-1)
        Cc = _f64(coeffs).reshape(-1)
        assert T.size % B == 0 and Cc.size == 18 * T.size
        N0, M = T.size // B, int(samples_per_piece)
        reps = (ClearanceReport * B)()
        clear = np.zeros(T.size * (M + 1)) if per_sample else None
        self._check(self.lib.isdf_check_collision(self.h, B, N0, _dp(T), _dp(Cc), M, float(margin), float(horizon), reps, _dp(clear)))
        out = [r.as_dict() for r in reps]
        return (out, clear.reshape(B, N0, M + 1)) if per_sample else out

    def check_collision_device(self, B, N0, d_T, d_coeffs, samples_per_piece, margin, horizon, d_reports, d_clearance=0, stream=0):
        """device-resident twin: raw device pointers (d_reports: B * 96 bytes, d_clearance may be 0), asynchronous on `stream`"""
        self._check(self.lib.isdf_check_collision_device(self.h, B, N0, C.c_void_p(d_T), C.c_void_p(d_coeffs), int(samples_per_piece), float(margin),
                                                         float(horizon), C.c_void_p(d_reports), C.c_void_p(d_clearance or None), C.c_void_p(stream)))

    def dbg_check_stats(self, n_samples=0):
        """counters of the last check {voxels in the body box, SDF values, mesh searches} and (after dbg_enable) per-sample cycles"""
        cnt = (C.c_ulonglong * 3)()
        cyc = np.zeros(n_samples, dtype=np.uint64)
        self.lib.isdf_dbg_check_stats.argtypes = [C.c_void_p, C.POINTER(C.c_ulonglong), C.c_void_p, C.c_longlong]
        if self.lib.isdf_dbg_check_stats(self.h, cnt, cyc.ctypes.data if n_samples else None, n_samples) != 0:
            raise IsdfError(-1, "isdf_dbg_check_stats failed")
        return dict(voxels_in_box=cnt[0], sdf_values=cnt[1], mesh_searches=cnt[2]), cyc

    def dbg_enable(self, on=True):
        self.lib.isdf_dbg_enable.argtypes = [C.c_void_p, C.c_int]
        if self.lib.isdf_dbg_enable(self.h, int(on)) != 0:
            raise IsdfError(-1, "isdf_dbg_enable failed")

    # ---- front end: attitude kernels (see include/isdf.h) ----
    def frontend_build_kernels(self, max_roll=45.0, max_pitch=45.0, ang_res=9.0, front_end_safeh=0.0):
        kc = KernelConfig(max_roll, max_pitch, ang_res, front_end_safeh)
        xk, yk = C.c_int(0), C.c_int(0)
        self._check(self.lib.isdf_frontend_build_kernels(self.h, C.byref(kc), C.byref(xk), C.byref(yk)))
        self.fe_dims = (xk.value, yk.value)
        return self.fe_dims

    def frontend_kernels(self, ks):
        xk, yk = self.fe_dims
        out = np.zeros(xk * yk * ks ** 3, dtype=np.uint8)
        self._check(self.lib.isdf_frontend_get_kernels(self.h, out.ctypes.data_as(C.POINTER(C.c_uint8)), out.size))
        return out.reshape(xk * yk, ks, ks, ks)

    def frontend_feasibility(self, X, Y, Z):
        out = np.zeros((X * Y * Z, 4), dtype=np.uint32)
        self._check(self.lib.isdf_frontend_feasibility(self.h, out.ctypes.data_as(C.POINTER(C.c_uint32))))
        return out

    def frontend_feasibility_device(self, d_masks, stream=None):
        self._check(self.lib.isdf_frontend_feasibility_device(self.h, d_masks, stream))

    def frontend_check_batch(self, ind, father):
        ind = np.ascontiguousarray(ind, dtype=np.int32).reshape(-1, 3)
        father = _f64(father).reshape(-1, 2)
        n = ind.shape[0]
        child, ok = np.zeros((n, 2)), np.zeros(n, dtype=np.uint8)
        self._check(self.lib.isdf_frontend_check_batch(self.h, n, ind.ctypes.data_as(C.POINTER(C.c_int32)), _dp(father.reshape(-1)), _dp(child.reshape(-1)),
                                                       ok.ctypes.data_as(C.POINTER(C.c_uint8))))
        return child, ok.astype(bool)

    # ---- multi-GPU reduction over peer memory (see include/isdf.h) ----
    def peer_export(self, world, max_doubles):
        buf = C.create_string_buffer(64)
        self._check(self.lib.isdf_peer_export(self.h, world, max_doubles, buf))
        return bytes(buf.raw)

    def peer_connect(self, world, rank, handles, fuse=True):
        blob = b"".join(handles)
        assert len(blob) == 64 * world
        self._check(self.lib.isdf_peer_connect(self.h, world, rank, blob, int(fuse)))

    def peer_allreduce_device(self, d_vec, n, stream=None):
        self._check(self.lib.isdf_peer_allreduce_device(self.h, d_vec, n, stream))

    def peer_status(self):
        self._check(self.lib.isdf_peer_status(self.h))

    def peer_disconnect(self):
        self._check(self.lib.isdf_peer_disconnect(self.h))

    def piece_costs(self, n):
        out = np.zeros(n)
        self._check(self.lib.isdf_get_piece_costs(self.h, _dp(out), n))
        return out

    def set_points(self, pts):
        pts = _f64(pts).reshape(-1, 3)
        self._check(self.lib.isdf_set_points(self.h, _dp(pts) if pts.size else None, pts.shape[0]))
        self.n_points = pts.shape[0]

    def eval_swept(self, T, coeffs, cost=0.0, gradC=None, gradT=None):
        T = _f64(T).reshape(-1)
        N = T.size
        Cc = _f64(coeffs).reshape(-1)
        gC = np.zeros(18 * N) if gradC is None else _f64(gradC).reshape(-1)
        gT = np.zeros(N) if gradT is None else _f64(gradT).reshape(-1)
        c = C.c_double(cost)
        self._check(self.lib.isdf_eval_swept(self.h, N, _dp(T), _dp(Cc), C.byref(c), _dp(gC), _dp(gT)))
        return c.value, gC, gT

    def eval_swept_given(self, T, coeffs, tstar, sdf, grel):
        T = _f64(T).reshape(-1)
        N = T.size
        Cc = _f64(coeffs).reshape(-1)
        gC, gT, c = np.zeros(18 * N), np.zeros(N), C.c_double(0.0)
        ts, sd, gr = _f64(tstar).reshape(-1), _f64(sdf).reshape(-1), _f64(grel).reshape(-1)
        self._check(self.lib.isdf_eval_swept_given(self.h, N, _dp(T), _dp(Cc), _dp(ts), _dp(sd), _dp(gr), C.byref(c), _dp(gC), _dp(gT)))
        return c.value, gC, gT

    def swept_results(self):
        P = self.n_points
        t, s, g = np.zeros(P), np.zeros(P), np.zeros((P, 3))
        self._check(self.lib.isdf_get_swept_results(self.h, _dp(t), _dp(s), _dp(g)))
        return t, s, g

    # ---- device-resident variants: raw device pointers (e.g. torch tensor .data_ptr()), asynchronous ----
    def eval_discrete_device(self, N, d_T, d_coeffs, d_out, stream=0):
        self._check(self.lib.isdf_eval_discrete_device(self.h, N, C.c_void_p(d_T), C.c_void_p(d_coeffs), C.c_void_p(d_out), C.c_void_p(stream)))

    def eval_swept_device(self, N, d_T, d_coeffs, d_out, stream=0):
        self._check(self.lib.isdf_eval_swept_device(self.h, N, C.c_void_p(d_T), C.c_void_p(d_coeffs), C.c_void_p(d_out), C.c_void_p(stream)))

    def set_shard(self, rank, world):
        self._check(self.lib.isdf_set_shard(self.h, rank, world))

    def stats(self):
        s = Stats()
        self._check(self.lib.isdf_get_stats(self.h, C.byref(s)))
        return s

    # ---- diagnostics (isdf_dbg_*: exported by the library, not part of include/isdf.h) ----
    def dbg_schedule(self, natural_order=False, warp_slots=0):
        """natural_order: every launch as a context's first one (no work items, nothing split); warp_slots > 0: build the work items as
        if the device had that many resident warps (huge values force every non-trivial sample to be split)."""
        vp = C.c_void_p
        self.lib.isdf_dbg_schedule.argtypes = [vp, C.c_int, C.c_int]
        if self.lib.isdf_dbg_schedule(self.h, int(natural_order), int(warp_slots)) != 0:
            raise IsdfError(-1, "isdf_dbg_schedule failed")

    def dbg_item_stats(self):
        n, parts = C.c_int(0), C.c_int(0)
        self.lib.isdf_dbg_item_stats.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        if self.lib.isdf_dbg_item_stats(self.h, C.byref(n), C.byref(parts)) != 0:
            raise IsdfError(-1, "isdf_dbg_item_stats failed")
        return n.value, parts.value

    def dbg_flatness(self, v, a, j, quat_grad, omg_grad, vel_grad):
        """device flatness map + adjoint as compiled into the epilogue kernel -> (quat, omg, gV, gA, gJ)"""
        vaj = np.ascontiguousarray(np.concatenate([_f64(v).reshape(-1, 3), _f64(a).reshape(-1, 3), _f64(j).reshape(-1, 3)], axis=1))
        gr = np.ascontiguousarray(np.concatenate([_f64(quat_grad).reshape(-1, 4), _f64(omg_grad).reshape(-1, 3), _f64(vel_grad).reshape(-1, 3)], axis=1))
        n = vaj.shape[0]
        out = np.zeros((n, 16))
        dp = C.POINTER(C.c_double)
        self.lib.isdf_dbg_flatness.argtypes = [C.c_void_p, C.c_int, dp, dp, dp]
        if self.lib.isdf_dbg_flatness(self.h, n, _dp(vaj), _dp(gr), _dp(out)) != 0:
            raise IsdfError(-1, "isdf_dbg_flatness failed")
        return out[:, 0:4], out[:, 4:7], out[:, 7:10], out[:, 10:13], out[:, 13:16]
