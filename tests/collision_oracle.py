"""ctypes binding of tests/collision_oracle.cpp — the oracle of the whole-body collision check (TEST INFRASTRUCTURE).
The library is compiled on first use into a temporary directory keyed by the sources' hash, with the oracle's flags (oracle/Makefile; OpenMP over independent samples)."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile
import numpy as np
import oracle_lib as O

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "collision_oracle.cpp")
ORACLE_DIR = os.path.join(os.path.dirname(HERE), "oracle")
dp = C.POINTER(C.c_double)


class Report(C.Structure):
    """orc_clearance_report == isdf_clearance_report"""
    _fields_ = [("min_clearance", C.c_double), ("t_min", C.c_double), ("p_min", C.c_double * 3), ("t_hit", C.c_double), ("p_hit", C.c_double * 3)] + \
               [(n, C.c_int32) for n in ["collides", "piece_min", "sample_min", "piece_hit", "sample_hit", "reserved_"]]

    def as_dict(self):
        return dict(min_clearance=self.min_clearance, t_min=self.t_min, p_min=np.array(self.p_min[:]), t_hit=self.t_hit, p_hit=np.array(self.p_hit[:]),
                    collides=bool(self.collides), piece_min=self.piece_min, sample_min=self.sample_min, piece_hit=self.piece_hit,
                    sample_hit=self.sample_hit)


_lib = None


def lib():
    global _lib
    if _lib is None:
        flags = ["-O3", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fopenmp", "-shared"]
        srcs = [SRC] + sorted(os.path.join(ORACLE_DIR, f) for f in os.listdir(ORACLE_DIR) if f.endswith(".hpp"))
        h = hashlib.sha256(" ".join(flags).encode() + b"".join(open(s, "rb").read() for s in srcs)).hexdigest()[:16]
        d = os.path.join(tempfile.gettempdir(), f"isdf_collision_oracle_{os.getuid()}")
        os.makedirs(d, exist_ok=True)
        so = os.path.join(d, f"libcollision_oracle_{h}.so")
        if not os.path.exists(so):
            cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
            tmp = so + f".{os.getpid()}.tmp"
            subprocess.check_call([cxx] + flags + ["-o", tmp, SRC])
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.orc_check_collision.argtypes = [dp, C.c_double, C.POINTER(C.c_uint8), C.c_int, C.c_int, C.c_int, dp, C.c_double, C.c_void_p, C.c_int, C.c_int,
                                          dp, dp, C.c_int, C.c_double, C.c_double, C.POINTER(Report), dp, C.c_int]
        _lib = L
    return _lib


def check_collision(cfg, occ, bmin, res, shape, T, coeffs, samples_per_piece, margin, horizon, B=1, unrestricted=False):
    """cfg: an isdf_config-layout struct; shape: oracle_lib.Shape. Returns (list of B report dicts, clearance (B, N0, M + 1))."""
    T = O.f64(T).reshape(-1)
    Cc = O.f64(coeffs).reshape(-1)
    N0, M = T.size // B, int(samples_per_piece)
    occ = np.ascontiguousarray(occ, dtype=np.uint8)
    X, Y, Z = occ.shape
    flat = O.f64([cfg.vehicle_mass, cfg.grav_acc, cfg.horiz_drag, cfg.vert_drag, cfg.paras_drag, cfg.speed_eps])
    bd = cfg.kernel_size * cfg.occupancy_resolution
    reps = (Report * B)()
    clear = np.zeros(T.size * (M + 1))
    lib().orc_check_collision(flat.ctypes.data_as(dp), bd, occ.ctypes.data_as(C.POINTER(C.c_uint8)), X, Y, Z, O.f64(bmin).ctypes.data_as(dp), float(res),
                              shape.h, B, N0, T.ctypes.data_as(dp), Cc.ctypes.data_as(dp), M, float(margin), float(horizon), reps,
                              clear.ctypes.data_as(dp), int(unrestricted))
    return [r.as_dict() for r in reps], clear.reshape(B, N0, M + 1)
