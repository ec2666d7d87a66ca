"""Whole-body collision check without a GPU: the oracle (tests/collision_oracle.cpp) against closed forms and a numpy brute force,
the box-restriction property of 1-Lipschitz SDFs, argument validation of the C ABI and the report's layout."""
import ctypes as C
import os
import subprocess
import numpy as np
import pytest
import isdf_b200 as I
import oracle_lib as O
import collision_oracle as CO
import workloads as W

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def ball_cfg():
    cfg = I.default_config_values()
    cfg.flags = I.WITH_COLLISION
    return cfg


def line_traj(p0, v, T):
    """one piece p(t) = p0 + v t (6 x 3 column-major coefficient block)"""
    Cc = np.zeros((3, 6))
    Cc[:, 0], Cc[:, 1] = p0, v
    return np.array([float(T)]), Cc.reshape(-1)


def piece_positions(T, Cc, M):
    """numpy: positions of every check sample (piece-major), local time j * (T_i * (1/M))"""
    N = T.size
    Cm = Cc.reshape(3, N, 6)
    out = []
    for i in range(N):
        step = T[i] * (1.0 / M)
        t = np.arange(M + 1) * step
        P = t[:, None] ** np.arange(6)[None, :]
        out.append(P @ Cm[:, i, :].T)
    return np.concatenate(out)


def test_ball_passing_one_voxel_closed_form():
    """a ball of radius 1 flies along x at 9 m/s and passes a single occupied voxel 3 m to the side: c = 3 - 1 at closest approach,
    and the first hit below a margin of 2.2 is the first sample with |9 t - 18| < sqrt(3.2^2 - 9)"""
    cfg = ball_cfg()
    occ = np.zeros((40, 20, 20), np.uint8)
    occ[20, 13, 10] = 1                                  # centre (20.5, 13.5, 10.5)
    T, Cc = line_traj([2.5, 10.5, 10.5], [9.0, 0, 0], 4.0)
    M, H, margin = 36, 2.5, 2.2
    rep, clear = CO.check_collision(cfg, occ, [0, 0, 0], 1.0, O.Shape.analytic(0, [1.0]), T, Cc, M, margin, H)
    r = rep[0]
    assert abs(r["min_clearance"] - 2.0) <= 1e-12
    assert r["piece_min"] == 0 and r["sample_min"] == 18 and abs(r["t_min"] - 2.0) <= 1e-12
    assert np.array_equal(r["p_min"], [20.5, 13.5, 10.5])
    t = np.arange(M + 1) * (4.0 / M)
    expect = np.minimum(H, np.sqrt((2.5 + 9 * t - 20.5) ** 2 + 9.0) - 1.0)
    assert np.abs(clear[0, 0] - expect).max() <= 1e-12
    j_hit = int(np.argmax(np.abs(9 * t - 18) < np.sqrt((margin + 1) ** 2 - 9)))
    assert j_hit == 17
    assert r["collides"] and r["sample_hit"] == j_hit and abs(r["t_hit"] - 17 / 9) <= 1e-12 and np.array_equal(r["p_hit"], [20.5, 13.5, 10.5])
    # a margin below the minimum: no hit, and the report says so
    rep2, _ = CO.check_collision(cfg, occ, [0, 0, 0], 1.0, O.Shape.analytic(0, [1.0]), T, Cc, M, 1.9, H)
    assert not rep2[0]["collides"] and rep2[0]["t_hit"] == -1 and rep2[0]["sample_hit"] == -1 and np.isnan(rep2[0]["p_hit"]).all()
    # nothing within the horizon: c == H everywhere and no argmin voxel
    rep3, clear3 = CO.check_collision(cfg, occ, [0, 0, 0], 1.0, O.Shape.analytic(0, [1.0]), T, Cc, M, 0.0, 1.5)
    assert (clear3 == 1.5).all() and rep3[0]["min_clearance"] == 1.5 and np.isnan(rep3[0]["p_min"]).all()
    assert rep3[0]["sample_min"] == 0 and not rep3[0]["collides"]


@pytest.mark.parametrize("radius,H", [(0.8, 0.866), (2.5, 1.0), (4.0, 3.0)])
def test_oracle_matches_numpy_brute_force_for_balls(radius, H):
    """Ball: sdf = |p| - r is rotation-free and the robot lies inside its kernel cube, so c = min(H, min over ALL occupied voxels)"""
    cfg = ball_cfg()
    occ = W.random_map(32, 32, 24, p=0.03, seed=4, slabs=1)
    T, Cc, _ = W.make_trajectory(3, [0, 0, 0], [32, 32, 24], seed=5, jitter=0.3)
    M = 12
    rep, clear = CO.check_collision(cfg, occ, [0, 0, 0], 1.0, O.Shape.analytic(0, [radius]), T, Cc, M, 0.0, H)
    P = piece_positions(T, Cc, M)
    vox = (np.argwhere(occ) + 0.5)
    d = np.sqrt(((P[:, None, :] - vox[None, :, :]) ** 2).sum(-1)) - radius
    expect = np.minimum(H, d.min(1))
    assert np.abs(clear.reshape(-1) - expect).max() <= 1e-12
    k = int(np.argmin(expect))
    assert rep[0]["min_clearance"] == clear.reshape(-1)[k] and rep[0]["piece_min"] * (M + 1) + rep[0]["sample_min"] == k
    if expect[k] < H:
        assert np.allclose(rep[0]["p_min"], vox[np.argmin(d[k])], atol=0)


def test_box_restriction_changes_nothing_for_an_exact_mesh_inside_its_cube():
    cfg = ball_cfg()
    occ = W.random_map(28, 28, 24, p=0.04, seed=7, slabs=1)
    T, Cc, _ = W.make_trajectory(3, [0, 0, 0], [28, 28, 24], seed=8, jitter=0.3)
    V, F = W.l_prism_mesh()
    sh = O.Shape.mesh(V, F, [0, 0, 0, 30, 10, 0])
    for H in (0.866, 2.0):
        a, ca = CO.check_collision(cfg, occ, [0, 0, 0], 1.0, sh, T, Cc, 6, 0.0, H)
        b, cb = CO.check_collision(cfg, occ, [0, 0, 0], 1.0, sh, T, Cc, 6, 0.0, H, unrestricted=True)
        assert np.array_equal(ca, cb)
        assert a[0]["min_clearance"] == b[0]["min_clearance"] and np.array_equal(a[0]["p_min"], b[0]["p_min"], equal_nan=True)
        assert (ca < H).any()


def _report_layout_from_c():
    src = r'''#include <stdio.h>
#include <stddef.h>
#include "isdf.h"
int main(void) {
    isdf_clearance_report r;
    r.collides = 0; (void)r;
    printf("%d %d %d %d %d %d %d %d %d %d %d %d\n", (int)sizeof(isdf_clearance_report), (int)offsetof(isdf_clearance_report, min_clearance),
           (int)offsetof(isdf_clearance_report, t_min), (int)offsetof(isdf_clearance_report, p_min), (int)offsetof(isdf_clearance_report, t_hit),
           (int)offsetof(isdf_clearance_report, p_hit), (int)offsetof(isdf_clearance_report, collides), (int)offsetof(isdf_clearance_report, piece_min),
           (int)offsetof(isdf_clearance_report, sample_min), (int)offsetof(isdf_clearance_report, piece_hit), (int)offsetof(isdf_clearance_report, sample_hit),
           (int)offsetof(isdf_clearance_report, reserved_));
    return 0;
}
'''
    return src


def test_report_layout_matches_the_header_and_compiles_as_c99(tmp_path):
    src = tmp_path / "rep.c"
    src.write_text(_report_layout_from_c())
    exe = str(tmp_path / "rep")
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe],
                       capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    got = [int(v) for v in subprocess.check_output([exe]).split()]
    R = I.ClearanceReport
    names = ["min_clearance", "t_min", "p_min", "t_hit", "p_hit", "collides", "piece_min", "sample_min", "piece_hit", "sample_hit", "reserved_"]
    assert got == [C.sizeof(R)] + [getattr(R, n).offset for n in names]
    assert C.sizeof(R) == 96 and C.sizeof(CO.Report) == 96
    assert [getattr(CO.Report, n).offset for n in names] == [getattr(R, n).offset for n in names]


def _call(lib, ctx, B, N0, M, margin, horizon, with_data=True):
    reps = (I.ClearanceReport * max(B, 1))()
    for r in reps:
        r.min_clearance, r.collides = 123.0, 0
    T, Cc = np.ones(max(B * N0, 1)), np.zeros(18 * max(B * N0, 1))
    dp = C.POINTER(C.c_double)
    rc = lib.isdf_check_collision(ctx, B, N0, T.ctypes.data_as(dp) if with_data else None, Cc.ctypes.data_as(dp) if with_data else None, M,
                                  margin, horizon, reps, None)
    return rc, reps


def test_argument_validation_poisons_every_report_without_a_gpu():
    lib = I.load_library()
    rc, reps = _call(lib, None, 3, 4, 16, 0.0, 1.0)
    assert rc == -1 and b"ctx" in lib.isdf_last_error()
    assert all(np.isnan(r.min_clearance) and r.collides == 1 for r in reps)          # a caller ignoring the status never reads "safe"
    for args, word in [((3, 4, 16, 1.5, 1.0), b"margin"), ((3, 4, 16, 0.0, 0.0), b"horizon"), ((3, 4, 16, 0.0, float("inf")), b"horizon"),
                       ((3, 4, 0, 0.0, 1.0), b"samples_per_piece"), ((3, 4, 4097, 0.0, 1.0), b"samples_per_piece"), ((0, 4, 16, 0.0, 1.0), b"N0"),
                       ((3, 0, 16, 0.0, 1.0), b"N0"), ((3, 4, 16, float("nan"), 1.0), b"margin")]:
        rc, reps = _call(lib, None, *args)
        assert rc == -1 and word in lib.isdf_last_error(), (args, lib.isdf_last_error())
        if args[0] > 0:
            assert all(np.isnan(r.min_clearance) and r.collides == 1 for r in reps)
    assert lib.isdf_check_collision_device(None, 1, 1, None, None, 16, 0.0, 1.0, None, None, None) == -1


def test_host_adapter_exports_the_verdict_hook():
    import host_lib
    host = os.path.join(ROOT, "implicit-sdf-planner_b200", "host", "libisdf_host.so")
    if not os.path.exists(host):
        import __graft_entry__ as G
        G.build()
    out = subprocess.check_output(["nm", "-D", "--defined-only", host]).decode()
    assert "isdf_host_backend_collides" in out
    assert host_lib.LIB == host
