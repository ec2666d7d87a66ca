"""Whole-body collision check on the device (isdf_check_collision, csrc/isdf_check.cuh) against its oracle (tests/collision_oracle.cpp):
per-sample clearance, verdict, first hit and argmin voxels; determinism and batch composition; edges; no side effects on the cost paths;
the random-restart selection recipe of INTEGRATION.md."""
import ctypes as C
import numpy as np
import pytest
import isdf_b200 as I
import oracle_lib as O
import collision_oracle as CO
import workloads as W
from common import small_case, BMIN, MESHES

pytestmark = pytest.mark.gpu

RES = 1.0
CUBE = RES * np.sqrt(3) / 2          # "no occupied voxel cube touches the robot" for a 1-Lipschitz SDF


def maps():
    cfg, occ, T, Cc, _ = small_case(N=4, K=16, seed=3)
    rocc = W.random_map(48, 48, 40, p=0.04, seed=21, slabs=2)
    rT, rC, _ = W.make_trajectory(4, [0, 0, 0], [48, 48, 40], seed=22, jitter=0.3)
    return cfg, [("three_slit", occ, T, Cc), ("random", rocc, rT, rC)]


def assert_parity(got, gclear, exp, eclear, margin, tol=1e-12, what=""):
    """per-sample clearance within tol; verdict, first hit and argmin voxels identical (cases have no value within 1e-9 of the margin)"""
    assert np.abs(gclear - eclear).max() <= tol, (what, np.abs(gclear - eclear).max())
    assert np.abs(eclear - margin).min() > 1e-9, what
    for g, e in zip(got, exp):
        assert g["collides"] == e["collides"], what
        assert (g["piece_hit"], g["sample_hit"]) == (e["piece_hit"], e["sample_hit"]), what
        assert np.array_equal(g["p_hit"], e["p_hit"], equal_nan=True), what
        assert abs(g["t_hit"] - e["t_hit"]) <= 1e-12 * max(1.0, abs(e["t_hit"])), what
        assert abs(g["min_clearance"] - e["min_clearance"]) <= tol, what
        if tol <= 1e-12:
            # the last sample of piece i and the first of piece i + 1 are the same pose up to rounding: where the minimum sits on such a
            # junction either one may be reported first, with the same voxel and the same time
            same = (g["piece_min"], g["sample_min"]) == (e["piece_min"], e["sample_min"])
            junction = (g["sample_min"] == 0 and g["piece_min"] == e["piece_min"] + 1 and e["sample_min"] == gclear.shape[-1] - 1) or \
                       (e["sample_min"] == 0 and e["piece_min"] == g["piece_min"] + 1 and g["sample_min"] == gclear.shape[-1] - 1)
            assert same or junction, (what, (g["piece_min"], g["sample_min"]), (e["piece_min"], e["sample_min"]))
            assert np.array_equal(g["p_min"], e["p_min"], equal_nan=True), what
            assert abs(g["t_min"] - e["t_min"]) <= 1e-12 * max(1.0, abs(e["t_min"])), what


def sweep(ev, osh, cfg, cases, Ms=(1, 16, 64), tol=1e-12, margins=(-0.05, 0.0, CUBE)):
    compared = 0
    for name, occ, T, Cc in cases:
        ev.set_map_u8(occ, BMIN, RES)
        for M in Ms:
            for H in (cfg.safety_hor, 1.0):
                for margin in margins:
                    what = f"{name} M={M} H={H} margin={margin}"
                    if margin > H:
                        with pytest.raises(I.IsdfError) as e:
                            ev.check_collision(T, Cc, M, margin, H)
                        assert e.value.code == -1
                        continue
                    got, gclear = ev.check_collision(T, Cc, M, margin, H, per_sample=True)
                    exp, eclear = CO.check_collision(cfg, occ, BMIN, RES, osh, T, Cc, M, margin, H)
                    assert_parity(got, gclear, exp, eclear, margin, tol, what)
                    compared += 1
    return compared


@pytest.mark.parametrize("shape", ["Ball", "CappedCone", "Torus", "SmoothIntersection", "WireframeBox", "Box"])
def test_analytic_shapes_match_the_oracle(shape):
    cfg, cases = maps()
    ev = I.Evaluator(cfg)
    if shape == "Box":
        R, t = W.rotation_from_poly_params([0.3, -0.2, 0.1, 30.0, -20.0, 45.0])
        ev.set_shape_analytic(I.SHAPE_KINDS["BOX"], [1.4, 0.6, 0.5], R, t)
        osh = O.Shape.analytic(I.SHAPE_KINDS["BOX"], [1.4, 0.6, 0.5], R, t)
    else:
        ev.set_shape_named(shape)
        osh = O.Shape.named(shape)
    n = sweep(ev, osh, cfg, cases)
    assert n >= 24
    ev.close()


def ref_mesh(name):
    d = np.load(__import__("os").path.join(__import__("os").path.dirname(__file__), "golden", "ref_meshes.npz"))
    return d[f"{name}_V"], d[f"{name}_F"], d[f"{name}_pp"]


@pytest.mark.parametrize("mesh", ["box", "lprism", "ico", "RoundedCone", "Lthick"])
def test_exact_sign_meshes_match_the_oracle(mesh):
    cfg, cases = maps()
    if mesh in MESHES:
        V, F = MESHES[mesh]()
        pp = [0, 0, 0, 30, -15, 60]
    else:
        V, F, pp = ref_mesh(mesh)
    ev = I.Evaluator(cfg)
    ev.set_shape_mesh(V, F, pp, I.MESH_SIGN_EXACT)
    osh = O.Shape.mesh(V, F, pp, wn_mode=O.WN_EXACT)
    n = sweep(ev, osh, cfg, cases, Ms=(1, 16) if mesh == "RoundedCone" else (1, 16, 64))
    assert n >= 16
    # branch-and-bound: most boxed voxels never reach a triangle
    ev.set_map_u8(cases[1][1], BMIN, RES)
    ev.check_collision(cases[1][2], cases[1][3], 16, 0.0, 1.0)
    cnt, _ = ev.dbg_check_stats()
    assert cnt["mesh_searches"] < cnt["voxels_in_box"], cnt
    ev.close()


def test_winding_sign_soup_matches_the_oracle_to_the_winding_approximation():
    """s = 1 - 2 w with the product's hierarchical w against the oracle's exact w: agreement is bounded by the tree's approximation
    (|dw| ~1e-4, tests/test_gpu_soup.py), not by rounding. Distances and the enumeration are exact, so the verdict agrees wherever no
    sample lies within that tolerance of the margin."""
    cfg, cases = maps()
    V, F = MESHES["rcone"]()
    keep = np.ones(len(F), bool)
    keep[3::7] = False
    V, F = V, F[keep]
    ev = I.Evaluator(cfg)
    ev.set_shape_mesh(V, F, [0, 0, 0, 120, 0, 0], I.MESH_SIGN_WINDING)
    osh = O.Shape.mesh(V, F, [0, 0, 0, 120, 0, 0], wn_mode=O.WN_RAW)
    tol, verdicts = 2e-3, 0
    for name, occ, T, Cc in cases:
        ev.set_map_u8(occ, BMIN, RES)
        for M in (1, 16):
            for margin in (-0.05, 0.0, 0.5):
                got, gclear = ev.check_collision(T, Cc, M, margin, 1.0, per_sample=True)
                exp, eclear = CO.check_collision(cfg, occ, BMIN, RES, osh, T, Cc, M, margin, 1.0)
                assert np.abs(gclear - eclear).max() <= tol, (name, M, np.abs(gclear - eclear).max())
                assert abs(got[0]["min_clearance"] - exp[0]["min_clearance"]) <= tol
                if np.abs(eclear - margin).min() > tol:
                    assert got[0]["collides"] == exp[0]["collides"]
                    assert (got[0]["piece_hit"], got[0]["sample_hit"]) == (exp[0]["piece_hit"], exp[0]["sample_hit"])
                    verdicts += 1
                a, ca = ev.check_collision(T, Cc, M, margin, 1.0, per_sample=True)
                assert np.array_equal(ca, gclear)                                          # deterministic
    assert verdicts >= 6
    ev.close()


@pytest.fixture(scope="module")
def big():
    X = 512
    occ = W.random_map(X, X, X, p=0.05, seed=1, slabs=3)
    cfg = I.default_config_values()
    cfg.integral_intervs = 256
    cfg.flags = I.WITH_COLLISION
    T, Cc, wp = W.make_trajectory(64, [0, 0, 0], [X, X, X], seed=11, jitter=0.2)
    return cfg, occ, T, Cc


def test_full_size_configs2_mesh_against_the_oracle(big):
    """configs[2]: 512^3 map, 64 pieces x 256 check intervals, the 3900-triangle mesh robot; every sample against the oracle"""
    cfg, occ, T, Cc = big
    V, F = W.rounded_cone_mesh()
    ev = I.Evaluator(cfg)
    ev.set_map_u8(occ, BMIN, RES)
    ev.set_shape_mesh(V, F, [0, 0, 0, 120, 0, 0], I.MESH_SIGN_EXACT)
    osh = O.Shape.mesh(V, F, [0, 0, 0, 120, 0, 0], wn_mode=O.WN_BH)
    margin, H = 0.0, cfg.safety_hor
    got, gclear = ev.check_collision(T, Cc, 256, margin, H, per_sample=True)
    exp, eclear = CO.check_collision(cfg, occ, BMIN, RES, osh, T, Cc, 256, margin, H)
    assert (eclear < H).mean() > 0.05
    assert_parity(got, gclear, exp, eclear, margin, 1e-12, "configs[2]")
    ev.close()


def test_determinism_batch_composition_and_device_entry_point():
    import torch
    cfg, occ, _, _, _ = small_case(N=4, K=16, seed=3)
    V, F = MESHES["lprism"]()
    ev = I.Evaluator(cfg)
    ev.set_map_u8(occ, BMIN, RES)
    N0, B, M = 4, 8, 32
    Ts, Cs = [], []
    for b in range(B):
        T, Cc, _ = W.make_trajectory(N0, [0, 0, 0], [50, 50, 34], seed=40 + b, jitter=0.3)
        Ts.append(T); Cs.append(Cc.reshape(3, 6 * N0))
    Tb = np.concatenate(Ts)
    Cb = np.concatenate(Cs, axis=1).reshape(-1)                 # column-major 6BN0 x 3: axis blocks of all pieces
    for setter in (lambda: ev.set_shape_named("CappedCone"), lambda: ev.set_shape_mesh(V, F, [0, 0, 0, 20, 0, 0], I.MESH_SIGN_EXACT),
                   lambda: ev.set_shape_mesh(V, F, [0, 0, 0, 20, 0, 0], I.MESH_SIGN_WINDING)):
        setter()
        a, ca = ev.check_collision(Tb, Cb, M, 0.0, 1.0, B=B, per_sample=True)
        b2, cb = ev.check_collision(Tb, Cb, M, 0.0, 1.0, B=B, per_sample=True)
        assert np.array_equal(ca, cb) and all(x == y or (np.isnan(x["t_hit"]) and np.isnan(y["t_hit"])) for x, y in
                                              zip([r["t_hit"] for r in a], [r["t_hit"] for r in b2]))
        for b in range(B):
            s, cs = ev.check_collision(Ts[b], Cs[b].reshape(-1), M, 0.0, 1.0, per_sample=True)
            assert np.array_equal(cs[0], ca[b]), b
            for k in ("min_clearance", "t_min", "t_hit", "collides", "piece_min", "sample_min", "piece_hit", "sample_hit"):
                assert s[0][k] == a[b][k] or (np.isnan(s[0][k]) and np.isnan(a[b][k])), (b, k)
            assert np.array_equal(s[0]["p_min"], a[b]["p_min"], equal_nan=True) and np.array_equal(s[0]["p_hit"], a[b]["p_hit"], equal_nan=True)
        # device entry point == host entry point
        dT, dC = torch.tensor(Tb, device="cuda"), torch.tensor(Cb, device="cuda")
        drep = torch.zeros(B * C.sizeof(I.ClearanceReport), dtype=torch.uint8, device="cuda")
        dclear = torch.zeros(ca.size, dtype=torch.float64, device="cuda")
        stream = torch.cuda.current_stream().cuda_stream
        ev.check_collision_device(B, N0, dT.data_ptr(), dC.data_ptr(), M, 0.0, 1.0, drep.data_ptr(), dclear.data_ptr(), stream)
        torch.cuda.synchronize()
        assert np.array_equal(dclear.cpu().numpy().reshape(ca.shape), ca)
        raw = drep.cpu().numpy().tobytes()
        reps = (I.ClearanceReport * B).from_buffer_copy(raw)
        for b in range(B):
            d = reps[b].as_dict()
            for k in ("min_clearance", "t_min", "t_hit", "collides", "piece_min", "sample_min", "piece_hit", "sample_hit"):
                assert d[k] == a[b][k] or (np.isnan(d[k]) and np.isnan(a[b][k])), (b, k)
        # the device entry point poisons its reports on failure
        with pytest.raises(I.IsdfError):
            ev.check_collision_device(B, N0, dT.data_ptr(), dC.data_ptr(), M, 2.0, 1.0, drep.data_ptr(), 0, stream)
        torch.cuda.synchronize()
        reps = (I.ClearanceReport * B).from_buffer_copy(drep.cpu().numpy().tobytes())
        assert all(np.isnan(r.min_clearance) and r.collides == 1 for r in reps)
    ev.close()


def test_edges_empty_map_outside_the_map_wall_and_state_errors():
    cfg = I.default_config_values()
    ev = I.Evaluator(cfg)
    T, Cc = np.array([4.0]), np.zeros((3, 6))
    Cc[:, 0], Cc[:, 1] = [2.3, 10.3, 10.6], [9.0, 0, 0]                   # straight flight along x at 9 m/s (off the voxel grid's symmetry)
    Cc = Cc.reshape(-1)
    # state errors: every report poisoned
    for setup in (lambda: None, lambda: ev.set_shape_named("Ball")):
        setup()
        reps = (I.ClearanceReport * 1)()
        dp = C.POINTER(C.c_double)
        r = ev.lib.isdf_check_collision(ev.h, 1, 1, T.ctypes.data_as(dp), Cc.ctypes.data_as(dp), 8, 0.0, 1.0, reps, None)
        assert r == -2 and np.isnan(reps[0].min_clearance) and reps[0].collides == 1
    # empty map: c = H everywhere, no hit, no argmin voxel
    ev.set_map_u8(np.zeros((40, 20, 20), np.uint8), BMIN, RES)
    rep, cl = ev.check_collision(T, Cc, 16, 0.0, 0.9, per_sample=True)
    assert (cl == 0.9).all() and rep[0]["min_clearance"] == 0.9 and not rep[0]["collides"] and rep[0]["t_hit"] == -1
    assert np.isnan(rep[0]["p_min"]).all() and np.isnan(rep[0]["p_hit"]).all()
    # a wall across the flight: a hit, first at the closed-form sample, the wall voxel nearest to the robot
    occ = np.zeros((40, 20, 20), np.uint8)
    occ[20, :, :] = 1
    osh = O.Shape.named("Ball")
    ev.set_shape_named("Ball")
    ev.set_map_u8(occ, BMIN, RES)
    rep, cl = ev.check_collision(T, Cc, 36, 0.0, 1.0, per_sample=True)
    exp, ecl = CO.check_collision(cfg, occ, BMIN, RES, osh, T, Cc, 36, 0.0, 1.0)
    assert_parity(rep, cl, exp, ecl, 0.0, 1e-12, "wall")
    r_ball = O.Shape.named("Ball").params()[0]
    t = np.arange(37) * (4.0 / 36)
    x = 2.3 + 9 * t
    expect = np.minimum(1.0, np.sqrt((x - 20.5) ** 2 + 0.05) - r_ball)    # nearest wall voxel: centre (20.5, 10.5, 10.5)
    assert np.abs(cl[0, 0] - expect).max() <= 1e-12
    assert rep[0]["collides"] and rep[0]["sample_hit"] == int(np.argmax(expect < 0.0))
    # partly outside the map: the map covers x < 20 only; samples beyond see free space
    occ2 = np.ones((20, 20, 20), np.uint8)
    occ2[:, 9:12, 9:12] = 0                                               # a tunnel: nearest wall voxel centres 1.8 m from the flight line
    ev.set_map_u8(occ2, BMIN, RES)
    rep, cl = ev.check_collision(T, Cc, 36, -0.05, 1.0, per_sample=True)
    exp, ecl = CO.check_collision(cfg, occ2, BMIN, RES, osh, T, Cc, 36, -0.05, 1.0)
    assert_parity(rep, cl, exp, ecl, -0.05, 1e-12, "outside")
    assert (cl[0, 0][x > 20 + 2] == 1.0).all() and (cl[0, 0][x < 19] < 1.0).all()          # past the map's end: free space
    ev.close()


def test_check_leaves_the_cost_paths_untouched():
    cfg, occ, T, Cc, wp = small_case(N=4, K=16, seed=3)
    V, F = MESHES["rcone"]()
    ev = I.Evaluator(cfg)
    ev.set_map_u8(occ, BMIN, RES)
    ev.set_shape_mesh(V, F, [0, 0, 0, 120, 0, 0])
    pts = W.gather_obstacle_points(occ, BMIN, RES, wp, cfg.kernel_size * cfg.occupancy_resolution / 3.0)[:200]
    ev.set_points(pts)
    d0, d1 = ev.eval_discrete(T, Cc), ev.eval_discrete(T, Cc)       # the second runs on the work items the first built
    s0 = ev.eval_swept(T, Cc)
    ts0 = ev.swept_results()[0].copy()
    T2, C2, _ = W.make_trajectory(6, [0, 0, 0], [50, 50, 34], seed=9, jitter=0.3)
    ev.check_collision(T2, C2, 64, 0.0, 1.0)
    ev.check_collision(T, Cc, 16, 0.0, cfg.safety_hor)
    d2 = ev.eval_discrete(T, Cc)
    assert d2[0] == d1[0] and np.array_equal(d2[1], d1[1]) and np.array_equal(d2[2], d1[2])
    assert np.array_equal(ev.swept_results()[0], ts0)               # lastTstar untouched by the check
    s1 = ev.eval_swept(T, Cc)
    ev.set_points(pts)
    s2 = ev.eval_swept(T, Cc)
    assert s2[0] == s0[0] and np.array_equal(s2[1], s0[1]) and np.array_equal(s2[2], s0[2])
    assert np.isfinite(s1[0]) and d0[0] == d1[0]
    ev.close()


def test_restart_recipe_selects_a_collision_free_trajectory():
    """INTEGRATION.md: isdf_lbfgs_batch -> isdf_callback_batch on the final x -> isdf_get_batch_trajectories -> isdf_check_collision(B)
    -> the lowest-cost trajectory that does not collide; the oracle agrees with its verdict"""
    from test_gpu_lbfgs_device import problems
    cfg, _, _, _, _ = small_case(N=6, K=16, seed=3)
    occ = W.random_map(64, 64, 48, p=0.003, seed=5, slabs=0)                  # sparse obstacles: some restarts end collision-free
    cfg.vmax, cfg.omgmax = 1.2, 0.5
    B, N0, rho = 16, 6, 20.0
    heads, tails, X = problems(B, N0, seed=300)
    ev = I.Evaluator(cfg)
    ev.set_map_u8(occ, BMIN, RES)
    ev.set_shape_named("Ball")
    res = ev.lbfgs_batch(heads, tails, rho, X, ev.lbfgs_params(max_iterations=30, mem_size=8, past=3, delta=1e-7))
    cost, _ = ev.callback_batch(heads, tails, rho, res["x"])
    T, Cc, _ = ev.batch_trajectories(B, N0)
    margin, H = 0.0, cfg.safety_hor
    reps = ev.check_collision(T, Cc, cfg.integral_intervs, margin, H, B=B)
    free = [b for b in range(B) if not reps[b]["collides"]]
    assert free, [r["min_clearance"] for r in reps]
    pick = min(free, key=lambda b: cost[b])
    Tp = T[pick * N0:(pick + 1) * N0]
    Cp = Cc.reshape(3, B, 6 * N0)[:, pick, :].reshape(-1)
    exp, _ = CO.check_collision(cfg, occ, BMIN, RES, O.Shape.named("Ball"), Tp, Cp, cfg.integral_intervs, margin, H)
    assert reps[pick]["collides"] == 0 and exp[0]["collides"] == 0
    assert abs(reps[pick]["min_clearance"] - exp[0]["min_clearance"]) <= 1e-12
    ev.close()
