"""Pins for the oracle itself (CPU): finite differences, independent restatements, known answers.
The reference ships no golden vectors for this path (SURVEY.md §4/§8c), so these are what anchors the checker."""
import ctypes as C
import os
import numpy as np
import pytest
import isdf_b200 as I
import oracle_lib as O
import workloads as W
from common import small_case, rel_l2, BMIN, tilted, MESHES


def ocfg(cfg=None):
    return O.config_from(cfg if cfg is not None else I.default_config_values())


def test_config_layout_matches_abi():
    assert C.sizeof(O.OrcConfig) == C.sizeof(I.Config) == 16 * 8 + 4 * 4


def test_flatness_adjoint_matches_central_differences():
    cfg = ocfg()
    rng = np.random.default_rng(0)
    for _ in range(25):
        v, a, j = rng.normal(size=3) * 3, rng.normal(size=3) * 3, rng.normal(size=3) * 3
        qb, ob = rng.normal(size=4), rng.normal(size=3)
        g = O.flat_backward(cfg, v, a, j, np.zeros(3), np.zeros(3), qb, ob)

        def L(v, a, j):
            q, o = O.flat_forward(cfg, v, a, j)
            return q @ qb + o @ ob
        num = np.zeros((3, 3))
        eps = 1e-6
        for k in range(3):
            for c in range(3):
                xp, xm = [v.copy(), a.copy(), j.copy()], [v.copy(), a.copy(), j.copy()]
                xp[k][c] += eps
                xm[k][c] -= eps
                num[k, c] = (L(*xp) - L(*xm)) / (2 * eps)
        assert np.abs(num - g[1:]).max() <= 1e-6 * (np.abs(g[1:]).max() + 1.0)
        q, _ = O.flat_forward(cfg, v, a, j)
        assert abs(np.linalg.norm(q) - 1) < 1e-12 and q[3] == 0.0   # unit quaternion, yaw == 0 (flat:80-84)


def test_flatness_passes_direct_grads_through():
    cfg = ocfg()
    rng = np.random.default_rng(1)
    v, a, j = rng.normal(size=3), rng.normal(size=3), rng.normal(size=3)
    pg, vg = rng.normal(size=3), rng.normal(size=3)
    g0 = O.flat_backward(cfg, v, a, j, np.zeros(3), np.zeros(3), np.ones(4), np.ones(3))
    g1 = O.flat_backward(cfg, v, a, j, pg, vg, np.ones(4), np.ones(3))
    assert np.allclose(g1[0], pg) and np.allclose(g1[1] - g0[1], vg)


@pytest.mark.parametrize("shape_name", ["Ball", "Torus", "RoundedCone"])
def test_discrete_gradient_is_the_gradient_of_the_cost(shape_name):
    # only exact distance fields: the reference normalises the FD gradient (Shape.hpp:56), so for the non-metric shapes
    # (smooth CSG, CappedCone, Trefoil, bend/twist) its "gradient" is by design not the derivative of the cost
    cfg, occ, T, Cc, _ = small_case(N=3, K=12, seed=5)
    cfg = ocfg(cfg)
    sh = O.Shape.named(shape_name)
    c0, gC, gT, npairs = O.eval_discrete(cfg, occ, BMIN, 1.0, sh, T, Cc)
    assert npairs > 100 and c0 > 0
    rng = np.random.default_rng(0)
    e = 1e-6
    # directional derivative along random directions (robust to isolated window-edge discontinuities)
    for _ in range(6):
        dC, dT = rng.normal(size=Cc.size), rng.normal(size=T.size) * 0.1
        cp = O.eval_discrete(cfg, occ, BMIN, 1.0, sh, T + e * dT, Cc + e * dC)[0]
        cm = O.eval_discrete(cfg, occ, BMIN, 1.0, sh, T - e * dT, Cc - e * dC)[0]
        num, ana = (cp - cm) / (2 * e), gC @ dC + gT @ dT
        assert abs(num - ana) <= 2e-4 * abs(ana) + 1e-3


def test_dynamics_only_terms_match_finite_differences():
    cfg, occ, T, Cc, _ = small_case(N=3, K=12, seed=7, flags=I.WITH_DYNAMICS)
    cfg.vmax, cfg.omgmax, cfg.thetamax = 0.8, 0.3, 0.2   # make every hinge active
    cfg = ocfg(cfg)
    c0, gC, gT, _ = O.eval_discrete(cfg, None, BMIN, 1.0, None, T, Cc)
    assert c0 > 0
    rng = np.random.default_rng(0)
    e = 1e-6
    for _ in range(5):
        dC, dT = rng.normal(size=Cc.size), rng.normal(size=T.size) * 0.1
        cp = O.eval_discrete(cfg, None, BMIN, 1.0, None, T + e * dT, Cc + e * dC)[0]
        cm = O.eval_discrete(cfg, None, BMIN, 1.0, None, T - e * dT, Cc - e * dC)[0]
        num, ana = (cp - cm) / (2 * e), gC @ dC + gT @ dT
        assert abs(num - ana) <= 1e-5 * abs(ana) + 1e-6


def test_omp_baseline_equals_serial_oracle():
    cfg, occ, T, Cc, _ = small_case(N=4, K=16, seed=2)
    cfg.threads_num = 4
    cfg = ocfg(cfg)
    sh = O.Shape.named("Torus")
    a = O.eval_discrete(cfg, occ, BMIN, 1.0, sh, T, Cc, use_omp=False)
    b = O.eval_discrete(cfg, occ, BMIN, 1.0, sh, T, Cc, use_omp=True)
    assert a[3] == b[3]
    assert abs(a[0] - b[0]) <= 1e-11 * abs(a[0]) and rel_l2(b[1], a[1]) < 1e-11 and rel_l2(b[2], a[2]) < 1e-11


def test_shard_partials_sum_to_full():
    cfg, occ, T, Cc, _ = small_case(N=3, K=10, seed=4)
    cfg = ocfg(cfg)
    sh = O.Shape.named("Ball")
    full = O.eval_discrete(cfg, occ, BMIN, 1.0, sh, T, Cc)
    parts = [O.eval_discrete(cfg, occ, BMIN, 1.0, sh, T, Cc, rank=r, world=3) for r in range(3)]
    assert abs(sum(p[0] for p in parts) - full[0]) <= 1e-12 * abs(full[0])
    assert rel_l2(sum(p[1] for p in parts), full[1]) < 1e-12
    assert sum(p[3] for p in parts) == full[3]


# ---- grid quirks (Gridmap3D.cpp:135-194, 239-284; PCSmap_manager.h:130-170) ------------------------------------------
def test_points_in_aabb_against_numpy_restatement():
    rng = np.random.default_rng(3)
    occ = (rng.random((20, 17, 13)) < 0.2).astype(np.uint8)
    bmin, res = np.array([-3.0, 1.0, 0.5]), 0.5
    bmax = bmin + np.array(occ.shape) * res
    for _ in range(30):
        c = bmin + (bmax - bmin) * (rng.random(3) * 1.6 - 0.3)   # also outside the map
        half = rng.uniform(0.3, 3.0)
        pts, n = O.points_in_aabb(occ, bmin, res, c, half)
        lo, hi = np.clip(c - half, bmin, bmax), np.clip(c + half, bmin, bmax)
        i0 = np.clip(np.floor((lo - bmin) / res).astype(int), 0, np.array(occ.shape) - 1)
        i1 = np.clip(np.floor((hi - bmin) / res).astype(int), 0, np.array(occ.shape) - 1)
        exp = []
        for i in range(i0[0], i1[0] + 1):
            for j in range(i0[1], i1[1] + 1):
                for k in range(i0[2], i1[2] + 1):
                    if occ[i, j, k]:
                        exp.append([(i + .5) * res + bmin[0], (j + .5) * res + bmin[1], (k + .5) * res + bmin[2]])
        assert n == len(exp)
        if n:
            assert np.array_equal(pts, np.array(exp))


# ---- shapes -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", I.NAMED_SHAPES)
def test_named_shapes_evaluate_and_have_unit_fd_gradient(name):
    R, t = tilted()
    sh = O.Shape.named(name, R, t)
    rng = np.random.default_rng(5)
    p = rng.uniform(-6, 6, size=(200, 3))
    sdf, g = sh.query(p, 2)
    assert np.all(np.isfinite(sdf)) and np.all(np.isfinite(g))
    n = np.linalg.norm(g, axis=1)
    ok = n > 0
    assert ok.mean() > 0.95 and np.allclose(n[ok], 1.0, atol=1e-9)
    s0, _ = sh.query(p, 0)
    _, g1 = sh.query(p, 1)
    assert np.array_equal(s0, sdf) and np.array_equal(g1, g)


def test_ball_closed_form():
    sh = O.Shape.named("Ball")
    p = np.random.default_rng(0).normal(size=(50, 3)) * 3
    s, g = sh.query(p)
    assert np.allclose(s, np.linalg.norm(p, axis=1) - 1.0, rtol=0, atol=1e-15)
    assert np.allclose(g, p / np.linalg.norm(p, axis=1, keepdims=True), atol=1e-15)


def test_box_gradient_is_one_sided_and_unnormalised():
    sh = O.Shape.analytic(I.SHAPE_KINDS["BOX"], [1.5, 0.15, 0.15])   # Shape.hpp:2363-2377 (quirk Q9)
    p = np.array([[2.0, 0.4, 0.3], [0.2, 0.05, 0.0]])
    s, g = sh.query(p)
    s0 = sh.query(p, 0)[0]
    for i in range(2):
        for a in range(3):
            q = p[i].copy()
            q[a] += 0.01
            assert abs(g[i, a] - (sh.query(q[None], 0)[0][0] - s0[i]) / 0.01) < 1e-12
    assert abs(np.linalg.norm(g[0]) - 1.0) > 1e-4   # near a corner the one-sided dx=0.01 FD is visibly not unit length


def test_analytic_rounded_cone_agrees_with_its_mesh():
    """cross-check of two independent SDF paths at mesh-discretisation tolerance (SURVEY §8c)"""
    V, F = W.rounded_cone_mesh(n_theta=64, n_prof=48)
    assert W.mesh_volume(V, F) > 0
    msh, ash = O.Shape.mesh(V, F), O.Shape.named("RoundedCone")
    p = np.random.default_rng(2).uniform(-4, 7, size=(300, 3))
    sm, gm = msh.query(p)
    sa, ga = ash.query(p)
    assert np.abs(sm - sa).max() < 0.02
    far = np.abs(sa) > 0.3
    assert np.all(np.sign(sm[far]) == np.sign(sa[far]))
    assert np.einsum("ij,ij->i", gm[far], ga[far]).min() > 0.97


# ---- mesh internals -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mesh", list(MESHES))
def test_bvh_closest_point_equals_brute_force(mesh):
    V, F = MESHES[mesh]()
    assert W.mesh_volume(V, F) > 0, "generator must produce outward-oriented closed meshes"
    sh = O.Shape.mesh(V, F)
    p = np.random.default_rng(1).uniform(-4, 6, size=(400, 3))
    r = sh.mesh_query(p)
    assert np.array_equal(r["d2"], r["d2_brute"])
    assert np.allclose(np.sum((p - r["closest"]) ** 2, axis=1), r["d2"], rtol=1e-12)


@pytest.mark.parametrize("mesh", list(MESHES))
def test_exact_winding_number_is_integer_for_closed_meshes(mesh):
    V, F = MESHES[mesh]()
    sh = O.Shape.mesh(V, F)
    p = np.random.default_rng(4).uniform(-3, 5, size=(300, 3))
    r = sh.mesh_query(p, brute=False)
    w = r["w_exact"]
    assert np.abs(w - np.round(w)).max() < 1e-9 and set(np.round(w).astype(int)) <= {0, 1}
    assert np.abs(r["w_bh"] - w).max() < 0.05                        # Barnes–Hut dipole tree, beta = 2
    assert np.array_equal(r["w_bh"] > 0.5, w > 0.5)


def fwn_kat_points():
    return np.random.default_rng(7).uniform(-3, 5, size=(500, 3))


def test_winding_number_against_reference_fwn_header():
    """KAT from the one reference file that compiles here (igl/FastWindingNumberForSoups.h -> oracle/_ref; where that build is absent,
    its committed answers in tests/golden/reference_pins.npz)."""
    zr = None if O.ref_fwn_available() else np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_pins.npz"))
    for mesh in MESHES:
        V, F = MESHES[mesh]()
        sh = O.Shape.mesh(V, F)
        p = fwn_kat_points()
        w_ref = O.RefFwn(V, F, order=2).query(p, 2.0) if zr is None else zr[f"fwn_{mesh}_w"]
        w_ex = sh.mesh_query(p, brute=False)["w_exact"]
        d = np.sqrt(sh.mesh_query(p, winding=False)["d2"])
        keep = d > 1e-3
        # the reference's FP32 order-2 approximation carries ~1e-5..1e-3 error (SURVEY §0.4); same inside/outside call
        assert np.abs(w_ref - w_ex)[keep].max() < 5e-3
        assert np.array_equal(w_ref[keep] > 0.5, w_ex[keep] > 0.5)


# ---- MINCO ---------------------------------------------------------------------------------------------------------------
def test_minco_matches_dense_numpy_solve_and_adjoint_matches_fd():
    rng = np.random.default_rng(0)
    N = 5
    wp = W.random_walk_waypoints(N, [0, 0, 0], [40, 40, 30], seed=1)
    T = 2.5 * (1 + 0.3 * (rng.random(N) - 0.5))
    head = np.zeros((3, 3)); tail = np.zeros((3, 3))
    head[:, 0], tail[:, 0] = wp[0], wp[-1]
    head[:, 1], tail[:, 2] = [0.3, -0.2, 0.1], [0.05, 0.0, -0.1]
    co, energy, gc, gt = O.minco_forward(head, tail, wp[1:-1].T, T)
    ref = W.minco_s3(wp, T, head_va=[head[:, 1], head[:, 2]], tail_va=[tail[:, 1], tail[:, 2]])
    assert rel_l2(co, ref) < 1e-9
    # energy = integral of squared jerk (numerical quadrature)
    Cm = co.reshape(3, 6 * N)
    num = 0.0
    for i in range(N):
        s = np.linspace(0, T[i], 4001)
        c3, c4, c5 = Cm[:, 6 * i + 3], Cm[:, 6 * i + 4], Cm[:, 6 * i + 5]
        jerk = 6 * c3[:, None] + 24 * c4[:, None] * s + 60 * c5[:, None] * s ** 2
        num += np.trapezoid((jerk ** 2).sum(0), s)
    assert abs(num - energy) < 1e-5 * energy
    # total derivative of a random linear functional of the coefficients + energy wrt (waypoints, T)
    wC = rng.normal(size=co.size)

    def J(inP, T):
        c, e, _, _ = O.minco_forward(head, tail, inP, T)
        return wC @ c + e
    gP, gT = O.minco_backward(head, tail, wp[1:-1].T, T, wC + gc, gt)
    eps = 1e-6
    inP = wp[1:-1].T.copy()
    for (a, b) in [(0, 0), (2, 1), (1, 3)]:
        ip, im = inP.copy(), inP.copy()
        ip[a, b] += eps; im[a, b] -= eps
        assert abs((J(ip, T) - J(im, T)) / (2 * eps) - gP[a, b]) <= 1e-5 * abs(gP[a, b]) + 1e-5
    for i in range(N):
        Tp, Tm = T.copy(), T.copy()
        Tp[i] += eps; Tm[i] -= eps
        assert abs((J(inP, Tp) - J(inP, Tm)) / (2 * eps) - gT[i]) <= 1e-5 * abs(gT[i]) + 1e-5


# ---- swept volume ---------------------------------------------------------------------------------------------------------
def _sv_case(N=4, seed=3):
    cfg, occ, T, Cc, wp = small_case(N=N, K=16, seed=seed, noise=0.05)
    pts = W.gather_obstacle_points(occ, BMIN, 1.0, wp, cfg.kernel_size * cfg.occupancy_resolution / 3.0)
    return cfg, occ, T, Cc, wp, pts


def test_swept_sdf_is_the_min_over_time_of_the_pose_sdf():
    cfg, occ, T, Cc, wp, pts = _sv_case()
    assert len(pts) > 50
    sh = O.Shape.named("Ball")
    r = O.eval_swept(ocfg(cfg), sh, T, Cc, pts[:80])
    assert r["nsdf"] > 0
    tt = np.linspace(0, T.sum(), 4001)
    xs = W.traj_eval(T, Cc, tt)
    for k in range(80):
        dense = np.linalg.norm(pts[k] - xs, axis=1).min() - 1.0      # ball SDF is rotation invariant
        if r["sdf"][k] < 9.99:
            assert abs(r["sdf"][k] - dense) < 2e-3, (k, r["sdf"][k], dense)
        else:
            assert dense > 2 * cfg.safety_hor + 0.1 - 1e-6           # never came within safty_hor_inf (swm:383)


def test_swept_tail_gradient_matches_finite_differences():
    cfg, occ, T, Cc, wp, pts = _sv_case(seed=5)
    sh = O.Shape.named("Ball")
    oc = ocfg(cfg)
    r = O.eval_swept(oc, sh, T, Cc, pts)
    assert r["cost"] > 0
    rng = np.random.default_rng(0)
    e = 1e-5
    ok = 0
    for _ in range(6):
        dC = rng.normal(size=Cc.size)
        cp = O.eval_swept(oc, sh, T, Cc + e * dC, pts)["cost"]
        cm = O.eval_swept(oc, sh, T, Cc - e * dC, pts)["cost"]
        num, ana = (cp - cm) / (2 * e), r["gradC"] @ dC
        if abs(num - ana) <= 2e-3 * abs(ana) + 1e-2:   # limited by the 1-D minimiser's tolerance (SURVEY §9)
            ok += 1
    assert ok >= 5


def test_swept_given_tail_reproduces_search_result():
    cfg, occ, T, Cc, wp, pts = _sv_case(seed=2)
    sh = O.Shape.named("Torus")
    oc = ocfg(cfg)
    a = O.eval_swept(oc, sh, T, Cc, pts)
    b = O.eval_swept(oc, sh, T, Cc, pts, given=(a["tstar"], a["sdf"], a["grel"]))
    assert a["cost"] == b["cost"] and np.array_equal(a["gradC"], b["gradC"]) and np.array_equal(a["gradT"], b["gradT"])
