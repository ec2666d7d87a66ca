"""Oracle pinned to REFERENCE-COMPILED code (kind "reference"), CPU only.

oracle/_ref/libref_flat.so is the reference's own utils/flatness.hpp (optimizated_forward :53-86 / :88-148, backwardthreadsafe
:230-406) compiled unmodified against an element-access-only Eigen stand-in (oracle/Makefile `ref`). The oracle's flatness map and its
HAND-DERIVED adjoint (oracle_math.hpp orc::Flat) must reproduce it to rounding; tests/golden/flat_reference.npz holds outputs of the
same reference build (made by tests/golden/make_reference_golden.py) so the pin also holds where oracle/_ref is absent. Every test here that
calls a reference-compiled library does so where oracle/_ref exists, and compares with that build's committed outputs elsewhere."""
import os
import numpy as np
import pytest
import isdf_b200 as I
import oracle_lib as O

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
N_RANDOM = 10000
FLAT_SAMPLE = np.sort(np.random.default_rng(1).choice(N_RANDOM, 512, replace=False))   # rows of flat_inputs(N_RANDOM) kept as golden data


def flat_inputs(n, seed=0):
    rng = np.random.default_rng(seed)
    scale = 10.0 ** rng.uniform(-2, 1.3, size=(n, 1))                 # speeds / accelerations from cm/s to ~20 m/s
    v, a, j = rng.normal(size=(n, 3)) * scale, rng.normal(size=(n, 3)) * scale * 1.5, rng.normal(size=(n, 3)) * scale * 3
    a[:, 2] = np.abs(a[:, 2]) * 0.3 - 2.0                             # keeps thrust away from the singular zu = -|zu| e_z
    pg, vg, og = rng.normal(size=(n, 3)), rng.normal(size=(n, 3)), rng.normal(size=(n, 3))
    qg = rng.normal(size=(n, 4))
    return v, a, j, pg, vg, qg, og


def relerr(x, ref):
    return np.max(np.abs(x - ref) / np.maximum(1.0, np.max(np.abs(ref), axis=-1, keepdims=True)))


def reference_pins():
    """outputs of the reference-compiled libraries and the reference's OBJ files (tests/golden/make_reference_golden.py)"""
    return np.load(os.path.join(G, "reference_pins.npz"))


def test_flatness_oracle_equals_reference_compiled_flatness_hpp():
    cfg = O.config_from(I.default_config_values())
    v, a, j, pg, vg, qg, og = flat_inputs(N_RANDOM)
    if O.ref_flat_available():
        ref = O.RefFlat(cfg)
        q_ref, o_ref = ref.forward(v, a, j)
        q_only = ref.forward_quat(v, a, j)
        b_ref = ref.backward(v, a, j, pg, vg, qg, og)
    else:
        z = reference_pins()
        v, a, j, pg, vg, qg, og = (x[FLAT_SAMPLE] for x in (v, a, j, pg, vg, qg, og))
        q_ref, o_ref, q_only, b_ref = z["flat_quat"], z["flat_omg"], z["flat_quat_only"], z["flat_back"]
    q, o = O.flat_forward_batch(cfg, v, a, j)
    assert np.array_equal(q_only, q_ref)
    assert relerr(q, q_ref) <= 1e-15 and relerr(o, o_ref) <= 1e-12
    b = O.flat_backward_batch(cfg, v, a, j, pg, vg, qg, og)
    assert relerr(b, b_ref) <= 1e-12, relerr(b, b_ref)
    assert np.array_equal(b[:, 0:3], pg)                               # pos_total_grad = pos_grad (flat:402-404)


def test_flatness_oracle_equals_committed_reference_outputs():
    z = np.load(os.path.join(G, "flat_reference.npz"))
    cfg = O.config_from(I.default_config_values())
    assert np.allclose(z["par"], [cfg.vehicle_mass, cfg.grav_acc, cfg.horiz_drag, cfg.vert_drag, cfg.paras_drag, cfg.speed_eps])
    q, o = O.flat_forward_batch(cfg, z["v"], z["a"], z["j"])
    b = O.flat_backward_batch(cfg, z["v"], z["a"], z["j"], z["pg"], z["vg"], z["qg"], z["og"])
    assert relerr(q, z["quat"]) <= 1e-15 and relerr(o, z["omg"]) <= 1e-12 and relerr(b, z["back"]) <= 1e-12


# ---- the robot meshes the reference ships (src/plan_manager/shapes/*.obj), committed as INPUT fixtures with reference-computed winding numbers
def ref_mesh_cases():
    z = np.load(os.path.join(G, "ref_meshes.npz"))
    return z, [str(n) for n in z["names"]]


@pytest.mark.parametrize("name", ["Lthick", "RoundedCone", "mybox", "drone", "kuang", "box"])
def test_reference_meshes_oracle_sign_and_distance(name):
    """oracle on the reference's own robot meshes: inside/outside == the reference-compiled FWN's (rounded), exact winding within the FWN's
    approximation error, BVH distance == brute force; and the reference-faithful mode s = 1 - 2 w_FWN differs from ±1 by ~1e-3."""
    z, _ = ref_mesh_cases()
    V, F, pp, q, w_ref = z[name + "_V"], z[name + "_F"], z[name + "_pp"], z[name + "_q"], z[name + "_w"]
    sh = O.Shape.mesh(V, F, pp)
    r = sh.mesh_query(q)
    assert np.array_equal(r["d2"], r["d2_brute"])
    keep = np.sqrt(r["d2"]) > 1e-3
    assert np.abs(r["w_exact"] - np.round(r["w_exact"])).max() < 1e-9          # closed, consistently oriented (what the product requires)
    assert np.abs(w_ref - r["w_exact"])[keep].max() < 5e-3
    sdf, _ = sh.query(q)
    assert np.array_equal(sdf[keep] < 0, w_ref[keep] > 0.5)
    if O.ref_fwn_available():
        sdf_ref, g_ref = O.Shape.mesh(V, F, pp, wn_mode=O.WN_REF).query(q)
    else:
        zr = reference_pins()
        sdf_ref, g_ref = zr[f"mesh_{name}_sdf_fwn"], zr[f"mesh_{name}_grad_fwn"]
    assert np.allclose(sdf_ref, (1 - 2 * w_ref) * np.sqrt(r["d2"]), rtol=1e-12, atol=1e-15)   # WN_REF mode = Shape.cpp:110-113 with the fixture's w
    dev = np.abs(sdf_ref - sdf)[keep] / np.abs(sdf)[keep]
    assert 1e-7 < dev.max() < 1e-2                                            # the FP32 order-2 tree's error reaches the SDF VALUE ...
    _, g = sh.query(q)
    assert np.abs(g_ref - g)[keep].max() < 1e-12                               # ... but not the (normalised) gradient


def test_obj_reader_matches_fixture_on_reference_files(tmp_path):
    """host/isdf_obj.hpp (read_triangle_mesh counterpart, Shape.cpp:36) on the reference's OBJ files (committed byte for byte)"""
    import host_lib as H
    zr = reference_pins()
    z, names = ref_mesh_cases()
    for name in names:
        (tmp_path / (name + ".obj")).write_bytes(zr["obj_" + name].tobytes())
        V, F = H.read_obj(str(tmp_path / (name + ".obj")))
        assert np.array_equal(V, z[name + "_V"]) and np.array_equal(F, z[name + "_F"])
    # independent numpy parse of one file
    rows = [ln.split() for ln in open(tmp_path / "RoundedCone.obj") if ln[:2] in ("v ", "f ")]
    Vn = np.array([[float(x) for x in r[1:4]] for r in rows if r[0] == "v"])
    Fn = np.array([[int(x.split("/")[0]) - 1 for x in r[1:4]] for r in rows if r[0] == "f"], dtype=np.int32)
    assert np.array_equal(Vn, z["RoundedCone_V"]) and np.array_equal(Fn, z["RoundedCone_F"])


def test_obj_reader_forms(tmp_path):
    """index forms i, i/t, i/t/n, i//n, negative (relative) indices, polygon fans, comments"""
    import host_lib as H
    p = tmp_path / "t.obj"
    p.write_text("# c\nv 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0 1.0\nvn 0 0 1\nvt 0 0\nf 1/1/1 2/1/1 3/1/1 4/1/1\nv 0 0 1\nf -1 1//1 2\nf 1/1 3/1 5/1\n")
    V, F = H.read_obj(str(p))
    assert V.shape == (5, 3) and np.array_equal(F, [[0, 1, 2], [0, 2, 3], [4, 0, 1], [0, 2, 4]])


def _lbfgs_problems():
    def rosen(x):
        f = np.sum(100.0 * (x[1:] - x[:-1] ** 2) ** 2 + (1 - x[:-1]) ** 2)
        g = np.zeros_like(x)
        g[:-1] = -400 * x[:-1] * (x[1:] - x[:-1] ** 2) - 2 * (1 - x[:-1])
        g[1:] += 200 * (x[1:] - x[:-1] ** 2)
        return f, g
    A = np.diag([1.0, 10.0, 100.0, 3.0, 0.25])

    def quad(x):
        return 0.5 * x @ A @ x, A @ x

    def hinge(x):       # smoothed-L1 like kink (the planner's penalty shape): piecewise cubic / linear, long line searches
        f, g = 0.0, np.zeros_like(x)
        for i, v in enumerate(x):
            a = abs(v - 0.3 * i)
            if a > 0.1:
                f += a - 0.05; g[i] = np.sign(v - 0.3 * i)
            else:
                f += (0.2 - a) * a ** 3 / (2 * 0.1 ** 3) * 10; g[i] = np.sign(v - 0.3 * i) * (0.6 * a ** 2 - 4 * a ** 3) / (2 * 0.1 ** 3) * 10
        return f + 0.05 * x @ x, g + 0.1 * x

    def flat_then_nan(x):   # a callback that turns NaN away from the start: the drivers must fail the same way
        if np.linalg.norm(x) > 3.0:
            return float("nan"), x
        return float(np.sum(np.cos(x))), -np.sin(x)
    rng = np.random.default_rng(4)
    return [("rosenbrock-6", rosen, np.array([-1.2, 1.0, -0.5, 0.8, 1.5, -0.3]), dict(mem_size=16, past=10, delta=1e-9, g_epsilon=0.0, max_iterations=300)),
            ("rosenbrock-2 gtol", rosen, np.array([-1.2, 1.0]), dict(mem_size=8, past=0, delta=1e-6, g_epsilon=1e-8, max_iterations=2000)),
            ("quadratic", quad, rng.normal(size=5), dict(mem_size=4, past=3, delta=1e-12, g_epsilon=1e-12, max_iterations=200)),
            ("hinge", hinge, rng.normal(size=7) * 2, dict(mem_size=16, past=10, delta=1e-6, g_epsilon=0.0, max_iterations=150)),
            ("iteration cap", rosen, np.array([-1.2, 1.0, 1.0, 1.0]), dict(mem_size=8, past=3, delta=1e-14, g_epsilon=0.0, max_iterations=7)),
            ("nan away from the start", flat_then_nan, np.array([0.5, -0.4, 0.3]), dict(mem_size=8, past=3, delta=1e-6, g_epsilon=1e-9, max_iterations=50)),
            ("stationary start", quad, np.zeros(5), dict(mem_size=8, past=3, delta=1e-6, g_epsilon=1e-5, max_iterations=50))]


def test_lbfgs_host_driver_equals_reference_compiled_lbfgs_hpp():
    """The product's sequential L-BFGS driver (host/isdf_lbfgs.hpp; the lock-step host and device drivers are tested bit-identical to it)
    against the reference's own utils/lbfgs.hpp compiled unmodified (oracle/_ref/libref_lbfgs.so, eager Eigen stand-in with left-to-right
    reductions): every point handed to the callback, in order, the solution, the value, the return code and the evaluation count are
    IDENTICAL — Lewis-Overton line search, cautious update, the fork's direction-reset patches (one extra evaluation), stop tests."""
    import host_lib as H
    ref = O.RefLbfgs() if os.path.exists(O.REF_LBFGS) else None
    zl = None if ref else np.load(os.path.join(G, "lbfgs_reference.npz"))
    for k, (name, fun, x0, kw) in enumerate(_lbfgs_problems()):
        if ref is not None:
            a = ref.minimize(fun, x0, **kw)
        else:
            a = dict(ret=int(zl[f"p{k}_ret"]), evaluations=int(zl[f"p{k}_evals"]), trace=list(zl[f"p{k}_trace"]), x=zl[f"p{k}_x"], f=float(zl[f"p{k}_f"]))
        b = H.lbfgs_minimize(fun, x0, **kw)
        assert a["ret"] == b["ret"], f"{name}: return code {a['ret']} (reference) vs {b['ret']}"
        assert a["evaluations"] == b["evaluations"] == len(b["trace"]), f"{name}: evaluations {a['evaluations']} vs {b['evaluations']}"
        for k, (p, q) in enumerate(zip(a["trace"], b["trace"])):
            assert np.array_equal(p, q), f"{name}: evaluation {k} at different points (max diff {np.abs(p - q).max():.3e})"
        assert np.array_equal(a["x"], b["x"]) and (a["f"] == b["f"] or (np.isnan(a["f"]) and np.isnan(b["f"]))), name


def _minco_cases():
    rng = np.random.default_rng(21)
    out = []
    for N in (2, 3, 8, 64):
        head = np.stack([rng.normal(size=3) * 5, rng.normal(size=3), rng.normal(size=3) * 0.3], axis=1)
        tail = np.stack([rng.normal(size=3) * 5 + 20, rng.normal(size=3), rng.normal(size=3) * 0.3], axis=1)
        inPs = np.cumsum(rng.normal(size=(3, N - 1)) * 2 + 1.0, axis=1)
        T = rng.uniform(0.4, 3.0, N)
        out.append((N, head, tail, inPs, T, rng.normal(size=18 * N), rng.normal(size=N)))
    return out


def test_minco_oracle_and_host_port_equal_reference_compiled_minco_hpp():
    """oracle_minco.hpp and host/isdf_minco.hpp against the reference's own utils/minco.hpp compiled unmodified (oracle/_ref/libref_minco.so, eager
    Eigen stand-in): banded LU + substitution (coefficients), energy and its partial gradients, the adjoint solve and propogateGrad. The ORACLE
    is bit-identical wherever no reduction is involved (coefficients, dE/dC, gradByPoints) and agrees to the last ulps where a sum's order is the
    stand-in's (energy, dE/dT, gradByTimes); the product's host port (device kernels bit-identical to it) agrees to 1e-12."""
    import host_lib as H
    ref = O.RefMinco() if os.path.exists(O.REF_MINCO) else None
    zm = None if ref else np.load(os.path.join(G, "minco_reference.npz"))
    for k, (N, head, tail, inPs, T, gC, gT) in enumerate(_minco_cases()):
        if ref is not None:
            rc, re, rgc, rgt = ref.forward(head, tail, inPs, T)
            rgp, rgto = ref.backward(head, tail, inPs, T, gC, gT)
        else:
            rc, re, rgc, rgt = zm[f"c{k}_coeffs"], float(zm[f"c{k}_energy"]), zm[f"c{k}_gdC"], zm[f"c{k}_gdT"]
            rgp, rgto = zm[f"c{k}_gradP"], zm[f"c{k}_gradT"]
        # the oracle follows the reference's operation order: identical bits wherever no reduction is involved
        c, e, gc, gt = O.minco_forward(head, tail, inPs, T)
        assert np.array_equal(c, rc), f"oracle N={N}: coefficients differ from the reference-compiled solve by {np.abs(c - rc).max():.3e}"
        assert np.array_equal(gc, rgc), f"oracle N={N}: dE/dC"
        assert abs(e - re) <= 4e-16 * abs(re) * 6 * N and np.allclose(gt, rgt, rtol=1e-14, atol=0), f"oracle N={N}: energy / dE/dT"
        gp, gto = O.minco_backward(head, tail, inPs, T, gC, gT)
        assert np.array_equal(np.asarray(gp).reshape(-1), np.asarray(rgp).reshape(-1)), f"oracle N={N}: gradByPoints (adjoint solve) differs by {np.abs(np.asarray(gp) - rgp).max():.3e}"
        assert np.allclose(gto, rgto, rtol=1e-13, atol=1e-13 * np.abs(rgto).max()), f"oracle N={N}: gradByTimes"
        # the product's host MINCO (the device kernels are bit-identical to it) keeps the band factored with reciprocal pivots: same
        # solution to rounding
        c, e, gc, gt = H.minco_forward(head, tail, inPs, T)
        scale = np.abs(rc).max()
        assert np.abs(c - rc).max() <= 1e-12 * scale, f"host N={N}: coefficients {np.abs(c - rc).max():.3e}"
        assert np.allclose(gc, rgc, rtol=0, atol=1e-11 * np.abs(rgc).max()) and abs(e - re) <= 1e-12 * abs(re) and np.allclose(gt, rgt, rtol=0, atol=1e-11 * np.abs(rgt).max())
        gp, gto = H.minco_backward(head, tail, inPs, T, gC, gT)
        assert np.allclose(np.asarray(gp).reshape(-1), np.asarray(rgp).reshape(-1), rtol=0, atol=1e-11 * np.abs(rgp).max()), f"host N={N}: gradByPoints"
        assert np.allclose(gto, rgto, rtol=0, atol=1e-11 * np.abs(rgto).max()), f"host N={N}: gradByTimes"
    # getTrajectory: the 3 x 6 coefficient matrices are the coefficient block transposed, highest power first
    N, head, tail, inPs, T, _, _ = _minco_cases()[2]
    if ref is not None:
        dur, cm = ref.trajectory(head, tail, inPs, T)
        co = ref.forward(head, tail, inPs, T)[0].reshape(3, 6 * N)
    else:
        zr = reference_pins()
        dur, cm = zr["traj_durations"], zr["traj_coeffs"]
        co = zm["c2_coeffs"].reshape(3, 6 * N)
    assert np.array_equal(dur, T)
    for i in range(N):
        assert np.array_equal(cm[i], co[:, 6 * i:6 * i + 6][:, ::-1])


def test_minco_and_lbfgs_equal_committed_reference_outputs():
    """the same two pins against the COMMITTED outputs of the reference-compiled libraries (tests/golden/make_reference_golden.py), so that they hold
    where /root/reference — and with it oracle/_ref — is absent"""
    import host_lib as H
    zm = np.load(os.path.join(G, "minco_reference.npz"))
    for k, (N, head, tail, inPs, T, gC, gT) in enumerate(_minco_cases()):
        c, e, gc, gt = O.minco_forward(head, tail, inPs, T)
        gp, gto = O.minco_backward(head, tail, inPs, T, gC, gT)
        assert np.array_equal(c, zm[f"c{k}_coeffs"]) and np.array_equal(gc, zm[f"c{k}_gdC"]) and np.array_equal(np.asarray(gp), zm[f"c{k}_gradP"])
        assert abs(e - float(zm[f"c{k}_energy"])) <= 1e-14 * abs(e) and np.allclose(gt, zm[f"c{k}_gdT"], rtol=1e-14, atol=0)
        assert np.allclose(gto, zm[f"c{k}_gradT"], rtol=0, atol=1e-13 * np.abs(gto).max())
        ev, piece, tloc, total = O.traj_eval(T, c, zm[f"c{k}_times"])
        assert np.array_equal(ev, zm[f"c{k}_pvaj"]) and np.array_equal(piece, zm[f"c{k}_piece"]) and np.array_equal(tloc, zm[f"c{k}_tloc"]) and total == float(zm[f"c{k}_total"])
    zl = np.load(os.path.join(G, "lbfgs_reference.npz"))
    for k, (name, fun, x0, kw) in enumerate(_lbfgs_problems()):
        b = H.lbfgs_minimize(fun, x0, **kw)
        assert b["ret"] == int(zl[f"p{k}_ret"]) and b["evaluations"] == int(zl[f"p{k}_evals"]), name
        assert np.array_equal(np.array(b["trace"]), zl[f"p{k}_trace"]) and np.array_equal(b["x"], zl[f"p{k}_x"]), name
        f_ref = float(zl[f"p{k}_f"])
        assert b["f"] == f_ref or (np.isnan(b["f"]) and np.isnan(f_ref)), name


def _traj_times(T, rng):
    """absolute times that exercise locatePieceIdx: inside pieces, EXACTLY on junctions (strict '>' keeps a junction in the earlier piece), the
    sums as the bench's sampling produces them, before 0 and past the end (clamped into the last piece, quirk Q12)"""
    cs = np.cumsum(T)
    return np.concatenate([rng.uniform(0, cs[-1], 200), cs, cs - 1e-13, cs + 1e-13, np.cumsum(np.full(40, cs[-1] / 40)), [0.0, -0.3, cs[-1] + 0.7, cs[-1] * 2]])


def test_trajectory_evaluation_equals_reference_compiled_trajectory_hpp():
    """orc::Traj (locatePieceIdx's sequential subtraction, Piece::getPos_Vel_Acc_Jerk's running powers) against the reference's own
    utils/trajectory.hpp compiled unmodified and fed by the reference's own MINCO getTrajectory: piece index, local time, position, velocity,
    acceleration and jerk IDENTICAL at every time, incl. junctions and out-of-range times. The device's traj_locate / traj_pvaj
    (csrc/isdf_swept.cuh) follow orc::Traj operation by operation and are compared with it by the GPU parity tests."""
    ref = O.RefMinco() if os.path.exists(O.REF_MINCO) else None
    zm = None if ref else np.load(os.path.join(G, "minco_reference.npz"))
    rng = np.random.default_rng(8)
    for k, (N, head, tail, inPs, T, _, _) in enumerate(_minco_cases()):
        if ref is not None:
            times = _traj_times(T, rng)
            r_out, r_piece, r_tloc, r_total = ref.traj_eval(head, tail, inPs, T, times)
        else:   # the committed outputs were taken at times drawn the same way from another seed
            times = zm[f"c{k}_times"]
            r_out, r_piece, r_tloc, r_total = zm[f"c{k}_pvaj"], zm[f"c{k}_piece"], zm[f"c{k}_tloc"], float(zm[f"c{k}_total"])
        coeffs = O.minco_forward(head, tail, inPs, T)[0]
        o_out, o_piece, o_tloc, o_total = O.traj_eval(T, coeffs, times)
        assert o_total == r_total and np.array_equal(o_piece, r_piece) and np.array_equal(o_tloc, r_tloc), f"N={N}: piece search"
        assert np.array_equal(o_out, r_out), f"N={N}: pos/vel/acc/jerk differ by {np.abs(o_out - r_out).max():.3e}"


def _grid_cases():
    rng = np.random.default_rng(12)
    out = []
    for dims, bmin, res in (((20, 16, 12), np.array([0.0, 0.0, 0.0]), 1.0), ((24, 10, 31), np.array([-3.0, 2.0, -7.5]), 0.5), ((9, 9, 9), np.array([1.0, -1.0, 0.25]), 0.25)):
        dims = np.array(dims)
        bmax = bmin + dims * res
        pts = np.concatenate([bmin + rng.random((400, 3)) * (bmax - bmin),                       # inside
                              bmin - 2 + rng.random((300, 3)) * (bmax - bmin + 4),               # in and around
                              np.array([bmin, bmax, bmin + (bmax - bmin) * [1, 0, 0], bmin + (bmax - bmin) * [0, 1, 1], (bmin + bmax) / 2]),   # corners / faces
                              bmin + np.floor(rng.random((100, 3)) * dims) * res])               # exactly on cell boundaries
        occ = (rng.random(tuple(dims)) < 0.2).astype(np.uint8)
        boxes = [(bmin - 1 + rng.random(3) * (bmax - bmin + 2), float(rng.choice([0.4, 1.3, 2.5, 6.5]) * res)) for _ in range(25)]
        out.append((dims, bmin, res, pts, occ, boxes))
    return out


def test_grid_oracle_equals_committed_reference_outputs():
    z = np.load(os.path.join(G, "grid_reference.npz"))
    for k, (dims, bmin, res, pts, occ, boxes) in enumerate(_grid_cases()):
        oi, oc, om = O.grid_index(dims, bmin, res, pts)
        assert np.array_equal(oi, z[f"g{k}_idx"]) and np.array_equal(oc, z[f"g{k}_centre"]) and np.array_equal(om, z[f"g{k}_inmap"])
        for b, (centre, half) in enumerate(boxes):
            op, on = O.points_in_aabb(occ, bmin, res, centre, half)
            assert on == int(z[f"g{k}_b{b}_n"]) and np.array_equal(op, z[f"g{k}_b{b}_pts"])


def test_grid_oracle_equals_reference_compiled_gridmap3d():
    """orc::Grid against the reference's own map_manager/src/Gridmap3D.cpp compiled unmodified: getGridIndex (with its clamping quirk: the
    'iy < 0' and 'iz < 0' branches reset ix), getGridCubeCenter, isInMap — at points inside, on every face, outside on every side; and the AABB
    gather PCSmapManager::getPointsInAABB built on them (projInMap + index box + isIndexOccupied + cube centres): same voxels, same order, same bits."""
    ref = O.RefGrid() if os.path.exists(O.REF_GRID) else None
    z = None if ref else np.load(os.path.join(G, "grid_reference.npz"))
    for k, (dims, bmin, res, pts, occ, boxes) in enumerate(_grid_cases()):
        if ref is not None:
            ri, rc, rm = ref.index(dims, bmin, res, pts)
        else:
            ri, rc, rm = z[f"g{k}_idx"], z[f"g{k}_centre"], z[f"g{k}_inmap"]
        oi, oc, om = O.grid_index(dims, bmin, res, pts)
        assert np.array_equal(ri, oi) and np.array_equal(rc, oc) and np.array_equal(rm, om), f"grid {dims} res {res}"
        for b, (centre, half) in enumerate(boxes):
            if ref is not None:
                rp, rn = ref.points_in_aabb(occ, bmin, res, centre, half)
            else:
                rp, rn = z[f"g{k}_b{b}_pts"], int(z[f"g{k}_b{b}_n"])
            op, on = O.points_in_aabb(occ, bmin, res, centre, half)
            assert rn == on and np.array_equal(rp, op), f"AABB gather at {centre} half {half}: {rn} vs {on} voxels"
