"""Golden vectors computed by REFERENCE-COMPILED code (oracle/_ref/*.so built from /root/reference by `make -C oracle ref`).
Run in the build container (where /root/reference exists):  python tests/golden/make_reference_golden.py
  flat_reference.npz — inputs and outputs of the reference's utils/flatness.hpp (optimizated_forward, backwardthreadsafe);
  ref_meshes.npz     — the robot meshes the reference ships and loads down its mesh Generalshape path (src/plan_manager/shapes/
                       {Lthick,drone,kuang,box,RoundedCone,mybox}.obj; INPUT data, read with the product's OBJ reader), the
                       poly_params of the config that names them, seeded query points, and the winding numbers the
                       reference-compiled igl/FastWindingNumberForSoups.h returns for them (order 2, accuracy scale 2.0: Shape.cpp:86,110);
  minco_reference.npz — outputs of the reference's utils/minco.hpp (MINCO_S3NU forward, energy gradients, propogateGrad) on seeded problems, and
                        of its utils/trajectory.hpp (getPos_Vel_Acc_Jerk, locatePieceIdx, getTotalDuration) on the resulting trajectories;
  lbfgs_reference.npz — what the reference's utils/lbfgs.hpp does on seeded problems: every evaluated point, solution, value, return code;
  grid_reference.npz  — the reference's map_manager/src/Gridmap3D.cpp: grid indices, cube centres, in-map flags and AABB gathers on seeded grids;
  reference_pins.npz  — what the tests that call the reference-compiled libraries compare against, for where oracle/_ref is absent: the
                        reference's OBJ files as shipped (bytes), flatness.hpp on a fixed sample of the 10000 random inputs, FWN winding
                        numbers, the FWN-signed oracle (s = 1 - 2 w) on the robot meshes and on the sign-policy cases, getTrajectory."""
import os
import sys
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "implicit-sdf-planner_b200", "py"))
import isdf_b200 as I          # noqa: E402
import oracle_lib as O         # noqa: E402
from test_reference_pins import flat_inputs, _minco_cases, _lbfgs_problems, _traj_times, _grid_cases, N_RANDOM, FLAT_SAMPLE   # noqa: E402


REF_SHAPES = "/root/reference/src/plan_manager/shapes"
# mesh -> poly_params: config_L.yaml:8-10 (Lthick), config_CappedCone.yaml:8-10 (RoundedCone), config_box.yaml:8-11 (mybox); drone / kuang /
# box are named by no shipped config (sw_manager.hpp:255-275 sends any unknown name down the mesh path): CappedCone's parameters
MESHES = {"Lthick": [0, 0, 0, 0, 0, 0], "RoundedCone": [0, 0, 0, 120, 0, 0], "mybox": [0, 0, 0, 0, 0, 0],
          "drone": [0, 0, 0, 120, 0, 0], "kuang": [0, 0, 0, 120, 0, 0], "box": [0, 0, 0, 120, 0, 0]}


def ref_meshes():
    import host_lib as H
    import workloads as W
    out = {}
    for name, pp in MESHES.items():
        V, F = H.read_obj(os.path.join(REF_SHAPES, name + ".obj"))
        R, t = W.rotation_from_poly_params(pp)
        Vt = V @ R.T + t                                            # Shape.cpp:38-50
        lo, hi = Vt.min(0) - 1.0, Vt.max(0) + 1.0
        rng = np.random.default_rng(abs(hash(name)) % 1000 + 5 if False else sum(map(ord, name)))
        q = lo + (hi - lo) * rng.random((600, 3))
        w = O.RefFwn(Vt, F, order=2).query(q, 2.0)
        out[name + "_V"], out[name + "_F"], out[name + "_pp"], out[name + "_q"], out[name + "_w"] = V, F, np.array(pp, float), q, w
        print(name, V.shape, F.shape, "w range", w.min(), w.max())
    np.savez_compressed(os.path.join(HERE, "ref_meshes.npz"), names=np.array(list(MESHES)), **out)
    print("ref_meshes.npz written")


def reference_pins():
    from common import MESHES as TEST_MESHES
    from test_oracle_pins import fwn_kat_points
    from test_gpu_reference_pins import sign_policy_case
    out = {}
    for name in MESHES:
        out["obj_" + name] = np.frombuffer(open(os.path.join(REF_SHAPES, name + ".obj"), "rb").read(), dtype=np.uint8)
    cfg = O.config_from(I.default_config_values())
    ref = O.RefFlat(cfg)
    v, a, j, pg, vg, qg, og = (x[FLAT_SAMPLE] for x in flat_inputs(N_RANDOM))
    out["flat_quat"], out["flat_omg"] = ref.forward(v, a, j)
    out["flat_quat_only"] = ref.forward_quat(v, a, j)
    out["flat_back"] = ref.backward(v, a, j, pg, vg, qg, og)
    for name, gen in TEST_MESHES.items():
        V, F = gen()
        out[f"fwn_{name}_w"] = O.RefFwn(V, F, order=2).query(fwn_kat_points(), 2.0)
    z = np.load(os.path.join(HERE, "ref_meshes.npz"))
    for name in MESHES:
        V, F, pp, q = z[name + "_V"], z[name + "_F"], z[name + "_pp"], z[name + "_q"]
        out[f"mesh_{name}_sdf_fwn"], out[f"mesh_{name}_grad_fwn"] = O.Shape.mesh(V, F, pp, wn_mode=O.WN_REF).query(q)
    for name in ("Lthick", "RoundedCone"):
        cfg_s, occ, T, Cc, V, F, pp = sign_policy_case(name)
        out[f"sign_{name}_cost"], out[f"sign_{name}_gradC"], out[f"sign_{name}_gradT"], _ = O.eval_discrete(
            O.config_from(cfg_s), occ, [0, 0, 0], 1.0, O.Shape.mesh(V, F, pp, wn_mode=O.WN_REF), T, Cc)
    N, head, tail, inPs, T, _, _ = _minco_cases()[2]
    out["traj_durations"], out["traj_coeffs"] = O.RefMinco().trajectory(head, tail, inPs, T)
    np.savez_compressed(os.path.join(HERE, "reference_pins.npz"), **out)
    print("reference_pins.npz written")


def main():
    O.build()
    ref_meshes()
    cfg = O.config_from(I.default_config_values())
    ref = O.RefFlat(cfg)
    v, a, j, pg, vg, qg, og = flat_inputs(256, seed=123)
    q, o = ref.forward(v, a, j)
    b = ref.backward(v, a, j, pg, vg, qg, og)
    np.savez(os.path.join(HERE, "flat_reference.npz"), par=ref.par, v=v, a=a, j=j, pg=pg, vg=vg, qg=qg, og=og, quat=q, omg=o, back=b)
    print("flat_reference.npz written")
    rm = O.RefMinco()
    out = {}
    for k, (N, head, tail, inPs, T, gC, gT) in enumerate(_minco_cases()):
        co, e, gc, gt = rm.forward(head, tail, inPs, T)
        gp, gto = rm.backward(head, tail, inPs, T, gC, gT)
        out.update({f"c{k}_coeffs": co, f"c{k}_energy": np.array(e), f"c{k}_gdC": gc, f"c{k}_gdT": gt, f"c{k}_gradP": np.asarray(gp), f"c{k}_gradT": gto})
        times = _traj_times(T, np.random.default_rng(100 + k))
        ev, piece, tloc, total = rm.traj_eval(head, tail, inPs, T, times)
        out.update({f"c{k}_times": times, f"c{k}_pvaj": ev, f"c{k}_piece": piece, f"c{k}_tloc": tloc, f"c{k}_total": np.array(total)})
    np.savez_compressed(os.path.join(HERE, "minco_reference.npz"), ncases=np.array(len(_minco_cases())), **out)
    print("minco_reference.npz written")
    rl = O.RefLbfgs()
    out = {}
    for k, (name, fun, x0, kw) in enumerate(_lbfgs_problems()):
        r = rl.minimize(fun, x0, **kw)
        out.update({f"p{k}_trace": np.array(r["trace"]), f"p{k}_x": r["x"], f"p{k}_f": np.array(r["f"]), f"p{k}_ret": np.array(r["ret"]), f"p{k}_evals": np.array(r["evaluations"])})
        print(name, r["ret"], r["evaluations"])
    np.savez_compressed(os.path.join(HERE, "lbfgs_reference.npz"), nproblems=np.array(len(_lbfgs_problems())), **out)
    print("lbfgs_reference.npz written")
    rg = O.RefGrid()
    out = {}
    for k, (dims, bmin, res, pts, occ, boxes) in enumerate(_grid_cases()):
        idx, ctr, inm = rg.index(dims, bmin, res, pts)
        out.update({f"g{k}_idx": idx, f"g{k}_centre": ctr, f"g{k}_inmap": inm})
        for b, (centre, half) in enumerate(boxes):
            p_, n_ = rg.points_in_aabb(occ, bmin, res, centre, half)
            out.update({f"g{k}_b{b}_pts": p_, f"g{k}_b{b}_n": np.array(n_)})
    np.savez_compressed(os.path.join(HERE, "grid_reference.npz"), **out)
    print("grid_reference.npz written")
    reference_pins()


if __name__ == "__main__":
    main()
