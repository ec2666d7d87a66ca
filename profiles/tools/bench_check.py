#!/usr/bin/env python
"""Timing of the whole-body collision check (isdf_check_collision_device, csrc/isdf_check.cuh) on one GPU.
  * the BASELINE configs[2] trajectory (512^3 map, 5 % occupancy + 3 wall slabs, 64 pieces) at M = 256 check intervals per piece,
    H = safety_hor and H = 1 m, for the 3900-triangle exact-sign mesh robot and an analytic robot (RoundedCone);
  * a 1024-restart batch at configs[4] size (64 pieces x 256 intervals each, the same map; MINCO trajectories of bench.py's restart problems);
  * what the branch-and-bound removes: voxels in the body box vs SDF values computed vs mesh searches;
  * the per-sample warp time spread (clock64 cycles per sample, one warp per sample);
  * the oracle's CPU time on the configs[2] input (tests/collision_oracle.cpp, OpenMP over samples, core count stated).
CUDA events around each call, L2 flushed (512 MiB write) before every timed call. Card name and power limit are read in the same run.
usage: bench_check.py [out.json] [--reps R] [--no-oracle]"""
import json, os, subprocess, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "implicit-sdf-planner_b200", "py")); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch
import isdf_b200 as I, workloads as W

args = [a for a in sys.argv[1:] if not a.startswith("--")]
out_path = args[0] if args else None
reps = int(sys.argv[sys.argv.index("--reps") + 1]) if "--reps" in sys.argv else 10
dev = torch.device("cuda:0")
card = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=dev)
stream = torch.cuda.current_stream().cuda_stream
X, N0, M = 512, 64, 256
occ = W.random_map(X, X, X, p=0.05, seed=1, slabs=3)
cfg = I.default_config_values()
cfg.integral_intervs = M
cfg.flags = I.WITH_COLLISION
T, Cc, _ = W.make_trajectory(N0, [0, 0, 0], [X, X, X], seed=11, jitter=0.2)
V, F = W.rounded_cone_mesh()
ev = I.Evaluator(cfg)
ev.set_map_u8(occ, [0, 0, 0], 1.0)
result = {"card": card, "l2": "flushed (512 MiB write) before every timed call", "timing": "CUDA events around isdf_check_collision_device",
          "workload": f"configs[2]: {X}^3 map (p = 0.05, 3 slabs), {N0} pieces x {M} check intervals ({N0 * (M + 1)} samples)", "runs": []}


def timed(B, n_pieces, dT, dC, H, margin=0.0, n=reps):
    drep = torch.zeros(B * 96, dtype=torch.uint8, device=dev)
    for _ in range(2):
        ev.check_collision_device(B, n_pieces, dT.data_ptr(), dC.data_ptr(), M, margin, H, drep.data_ptr(), 0, stream)
    ts = []
    for _ in range(n):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ev.check_collision_device(B, n_pieces, dT.data_ptr(), dC.data_ptr(), M, margin, H, drep.data_ptr(), 0, stream)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    cnt, _ = ev.dbg_check_stats()
    reps_h = (I.ClearanceReport * B).from_buffer_copy(drep.cpu().numpy().tobytes())
    return dict(ms_median=float(np.median(ts)), ms_min=float(np.min(ts)), ms_max=float(np.max(ts)), calls=n, **cnt,
                collides=int(sum(r.collides for r in reps_h)), min_clearance_first=reps_h[0].min_clearance)


def spread(B, n_pieces, T_h, C_h, H):
    """one untimed call with per-sample cycle recording"""
    ev.dbg_enable(True)
    ev.check_collision(T_h, C_h, M, 0.0, H, B=B)
    _, cyc = ev.dbg_check_stats(B * n_pieces * (M + 1))
    ev.dbg_enable(False)
    q = np.percentile(cyc, [50, 90, 99, 100])
    return dict(cycles_p50=float(q[0]), cycles_p90=float(q[1]), cycles_p99=float(q[2]), cycles_max=float(q[3]), cycles_mean=float(cyc.mean()))


dT, dC = torch.tensor(T, device=dev), torch.tensor(Cc, device=dev)
for robot in ("mesh3900", "RoundedCone"):
    if robot == "mesh3900":
        ev.set_shape_mesh(V, F, [0, 0, 0, 120, 0, 0], I.MESH_SIGN_EXACT)
    else:
        ev.set_shape_named(robot)
    for H in (cfg.safety_hor, 1.0):
        r = dict(robot=robot, H=H, B=1, **timed(1, N0, dT, dC, H), **spread(1, N0, T, Cc, H))
        print(json.dumps(r), flush=True)
        result["runs"].append(r)

# configs[4] size: 1024 restarts, trajectories from MINCO through bench.py's restart problems (callback on the device)
sys.path.insert(0, ROOT)
from bench import batch_problems
B = 1024
xs, heads, tails = batch_problems(B, N0, X)
h3, t3 = heads.reshape(B, 3, 3).transpose(0, 2, 1), tails.reshape(B, 3, 3).transpose(0, 2, 1)   # column-major 3x3 -> row-major
ev.set_shape_mesh(V, F, [0, 0, 0, 120, 0, 0], I.MESH_SIGN_EXACT)
ev.callback_batch(h3, t3, 20.0, xs)
Tb, Cb, _ = ev.batch_trajectories(B, N0)
dTb, dCb = torch.tensor(Tb, device=dev), torch.tensor(Cb, device=dev)
for H in (cfg.safety_hor,):
    r = dict(robot="mesh3900", H=H, B=B, **timed(B, N0, dTb, dCb, H, n=max(3, reps // 3)), **spread(B, N0, Tb, Cb, H))
    print(json.dumps(r), flush=True)
    result["runs"].append(r)

if "--no-oracle" not in sys.argv:
    import oracle_lib as O, collision_oracle as CO
    osh = O.Shape.mesh(V, F, [0, 0, 0, 120, 0, 0], wn_mode=O.WN_BH)
    CO.lib()
    t0 = time.perf_counter()
    rep, _ = CO.check_collision(cfg, occ, [0, 0, 0], 1.0, osh, T, Cc, M, 0.0, cfg.safety_hor)
    dt = time.perf_counter() - t0
    result["oracle_cpu"] = dict(robot="mesh3900", H=cfg.safety_hor, seconds=dt, threads=os.cpu_count(),
                                note="OpenMP over samples; the mesh sign from the oracle's Barnes-Hut winding number (thresholded)",
                                min_clearance=rep[0]["min_clearance"])
    print(json.dumps(result["oracle_cpu"]), flush=True)
ev.close()
if out_path:
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    json.dump(result, open(out_path, "w"), indent=1)
