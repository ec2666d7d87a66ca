#!/usr/bin/env python
"""bench.py — collision cost+gradient evaluations/s of the discrete hot path on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, through libisdf_b200.so)
  python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU algorithm (OpenMP structure) on host cores

Workload (N=1 and every N: strong scaling, total work fixed): BASELINE.json configs[2] — the configuration the
north_star target is quoted on: 512^3 random voxel map (Bernoulli 5 % + wall slabs), 64-piece MINCO trajectory,
256 samples/piece (S = 16448 pose samples), robot = 3900-triangle closed mesh (rounded cone, the mesh-SDF path).
One "step" = one cost + gradC (6N x 3) + gradT (N) evaluation of the collision term over the whole trajectory.
Every step evaluates a DIFFERENT iterate (the trajectory moved by a small optimiser-like step), so the longest-first work-item
schedule each step uses was learned from another trajectory — as in a real optimiser run; the same-iterate and cold (first
evaluation) figures are reported beside it in `extra`.
At N > 1 every rank evaluates the pose samples s % N == rank and the 19N+1 doubles are summed over NVLink peer memory.
Other BASELINE configs as strong-scaling workloads of their own: --workload swept (configs[3]), --workload batch1024 (configs[4]).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "implicit-sdf-planner_b200", "py"))

METRIC = "collision_cost_grad_evals_per_s"
UNIT = "evals/s"
WORKLOAD = dict(map_dim=512, occupancy=0.05, pieces=64, samples_per_piece=256, kernel_size=13, mesh="rounded_cone_3900tri",
                poly_params=[0.0, 0.0, 0.0, 120.0, 0.0, 0.0])


# ---- distributed helpers (also exercised by tests/test_multi_rank_gloo.py on CPU/gloo) ------------------------------
def dist_ready():
    import torch.distributed as dist
    return dist.is_available() and dist.is_initialized()


def allreduce_partials(t):
    """sum the per-rank partial [cost | gradC | gradT] vectors in place (NCCL over NVLink on GPU tensors, gloo on CPU)."""
    if dist_ready():
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t


def max_over_ranks(x):
    if not dist_ready():
        return float(x)
    import torch
    import torch.distributed as dist
    dev = "cuda" if dist.get_backend() == "nccl" else "cpu"
    t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier():
    if dist_ready():
        import torch.distributed as dist
        dist.barrier()


_release = {}


def release_together():
    """N > 1: enqueue a tiny all-reduce on the current stream right before the timed step. The host has already passed a barrier; this makes the
    DEVICES leave the collective within a few microseconds of each other, so the timed region (CUDA events, max over ranks) measures the step
    and not the scatter of eight python processes' launch times (30-50 us, as large as the sharded step itself)."""
    if dist_ready():
        import torch
        import torch.distributed as dist
        if dist.get_backend() == "nccl":
            if "t" not in _release:
                _release["t"] = torch.zeros(1, device="cuda")
            dist.all_reduce(_release["t"])


# ---- workload ------------------------------------------------------------------------------------------------------------
def make_workload(small=False):
    import isdf_b200 as I
    import workloads as W
    w = dict(WORKLOAD)
    if small:
        w.update(map_dim=128, pieces=8, samples_per_piece=32)
    X = w["map_dim"]
    occ = W.random_map(X, X, X, p=w["occupancy"], seed=1, slabs=3)
    cfg = I.default_config_values()
    cfg.integral_intervs = w["samples_per_piece"]
    cfg.kernel_size = w["kernel_size"]
    cfg.flags = I.WITH_COLLISION | I.WITH_DYNAMICS
    T, Cc, wp = W.make_trajectory(w["pieces"], [0, 0, 0], [X, X, X], seed=11, jitter=0.2)
    V, F = W.rounded_cone_mesh()
    return w, cfg, occ, T, Cc, V, F


def algorithmic_bytes(w):
    """SURVEY.md §8(d): S*W^3 bytes of occupancy (1 B/voxel, each sample's window counted once) + coeff/T read + grads written."""
    N, K, Wk = w["pieces"], w["samples_per_piece"], w["kernel_size"]
    S = N * (K + 1)
    return S * Wk ** 3 + 8 * 19 * N + 8 * (19 * N + 1)


def make_iterates(w, T, Cc, n, seed=5, step_m=0.01):
    """n distinct iterates around (T, Cc): iterate k = Cc + k * delta, delta a fixed random direction whose power-k coefficients are
    scaled by piece_time^-k so that each step moves the trajectory by ~step_m metres (1 cm: a typical L-BFGS step of this problem)."""
    N = w["pieces"]
    rng = np.random.default_rng(seed)
    d = rng.normal(size=(3, N, 6)) * step_m / (2.5 ** np.arange(6))[None, None, :]
    delta = d.reshape(-1)
    return np.stack([Cc + k * delta for k in range(n)])


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.p:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            txt, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            return out
        sm, mx, reasons = [], [], set()
        for line in txt.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            # the first samples precede the GPU work: report the median of the upper half (clocks under load)
            sm_sorted = sorted(sm)
            out = {"sm_mhz": statistics.median(sm_sorted[len(sm_sorted) // 2:]), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                   "samples": len(sm), "sm_mhz_min": min(sm)}
        return out


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_capture(key="k_discrete_dram_bytes_per_launch"):
    """a figure of the dominant kernel from the committed ncu --set full capture (profiles/roofline_traffic.json), or None."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(key)
        except Exception:
            return None
    return None


def ncu_traffic():
    return ncu_capture("k_discrete_dram_bytes_per_launch")


# ---- CPU arm: the reference's algorithm (oracle port, OpenMP `parallel for schedule(dynamic)` + `critical`) -----------------
def usable_cores():
    """threads the CPU arms may really use: logical CPUs, narrowed by the affinity mask and a cgroup CPU quota (a container that sees 128
    CPUs but is throttled to a few cores' worth of time runs SLOWER with 128 threads — the CPU arm should get its best shot)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, int(q / per + 0.5)))
        except Exception:
            pass
    return max(1, n)


def cpu_sample_eval(w, cfg, occ, T, Cc, V, F, pieces, threads, mode=1):
    """one evaluation restricted to `pieces` pieces spread evenly over the trajectory (a bounded, representative sample of the same
    workload — the term couples nothing across pieces); mode 1 = the reference's loop structure (parallel for dynamic + critical),
    mode 2 = the "fair CPU" arm (per-thread accumulators + the exact culls the GPU uses). Returns (seconds, oracle result)"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O     # bench's CPU legs are one of the three places allowed to execute oracle/
    N = w["pieces"]
    sel = np.unique(np.linspace(0, N - 1, pieces).round().astype(int)) if pieces < N else np.arange(N)
    assert len(sel) == pieces
    Cm = Cc.reshape(3, 6 * N)
    sub = np.concatenate([np.concatenate([Cm[ax, 6 * i:6 * i + 6] for i in sel]) for ax in range(3)])
    oc = O.config_from(cfg)
    oc.threads_num = threads
    if not hasattr(cpu_sample_eval, "shape"):
        cpu_sample_eval.shape = O.Shape.mesh(V, F, w["poly_params"], wn_mode=O.WN_BH)
    t0 = time.perf_counter()
    r = O.eval_discrete(oc, occ, [0, 0, 0], 1.0, cpu_sample_eval.shape, np.ascontiguousarray(T[sel]), sub, use_omp=mode)
    return time.perf_counter() - t0, r


def cpu_baseline(w, cfg, occ, T, Cc, V, F, budget_s=20.0):
    """returns (cpu_baseline object, full-workload oracle result or None, fair-arm object)"""
    cores = usable_cores()
    pieces = 1
    dt, r = cpu_sample_eval(w, cfg, occ, T, Cc, V, F, pieces, cores)
    # grow the sample until it is worth ~budget/2 of CPU time, never beyond the full trajectory
    while dt < budget_s / 4 and pieces < w["pieces"]:
        pieces = min(w["pieces"], pieces * 2)
        dt, r = cpu_sample_eval(w, cfg, occ, T, Cc, V, F, pieces, cores)
    evals_per_s = 1.0 / (dt * w["pieces"] / pieces)
    full = r if pieces == w["pieces"] else None
    # context (SURVEY 8d): one thread, and the README's 1.5 x nproc oversubscription (README.md:148), on bounded samples of the same workload
    dt1, _ = cpu_sample_eval(w, cfg, occ, T, Cc, V, F, 1, 1)
    dto, _ = cpu_sample_eval(w, cfg, occ, T, Cc, V, F, pieces, int(1.5 * cores))
    # the "fair CPU" arm of BASELINE.md §2: per-thread accumulators instead of the critical section AND the exact culls the GPU kernels use
    # (inflated-AABB skip, search bounded by safety_hor, sign only where needed): same cost and gradient, best of 3 whole-workload runs
    dtf, rf = min((cpu_sample_eval(w, cfg, occ, T, Cc, V, F, w["pieces"], cores, mode=2) for _ in range(3)), key=lambda x: x[0])
    fair = {"value": 1.0 / dtf, "unit": UNIT, "cores": cores, "ms_per_eval": 1e3 * dtf,
            "what": "same oracle, per-thread accumulators (no critical section) + the GPU path's exact culls (inflated-AABB skip, BVH search bounded by safety_hor, "
                    "winding number only for pairs with no triangle in reach); whole workload, best of 3",
            "us_per_pair_per_thread": 1e6 * dtf * cores / max(rf[3], 1)}
    if full is not None:
        g, gf = np.concatenate([full[1], full[2]]), np.concatenate([rf[1], rf[2]])
        fair["rel_vs_reference_structure"] = {"cost": abs(rf[0] - full[0]) / abs(full[0]), "grad_l2": float(np.linalg.norm(gf - g) / np.linalg.norm(g))}
    base = {"value": evals_per_s, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{pieces} of {w['pieces']} pieces, evenly spread ({pieces * (w['samples_per_piece'] + 1)} pose samples) of the same workload, "
                      f"{dt:.2f} s wall with {cores} OpenMP threads (schedule(dynamic) + critical, g++ -O3), scaled by pieces",
            "one_thread_evals_per_s": 1.0 / (dt1 * w["pieces"]), "oversubscribed_1p5x_evals_per_s": 1.0 / (dto * w["pieces"] / pieces),
            "us_per_pair_per_thread": 1e6 * dt * cores / max(r[3], 1), "pairs": int(r[3]),
            "note": "reference loop structure: every (pose, voxel) pair inside the body-frame box pays a full closest-triangle search + winding number "
                    "(Shape.cpp:139-151 has no early out); the fair arm beside it (extra.cpu_fair) shows what exact culls buy on the CPU"}
    return base, full, fair


# ---- secondary metric: L-BFGS iterations/s over the whole callback (MINCO -> swept-volume term -> time integral -> adjoint) -------
def lbfgs_workload():
    import isdf_b200 as I
    import workloads as W
    X = 256
    occ = W.random_map(X, X, X, p=0.05, seed=2, slabs=3)
    cfg = I.default_config_values()
    cfg.flags = I.WITH_DYNAMICS                      # the live reference callback: collision through the swept-volume term
    N = 64
    wp = W.random_walk_waypoints(N, [0, 0, 0], [X, X, X], seed=11)
    pts = W.gather_obstacle_points(occ, [0, 0, 0], 1.0, wp, cfg.kernel_size * cfg.occupancy_resolution / 3.0)
    head, tail = np.zeros((3, 3)), np.zeros((3, 3))
    head[:, 0], tail[:, 0] = wp[0], wp[-1]
    x0 = np.concatenate([np.full(N, 1.2), wp[1:-1].reshape(-1)])   # tau = 1.2 -> T = 2.92 s per piece
    return cfg, N, wp, pts, head, tail, x0, "Torus_big"


def lbfgs_ours(device, max_iterations=40):
    import ctypes as CT
    import isdf_b200 as I
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import host_lib as H
    cfg, N, wp, pts, head, tail, x0, shape = lbfgs_workload()
    ev = I.Evaluator(cfg, device=device)
    ev.set_shape_named(shape)
    ev.set_points(pts)
    L = H.lib()
    hh, tt = np.asfortranarray(head), np.asfortranarray(tail)
    out = {}
    for rep in range(2):                                           # first run warms up allocations / work-item tables
        be = L.isdf_host_backend_create(ev.h, N, hh.ctypes.data_as(H.dp), tt.ctypes.data_as(H.dp), 20.0, 1, 1)
        x = x0.copy()
        fx, it, evs = CT.c_double(0), CT.c_int(0), CT.c_int(0)
        t0 = time.perf_counter()
        r = L.isdf_host_lbfgs_backend(be, x.ctypes.data_as(H.dp), x.size, CT.byref(fx), 16, 10, 1e-6, 0.0, max_iterations, CT.byref(it), CT.byref(evs))
        dt = time.perf_counter() - t0
        L.isdf_host_backend_destroy(be)
        out = {"iters_per_s": it.value / dt, "callback_evals_per_s": evs.value / dt, "iterations": it.value, "evaluations": evs.value,
               "seconds": dt, "ret": r, "final_cost": fx.value,
               "config": f"256^3 map p=0.05, 64 pieces, {len(pts)} obstacle points, robot {shape}, callback = MINCO + swept-volume term + "
                         "time-integral dynamics + adjoint (back_end_optimizer.hpp:358-430), L-BFGS mem 16 past 10 (config_CappedCone.yaml:99-102)"}
    ev.close()
    return out


def lbfgs_cpu(max_iterations=2):
    """same driver, callback assembled from the oracle (OpenMP, all host threads)"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import host_lib as H
    import oracle_lib as O
    cfg, N, wp, pts, head, tail, x0, shape = lbfgs_workload()
    oc = O.config_from(cfg)
    oc.threads_num = usable_cores()
    sh = O.Shape.named(shape)
    rho = 20.0

    def fun(x):
        tau = x[:N]
        T = np.where(tau > 0, (0.5 * tau + 1) * tau + 1, 1 / ((0.5 * tau - 1) * tau + 1))
        inP = x[N:].reshape(-1, 3).T
        co, energy, gC, gT = O.minco_forward(head, tail, inP, T)
        sv = O.eval_swept(oc, sh, T, co, pts, use_omp=True)
        di = O.eval_discrete(oc, None, [0, 0, 0], 1.0, None, T, co, use_omp=True)
        cost = energy + sv["cost"] + di[0] + rho * T.sum()
        gp, gt = O.minco_backward(head, tail, inP, T, gC + sv["gradC"] + di[1], gT + sv["gradT"] + di[2])
        gt = gt + rho
        gtau = np.where(tau > 0, gt * (tau + 1), gt * (1 - tau) / ((0.5 * tau - 1) * tau + 1) ** 2)
        return cost, np.concatenate([gtau, gp.T.reshape(-1)])
    t0 = time.perf_counter()
    r = H.lbfgs_minimize(fun, x0, mem_size=16, past=10, delta=1e-6, g_epsilon=0.0, max_iterations=max_iterations)
    dt = time.perf_counter() - t0
    return {"iters_per_s": r["iterations"] / dt, "callback_evals_per_s": r["evaluations"] / dt, "iterations": r["iterations"],
            "evaluations": r["evaluations"], "seconds": dt, "cores": oc.threads_num}


# ---- secondary metric: the swept-volume term alone (BASELINE configs[3]), mesh robot = the reference's live default ---------------
def swept_ours(device, with_cpu, cpu_points=423):
    import isdf_b200 as I
    import workloads as W
    X = 256
    occ = W.random_map(X, X, X, p=0.02, seed=2, slabs=3)
    cfg = I.default_config_values()
    cfg.flags = I.WITH_DYNAMICS
    T, Cc, wp = W.make_trajectory(64, [0, 0, 0], [X, X, X], seed=11, jitter=0.2)
    pts = W.gather_obstacle_points(occ, [0, 0, 0], 1.0, wp, cfg.kernel_size / 3.0)
    V, F = W.rounded_cone_mesh()
    poly = [0, 0, 0, 120, 0, 0]
    ev = I.Evaluator(cfg, device=device)
    ev.set_shape_mesh(V, F, poly)
    ev.set_points(pts)
    for _ in range(3):
        ev.eval_swept(T, Cc)
    ks, es = [], []
    for _ in range(10):
        t0 = time.perf_counter(); ev.eval_swept(T, Cc); es.append(time.perf_counter() - t0)
        ks.append(ev.stats().last_kernel_ms)
    st = ev.stats()
    out = {"config": f"BASELINE configs[3]: 256^3 map, 64-piece trajectory ({T.sum():.0f} s), {len(pts)} obstacle points, 3900-triangle mesh robot; "
                     "SV-SDF query (coarse 0.2 s scan, fine 0.02 s scan, sign descent) + chain rule per point",
           "kernel_ms": statistics.median(ks), "e2e_ms": 1e3 * statistics.median(es), "points_per_s": len(pts) / (statistics.median(ks) * 1e-3),
           "reference_equivalent_sdf_evals": int(st.last_sdf_evals)}
    ev.close()
    if with_cpu:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib as O
        oc = O.config_from(cfg); oc.threads_num = usable_cores()
        sh = O.Shape.mesh(V, F, poly, wn_mode=O.WN_BH)
        n = min(len(pts), cpu_points)
        idx = np.linspace(0, len(pts) - 1, n).astype(int)          # spread over the trajectory: per-point work is very uneven
        O.eval_swept(oc, sh, T, Cc, pts[idx[:32]], use_omp=True)      # wake the OpenMP pool
        dts = []
        for _ in range(2):
            t0 = time.perf_counter(); O.eval_swept(oc, sh, T, Cc, pts[idx], use_omp=True); dts.append(time.perf_counter() - t0)
        dt = min(dts)                                                 # the faster run: the CPU arm gets the benefit of the doubt
        out["cpu"] = {"ms_full_estimate": 1e3 * dt * len(pts) / n, "cores": oc.threads_num, "sample": f"{n} of {len(pts)} points, OpenMP oracle port, best of 2"}
        out["speedup_kernel_vs_cpu"] = out["cpu"]["ms_full_estimate"] / out["kernel_ms"]
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    w, cfg, occ, T, Cc, V, F = make_workload(args.small)
    cores = usable_cores()
    pieces = max(1, min(args.ref_pieces, w["pieces"]))
    for _ in range(max(0, min(args.warmup, 1))):
        cpu_sample_eval(w, cfg, occ, T, Cc, V, F, pieces, cores)
    times = []
    for _ in range(args.steps):
        dt, _ = cpu_sample_eval(w, cfg, occ, T, Cc, V, F, pieces, cores)
        times.append(dt)
    ms = 1e3 * statistics.mean(times) * w["pieces"] / pieces
    val = 1e3 / ms
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(w), **w},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": (f"each step = the whole workload ({pieces} pieces); " if pieces == w["pieces"] else
                                        f"each step = {pieces} of {w['pieces']} pieces, evenly spread, time scaled by {w['pieces']}/{pieces}; ") +
                                       f"{cores} OpenMP threads, reference loop structure (parallel for dynamic + critical)"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


def batch_callback_bench(ev, w, cfg, dev, rank, world, B, barrier, max_over_ranks, reps=3):
    """B problems per GPU through isdf_callback_batch_device: x -> MINCO -> time-integral term with the discrete collision loop over the
    concatenated B*N pieces -> adjoint -> grad(x). Problems differ per rank (seeds), nothing is exchanged: weak scaling by construction."""
    import torch
    import workloads as W
    N0, X = w["pieces"], w["map_dim"]
    dim = 4 * N0 - 3
    xs, heads, tails = np.zeros((B, dim)), np.zeros((B, 9)), np.zeros((B, 9))
    for b in range(B):
        wp = W.random_walk_waypoints(N0, [0, 0, 0], [X, X, X], seed=1000 + rank * B + b)
        xs[b, :N0] = 1.0                                   # tau = 1 -> T = 2.5 s (inittime)
        xs[b, N0:] = wp[1:-1].reshape(-1)
        heads[b, 0:3], tails[b, 0:3] = wp[0], wp[-1]       # column-major 3x3: first column = position
    d_x, d_h, d_t = (torch.from_numpy(a).to(dev) for a in (xs, heads, tails))
    d_cost = torch.zeros(B, dtype=torch.float64, device=dev)
    d_grad = torch.zeros(B, dim, dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    ev.set_shard(0, 1)

    def step():
        ev.callback_batch_device(B, N0, d_h.data_ptr(), d_t.data_ptr(), 1, 20.0, d_x.data_ptr(), d_cost.data_ptr(), d_grad.data_ptr(), stream)
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); barrier()
        e0.record(); step(); e1.record()
        torch.cuda.synchronize()
        ts.append(max_over_ranks(e0.elapsed_time(e1)))
    ms = statistics.mean(ts)
    c = d_cost.cpu().numpy()
    per_problem = None
    if world == 1:
        # the same problems one at a time through the host adapter (host MINCO port + isdf_eval_discrete with host buffers)
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import host_lib as H
        from ctypes import c_int as C_int
        L = H.lib()
        nb = min(B, 16)
        g = np.zeros(dim)
        t0 = time.perf_counter()
        cs = []
        for b in range(nb):
            be = L.isdf_host_backend_create(ev.h, N0, heads[b].ctypes.data_as(H.dp), tails[b].ctypes.data_as(H.dp), 20.0, 0, 1)
            cs.append(L.isdf_host_backend_cost(be, xs[b].ctypes.data_as(H.dp), g.ctypes.data_as(H.dp), dim))
            L.isdf_host_backend_destroy(be)
        dt = time.perf_counter() - t0
        per_problem = {"callbacks_per_s": nb / dt, "problems": nb, "max_rel_cost_diff_vs_batched": float(np.max(np.abs(np.array(cs) - c[:nb]) / np.abs(c[:nb])))}
    lockstep = None
    if world == 1:
        # B restarts under the lock-step batched L-BFGS driver (host/isdf_lbfgs.hpp): every round = one batched device callback
        try:
            nb = min(B, 32)
            Xl = np.ascontiguousarray(xs[:nb]).copy().reshape(-1)
            fl, rl = np.zeros(nb), np.zeros(nb, dtype=np.int32)
            itl, evl, stl = np.zeros(nb, dtype=np.int32), np.zeros(nb, dtype=np.int32), C_int()
            ipt = H.C.POINTER(H.C.c_int)
            t0 = time.perf_counter()
            rounds = L.isdf_host_lbfgs_batch_backend(ev.h, nb, N0, np.ascontiguousarray(heads[:nb]).ctypes.data_as(H.dp), np.ascontiguousarray(tails[:nb]).ctypes.data_as(H.dp),
                                                     20.0, Xl.ctypes.data_as(H.dp), fl.ctypes.data_as(H.dp), rl.ctypes.data_as(ipt), 16, 10, 1e-6, 0.0, 12,
                                                     itl.ctypes.data_as(ipt), evl.ctypes.data_as(ipt), H.C.byref(stl))
            dt = time.perf_counter() - t0
            lockstep = {"problems": nb, "rounds": int(rounds), "iterations_total": int(itl.sum()), "evaluations_total": int(evl.sum()), "seconds": dt,
                        "iters_per_s": float(itl.sum() / dt), "callback_evals_per_s": float(evl.sum() / dt), "status": int(stl.value),
                        "mean_cost_start": float(c[:nb].mean()), "mean_cost_end": float(fl.mean()), "max_iterations": 12}
        except Exception as e:
            lockstep = {"error": repr(e)}
        try:   # the same restarts under the DEVICE-RESIDENT lock-step driver (isdf_lbfgs_batch: iterates never leave the GPU)
            nb = min(B, 32)
            prm = ev.lbfgs_params(max_iterations=12)
            hh3 = heads[:nb].reshape(nb, 3, 3).transpose(0, 2, 1)
            tt3 = tails[:nb].reshape(nb, 3, 3).transpose(0, 2, 1)
            t0 = time.perf_counter()
            rd = ev.lbfgs_batch(hh3, tt3, 20.0, xs[:nb], prm)
            dt = time.perf_counter() - t0
            lockstep["device_resident"] = {"problems": nb, "rounds": int(rd["rounds"]), "iterations_total": int(rd["iterations"].sum()), "evaluations_total": int(rd["evaluations"].sum()),
                                           "seconds": dt, "iters_per_s": float(rd["iterations"].sum() / dt), "callback_evals_per_s": float(rd["evaluations"].sum() / dt),
                                           "batched_evals_per_s_incl_finished_instances": float(nb * rd["rounds"] / dt), "mean_cost_end": float(rd["f"].mean()),
                                           "identical_to_host_lockstep": bool(np.array_equal(rd["x"].reshape(-1), Xl) and np.array_equal(rd["f"], fl))}
        except Exception as e:
            if isinstance(lockstep, dict):
                lockstep["device_resident"] = {"error": repr(e)}
    return {"callbacks_per_s": world * B * 1e3 / ms, "host_adapter_one_at_a_time": per_problem, "lockstep_lbfgs": lockstep, "ms_per_batch_max_over_ranks": ms, "problems_per_gpu": B, "problems_total": world * B,
            "scaling": "weak", "finite_costs": bool(np.all(np.isfinite(c))), "mean_cost": float(c.mean()),
            "what": f"BASELINE configs[4]: {world * B} random-restart problems ({N0} pieces x {w['samples_per_piece']} samples, shared {X}^3 map, mesh robot), "
                    "decision vector in -> cost and gradient out, MINCO forward/adjoint + time-integral/collision term all on the device; no collective"}


def frontend_bench(ev, w, occ, V, F, dev, with_cpu, reps=3):
    """SURVEY 8f row 4 on the bench map: which of the 121 (roll, pitch) attitudes of the mesh robot fit at EVERY voxel (128-bit mask per voxel)."""
    import torch
    X = w["map_dim"]
    t0 = time.perf_counter()
    xk, yk = ev.frontend_build_kernels(45.0, 45.0, 9.0, 0.0)          # config_CappedCone.yaml:62-64
    t_build = time.perf_counter() - t0
    nvox = X ** 3
    d_masks = torch.empty(nvox * 4, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    ev.frontend_feasibility_device(d_masks.data_ptr(), stream)
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); ev.frontend_feasibility_device(d_masks.data_ptr(), stream); e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ms = statistics.median(ts)
    fit = int((d_masks.view(-1, 4) != 0).any(dim=1).sum().item())
    peak, peak_src = measured_peak_hbm()
    nbytes = nvox * 16 + nvox // 8
    out = {"what": f"attitude-kernel feasibility of all {X}^3 voxels x {xk * yk} attitudes (kernel {w['kernel_size']}^3, mesh robot): kernelConv<true> of "
                   "sw_manager.hpp:821-846 for every voxel, 128-bit mask out",
           "ms": ms, "voxels_per_s": nvox / (ms * 1e-3), "voxel_attitude_checks_per_s": nvox * xk * yk / (ms * 1e-3), "kernel_build_s": t_build,
           "voxels_with_a_fitting_attitude": fit,
           "roofline": {"bound": "hbm", "achieved": nbytes / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": nbytes / (ms * 1e-3) / 1e9 / peak,
                        "algorithmic_bytes_per_launch": nbytes, "peak_source": peak_src,
                        "note": "16 B mask written + 1 bit occupancy read per voxel; the window reads hit L1/L2"}}
    del d_masks
    if with_cpu:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib as O
        sub = np.ascontiguousarray(occ[:96, :96, :96])
        fe = O.FrontEnd(O.Shape.mesh(V, F, w["poly_params"], wn_mode=O.WN_BH), sub, ks=w["kernel_size"])
        rng = np.random.default_rng(0)
        n = 200000
        ind = rng.integers(0, 96, (n, 3))
        O.lib().orc_set_num_threads(usable_cores())                   # the front-end loop uses OpenMP's default team
        fe.feasibility(ind[:2000])                                    # wake the OpenMP pool
        dts = []
        for _ in range(2):
            t0 = time.perf_counter(); fe.feasibility(ind); dts.append(time.perf_counter() - t0)
        dt = min(dts)
        out["cpu"] = {"voxels_per_s": n / dt, "cores": usable_cores(), "sample": f"{n} random voxels of a 96^3 corner of the same map, oracle byte-kernel port, OpenMP, best of 2"}
        out["speedup_vs_cpu"] = out["voxels_per_s"] / out["cpu"]["voxels_per_s"]
    return out


def workload_name(w):
    return (f"BASELINE configs[2]: random {w['map_dim']}^3 voxel map (p={w['occupancy']}, wall slabs), {w['pieces']}-piece MINCO traj, "
            f"{w['samples_per_piece']} samples/piece, mesh-SDF robot ({w['mesh']}), discrete collision cost+grad")


def dump_outputs(out_dir, **arrays):
    """--dump-outputs: one float64 .npy per array, so that two builds run with the same arguments can be compared output for output"""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


# ---- GPU arm ----------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import isdf_b200 as I
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    w, cfg, occ, T, Cc, V, F = make_workload(args.small)
    N = w["pieces"]
    ev = I.Evaluator(cfg, device=local)
    ev.set_map_u8(occ, [0, 0, 0], 1.0)
    if args.robot == "mesh":
        ev.set_shape_mesh(V, F, w["poly_params"])
    else:
        import workloads as W
        R, t = W.rotation_from_poly_params(w["poly_params"])
        ev.set_shape_named(args.robot, R, t)
        w["mesh"] = "analytic:" + args.robot
        args.no_cpu_baseline = True
    ev.set_shard(rank, world)
    dev = torch.device("cuda", local)
    n_warm = max(args.warmup, 3)
    n_e2e_warm = 3
    n_iter = n_warm + args.steps + n_e2e_warm + args.steps + 2
    iters = make_iterates(w, T, Cc, n_iter)                 # iterate 0 = the unperturbed trajectory (parity is checked on it)
    d_T = torch.from_numpy(T).to(dev)
    d_Cs = torch.from_numpy(iters).to(dev)                  # every iterate resident in HBM before the timed region
    d_out = torch.zeros(19 * N + 1, dtype=torch.float64, device=dev)
    flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2
    stream = torch.cuda.current_stream().cuda_stream
    ref_nccl = None
    if world > 1:                                         # untimed cross-check for the fused exchange: same shards, NCCL sum
        ev.eval_discrete_device(N, d_T.data_ptr(), d_Cs[0].data_ptr(), d_out.data_ptr(), stream)
        allreduce_partials(d_out)
        torch.cuda.synchronize()
        ref_nccl = d_out.cpu().numpy().copy()
    # multi-GPU reduction: fused into the evaluation through NVLink peer memory (isdf_peer_*); NCCL all-reduce if that cannot be set up
    collective = "none"
    if world > 1:
        import torch.distributed as dist
        collective = "nccl"
        if args.collective == "peer":
            try:
                handles = [None] * world
                dist.all_gather_object(handles, ev.peer_export(world, 19 * N + 1))
                ev.peer_connect(world, rank, handles, fuse=True)
                okf = torch.ones(1, device=dev)
            except Exception as e:
                okf = torch.zeros(1, device=dev)
                if rank == 0:
                    print(f"bench: peer-memory exchange unavailable ({e}); using NCCL", file=sys.stderr)
            dist.all_reduce(okf, op=dist.ReduceOp.MIN)
            if okf.item() == 1:
                collective = "peer"
            else:
                try:
                    ev.peer_disconnect()
                except Exception:
                    pass
            dist.barrier()

    def step_device(k):
        ev.eval_discrete_device(N, d_T.data_ptr(), d_Cs[k].data_ptr(), d_out.data_ptr(), stream)   # collective == "peer": includes the exchange
        if collective == "nccl":
            allreduce_partials(d_out)

    def timed(ks, do_flush=True):
        out = []
        for k in ks:
            if do_flush:
                flush.zero_()                               # L2 flush between timed iterations (not timed)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            barrier()
            release_together()
            e0.record()
            step_device(k)
            e1.record()
            torch.cuda.synchronize()
            out.append(max_over_ranks(e0.elapsed_time(e1)))
        return out

    sampler = ClockSampler(local) if rank == 0 else None   # nvidia-smi needs ~0.5 s to start: begin before the warm-up
    step_device(0)                                          # iterate 0 first: its result is the one compared with the CPU arm
    torch.cuda.synchronize()
    result = d_out.cpu().numpy().copy()
    for k in range(1, n_warm):
        step_device(k)
    torch.cuda.synchronize()
    barrier()
    l0 = ev.stats().kernel_launches
    t_wall0 = time.perf_counter()
    times = timed(range(n_warm, n_warm + args.steps))       # THE timed region: K distinct iterates, each on the schedule of its predecessor
    barrier()
    wall = time.perf_counter() - t_wall0
    launches = ev.stats().kernel_launches - l0
    last = d_out.cpu().numpy().copy()                       # [cost | gradC | gradT] of the last timed step (--dump-outputs)
    k_last = n_warm + args.steps - 1
    # context figures (not the headline): warm L2; the SAME iterate repeated (round 1's measurement: the schedule is a perfect predictor);
    # cold = a context's first evaluation (natural sample order, nothing split)
    warm = timed(range(n_warm, n_warm + min(args.steps, 10)), do_flush=False)
    same = timed([k_last] * (2 + min(args.steps, 10)))[2:]
    cold = None
    try:
        ev.dbg_schedule(natural_order=True)
        cold = timed([k_last] * 5)
        ev.dbg_schedule(natural_order=False)
        for k in range(2):
            step_device(k_last)
    except Exception:
        cold = None
    # the timed region is only tens of milliseconds: keep the same kernel running (untimed) until nvidia-smi has sampled it
    for _ in range(40):                                     # a FIXED count: every rank must run the same number of (exchanging) evaluations
        for _ in range(50):
            step_device(k_last)
        torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None
    ms = statistics.mean(times)

    # ---- e2e: the reference-facing C-ABI call with HOST buffers (H2D + kernel + D2H inside the timed region), distinct iterates ----
    e2e_times = []
    h_part = torch.empty(19 * N + 1, dtype=torch.float64).pin_memory()
    k0 = n_warm + args.steps
    for it in range(n_e2e_warm + args.steps):
        Ck = iters[k0 + it]
        flush.zero_()
        torch.cuda.synchronize(); barrier()
        t0 = time.perf_counter()
        c, gC, gT = ev.eval_discrete(T, Ck)               # isdf_eval_discrete: pinned staging, H2D, kernel, D2H, sync
        if collective == "nccl":
            h_part[0] = c; h_part[1:1 + 18 * N] = torch.from_numpy(gC); h_part[1 + 18 * N:] = torch.from_numpy(gT)
            d_tmp = h_part.to(dev, non_blocking=True)
            allreduce_partials(d_tmp)
            h_part.copy_(d_tmp)
            torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) * 1e3
        if it >= n_e2e_warm:
            e2e_times.append(max_over_ranks(dt))
    pairs = ev.stats().last_pairs
    kernel_ms_alone = ev.stats().last_kernel_ms
    ms_e2e = statistics.mean(e2e_times)

    # ---- context for N > 1: batch of random restarts, one trajectory per GPU, no collective (BASELINE configs[4] in miniature) ----
    batch_weak = None
    if world > 1:
        import workloads as W
        Tb, Cb, _ = W.make_trajectory(N, [0, 0, 0], [w["map_dim"]] * 3, seed=11 + rank, jitter=0.2)
        ev.set_shard(0, 1)
        d_Tb, d_Cb = torch.from_numpy(Tb).to(dev), torch.from_numpy(Cb).to(dev)
        for _ in range(4):
            ev.eval_discrete_device(N, d_Tb.data_ptr(), d_Cb.data_ptr(), d_out.data_ptr(), stream)
        tb = []
        for _ in range(args.steps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(); barrier()
            e0.record(); ev.eval_discrete_device(N, d_Tb.data_ptr(), d_Cb.data_ptr(), d_out.data_ptr(), stream); e1.record()
            torch.cuda.synchronize()
            tb.append(max_over_ranks(e0.elapsed_time(e1)))
        ev.set_shard(rank, world)
        batch_weak = {"evals_per_s": world * 1e3 / statistics.mean(tb), "ms_per_step_max_over_ranks": statistics.mean(tb), "scaling": "weak",
                      "what": f"{world} different trajectories (seed 11+rank), one per GPU, evaluated concurrently; no collective"}

    # ---- BASELINE configs[4]: batch of random restarts, whole callback on the device, B_local problems per GPU, no collective ----
    batch_cb = None
    if not args.no_batch and not args.small:
        try:
            batch_cb = batch_callback_bench(ev, w, cfg, dev, rank, world, args.batch_per_gpu, barrier, max_over_ranks)
        except Exception as e:
            batch_cb = {"error": repr(e)}
        ev.set_shard(rank, world)

    if rank == 0:
        peak, peak_src = measured_peak_hbm()
        ab = algorithmic_bytes(w)
        achieved = ab / (ms * 1e-3) / 1e9 if world == 1 else ab / world / (ms * 1e-3) / 1e9
        line = {"metric": METRIC, "value": 1e3 / ms, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": workload_name(w), **w, "l2": "flushed (512 MiB write) between timed steps",
                           "iterates": f"{args.steps} distinct iterates (trajectory moved ~1 cm per step), each evaluated on the work-item schedule learned from its predecessor",
                           "term": "discrete collision term = grad_cost_p wired into addTimeIntPenaltyParallel (back_end_optimizer.hpp:766-824, the north star's / IROS-2023 form); "
                                   "it is DEAD CODE in the reference snapshot, whose live collision term is the swept-volume one (extra.swept, --workload swept)",
                           "parallelism": (f"sample-interleaved shards x{world} + " + (f"rank-ordered sum of {19 * N + 1} doubles over NVLink peer memory, fused into the epilogue kernel"
                                                                                      if collective == "peer" else f"1 NCCL all-reduce of {19 * N + 1} doubles")) if world > 1 else "1 GPU"},
                "clocks": clocks,
                "e2e": {"value": 1e3 / ms_e2e, "unit": UNIT, "h2d_bytes_per_step": 8 * 19 * N, "d2h_bytes_per_step": 8 * (19 * N + 1) + 8,
                        "ms_per_step": ms_e2e, "api": "isdf_eval_discrete (host buffers)"},
                "gpu_launches": int(launches),
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic(),
                             "peak_source": peak_src, "kernel": "k_discrete_mesh", "algorithmic_bytes_per_launch": ab // world,
                             "fp64_pipe_active_pct_ncu": ncu_capture("fp64_pipe_active_pct"), "issue_slots_busy_pct_ncu": ncu_capture("issue_slots_busy_pct"),
                             "note": "window bytes counted at 1 B/voxel per sample (SURVEY §8d); the kernel is FP64/latency bound, see DESIGN.md"},
                "extra": {"pairs_per_eval": int(pairs), "pairs_per_s": pairs / (ms * 1e-3), "ms_per_step_warm_l2": statistics.mean(warm),
                          "evals_per_s_warm_l2": 1e3 / statistics.mean(warm), "ms_min": min(times), "ms_max": max(times),
                          "ms_per_step_same_iterate": statistics.mean(same), "ms_per_step_cold": (statistics.mean(cold) if cold else None),
                          "schedule_note": "value = distinct iterates on a stale (previous iterate's) schedule; same_iterate = round 1's measurement (identical trajectory "
                                           "every step); cold = first evaluation of a context: natural sample order, nothing split",
                          "kernel_ms_in_host_call": kernel_ms_alone, "wall_s_timed_loop": wall,
                          "cost": float(result[0]), "grad_norm": float(np.linalg.norm(result[1:])), "batch_weak": batch_weak,
                          "collective": collective,
                          "collective_vs_nccl_rel_l2": (float(np.linalg.norm(result - ref_nccl) / np.linalg.norm(ref_nccl)) if ref_nccl is not None else None),
                          "batch_callback": batch_cb}}
        if world == 1 and not args.no_lbfgs:
            try:
                line["extra"]["lbfgs"] = lbfgs_ours(local)
                if not args.no_cpu_baseline:
                    line["extra"]["lbfgs"]["cpu"] = lbfgs_cpu()
            except Exception as e:   # secondary metric must never take the headline line down
                line["extra"]["lbfgs"] = {"error": repr(e)}
        if world == 1 and not args.no_frontend and args.robot == "mesh" and not args.small:
            try:
                line["extra"]["frontend"] = frontend_bench(ev, w, occ, V, F, dev, not args.no_cpu_baseline)
            except Exception as e:
                line["extra"]["frontend"] = {"error": repr(e)}
        if world == 1 and not args.no_swept:
            try:
                line["extra"]["swept"] = swept_ours(local, not args.no_cpu_baseline)
            except Exception as e:
                line["extra"]["swept"] = {"error": repr(e)}
        if world == 1 and not args.no_cpu_baseline:
            base, full, fair = cpu_baseline(w, cfg, occ, T, Cc, V, F, budget_s=args.cpu_budget)
            line["cpu_baseline"] = base
            line["extra"]["cpu_fair"] = fair
            line["extra"]["speedup_kernel_vs_cpu"] = line["value"] / base["value"]
            line["extra"]["speedup_e2e_vs_cpu"] = line["e2e"]["value"] / base["value"]
            line["extra"]["speedup_e2e_vs_cpu_fair"] = line["e2e"]["value"] / fair["value"]
            if full is not None:   # parity of the benchmark workload itself (iterate 0): GPU result against the CPU arm's full-size result
                og = np.concatenate([full[1], full[2]])
                line["parity"] = {"cost_rel": abs(float(result[0]) - full[0]) / abs(full[0]),
                                  "grad_rel_l2": float(np.linalg.norm(result[1:] - og) / np.linalg.norm(og)),
                                  "against": "oracle (OpenMP order), whole benchmark workload, same inputs",
                                  "tolerance": 1e-6}
            try:   # deviation of the product's ±1 sign policy from the reference-faithful s = 1 - 2 w_FWN (w from the reference-compiled FWN header)
                sys.path.insert(0, os.path.join(ROOT, "tests"))
                import oracle_lib as O
                if O.ref_fwn_available():
                    oc = O.config_from(cfg); oc.threads_num = usable_cores()
                    rf = O.eval_discrete(oc, occ, [0, 0, 0], 1.0, O.Shape.mesh(V, F, w["poly_params"], wn_mode=O.WN_REF), T, Cc, use_omp=True)
                    rg = np.concatenate([rf[1], rf[2]])
                    line["extra"]["sign_policy_deviation_vs_reference_fwn"] = {
                        "cost_rel": abs(float(result[0]) - rf[0]) / abs(rf[0]), "grad_rel_l2": float(np.linalg.norm(result[1:] - rg) / np.linalg.norm(rg)),
                        "what": "product (sign = ±1, exact inside/outside) against the oracle with the reference's un-thresholded s = 1 - 2 w, w from "
                                "oracle/_ref/libref_fwn.so (the reference's own FastWindingNumberForSoups.h, FP32 order 2, beta 2); this is the FWN's approximation "
                                "error seen through the hinge, reported as SURVEY 8c demands — not a parity claim"}
            except Exception as e:
                line["extra"]["sign_policy_deviation_vs_reference_fwn"] = {"error": repr(e)}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, cost=last[:1], gradC=last[1:1 + 18 * N], gradT=last[1 + 18 * N:])
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        torch.cuda.synchronize()
        dist.barrier()
        if collective == "peer":
            ev.peer_status()
            ev.peer_disconnect()
    ev.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


# ---- other BASELINE configs as strong-scaling workloads of their own ----------------------------------------------------------
def _dist_setup():
    import torch
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local


def _peer_setup(ev, world, rank, n, dev):
    """fused exchange over NVLink peer memory for the sharded evaluation; returns 'peer' or 'nccl'"""
    import torch
    import torch.distributed as dist
    try:
        handles = [None] * world
        dist.all_gather_object(handles, ev.peer_export(world, n))
        ev.peer_connect(world, rank, handles, fuse=True)
        okf = torch.ones(1, device=dev)
    except Exception as e:
        okf = torch.zeros(1, device=dev)
        if rank == 0:
            print(f"bench: peer-memory exchange unavailable ({e}); using NCCL", file=sys.stderr)
    dist.all_reduce(okf, op=dist.ReduceOp.MIN)
    if okf.item() != 1:
        try:
            ev.peer_disconnect()
        except Exception:
            pass
        return "nccl"
    dist.barrier()
    return "peer"


def swept_workload():
    import isdf_b200 as I
    import workloads as W
    X = 256
    occ = W.random_map(X, X, X, p=0.02, seed=2, slabs=3)
    cfg = I.default_config_values()
    cfg.flags = I.WITH_DYNAMICS
    T, Cc, wp = W.make_trajectory(64, [0, 0, 0], [X, X, X], seed=11, jitter=0.2)
    pts = W.gather_obstacle_points(occ, [0, 0, 0], 1.0, wp, cfg.kernel_size / 3.0)
    V, F = W.rounded_cone_mesh()
    w = dict(map_dim=X, occupancy=0.02, pieces=64, points=int(len(pts)), mesh="rounded_cone_3900tri", poly_params=[0.0, 0.0, 0.0, 120.0, 0.0, 0.0],
             workload=f"BASELINE configs[3]: swept-volume SV-SDF collision term, 256^3 map, 64-piece trajectory ({T.sum():.0f} s), {len(pts)} obstacle points, mesh robot")
    return w, cfg, T, Cc, pts, V, F


def run_swept(args):
    """configs[3] as a strong-scaling workload: one step = one swept-volume cost+grad evaluation; obstacle points sharded over the ranks
    (interleaved), the 19N+1 doubles summed over NVLink peer memory by the evaluation's last kernel"""
    import torch
    import isdf_b200 as I
    rank, world, local = _dist_setup()
    w, cfg, T, Cc, pts, V, F = swept_workload()
    N = w["pieces"]
    dev = torch.device("cuda", local)
    ev = I.Evaluator(cfg, device=local)
    ev.set_shape_mesh(V, F, w["poly_params"])
    ev.set_points(pts)
    ev.set_shard(rank, world)
    collective = _peer_setup(ev, world, rank, 19 * N + 1, dev) if world > 1 else "none"
    n_warm = max(args.warmup, 3)
    iters = make_iterates(w, T, Cc, 2 * (n_warm + args.steps) + 1)
    d_T, d_Cs = torch.from_numpy(T).to(dev), torch.from_numpy(iters).to(dev)
    d_out = torch.zeros(19 * N + 1, dtype=torch.float64, device=dev)
    flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def step(k):
        ev.eval_swept_device(N, d_T.data_ptr(), d_Cs[k].data_ptr(), d_out.data_ptr(), stream)
        if collective == "nccl":
            allreduce_partials(d_out)
    sampler = ClockSampler(local) if rank == 0 else None
    for k in range(n_warm):
        step(k)
    torch.cuda.synchronize(); barrier()
    l0 = ev.stats().kernel_launches
    times = []
    for k in range(n_warm, n_warm + args.steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); barrier(); release_together()
        e0.record(); step(k); e1.record()
        torch.cuda.synchronize()
        times.append(max_over_ranks(e0.elapsed_time(e1)))
    launches = ev.stats().kernel_launches - l0
    e2e = []
    for it in range(n_warm + args.steps):
        Ck = iters[it]                                      # the iterates of the device-timed loop, in the same order
        flush.zero_()
        torch.cuda.synchronize(); barrier()
        t0 = time.perf_counter()
        c, gC, gT = ev.eval_swept(T, Ck)
        if collective == "nccl":
            part = torch.from_numpy(np.concatenate([[c], gC, gT])).to(dev)
            allreduce_partials(part); part.cpu()
        dt = (time.perf_counter() - t0) * 1e3
        if it >= n_warm:
            e2e.append(max_over_ranks(dt))
    nsdf = ev.stats().last_sdf_evals
    for _ in range(30):                                     # fixed count on every rank (matching exchange epochs)
        for _ in range(30):
            step(0)
        torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None
    if rank == 0:
        ms, ms_e2e = statistics.mean(times), statistics.mean(e2e)
        peak, peak_src = measured_peak_hbm()
        ab = 40 * len(pts) + 8 * 19 * N + 8 * (19 * N + 1)
        line = {"metric": "swept_collision_cost_grad_evals_per_s", "value": 1e3 / ms, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": n_warm,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {**w, "l2": "flushed (512 MiB write) between timed steps", "iterates": "distinct (trajectory moved ~1 cm per step)",
                           "parallelism": f"obstacle points interleaved over {world} rank(s)" + (f", {collective} sum of {19 * N + 1} doubles" if world > 1 else "")},
                "clocks": clocks, "gpu_launches": int(launches),
                "e2e": {"value": 1e3 / ms_e2e, "unit": UNIT, "h2d_bytes_per_step": 8 * 19 * N, "d2h_bytes_per_step": 8 * (19 * N + 1) + 8, "ms_per_step": ms_e2e,
                        "api": "isdf_eval_swept (host buffers)"},
                "roofline": {"bound": "hbm", "achieved": ab / world / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": ab / world / (ms * 1e-3) / 1e9 / peak, "traffic": None,
                             "peak_source": peak_src, "kernel": "k_sv_points_cta<true>", "algorithmic_bytes_per_launch": ab // world,
                             "note": "compute/latency bound by construction (SURVEY 8d): the primary figure is reference-equivalent SDF evaluations per second",
                             "sdf_evals_per_eval_this_rank": int(nsdf), "sdf_evals_per_s_this_rank": nsdf / (ms * 1e-3)}}
        if world == 1 and not args.no_cpu_baseline:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import oracle_lib as O
            oc = O.config_from(cfg); oc.threads_num = usable_cores()
            sh = O.Shape.mesh(V, F, w["poly_params"], wn_mode=O.WN_BH)
            O.eval_swept(oc, sh, T, Cc, pts[:32], use_omp=True)
            dts = []
            for _ in range(2):
                t0 = time.perf_counter(); ref = O.eval_swept(oc, sh, T, iters[0], pts, use_omp=True); dts.append(time.perf_counter() - t0)
            line["cpu_baseline"] = {"value": 1.0 / min(dts), "unit": UNIT, "cores": oc.threads_num, "kind": "port",
                                    "sample": f"whole workload ({len(pts)} points), OpenMP oracle port (parallel for dynamic + critical), best of 2"}
            c, gC, gT = ev.eval_swept(T, iters[0])
            g, og = np.concatenate([gC, gT]), np.concatenate([ref["gradC"], ref["gradT"]])
            line["parity"] = {"cost_rel": abs(c - ref["cost"]) / abs(ref["cost"]), "grad_rel_l2": float(np.linalg.norm(g - og) / np.linalg.norm(og)), "tolerance": 1e-6}
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        torch.cuda.synchronize(); dist.barrier()
        if collective == "peer":
            ev.peer_status(); ev.peer_disconnect()
    ev.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def batch_problems(B, N0, X, first=0):
    import workloads as W
    dim = 4 * N0 - 3
    xs, heads, tails = np.zeros((B, dim)), np.zeros((B, 9)), np.zeros((B, 9))
    for b in range(B):
        wp = W.random_walk_waypoints(N0, [0, 0, 0], [X, X, X], seed=1000 + first + b)
        xs[b, :N0] = 1.0                                   # tau = 1 -> T = 2.5 s (inittime)
        xs[b, N0:] = wp[1:-1].reshape(-1)
        heads[b, 0:3], tails[b, 0:3] = wp[0], wp[-1]       # column-major 3x3: first column = position
    return xs, heads, tails


def run_batch(args):
    """configs[4] as a strong-scaling workload: a FIXED batch of 1024 random-restart problems, sharded by problem over the ranks; one step =
    the whole optimiser callback (MINCO -> time-integral + discrete collision term -> adjoint) for all of them; no collective"""
    import torch
    import isdf_b200 as I
    rank, world, local = _dist_setup()
    w, cfg, occ, T, Cc, V, F = make_workload(False)
    N0, X, Btot = w["pieces"], w["map_dim"], args.batch_total
    B = Btot // world
    dim = 4 * N0 - 3
    dev = torch.device("cuda", local)
    ev = I.Evaluator(cfg, device=local)
    ev.set_map_u8(occ, [0, 0, 0], 1.0)
    ev.set_shape_mesh(V, F, w["poly_params"])
    xs, heads, tails = batch_problems(B, N0, X, first=rank * B)
    d_x, d_h, d_t = (torch.from_numpy(a).to(dev) for a in (xs, heads, tails))
    d_cost = torch.zeros(B, dtype=torch.float64, device=dev)
    d_grad = torch.zeros(B, dim, dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def step():
        ev.callback_batch_device(B, N0, d_h.data_ptr(), d_t.data_ptr(), 1, 20.0, d_x.data_ptr(), d_cost.data_ptr(), d_grad.data_ptr(), stream)
    sampler = ClockSampler(local) if rank == 0 else None
    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize(); barrier()
    l0 = ev.stats().kernel_launches
    times = []
    for _ in range(args.steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); barrier()
        e0.record(); step(); e1.record()
        torch.cuda.synchronize()
        times.append(max_over_ranks(e0.elapsed_time(e1)))
    launches = ev.stats().kernel_launches - l0
    e2e = []
    hh, tt = heads.reshape(B, 3, 3).transpose(0, 2, 1), tails.reshape(B, 3, 3).transpose(0, 2, 1)   # back to row-major 3x3 for the python wrapper
    for it in range(2 + max(3, args.steps // 4)):
        torch.cuda.synchronize(); barrier()
        t0 = time.perf_counter()
        c, g = ev.callback_batch(hh, tt, 20.0, xs)
        dt = (time.perf_counter() - t0) * 1e3
        if it >= 2:
            e2e.append(max_over_ranks(dt))
    clocks = sampler.stop() if sampler else None
    fin = bool(np.all(np.isfinite(c)))
    # BASELINE metric (ii): L-BFGS iterations/s — every rank optimises its own problems with the device-resident lock-step driver
    lb = None
    try:
        prm = ev.lbfgs_params(max_iterations=args.lbfgs_iterations)
        torch.cuda.synchronize(); barrier()
        t0 = time.perf_counter()
        rd = ev.lbfgs_batch(hh, tt, 20.0, xs, prm)
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
        tot = torch.tensor([float(rd["iterations"].sum()), float(rd["evaluations"].sum()), float(rd["f"].sum()), float(c.sum())], dtype=torch.float64, device=dev)
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(tot)
        tot = tot.cpu().numpy()
        lb = {"iters_per_s": tot[0] / dt, "callback_evals_per_s": tot[1] / dt, "iterations_total": int(tot[0]), "evaluations_total": int(tot[1]), "seconds_max_over_ranks": dt,
              "rounds_rank0": int(rd["rounds"]), "max_iterations": args.lbfgs_iterations, "mean_cost_start": tot[3] / Btot, "mean_cost_end": tot[2] / Btot,
              "what": f"{Btot} restarts, each under the reference fork's L-BFGS (mem 16, past 10), lock-step on the device: one batched callback per round, "
                      "iterates and histories resident in HBM; problems sharded over the ranks, no collective"}
    except Exception as e:
        lb = {"error": repr(e)}
    if rank == 0:
        ms, ms_e2e = statistics.mean(times), statistics.mean(e2e)
        S = Btot * N0 * (w["samples_per_piece"] + 1)
        ab = S * w["kernel_size"] ** 3 + 2 * 8 * Btot * dim
        peak, peak_src = measured_peak_hbm()
        line = {"metric": "batched_callback_problems_per_s", "value": Btot * 1e3 / ms, "unit": "problems/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": f"BASELINE configs[4]: {Btot} random-restart problems ({N0} pieces x {w['samples_per_piece']} samples) on the shared {X}^3 map, mesh robot; "
                                       "one step = cost and gradient of every problem (MINCO forward, time-integral + discrete collision term, adjoint), all on the device",
                           "problems_total": Btot, "problems_per_gpu": B, "l2": "the per-step working set (16.8 M pose windows) exceeds L2", "parallelism": f"problems sharded over {world} rank(s), no collective"},
                "clocks": clocks, "gpu_launches": int(launches),
                "e2e": {"value": Btot * 1e3 / ms_e2e, "unit": "problems/s", "h2d_bytes_per_step": 8 * B * (dim + 18), "d2h_bytes_per_step": 8 * B * (dim + 1), "ms_per_step": ms_e2e,
                        "api": "isdf_callback_batch (host buffers: decision vectors in, costs and gradients out)"},
                "roofline": {"bound": "hbm", "achieved": ab / world / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": ab / world / (ms * 1e-3) / 1e9 / peak, "traffic": None,
                             "peak_source": peak_src, "kernel": "k_discrete_mesh", "algorithmic_bytes_per_launch": ab // world},
                "extra": {"finite_costs": fin, "lbfgs": lb}}
        if world == 1 and not args.no_cpu_baseline:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import oracle_lib as O
            oc = O.config_from(cfg); oc.threads_num = usable_cores()
            osh = O.Shape.mesh(V, F, w["poly_params"], wn_mode=O.WN_BH)
            nb, t0 = 4, time.perf_counter()
            worst = 0.0
            for b in range(nb):
                tau = xs[b, :N0]; Tt = np.where(tau > 0, (0.5 * tau + 1) * tau + 1, 1 / ((0.5 * tau - 1) * tau + 1))
                inP = xs[b, N0:].reshape(-1, 3).T
                hb, tb = heads[b].reshape(3, 3).T, tails[b].reshape(3, 3).T
                co, energy, gC, gT = O.minco_forward(hb, tb, inP, Tt)
                di = O.eval_discrete(oc, occ, [0, 0, 0], 1.0, osh, Tt, co, use_omp=True)
                c_ref = energy + di[0] + 20.0 * Tt.sum()
                O.minco_backward(hb, tb, inP, Tt, gC + di[1], gT + di[2])
                worst = max(worst, abs(c[b] - c_ref) / abs(c_ref))
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": nb / dt, "unit": "problems/s", "cores": oc.threads_num, "kind": "port",
                                    "sample": f"{nb} of the {Btot} problems, one at a time: oracle MINCO + OpenMP discrete term (reference loop structure) + oracle adjoint"}
            line["parity"] = {"cost_rel_max_over_sample": worst, "tolerance": 1e-6}
        print(json.dumps(line))
    ev.close()
    if world > 1:
        import torch.distributed as dist
        torch.cuda.synchronize(); dist.barrier(); dist.destroy_process_group()
    return 0


def run_reference_other(args):
    """--impl reference for --workload swept / batch1024: the oracle's OpenMP port on the host cores (rank 0 only)"""
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    cores = usable_cores()
    if args.workload == "swept":
        w, cfg, T, Cc, pts, V, F = swept_workload()
        oc = O.config_from(cfg); oc.threads_num = cores
        sh = O.Shape.mesh(V, F, w["poly_params"], wn_mode=O.WN_BH)
        O.eval_swept(oc, sh, T, Cc, pts[:32], use_omp=True)
        ts = []
        for _ in range(args.steps):
            t0 = time.perf_counter(); O.eval_swept(oc, sh, T, Cc, pts, use_omp=True); ts.append(time.perf_counter() - t0)
        ms = 1e3 * statistics.mean(ts)
        metric, unit, val, sample = "swept_collision_cost_grad_evals_per_s", UNIT, 1e3 / ms, f"each step = the whole workload ({len(pts)} points)"
    else:
        w, cfg, occ, T, Cc, V, F = make_workload(False)
        N0, X = w["pieces"], w["map_dim"]
        oc = O.config_from(cfg); oc.threads_num = cores
        osh = O.Shape.mesh(V, F, w["poly_params"], wn_mode=O.WN_BH)
        xs, heads, tails = batch_problems(2, N0, X)
        ts = []
        for k in range(args.steps):
            b = k % 2
            tau = xs[b, :N0]; Tt = np.where(tau > 0, (0.5 * tau + 1) * tau + 1, 1 / ((0.5 * tau - 1) * tau + 1))
            inP = xs[b, N0:].reshape(-1, 3).T
            hb, tb = heads[b].reshape(3, 3).T, tails[b].reshape(3, 3).T
            t0 = time.perf_counter()
            co, energy, gC, gT = O.minco_forward(hb, tb, inP, Tt)
            di = O.eval_discrete(oc, occ, [0, 0, 0], 1.0, osh, Tt, co, use_omp=True)
            O.minco_backward(hb, tb, inP, Tt, gC + di[1], gT + di[2])
            ts.append(time.perf_counter() - t0)
        ms = 1e3 * statistics.mean(ts) * args.batch_total
        metric, unit, val, sample = "batched_callback_problems_per_s", "problems/s", args.batch_total * 1e3 / ms, f"each step = 1 of the {args.batch_total} problems, time scaled by {args.batch_total}"
        w = {"workload": "BASELINE configs[4]", "problems_total": args.batch_total}
    line = {"impl": "reference", "metric": metric, "value": val, "unit": unit, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": w,
            "cpu_baseline": {"value": val, "unit": unit, "cores": cores, "kind": "port", "sample": sample + f"; {cores} OpenMP threads, reference loop structure"},
            "e2e": {"value": val, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--small", action="store_true", help="tiny workload for plumbing checks (not a bench value)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-lbfgs", action="store_true", help="skip the secondary L-BFGS iterations/s measurement")
    ap.add_argument("--collective", default="peer", choices=["peer", "nccl"], help="N > 1: reduction of the sharded evaluation")
    ap.add_argument("--no-batch", action="store_true", help="skip the batched device-callback measurement (configs[4])")
    ap.add_argument("--batch-per-gpu", type=int, default=128, help="problems per GPU in the batched callback measurement (1024 / 8 GPUs)")
    ap.add_argument("--no-frontend", action="store_true", help="skip the front-end attitude-kernel feasibility measurement")
    ap.add_argument("--no-swept", action="store_true", help="skip the secondary swept-volume (SV-SDF) measurement")
    ap.add_argument("--cpu-budget", type=float, default=20.0)
    ap.add_argument("--ref-pieces", type=int, default=64, help="--impl reference: pieces per step sample (of 64; evenly spread; 64 = the whole workload, ~1-2 s per step)")
    ap.add_argument("--robot", default="mesh", help="mesh (headline) or an analytic shape name, e.g. SmoothIntersection (diagnostic runs)")
    ap.add_argument("--workload", default="discrete", choices=["discrete", "swept", "batch1024"],
                    help="discrete = BASELINE configs[2] (headline); swept = configs[3]; batch1024 = configs[4] — each a strong-scaling workload of its own")
    ap.add_argument("--batch-total", type=int, default=1024, help="--workload batch1024: total problems (sharded over the ranks)")
    ap.add_argument("--lbfgs-iterations", type=int, default=8, help="--workload batch1024: iteration cap of the device-resident L-BFGS measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write cost, gradC and gradT of the last timed step as DIR/<name>.npy "
                                                           "(float64; default discrete workload only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "discrete"):
        ap.error("--dump-outputs applies to the default discrete workload of --impl ours")
    if args.impl == "reference":
        return run_reference(args) if args.workload == "discrete" else run_reference_other(args)
    if args.workload == "swept":
        return run_swept(args)
    if args.workload == "batch1024":
        return run_batch(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
