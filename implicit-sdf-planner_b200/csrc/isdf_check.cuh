// Whole-body trajectory collision check (include/isdf.h, isdf_check_collision): per check sample the clearance
//   c = min(H, min over occupied voxels v inside the body box inflated by H of sdf_robot(R^T (p_v - x)))
// and, per trajectory, the deterministic reduction of those samples into a verdict report. This is the implementation behind the
// call site the reference has but never filled (PlannerManager::generateTraj -> SweptVolumeManager::isTrajCollide, swm:759-767).
//
// Same machinery as the discrete cost path (isdf_discrete.cuh), only the reduction differs: a minimum instead of a hinge sum.
//   * k_check_samples — persistent warps draw check samples from one counter; a warp evaluates the sample's pose (piece_pose),
//     scans the occupied voxels of the world AABB of the inflated body box from the bit-packed map (scan_window / row_bits, 32
//     voxels per pass in (x, y, z) order) and keeps the running minimum with its argmin voxel:
//       - analytic shapes: lane per voxel, closed-form SDF, warp min + argmin at the end of the sample;
//       - exact-sign mesh: BRANCH-AND-BOUND. The warp's running minimum `best` starts at H. Every voxel of a pass gets an exact lower
//         bound on its SDF (distance to the mesh AABB when outside it; the cell record's d_centre - ghd; gpad outside the cell grid).
//         The warp then searches the pass's voxels in ascending bound order, each with reach = best (a voxel farther than best is
//         never resolved to a triangle), and stops as soon as the smallest remaining bound lies STRICTLY above best — so ties are
//         always evaluated and the argmin tie rule holds whatever the order;
//       - winding-sign mesh: s = 1 - 2 w is not ±1, so no distance bound decides anything: every voxel in the box is answered by an
//         unbounded warp-cooperative search, then the signs are evaluated one voxel per lane.
//   * k_check_finish — one CTA per trajectory reduces its samples in (piece, j) order (lexicographic (value, sample) minimum and the
//     smallest hitting sample: exact operations, no floating-point atomics), so the report is independent of scheduling.
// The minimum and its argmin are exact functions of the per-voxel SDF values; the SDF of a voxel does not depend on the reach its search
// was given. Hence the result is bit-identical whatever warp takes which sample, and alone or inside a batch.
//
// Included by isdf_api.cu (launch interface only) and isdf_discrete_tu.cu (ISDF_DISCRETE_TU: the kernels, FMA contract — nothing here
// replays a sequential decision of the reference).
#pragma once
#include "isdf_discrete.cuh"

namespace isdf {

constexpr int CHECK_WARPS = 4;
constexpr int CHECK_THREADS = CHECK_WARPS * 32;
constexpr int CHECK_FIN_THREADS = 256;
constexpr int CHECK_MAX_SAMPLES_PER_PIECE = 4096;
enum { CHECK_ANALYTIC = 0, CHECK_MESH_EXACT = 1, CHECK_MESH_WINDING = 2 };
enum { CHECK_CNT_BOX = 0, CHECK_CNT_SDF = 1, CHECK_CNT_SEARCH = 2, CHECK_NCOUNTERS = 3 };

struct CheckArgs {
    DevCfg cfg;
    DevGrid grid;
    DevShape shape;
    int N;                  // pieces in the block (B * N0)
    int N0;                 // pieces per trajectory
    int M;                  // check intervals per piece: samples j = 0..M
    const double *T;        // N
    const double *C;        // 6N x 3 column-major
    double margin, horizon;
    double *clear;          // N * (M + 1): per-sample clearance
    long long *arg;         // N * (M + 1): linear address of the sample's argmin voxel, -1 = none (c == horizon or NaN)
    int *cursor;            // persistent-warp sample counter (zero on entry; k_check_finish zeroes it again)
    unsigned long long *counters;   // CHECK_NCOUNTERS: voxels in the box, SDF values computed, mesh searches
    unsigned long long *cycles;     // may be null: per-sample clock64 cycles of its warp
    isdf_clearance_report *reports; // B
};

#ifdef ISDF_DISCRETE_TU
// lexicographic (value, linear address) order; address -1 (no voxel) sorts last
__device__ __forceinline__ bool check_better(double v, long long a, double bv, long long ba) {
    return v < bv || (v == bv && (unsigned long long)a < (unsigned long long)ba);
}
__device__ __forceinline__ void check_warp_min(double &v, long long &a) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, v, o);
        const long long oa = __shfl_xor_sync(0xffffffffu, a, o);
        if (check_better(ov, oa, v, a)) { v = ov; a = oa; }
    }
}

// Occupied voxels that can lie in the body box |R^T (p - x)|_inf <= hb: the box's world AABB (half extent hb * sum_k |R(a, k)| per axis),
// one voxel wider on every side, intersected with the map. Voxels outside the map are free, so nothing is clamped INTO the map.
__device__ __forceinline__ bool check_window(const DevGrid &G, d3 pos, const rot3 &R, double hb, Window &W) {
    const double e[3] = {hb * (fabs(R.r0.x) + fabs(R.r0.y) + fabs(R.r0.z)), hb * (fabs(R.r1.x) + fabs(R.r1.y) + fabs(R.r1.z)),
                         hb * (fabs(R.r2.x) + fabs(R.r2.y) + fabs(R.r2.z))};
    const double p[3] = {pos.x, pos.y, pos.z};
    const int n[3] = {G.X, G.Y, G.Z};
    int lo[3], hi[3];
#pragma unroll
    for (int a = 0; a < 3; a++) {
        const double l = floor((p[a] - e[a] - G.bmin[a]) / G.res) - 1.0, h = floor((p[a] + e[a] - G.bmin[a]) / G.res) + 1.0;
        if (!(l <= (double)(n[a] - 1) && h >= 0.0)) return false;   // also false for a non-finite pose
        lo[a] = (int)fmax(l, 0.0); hi[a] = (int)fmin(h, (double)(n[a] - 1));
    }
    W.ix0 = lo[0]; W.ix1 = hi[0]; W.iy0 = lo[1]; W.iy1 = hi[1]; W.iz0 = lo[2]; W.iz1 = hi[2];
    return true;
}

// exact lower bound on the exact-sign mesh SDF at body-frame point p (1-Lipschitz): outside the mesh AABB the SDF is the positive
// distance, which is at least the distance to the AABB; inside the cell grid every point of a cell is >= d_centre - ghd; outside the
// grid at least gpad. The bound is lowered by 1e-12 so that its own rounding can never prune a voxel the definition keeps.
__device__ __forceinline__ double mesh_sdf_lower_bound(const DevMesh &Mh, d3 p, uint4 &rec) {
    const double ax = fmax(fmax(Mh.blo[0] - p.x, p.x - Mh.bhi[0]), 0.0), ay = fmax(fmax(Mh.blo[1] - p.y, p.y - Mh.bhi[1]), 0.0),
                 az = fmax(fmax(Mh.blo[2] - p.z, p.z - Mh.bhi[2]), 0.0);
    const double da = ax * ax + ay * ay + az * az;
    double lb = da > 0.0 ? sqrt(da) : -1e300;
    rec = make_uint4(0u, 0xffffffffu, 0u, 0u);   // {dist bits, seed, off, cnt}; seed 0xffffffff = outside the cell grid
    const int cx = (int)floor((p.x - Mh.glo[0]) * Mh.inv_gcell), cy = (int)floor((p.y - Mh.glo[1]) * Mh.inv_gcell),
              cz = (int)floor((p.z - Mh.glo[2]) * Mh.inv_gcell);
    if (cx < 0 || cy < 0 || cz < 0 || cx >= Mh.gdim[0] || cy >= Mh.gdim[1] || cz >= Mh.gdim[2]) lb = fmax(lb, Mh.gpad);
    else {
        rec = __ldg(Mh.cell_rec + ((size_t)(cx * Mh.gdim[1] + cy) * Mh.gdim[2] + cz));
        lb = fmax(lb, (double)__uint_as_float(rec.x) - Mh.ghd);
    }
    return lb - 1e-12;
}

template <int MODE>
__global__ void __launch_bounds__(CHECK_THREADS) k_check_samples(const __grid_constant__ CheckArgs A) {
    __shared__ WideStack wstk[CHECK_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const DevGrid &G = A.grid;
    const DevMesh &Mh = A.shape.mesh;
    const int M = A.M;
    const long long S = (long long)A.N * (M + 1);
    const double H = A.horizon, hb = A.cfg.half_bd + A.horizon;
    unsigned long long nbox = 0, nsdf = 0, nsearch = 0;
    for (;;) {
        int s = 0;
        if (lane == 0) s = atomicAdd(A.cursor, 1);
        s = __shfl_sync(0xffffffffu, s, 0);
        if (s >= S) break;
        const long long t_begin = A.cycles ? clock64() : 0;
        const int i = s / (M + 1), j = s - i * (M + 1);
        const double step = __ldg(A.T + i) * (1.0 / M);
        d3 pos; quat4 q; rot3 R;
        piece_pose(A.C, A.N, i, j, step, A.cfg.fp, pos, q, R);
        double best = H;        // running minimum (MESH_EXACT: warp-uniform; otherwise per lane until the final warp min)
        long long barg = -1;
        Window W;
        const bool finite = isfinite(pos.x) && isfinite(pos.y) && isfinite(pos.z) && isfinite(R.r0.x) && isfinite(R.r1.y) && isfinite(R.r2.z);
        if (finite && check_window(G, pos, R, hb, W)) {
            scan_window(G, W, lane, [&](bool valid, int vx, int vy, int vz, int) {
                bool inbox = false;
                d3 prel = mk3(0, 0, 0);
                long long addr = -1;
                if (valid) {
                    prel = rot_applyT(R, voxel_centre(G, vx, vy, vz) - pos);
                    inbox = !(fabs(prel.x) > hb || fabs(prel.y) > hb || fabs(prel.z) > hb);
                    addr = ((long long)vx * G.Y + vy) * G.Z + vz;
                }
                const unsigned boxed = __ballot_sync(0xffffffffu, inbox);
                nbox += __popc(boxed);
                if (MODE == CHECK_ANALYTIC) {
                    if (inbox) {
                        const double v = shape_sdf_analytic(A.shape, prel);
                        if (v < H && check_better(v, addr, best, barg)) { best = v; barg = addr; }
                    }
                    nsdf += __popc(boxed);
                } else if (MODE == CHECK_MESH_EXACT) {
                    uint4 rec = make_uint4(0u, 0xffffffffu, 0u, 0u);
                    double lb = 1e300;
                    if (inbox) lb = mesh_sdf_lower_bound(Mh, prel, rec);
                    unsigned live = boxed;
                    while (live) {
                        // the live voxel with the smallest bound (lowest lane among equal bounds)
                        double mlb = ((live >> lane) & 1u) ? lb : 1e300;
                        int src = lane;
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) {
                            const double ol = __shfl_xor_sync(0xffffffffu, mlb, o);
                            const int os = __shfl_xor_sync(0xffffffffu, src, o);
                            if (ol < mlb || (ol == mlb && os < src)) { mlb = ol; src = os; }
                        }
                        if (mlb > best) break;   // every remaining voxel is strictly farther than the running minimum
                        live &= ~(1u << src);
                        const d3 p = mk3(__shfl_sync(0xffffffffu, prel.x, src), __shfl_sync(0xffffffffu, prel.y, src), __shfl_sync(0xffffffffu, prel.z, src));
                        const long long va = __shfl_sync(0xffffffffu, addr, src);
                        const uint32_t cnt = __shfl_sync(0xffffffffu, rec.w, src), off = __shfl_sync(0xffffffffu, rec.z, src);
                        const uint32_t seed = __shfl_sync(0xffffffffu, rec.y, src), dbits = __shfl_sync(0xffffffffu, rec.x, src);
                        const bool inside = seed != 0xffffffffu && __uint_as_float(dbits) < 0.0f;
                        const int first_id = (lane < (int)cnt) ? (int)__ldg(Mh.cand + off + lane) : -1;
                        // reach a hair above best: a voxel whose SDF EQUALS best is still resolved (tie rule)
                        const double reach = best + 1e-12 * (1.0 + fabs(best));
                        double d2; d3 c; int tri, feat;
                        nsearch++;
                        if (mesh_search_rec(Mh, p, reach, lane, &wstk[warp], (int)cnt, off, first_id, seed == 0xffffffffu ? -1 : (int)seed, inside, d2, c, tri, feat)) {
                            d3 g;
                            const double v = mesh_finish_t<false>(Mh, p, p - c, d2, tri, feat, g);
                            nsdf++;
                            if (v < H && check_better(v, va, best, barg)) { best = v; barg = va; }
                        }
                    }
                } else {   // CHECK_MESH_WINDING: every voxel in the box, exactly
                    d3 e = mk3(0, 0, 0); double d2 = 0.0; int tri = -1, feat = 0;
                    unsigned live = boxed;
                    while (live) {
                        const int src = __ffs(live) - 1;
                        live &= live - 1;
                        const d3 p = mk3(__shfl_sync(0xffffffffu, prel.x, src), __shfl_sync(0xffffffffu, prel.y, src), __shfl_sync(0xffffffffu, prel.z, src));
                        uint4 rec;
                        mesh_sdf_lower_bound(Mh, p, rec);   // the bound decides nothing here: only the cell's candidate list and seed are used
                        const int first_id = (lane < (int)rec.w) ? (int)__ldg(Mh.cand + rec.z + lane) : -1;
                        double sd2; d3 c; int st, sf;
                        mesh_search_rec(Mh, p, 1e300, lane, &wstk[warp], (int)rec.w, rec.z, first_id, rec.y == 0xffffffffu ? -1 : (int)rec.y, false, sd2, c, st, sf);
                        nsearch++;
                        if (lane == src) { e = p - c; d2 = sd2; tri = st; feat = sf; }
                    }
                    if (inbox) {
                        d3 g;
                        const double v = mesh_finish_t<true>(Mh, prel, e, d2, tri, feat, g);
                        if (v < H && check_better(v, addr, best, barg)) { best = v; barg = addr; }
                    }
                    nsdf += __popc(boxed);
                }
            });
            if (MODE != CHECK_MESH_EXACT) check_warp_min(best, barg);
        }
        if (!finite) { best = nan(""); barg = -1; }
        if (lane == 0) {
            A.clear[s] = best; A.arg[s] = barg;
            if (A.cycles) A.cycles[s] = (unsigned long long)(clock64() - t_begin);
        }
        __syncwarp();
    }
    if (lane == 0) {
        atomicAdd(A.counters + CHECK_CNT_BOX, nbox);
        atomicAdd(A.counters + CHECK_CNT_SDF, nsdf);
        atomicAdd(A.counters + CHECK_CNT_SEARCH, nsearch);
    }
}

// (value, sample) order of the report's minimum; a NaN sample (non-finite pose) sorts first
__device__ __forceinline__ bool check_sample_less(double v, int k, double bv, int bk) {
    const bool n = isnan(v), bn = isnan(bv);
    if (n != bn) return n;
    if (!n && v != bv) return v < bv;
    return k < bk;
}

__device__ __forceinline__ void check_centre(const DevGrid &G, long long a, double *p) {
    if (a < 0) { p[0] = p[1] = p[2] = nan(""); return; }
    const long long yz = (long long)G.Y * G.Z;
    const int ix = (int)(a / yz), iy = (int)((a - ix * yz) / G.Z), iz = (int)(a - ix * yz - (long long)iy * G.Z);
    const d3 c = voxel_centre(G, ix, iy, iz);
    p[0] = c.x; p[1] = c.y; p[2] = c.z;
}

// trajectory time of local sample k (pieces summed in ascending order, like Trajectory::getTotalDuration)
__device__ __forceinline__ double check_time(const CheckArgs &A, int b, int k, int &piece, int &j) {
    piece = k / (A.M + 1); j = k - piece * (A.M + 1);
    double t = 0.0;
    for (int p = 0; p < piece; p++) t += __ldg(A.T + (size_t)b * A.N0 + p);
    return t + j * (__ldg(A.T + (size_t)b * A.N0 + piece) * (1.0 / A.M));
}

// one CTA per trajectory: minimum in (value, sample) order and the first sample below the margin
__global__ void __launch_bounds__(CHECK_FIN_THREADS) k_check_finish(const __grid_constant__ CheckArgs A) {
    __shared__ double sv[CHECK_FIN_THREADS];
    __shared__ int sk[CHECK_FIN_THREADS], sh[CHECK_FIN_THREADS];
    const int b = blockIdx.x, tid = threadIdx.x;
    const int n = A.N0 * (A.M + 1);
    const size_t base = (size_t)b * n;
    double bv = 0.0; int bk = 0x7fffffff, hk = 0x7fffffff;
    for (int k = tid; k < n; k += CHECK_FIN_THREADS) {
        const double v = __ldcg(A.clear + base + k);
        if (bk == 0x7fffffff || check_sample_less(v, k, bv, bk)) { bv = v; bk = k; }
        if (!(v >= A.margin) && k < hk) hk = k;
    }
    sv[tid] = bv; sk[tid] = bk; sh[tid] = hk;
    __syncthreads();
    for (int w = CHECK_FIN_THREADS / 2; w > 0; w >>= 1) {
        if (tid < w) {
            const double ov = sv[tid + w]; const int ok = sk[tid + w];
            if (ok != 0x7fffffff && (sk[tid] == 0x7fffffff || check_sample_less(ov, ok, sv[tid], sk[tid]))) { sv[tid] = ov; sk[tid] = ok; }
            sh[tid] = min(sh[tid], sh[tid + w]);
        }
        __syncthreads();
    }
    if (tid == 0) {
        isdf_clearance_report r;
        int pc, jj;
        const int k = sk[0];
        r.min_clearance = sv[0];
        r.t_min = check_time(A, b, k, pc, jj);
        r.piece_min = pc; r.sample_min = jj;
        check_centre(A.grid, __ldcg(A.arg + base + k), r.p_min);
        const int h = sh[0];
        r.collides = h != 0x7fffffff;
        if (r.collides) {
            r.t_hit = check_time(A, b, h, pc, jj);
            r.piece_hit = pc; r.sample_hit = jj;
            check_centre(A.grid, __ldcg(A.arg + base + h), r.p_hit);
        } else {
            r.t_hit = -1.0; r.piece_hit = -1; r.sample_hit = -1;
            r.p_hit[0] = r.p_hit[1] = r.p_hit[2] = nan("");
        }
        r.reserved_ = 0;
        A.reports[b] = r;
        if (b == 0) *A.cursor = 0;
    }
}

// failure path of the device entry point: every report reads "not safe"
__global__ void k_check_poison(isdf_clearance_report *reports, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    isdf_clearance_report r;
    r.min_clearance = nan(""); r.t_min = nan(""); r.t_hit = nan("");
    for (int a = 0; a < 3; a++) { r.p_min[a] = nan(""); r.p_hit[a] = nan(""); }
    r.collides = 1; r.piece_min = r.sample_min = r.piece_hit = r.sample_hit = -1; r.reserved_ = 0;
    reports[b] = r;
}
#endif  // ISDF_DISCRETE_TU

// ---- launch interface (isdf_discrete_tu.cu) -----------------------------------------------------------------------------------
// mode: CHECK_ANALYTIC / CHECK_MESH_EXACT / CHECK_MESH_WINDING; B trajectories -> the sample kernel on a persistent grid, then the finisher
cudaError_t check_launch(const CheckArgs &A, int mode, int B, int sm_count, cudaStream_t st);
cudaError_t check_launch_poison(isdf_clearance_report *d_reports, int B, cudaStream_t st);

}  // namespace isdf
