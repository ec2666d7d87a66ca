// Discrete collision cost/gradient kernels: a scan kernel (persistent warps drawing pose-sample work items) and an epilogue kernel
// (thread per sample, CTA per piece) per optimiser step.
//
// Reference semantics: addTimeIntPenaltyParallel (back_end_optimizer.hpp:432-554) with grad_cost_p (hpp:766-824)
// wired into the sample loop exactly as hpp:619-626 wires its swept-volume sibling; PCSmapManager::getPointsInAABB
// (PCSmap_manager.h:148-170); getSDFWithGradWhenRobotAtState (sw_manager.hpp:537-541).
//
// Mapping (B200-first, not the reference's OpenMP-over-samples + critical section):
//   * the pose window is read from the BIT-packed occupancy: lane = (x,y) row, one or two 32-bit loads + funnel shift give the
//     row's z-run; only the occupied voxels are enumerated, in the reference's (x, y, z) order per row, and compacted through a
//     per-warp shared-memory queue so that every cull pass runs on 32 live voxels (the reference tests every voxel and
//     heap-allocates a vector per sample, hpp:787);
//   * PERSISTENT warps draw work items (longest first) from one device counter: a warp that finishes a light sample takes the
//     next item at once instead of idling until its CTA's slowest warp is done;
//   * work items: the per-sample work measured in the previous evaluation (an optimiser moves the trajectory only a little
//     between steps) sorts the samples, and a sample that grazes an obstacle (dozens of mesh queries) is split into 2..32 items,
//     each a contiguous range of the 32 interleaved voxel CLASSES (window voxel (row r, z offset dz) belongs to class (r + 5 dz) % 32).
//     The per-sample sum is
//     ALWAYS formed class by class in the same order, whether one warp walks all classes or 32 warps take one each, so the split
//     never changes a bit of the result;
//   * k_discrete_analytic — two warp-level compaction queues keep lanes dense: queue A = voxels inside the body-frame
//     cull box, queue B = voxels whose hinge is active (sdf < safety_hor) and therefore need the 6 extra finite-
//     difference SDF evaluations of getSDFwithGrad1 (Shape.hpp:58-87). Evaluating those only for active voxels is exact
//     because an inactive voxel contributes nothing (hpp:809-821);
//   * k_discrete_mesh — voxels that survive the exact culls (body-frame box, inflated mesh AABB, per-cell distance lower
//     bound) are answered by WARP-COOPERATIVE nearest-triangle searches (the cell's exact candidate list near the surface, 64
//     candidates per pass with a division-free closest-point test; elsewhere the 32-ary tree seeded with the cell's nearest
//     triangle); sign, gradient, hinge and pose chain rule of the answered voxels are DEFERRED and evaluated one voxel per lane;
//     the warp-uniform pose (position, rotation, quaternion) lives in shared memory, not in 16 x 2 registers of every lane;
//   * k_discrete_epilogue — the per-sample chain rule (penalties, flatness adjoint, beta-basis outer products) as one THREAD
//     per sample, then a deterministic reduction inside the piece's CTA from shared memory: 20 threads add the partials in
//     ascending sample order; the last CTA adds the piece costs in ascending order and (several GPUs) runs the peer-memory
//     exchange — independent of scheduling, so results are bit-reproducible run to run and identical on every rank.
//
// This header is included by two translation units: isdf_api.cu (argument block, host-side constants, the device helpers the
// service kernels share) and isdf_discrete_tu.cu, which defines ISDF_DISCRETE_TU and is the only one that instantiates the
// kernels — compiled WITH FMA contraction, while the swept-volume TU keeps -fmad=false for its sequential decision replay.
#pragma once
#include "isdf_types.cuh"
#include "isdf_peer.cuh"

namespace isdf {

constexpr int DISC_WARPS = 4;
constexpr int DISC_THREADS = DISC_WARPS * 32;
constexpr int QCAP = 64;
constexpr int ROW_CLASSES = 32;         // a pose window's voxels are summed in 32 interleaved classes (canonical order): (row r, z offset dz) -> class (r + 5 dz) % 32
constexpr unsigned SPLIT_WORK_MIN = 256u;  // never split a sample lighter than this (work units: 64 per mesh query + 1 per culled pair)
constexpr int MAX_SPLIT_SLOTS = 16384;  // split samples per launch (2 KB of class sums each)
constexpr int WINDOW_AXIS_MAX = 1023;   // voxels per window axis: window offsets are packed 10 bits per axis
// CTAs per SM the register allocator must leave room for — A/B-measured on B200 (profiles/r01_tuning.md, r02_tuning.md)
constexpr int ANALYTIC_MIN_BLOCKS = 4;
#ifndef ISDF_MESH_MIN_BLOCKS
#define ISDF_MESH_MIN_BLOCKS 4
#endif
constexpr int MESH_MIN_BLOCKS = ISDF_MESH_MIN_BLOCKS;
constexpr int EPI_THREADS = 288;
constexpr int ITEMS_CACHE = 24;   // k_build_items: samples per thread whose work value is kept in registers (M <= 24576: any single trajectory)

struct DiscArgs {
    DevCfg cfg;
    DevGrid grid;
    DevShape shape;
    int N;
    const double *T;       // N
    const double *C;       // 6N x 3 column-major
    double *tot;           // S x 8: collision sums of a sample evaluated as ONE work item {costp, gradp(3), grad_quat(4)}
    int *pieces_done;      // 1  (zero on entry, zero on exit)
    double *piece_cost;    // N
    double *out;           // 19N+1: cost | gradC | gradT
    unsigned long long *pair_counter;  // may be null
    double *count_out;                 // host entry point only: the pair count (bit pattern) lands behind the result vector, one D2H copy fetches both
    unsigned long long *dbg;           // may be null: per sample {cycles, pairs, work}
    unsigned long long *trace;         // may be null: per work-item slot {begin, end} in ns of the global timer (+ 6 phase cycle counts with -DISDF_PHASE_TIMING)
    const int *items;                  // may be null: 3 ints per work item {local sample m, -1 = all classes or c0 | c1 << 8, split slot or -1}
    const int *item_count;             // number of valid items (device)
    int *item_cursor;                  // persistent warps draw items from this counter (zero on entry; the epilogue zeroes it again)
    double *subsum;                    // split slot x ROW_CLASSES x 8 class sums
    unsigned *split_work;              // split slot -> work accumulated by the parts (zero on entry, zeroed by the sample's last part)
    unsigned *split_done;              // split slot -> parts finished (zero on entry, zeroed by the sample's last part)
    unsigned *work;                    // may be null: per global sample, work measure written for the next evaluation
    int rank, world;       // this launch evaluates samples s with s % world == rank
    PeerArgs peer;         // peer.world > 1: the epilogue's last CTA also sums `out` over the ranks through peer memory (isdf_peer.cuh)
};

struct PairAcc { double c, gx, gy, gz, q0, q1, q2, q3; };

// hpp:809-821 for one (pose, voxel) pair
__device__ __forceinline__ void pair_accumulate(const DevCfg &cfg, const rot3 &R, quat4 q, d3 d, double sdf, d3 g, PairAcc &a) {
    double f, df;
    hinge(cfg.safety - sdf, cfg.mu, f, df);
    if (f > 0.0) {
        a.c += f;
        const d3 wg = rot_apply(R, g);
        a.gx += df * wg.x; a.gy += df * wg.y; a.gz += df * wg.z;
        double jq[4];
        quat_pull(q, g, d, jq);
        a.q0 += -df * jq[0]; a.q1 += -df * jq[1]; a.q2 += -df * jq[2]; a.q3 += -df * jq[3];
    }
}

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
__device__ __forceinline__ double clampr(double v, double lo, double hi) { return v < lo ? lo : (v > hi ? hi : v); }

// GridMap3D::getGridIndex after PCSmapManager::projInMap (Gridmap3D.cpp:135-175, PCSmap_manager.h:130-137)
__device__ __forceinline__ int grid_axis_index(double coord, double bmin, double bmax, double res, int size) {
    const double c = clampr(coord, bmin, bmax);
    return clampi((int)floor((c - bmin) / res), 0, size - 1);
}

struct Window { int ix0, ix1, iy0, iy1, iz0, iz1; };

__device__ __forceinline__ Window window_of(const DevGrid &G, d3 pos, double h) {
    Window w;
    w.ix0 = grid_axis_index(pos.x - h, G.bmin[0], G.bmax[0], G.res, G.X);
    w.ix1 = grid_axis_index(pos.x + h, G.bmin[0], G.bmax[0], G.res, G.X);
    w.iy0 = grid_axis_index(pos.y - h, G.bmin[1], G.bmax[1], G.res, G.Y);
    w.iy1 = grid_axis_index(pos.y + h, G.bmin[1], G.bmax[1], G.res, G.Y);
    w.iz0 = grid_axis_index(pos.z - h, G.bmin[2], G.bmax[2], G.res, G.Z);
    w.iz1 = grid_axis_index(pos.z + h, G.bmin[2], G.bmax[2], G.res, G.Z);
    return w;
}
__device__ __forceinline__ d3 voxel_centre(const DevGrid &G, int ix, int iy, int iz) {   // getGridCubeCenter (Gridmap3D.cpp:177-194)
    return mk3((ix + 0.5) * G.res + G.bmin[0], (iy + 0.5) * G.res + G.bmin[1], (iz + 0.5) * G.res + G.bmin[2]);
}

// one window row's z-run [zs, zs + nzc) as a bit mask (bit k = voxel zs + k)
__device__ __forceinline__ uint32_t row_bits(const DevGrid &G, int ix, int iy, int zs, uint32_t zmask) {
    const uint32_t *row = G.bits + ((size_t)ix * G.Y + iy) * G.Zw;
    const int wz = zs >> 5, sh = zs & 31;
    const uint32_t lo = __ldg(row + wz);
    const uint32_t hi = (sh != 0 && wz + 1 < G.Zw) ? __ldg(row + wz + 1) : 0u;
    return __funnelshift_r(lo, hi, sh) & zmask;
}

// Enumerate the occupied voxels of a window, 32 at a time, in the reference's order (x, then y, then z ascending).
// visit(valid, ix, iy, iz, r) is called by the whole warp; lanes without a voxel pass valid = false. (analytic kernel)
template <class Visit>
__device__ __forceinline__ void scan_window(const DevGrid &G, const Window &W, int lane, Visit &&visit) {
    const int ny = W.iy1 - W.iy0 + 1;
    const int nrows = (W.ix1 - W.ix0 + 1) * ny;
    for (int zs = W.iz0; zs <= W.iz1; zs += 32) {
        const int nzc = min(32, W.iz1 - zs + 1);
        const uint32_t zmask = (nzc == 32) ? 0xffffffffu : ((1u << nzc) - 1u);
        for (int rb = 0; rb < nrows; rb += 32) {
            const int r = rb + lane;
            uint32_t bits = 0;
            int rx = 0, ry = 0;
            if (r < nrows) {
                rx = r / ny; ry = r - rx * ny;
                bits = row_bits(G, W.ix0 + rx, W.iy0 + ry, zs, zmask);
            }
            const int cnt = __popc(bits);
            int incl = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
            const int total = __shfl_sync(0xffffffffu, incl, 31);
            for (int base = 0; base < total; base += 32) {
                const int kk = base + lane;
                // source lane = number of lanes whose inclusive count is <= kk (binary search over the scan)
                int src = 0;
#pragma unroll
                for (int stp = 16; stp > 0; stp >>= 1) {
                    const int probe = src + stp - 1;
                    const int v = __shfl_sync(0xffffffffu, incl, probe & 31);
                    if (probe < 32 && v <= kk) src += stp;
                }
                src = min(src, 31);
                const int s_incl = __shfl_sync(0xffffffffu, incl, src);
                const int s_cnt = __shfl_sync(0xffffffffu, cnt, src);
                uint32_t s_bits = __shfl_sync(0xffffffffu, bits, src);
                const int s_rx = __shfl_sync(0xffffffffu, rx, src), s_ry = __shfl_sync(0xffffffffu, ry, src);
                const int s_r = __shfl_sync(0xffffffffu, r, src);
                const bool valid = kk < total;
                int bz = 0;
                if (valid) {
                    // position of the nth set bit: clear the n lowest set bits, then find-first-set
                    int nth = kk - (s_incl - s_cnt);
                    while (nth-- > 0) s_bits &= s_bits - 1;
                    bz = __ffs(s_bits) - 1;
                }
                visit(valid, W.ix0 + s_rx, W.iy0 + s_ry, zs + bz, s_r);
            }
        }
    }
}

// pose of piece i of the 6N x 3 column-major block C at local time j * step: position, flatness quaternion, rotation (hpp:456-492)
__device__ __forceinline__ void piece_pose(const double *C, int N, int i, int j, double step, const FlatParams &fp, d3 &pos, quat4 &q, rot3 &R) {
    double cx[6], cy[6], cz[6];
#pragma unroll
    for (int k = 0; k < 6; k++) {
        cx[k] = __ldg(C + 6 * i + k);
        cy[k] = __ldg(C + 6 * N + 6 * i + k);
        cz[k] = __ldg(C + 12 * N + 6 * i + k);
    }
    PieceEval pe;
    piece_eval(cx, cy, cz, j * step, pe);
    q = flat_quat_only(fp, pe.vel, pe.acc);
    pos = pe.pos;
    R = quat_rot(q);
}
// pose of sample (i, j)
__device__ __forceinline__ void sample_pose(const DiscArgs &A, int i, int j, double step, d3 &pos, quat4 &q, rot3 &R) {
    piece_pose(A.C, A.N, i, j, step, A.cfg.fp, pos, q, R);
}

// hpp:505-551 for one sample given the reduced collision sums; writes the 20 per-sample partials to st[]
__device__ __forceinline__ void sample_epilogue(const DiscArgs &A, int i, int j, double Ti, double costp, d3 gp,
                                                double gq0, double gq1, double gq2, double gq3, double *st) {
    const DevCfg &cfg = A.cfg;
    const int K = cfg.K;
    const double frac = 1.0 / K;
    const double step = Ti * frac;
    double cx[6], cy[6], cz[6];
#pragma unroll
    for (int k = 0; k < 6; k++) {
        cx[k] = __ldg(A.C + 6 * i + k);
        cy[k] = __ldg(A.C + 6 * A.N + 6 * i + k);
        cz[k] = __ldg(A.C + 12 * A.N + 6 * i + k);
    }
    PieceEval pe;
    piece_eval(cx, cy, cz, j * step, pe);
    FlatState fs;
    flat_state(cfg.fp, pe.vel, pe.acc, pe.jer, fs);
    const quat4 q = flat_quat(fs);
    const d3 omg = flat_omega(fs);
    double pena = 0.0;
    d3 gradVel = mk3(0, 0, 0), gradOmg = mk3(0, 0, 0), gradPos = mk3(0, 0, 0);
    double gradQuat[4] = {0, 0, 0, 0};
    if (cfg.flags & ISDF_WITH_DYNAMICS) {
        const double cos_theta = 1.0 - 2.0 * (q.x * q.x + q.y * q.y);
        double f, df;
        if (hinge(dot3(pe.vel, pe.vel) - cfg.vmax2, cfg.mu, f, df)) {
            const double sc = cfg.wv * df * 2.0;
            gradVel = mk3(sc * pe.vel.x, sc * pe.vel.y, sc * pe.vel.z); pena += cfg.wv * f;
        }
        if (hinge(dot3(omg, omg) - cfg.omgmax2, cfg.mu, f, df)) {
            const double sc = cfg.womg * df * 2.0;
            gradOmg = mk3(sc * omg.x, sc * omg.y, sc * omg.z); pena += cfg.womg * f;
        }
        if (hinge(acos(cos_theta) - cfg.thetamax, cfg.mu, f, df)) {
            const double sc = cfg.wtheta * df / sqrt(1.0 - cos_theta * cos_theta) * 4.0;
            gradQuat[1] += sc * q.x; gradQuat[2] += sc * q.y; pena += cfg.wtheta * f;
        }
    }
    if (costp > 0.0) {  // grad_cost_p returns (costp > 0), hpp:823
        gradPos = mk3(cfg.wp * gp.x, cfg.wp * gp.y, cfg.wp * gp.z);
        gradQuat[0] += cfg.wp * gq0; gradQuat[1] += cfg.wp * gq1; gradQuat[2] += cfg.wp * gq2; gradQuat[3] += cfg.wp * gq3;
        pena += cfg.wp * costp;
    }
    d3 gV, gA, gJ;
    flat_adjoint(cfg.fp, fs, pe.vel, pe.acc, gradQuat, gradOmg, gradVel, gV, gA, gJ);
    const d3 gP = gradPos;
    const double node = (j == 0 || j == K) ? 0.5 : 1.0;
    const double alpha = j * frac;
    const double w = node * step;
#pragma unroll
    for (int k = 0; k < 6; k++) {
        st[k] = (pe.b0[k] * gP.x + pe.b1[k] * gV.x + pe.b2[k] * gA.x + pe.b3[k] * gJ.x) * w;
        st[6 + k] = (pe.b0[k] * gP.y + pe.b1[k] * gV.y + pe.b2[k] * gA.y + pe.b3[k] * gJ.y) * w;
        st[12 + k] = (pe.b0[k] * gP.z + pe.b1[k] * gV.z + pe.b2[k] * gA.z + pe.b3[k] * gJ.z) * w;
    }
    st[18] = (dot3(gP, pe.vel) + dot3(gV, pe.acc) + dot3(gA, pe.jer) + dot3(gJ, pe.sna)) * alpha * node * step + node * frac * pena;
    st[19] = node * step * pena;
}

// ============================================================================================================================
// Work item of a warp: {global sample, first class, one-past-last class, split slot}.
struct Item { int s, c0, c1, hslot, slot; };
__device__ __forceinline__ unsigned long long global_ns() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#ifdef ISDF_PHASE_TIMING
constexpr int TRACE_STRIDE = 8;
#define ISDF_PT(x) x
#else
constexpr int TRACE_STRIDE = 2;
#define ISDF_PT(x)
#endif

// Persistent-warp scheduler: the warp's next work item, or false when the table is exhausted. Which warp takes which item
// never touches the arithmetic, so results stay bit-reproducible.
__device__ __forceinline__ bool next_item(const DiscArgs &A, Item &it, int lane) {
    const int K = A.cfg.K;
    const int S = A.N * (K + 1);
    const int M = (S - A.rank + A.world - 1) / A.world;   // local samples; local m -> global s = rank + world * m
    int slot = 0;
    if (lane == 0) slot = atomicAdd(A.item_cursor, 1);
    slot = __shfl_sync(0xffffffffu, slot, 0);
    it.slot = slot;
    if (A.items) {
        if (slot >= __ldg(A.item_count)) return false;
        const int m = __ldg(A.items + 3 * slot), part = __ldg(A.items + 3 * slot + 1);
        it.s = A.rank + A.world * m;
        it.c0 = part < 0 ? 0 : (part & 0xff); it.c1 = part < 0 ? ROW_CLASSES : (part >> 8);
        it.hslot = __ldg(A.items + 3 * slot + 2);
        return true;
    }
    if (slot >= M) return false;
    it.s = A.rank + A.world * slot; it.c0 = 0; it.c1 = ROW_CLASSES; it.hslot = -1;
    return true;
}

// Shared tail of both scan kernels for an item that covers the WHOLE sample: lanes 0..7 hold the eight collision sums.
// The per-sample chain rule and the per-piece reduction run afterwards in k_discrete_epilogue with one THREAD per sample.
__device__ __forceinline__ void sample_finish_whole(const DiscArgs &A, const Item &it, double mine, unsigned npairs, long long t_begin, unsigned work) {
    const int lane = threadIdx.x & 31;
    const int s = it.s;
    if (lane < 8) A.tot[(size_t)s * 8 + lane] = mine;
    if (lane == 0) {
        if (A.pair_counter && npairs) atomicAdd(A.pair_counter, (unsigned long long)npairs);
        if (A.work) A.work[s] = work;
        if (A.dbg) { A.dbg[3 * (size_t)s] = (unsigned long long)(clock64() - t_begin); A.dbg[3 * (size_t)s + 1] = npairs; A.dbg[3 * (size_t)s + 2] = work; }
    }
}

#ifdef ISDF_DISCRETE_TU
// ============================================================================================================================
// One CTA per piece, one thread per pose sample of the piece: hpp:505-551 (dynamic penalties, flatness adjoint, chain rule onto the
// piece's 6x3 coefficients and its duration), then the deterministic per-piece reduction — the samples' 20 partials are staged in
// shared memory and 20 threads, one per output component, add them in ascending sample order — and, in the last CTA to finish,
// the total cost in ascending piece order.
__global__ void __launch_bounds__(EPI_THREADS) k_discrete_epilogue(const __grid_constant__ DiscArgs A) {
    __shared__ double sp[PARTIAL_STRIDE][EPI_THREADS + 1];   // component-major, padded: conflict-free writes, <= 2-way reads
    const int K = A.cfg.K, N = A.N, i = blockIdx.x;
    const int first_s = i * (K + 1), last_s = first_s + K;
    const int f0 = first_s + ((A.rank - first_s) % A.world + A.world) % A.world;  // first local sample >= first_s
    const int local_cnt = (f0 > last_s) ? 0 : ((last_s - f0) / A.world + 1);
    const double Ti = __ldg(A.T + i);
    double run = 0.0;   // threads 0..19: running sum of output component threadIdx.x
    for (int chunk = 0; chunk < local_cnt; chunk += EPI_THREADS) {
        const int idx = chunk + threadIdx.x;
        if (idx < local_cnt) {
            const int s = f0 + idx * A.world;
            const int j = s - first_s;
            double tot[8];   // the sample's collision sums (a split sample's row was finished by its last part, in class order)
            {
                const double2 *tp = reinterpret_cast<const double2 *>(A.tot + (size_t)s * 8);
                const double2 t0 = __ldcg(tp), t1 = __ldcg(tp + 1), t2 = __ldcg(tp + 2), t3 = __ldcg(tp + 3);
                tot[0] = t0.x; tot[1] = t0.y; tot[2] = t1.x; tot[3] = t1.y; tot[4] = t2.x; tot[5] = t2.y; tot[6] = t3.x; tot[7] = t3.y;
            }
            double st[PARTIAL_STRIDE];
            sample_epilogue(A, i, j, Ti, tot[0], mk3(tot[1], tot[2], tot[3]), tot[4], tot[5], tot[6], tot[7], st);
#pragma unroll
            for (int v = 0; v < PARTIAL_STRIDE; v++) sp[v][threadIdx.x] = st[v];
        }
        __syncthreads();
        if (threadIdx.x < PARTIAL_STRIDE) {
            const int n = min(EPI_THREADS, local_cnt - chunk);
            const double *row = sp[threadIdx.x];
            int k = 0;
            for (; k + 8 <= n; k += 8) {   // 8 loads in flight per step; the additions stay in ascending-sample order
                double v[8];
#pragma unroll
                for (int u = 0; u < 8; u++) v[u] = row[k + u];
#pragma unroll
                for (int u = 0; u < 8; u++) run += v[u];
            }
            for (; k < n; k++) run += row[k];
        }
        __syncthreads();
    }
    if (threadIdx.x < PARTIAL_STRIDE) {
        const int comp = threadIdx.x;
        if (comp < 18) { const int ax = comp / 6, k = comp - 6 * ax; A.out[1 + (size_t)ax * 6 * N + 6 * i + k] = run; }
        else if (comp == 18) A.out[1 + 18 * N + i] = run;
        else A.piece_cost[i] = run;
    }
    // last CTA to finish: total cost = piece costs added in ascending order, then (multi-GPU) the exchange over peer memory
    __shared__ int s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(A.pieces_done, 1) == N - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    if (threadIdx.x < 32) {
        const int lane = threadIdx.x;
        double c = 0.0;
        for (int base = 0; base < N; base += 32) {
            const double v = (base + lane < N) ? __ldcg(A.piece_cost + base + lane) : 0.0;
            for (int u = 0; u < 32 && base + u < N; u++) c += __shfl_sync(0xffffffffu, v, u);
        }
        if (lane == 0) {
            A.out[0] = c; *A.pieces_done = 0; *A.item_cursor = 0;
            if (A.count_out) *A.count_out = __longlong_as_double(A.pair_counter ? (long long)*(volatile unsigned long long *)A.pair_counter : 0ll);
        }
    }
    if (A.peer.world > 1) {
        __threadfence();
        __syncthreads();
        peer_allreduce_block(A.peer, A.out, 19 * N + 1);
    }
}

// ============================================================================================================================
// analytic shapes
__global__ void __launch_bounds__(DISC_THREADS, ANALYTIC_MIN_BLOCKS) k_discrete_analytic(const __grid_constant__ DiscArgs A) {
    __shared__ uint32_t qA[DISC_WARPS][QCAP];
    __shared__ uint32_t qB[DISC_WARPS][QCAP];
    __shared__ double qBs[DISC_WARPS][QCAP];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    const DevCfg &cfg = A.cfg;
    const int K = cfg.K;
    Item it;
    while (next_item(A, it, lane)) {
        const int s = it.s;
        const int i = s / (K + 1), j = s - i * (K + 1);
        const double Ti = __ldg(A.T + i);
        const double step = Ti * (1.0 / K);
        const long long t_begin = A.dbg ? clock64() : 0;

        d3 pos; quat4 q; rot3 R;
        sample_pose(A, i, j, step, pos, q, R);

        double mine = 0.0;
        unsigned npairs = 0;

        if (cfg.flags & ISDF_WITH_COLLISION) {
            const DevGrid &G = A.grid;
            const double h = cfg.half_bd;
            const Window W = window_of(G, pos, h);
            PairAcc acc = {0, 0, 0, 0, 0, 0, 0, 0};
            int nA = 0, nB = 0;  // queue fill (warp-uniform)

            auto entry_centre = [&](uint32_t e) { return voxel_centre(G, W.ix0 + (int)(e & 0x3ffu), W.iy0 + (int)((e >> 10) & 0x3ffu), W.iz0 + (int)(e >> 20)); };
            // queue B consumer: finite-difference gradient + accumulation for `cnt` active voxels
            auto drain_B = [&](int cnt) {
                if (lane < cnt) {
                    const double sdf = qBs[warp][lane];
                    const d3 d = entry_centre(qB[warp][lane]) - pos;
                    const d3 prel = rot_applyT(R, d);
                    const d3 g = shape_grad_analytic(A.shape, prel, sdf);
                    pair_accumulate(cfg, R, q, d, sdf, g, acc);
                }
                __syncwarp();
                const int rest = nB - cnt;
                uint32_t e2 = 0; double s2 = 0;
                if (lane < rest) { e2 = qB[warp][cnt + lane]; s2 = qBs[warp][cnt + lane]; }
                __syncwarp();
                if (lane < rest) { qB[warp][lane] = e2; qBs[warp][lane] = s2; }
                __syncwarp();
                nB = rest;
            };
            // queue A consumer: SDF for `cnt` voxels inside the cull box
            auto drain_A = [&](int cnt) {
                bool active = false; uint32_t e = 0; double sdf = 0.0;
                if (lane < cnt) {
                    e = qA[warp][lane];
                    const d3 prel = rot_applyT(R, entry_centre(e) - pos);
                    sdf = shape_sdf_analytic(A.shape, prel);
                    active = (cfg.safety - sdf) > 0.0;
                }
                __syncwarp();
                const int rest = nA - cnt;
                uint32_t e2 = 0;
                if (lane < rest) e2 = qA[warp][cnt + lane];
                __syncwarp();
                if (lane < rest) qA[warp][lane] = e2;
                nA = rest;
                const unsigned bal = __ballot_sync(0xffffffffu, active);
                if (active) { const int p = nB + __popc(bal & lt_mask); qB[warp][p] = e; qBs[warp][p] = sdf; }
                nB += __popc(bal);
                __syncwarp();
                if (nB >= 32) drain_B(32);
            };

            scan_window(G, W, lane, [&](bool valid, int vx, int vy, int vz, int) {
                bool pass = false;
                if (valid) {
                    const d3 prel = rot_applyT(R, voxel_centre(G, vx, vy, vz) - pos);
                    pass = !(fabs(prel.x) > h || fabs(prel.y) > h || fabs(prel.z) > h);  // hpp:800
                }
                const unsigned bal = __ballot_sync(0xffffffffu, pass);
                npairs += __popc(bal);
                if (pass) qA[warp][nA + __popc(bal & lt_mask)] = (uint32_t)(vx - W.ix0) | ((uint32_t)(vy - W.iy0) << 10) | ((uint32_t)(vz - W.iz0) << 20);
                nA += __popc(bal);
                __syncwarp();
                if (nA >= 32) drain_A(32);
            });
            if (nA > 0) drain_A(nA);
            if (nB > 0) drain_B(nB);
            // xor butterfly: fixed order (analytic samples are never split: their work is near-uniform)
            const double t0 = warp_sum(acc.c), t1 = warp_sum(acc.gx), t2 = warp_sum(acc.gy), t3 = warp_sum(acc.gz);
            const double t4 = warp_sum(acc.q0), t5 = warp_sum(acc.q1), t6 = warp_sum(acc.q2), t7 = warp_sum(acc.q3);
            mine = lane == 0 ? t0 : lane == 1 ? t1 : lane == 2 ? t2 : lane == 3 ? t3 : lane == 4 ? t4 : lane == 5 ? t5 : lane == 6 ? t6 : t7;
        }
        sample_finish_whole(A, it, mine, npairs, t_begin, npairs);
        __syncwarp();
    }
}

// ============================================================================================================================
// mesh shapes
struct QRes { double ex, ey, ez; int tri; uint32_t code; int fc; };   // an answered voxel awaiting its deferred tail: e = p - closest point, triangle, voxel code, feature | class << 8 (40 bytes: with the float bounds of WideStack the kernel's shared memory fits the 132 KB carve-out at 4 CTAs/SM, i.e. 124 KB of L1 instead of 92)
struct Survivor { double px, py, pz; uint32_t off, cnt, seed, code; };   // a voxel that passed the exact culls: body-frame point, its cell's list (cnt bit 31: cell centre inside), seed triangle (0xffffffff: none)
struct MeshWarpSmem {
    double pose[16];                     // warp-uniform pose: pos 0..2, R rows 3..11, q (w, x, y, z) 12..15
    double cacc[ROW_CLASSES][8];         // class accumulators
    double vals[32][8];                  // deferred tails: one voxel's eight contributions per lane
    QRes qr[32];
    Survivor sv[32];                     // culled voxels awaiting their search
    uint32_t vq[64];                     // ring of occupied-voxel codes (dx | dy << 10 | dz << 20, relative to the window origin)
    WideStack stk;
};

__device__ __forceinline__ d3 smem_pos(const double *ps) { return mk3(ps[0], ps[1], ps[2]); }
__device__ __forceinline__ rot3 smem_rot(const double *ps) {
    rot3 R; R.r0 = mk3(ps[3], ps[4], ps[5]); R.r1 = mk3(ps[6], ps[7], ps[8]); R.r2 = mk3(ps[9], ps[10], ps[11]); return R;
}
// r / ny for 0 <= r < 2^20, 1 <= ny <= 1023 without an integer division: float estimate + one correction step
__device__ __forceinline__ void row_split(int r, int ny, float inv_ny, int &rx, int &ry) {
    rx = (int)(((float)r + 0.5f) * inv_ny);
    ry = r - rx * ny;
    if (ry < 0) { rx--; ry += ny; } else if (ry >= ny) { rx++; ry -= ny; }
}

template <bool WINDING>
__global__ void __launch_bounds__(DISC_THREADS, MESH_MIN_BLOCKS) k_discrete_mesh(const __grid_constant__ DiscArgs A) {
    __shared__ MeshWarpSmem wsm[DISC_WARPS];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    const DevCfg &cfg = A.cfg;
    const DevMesh &Mh = A.shape.mesh;
    const DevGrid &G = A.grid;
    const int K = cfg.K;
    MeshWarpSmem &sm = wsm[warp];
    const double h = cfg.half_bd, sf = cfg.safety;
    Item it;
    while (next_item(A, it, lane)) {
        const int s = it.s;
        const int i = s / (K + 1), j = s - i * (K + 1);
        const long long t_begin = A.dbg ? clock64() : 0;
        if (A.trace && lane == 0) A.trace[TRACE_STRIDE * (size_t)it.slot] = global_ns();
        ISDF_PT(long long pt_pose = 0; long long pt_cull = 0; long long pt_search = 0; long long pt_tail = 0; long long pt_t0 = clock64(); long long pt_all0 = pt_t0;)
        unsigned npairs = 0, nquery = 0;
        const bool whole = (it.c1 - it.c0) == ROW_CLASSES;

        if (cfg.flags & ISDF_WITH_COLLISION) {
            Window W;
            {   // pose -> shared memory (every lane computes the same values; lane 0 publishes them)
                const double Ti = __ldg(A.T + i);
                d3 pos; quat4 q; rot3 R;
                sample_pose(A, i, j, Ti * (1.0 / K), pos, q, R);
                W = window_of(G, pos, h);
                if (lane == 0) {
                    double *ps = sm.pose;
                    ps[0] = pos.x; ps[1] = pos.y; ps[2] = pos.z;
                    ps[3] = R.r0.x; ps[4] = R.r0.y; ps[5] = R.r0.z; ps[6] = R.r1.x; ps[7] = R.r1.y; ps[8] = R.r1.z;
                    ps[9] = R.r2.x; ps[10] = R.r2.y; ps[11] = R.r2.z;
                    ps[12] = q.w; ps[13] = q.x; ps[14] = q.y; ps[15] = q.z;
                }
            }
            for (int k = lane; k < ROW_CLASSES * 8; k += 32) (&sm.cacc[0][0])[k] = 0.0;
            __syncwarp();
            ISDF_PT(pt_pose = clock64() - pt_t0;)
            const int ny = W.iy1 - W.iy0 + 1;
            const int nrows = (W.ix1 - W.ix0 + 1) * ny;
            const float inv_ny = 1.0f / (float)ny;
            int nq = 0, head = 0, nres = 0;   // voxel ring fill / head, answered voxels awaiting their tail (warp-uniform)

            // deferred tails: sign, gradient, hinge, chain rule onto (position, quaternion) — one answered voxel per lane; the
            // contributions are then added to the class accumulators in voxel order by lanes 0..7 (one per component)
            auto flush_tails = [&]() __attribute__((always_inline)) {
                __syncwarp();
                ISDF_PT(const long long pt_a = clock64();)
                bool active = false;
                if (lane < nres) {
                    const QRes r = sm.qr[lane];
                    d3 g = mk3(0, 0, 0);
                    const double *ps = sm.pose;
                    const d3 d = voxel_centre(G, W.ix0 + (int)(r.code & 0x3ffu), W.iy0 + (int)((r.code >> 10) & 0x3ffu), W.iz0 + (int)(r.code >> 20)) - smem_pos(ps);
                    const double sdf = mesh_finish_t<WINDING>(Mh, rot_applyT(smem_rot(ps), d), mk3(r.ex, r.ey, r.ez), r.ex * r.ex + r.ey * r.ey + r.ez * r.ez, r.tri, r.fc & 0xff, g);
                    quat4 q; q.w = ps[12]; q.x = ps[13]; q.y = ps[14]; q.z = ps[15];
                    PairAcc one = {0, 0, 0, 0, 0, 0, 0, 0};
                    pair_accumulate(cfg, smem_rot(ps), q, d, sdf, g, one);
                    active = one.c > 0.0;
                    double *v = sm.vals[lane];
                    v[0] = one.c; v[1] = one.gx; v[2] = one.gy; v[3] = one.gz; v[4] = one.q0; v[5] = one.q1; v[6] = one.q2; v[7] = one.q3;
                }
                unsigned act = __ballot_sync(0xffffffffu, active);
                __syncwarp();
                if (lane < 8) {
                    while (act) {
                        const int k = __ffs(act) - 1;
                        act &= act - 1;
                        sm.cacc[sm.qr[k].fc >> 8][lane] += sm.vals[k][lane];
                    }
                }
                __syncwarp();
                nres = 0;
                ISDF_PT(pt_tail += clock64() - pt_a;)
            };

            int nsv = 0;   // queued survivors (warp-uniform)
            // cull stage for the n oldest voxels of the ring (n <= 32): survivors are appended to the survivor queue
            auto cull = [&](int n) __attribute__((always_inline)) {
                ISDF_PT(const long long pt_a = clock64();)
                bool pass = false, box = false;
                uint32_t code = 0;
                d3 prel = mk3(0, 0, 0);
                uint4 rec = make_uint4(0u, 0xffffffffu, 0u, 0u);   // {dist bits, seed, off, cnt}; seed 0xffffffff = outside the cell grid
                if (lane < n) {
                    code = sm.vq[(head + lane) & 63];
                    const double *ps = sm.pose;
                    const d3 d = voxel_centre(G, W.ix0 + (int)(code & 0x3ffu), W.iy0 + (int)((code >> 10) & 0x3ffu), W.iz0 + (int)(code >> 20)) - smem_pos(ps);
                    prel = rot_applyT(smem_rot(ps), d);
                    box = !(fabs(prel.x) > h || fabs(prel.y) > h || fabs(prel.z) > h);  // hpp:800
                    // exact skips: outside the mesh AABB inflated by safety_hor, or in a cell whose every point is >= safety_hor away
                    // (with the un-thresholded winding sign s = 1 - 2 w no distance bound decides the hinge: every voxel in the box is answered)
                    constexpr bool wn = WINDING;
                    pass = box && (wn || !(prel.x < Mh.blo[0] - sf || prel.x > Mh.bhi[0] + sf || prel.y < Mh.blo[1] - sf || prel.y > Mh.bhi[1] + sf ||
                                           prel.z < Mh.blo[2] - sf || prel.z > Mh.bhi[2] + sf));
                    if (pass) {
                        const int cx = (int)floor((prel.x - Mh.glo[0]) * Mh.inv_gcell), cy = (int)floor((prel.y - Mh.glo[1]) * Mh.inv_gcell),
                                  cz = (int)floor((prel.z - Mh.glo[2]) * Mh.inv_gcell);
                        if (cx < 0 || cy < 0 || cz < 0 || cx >= Mh.gdim[0] || cy >= Mh.gdim[1] || cz >= Mh.gdim[2]) pass = wn || !(sf <= Mh.gpad);   // outside the grid: >= gpad away
                        else {
                            rec = __ldg(Mh.cell_rec + ((size_t)(cx * Mh.gdim[1] + cy) * Mh.gdim[2] + cz));
                            pass = wn || !((double)__uint_as_float(rec.x) - Mh.ghd >= sf);
                        }
                    }
                }
                head = (head + n) & 63; nq -= n;
                npairs += __popc(__ballot_sync(0xffffffffu, box));
                const unsigned bal = __ballot_sync(0xffffffffu, pass);
                if (pass) {
                    Survivor &v = sm.sv[nsv + __popc(bal & lt_mask)];
                    v.px = prel.x; v.py = prel.y; v.pz = prel.z; v.off = rec.z; v.seed = rec.y; v.code = code;
                    v.cnt = rec.w | ((rec.y != 0xffffffffu && __uint_as_float(rec.x) < 0.0f) ? 0x80000000u : 0u);
                }
                nsv += __popc(bal);
                __syncwarp();
                ISDF_PT(pt_cull += clock64() - pt_a;)
            };
            // search stage for every queued survivor, in voxel order, software-pipelined ACROSS queries: while query k runs, the
            // first 32 candidate ids of query k+2 are being loaded and the triangle records of query k+1's first pass are
            // prefetched into L1 — the id -> record -> arithmetic chain of a query starts with its operands already close
            auto search_all = [&](bool final) __attribute__((always_inline)) {
                ISDF_PT(const long long pt_a = clock64(); const long long pt_tail0 = pt_tail;)
                nquery += nsv;
                auto first_ids = [&](int k) -> int {
                    if (k >= nsv) return -1;
                    const uint32_t cnt = sm.sv[k].cnt & 0x7fffffffu;
                    return (lane < (int)cnt) ? (int)__ldg(Mh.cand + sm.sv[k].off + lane) : -1;
                };
                int ids0 = first_ids(0), ids1 = first_ids(1);
                int k = 0;
                do {
                    if (k < nsv) {
                        const int ids2 = first_ids(k + 2);
                        const Survivor &v = sm.sv[k];
                        const d3 p = mk3(v.px, v.py, v.pz);
                        const uint32_t cnt_in = v.cnt, qcode = v.code;
                        double d2; d3 c = mk3(0, 0, 0); int tri, feat;
                        if (mesh_search_rec(Mh, p, sf, lane, &sm.stk, (int)(cnt_in & 0x7fffffffu), v.off, ids0, (int)v.seed, (cnt_in >> 31) != 0u, d2, c, tri, feat)) {
                            if (lane == 0) {
                                QRes r;
                                r.ex = p.x - c.x; r.ey = p.y - c.y; r.ez = p.z - c.z; r.tri = tri; r.code = qcode;
                                r.fc = feat | ((int)(((qcode & 0x3ffu) * (uint32_t)ny + ((qcode >> 10) & 0x3ffu) + 5u * (qcode >> 20)) % ROW_CLASSES) << 8);   // class = (r + 5 dz) % 32
                                sm.qr[nres] = r;
                            }
                            nres++;
                        }
                        ids0 = ids1; ids1 = ids2;
                    }
                    k++;
                    if (nres == 32 || (final && k >= nsv && nres > 0)) flush_tails();   // the only call site
                } while (k < nsv);
                __syncwarp();
                nsv = 0;
                ISDF_PT(pt_search += (clock64() - pt_a) - (pt_tail - pt_tail0);)
            };

            // Producer loop (one cull and one search call site): batches of 32 window rows are loaded (lane = row), their occupied voxels
            // are appended to the ring, and whenever 32 voxels are queued — or the window is exhausted — they are processed.
            // Voxel (row r, z offset dz) of the window belongs to class (r + 5 dz) % 32: the voxels an obstacle patch puts near the robot
            // — a few rows x a few z, the ones that cost mesh queries — land in ~as many different classes as there are voxels, so the
            // parts of a split sample get near-equal numbers of queries (row-interleaved classes gave a wall patch to 5 of 32 classes:
            // item timeline in profiles/r02_tuning.md). A split part scans the same rows and keeps its classes' voxels (a bit filter).
            // Lanes are rows in ascending order and a lane emits its voxels z-ascending, so emitting a batch lane by lane — at once when it
            // fits into the ring, else row by row (dense walls) — keeps every CLASS's voxels in (row, z) order for whole samples and parts.
            const int w = it.c1 - it.c0;
            int zs = W.iz0, kb = -32;
            uint32_t bits = 0, rowcode = 0;
            unsigned pending = 0;
            bool finished = false;
            for (;;) {
                if (!finished) {
                    if (pending == 0u) {   // next batch of rows
                        kb += 32;
                        if (kb >= nrows) { kb = 0; zs += 32; }
                        if (zs > W.iz1) finished = true;
                        else {
                            const int nzc = min(32, W.iz1 - zs + 1);
                            const uint32_t zmask = (nzc == 32) ? 0xffffffffu : ((1u << nzc) - 1u);
                            const int r = kb + lane;
                            bits = 0;
                            if (r < nrows) {
                                int rx, ry;
                                row_split(r, ny, inv_ny, rx, ry);
                                bits = row_bits(G, W.ix0 + rx, W.iy0 + ry, zs, zmask);
                                rowcode = (uint32_t)rx | ((uint32_t)ry << 10) | ((uint32_t)(zs - W.iz0) << 20);
                                if (!whole && bits != 0u) {   // keep the voxels of the classes [c0, c1)
                                    uint32_t keep = 0u;
                                    unsigned cls = (unsigned)(r + 5 * (zs - W.iz0)) & 31u;
                                    for (int k = 0; k < nzc; k++) { keep |= (((cls - (unsigned)it.c0) & 31u) < (unsigned)w ? 1u : 0u) << k; cls = (cls + 5u) & 31u; }
                                    bits &= keep;
                                }
                            }
                            pending = __ballot_sync(0xffffffffu, bits != 0u);
                            if (pending != 0u) {
                                int incl = __popc(bits);
#pragma unroll
                                for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
                                const int total = __shfl_sync(0xffffffffu, incl, 31);
                                if (nq + total <= 64) {   // the whole batch fits: emit it at once
                                    int pos = head + nq + incl - __popc(bits);
                                    while (bits != 0u) {
                                        const int z = __ffs(bits) - 1;
                                        bits &= bits - 1;
                                        sm.vq[pos & 63] = rowcode + ((uint32_t)z << 20);
                                        pos++;
                                    }
                                    nq += total;
                                    pending = 0u;
                                }
                            }
                        }
                    } else {               // one row: lane z emits voxel z of the lowest pending row
                        const int src = __ffs(pending) - 1;
                        pending &= pending - 1;
                        const uint32_t b = __shfl_sync(0xffffffffu, bits, src);
                        const uint32_t rc = __shfl_sync(0xffffffffu, rowcode, src);
                        if ((b >> lane) & 1u) sm.vq[(head + nq + __popc(b & lt_mask)) & 63] = rc + ((uint32_t)lane << 20);
                        nq += __popc(b);
                    }
                    __syncwarp();
                }
                if (nq >= 32 || (finished && nq > 0)) cull(min(nq, 32));
                // single call site; the final round runs even without survivors when answered voxels still await their tail
                const bool last_round = finished && nq == 0;
                if (nsv > 0 || (last_round && nres > 0)) {
                    search_all(last_round);
                }
                if (last_round) break;
            }
            __syncwarp();
            // sample (or part) total: class sums added in class order
            if (whole) {
                double mine = 0.0;
                if (lane < 8) for (int c = 0; c < ROW_CLASSES; c++) mine += sm.cacc[c][lane];
                sample_finish_whole(A, it, mine, npairs, t_begin, 64u * nquery + npairs);
            } else {
                // split part: publish this part's class sums; the LAST part of the sample to arrive (one ticket per split slot) adds
                // all 32 class sums in class order — the same additions a whole-sample item performs — so that the epilogue sees
                // one finished row per sample whether or not it was split
                double *sub = A.subsum + (size_t)it.hslot * ROW_CLASSES * 8;
                if (lane < 8) for (int c = it.c0; c < it.c1; c++) __stcg(sub + c * 8 + lane, sm.cacc[c][lane]);
                __threadfence();
                __syncwarp();
                unsigned mywork = 64u * nquery + npairs, prev = 0;
                if (lane == 0) {
                    if (A.pair_counter && npairs) atomicAdd(A.pair_counter, (unsigned long long)npairs);
                    atomicAdd(A.split_work + it.hslot, mywork);
                    prev = atomicAdd(A.split_done + it.hslot, 1u);
                }
                prev = __shfl_sync(0xffffffffu, prev, 0);
                if ((int)prev == ROW_CLASSES / w - 1) {   // last of the f = 32 / w parts
                    __threadfence();
                    double mine = 0.0;
                    if (lane < 8) for (int c = 0; c < ROW_CLASSES; c++) mine += __ldcg(sub + c * 8 + lane);
                    unsigned total_work = 0;
                    if (lane == 0) { total_work = atomicExch(A.split_work + it.hslot, 0u); A.split_done[it.hslot] = 0u; }
                    total_work = __shfl_sync(0xffffffffu, total_work, 0);
                    sample_finish_whole(A, it, mine, 0u, t_begin, total_work);
                }
            }
        } else {
            sample_finish_whole(A, it, 0.0, 0u, t_begin, 0u);
        }
        if (A.trace && lane == 0) {
            unsigned long long *tr = A.trace + TRACE_STRIDE * (size_t)it.slot;
            tr[1] = global_ns();
            ISDF_PT(tr[2] = pt_pose; tr[3] = pt_cull; tr[4] = pt_search; tr[5] = pt_tail; tr[6] = clock64() - pt_all0; tr[7] = ((unsigned long long)nquery << 32) | npairs;)
        }
        __syncwarp();
    }
}


// Work items for the next evaluation: bucket sort by reported work, descending. A sample is split into f = 2..32 items (each a
// contiguous range of 32/f row classes, work/f each) only when it alone would outlast the launch's balanced share:
// work > thr = 0.7 * total / warp_slots, f = the power of two that brings a part down to ~thr. With one GPU almost nothing is
// split (splitting costs redundant pose work and sparse row scans); with the samples sharded over 8 GPUs the same trajectory has
// 8x less work per GPU and its heavy samples are spread over up to 32 warps each. Placement inside a bucket uses shared-memory
// atomics: the order only decides WHICH warp takes WHICH item, never the arithmetic, so results stay bit-reproducible.
// One CTA, ~10 us, off the critical path of the evaluation that produced `work`.
constexpr int ORDER_BUCKETS = 1024;
__device__ __forceinline__ int order_bucket(unsigned w) { return (int)min(w >> 3, (unsigned)ORDER_BUCKETS - 1u); }

// inclusive scan of one int per thread over the 1024-thread block (warp scans + a scan of the 32 warp totals)
__device__ __forceinline__ int block_scan_inclusive_1024(int v, int *warp_tot) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += t; }
    if (lane == 31) warp_tot[wid] = v;
    __syncthreads();
    if (wid == 0) {
        int t = warp_tot[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, t, o); if (lane >= o) t += u; }
        warp_tot[lane] = t;
    }
    __syncthreads();
    const int r = v + (wid > 0 ? warp_tot[wid - 1] : 0);
    __syncthreads();
    return r;
}

template <bool CACHED>
__global__ void __launch_bounds__(1024) k_build_items(const unsigned *work, int rank, int world, int M, int max_split, int warp_slots,
                                                      int *items, int *item_count) {
    __shared__ int hist[ORDER_BUCKETS];
    __shared__ int cursor[ORDER_BUCKETS];
    __shared__ int warp_tot[32];
    __shared__ int nsplit, first_over;
    __shared__ unsigned long long total_work;
    int *scratch = items + 3 * ((size_t)M + (size_t)(ROW_CLASSES - 1) * max_split);   // behind the item table: per sample (slot << 6) | f, or -1
    const int tid = threadIdx.x;
    unsigned wv[CACHED ? ITEMS_CACHE : 1];
    if (CACHED) {
#pragma unroll
        for (int u = 0; u < ITEMS_CACHE; u++) { const int m = tid + u * 1024; wv[u] = (m < M) ? __ldcg(work + rank + (size_t)world * m) : 0u; }
    }
    auto work_of = [&](int u, int m) -> unsigned { return CACHED ? wv[u] : __ldcg(work + rank + (size_t)world * m); };
    hist[tid] = 0; cursor[tid] = 0;
    if (tid == 0) { nsplit = 0; total_work = 0ull; first_over = ORDER_BUCKETS; }
    __syncthreads();
    {   // per-sample work histogram (cursor[]) and total work
        unsigned long long mine = 0ull;
        if (CACHED) {
#pragma unroll
            for (int u = 0; u < ITEMS_CACHE; u++) { const int m = tid + u * 1024; if (m < M) { mine += wv[u]; atomicAdd(&cursor[order_bucket(wv[u])], 1); } }
        } else {
            for (int m = tid; m < M; m += 1024) { const unsigned w = work_of(0, m); mine += w; atomicAdd(&cursor[order_bucket(w)], 1); }
        }
        for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
        if ((tid & 31) == 0) atomicAdd(&total_work, mine);
    }
    __syncthreads();
    // balanced-share threshold, raised if needed so that only the max_split HEAVIEST samples qualify: walking the buckets from the
    // top, b = the first bucket whose samples no longer fit into the split slots (thread t looks at bucket 1023 - t)
    {
        const int cum = block_scan_inclusive_1024(cursor[ORDER_BUCKETS - 1 - tid], warp_tot);
        if (cum > max_split) atomicMin(&first_over, tid);
    }
    __syncthreads();
    unsigned THR;
    {
        const unsigned long long t = (total_work * 7ull) / (10ull * (unsigned long long)max(warp_slots, 1));
        THR = (unsigned)min(max(t, (unsigned long long)SPLIT_WORK_MIN), 0xffffffffull);
        if (first_over < ORDER_BUCKETS) {
            const int b = ORDER_BUCKETS - 1 - first_over;
            THR = max(THR, (unsigned)(b + 1) << 3);           // buckets above b fit into the split slots
            if (b == ORDER_BUCKETS - 1) THR = 0xffffffffu;     // even the top bucket alone overflows: no splitting
        }
    }
    __syncthreads();
    cursor[tid] = 0;
    __syncthreads();
    // pass 1: decide splits (first come first served up to max_split) and their factor, histogram the item keys
    auto decide = [&](int m, unsigned w) {
        int code = -1;
        if (w >= THR) {
            const int hs = atomicAdd(&nsplit, 1);
            if (hs < max_split) {
                int f = 2;
                while (f < ROW_CLASSES && (unsigned long long)THR * (unsigned)f < (unsigned long long)w) f <<= 1;
                code = (hs << 6) | f;
                atomicAdd(&hist[order_bucket(w / (unsigned)f)], f);
            }
        }
        if (code < 0) atomicAdd(&hist[order_bucket(w)], 1);
        scratch[m] = code;
    };
    if (CACHED) {
#pragma unroll
        for (int u = 0; u < ITEMS_CACHE; u++) { const int m = tid + u * 1024; if (m < M) decide(m, wv[u]); }
    } else {
        for (int m = tid; m < M; m += 1024) decide(m, work_of(0, m));
    }
    __syncthreads();
    {   // exclusive scan over buckets in DESCENDING bucket order
        const int b = ORDER_BUCKETS - 1 - tid;
        const int incl = block_scan_inclusive_1024(hist[b], warp_tot);
        cursor[b] = incl - hist[b];
        if (tid == ORDER_BUCKETS - 1) *item_count = incl;
    }
    __syncthreads();
    auto place = [&](int m, unsigned w) {
        const int code = scratch[m];
        if (code >= 0) {
            const int hs = code >> 6, f = code & 63, cw = ROW_CLASSES / f;
            const int pos = atomicAdd(&cursor[order_bucket(w / (unsigned)f)], f);
            for (int p = 0; p < f; p++) { items[3 * (pos + p)] = m; items[3 * (pos + p) + 1] = (p * cw) | ((p * cw + cw) << 8); items[3 * (pos + p) + 2] = hs; }
        } else {
            const int pos = atomicAdd(&cursor[order_bucket(w)], 1);
            items[3 * pos] = m; items[3 * pos + 1] = -1; items[3 * pos + 2] = -1;
        }
    };
    if (CACHED) {
#pragma unroll
        for (int u = 0; u < ITEMS_CACHE; u++) { const int m = tid + u * 1024; if (m < M) place(m, wv[u]); }
    } else {
        for (int m = tid; m < M; m += 1024) place(m, work_of(0, m));
    }
}
#endif  // ISDF_DISCRETE_TU

// ---- launch interface of the discrete translation unit (isdf_discrete_tu.cu) ------------------------------------------------------
cudaError_t discrete_launch_scan(const DiscArgs &A, bool mesh, unsigned grid, cudaStream_t st);
cudaError_t discrete_launch_epilogue(const DiscArgs &A, cudaStream_t st);
cudaError_t discrete_launch_build_items(const unsigned *work, int rank, int world, int M, int max_split, int warp_slots, int *items,
                                        int *item_count, cudaStream_t st);
// resident CTAs per SM of the scan kernels (occupancy API); also the "can this image run here" probe of isdf_create
cudaError_t discrete_resident_blocks(int *mesh_blocks, int *analytic_blocks);
// diagnostics: the device flatness map / adjoint exactly as the epilogue compiles it (tests pin it to the reference's flatness.hpp)
cudaError_t discrete_launch_dbg_flatness(const FlatParams &fp, int n, const double *vaj, const double *grads, double *out, cudaStream_t st);

}  // namespace isdf
