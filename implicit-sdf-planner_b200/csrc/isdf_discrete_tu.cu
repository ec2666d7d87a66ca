// Translation unit of the discrete-path kernels (isdf_discrete.cuh): k_discrete_mesh, k_discrete_analytic, k_discrete_epilogue,
// k_build_items, and the collision-check kernels (isdf_check.cuh: k_check_samples, k_check_finish). Compiled WITH FMA contraction (nvcc default): nothing on this path replays a sequential decision of the
// reference, its parity bar is the north star's 1e-6 (observed ~1e-15), and un-fused FP64 cost the mesh kernel ~12 % (ncu,
// profiles/r01_p). The swept-volume search, whose accept/reject sequence must replay the reference's bit for bit, stays in
// isdf_api.cu under -fmad=false. ISDF_FAST_TRI selects the division-free closest-point test (isdf_mesh.cuh) for this TU only.
#define ISDF_DISCRETE_TU 1
#ifndef ISDF_NO_FAST_TRI   // A/B builds only
#define ISDF_FAST_TRI 1
#endif
#include "../../include/isdf.h"
#include "isdf_types.cuh"
#include "isdf_discrete.cuh"
#include "isdf_check.cuh"
#include <algorithm>

namespace isdf {

cudaError_t discrete_launch_scan(const DiscArgs &A, bool mesh, unsigned grid, cudaStream_t st) {
#ifdef ISDF_CARVEOUT
    static bool carved = false;   // A/B: ask for the smallest shared-memory carve-out that still holds 4 CTAs/SM (132 KB -> 124 KB of L1)
    if (!carved) {
        carved = true;
        cudaFuncSetAttribute(k_discrete_mesh<false>, cudaFuncAttributePreferredSharedMemoryCarveout, ISDF_CARVEOUT);
        cudaFuncSetAttribute(k_discrete_mesh<true>, cudaFuncAttributePreferredSharedMemoryCarveout, ISDF_CARVEOUT);
    }
#endif
    if (mesh && A.shape.mesh.sign_mode == MESH_SIGN_WINDING) k_discrete_mesh<true><<<grid, DISC_THREADS, 0, st>>>(A);
    else if (mesh) k_discrete_mesh<false><<<grid, DISC_THREADS, 0, st>>>(A);
    else k_discrete_analytic<<<grid, DISC_THREADS, 0, st>>>(A);
    return cudaGetLastError();
}

cudaError_t discrete_launch_epilogue(const DiscArgs &A, cudaStream_t st) {
    k_discrete_epilogue<<<(unsigned)A.N, EPI_THREADS, 0, st>>>(A);
    return cudaGetLastError();
}

cudaError_t discrete_launch_build_items(const unsigned *work, int rank, int world, int M, int max_split, int warp_slots, int *items,
                                        int *item_count, cudaStream_t st) {
    if (M <= 1024 * ITEMS_CACHE) k_build_items<true><<<1, 1024, 0, st>>>(work, rank, world, M, max_split, warp_slots, items, item_count);
    else k_build_items<false><<<1, 1024, 0, st>>>(work, rank, world, M, max_split, warp_slots, items, item_count);
    return cudaGetLastError();
}

cudaError_t discrete_resident_blocks(int *mesh_blocks, int *analytic_blocks) {
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, (const void *)k_discrete_analytic);   // fails loudly if the sm_100a image cannot run here
    if (e != cudaSuccess) return e;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(mesh_blocks, k_discrete_mesh<false>, DISC_THREADS, 0);
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(analytic_blocks, k_discrete_analytic, DISC_THREADS, 0);
}

// vaj: n x 9 (vel, acc, jer); grads: n x 10 (quat_grad 4, omg_grad 3, vel_grad 3); out: n x 16 (quat 4, omg 3, gV 3, gA 3, gJ 3)
__global__ void k_dbg_flatness(const FlatParams fp, int n, const double *vaj, const double *grads, double *out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double *x = vaj + 9 * (size_t)i, *gr = grads + 10 * (size_t)i;
    const d3 v = mk3(x[0], x[1], x[2]), a = mk3(x[3], x[4], x[5]), j = mk3(x[6], x[7], x[8]);
    FlatState fs;
    flat_state(fp, v, a, j, fs);
    const quat4 q = flat_quat(fs);
    const quat4 q2 = flat_quat_only(fp, v, a);
    const d3 om = flat_omega(fs);
    const double qb[4] = {gr[0], gr[1], gr[2], gr[3]};
    d3 gV, gA, gJ;
    flat_adjoint(fp, fs, v, a, qb, mk3(gr[4], gr[5], gr[6]), mk3(gr[7], gr[8], gr[9]), gV, gA, gJ);
    double *o = out + 16 * (size_t)i;
    const bool same = (q.w == q2.w && q.x == q2.x && q.y == q2.y && q.z == q2.z);   // the scan kernels' quaternion-only forward
    o[0] = same ? q.w : nan(""); o[1] = q.x; o[2] = q.y; o[3] = q.z; o[4] = om.x; o[5] = om.y; o[6] = om.z;
    o[7] = gV.x; o[8] = gV.y; o[9] = gV.z; o[10] = gA.x; o[11] = gA.y; o[12] = gA.z; o[13] = gJ.x; o[14] = gJ.y; o[15] = gJ.z;
}

cudaError_t discrete_launch_dbg_flatness(const FlatParams &fp, int n, const double *vaj, const double *grads, double *out, cudaStream_t st) {
    k_dbg_flatness<<<(n + 127) / 128, 128, 0, st>>>(fp, n, vaj, grads, out);
    return cudaGetLastError();
}

cudaError_t check_launch(const CheckArgs &A, int mode, int B, int sm_count, cudaStream_t st) {
    static int resident[3] = {0, 0, 0};   // CTAs per SM of each sample kernel (occupancy API, asked once)
    const void *fn = mode == CHECK_ANALYTIC ? (const void *)k_check_samples<CHECK_ANALYTIC>
                   : mode == CHECK_MESH_EXACT ? (const void *)k_check_samples<CHECK_MESH_EXACT> : (const void *)k_check_samples<CHECK_MESH_WINDING>;
    if (resident[mode] == 0) {
        cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident[mode], fn, CHECK_THREADS, 0);
        if (e != cudaSuccess) return e;
        resident[mode] = std::max(resident[mode], 1);
    }
    // persistent grid: one CTA per resident slot, or fewer when there are fewer samples than warps
    const long long S = (long long)A.N * (A.M + 1);
    const long long grid = std::max(1ll, std::min((S + CHECK_WARPS - 1) / CHECK_WARPS, (long long)sm_count * resident[mode]));
    if (mode == CHECK_ANALYTIC) k_check_samples<CHECK_ANALYTIC><<<(unsigned)grid, CHECK_THREADS, 0, st>>>(A);
    else if (mode == CHECK_MESH_EXACT) k_check_samples<CHECK_MESH_EXACT><<<(unsigned)grid, CHECK_THREADS, 0, st>>>(A);
    else k_check_samples<CHECK_MESH_WINDING><<<(unsigned)grid, CHECK_THREADS, 0, st>>>(A);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    k_check_finish<<<(unsigned)B, CHECK_FIN_THREADS, 0, st>>>(A);
    return cudaGetLastError();
}

cudaError_t check_launch_poison(isdf_clearance_report *d_reports, int B, cudaStream_t st) {
    k_check_poison<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(d_reports, B);
    return cudaGetLastError();
}

}  // namespace isdf
