// libisdf_b200.so — C-ABI layer (include/isdf.h) over the sm_100a kernels. No CPU fallback anywhere: every entry
// point either runs CUDA kernels or fails with ISDF_ERR_CUDA / ISDF_ERR_STATE.
#include "../../include/isdf.h"
#include "isdf_types.cuh"
#include "isdf_discrete.cuh"
#include "isdf_check.cuh"
#include "isdf_swept.cuh"
#include "isdf_minco.cuh"
#include "isdf_frontend.cuh"
#include "isdf_lbfgs.cuh"
#include <queue>
#include "isdf_host_mesh.cuh"
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <string>
#include <vector>
#include <limits>

using namespace isdf;

__global__ void k_mesh_cells(const __grid_constant__ DevMesh M, int nx, int ny, int nz, double lx, double ly, double lz, double cell,
                             float *dist, uint32_t *seed);

__global__ void k_mesh_cell_lists(const __grid_constant__ DevMesh M, long long ncell, double hd, double list_reach, uint16_t *cnt,
                                  const uint32_t *off, uint32_t *cand);
__global__ void k_mesh_cell_pack(long long ncell, const float *dist, const uint32_t *seed, const uint32_t *off, const uint16_t *cnt, uint4 *rec);

static thread_local std::string g_err;
static int fail(int code, const std::string &msg) { g_err = msg; return code; }

#define CU_TRY(expr)                                                                                  \
    do {                                                                                              \
        cudaError_t e__ = (expr);                                                                     \
        if (e__ != cudaSuccess) {                                                                     \
            return fail(ISDF_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));          \
        }                                                                                             \
    } while (0)

struct isdf_ctx {
    int device = 0;
    isdf_config cfg;
    DevCfg dcfg;
    cudaStream_t stream = nullptr, aux_stream = nullptr;   // aux: work-item build, off the evaluation's critical path
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_main_done = nullptr, ev_items_done = nullptr;
    bool items_pending = false;
    // map
    bool have_map = false;
    DevGrid grid;
    DevBuf<uint32_t> d_bits;
    // shape
    bool have_shape = false;
    DevShape shape;
    DevBuf<BvhNode> d_nodes; DevBuf<WideNode> d_wnodes; DevBuf<double> d_tris, d_pn, d_obb; DevBuf<float> d_cell_dist; DevBuf<uint32_t> d_cell_seed, d_cell_off, d_cand; DevBuf<uint16_t> d_cell_cnt; DevBuf<uint4> d_cell_rec; DevBuf<WnNode> d_wn;
    // evaluation scratch
    DevBuf<double> d_T, d_C, d_out, d_piece_cost;
    double *count_out_dev = nullptr;   // host entry points: where the epilogue drops the pair count (behind the result vector)
    DevBuf<int> d_tickets;       // pieces_done counter of the epilogue kernel
    DevBuf<double> d_tot; DevBuf<unsigned> d_split_done;   // per-sample collision sums handed from the scan kernels to the epilogue
    DevBuf<int> d_items, d_item_count; DevBuf<unsigned> d_work, d_split_work; DevBuf<double> d_subsum;   // work items (longest first, heavy samples split)
    int warp_slots = 148 * 16;   // resident warps of the mesh kernel on this device (SMs x CTAs/SM x warps/CTA)
    int sm_count = 148, mesh_blocks = 4, analytic_blocks = 4;   // persistent grids: one CTA per resident slot
    long long order_for = -1;    // (N, rank, world) signature the order array is valid for
    DevBuf<unsigned long long> d_counter, d_dbg, d_trace;
    DevBuf<double> d_mx, d_mbc, d_mT, d_mC, d_mlu, d_men, d_mgC, d_mgT, d_mcost, d_mgrad, d_mout, d_mCpp, d_msv;   // batched callback (isdf_minco.cuh)
    int minco_B = 0, minco_N = 0;
    DevBuf<double> d_lb_x, d_lb_f, d_lb_grad, d_lb_state; DevBuf<int> d_lb_int, d_lb_head;   // device-resident lock-step L-BFGS (isdf_lbfgs.cuh)
    int *h_lb_active = nullptr;  // pinned
    bool dbg_on = false;
    bool no_items = false;       // diagnostics: always launch in natural order, never split (isdf_dbg_schedule)
    int warp_slots_override = 0; // diagnostics: pretend the device has this many resident warps (forces splitting)
    double *h_stage = nullptr;   // pinned
    size_t h_stage_n = 0;
    // swept volume
    SweptState sv;
    // shard
    int rank = 0, world = 1;
    // front end attitude kernels (isdf_frontend.cuh)
    DevBuf<double> d_fe_rot; DevBuf<uint8_t> d_fe_kernels, d_fe_order, d_fe_ok; DevBuf<uint32_t> d_fe_masks, d_fe_out;
    DevBuf<int> d_fe_ind; DevBuf<double> d_fe_father, d_fe_child;
    DevBuf<uint2> d_fe_core, d_fe_urows, d_fe_surv, d_fe_chunks; DevBuf<uint4> d_fe_tab; int fe_nurow = 0, fe_nchunk = 0, fe_ntab = 0; DevBuf<unsigned> d_fe_count; int fe_ncore = 0;
    bool fe_ready = false;
    int fe_xk = 0, fe_yk = 0, fe_ks = 0;
    double fe_max_roll = 0, fe_max_pitch = 0, fe_ang_res = 0, fe_margin = 0;
    // peer-memory reduction (isdf_peer.cuh)
    void *peer_buf = nullptr;            // own exchange buffer (cudaMalloc, exported through CUDA IPC)
    void *peer_open[PEER_MAX] = {};      // peers' buffers opened here (null for self / unused)
    PeerArgs peer = {};                  // world == 0: not connected
    bool peer_fused = false;             // sharded *_device evaluations finish with the exchange
    int peer_world_alloc = 0, peer_cap = 0;
    DevBuf<int> d_peer_status;
    // collision check (isdf_check.cuh): its own buffers, so that a check leaves the cost paths' state alone
    DevBuf<double> d_ck_in, d_ck_clear; DevBuf<long long> d_ck_arg; DevBuf<int> d_ck_cursor; DevBuf<unsigned long long> d_ck_counters, d_ck_cycles;
    DevBuf<isdf_clearance_report> d_ck_rep;
    isdf_stats stats;
};

static int set_device(isdf_ctx *c) { CU_TRY(cudaSetDevice(c->device)); return 0; }

static int ensure_stage(isdf_ctx *c, size_t n) {
    if (n <= c->h_stage_n) return 0;
    if (c->h_stage) cudaFreeHost(c->h_stage);
    c->h_stage = nullptr; c->h_stage_n = 0;
    CU_TRY(cudaMallocHost((void **)&c->h_stage, n * sizeof(double)));
    c->h_stage_n = n;
    return 0;
}

extern "C" const char *isdf_last_error(void) { return g_err.c_str(); }

extern "C" int isdf_default_config(isdf_config *cfg) {
    if (!cfg) return fail(ISDF_ERR_INVALID, "cfg is NULL");
    // plan_manager/config/config_CappedCone.yaml
    cfg->vehicle_mass = 0.61; cfg->grav_acc = 9.8; cfg->horiz_drag = 0.10; cfg->vert_drag = 0.10; cfg->paras_drag = 0.01; cfg->speed_eps = 0.0001;
    cfg->vmax = 10; cfg->omgmax = 10; cfg->thetamax = 100.0;
    cfg->weight_v = 1000.0; cfg->weight_p = 4000.0; cfg->weight_omg = 1000.0; cfg->weight_theta = 1000.0;
    cfg->smoothing_eps = 1.0e-2; cfg->safety_hor = 0.866; cfg->occupancy_resolution = 1.0;
    cfg->kernel_size = 13; cfg->integral_intervs = 64; cfg->threads_num = 30;
    // the LIVE reference callback (hpp:358-430): collision through the swept-volume term only; grad_cost_p is dead code there, so the
    // discrete collision term is opt-in (flags |= ISDF_WITH_COLLISION) — a default BackEnd must not penalise collision twice
    cfg->flags = ISDF_WITH_DYNAMICS;
    return 0;
}

extern "C" int isdf_create(const isdf_config *cfg, int device, isdf_ctx **out) {
    if (!cfg || !out) return fail(ISDF_ERR_INVALID, "cfg/out is NULL");
    if (cfg->integral_intervs < 1 || cfg->kernel_size < 1 || !(cfg->occupancy_resolution > 0) || !(cfg->vehicle_mass > 0) ||
        !(cfg->smoothing_eps > 0))
        return fail(ISDF_ERR_INVALID, "config out of range");
    int ndev = 0;
    CU_TRY(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(ISDF_ERR_CUDA, "no such CUDA device (this library has no CPU fallback)");
    CU_TRY(cudaSetDevice(device));
    // fail loudly if the sm_100a image cannot run here
    int nb_mesh = 0, nb_analytic = 0;
    CU_TRY(discrete_resident_blocks(&nb_mesh, &nb_analytic));
    // pose-window offsets are packed 10 bits per axis (isdf_discrete.cuh); the inclusive index range of a window is at most
    // kernel_size + 2 voxels when the map resolution equals occupancy_resolution (isdf_set_map checks the resolution)
    if (cfg->kernel_size + 2 > WINDOW_AXIS_MAX) return fail(ISDF_ERR_UNSUPPORTED, "kernel_size too large (pose windows are limited to 1023 voxels per axis)");
    isdf_ctx *c = new isdf_ctx();
    c->device = device; c->cfg = *cfg;
    {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, device) == cudaSuccess && nb_mesh > 0 && nb_analytic > 0) {
            c->sm_count = prop.multiProcessorCount;
            c->mesh_blocks = nb_mesh; c->analytic_blocks = nb_analytic;
            c->warp_slots = prop.multiProcessorCount * nb_mesh * DISC_WARPS;
        }
    }
    std::memset(&c->stats, 0, sizeof(c->stats));
    std::memset(&c->grid, 0, sizeof(c->grid));
    std::memset(&c->shape, 0, sizeof(c->shape));
    DevCfg &d = c->dcfg;
    d.fp.mass = cfg->vehicle_mass; d.fp.grav = cfg->grav_acc; d.fp.dh_over_m = cfg->horiz_drag / cfg->vehicle_mass;
    d.fp.cp = cfg->paras_drag; d.fp.veps = cfg->speed_eps;
    d.vmax2 = cfg->vmax * cfg->vmax; d.omgmax2 = cfg->omgmax * cfg->omgmax; d.thetamax = cfg->thetamax;
    d.wv = cfg->weight_v; d.wp = cfg->weight_p; d.womg = cfg->weight_omg; d.wtheta = cfg->weight_theta;
    d.mu = cfg->smoothing_eps; d.safety = cfg->safety_hor;
    d.half_bd = (cfg->kernel_size * cfg->occupancy_resolution) / 2;
    d.K = cfg->integral_intervs; d.flags = cfg->flags;
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->aux_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_main_done, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_items_done, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev1);
    if (e == cudaSuccess) e = c->d_counter.ensure(4);
    if (e == cudaSuccess) e = cudaMemset(c->d_counter.p, 0, 4 * sizeof(unsigned long long));
    if (e != cudaSuccess) { delete c; return fail(ISDF_ERR_CUDA, std::string("isdf_create: ") + cudaGetErrorString(e)); }
    *out = c;
    return 0;
}

extern "C" int isdf_destroy(isdf_ctx *c) {
    if (!c) return 0;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    if (c->aux_stream) cudaStreamSynchronize(c->aux_stream);
    c->d_bits.release(); c->d_nodes.release(); c->d_wnodes.release(); c->d_tris.release(); c->d_pn.release(); c->d_obb.release(); c->d_cell_dist.release(); c->d_cell_seed.release(); c->d_cell_off.release(); c->d_cand.release(); c->d_cell_cnt.release(); c->d_cell_rec.release(); c->d_wn.release();
    c->d_T.release(); c->d_C.release(); c->d_out.release(); c->d_piece_cost.release();
    c->d_tickets.release(); c->d_counter.release(); c->d_items.release(); c->d_item_count.release(); c->d_tot.release(); c->d_split_done.release(); c->d_work.release(); c->d_split_work.release(); c->d_subsum.release(); c->d_dbg.release(); c->d_trace.release();
    for (int p = 0; p < PEER_MAX; p++) if (c->peer_open[p]) cudaIpcCloseMemHandle(c->peer_open[p]);
    if (c->peer_buf) cudaFree(c->peer_buf);
    c->d_peer_status.release();
    c->d_fe_rot.release(); c->d_fe_kernels.release(); c->d_fe_order.release(); c->d_fe_ok.release(); c->d_fe_masks.release(); c->d_fe_out.release(); c->d_fe_ind.release(); c->d_fe_father.release(); c->d_fe_child.release(); c->d_fe_core.release(); c->d_fe_urows.release(); c->d_fe_surv.release(); c->d_fe_chunks.release(); c->d_fe_tab.release(); c->d_fe_count.release();
    c->d_mx.release(); c->d_mbc.release(); c->d_mT.release(); c->d_mC.release(); c->d_mlu.release(); c->d_men.release(); c->d_mgC.release(); c->d_mgT.release(); c->d_mcost.release(); c->d_mgrad.release(); c->d_mout.release(); c->d_mCpp.release(); c->d_msv.release();
    c->sv.release();
    c->d_ck_in.release(); c->d_ck_clear.release(); c->d_ck_arg.release(); c->d_ck_cursor.release(); c->d_ck_counters.release(); c->d_ck_cycles.release(); c->d_ck_rep.release();
    if (c->h_stage) cudaFreeHost(c->h_stage);
    if (c->h_lb_active) cudaFreeHost(c->h_lb_active);
    c->d_lb_x.release(); c->d_lb_f.release(); c->d_lb_grad.release(); c->d_lb_state.release(); c->d_lb_int.release(); c->d_lb_head.release();
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->ev_main_done) cudaEventDestroy(c->ev_main_done);
    if (c->ev_items_done) cudaEventDestroy(c->ev_items_done);
    if (c->aux_stream) cudaStreamDestroy(c->aux_stream);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return 0;
}

extern "C" int isdf_get_stats(isdf_ctx *c, isdf_stats *out) {
    if (!c || !out) return fail(ISDF_ERR_INVALID, "NULL argument");
    *out = c->stats;
    return 0;
}

extern "C" int isdf_set_shard(isdf_ctx *c, int rank, int world) {
    if (!c || world < 1 || rank < 0 || rank >= world) return fail(ISDF_ERR_INVALID, "bad shard");
    if (world > c->cfg.integral_intervs + 1) return fail(ISDF_ERR_INVALID, "world larger than samples per piece");
    c->rank = rank; c->world = world; c->order_for = -1;
    return 0;
}

// ---- shapes ---------------------------------------------------------------------------------------------------
static void shape_common(isdf_ctx *c, const double *rot, const double *trans) {
    DevShape &s = c->shape;
    const double I[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    for (int i = 0; i < 9; i++) s.rot[i] = rot ? rot[i] : I[i];
    for (int i = 0; i < 3; i++) s.trans[i] = trans ? trans[i] : 0.0;
    // CSG helper rotations: rotate(other, angle = acos(0), axis) of Shape.hpp:2021-2041 for axis = Y x X and Z x X
    const double ang = std::acos(0.0), sn = std::sin(ang), cs = std::cos(ang), mm = 1 - cs;
    auto fill = [&](double x, double y, double z, double *R) {
        R[0] = mm * x * x + cs;     R[1] = mm * x * y + z * sn; R[2] = mm * z * x - y * sn;
        R[3] = mm * x * y - z * sn; R[4] = mm * y * y + cs;     R[5] = mm * y * z + x * sn;
        R[6] = mm * z * x + y * sn; R[7] = mm * y * z - x * sn; R[8] = mm * z * z + cs;
    };
    fill(0, 0, -1, s.csg_ry);  // (0,1,0) x (1,0,0)
    fill(0, 1, 0, s.csg_rz);   // (0,0,1) x (1,0,0)
}

extern "C" int isdf_set_shape_analytic(isdf_ctx *c, int kind, const double *params, int nparams, const double *rot, const double *trans) {
    if (!c) return fail(ISDF_ERR_INVALID, "ctx is NULL");
    if (kind < 0 || kind >= ISDF_SHAPE_MESH) return fail(ISDF_ERR_INVALID, "kind is not an analytic shape");
    if (nparams < 0 || nparams > 12 || (nparams > 0 && !params)) return fail(ISDF_ERR_INVALID, "bad params");
    std::memset(&c->shape, 0, sizeof(c->shape));
    c->shape.kind = kind;
    for (int i = 0; i < nparams; i++) c->shape.par[i] = params[i];
    shape_common(c, rot, trans);
    c->have_shape = true; c->fe_ready = false;
    c->order_for = -1;   // work items of another shape class may carry split slots
    return 0;
}

extern "C" int isdf_set_shape_named(isdf_ctx *c, const char *name, const double *rot, const double *trans) {
    if (!c || !name) return fail(ISDF_ERR_INVALID, "NULL argument");
    struct Entry { const char *name; int kind; int n; double p[12]; };
    // constants are the reference classes' hard-coded members (Shape.hpp:609,827,863,898-900,936,1003-1005,1052,1149,1214,
    // 1239,1293,1346-1349,1520,1575,1630)
    static const Entry table[] = {
        {"Ball", ISDF_SHAPE_BALL, 1, {1.0}},
        {"Point", ISDF_SHAPE_POINT, 0, {0}},
        {"Torus", ISDF_SHAPE_TORUS, 2, {2.5, 0.3}},
        {"Torus_big", ISDF_SHAPE_TORUS, 2, {3.5, 0.3}},
        {"Cappedtorus", ISDF_SHAPE_CAPPED_TORUS, 4, {0, 0, 3.5, 0.3}},  // sc filled below: (sin 40, cos 40), radians
        {"CappedCone", ISDF_SHAPE_CAPPED_CONE, 2, {2.0, 0.8}},
        {"RoundedCone", ISDF_SHAPE_ROUNDED_CONE, 3, {1.5, 0.6, 4.5}},
        {"WireframeBox", ISDF_SHAPE_WIREFRAME_BOX, 4, {1.8, 2.5, 3.5, 0.1}},
        {"BendLinear", ISDF_SHAPE_BEND_LINEAR, 2, {2.0, 0.25}},
        {"BendLinear_big", ISDF_SHAPE_BEND_LINEAR, 2, {3.2, 0.45}},
        {"TwistBox", ISDF_SHAPE_TWIST_BOX, 4, {2.0, 2.0, 2.0, 3.14159265358979323846 / 6}},
        {"BendBox", ISDF_SHAPE_BEND_BOX, 4, {2.0, 2.0, 2.0, 0.5}},
        {"Table", ISDF_SHAPE_TABLE, 12, {0.0, 0.0, 0.0, 3.5, 1.75, 0.7, 2.8, 1.05, 0.0, 3.5, 1.75, 2.8}},
        {"Trefoil", ISDF_SHAPE_TREFOIL, 0, {0}},
        {"SmoothDifference", ISDF_SHAPE_SMOOTH_DIFFERENCE, 4, {3.0, 3.0, 0.5, 1.0}},
        {"SmoothIntersection", ISDF_SHAPE_SMOOTH_INTERSECTION, 4, {3.0, 3.0, 0.5, 1.0}},
        {"SmoothIntersection_big", ISDF_SHAPE_SMOOTH_INTERSECTION, 4, {9.0, 9.0, 1.5, 3.0}},
        {"CSG", ISDF_SHAPE_CSG, 0, {0}},
    };
    for (const Entry &e : table) {
        if (std::strcmp(e.name, name) == 0) {
            double p[12];
            for (int i = 0; i < 12; i++) p[i] = e.p[i];
            if (e.kind == ISDF_SHAPE_CAPPED_TORUS) { p[0] = std::sin(40); p[1] = std::cos(40); }
            return isdf_set_shape_analytic(c, e.kind, p, e.n, rot, trans);
        }
    }
    // the reference falls back to the mesh Generalshape for unknown names (swm:269-274); a mesh needs its geometry
    return fail(ISDF_ERR_INVALID, std::string("unknown analytic shape name '") + name + "' (use isdf_set_shape_mesh for OBJ bodies)");
}

extern "C" int isdf_set_shape_mesh(isdf_ctx *c, const double *V, int nV, const int32_t *F, int nF, const double *poly_params) {
    return isdf_set_shape_mesh_ex(c, V, nV, F, nF, poly_params, ISDF_MESH_SIGN_AUTO);
}

extern "C" int isdf_set_shape_mesh_ex(isdf_ctx *c, const double *V, int nV, const int32_t *F, int nF, const double *poly_params, int sign_mode) {
    if (!c || !V || !F) return fail(ISDF_ERR_INVALID, "NULL argument");
    if (sign_mode < 0 || sign_mode > 2) return fail(ISDF_ERR_INVALID, "bad sign_mode");
    if (set_device(c)) return ISDF_ERR_CUDA;
    HostMesh hm; std::string err;
    // the bitmap shortcut is sized for the smallest bound the kernels use: safety_hor (discrete) — the swept path uses
    // 2*safety_hor + 0.1 >= safety_hor
    if (!build_host_mesh(V, nV, F, nF, poly_params, c->cfg.safety_hor, hm, err, sign_mode))
        return fail(err.find("not a closed") != std::string::npos ? ISDF_ERR_UNSUPPORTED : ISDF_ERR_INVALID, err);
    if (!hm.wn.empty()) CU_TRY(c->d_wn.upload(hm.wn.data(), hm.wn.size(), c->stream));
    CU_TRY(c->d_nodes.upload(hm.nodes.data(), hm.nodes.size(), c->stream));
    CU_TRY(c->d_wnodes.upload(hm.wnodes.data(), hm.wnodes.size(), c->stream));
    CU_TRY(c->d_tris.upload(hm.tris.data(), hm.tris.size(), c->stream));
    CU_TRY(c->d_pn.upload(hm.pnormals.data(), hm.pnormals.size(), c->stream));
    CU_TRY(c->d_obb.upload(hm.leaf_obb.data(), hm.leaf_obb.size(), c->stream));
    CU_TRY(cudaStreamSynchronize(c->stream));
    std::memset(&c->shape, 0, sizeof(c->shape));
    c->shape.kind = ISDF_SHAPE_MESH;
    shape_common(c, nullptr, nullptr);
    DevMesh m = hm.view();
    m.nodes = c->d_nodes.p; m.wnodes = c->d_wnodes.p; m.tris = c->d_tris.p; m.pnormals = c->d_pn.p; m.leaf_obb = c->d_obb.p;
    m.wn = hm.wn.empty() ? nullptr : c->d_wn.p;
    // per-cell signed distance + seed triangle, computed on the device with the freshly uploaded BVH
    const size_t ncell = (size_t)m.gdim[0] * m.gdim[1] * m.gdim[2];
    CU_TRY(c->d_cell_dist.ensure(ncell));
    CU_TRY(c->d_cell_seed.ensure(ncell));
    {
        DevMesh build = m;
        build.gdim[0] = 0;            // no grid while it is being built: plain unbounded BVH queries
        build.cell_dist = nullptr; build.cell_seed = nullptr; build.cell_off = nullptr; build.cell_cnt = nullptr; build.cand = nullptr;
        k_mesh_cells<<<(unsigned)((ncell + 127) / 128), 128, 0, c->stream>>>(build, m.gdim[0], m.gdim[1], m.gdim[2], m.glo[0], m.glo[1], m.glo[2],
                                                                           m.gcell, c->d_cell_dist.p, c->d_cell_seed.p);
        c->stats.kernel_launches++;
        CU_TRY(cudaGetLastError());
        CU_TRY(cudaStreamSynchronize(c->stream));
    }
    m.cell_dist = c->d_cell_dist.p; m.cell_seed = c->d_cell_seed.p;
    m.cell_off = nullptr; m.cell_cnt = nullptr; m.cand = nullptr;
    // exact candidate lists for every cell a query can land in and not be settled by the cell's distance bracket alone: the discrete
    // path queries within safety_hor of the surface, the swept-volume path within its range bound 2*safety_hor + 0.1 (swm:383) — a
    // flat pass over ~100 listed triangles answers such a query in a tenth of the time of a far-field tree search, and the sign
    // descent of the swept-volume path is a CHAIN of them (profiles/r02_tuning.md, swept path)
    {
        const double hd = 0.5 * std::sqrt(3.0) * m.gcell;
        const double list_reach = std::max(c->cfg.safety_hor, 2.0 * c->cfg.safety_hor + 0.1) + 2.0 * m.ghd;
        CU_TRY(c->d_cell_cnt.ensure(ncell)); CU_TRY(c->d_cell_off.ensure(ncell));
        const unsigned warps_grid = (unsigned)((ncell + 3) / 4);
        k_mesh_cell_lists<<<warps_grid, 128, 0, c->stream>>>(m, (long long)ncell, hd, list_reach, c->d_cell_cnt.p, nullptr, nullptr);
        c->stats.kernel_launches++;
        CU_TRY(cudaGetLastError());
        std::vector<uint16_t> cnt(ncell);
        CU_TRY(cudaMemcpyAsync(cnt.data(), c->d_cell_cnt.p, sizeof(uint16_t) * ncell, cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(cudaStreamSynchronize(c->stream));
        std::vector<uint32_t> off(ncell);
        size_t total = 0;
        for (size_t i = 0; i < ncell; i++) { off[i] = (uint32_t)total; total += cnt[i]; }
        if (total > 0 && total < (1ull << 31)) {
            CU_TRY(c->d_cand.ensure(total));
            CU_TRY(cudaMemcpyAsync(c->d_cell_off.p, off.data(), sizeof(uint32_t) * ncell, cudaMemcpyHostToDevice, c->stream));
            k_mesh_cell_lists<<<warps_grid, 128, 0, c->stream>>>(m, (long long)ncell, hd, list_reach, c->d_cell_cnt.p, c->d_cell_off.p, c->d_cand.p);
            c->stats.kernel_launches++;
            CU_TRY(cudaGetLastError());
            CU_TRY(cudaStreamSynchronize(c->stream));
            m.cell_off = c->d_cell_off.p; m.cell_cnt = c->d_cell_cnt.p; m.cand = c->d_cand.p;
        }
        if (getenv("ISDF_VERBOSE")) {
            size_t listed = 0; for (size_t i = 0; i < ncell; i++) listed += cnt[i] != 0;
            fprintf(stderr, "[isdf] mesh cell grid %d x %d x %d (cell %.3f m), %zu cells with a candidate list, %zu candidates (%.1f MB)\n", m.gdim[0], m.gdim[1], m.gdim[2],
                    m.gcell, listed, total, total * 4e-6);
        }
    }
    // fused 16-byte cell records for the discrete scan kernel's cull stage
    CU_TRY(c->d_cell_rec.ensure(ncell));
    k_mesh_cell_pack<<<(unsigned)((ncell + 255) / 256), 256, 0, c->stream>>>((long long)ncell, m.cell_dist, m.cell_seed, m.cell_off, m.cell_cnt, c->d_cell_rec.p);
    c->stats.kernel_launches++;
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaStreamSynchronize(c->stream));
    m.cell_rec = c->d_cell_rec.p;
    c->shape.mesh = m;
    c->have_shape = true; c->fe_ready = false;
    c->order_for = -1;
    return 0;
}

__global__ void k_mesh_cell_pack(long long ncell, const float *dist, const uint32_t *seed, const uint32_t *off, const uint16_t *cnt, uint4 *rec) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ncell) return;
    rec[i] = make_uint4(__float_as_uint(dist[i]), seed[i], (off && cnt) ? off[i] : 0u, (off && cnt) ? (uint32_t)cnt[i] : 0u);
}

// signed distance + nearest triangle at every cell centre of the body-frame grid (one thread per cell)
__global__ void k_mesh_cells(const __grid_constant__ DevMesh M, int nx, int ny, int nz, double lx, double ly, double lz, double cell,
                             float *dist, uint32_t *seed) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)nx * ny * nz) return;
    const int iz = (int)(idx % nz), iy = (int)((idx / nz) % ny), ix = (int)(idx / ((size_t)nz * ny));
    const d3 p = mk3(lx + (ix + 0.5) * cell, ly + (iy + 0.5) * cell, lz + (iz + 0.5) * cell);
    d3 c = mk3(0, 0, 0); int tri, feat;
    const double d2 = mesh_closest(M, p, 1e300, c, tri, feat);
    const d3 e = p - c;
    const double *pn = M.pnormals + 21 * (size_t)tri + 3 * feat;
    double side = e.x * pn[0] + e.y * pn[1] + e.z * pn[2];
    if (side == 0.0) { const double *fn = M.pnormals + 21 * (size_t)tri; side = e.x * fn[0] + e.y * fn[1] + e.z * fn[2]; }
    dist[idx] = (float)((side < 0.0 ? -1.0 : 1.0) * sqrt(d2));
    seed[idx] = (uint32_t)tri;
}

// Candidate lists (one warp per cell). Pass 1 (cand == nullptr): count the triangles within d_c + 2 hd of the cell centre and
// store the count (0 for cells that are too far, too deep or whose list would exceed LIST_CAP). Pass 2: fill the lists.
constexpr int LIST_CAP = MESH_LIST_CAP;
__global__ void __launch_bounds__(128) k_mesh_cell_lists(const __grid_constant__ DevMesh M, long long ncell, double hd, double list_reach,
                                                         uint16_t *cnt, const uint32_t *off, uint32_t *cand) {
    __shared__ WideStack stk[4];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long cell = (long long)blockIdx.x * 4 + warp;
    if (cell >= ncell) return;
    const double dc = fabs((double)M.cell_dist[cell]);
    if (cand == nullptr) { if (lane == 0) cnt[cell] = 0; }
    else if (cnt[cell] == 0) return;
    if (dc > list_reach) return;
    const int nz = M.gdim[2], ny = M.gdim[1];
    const int iz = (int)(cell % nz), iy = (int)((cell / nz) % ny), ix = (int)(cell / ((long long)nz * ny));
    const d3 ctr = mk3(M.glo[0] + (ix + 0.5) * M.gcell, M.glo[1] + (iy + 0.5) * M.gcell, M.glo[2] + (iz + 0.5) * M.gcell);
    // radius: centre distance (float-rounded: add its slack) + two half diagonals, then a relative safety margin
    const double R = (dc + (M.ghd - hd) + 2.0 * hd) * (1.0 + 1e-9) + 1e-12;
    const unsigned lt_mask = (1u << lane) - 1u;
    int n = 0;
    const uint32_t base = cand ? off[cell] : 0u;
    wide_range(M, ctr, R * R, lane, &stk[warp], [&](bool hit, int t) {
        const unsigned bal = __ballot_sync(0xffffffffu, hit);
        if (cand && hit) cand[base + n + __popc(bal & lt_mask)] = (uint32_t)t;
        n += __popc(bal);
    });
    if (cand == nullptr && lane == 0) cnt[cell] = (n <= LIST_CAP) ? (uint16_t)n : (uint16_t)0;
}

__global__ void k_shape_query(const __grid_constant__ DevShape S, const double *p, int n, double *sdf, double *grad, int what) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const d3 q = mk3(p[3 * i], p[3 * i + 1], p[3 * i + 2]);
    d3 g = mk3(0, 0, 0);
    double s = 0;
    if (what == ISDF_QUERY_SDF) s = shape_sdf(S, q);
    else if (what == ISDF_QUERY_GRAD) g = shape_grad(S, q);
    else s = shape_sdf_grad(S, q, g);
    if (sdf && what != ISDF_QUERY_GRAD) sdf[i] = s;
    if (grad && what != ISDF_QUERY_SDF) { grad[3 * i] = g.x; grad[3 * i + 1] = g.y; grad[3 * i + 2] = g.z; }
}

extern "C" int isdf_shape_query(isdf_ctx *c, const double *p_rel, int n, double *sdf, double *grad, int what) {
    if (!c || !p_rel || n < 0) return fail(ISDF_ERR_INVALID, "bad argument");
    if (!c->have_shape) return fail(ISDF_ERR_STATE, "shape not set");
    if (what < 0 || what > 2) return fail(ISDF_ERR_INVALID, "bad query kind");
    if (n == 0) return 0;
    if (set_device(c)) return ISDF_ERR_CUDA;
    ScopedDevBuf<double> dp, ds, dg;
    CU_TRY(dp.upload(p_rel, (size_t)3 * n, c->stream));
    CU_TRY(ds.ensure(n)); CU_TRY(dg.ensure((size_t)3 * n));
    k_shape_query<<<(n + 127) / 128, 128, 0, c->stream>>>(c->shape, dp.p, n, ds.p, dg.p, what);
    c->stats.kernel_launches++;
    CU_TRY(cudaGetLastError());
    std::vector<double> hs(n), hg((size_t)3 * n);
    CU_TRY(cudaMemcpyAsync(hs.data(), ds.p, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(cudaMemcpyAsync(hg.data(), dg.p, sizeof(double) * 3 * n, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(cudaStreamSynchronize(c->stream));
    if (sdf && what != ISDF_QUERY_GRAD) std::memcpy(sdf, hs.data(), sizeof(double) * n);
    if (grad && what != ISDF_QUERY_SDF) std::memcpy(grad, hg.data(), sizeof(double) * 3 * n);
    return 0;
}

// ---- map ------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void k_pack_bits(const T *occ, uint32_t *bits, int rows, int Z, int Zw) {
    // one warp per 32-voxel word: ballot of "voxel != 0"
    const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    const long long nwords = (long long)rows * Zw;
    if (gw >= nwords) return;
    const int row = (int)(gw / Zw), w = (int)(gw - (long long)row * Zw);
    const int z = w * 32 + lane;
    const bool o = (z < Z) && (occ[(size_t)row * Z + z] != (T)0);
    const unsigned b = __ballot_sync(0xffffffffu, o);
    if (lane == 0) bits[gw] = b;
}

template <typename T>
static int set_map_impl(isdf_ctx *c, const T *occ, int X, int Y, int Z, const double *bmin, double res) {
    if (!c || !occ || !bmin) return fail(ISDF_ERR_INVALID, "NULL argument");
    if (X < 1 || Y < 1 || Z < 1 || !(res > 0)) return fail(ISDF_ERR_INVALID, "bad map size");
    if ((long long)X * Y >= (1ll << 31) / ((Z + 31) / 32)) return fail(ISDF_ERR_INVALID, "map too large");
    if (Z > 65535) return fail(ISDF_ERR_UNSUPPORTED, "Z > 65535");
    // a pose window spans 2 * half_bd / res + 2 voxels per axis of THIS map (its resolution need not equal occupancy_resolution); the scan
    // kernels pack window offsets into 10 bits per axis
    if (c && 2.0 * c->dcfg.half_bd / res + 2.0 > (double)WINDOW_AXIS_MAX)
        return fail(ISDF_ERR_UNSUPPORTED, "map resolution too fine for kernel_size * occupancy_resolution: a pose window would exceed 1023 voxels per axis");
    if (set_device(c)) return ISDF_ERR_CUDA;
    const size_t nvox = (size_t)X * Y * Z;
    T *d_occ = nullptr;
    CU_TRY(cudaMalloc((void **)&d_occ, nvox * sizeof(T)));
    cudaError_t e = cudaMemcpyAsync(d_occ, occ, nvox * sizeof(T), cudaMemcpyHostToDevice, c->stream);
    const int Zw = (Z + 31) / 32;
    const size_t nwords = (size_t)X * Y * Zw;
    if (e == cudaSuccess) e = c->d_bits.ensure(nwords);
    if (e == cudaSuccess) {
        const long long threads = (long long)nwords * 32;
        k_pack_bits<T><<<(unsigned)((threads + 255) / 256), 256, 0, c->stream>>>(d_occ, c->d_bits.p, X * Y, Z, Zw);
        c->stats.kernel_launches++;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(d_occ);
    if (e != cudaSuccess) return fail(ISDF_ERR_CUDA, std::string("isdf_set_map: ") + cudaGetErrorString(e));
    DevGrid &g = c->grid;
    g.bits = c->d_bits.p; g.X = X; g.Y = Y; g.Z = Z; g.Zw = Zw; g.res = res;
    const int dims[3] = {X, Y, Z};
    for (int a = 0; a < 3; a++) { g.bmin[a] = bmin[a]; g.bmax[a] = bmin[a] + dims[a] * res; }
    c->have_map = true;
    return 0;
}

extern "C" int isdf_set_map_u8(isdf_ctx *c, const uint8_t *occ, int X, int Y, int Z, const double *bmin, double res) {
    return set_map_impl<uint8_t>(c, occ, X, Y, Z, bmin, res);
}
extern "C" int isdf_set_map_f64(isdf_ctx *c, const double *grid_map, int X, int Y, int Z, const double *bmin, double res) {
    return set_map_impl<double>(c, grid_map, X, Y, Z, bmin, res);
}

// getPointsInAABB (pcs:148-170): one CTA; thread = (x, y) row of the clamped index box — popcount of the row's z-run, block-wide exclusive scan
// for the row's output offset, then every thread writes its row's voxel centres in z order: the reference's x -> y -> z output order
__global__ void __launch_bounds__(256) k_points_in_aabb(const DevGrid G, double cx, double cy, double cz, double h, double *out, int cap, int *count) {
    __shared__ int warp_tot[8];
    __shared__ int running;
    const int ix0 = grid_axis_index(cx - h, G.bmin[0], G.bmax[0], G.res, G.X), ix1 = grid_axis_index(cx + h, G.bmin[0], G.bmax[0], G.res, G.X);
    const int iy0 = grid_axis_index(cy - h, G.bmin[1], G.bmax[1], G.res, G.Y), iy1 = grid_axis_index(cy + h, G.bmin[1], G.bmax[1], G.res, G.Y);
    const int iz0 = grid_axis_index(cz - h, G.bmin[2], G.bmax[2], G.res, G.Z), iz1 = grid_axis_index(cz + h, G.bmin[2], G.bmax[2], G.res, G.Z);
    const int ny = iy1 - iy0 + 1, nrows = (ix1 - ix0 + 1) * ny;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) running = 0;
    __syncthreads();
    for (int base = 0; base < nrows; base += blockDim.x) {
        const int r = base + threadIdx.x;
        int i = 0, j = 0, cnt = 0;
        if (r < nrows) {
            i = ix0 + r / ny; j = iy0 + r % ny;
            const uint32_t *row = G.bits + ((size_t)i * G.Y + j) * G.Zw;
            for (int wz = iz0 >> 5; wz <= (iz1 >> 5); wz++) {
                uint32_t w = row[wz];
                if (wz == (iz0 >> 5)) w &= 0xffffffffu << (iz0 & 31);
                if (wz == (iz1 >> 5) && (iz1 & 31) != 31) w &= (1u << ((iz1 & 31) + 1)) - 1u;
                cnt += __popc(w);
            }
        }
        int incl = cnt;
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
        if (lane == 31) warp_tot[warp] = incl;
        __syncthreads();
        int off = running + incl - cnt;
        for (int w = 0; w < warp; w++) off += warp_tot[w];
        if (r < nrows && cnt > 0) {
            const uint32_t *row = G.bits + ((size_t)i * G.Y + j) * G.Zw;
            for (int k = iz0; k <= iz1; k++)
                if ((row[k >> 5] >> (k & 31)) & 1u) {
                    if (off < cap) { out[3 * off] = (i + 0.5) * G.res + G.bmin[0]; out[3 * off + 1] = (j + 0.5) * G.res + G.bmin[1]; out[3 * off + 2] = (k + 0.5) * G.res + G.bmin[2]; }
                    off++;
                }
        }
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int w = 0; w < 8; w++) t += warp_tot[w]; running += t; }
        __syncthreads();
    }
    if (threadIdx.x == 0) *count = running;
}

extern "C" int isdf_points_in_aabb(isdf_ctx *c, const double *centre, double half_extent, double *out_points, int cap, int *n) {
    if (!c || !centre || !n || cap < 0 || (cap > 0 && !out_points)) return fail(ISDF_ERR_INVALID, "bad argument");
    if (!c->have_map) return fail(ISDF_ERR_STATE, "map not set");
    if (set_device(c)) return ISDF_ERR_CUDA;
    ScopedDevBuf<double> d; ScopedDevBuf<int> dn;
    CU_TRY(d.ensure((size_t)3 * (cap > 0 ? cap : 1))); CU_TRY(dn.ensure(1));
    k_points_in_aabb<<<1, 256, 0, c->stream>>>(c->grid, centre[0], centre[1], centre[2], half_extent, d.p, cap, dn.p);
    c->stats.kernel_launches++;
    CU_TRY(cudaGetLastError());
    int cnt = 0;
    CU_TRY(cudaMemcpyAsync(&cnt, dn.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(cudaStreamSynchronize(c->stream));
    const int m = cnt < cap ? cnt : cap;
    if (m > 0) CU_TRY(cudaMemcpy(out_points, d.p, sizeof(double) * 3 * m, cudaMemcpyDeviceToHost));
    *n = cnt;
    return 0;
}

// ---- obstacle gather (plan_manager.cpp:232-254 / pcs:182-216) -------------------------------------------------------------
struct GatherBox { int a0[3], a1[3], l0[3], l1[3]; };
__device__ __forceinline__ bool gather_includes(const DevGrid &G, const GatherBox &b, int i, int j, int k) {
    if (i < b.a0[0] || i > b.a1[0] || j < b.a0[1] || j > b.a1[1] || k < b.a0[2] || k > b.a1[2]) return false;
    if (!(i > b.l1[0] || i < b.l0[0] || j > b.l1[1] || j < b.l0[1] || k > b.l1[2] || k < b.l0[2])) return false;
    return (G.bits[((size_t)i * G.Y + j) * G.Zw + (k >> 5)] >> (k & 31)) & 1u;
}
// Obstacle gather, one CTA per waypoint, three launches: k_gather_boxes (index boxes of every waypoint), k_gather_points<false> (how many
// voxels each waypoint emits: a voxel belongs to the FIRST waypoint whose box includes it) and, after an exclusive scan over the waypoints
// inside the kernel, k_gather_points<true> (ordered compaction inside the CTA at the waypoint's offset). Output order = the reference's:
// waypoint by waypoint, each box in x -> y -> z order.
__global__ void k_gather_boxes(const DevGrid G, const double *wps, int nQ, double h, double ox, double oy, double oz, GatherBox *boxes) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nQ) return;
    GatherBox b;
    const double c[3] = {wps[3 * q] + ox, wps[3 * q + 1] + oy, wps[3 * q + 2] + oz};
    const double l[3] = {q == 0 ? 999.0 : wps[3 * (q - 1)], q == 0 ? 999.0 : wps[3 * (q - 1) + 1], q == 0 ? 999.0 : wps[3 * (q - 1) + 2]};
    const int dims[3] = {G.X, G.Y, G.Z};
    for (int a = 0; a < 3; a++) {
        b.a0[a] = grid_axis_index(c[a] - h, G.bmin[a], G.bmax[a], G.res, dims[a]); b.a1[a] = grid_axis_index(c[a] + h, G.bmin[a], G.bmax[a], G.res, dims[a]);
        b.l0[a] = grid_axis_index(l[a] - h, G.bmin[a], G.bmax[a], G.res, dims[a]); b.l1[a] = grid_axis_index(l[a] + h, G.bmin[a], G.bmax[a], G.res, dims[a]);
    }
    boxes[q] = b;
}
template <bool WRITE>
__global__ void __launch_bounds__(256) k_gather_points(const DevGrid G, int nQ, const GatherBox *boxes, int *counts, double *out, int cap, int *count) {
    __shared__ int warp_cnt[8];
    __shared__ int running;
    const int q = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        int off = 0;
        if (WRITE) { for (int p = 0; p < q; p++) off += counts[p]; if (q == nQ - 1) *count = off + counts[q]; }
        running = off;
    }
    __syncthreads();
    const GatherBox b = boxes[q];
    const int ny = b.a1[1] - b.a0[1] + 1, nz = b.a1[2] - b.a0[2] + 1;
    const int nvox = (b.a1[0] - b.a0[0] + 1) * ny * nz;
    for (int base = 0; base < nvox; base += blockDim.x) {
        const int v = base + threadIdx.x;
        bool emit = false; int i = 0, j = 0, k = 0;
        if (v < nvox) {
            i = b.a0[0] + v / (ny * nz); j = b.a0[1] + (v / nz) % ny; k = b.a0[2] + v % nz;
            emit = gather_includes(G, b, i, j, k);
            for (int p = 0; emit && p < q; p++) if (gather_includes(G, boxes[p], i, j, k)) emit = false;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, emit);
        if (lane == 0) warp_cnt[warp] = __popc(bal);
        __syncthreads();
        if (WRITE) {
            int off = running;
            for (int w = 0; w < warp; w++) off += warp_cnt[w];
            if (emit) {
                const int pos = off + __popc(bal & ((1u << lane) - 1u));
                if (pos < cap) { out[3 * pos] = (i + 0.5) * G.res + G.bmin[0]; out[3 * pos + 1] = (j + 0.5) * G.res + G.bmin[1]; out[3 * pos + 2] = (k + 0.5) * G.res + G.bmin[2]; }
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int w = 0; w < 8; w++) t += warp_cnt[w]; running += t; }
        __syncthreads();
    }
    if (!WRITE && threadIdx.x == 0) counts[q] = running;
}

extern "C" int isdf_gather_obstacle_points(isdf_ctx *c, const double *waypoints, int nQ, double half_extent, const double *offset,
                                           double *out_points, int cap, int *n, int set_as_points) {
    if (!c || !waypoints || nQ < 1 || !n || cap < 0 || (cap > 0 && !out_points && !set_as_points)) return fail(ISDF_ERR_INVALID, "bad argument");
    if (!c->have_map) return fail(ISDF_ERR_STATE, "map not set");
    if (set_device(c)) return ISDF_ERR_CUDA;
    ScopedDevBuf<double> dw, dout; ScopedDevBuf<GatherBox> db; ScopedDevBuf<int> dn;
    const int capd = cap > 0 ? cap : 1;
    CU_TRY(dw.upload(waypoints, (size_t)3 * nQ, c->stream));
    CU_TRY(dout.ensure((size_t)3 * capd)); CU_TRY(db.ensure(nQ)); CU_TRY(dn.ensure((size_t)nQ + 1));
    const double ox = offset ? offset[0] : 0.0, oy = offset ? offset[1] : 0.0, oz = offset ? offset[2] : 0.0;
    k_gather_boxes<<<(nQ + 127) / 128, 128, 0, c->stream>>>(c->grid, dw.p, nQ, half_extent, ox, oy, oz, db.p);
    k_gather_points<false><<<nQ, 256, 0, c->stream>>>(c->grid, nQ, db.p, dn.p + 1, nullptr, 0, dn.p);
    k_gather_points<true><<<nQ, 256, 0, c->stream>>>(c->grid, nQ, db.p, dn.p + 1, dout.p, capd, dn.p);
    c->stats.kernel_launches += 3;
    CU_TRY(cudaGetLastError());
    int cnt = 0;
    CU_TRY(cudaMemcpyAsync(&cnt, dn.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(cudaStreamSynchronize(c->stream));
    *n = cnt;
    const int m = cnt < cap ? cnt : cap;
    int rc = 0;
    if (m > 0 && out_points) CU_TRY(cudaMemcpy(out_points, dout.p, sizeof(double) * 3 * m, cudaMemcpyDeviceToHost));
    if (set_as_points) {
        if (cnt > cap) rc = fail(ISDF_ERR_INVALID, "cap smaller than the obstacle list");
        else {
            std::vector<double> tmp((size_t)3 * (m > 0 ? m : 1));
            if (m > 0) CU_TRY(cudaMemcpy(tmp.data(), dout.p, sizeof(double) * 3 * m, cudaMemcpyDeviceToHost));
            cudaError_t e = c->sv.set_points(tmp.data(), m, c->stream);
            if (e != cudaSuccess) rc = fail(ISDF_ERR_CUDA, cudaGetErrorString(e));
        }
    }
    return rc;
}

// ---- discrete evaluation ------------------------------------------------------------------------------------
static int launch_discrete(isdf_ctx *c, int N, const double *d_T, const double *d_C, double *d_out, cudaStream_t st) {
    const int K = c->cfg.integral_intervs;
    const long long S = (long long)N * (K + 1);
    if (S > 0x7fffffffll) return fail(ISDF_ERR_UNSUPPORTED, "N * (integral_intervs + 1) must fit in 31 bits");
    CU_TRY(c->d_piece_cost.ensure(N));
    if (c->d_tickets.n < 2) {   // [0] pieces_done of the epilogue, [1] work-item cursor of the persistent scan warps
        CU_TRY(c->d_tickets.ensure(2));
        CU_TRY(cudaMemsetAsync(c->d_tickets.p, 0, 2 * sizeof(int), st));
    }
    CU_TRY(c->d_tot.ensure((size_t)S * 8));
    DiscArgs A;
    A.cfg = c->dcfg; A.grid = c->grid; A.shape = c->shape; A.N = N; A.T = d_T; A.C = d_C;
    A.tot = c->d_tot.p; A.pieces_done = c->d_tickets.p; A.item_cursor = c->d_tickets.p + 1;
    A.piece_cost = c->d_piece_cost.p; A.out = d_out; A.pair_counter = c->d_counter.p; A.count_out = c->count_out_dev;
    A.rank = c->rank; A.world = c->world;
    A.peer = PeerArgs{};
    const bool fused = c->peer_fused && c->peer.world > 1 && c->world > 1;   // an unsharded call (isdf_set_shard(ctx, 0, 1)) stays local
    if (fused) {
        if (c->peer.world != c->world || c->peer.rank != c->rank) return fail(ISDF_ERR_STATE, "peer group does not match isdf_set_shard");
        if (19 * N + 1 > c->peer.cap) return fail(ISDF_ERR_INVALID, "peer exchange buffer too small for this N (isdf_peer_export max_doubles)");
        A.peer = c->peer; A.peer.epoch = c->peer.epoch + 1;   // committed below, once the exchange kernel is really enqueued
    }
    A.dbg = nullptr;
    A.trace = nullptr;
    if (c->dbg_on) { CU_TRY(c->d_dbg.ensure((size_t)3 * S)); CU_TRY(cudaMemsetAsync(c->d_dbg.p, 0, sizeof(unsigned long long) * 3 * S, st)); A.dbg = c->d_dbg.p; }
    const long long M = (S - c->rank + c->world - 1) / c->world;
    CU_TRY(cudaMemsetAsync(c->d_counter.p, 0, sizeof(unsigned long long), st));
    // longest-first order from the previous evaluation of the same problem shape (first evaluation: natural order)
    const long long sig = ((long long)N << 20) ^ ((long long)c->rank << 10) ^ c->world ^ ((long long)K << 40);
    const bool mesh = (c->shape.kind == ISDF_SHAPE_MESH);
    // only mesh samples have a heavy tail worth splitting. Every sample of a launch may be split (item trace at world = 8, profiles/r02_tuning.md:
    // with M/4 slots the 515 heaviest samples were split and the NEXT heaviest — unsplit, 15-25 queries, 80-110 us — set the kernel time)
    const int max_split = mesh ? (int)std::min<long long>(M, MAX_SPLIT_SLOTS) : 0;
    const size_t max_items = (size_t)M + (size_t)(ROW_CLASSES - 1) * max_split;
    CU_TRY(c->d_work.ensure((size_t)S));
    if (c->d_items.n < 3 * max_items + (size_t)M) { CU_TRY(c->d_items.ensure(3 * max_items + (size_t)M)); c->order_for = -1; }   // a regrown table holds no items yet
    CU_TRY(c->d_item_count.ensure(1));
    CU_TRY(c->d_subsum.ensure((size_t)std::max(max_split, 1) * ROW_CLASSES * 8));
    if (c->d_split_work.n < (size_t)std::max(max_split, 1)) {
        CU_TRY(c->d_split_work.ensure((size_t)std::max(max_split, 1)));
        CU_TRY(cudaMemsetAsync(c->d_split_work.p, 0, sizeof(unsigned) * std::max(max_split, 1), st));
    }
    if (c->d_split_done.n < (size_t)std::max(max_split, 1)) {
        CU_TRY(c->d_split_done.ensure((size_t)std::max(max_split, 1)));
        CU_TRY(cudaMemsetAsync(c->d_split_done.p, 0, sizeof(unsigned) * std::max(max_split, 1), st));
    }
    A.work = c->d_work.p;
    if (c->dbg_on) { CU_TRY(c->d_trace.ensure(TRACE_STRIDE * max_items)); CU_TRY(cudaMemsetAsync(c->d_trace.p, 0, sizeof(unsigned long long) * TRACE_STRIDE * max_items, st)); A.trace = c->d_trace.p; }
    // a launch with far more samples than resident warps (batched callbacks: millions) balances itself through the persistent warps'
    // dynamic item counter: sorting / splitting would only cost a long single-CTA pass over the work array
    const bool want_items = !c->no_items && M <= 1024ll * ITEMS_CACHE * 4;
    const bool have_items = (c->order_for == sig) && want_items;
    A.items = have_items ? c->d_items.p : nullptr;
    A.item_count = c->d_item_count.p; A.subsum = c->d_subsum.p; A.split_work = c->d_split_work.p; A.split_done = c->d_split_done.p;
    // persistent grid: one CTA per resident slot (or fewer when there are fewer items than warps)
    const long long want = ((have_items ? (long long)max_items : M) + DISC_WARPS - 1) / DISC_WARPS;
    const long long resident = (long long)c->sm_count * (mesh ? c->mesh_blocks : c->analytic_blocks);
    const unsigned grid = (unsigned)std::max<long long>(1, std::min(want, resident));
    if (c->items_pending) CU_TRY(cudaStreamWaitEvent(st, c->ev_items_done, 0));   // the table this launch reads (or overwrites next)
    CU_TRY(discrete_launch_scan(A, mesh, grid, st));
    CU_TRY(discrete_launch_epilogue(A, st));
    if (fused) c->peer.epoch = A.peer.epoch;
    // build the next evaluation's work items on the aux stream: overlaps the caller's D2H / all-reduce / host work
    if (want_items) {
        CU_TRY(cudaEventRecord(c->ev_main_done, st));
        CU_TRY(cudaStreamWaitEvent(c->aux_stream, c->ev_main_done, 0));
        CU_TRY(discrete_launch_build_items(c->d_work.p, c->rank, c->world, (int)M, max_split, c->warp_slots_override > 0 ? c->warp_slots_override : c->warp_slots, c->d_items.p, c->d_item_count.p, c->aux_stream));
        CU_TRY(cudaEventRecord(c->ev_items_done, c->aux_stream));
        c->items_pending = true;
        c->order_for = sig;
        c->stats.kernel_launches++;   // work-item builder
    }
    c->stats.kernel_launches += 2;   // scan kernel, epilogue
    c->stats.evals_discrete++;
    return 0;
}

static int check_eval_state(isdf_ctx *c, int N, bool need_map) {
    if (!c) return fail(ISDF_ERR_INVALID, "ctx is NULL");
    if (N < 1) return fail(ISDF_ERR_INVALID, "N < 1");
    const bool coll = (c->cfg.flags & ISDF_WITH_COLLISION) != 0;
    if (coll && !c->have_shape) return fail(ISDF_ERR_STATE, "shape not set");
    if (need_map && coll && !c->have_map) return fail(ISDF_ERR_STATE, "map not set");
    return 0;
}

extern "C" int isdf_eval_discrete_device(isdf_ctx *c, int N, const double *d_T, const double *d_coeffs, double *d_out, void *cuda_stream) {
    int r = check_eval_state(c, N, true);
    if (r) return r;
    if (!d_T || !d_coeffs || !d_out) return fail(ISDF_ERR_INVALID, "NULL device pointer");
    if (set_device(c)) return ISDF_ERR_CUDA;
    return launch_discrete(c, N, d_T, d_coeffs, d_out, (cudaStream_t)cuda_stream);
}

static void poison(double *cost) { if (cost) *cost = std::numeric_limits<double>::quiet_NaN(); }

extern "C" int isdf_eval_discrete(isdf_ctx *c, int N, const double *T, const double *coeffs, double *cost, double *gradC, double *gradT) {
    int r = check_eval_state(c, N, true);
    if (r) { poison(cost); return r; }
    if (!T || !coeffs || !cost || !gradC || !gradT) { poison(cost); return fail(ISDF_ERR_INVALID, "NULL argument"); }
    auto body = [&]() -> int {
        if (set_device(c)) return ISDF_ERR_CUDA;
        const size_t nin = (size_t)19 * N, nout = (size_t)19 * N + 1;
        // one pinned staging block, ONE copy each way: [coefficients 18N | durations N] in, [cost | gradC | gradT | pair count] out
        if (ensure_stage(c, nin + nout + 1)) return ISDF_ERR_CUDA;
        CU_TRY(c->d_C.ensure(nin)); CU_TRY(c->d_out.ensure(nout + 1));
        std::memcpy(c->h_stage, coeffs, sizeof(double) * 18 * N);
        std::memcpy(c->h_stage + 18 * (size_t)N, T, sizeof(double) * N);
        CU_TRY(cudaMemcpyAsync(c->d_C.p, c->h_stage, sizeof(double) * nin, cudaMemcpyHostToDevice, c->stream));
        CU_TRY(cudaEventRecord(c->ev0, c->stream));
        c->count_out_dev = c->d_out.p + nout;
        int rr = launch_discrete(c, N, c->d_C.p + 18 * (size_t)N, c->d_C.p, c->d_out.p, c->stream);
        c->count_out_dev = nullptr;
        if (rr) return rr;
        CU_TRY(cudaEventRecord(c->ev1, c->stream));
        double *h_out = c->h_stage + nin;
        CU_TRY(cudaMemcpyAsync(h_out, c->d_out.p, sizeof(double) * (nout + 1), cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(cudaStreamSynchronize(c->stream));
        unsigned long long pairs = 0;
        std::memcpy(&pairs, h_out + nout, sizeof(pairs));
        if (c->peer_fused && c->peer.world > 1 && c->world > 1 && isdf_peer_status(c) != ISDF_OK) return ISDF_ERR_CUDA;   // exchange timed out: the vector is NaN
        float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1);
        c->stats.last_kernel_ms = ms; c->stats.last_pairs = (int64_t)pairs;
        *cost += h_out[0];                                   // accumulate like hpp:539-550
        for (size_t k = 0; k < (size_t)18 * N; k++) gradC[k] += h_out[1 + k];
        for (int k = 0; k < N; k++) gradT[k] += h_out[1 + 18 * N + k];
        return 0;
    };
    r = body();
    if (r) poison(cost);
    return r;
}

extern "C" int isdf_get_piece_costs(isdf_ctx *c, double *piece_cost, int n) {
    if (!c || !piece_cost || n < 0) return fail(ISDF_ERR_INVALID, "bad argument");
    if ((size_t)n > c->d_piece_cost.n) return fail(ISDF_ERR_STATE, "no discrete evaluation with that many pieces yet");
    if (set_device(c)) return ISDF_ERR_CUDA;
    CU_TRY(cudaStreamSynchronize(c->stream));
    CU_TRY(cudaMemcpy(piece_cost, c->d_piece_cost.p, sizeof(double) * n, cudaMemcpyDeviceToHost));
    return 0;
}

// ---- batched optimiser callback on the device (MINCO -> time-integral term -> adjoint), SURVEY §8f row 1 ----------------------
static int callback_batch_launch(isdf_ctx *c, int B, int N0, const double *d_head, const double *d_tail, int bc_stride, double rho,
                                 const double *d_x, double *d_cost, double *d_grad, cudaStream_t st) {
    const size_t BN = (size_t)B * N0;
    const size_t smem = minco_smem_bytes(N0);
    if (smem > 220 * 1024) return fail(ISDF_ERR_UNSUPPORTED, "pieces per problem too large for the shared-memory banded solver (N0 <= 290)");
    if (BN * (size_t)(c->cfg.integral_intervs + 1) > 0x7fffffffull) return fail(ISDF_ERR_UNSUPPORTED, "batch too large: B*N0*(K+1) must fit in 31 bits");
    CU_TRY(c->d_mT.ensure(BN)); CU_TRY(c->d_mC.ensure(18 * BN)); CU_TRY(c->d_mlu.ensure(78 * BN)); CU_TRY(c->d_men.ensure(B));
    CU_TRY(c->d_mgC.ensure(18 * BN)); CU_TRY(c->d_mgT.ensure(BN)); CU_TRY(c->d_mout.ensure(19 * BN + 1));
    MincoArgs M;
    M.B = B; M.N = N0; M.x = d_x; M.head = d_head; M.tail = d_tail; M.bc_stride = bc_stride; M.rho = rho;
    M.T = c->d_mT.p; M.C = c->d_mC.p; M.lu = c->d_mlu.p; M.energy = c->d_men.p; M.gC_e = c->d_mgC.p; M.gT_e = c->d_mgT.p;
    M.disc_out = nullptr; M.piece_cost = nullptr; M.cost = d_cost; M.grad = d_grad;
    // per-problem obstacle point sets registered for exactly this batch (isdf_set_points_batch): the LIVE composition of costFunctionLmbm
    // (hpp:386-405) — swept-volume term, then time-integral term
    const bool with_swept = (c->sv.B == B);
    M.Cpp = nullptr; M.sv_out = nullptr;
    if (with_swept) {
        if (c->shape.kind == ISDF_SHAPE_MESH && c->shape.mesh.sign_mode == MESH_SIGN_WINDING)
            return fail(ISDF_ERR_UNSUPPORTED, "swept-volume term with a winding-sign mesh (see isdf_set_shape_mesh_ex)");
        CU_TRY(c->d_mCpp.ensure(18 * BN)); CU_TRY(c->d_msv.ensure((size_t)B * (19 * (size_t)N0 + 1)));
        M.Cpp = c->d_mCpp.p;
    }
    CU_TRY(cudaFuncSetAttribute(k_minco_forward, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CU_TRY(cudaFuncSetAttribute(k_minco_backward, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_minco_forward<<<B, 32, smem, st>>>(M);
    if (with_swept) {
        int launches = 0;
        cudaError_t e = c->sv.launch_batch(c->dcfg, c->shape, N0, M.T, M.Cpp, c->d_msv.p, st, &launches);
        c->stats.kernel_launches += launches;
        c->stats.evals_swept++;
        if (e != cudaSuccess) return fail(e == cudaErrorInvalidValue ? ISDF_ERR_INVALID : ISDF_ERR_CUDA, std::string("batched swept: ") + cudaGetErrorString(e));
        M.sv_out = c->d_msv.p;
    }
    int r = launch_discrete(c, (int)BN, M.T, M.C, c->d_mout.p, st);
    if (r) return r;
    M.disc_out = c->d_mout.p; M.piece_cost = c->d_piece_cost.p;
    k_minco_backward<<<B, 32, smem, st>>>(M);
    c->stats.kernel_launches += 2;
    c->minco_B = B; c->minco_N = N0;
    CU_TRY(cudaGetLastError());
    return 0;
}

static int callback_batch_check(isdf_ctx *c, int B, int N0) {
    if (!c) return fail(ISDF_ERR_INVALID, "ctx is NULL");
    if (B < 1 || N0 < 1) return fail(ISDF_ERR_INVALID, "B < 1 or N0 < 1");
    if ((long long)B * N0 > 0x7fffffffll) return fail(ISDF_ERR_INVALID, "B*N0 overflows");
    if (c->world != 1) return fail(ISDF_ERR_STATE, "the batched callback shards by PROBLEM: keep isdf_set_shard(ctx, 0, 1) and give each rank its own problems");
    return check_eval_state(c, B * N0, true);
}

extern "C" int isdf_callback_batch_device(isdf_ctx *c, int B, int N0, const double *d_head, const double *d_tail, int per_problem_bc, double rho,
                                          const double *d_x, double *d_cost, double *d_grad, void *cuda_stream) {
    int r = callback_batch_check(c, B, N0);
    if (r) return r;
    if (!d_head || !d_tail || !d_x || !d_cost || !d_grad) return fail(ISDF_ERR_INVALID, "NULL device pointer");
    if (set_device(c)) return ISDF_ERR_CUDA;
    return callback_batch_launch(c, B, N0, d_head, d_tail, per_problem_bc ? 9 : 0, rho, d_x, d_cost, d_grad, (cudaStream_t)cuda_stream);
}

extern "C" int isdf_callback_batch(isdf_ctx *c, int B, int N0, const double *head, const double *tail, int per_problem_bc, double rho,
                                   const double *x, double *cost, double *grad) {
    auto poison_all = [&]() { if (cost && B > 0) for (int b = 0; b < B; b++) cost[b] = std::numeric_limits<double>::quiet_NaN(); };
    int r = callback_batch_check(c, B, N0);
    if (r) { poison_all(); return r; }
    if (!head || !tail || !x || !cost || !grad) { poison_all(); return fail(ISDF_ERR_INVALID, "NULL argument"); }
    auto body = [&]() -> int {
        if (set_device(c)) return ISDF_ERR_CUDA;
        const size_t dim = (size_t)N0 + 3 * (size_t)(N0 - 1), nbc = per_problem_bc ? (size_t)9 * B : 9;
        CU_TRY(c->d_mx.upload(x, dim * B, c->stream));
        CU_TRY(c->d_mbc.ensure(2 * nbc));
        CU_TRY(cudaMemcpyAsync(c->d_mbc.p, head, sizeof(double) * nbc, cudaMemcpyHostToDevice, c->stream));
        CU_TRY(cudaMemcpyAsync(c->d_mbc.p + nbc, tail, sizeof(double) * nbc, cudaMemcpyHostToDevice, c->stream));
        CU_TRY(c->d_mcost.ensure(B)); CU_TRY(c->d_mgrad.ensure(dim * B));
        CU_TRY(cudaEventRecord(c->ev0, c->stream));
        int rr = callback_batch_launch(c, B, N0, c->d_mbc.p, c->d_mbc.p + nbc, per_problem_bc ? 9 : 0, rho, c->d_mx.p, c->d_mcost.p, c->d_mgrad.p, c->stream);
        if (rr) return rr;
        CU_TRY(cudaEventRecord(c->ev1, c->stream));
        CU_TRY(cudaMemcpyAsync(cost, c->d_mcost.p, sizeof(double) * B, cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(cudaMemcpyAsync(grad, c->d_mgrad.p, sizeof(double) * dim * B, cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(cudaStreamSynchronize(c->stream));
        float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1);
        c->stats.last_kernel_ms = ms;
        return 0;
    };
    r = body();
    if (r) poison_all();
    return r;
}

// ---- device-resident lock-step L-BFGS over the batched callback (SURVEY §8f row 2; isdf_lbfgs.cuh) ----------------------------------------
static int lbfgs_check(const isdf_lbfgs_params *p) {
    if (!p) return fail(ISDF_ERR_INVALID, "params is NULL");
    if (p->mem_size <= 0 || p->mem_size > 64) return fail(ISDF_ERR_INVALID, "mem_size out of range (1..64)");
    if (p->past < 0 || p->g_epsilon < 0.0 || p->delta < 0.0 || p->min_step < 0.0 || p->max_step < p->min_step || !(p->f_dec_coeff > 0.0 && p->f_dec_coeff < 1.0) ||
        !(p->machine_prec > 0.0) || p->max_linesearch <= 0 || p->max_iterations < 0 || p->max_rounds < 0)
        return fail(ISDF_ERR_INVALID, "L-BFGS parameter out of range");
    return 0;
}

extern "C" int isdf_lbfgs_default_params(isdf_lbfgs_params *p) {
    if (!p) return fail(ISDF_ERR_INVALID, "params is NULL");
    // lbfgs_parameter_t defaults (lbfgs.hpp:40-142) with the back end's settings (config_CappedCone.yaml:99-102: mem 16, past 10, min_step 1e-32, g_epsilon 0)
    p->mem_size = 16; p->past = 10; p->max_iterations = 0; p->max_linesearch = 64; p->max_rounds = 0;
    p->g_epsilon = 0.0; p->delta = 1.0e-6; p->min_step = 1.0e-32; p->max_step = 1.0e+20; p->f_dec_coeff = 1.0e-4; p->cautious_factor = 1.0e-6; p->machine_prec = 1.0e-16;
    return 0;
}

// d_x: B x n (in: starting points, out: solutions); d_f: B; d_ret / d_iterations / d_evaluations: B ints (any of the three may be null).
// Synchronous with respect to the host (one 4-byte read per round decides termination), all data stays on the device.
extern "C" int isdf_lbfgs_batch_device(isdf_ctx *c, int B, int N0, const double *d_head, const double *d_tail, int per_problem_bc, double rho,
                                       const isdf_lbfgs_params *prm, double *d_x, double *d_f, int *d_ret, int *d_iterations, int *d_evaluations,
                                       int *rounds_out, void *cuda_stream) {
    int r = callback_batch_check(c, B, N0);
    if (r) return r;
    if ((r = lbfgs_check(prm))) return r;
    if (!d_head || !d_tail || !d_x || !d_f) return fail(ISDF_ERR_INVALID, "NULL device pointer");
    if (set_device(c)) return ISDF_ERR_CUDA;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const int n = 4 * N0 - 3, m = prm->mem_size, npf = prm->past > 1 ? prm->past : 1;
    const size_t per = (size_t)4 * n + npf + 2 * (size_t)m + 2 * (size_t)m * n + LB_NSCALAR;   // doubles of state per instance
    CU_TRY(c->d_lb_state.ensure(per * B)); CU_TRY(c->d_lb_grad.ensure((size_t)B * n)); CU_TRY(c->d_lb_int.ensure((size_t)B * LB_NINT + 4));
    if (!c->h_lb_active) CU_TRY(cudaMallocHost((void **)&c->h_lb_active, sizeof(int)));
    CU_TRY(cudaMemsetAsync(c->d_lb_state.p, 0, sizeof(double) * per * B, st));
    CU_TRY(cudaMemsetAsync(c->d_lb_int.p, 0, sizeof(int) * ((size_t)B * LB_NINT + 4), st));   // phase = WANT_INIT
    LbfgsArgs L;
    L.B = B; L.n = n;
    L.pr.mem_size = m; L.pr.past = prm->past; L.pr.max_iterations = prm->max_iterations; L.pr.max_linesearch = prm->max_linesearch;
    L.pr.g_epsilon = prm->g_epsilon; L.pr.delta = prm->delta; L.pr.min_step = prm->min_step; L.pr.max_step = prm->max_step;
    L.pr.f_dec_coeff = prm->f_dec_coeff; L.pr.cautious_factor = prm->cautious_factor; L.pr.machine_prec = prm->machine_prec;
    double *p = c->d_lb_state.p;
    L.x = d_x; L.f = d_f; L.grad = c->d_lb_grad.p;
    L.xp = p; p += (size_t)B * n; L.g = p; p += (size_t)B * n; L.gp = p; p += (size_t)B * n; L.d = p; p += (size_t)B * n;
    L.pf = p; p += (size_t)B * npf; L.alpha = p; p += (size_t)B * m; L.ys = p; p += (size_t)B * m;
    L.S = p; p += (size_t)B * m * n; L.Y = p; p += (size_t)B * m * n; L.sc = p;
    L.st = c->d_lb_int.p; L.active = c->d_lb_int.p + (size_t)B * LB_NINT;
    // olddnorm starts at 1 (lbfgs.hpp:541): scalar slot 2 of every instance
    {
        std::vector<double> init((size_t)B * LB_NSCALAR, 0.0);
        for (int b = 0; b < B; b++) init[(size_t)b * LB_NSCALAR + 2] = 1.0;
        CU_TRY(cudaMemcpyAsync(L.sc, init.data(), sizeof(double) * init.size(), cudaMemcpyHostToDevice, st));
        CU_TRY(cudaStreamSynchronize(st));
    }
    int rounds = 0;
    for (;;) {
        // every instance's requested point is evaluated (finished instances ride along unchanged: their state is frozen)
        r = callback_batch_launch(c, B, N0, d_head, d_tail, per_problem_bc ? 9 : 0, rho, d_x, d_f, c->d_lb_grad.p, st);
        if (r) return r;
        CU_TRY(cudaMemsetAsync(L.active, 0, sizeof(int), st));
        k_lbfgs_feed<<<(unsigned)((B + 63) / 64), 64, 0, st>>>(L);
        c->stats.kernel_launches++;
        CU_TRY(cudaGetLastError());
        CU_TRY(cudaMemcpyAsync(c->h_lb_active, L.active, sizeof(int), cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
        ++rounds;
        if (*c->h_lb_active == 0) break;
        if (prm->max_rounds > 0 && rounds >= prm->max_rounds) break;
    }
    // results: f = fx of every instance (scalar slot 0), return codes and counters
    CU_TRY(cudaMemcpy2DAsync(d_f, sizeof(double), L.sc, sizeof(double) * LB_NSCALAR, sizeof(double), B, cudaMemcpyDeviceToDevice, st));
    if (d_ret) CU_TRY(cudaMemcpy2DAsync(d_ret, sizeof(int), L.st + 1, sizeof(int) * LB_NINT, sizeof(int), B, cudaMemcpyDeviceToDevice, st));
    if (d_iterations) CU_TRY(cudaMemcpy2DAsync(d_iterations, sizeof(int), L.st + 8, sizeof(int) * LB_NINT, sizeof(int), B, cudaMemcpyDeviceToDevice, st));
    if (d_evaluations) CU_TRY(cudaMemcpy2DAsync(d_evaluations, sizeof(int), L.st + 9, sizeof(int) * LB_NINT, sizeof(int), B, cudaMemcpyDeviceToDevice, st));
    CU_TRY(cudaStreamSynchronize(st));
    if (rounds_out) *rounds_out = rounds;
    return 0;
}

extern "C" int isdf_lbfgs_batch(isdf_ctx *c, int B, int N0, const double *head, const double *tail, int per_problem_bc, double rho,
                                const isdf_lbfgs_params *prm, double *x, double *f, int *ret, int *iterations, int *evaluations, int *rounds_out) {
    int r = callback_batch_check(c, B, N0);
    if (r) return r;
    if (!head || !tail || !x || !f) return fail(ISDF_ERR_INVALID, "NULL argument");
    if (set_device(c)) return ISDF_ERR_CUDA;
    const size_t n = (size_t)4 * N0 - 3, nbc = per_problem_bc ? (size_t)9 * B : 9;
    CU_TRY(c->d_lb_x.upload(x, n * B, c->stream));
    CU_TRY(c->d_mbc.ensure(2 * nbc));
    CU_TRY(cudaMemcpyAsync(c->d_mbc.p, head, sizeof(double) * nbc, cudaMemcpyHostToDevice, c->stream));
    CU_TRY(cudaMemcpyAsync(c->d_mbc.p + nbc, tail, sizeof(double) * nbc, cudaMemcpyHostToDevice, c->stream));
    CU_TRY(c->d_lb_f.ensure(B)); CU_TRY(c->d_lb_head.ensure((size_t)3 * B));
    r = isdf_lbfgs_batch_device(c, B, N0, c->d_mbc.p, c->d_mbc.p + nbc, per_problem_bc, rho, prm, c->d_lb_x.p, c->d_lb_f.p, c->d_lb_head.p, c->d_lb_head.p + B,
                                c->d_lb_head.p + 2 * (size_t)B, rounds_out, c->stream);
    if (r) return r;
    CU_TRY(cudaMemcpy(x, c->d_lb_x.p, sizeof(double) * n * B, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(f, c->d_lb_f.p, sizeof(double) * B, cudaMemcpyDeviceToHost));
    if (ret) CU_TRY(cudaMemcpy(ret, c->d_lb_head.p, sizeof(int) * B, cudaMemcpyDeviceToHost));
    if (iterations) CU_TRY(cudaMemcpy(iterations, c->d_lb_head.p + B, sizeof(int) * B, cudaMemcpyDeviceToHost));
    if (evaluations) CU_TRY(cudaMemcpy(evaluations, c->d_lb_head.p + 2 * (size_t)B, sizeof(int) * B, cudaMemcpyDeviceToHost));
    return 0;
}

extern "C" int isdf_get_batch_trajectories(isdf_ctx *c, double *T, double *coeffs, double *energy) {
    if (!c) return fail(ISDF_ERR_INVALID, "ctx is NULL");
    if (c->minco_B <= 0) return fail(ISDF_ERR_STATE, "no batched callback evaluated yet");
    if (set_device(c)) return ISDF_ERR_CUDA;
    const size_t BN = (size_t)c->minco_B * c->minco_N;
    CU_TRY(cudaStreamSynchronize(c->stream));
    if (T) CU_TRY(cudaMemcpy(T, c->d_mT.p, sizeof(double) * BN, cudaMemcpyDeviceToHost));
    if (coeffs) CU_TRY(cudaMemcpy(coeffs, c->d_mC.p, sizeof(double) * 18 * BN, cudaMemcpyDeviceToHost));
    if (energy) CU_TRY(cudaMemcpy(energy, c->d_men.p, sizeof(double) * c->minco_B, cudaMemcpyDeviceToHost));
    return 0;
}

// ---- multi-GPU: rank-ordered sum of the sharded evaluation through NVLink peer memory (isdf_peer.cuh) ------------------------------
static size_t peer_bytes(int world, int cap) { return sizeof(unsigned long long) * 2 * PEER_MAX + sizeof(double) * 2 * (size_t)world * cap; }

extern "C" int isdf_peer_export(isdf_ctx *c, int world, int max_doubles, unsigned char *handle64) {
    if (!c || !handle64 || world < 2 || world > PEER_MAX || max_doubles < 1) return fail(ISDF_ERR_INVALID, "bad argument (2 <= world <= 16)");
    if (set_device(c)) return ISDF_ERR_CUDA;
    if (c->peer.world) return fail(ISDF_ERR_STATE, "already connected: isdf_peer_disconnect first");
    if (c->peer_buf) { cudaFree(c->peer_buf); c->peer_buf = nullptr; }
    CU_TRY(cudaMalloc(&c->peer_buf, peer_bytes(world, max_doubles)));
    CU_TRY(cudaMemset(c->peer_buf, 0, peer_bytes(world, max_doubles)));
    CU_TRY(c->d_peer_status.ensure(1));
    CU_TRY(cudaMemset(c->d_peer_status.p, 0, sizeof(int)));
    cudaIpcMemHandle_t h;
    CU_TRY(cudaIpcGetMemHandle(&h, c->peer_buf));
    static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
    std::memcpy(handle64, &h, 64);
    c->peer_world_alloc = world; c->peer_cap = max_doubles;
    return 0;
}

extern "C" int isdf_peer_connect(isdf_ctx *c, int world, int rank, const unsigned char *handles, int fuse_into_eval) {
    if (!c || !handles || rank < 0 || rank >= world) return fail(ISDF_ERR_INVALID, "bad argument");
    if (!c->peer_buf || world != c->peer_world_alloc) return fail(ISDF_ERR_STATE, "isdf_peer_export with the same world first");
    if (c->peer.world != 0) return fail(ISDF_ERR_STATE, "already connected: isdf_peer_disconnect first");
    if (set_device(c)) return ISDF_ERR_CUDA;
    PeerArgs P = {};
    P.world = world; P.rank = rank; P.cap = c->peer_cap; P.epoch = 0; P.status = c->d_peer_status.p;
    for (int p = 0; p < world; p++) {
        void *base = c->peer_buf;
        if (p != rank) {
            cudaIpcMemHandle_t h;
            std::memcpy(&h, handles + (size_t)64 * p, 64);
            cudaError_t e = cudaIpcOpenMemHandle(&base, h, cudaIpcMemLazyEnablePeerAccess);
            if (e != cudaSuccess) {
                for (int q = 0; q < p; q++) if (c->peer_open[q]) { cudaIpcCloseMemHandle(c->peer_open[q]); c->peer_open[q] = nullptr; }
                return fail(ISDF_ERR_CUDA, std::string("cudaIpcOpenMemHandle: ") + cudaGetErrorString(e));
            }
            c->peer_open[p] = base;
        }
        P.flags[p] = (unsigned long long *)base;
        P.slots[p] = (double *)((char *)base + sizeof(unsigned long long) * 2 * PEER_MAX);
    }
    c->peer = P;
    c->peer_fused = fuse_into_eval != 0;
    return 0;
}

extern "C" int isdf_peer_allreduce_device(isdf_ctx *c, double *d_vec, int n, void *cuda_stream) {
    if (!c || !d_vec || n < 1) return fail(ISDF_ERR_INVALID, "bad argument");
    if (c->peer.world < 2) return fail(ISDF_ERR_STATE, "not connected (isdf_peer_connect)");
    if (n > c->peer.cap) return fail(ISDF_ERR_INVALID, "vector longer than the exchange buffer");
    if (set_device(c)) return ISDF_ERR_CUDA;
    PeerArgs P = c->peer;
    P.epoch = c->peer.epoch + 1;
    k_peer_allreduce<<<1, 512, 0, (cudaStream_t)cuda_stream>>>(P, d_vec, n);
    c->stats.kernel_launches++;
    CU_TRY(cudaGetLastError());
    c->peer.epoch = P.epoch;
    return 0;
}

extern "C" int isdf_peer_status(isdf_ctx *c) {
    if (!c) return fail(ISDF_ERR_INVALID, "ctx is NULL");
    if (!c->d_peer_status.p) return 0;
    if (set_device(c)) return ISDF_ERR_CUDA;
    int st = 0;
    CU_TRY(cudaMemcpy(&st, c->d_peer_status.p, sizeof(int), cudaMemcpyDeviceToHost));
    if (st) return fail(ISDF_ERR_CUDA, "peer exchange timed out: a rank did not reach the same evaluation");
    return 0;
}

extern "C" int isdf_peer_disconnect(isdf_ctx *c) {
    if (!c) return fail(ISDF_ERR_INVALID, "ctx is NULL");
    if (set_device(c)) return ISDF_ERR_CUDA;
    cudaDeviceSynchronize();
    for (int p = 0; p < PEER_MAX; p++) if (c->peer_open[p]) { cudaIpcCloseMemHandle(c->peer_open[p]); c->peer_open[p] = nullptr; }
    if (c->peer_buf) { cudaFree(c->peer_buf); c->peer_buf = nullptr; }
    c->peer = PeerArgs{}; c->peer_fused = false; c->peer_world_alloc = 0; c->peer_cap = 0;
    return 0;
}

// ---- front end: attitude-kernel feasibility (isdf_frontend.cuh), SURVEY §8f row 4 ------------------------------------------------
// Eigen::AngleAxisd(rotx, UnitX) * Eigen::AngleAxisd(roty, UnitY) -> Matrix3d (Shape.hpp:431): quaternion product, toRotationMatrix
static void attitude_rotation(double rotx, double roty, double R[9]) {
    const double sa = std::sin(0.5 * rotx), sb = std::sin(0.5 * roty);
    const double aw = std::cos(0.5 * rotx), ax = sa * 1.0, ay = sa * 0.0, az = sa * 0.0;
    const double bw = std::cos(0.5 * roty), bx = sb * 0.0, by = sb * 1.0, bz = sb * 0.0;
    const double w = aw * bw - ax * bx - ay * by - az * bz;
    const double x = aw * bx + ax * bw + ay * bz - az * by;
    const double y = aw * by + ay * bw + az * bx - ax * bz;
    const double z = aw * bz + az * bw + ax * by - ay * bx;
    const double tx = 2.0 * x, ty = 2.0 * y, tz = 2.0 * z;
    const double twx = tx * w, twy = ty * w, twz = tz * w, txx = tx * x, txy = ty * x, txz = tz * x, tyy = ty * y, tyz = tz * y, tzz = tz * z;
    R[0] = 1.0 - (tyy + tzz); R[1] = txy - twz; R[2] = txz + twy;
    R[3] = txy + twz; R[4] = 1.0 - (txx + tzz); R[5] = tyz - twx;
    R[6] = txz - twy; R[7] = tyz + twx; R[8] = 1.0 - (txx + tyy);
}

static FrontArgs front_args(isdf_ctx *c) {
    FrontArgs A = {};
    A.grid = c->grid; A.shape = c->shape;
    for (int i = 0; i < 9; i++) A.rot[i] = c->shape.rot[i];
    for (int i = 0; i < 3; i++) A.trans[i] = c->shape.trans[i];
    if (c->shape.kind != ISDF_SHAPE_MESH) {   // the kernel applies ((pos - trans) * Rotate) * R_obj itself and evaluates the bare body
        const double I[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
        for (int i = 0; i < 9; i++) A.shape.rot[i] = I[i];
        for (int i = 0; i < 3; i++) A.shape.trans[i] = 0.0;
    }
    A.ks = c->fe_ks; A.xk = c->fe_xk; A.yk = c->fe_yk; A.natt = c->fe_xk * c->fe_yk;
    A.res = c->cfg.occupancy_resolution; A.margin = c->fe_margin;
    A.att_rot = c->d_fe_rot.p; A.kernels = c->d_fe_kernels.p; A.offset_masks = c->d_fe_masks.p; A.order = c->d_fe_order.p;
    A.max_roll = c->fe_max_roll; A.max_pitch = c->fe_max_pitch; A.ang_res = c->fe_ang_res;
    A.core_rows = c->d_fe_core.p; A.ncore = c->fe_ncore; A.urows = c->d_fe_urows.p; A.nurow = c->fe_nurow; A.chunks = c->d_fe_chunks.p; A.nchunk = c->fe_nchunk; A.tab = c->d_fe_tab.p; A.ntab = c->fe_ntab; A.surv = c->d_fe_surv.p; A.surv_count = c->d_fe_count.p;
    return A;
}

extern "C" int isdf_frontend_build_kernels(isdf_ctx *c, const isdf_kernel_config *kc, int *xkernel_size, int *ykernel_size) {
    if (!c || !kc) return fail(ISDF_ERR_INVALID, "NULL argument");
    if (!c->have_shape) return fail(ISDF_ERR_STATE, "shape not set");
    if (!(kc->kernel_ang_res > 0) || kc->kernel_max_roll < 0 || kc->kernel_max_pitch < 0) return fail(ISDF_ERR_INVALID, "bad attitude grid");
    const int ks = c->cfg.kernel_size;
    if (ks < 1 || (ks & 1) == 0) return fail(ISDF_ERR_INVALID, "kernel_size must be odd (Shape.hpp:258)");
    if (ks > 29) return fail(ISDF_ERR_UNSUPPORTED, "kernel_size > 29");
    const int xk = (int)std::floor(2 * kc->kernel_max_roll / kc->kernel_ang_res) + 1, yk = (int)std::floor(2 * kc->kernel_max_pitch / kc->kernel_ang_res) + 1;   // swm:135-136
    if (xk * yk > FE_MAX_ATT) return fail(ISDF_ERR_UNSUPPORTED, "more than 128 attitudes");
    if (set_device(c)) return ISDF_ERR_CUDA;
    const int natt = xk * yk, n3 = ks * ks * ks;
    std::vector<double> rot((size_t)9 * natt, 0.0);
    {
        int i = 0;
        for (double roll = -kc->kernel_max_roll; roll <= kc->kernel_max_roll && i < xk; roll += kc->kernel_ang_res, i++) {   // Shape.hpp:424-427
            int j = 0;
            for (double pitch = -kc->kernel_max_pitch; pitch <= kc->kernel_max_pitch && j < yk; pitch += kc->kernel_ang_res, j++)
                attitude_rotation(roll * M_PI / 180.0, pitch * M_PI / 180.0, &rot[(size_t)9 * (i * yk + j)]);
        }
    }
    // visiting order of visit_kernels_by_distance for every start attitude: level pose, then the BFS sequence without it
    std::vector<uint8_t> order((size_t)natt * natt, 0xff);
    const int zi = (xk - 1) / 2, zj = (yk - 1) / 2;
    for (int sx = 0; sx < xk; sx++)
        for (int sy = 0; sy < yk; sy++) {
            uint8_t *o = &order[(size_t)(sx * yk + sy) * natt];
            int n = 0;
            o[n++] = (uint8_t)(zi * yk + zj);
            std::vector<uint8_t> vis((size_t)natt, 0);
            std::queue<std::pair<int, int>> q;
            q.push({sx, sy}); vis[sx * yk + sy] = 1;
            const int dirs[4][2] = {{0, 1}, {0, -1}, {1, 0}, {-1, 0}};
            int deep = 0;
            while (!q.empty()) {
                deep++;
                const int x = q.front().first, y = q.front().second;
                q.pop();
                if (x != zi || y != zj) o[n++] = (uint8_t)(x * yk + y);
                for (auto &d : dirs) {
                    const int nx = x + d[0], ny = y + d[1];
                    if (nx < 0 || nx >= xk || ny < 0 || ny >= yk || vis[nx * yk + ny]) continue;
                    vis[nx * yk + ny] = 1;
                    q.push({nx, ny});
                }
                if (deep > 800) break;   // maxdeepth (swm:852)
            }
        }
    CU_TRY(c->d_fe_rot.upload(rot.data(), rot.size(), c->stream));
    CU_TRY(c->d_fe_order.upload(order.data(), order.size(), c->stream));
    CU_TRY(c->d_fe_kernels.ensure((size_t)natt * n3));
    CU_TRY(c->d_fe_masks.ensure((size_t)4 * n3));
    c->fe_xk = xk; c->fe_yk = yk; c->fe_ks = ks;
    c->fe_max_roll = kc->kernel_max_roll; c->fe_max_pitch = kc->kernel_max_pitch; c->fe_ang_res = kc->kernel_ang_res;
    c->fe_margin = std::max(kc->front_end_safeh, c->cfg.occupancy_resolution / 2);   // Shape.hpp:423
    FrontArgs A = front_args(c);
    const long long nt = (long long)natt * n3;
    k_frontend_kernels<<<(unsigned)((nt + 255) / 256), 256, 0, c->stream>>>(A);
    k_frontend_offset_masks<<<(unsigned)((n3 + 255) / 256), 256, 0, c->stream>>>(A);
    c->stats.kernel_launches += 2;
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaStreamSynchronize(c->stream));
    // the kernel core (offsets every attitude occupies), row by row, densest rows first: pass 1 of the two-pass feasibility kernel
    {
        std::vector<uint32_t> om((size_t)4 * n3);
        CU_TRY(cudaMemcpy(om.data(), c->d_fe_masks.p, sizeof(uint32_t) * om.size(), cudaMemcpyDeviceToHost));
        uint32_t valid[4];
        for (int k = 0; k < 4; k++) { const int lo = 32 * k; valid[k] = natt >= lo + 32 ? 0xffffffffu : (natt > lo ? ((1u << (natt - lo)) - 1u) : 0u); }
        std::vector<uint2> rows, urows;
        for (int a = 0; a < ks; a++)
            for (int b = 0; b < ks; b++) {
                uint32_t bits = 0, ubits = 0;
                for (int cc = 0; cc < ks; cc++) {
                    const uint32_t *m = &om[(size_t)4 * ((a * ks + b) * ks + cc)];
                    if (m[0] == valid[0] && m[1] == valid[1] && m[2] == valid[2] && m[3] == valid[3]) bits |= 1u << cc;
                    if (m[0] | m[1] | m[2] | m[3]) ubits |= 1u << cc;
                }
                if (bits) rows.push_back(make_uint2((uint32_t)a | ((uint32_t)b << 8), bits));
                if (ubits) urows.push_back(make_uint2((uint32_t)a | ((uint32_t)b << 8), ubits));
            }
        c->fe_nurow = (int)urows.size();
        if (!urows.empty()) CU_TRY(c->d_fe_urows.upload(urows.data(), urows.size(), c->stream));
        // pattern tables of the union rows, in chunks of <= FE_CHUNK_BITS offsets (pass 2 of the table-driven kernels)
        std::vector<uint2> chunks; std::vector<uint4> tab;
        for (const uint2 &ur : urows) {
            const int a = (int)(ur.x & 0xffu), b = (int)(ur.x >> 8);
            const int lo = __builtin_ctz(ur.y), hi = 31 - __builtin_clz(ur.y);
            for (int c0 = lo; c0 <= hi; c0 += FE_CHUNK_BITS) {
                const int len = std::min(FE_CHUNK_BITS, hi - c0 + 1);
                if (((ur.y >> c0) & ((1u << len) - 1u)) == 0u) continue;
                chunks.push_back(make_uint2(ur.x | ((uint32_t)c0 << 16) | ((uint32_t)len << 24), (uint32_t)tab.size()));
                for (uint32_t pat = 0; pat < (1u << len); pat++) {
                    uint4 e = make_uint4(0u, 0u, 0u, 0u);
                    for (int i = 0; i < len; i++)
                        if ((pat >> i) & 1u) { const uint32_t *m = &om[(size_t)4 * ((a * ks + b) * ks + c0 + i)]; e.x |= m[0]; e.y |= m[1]; e.z |= m[2]; e.w |= m[3]; }
                    tab.push_back(e);
                }
            }
        }
        c->fe_nchunk = (int)chunks.size(); c->fe_ntab = (int)tab.size();
        if (getenv("ISDF_VERBOSE")) fprintf(stderr, "[isdf] front end: %d attitudes, kernel core %zu rows, union %zu rows, %zu chunks, %zu table entries (%.1f KB)\n", natt, rows.size(), urows.size(), chunks.size(), tab.size(), tab.size() * 16e-3);
        if (!chunks.empty()) { CU_TRY(c->d_fe_chunks.upload(chunks.data(), chunks.size(), c->stream)); CU_TRY(c->d_fe_tab.upload(tab.data(), tab.size(), c->stream)); }
        std::stable_sort(rows.begin(), rows.end(), [](const uint2 &p, const uint2 &q) { return __builtin_popcount(p.y) > __builtin_popcount(q.y); });
        c->fe_ncore = (int)rows.size();
        if (!rows.empty()) CU_TRY(c->d_fe_core.upload(rows.data(), rows.size(), c->stream));
        CU_TRY(cudaStreamSynchronize(c->stream));
    }
    c->fe_ready = true;
    if (xkernel_size) *xkernel_size = xk;
    if (ykernel_size) *ykernel_size = yk;
    return 0;
}

extern "C" int isdf_frontend_get_kernels(isdf_ctx *c, uint8_t *out, int n) {
    if (!c || !out) return fail(ISDF_ERR_INVALID, "NULL argument");
    if (!c->fe_ready) return fail(ISDF_ERR_STATE, "isdf_frontend_build_kernels first (and again after changing the shape)");
    const size_t want = (size_t)c->fe_xk * c->fe_yk * c->fe_ks * c->fe_ks * c->fe_ks;
    if ((size_t)n != want) return fail(ISDF_ERR_INVALID, "n must be xkernel_size * ykernel_size * kernel_size^3");
    if (set_device(c)) return ISDF_ERR_CUDA;
    CU_TRY(cudaMemcpy(out, c->d_fe_kernels.p, want, cudaMemcpyDeviceToHost));
    return 0;
}

static int frontend_state(isdf_ctx *c) {
    if (!c) return fail(ISDF_ERR_INVALID, "ctx is NULL");
    if (!c->fe_ready) return fail(ISDF_ERR_STATE, "isdf_frontend_build_kernels first (and again after changing the shape)");
    if (!c->have_map) return fail(ISDF_ERR_STATE, "map not set");
    return 0;
}

extern "C" int isdf_frontend_feasibility_device(isdf_ctx *c, uint32_t *d_masks, void *cuda_stream) {
    int r = frontend_state(c);
    if (r) return r;
    if (!d_masks) return fail(ISDF_ERR_INVALID, "NULL device pointer");
    if (set_device(c)) return ISDF_ERR_CUDA;
    FrontArgs A = front_args(c);
    A.out = d_masks;
    const size_t smem = sizeof(uint32_t) * 4 * (size_t)A.ks * A.ks * A.ks;
    CU_TRY(cudaFuncSetAttribute(k_frontend_feasibility, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long nrun = (long long)c->grid.X * c->grid.Y * ((c->grid.Z + FE_ZRUN - 1) / FE_ZRUN);
    const unsigned grid = (unsigned)std::min<long long>((nrun + 255) / 256, 148ll * 64);
    if (c->fe_ncore > 0 && nrun < (1ll << 32) && !getenv("ISDF_FE_ONE_PASS")) {
        // two passes: the kernel core settles most voxels of a cluttered map, the mask accumulation runs on the survivors only
        CU_TRY(c->d_fe_surv.ensure((size_t)nrun));
        CU_TRY(c->d_fe_count.ensure(1));
        A.surv = c->d_fe_surv.p; A.surv_count = c->d_fe_count.p;
        CU_TRY(cudaMemsetAsync(c->d_fe_count.p, 0, sizeof(unsigned), (cudaStream_t)cuda_stream));
        const size_t tsmem = sizeof(uint4) * ((size_t)c->fe_ntab + (size_t)c->fe_nchunk);
        if (c->fe_nchunk > 0 && tsmem <= 200 * 1024 && !getenv("ISDF_FE_NO_TABLES")) {
            // throughput form: zero-filled output, bit-parallel core pass (32 voxels per thread), table-driven accumulation on the survivors
            const long long nvox = (long long)c->grid.X * c->grid.Y * c->grid.Z;
            CU_TRY(cudaMemsetAsync(d_masks, 0, sizeof(uint32_t) * 4 * (size_t)nvox, (cudaStream_t)cuda_stream));
            const long long nword = (long long)c->grid.X * c->grid.Y * c->grid.Zw;
            CU_TRY(cudaFuncSetAttribute(k_frontend_survivors_tab, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tsmem));
            k_frontend_core_words<<<(unsigned)std::min<long long>((nword + 255) / 256, 148ll * 32), 256, 0, (cudaStream_t)cuda_stream>>>(A);
            // 32 warps per SM hide the row reads: two CTAs of 512 threads when two tables fit into shared memory, else one of 1024
            if (2 * (tsmem + 1024) <= 220 * 1024) k_frontend_survivors_tab<<<148 * 2, 512, tsmem, (cudaStream_t)cuda_stream>>>(A);
            else k_frontend_survivors_tab<<<148, 1024, tsmem, (cudaStream_t)cuda_stream>>>(A);
        } else {
            CU_TRY(cudaFuncSetAttribute(k_frontend_survivors, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            k_frontend_core<<<grid, 256, 0, (cudaStream_t)cuda_stream>>>(A);
            k_frontend_survivors<<<148 * 16, 256, smem, (cudaStream_t)cuda_stream>>>(A);
        }
        c->stats.kernel_launches += 2;
    } else {
        k_frontend_feasibility<<<grid, 256, smem, (cudaStream_t)cuda_stream>>>(A);
        c->stats.kernel_launches++;
    }
    CU_TRY(cudaGetLastError());
    return 0;
}

extern "C" int isdf_frontend_feasibility(isdf_ctx *c, uint32_t *masks) {
    int r = frontend_state(c);
    if (r) return r;
    if (!masks) return fail(ISDF_ERR_INVALID, "NULL argument");
    if (set_device(c)) return ISDF_ERR_CUDA;
    const size_t nvox = (size_t)c->grid.X * c->grid.Y * c->grid.Z;
    CU_TRY(c->d_fe_out.ensure(4 * nvox));
    CU_TRY(cudaEventRecord(c->ev0, c->stream));
    r = isdf_frontend_feasibility_device(c, c->d_fe_out.p, c->stream);
    if (r) return r;
    CU_TRY(cudaEventRecord(c->ev1, c->stream));
    CU_TRY(cudaMemcpyAsync(masks, c->d_fe_out.p, sizeof(uint32_t) * 4 * nvox, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(cudaStreamSynchronize(c->stream));
    float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1);
    c->stats.last_kernel_ms = ms;
    return 0;
}

extern "C" int isdf_frontend_check_batch(isdf_ctx *c, int n, const int32_t *ind, const double *father_roll_pitch, double *child_roll_pitch, uint8_t *ok) {
    int r = frontend_state(c);
    if (r) return r;
    if (n < 0 || (n > 0 && (!ind || !father_roll_pitch || !child_roll_pitch || !ok))) return fail(ISDF_ERR_INVALID, "bad argument");
    if (n == 0) return 0;
    for (int q = 0; q < n; q++)
        if (ind[3 * q] < 0 || ind[3 * q] >= c->grid.X || ind[3 * q + 1] < 0 || ind[3 * q + 1] >= c->grid.Y || ind[3 * q + 2] < 0 || ind[3 * q + 2] >= c->grid.Z)
            return fail(ISDF_ERR_INVALID, "voxel index outside the map");
    if (set_device(c)) return ISDF_ERR_CUDA;
    CU_TRY(c->d_fe_ind.upload(ind, (size_t)3 * n, c->stream));
    CU_TRY(c->d_fe_father.upload(father_roll_pitch, (size_t)2 * n, c->stream));
    CU_TRY(c->d_fe_child.ensure((size_t)2 * n)); CU_TRY(c->d_fe_ok.ensure(n)); CU_TRY(c->d_fe_out.ensure((size_t)4 * n));
    FrontArgs A = front_args(c);
    A.out = c->d_fe_out.p; A.nq = n; A.q_ind = c->d_fe_ind.p; A.q_father = c->d_fe_father.p; A.q_child = c->d_fe_child.p; A.q_ok = c->d_fe_ok.p;
    const size_t smem = sizeof(uint32_t) * 4 * (size_t)A.ks * A.ks * A.ks;
    CU_TRY(cudaFuncSetAttribute(k_frontend_check, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_frontend_check<<<(unsigned)((n + 255) / 256), 256, smem, c->stream>>>(A);
    c->stats.kernel_launches++;
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(child_roll_pitch, c->d_fe_child.p, sizeof(double) * 2 * n, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(cudaMemcpyAsync(ok, c->d_fe_ok.p, n, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(cudaStreamSynchronize(c->stream));
    return 0;
}

// ---- swept volume -------------------------------------------------------------------------------------------
extern "C" int isdf_set_points(isdf_ctx *c, const double *pts, int P) {
    if (!c || P < 0 || (P > 0 && !pts)) return fail(ISDF_ERR_INVALID, "bad argument");
    if (set_device(c)) return ISDF_ERR_CUDA;
    c->sv.B = 0;   // a single point set replaces any per-problem sets
    CU_TRY(c->sv.set_points(pts, P, c->stream));
    return 0;
}

extern "C" int isdf_set_points_batch(isdf_ctx *c, int B, const int32_t *offsets, const double *pts) {
    if (!c || B < 0 || (B > 0 && !offsets)) return fail(ISDF_ERR_INVALID, "bad argument");
    if (set_device(c)) return ISDF_ERR_CUDA;
    if (B == 0) { c->sv.B = 0; return 0; }
    if (offsets[0] != 0) return fail(ISDF_ERR_INVALID, "offsets[0] must be 0");
    for (int b = 0; b < B; b++) if (offsets[b + 1] < offsets[b]) return fail(ISDF_ERR_INVALID, "offsets must be non-decreasing");
    if (offsets[B] > 0 && !pts) return fail(ISDF_ERR_INVALID, "pts is NULL");
    if (offsets[B] == 0) return fail(ISDF_ERR_INVALID, "no points at all: use B = 0 to switch the batched swept-volume term off");
    CU_TRY(c->sv.set_points_batch(B, offsets, pts, c->stream));
    return 0;
}

static int swept_common(isdf_ctx *c, int N, const double *d_T, const double *d_C, double *d_out, cudaStream_t st,
                        const double *g_t, const double *g_s, const double *g_g) {
    if (c->sv.P <= 0) return fail(ISDF_ERR_STATE, "obstacle points not set (isdf_set_points)");
    if (c->shape.kind == ISDF_SHAPE_MESH && c->shape.mesh.sign_mode == MESH_SIGN_WINDING)
        return fail(ISDF_ERR_UNSUPPORTED, "the swept-volume search prunes with distance brackets that need a true distance function: winding-sign meshes "
                                          "(open meshes / soups, ISDF_MESH_SIGN_WINDING) are supported by the discrete path and isdf_shape_query only");
    int launches = 0;
    cudaError_t e = c->sv.launch(c->dcfg, c->shape, N, d_T, d_C, d_out, c->rank, c->world, st, g_t, g_s, g_g, &launches);
    c->stats.kernel_launches += launches;
    c->stats.evals_swept++;
    if (e != cudaSuccess) return fail(e == cudaErrorInvalidValue ? ISDF_ERR_INVALID : ISDF_ERR_CUDA, std::string("swept: ") + cudaGetErrorString(e));
    if (c->peer_fused && c->peer.world > 1 && c->world > 1) {   // an unsharded call (isdf_set_shard(ctx, 0, 1)) stays local
        if (c->peer.world != c->world || c->peer.rank != c->rank) return fail(ISDF_ERR_STATE, "peer group does not match isdf_set_shard");
        if (19 * N + 1 > c->peer.cap) return fail(ISDF_ERR_INVALID, "peer exchange buffer too small for this N (isdf_peer_export max_doubles)");
        PeerArgs P = c->peer;
        P.epoch = c->peer.epoch + 1;
        k_peer_allreduce<<<1, 512, 0, st>>>(P, d_out, 19 * N + 1);
        c->stats.kernel_launches++;
        CU_TRY(cudaGetLastError());
        c->peer.epoch = P.epoch;   // committed only once the exchange is enqueued: a local failure must not leave this rank one epoch ahead
    }
    return 0;
}

extern "C" int isdf_eval_swept_device(isdf_ctx *c, int N, const double *d_T, const double *d_coeffs, double *d_out, void *cuda_stream) {
    int r = check_eval_state(c, N, false);
    if (r) return r;
    if (!c->have_shape) return fail(ISDF_ERR_STATE, "shape not set");
    if (!d_T || !d_coeffs || !d_out) return fail(ISDF_ERR_INVALID, "NULL device pointer");
    if (set_device(c)) return ISDF_ERR_CUDA;
    return swept_common(c, N, d_T, d_coeffs, d_out, (cudaStream_t)cuda_stream, nullptr, nullptr, nullptr);
}

static int eval_swept_host(isdf_ctx *c, int N, const double *T, const double *coeffs, const double *g_t, const double *g_s,
                           const double *g_g, double *cost, double *gradC, double *gradT) {
    int r = check_eval_state(c, N, false);
    if (r) { poison(cost); return r; }
    if (!c->have_shape) { poison(cost); return fail(ISDF_ERR_STATE, "shape not set"); }
    if (!T || !coeffs || !cost || !gradC || !gradT) { poison(cost); return fail(ISDF_ERR_INVALID, "NULL argument"); }
    auto body = [&]() -> int {
        if (set_device(c)) return ISDF_ERR_CUDA;
        const size_t nin = (size_t)19 * N, nout = (size_t)19 * N + 1;
        if (ensure_stage(c, nin + nout + 1)) return ISDF_ERR_CUDA;
        CU_TRY(c->d_C.ensure(nin)); CU_TRY(c->d_out.ensure(nout + 1));
        std::memcpy(c->h_stage, coeffs, sizeof(double) * 18 * N);
        std::memcpy(c->h_stage + 18 * (size_t)N, T, sizeof(double) * N);
        CU_TRY(cudaMemcpyAsync(c->d_C.p, c->h_stage, sizeof(double) * nin, cudaMemcpyHostToDevice, c->stream));
        ScopedDevBuf<double> dgt, dgs, dgg;
        if (g_t) {
            CU_TRY(dgt.upload(g_t, c->sv.P, c->stream)); CU_TRY(dgs.upload(g_s, c->sv.P, c->stream));
            CU_TRY(dgg.upload(g_g, (size_t)3 * c->sv.P, c->stream));
        }
        CU_TRY(cudaEventRecord(c->ev0, c->stream));
        c->sv.count_out = c->d_out.p + nout;
        int rr = swept_common(c, N, c->d_C.p + 18 * (size_t)N, c->d_C.p, c->d_out.p, c->stream, dgt.p, dgs.p, dgg.p);
        c->sv.count_out = nullptr;
        if (rr) return rr;
        CU_TRY(cudaEventRecord(c->ev1, c->stream));
        double *h_out = c->h_stage + nin;
        CU_TRY(cudaMemcpyAsync(h_out, c->d_out.p, sizeof(double) * (nout + 1), cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(cudaStreamSynchronize(c->stream));
        unsigned long long nsdf = 0;
        std::memcpy(&nsdf, h_out + nout, sizeof(nsdf));
        if (c->peer_fused && c->peer.world > 1 && c->world > 1 && isdf_peer_status(c) != ISDF_OK) return ISDF_ERR_CUDA;   // exchange timed out: the vector is NaN
        float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1);
        c->stats.last_kernel_ms = ms; c->stats.last_sdf_evals = (int64_t)nsdf;
        *cost += h_out[0];                                   // accumulate like hpp:640-645
        for (size_t k = 0; k < (size_t)18 * N; k++) gradC[k] += h_out[1 + k];
        for (int k = 0; k < N; k++) gradT[k] += h_out[1 + 18 * N + k];
        return 0;
    };
    r = body();
    if (r) poison(cost);
    return r;
}

extern "C" int isdf_eval_swept(isdf_ctx *c, int N, const double *T, const double *coeffs, double *cost, double *gradC, double *gradT) {
    return eval_swept_host(c, N, T, coeffs, nullptr, nullptr, nullptr, cost, gradC, gradT);
}

extern "C" int isdf_eval_swept_given(isdf_ctx *c, int N, const double *T, const double *coeffs, const double *tstar, const double *sdf,
                          const double *grel, double *cost, double *gradC, double *gradT) {
    if (!tstar || !sdf || !grel) { poison(cost); return fail(ISDF_ERR_INVALID, "NULL argument"); }
    return eval_swept_host(c, N, T, coeffs, tstar, sdf, grel, cost, gradC, gradT);
}

extern "C" int isdf_get_swept_results(isdf_ctx *c, double *tstar, double *sdf, double *grel) {
    if (!c) return fail(ISDF_ERR_INVALID, "ctx is NULL");
    if (c->sv.P <= 0) return fail(ISDF_ERR_STATE, "obstacle points not set");
    if (set_device(c)) return ISDF_ERR_CUDA;
    const size_t P = c->sv.P;
    if (tstar) CU_TRY(cudaMemcpy(tstar, c->sv.d_tstar.p, sizeof(double) * P, cudaMemcpyDeviceToHost));
    if (sdf) CU_TRY(cudaMemcpy(sdf, c->sv.d_sdf.p, sizeof(double) * P, cudaMemcpyDeviceToHost));
    if (grel) CU_TRY(cudaMemcpy(grel, c->sv.d_grel.p, sizeof(double) * 3 * P, cudaMemcpyDeviceToHost));
    return 0;
}


// ---- whole-body collision check (isdf_check.cuh) ------------------------------------------------------------------
static void poison_reports(isdf_clearance_report *r, int B) {
    if (!r || B < 1) return;
    const double nan = std::numeric_limits<double>::quiet_NaN();
    for (int b = 0; b < B; b++) {
        isdf_clearance_report &x = r[b];
        x.min_clearance = x.t_min = x.t_hit = nan;
        for (int a = 0; a < 3; a++) x.p_min[a] = x.p_hit[a] = nan;
        x.collides = 1; x.piece_min = x.sample_min = x.piece_hit = x.sample_hit = -1; x.reserved_ = 0;
    }
}

static int check_args(isdf_ctx *c, int B, int N0, int M, double margin, double horizon) {
    if (B < 1 || N0 < 1) return fail(ISDF_ERR_INVALID, "B and N0 must be >= 1");
    if (M < 1 || M > CHECK_MAX_SAMPLES_PER_PIECE) return fail(ISDF_ERR_INVALID, "samples_per_piece must be in [1, 4096]");
    if ((long long)B * N0 > 0x7fffffffll || (long long)B * N0 * (M + 1) > 0x7fffffffll) return fail(ISDF_ERR_INVALID, "B * N0 * (samples_per_piece + 1) must fit in 31 bits");
    if (!std::isfinite(horizon) || !(horizon > 0.0)) return fail(ISDF_ERR_INVALID, "horizon must be finite and > 0");
    if (!std::isfinite(margin) || margin > horizon) return fail(ISDF_ERR_INVALID, "margin must be finite and <= horizon");
    if (!c) return fail(ISDF_ERR_INVALID, "ctx is NULL");
    if (!c->have_map) return fail(ISDF_ERR_STATE, "map not set");
    if (!c->have_shape) return fail(ISDF_ERR_STATE, "shape not set");
    return 0;
}

// both entry points: per-sample kernel + per-trajectory finisher on st (asynchronous)
static int check_launch_ctx(isdf_ctx *c, int B, int N0, const double *d_T, const double *d_C, int M, double margin, double horizon,
                            isdf_clearance_report *d_rep, double *d_clear, cudaStream_t st) {
    const int N = B * N0;
    const size_t S = (size_t)N * (M + 1);
    if (c->d_ck_cursor.n < 1) {
        CU_TRY(c->d_ck_cursor.ensure(1));
        CU_TRY(cudaMemsetAsync(c->d_ck_cursor.p, 0, sizeof(int), st));
    }
    CU_TRY(c->d_ck_arg.ensure(S));
    if (!d_clear) { CU_TRY(c->d_ck_clear.ensure(S)); d_clear = c->d_ck_clear.p; }
    CU_TRY(c->d_ck_counters.ensure(CHECK_NCOUNTERS));
    CU_TRY(cudaMemsetAsync(c->d_ck_counters.p, 0, sizeof(unsigned long long) * CHECK_NCOUNTERS, st));
    CheckArgs A;
    A.cfg = c->dcfg; A.grid = c->grid; A.shape = c->shape;
    A.N = N; A.N0 = N0; A.M = M; A.T = d_T; A.C = d_C; A.margin = margin; A.horizon = horizon;
    A.clear = d_clear; A.arg = c->d_ck_arg.p; A.cursor = c->d_ck_cursor.p; A.counters = c->d_ck_counters.p; A.reports = d_rep;
    A.cycles = nullptr;
    if (c->dbg_on) { CU_TRY(c->d_ck_cycles.ensure(S)); A.cycles = c->d_ck_cycles.p; }
    const int mode = c->shape.kind != ISDF_SHAPE_MESH ? CHECK_ANALYTIC : (c->shape.mesh.sign_mode == MESH_SIGN_WINDING ? CHECK_MESH_WINDING : CHECK_MESH_EXACT);
    CU_TRY(check_launch(A, mode, B, c->sm_count, st));
    c->stats.kernel_launches += 2;
    return 0;
}

extern "C" int isdf_check_collision(isdf_ctx *c, int B, int N0, const double *T, const double *coeffs, int samples_per_piece,
                                    double margin, double horizon, isdf_clearance_report *reports, double *clearance) {
    poison_reports(reports, B);
    int r = check_args(c, B, N0, samples_per_piece, margin, horizon);
    if (r) return r;
    if (!T || !coeffs || !reports) return fail(ISDF_ERR_INVALID, "NULL argument");
    auto body = [&]() -> int {
        if (set_device(c)) return ISDF_ERR_CUDA;
        const int N = B * N0;
        const size_t S = (size_t)N * (samples_per_piece + 1);
        // [coefficients 18N | durations N] in one copy
        CU_TRY(c->d_ck_in.ensure((size_t)19 * N));
        CU_TRY(cudaMemcpyAsync(c->d_ck_in.p, coeffs, sizeof(double) * 18 * N, cudaMemcpyHostToDevice, c->stream));
        CU_TRY(cudaMemcpyAsync(c->d_ck_in.p + 18 * (size_t)N, T, sizeof(double) * N, cudaMemcpyHostToDevice, c->stream));
        CU_TRY(c->d_ck_rep.ensure(B));
        int rr = check_launch_ctx(c, B, N0, c->d_ck_in.p + 18 * (size_t)N, c->d_ck_in.p, samples_per_piece, margin, horizon, c->d_ck_rep.p,
                                  nullptr, c->stream);
        if (rr) return rr;
        std::vector<isdf_clearance_report> tmp(B);
        CU_TRY(cudaMemcpyAsync(tmp.data(), c->d_ck_rep.p, sizeof(isdf_clearance_report) * B, cudaMemcpyDeviceToHost, c->stream));
        if (clearance) CU_TRY(cudaMemcpyAsync(clearance, c->d_ck_clear.p, sizeof(double) * S, cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(cudaStreamSynchronize(c->stream));
        std::memcpy(reports, tmp.data(), sizeof(isdf_clearance_report) * B);
        return 0;
    };
    r = body();
    if (r) poison_reports(reports, B);
    return r;
}

extern "C" int isdf_check_collision_device(isdf_ctx *c, int B, int N0, const double *d_T, const double *d_coeffs, int samples_per_piece,
                                           double margin, double horizon, isdf_clearance_report *d_reports, double *d_clearance,
                                           void *cuda_stream) {
    const cudaStream_t st = (cudaStream_t)cuda_stream;
    auto poison_dev = [&]() {   // the device reports read "not safe" on every failure (best effort: the launch itself may be what failed)
        if (!d_reports || B < 1) return;
        int dev = -1;
        if (c) dev = c->device;
        else {
            cudaPointerAttributes pa;
            if (cudaPointerGetAttributes(&pa, d_reports) != cudaSuccess || pa.type != cudaMemoryTypeDevice) { cudaGetLastError(); return; }
            dev = pa.device;
        }
        if (cudaSetDevice(dev) == cudaSuccess) check_launch_poison(d_reports, B, st);
        cudaGetLastError();
    };
    int r = check_args(c, B, N0, samples_per_piece, margin, horizon);
    if (!r && (!d_T || !d_coeffs || !d_reports)) r = fail(ISDF_ERR_INVALID, "NULL device pointer");
    if (!r && set_device(c)) r = ISDF_ERR_CUDA;
    if (!r) r = check_launch_ctx(c, B, N0, d_T, d_coeffs, samples_per_piece, margin, horizon, d_reports, d_clearance, st);
    if (r) poison_dev();
    return r;
}

// ---- internal diagnostics (not part of include/isdf.h) ------------------------------------------------------------
extern "C" int isdf_dbg_enable(isdf_ctx *c, int on) { if (!c) return -1; c->dbg_on = on != 0; c->sv.dbg_on = on != 0; return 0; }
// scheduling diagnostics: natural_order != 0 -> every launch in natural sample order, nothing split (the state of a context's FIRST
// evaluation); warp_slots > 0 -> build the work items as if the device had that many resident warps (huge values shrink the
// balanced share per warp and force every non-trivial sample to be split, so tests can compare split parts against the oracle on one
// GPU); 0 restores the device's own figure.
extern "C" int isdf_dbg_schedule(isdf_ctx *c, int natural_order, int warp_slots) {
    if (!c) return -1;
    c->no_items = natural_order != 0; c->warp_slots_override = warp_slots > 0 ? warp_slots : 0; c->order_for = -1;
    return 0;
}
// number of work items / split samples of the table built by the last discrete evaluation
extern "C" int isdf_dbg_item_stats(isdf_ctx *c, int *item_count, int *split_parts) {
    if (!c || !item_count || !split_parts || !c->d_item_count.p) return -1;
    if (cudaSetDevice(c->device) != cudaSuccess) return -3;
    cudaStreamSynchronize(c->stream); cudaStreamSynchronize(c->aux_stream);
    int n = 0;
    if (cudaMemcpy(&n, c->d_item_count.p, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return -3;
    std::vector<int> it((size_t)3 * std::max(n, 1));
    if (n > 0 && cudaMemcpy(it.data(), c->d_items.p, sizeof(int) * 3 * n, cudaMemcpyDeviceToHost) != cudaSuccess) return -3;
    int parts = 0;
    for (int k = 0; k < n; k++) if (it[3 * k + 2] >= 0) parts++;
    *item_count = n; *split_parts = parts;
    return 0;
}
// the device flatness map and its adjoint as compiled into the epilogue kernel: vaj n x 9 (vel, acc, jer), grads n x 10
// (quat_grad 4, omg_grad 3, vel_grad 3) -> out n x 16 (quat 4, omg 3, total grads wrt vel, acc, jer)
extern "C" int isdf_dbg_flatness(isdf_ctx *c, int n, const double *vaj, const double *grads, double *out) {
    if (!c || n < 1 || !vaj || !grads || !out) return -1;
    if (cudaSetDevice(c->device) != cudaSuccess) return -3;
    ScopedDevBuf<double> dv, dg, dout;
    cudaError_t e = dv.upload(vaj, (size_t)9 * n, c->stream);
    if (e == cudaSuccess) e = dg.upload(grads, (size_t)10 * n, c->stream);
    if (e == cudaSuccess) e = dout.ensure((size_t)16 * n);
    if (e == cudaSuccess) e = discrete_launch_dbg_flatness(c->dcfg.fp, n, dv.p, dg.p, dout.p, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, dout.p, sizeof(double) * 16 * n, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    return e == cudaSuccess ? 0 : -3;
}
extern "C" int isdf_dbg_swept_stats(isdf_ctx *c, unsigned long long *out, long long n) {
    if (!c || !out || (size_t)n > c->sv.d_dbg.n) return -1;
    cudaStreamSynchronize(c->stream);
    return cudaMemcpy(out, c->sv.d_dbg.p, sizeof(unsigned long long) * n, cudaMemcpyDeviceToHost) == cudaSuccess ? 0 : -3;
}
extern "C" int isdf_dbg_trace_stride(void) { return TRACE_STRIDE; }
extern "C" int isdf_dbg_item_trace(isdf_ctx *c, unsigned long long *out, long long n) {
    if (!c || !out || (size_t)n > c->d_trace.n) return -1;
    if (cudaSetDevice(c->device) != cudaSuccess) return -3;
    return cudaMemcpy(out, c->d_trace.p, sizeof(unsigned long long) * n, cudaMemcpyDeviceToHost) == cudaSuccess ? 0 : -3;
}
extern "C" int isdf_dbg_sample_stats(isdf_ctx *c, unsigned long long *out, long long n) {
    if (!c || !out || (size_t)n > c->d_dbg.n) return -1;
    if (cudaSetDevice(c->device) != cudaSuccess) return -3;
    return cudaMemcpy(out, c->d_dbg.p, sizeof(unsigned long long) * n, cudaMemcpyDeviceToHost) == cudaSuccess ? 0 : -3;
}
// collision check diagnostics: counters {voxels in the body box, SDF values computed, mesh searches} of the last check and, after
// isdf_dbg_enable(ctx, 1), the per-sample clock64 cycles of its warp (n = samples of that check; may be 0)
extern "C" int isdf_dbg_check_stats(isdf_ctx *c, unsigned long long *counters3, unsigned long long *cycles, long long n) {
    if (!c || !counters3 || !c->d_ck_counters.p || (n > 0 && (!cycles || (size_t)n > c->d_ck_cycles.n))) return -1;
    if (cudaSetDevice(c->device) != cudaSuccess) return -3;
    if (cudaStreamSynchronize(c->stream) != cudaSuccess) return -3;
    if (cudaMemcpy(counters3, c->d_ck_counters.p, sizeof(unsigned long long) * CHECK_NCOUNTERS, cudaMemcpyDeviceToHost) != cudaSuccess) return -3;
    if (n > 0 && cudaMemcpy(cycles, c->d_ck_cycles.p, sizeof(unsigned long long) * n, cudaMemcpyDeviceToHost) != cudaSuccess) return -3;
    return 0;
}
