/* isdf.h — C ABI of libisdf_b200.so: B200-native (sm_100a) collision cost/gradient evaluator for the
 * Implicit-SDF-Planner back end. Plain pointers and sizes only; no torch / Eigen / ROS types.
 *
 * Every entry point names the reference interface it replaces (paths relative to /root/reference/src):
 *   hpp   = planner_algorithm/include/planner_algorithm/back_end_optimizer.hpp
 *   swm   = swept_volume/include/swept_volume/sw_manager.hpp
 *   Shape = utils/include/utils/Shape.hpp, utils/src/Shape.cpp
 *   pcs   = map_manager/include/map_manager/PCSmap_manager.h ; grid = map_manager/src/Gridmap3D.cpp
 *   minco = utils/include/utils/minco.hpp ; lmbm = utils/include/lmbm/lmbm.h ; lbfgs = utils/include/utils/lbfgs.hpp
 *
 * Conventions
 *   - All functions return 0 on success, a negative isdf_status on failure; isdf_last_error() gives the message.
 *     On failure every output cost is set to NaN so that either optimiser driver terminates
 *     (the LMBM callback has no error channel, lmbm_call.f:125; L-BFGS aborts on NaN, lbfgs.hpp:148-197).
 *   - Matrices follow Eigen's defaults: `coeffs`/`gradC` are MatrixX3d (6N x 3) COLUMN-major:
 *     element (6*i + k, axis) at [axis*6N + 6*i + k] = t^k coefficient of piece i (hpp:434,460).
 *   - There is no CPU fallback: if no CUDA device / kernel image is usable, isdf_create fails.
 */
#ifndef ISDF_H
#define ISDF_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct isdf_ctx isdf_ctx;

typedef enum isdf_status {
    ISDF_OK = 0,
    ISDF_ERR_INVALID = -1,   /* bad argument */
    ISDF_ERR_STATE = -2,     /* map / shape / points not set */
    ISDF_ERR_CUDA = -3,      /* CUDA runtime or launch failure (message has the CUDA error string) */
    ISDF_ERR_UNSUPPORTED = -4
} isdf_status;

/* Subset of struct Config (utils/include/utils/config.hpp:13-203) that the hot path reads, in the units of
 * plan_manager/config/ *.yaml. Same field order as oracle/oracle_capi.cpp::orc_config. */
typedef struct isdf_config {
    double vehicle_mass, grav_acc, horiz_drag, vert_drag, paras_drag, speed_eps; /* FlatnessMap::reset, flatness.hpp:36-51 */
    double vmax, omgmax, thetamax;                                               /* hpp:678-680 */
    double weight_v, weight_p, weight_omg, weight_theta;                         /* hpp:683-687 */
    double smoothing_eps;        /* smooth_fac, hpp:689 */
    double safety_hor;           /* hpp:691 */
    double occupancy_resolution; /* bd = kernel_size * occupancy_resolution, hpp:692 */
    int32_t kernel_size;
    int32_t integral_intervs;    /* integralRes K, hpp:690: K+1 trapezoid nodes per piece */
    int32_t threads_num;         /* kept for interface parity (config.hpp:16); ignored by the GPU path */
    int32_t flags;               /* isdf_flags */
} isdf_config;

typedef enum isdf_flags {
    ISDF_WITH_DYNAMICS = 1,   /* velocity / body-rate / tilt penalties of addTimeIntPenaltyParallel (hpp:505-534) */
    ISDF_WITH_COLLISION = 2   /* grad_cost_p (hpp:766-824) wired into the sample loop as hpp:619-626 wires its SV sibling */
} isdf_flags;

/* Numeric ids shared with oracle/oracle_shapes.hpp::ShapeKind. params[] layout per kind is documented in
 * implicit-sdf-planner_b200/csrc/isdf_shapes.cuh; isdf_set_shape_named() fills the reference's hard-coded constants. */
typedef enum isdf_shape_kind {
    ISDF_SHAPE_BALL = 0, ISDF_SHAPE_POINT = 1, ISDF_SHAPE_TORUS = 2, ISDF_SHAPE_CAPPED_TORUS = 3,
    ISDF_SHAPE_CAPPED_CONE = 4, ISDF_SHAPE_ROUNDED_CONE = 5, ISDF_SHAPE_WIREFRAME_BOX = 6,
    ISDF_SHAPE_BEND_LINEAR = 7, ISDF_SHAPE_TWIST_BOX = 8, ISDF_SHAPE_BEND_BOX = 9, ISDF_SHAPE_TABLE = 10,
    ISDF_SHAPE_TREFOIL = 11, ISDF_SHAPE_SMOOTH_DIFFERENCE = 12, ISDF_SHAPE_SMOOTH_INTERSECTION = 13,
    ISDF_SHAPE_CSG = 14, ISDF_SHAPE_BOX = 15, ISDF_SHAPE_MESH = 16
} isdf_shape_kind;

/* What isdf_shape_query computes — the four BasicShape virtuals (Shape.hpp:469-472). */
typedef enum isdf_query {
    ISDF_QUERY_SDF = 0,       /* getonlySDF(pos_rel) */
    ISDF_QUERY_GRAD = 1,      /* getonlyGrad1(pos_rel) */
    ISDF_QUERY_SDF_GRAD = 2   /* getSDFwithGrad1(pos_rel, grad) */
} isdf_query;

/* attitude grid of the front end's collision kernels (config yaml: kernel_max_roll / kernel_max_pitch / kernel_ang_res, degrees;
 * front_end_safeh); kernel_size and occupancy_resolution come from isdf_config */
typedef struct isdf_kernel_config {
    double kernel_max_roll, kernel_max_pitch, kernel_ang_res, front_end_safeh;
} isdf_kernel_config;

typedef struct isdf_stats {
    int64_t kernel_launches;   /* kernels of this library launched since isdf_create */
    int64_t evals_discrete;    /* isdf_eval_discrete* calls */
    int64_t evals_swept;       /* isdf_eval_swept* calls */
    int64_t last_pairs;        /* (sample, voxel) pairs that reached the SDF in the last discrete evaluation */
    int64_t last_sdf_evals;    /* SDF evaluations in the last swept-volume evaluation */
    double last_kernel_ms;     /* device time of the last evaluation's kernels (CUDA events on the launch stream) */
} isdf_stats;

/* ---- lifetime -------------------------------------------------------------------------------------------- */
/* values of plan_manager/config/config_CappedCone.yaml; flags = DYNAMICS (the live reference callback; add ISDF_WITH_COLLISION for the discrete grad_cost_p term) */
int isdf_default_config(isdf_config *cfg);
/* replaces TrajOptimizer::setParam (hpp:667-722) + SweptVolumeManager ctor (swm:135-150). device = CUDA ordinal. */
int isdf_create(const isdf_config *cfg, int device, isdf_ctx **out);
int isdf_destroy(isdf_ctx *ctx);
const char *isdf_last_error(void);
int isdf_get_stats(isdf_ctx *ctx, isdf_stats *out);
/* Shard the evaluation: this context evaluates samples / obstacle points with index % world == rank and returns
 * partial sums (caller all-reduces 19N+1 doubles). Default rank 0 / world 1. */
int isdf_set_shard(isdf_ctx *ctx, int rank, int world);

/* ---- robot shape: replaces SweptVolumeManager::initShape (swm:255-275) and the Generalshape ctor (Shape.cpp:27-103) */
/* rotate_rowmajor / trans = Generalshape::Rotate / trans from poly_params (Shape.hpp:776-780); NULL = identity / zero */
int isdf_set_shape_analytic(isdf_ctx *ctx, int kind, const double *params, int nparams,
                            const double *rotate_rowmajor, const double *trans);
/* factory keyed by the OBJ basename like shapeConstructors (swm:74-123): "Torus", "CSG", ...; plus "Ball", "Point" */
int isdf_set_shape_named(isdf_ctx *ctx, const char *name, const double *rotate_rowmajor, const double *trans);
/* triangle mesh (V: nV x 3 row-major, F: nF x 3 row-major); poly_params = {tx,ty,tz, roll,pitch,yaw in degrees} pre-transform as
 * Shape.cpp:38-50, NULL = none. SDF = s * dist (Shape.cpp:105-151); the distance is exact, the sign factor s depends on the mode:
 *   ISDF_MESH_SIGN_AUTO    closed, consistently oriented mesh -> ISDF_MESH_SIGN_EXACT, anything else (open mesh, triangle soup) ->
 *                          ISDF_MESH_SIGN_WINDING (as igl::fast_winding_number accepts any soup);
 *   ISDF_MESH_SIGN_EXACT   s = ±1, the exact inside/outside classification (angle-weighted pseudonormals); ISDF_ERR_UNSUPPORTED if the mesh
 *                          is not closed. This is what the reference's s = 1 - 2 w rounds to; DESIGN.md "mesh sign" reports the deviation;
 *   ISDF_MESH_SIGN_WINDING s = 1 - 2 w with w the generalised winding number, NOT thresholded — the reference's form (Shape.cpp:110-111).
 *                          w is evaluated hierarchically in FP64 (first-order expansion, exact near field), i.e. closer to the true winding
 *                          number than the reference's FP32 tree, not bit-equal to it. Discrete path, isdf_shape_query and the front end
 *                          support this mode; the swept-volume entry points return ISDF_ERR_UNSUPPORTED for it.
 * isdf_set_shape_mesh = isdf_set_shape_mesh_ex(..., ISDF_MESH_SIGN_AUTO). */
typedef enum isdf_mesh_sign { ISDF_MESH_SIGN_AUTO = 0, ISDF_MESH_SIGN_EXACT = 1, ISDF_MESH_SIGN_WINDING = 2 } isdf_mesh_sign;
int isdf_set_shape_mesh(isdf_ctx *ctx, const double *V, int nV, const int32_t *F, int nF, const double *poly_params);
int isdf_set_shape_mesh_ex(isdf_ctx *ctx, const double *V, int nV, const int32_t *F, int nF, const double *poly_params, int sign_mode);
/* the BasicShape virtual surface (Shape.hpp:469-472) for n body-frame points (n x 3 row-major); sdf/grad may be NULL */
int isdf_shape_query(isdf_ctx *ctx, const double *p_rel, int n, double *sdf, double *grad, int what);

/* ---- occupancy map: replaces GridMap3D::createGridMap + the fill in PCSmap_manager.cpp:148-181 ------------ */
/* occ: X*Y*Z bytes, address ix*Y*Z + iy*Z + iz (GridMap3D.h:194-195), non-zero = occupied.
 * boundary_xyzmax is taken as bmin + size*res. */
int isdf_set_map_u8(isdf_ctx *ctx, const uint8_t *occ, int X, int Y, int Z, const double *bmin, double res);
/* the reference's own storage: one double per voxel (GridMap3D.h:215) */
int isdf_set_map_f64(isdf_ctx *ctx, const double *grid_map, int X, int Y, int Z, const double *bmin, double res);
/* PCSmapManager::getPointsInAABB (pcs:148-170) on the device map; writes up to cap centres (cap x 3), returns count in *n */
int isdf_points_in_aabb(isdf_ctx *ctx, const double *centre, double half_extent, double *out_points, int cap, int *n);

/* The obstacle list of PlannerManager::generateTraj (plan_manager.cpp:232-254): for every waypoint in order, the occupied voxels of
 * box(wp + offset, half) that are not in box(previous wp, half) (PCSmapManager::getPointsInAABBOutOfLastOne, pcs:182-216),
 * de-duplicated by voxel. waypoints: nQ x 3 row-major. Writes up to cap centres in (first-including waypoint, voxel address)
 * order and the total in *n. If set_as_points != 0 the list also becomes the swept-volume point set (== isdf_set_points). */
int isdf_gather_obstacle_points(isdf_ctx *ctx, const double *waypoints, int nQ, double half_extent, const double *offset,
                                double *out_points, int cap, int *n, int set_as_points);

/* ---- discrete collision term: addTimeIntPenaltyParallel (hpp:432-554) with grad_cost_p (hpp:766-824) wired in */
/* ACCUMULATES into *cost, gradC (6N x 3 col-major), gradT (N) exactly like the reference's reference arguments. */
int isdf_eval_discrete(isdf_ctx *ctx, int N, const double *T, const double *coeffs,
                       double *cost, double *gradC, double *gradT);
/* device-resident variant: d_T (N), d_coeffs (18N) and d_out (19N+1 = [cost | gradC 18N | gradT N], OVERWRITTEN)
 * are device pointers on ctx's device; cuda_stream is a cudaStream_t (NULL = default stream). Asynchronous. */
int isdf_eval_discrete_device(isdf_ctx *ctx, int N, const double *d_T, const double *d_coeffs, double *d_out,
                              void *cuda_stream);

/* per-piece cost terms of the last discrete evaluation (n <= N doubles). With B independent trajectories concatenated into one
 * call (pieces b*N0 .. b*N0+N0-1 belong to trajectory b — the discrete term couples nothing across pieces, so a batch of
 * random restarts is simply a longer coefficient block) the cost of trajectory b is the sum of its N0 entries. */
int isdf_get_piece_costs(isdf_ctx *ctx, double *piece_cost, int n);

/* ---- batched optimiser callback on the device (SURVEY §8f row 1: MINCO on both sides of the hot loop) -------------------- */
/* B independent problems (random restarts, BASELINE configs[4]) in one call. Restates TrajOptimizer::costFunctionLmbm
 * (back_end_optimizer.hpp:358-430) with the time-integral term as the only penalty (use the per-problem host adapter
 * host/isdf_cost_callback.hpp when the swept-volume term is wanted: obstacle point sets are per trajectory):
 *   x_b = [tau (N0) | xi (3(N0-1), waypoint-major)] -> forwardT (hpp:214-241) -> MINCO_S3NU::setParameters (minco.hpp:433-513,
 *   banded LU :99-135) -> getEnergy + partials (:530-582) -> addTimeIntPenaltyParallel over the concatenated B*N0 pieces ->
 *   propogateGrad (:584-654) -> + rho*sum(T) -> backwardGradT / backwardGradP (hpp:283-330).
 * head / tail: 3x3 column-major (columns p, v, a), one pair shared by the batch (per_problem_bc = 0) or B pairs (= 1).
 * x: B x (4*N0-3) row-major; cost: B; grad: B x (4*N0-3). On failure every cost[b] is NaN. N0 <= 290.
 * Multi-GPU: shard by problem (each rank calls this with its own problems and isdf_set_shard(ctx, 0, 1)); no collective.
 * With per-problem obstacle point sets registered for the same B (isdf_set_points_batch) the callback is the LIVE composition of the
 * reference — swept-volume term (addSaftyPenaOnSweptVolumeParallel, hpp:386-391) then time-integral term (hpp:399-405) — for every problem,
 * each stage one launch over the whole batch (grid.y = problem). */
/* problem b owns the points [offsets[b], offsets[b+1]) of pts (offsets: B+1 ints, offsets[0] = 0; what plan_manager.cpp:232-254 builds per plan);
 * t* of every point starts at 0 and persists across evaluations like lastTstar. B = 0 switches the batched swept-volume term off again. */
int isdf_set_points_batch(isdf_ctx *ctx, int B, const int32_t *offsets, const double *pts);
int isdf_callback_batch(isdf_ctx *ctx, int B, int N0, const double *head, const double *tail, int per_problem_bc, double rho,
                        const double *x, double *cost, double *grad);
/* device-resident variant (all pointers on ctx's device, asynchronous on cuda_stream) */
int isdf_callback_batch_device(isdf_ctx *ctx, int B, int N0, const double *d_head, const double *d_tail, int per_problem_bc,
                               double rho, const double *d_x, double *d_cost, double *d_grad, void *cuda_stream);
/* the trajectories of the last batched callback: durations (B*N0), coefficient block (6*B*N0 x 3 column-major, piece b*N0+i),
 * jerk energies (B); any may be NULL */
int isdf_get_batch_trajectories(isdf_ctx *ctx, double *T, double *coeffs, double *energy);

/* ---- device-resident lock-step L-BFGS over the batched callback (SURVEY §8f row 2) ------------------------------------------------
 * B independent instances of the reference's patched LBFGS-Lite fork (utils/include/utils/lbfgs.hpp:480-830: Lewis-Overton bracketing that
 * returns on Armijo :290-430, cautious update + two-loop recursion :742-786, the fork's direction reset :788-811, stop tests :656-690; same
 * return codes :148-197) advanced together: every round is ONE isdf_callback_batch_device evaluation of all instances' requested points plus
 * one bookkeeping kernel; iterates and histories never leave the device. Each instance's iterates, counts and return code are bit-identical
 * to the sequential driver host/isdf_lbfgs.hpp run on the same callback. The reference's own driver is single-instance (and its live LMBM
 * shim non-re-entrant, lmbm/lmbm.cpp:4-6). */
typedef struct isdf_lbfgs_params {     /* lbfgs_parameter_t (lbfgs.hpp:40-142); with_tole_ls / cast_x_range off as in the shipped configs */
    int32_t mem_size, past, max_iterations, max_linesearch;
    int32_t max_rounds;                /* 0 = until every instance has stopped; otherwise a cap on batched evaluations */
    int32_t reserved_;
    double g_epsilon, delta, min_step, max_step, f_dec_coeff, cautious_factor, machine_prec;
} isdf_lbfgs_params;
int isdf_lbfgs_default_params(isdf_lbfgs_params *p);   /* config_CappedCone.yaml:99-102: mem 16, past 10, min_step 1e-32, g_epsilon 0, delta 1e-6 */
/* x: B x (4*N0-3) in/out; f: B; ret / iterations / evaluations: B (any may be NULL); rounds: batched evaluations used (may be NULL).
 * head / tail / rho / per_problem_bc as isdf_callback_batch. */
int isdf_lbfgs_batch(isdf_ctx *ctx, int B, int N0, const double *head, const double *tail, int per_problem_bc, double rho,
                     const isdf_lbfgs_params *params, double *x, double *f, int32_t *ret, int32_t *iterations, int32_t *evaluations, int32_t *rounds);
/* device-resident variant (all pointers on ctx's device; returns when every instance has stopped — one 4-byte read per round) */
int isdf_lbfgs_batch_device(isdf_ctx *ctx, int B, int N0, const double *d_head, const double *d_tail, int per_problem_bc, double rho,
                            const isdf_lbfgs_params *params, double *d_x, double *d_f, int32_t *d_ret, int32_t *d_iterations, int32_t *d_evaluations,
                            int32_t *rounds, void *cuda_stream);

/* ---- whole-body collision check: the verdict PlannerManager::generateTraj asks for after every optimisation
 * (plan_manager.cpp:306, :383) and SweptVolumeManager::isTrajCollide (swm:759-767) leaves as a stub that always returns false.
 * The cost terms above are soft (hinge penalties, zero beyond safety_hor, smoothed over mu) and an optimiser may stop with obstacles
 * inside the robot; this is the hard answer.
 *
 * Check samples: piece i is checked at M + 1 local times j * (T_i * (1/M)), j = 0..M (M = samples_per_piece, the rule of the discrete
 * path's integral nodes; M = integral_intervs is the natural choice). Pose as the discrete path: position from the piece polynomial,
 * attitude R from the flatness quaternion.
 * Clearance of a sample, H = horizon > 0, half_bd = kernel_size * occupancy_resolution / 2 (the body box of hpp:800):
 *     c = min( H, min over occupied voxels v with |R^T (p_v - x)|_inf <= half_bd + H of sdf_robot(R^T (p_v - x)) )
 * p_v = voxel centre (getGridCubeCenter). Voxels outside the map are free (no projInMap clamping: a geometric query, not a replay of
 * the gather). sdf_robot = the SDF of the current shape: any analytic kind, a mesh with ISDF_MESH_SIGN_EXACT, or a mesh with
 * ISDF_MESH_SIGN_WINDING (s = 1 - 2 w). For a 1-Lipschitz SDF (exact-sign mesh, Ball, Box) of a robot inside its kernel cube the box
 * changes nothing: c = min(H, minimum over ALL occupied voxel centres).
 * Verdict: the trajectory COLLIDES when some check sample has c < margin (margin <= H; a negative margin is a penetration tolerance).
 * For a 1-Lipschitz SDF, margin = res * sqrt(3) / 2 means "no occupied voxel cube touches the robot at any check sample".
 * A sample whose pose is not finite has c = NaN and counts as a hit. Nothing between check samples is certified.
 * First hit = the smallest (piece, j) with c < margin. Argmin voxel: among equal SDF values the smallest linear address
 * ix*Y*Z + iy*Z + iz; the reported minimum is the first sample in (piece, j) order that attains it.
 * Results are independent of scheduling: bit-identical run to run, alone or inside a batch, host or device entry point. */
typedef struct isdf_clearance_report {      /* one per trajectory */
    double min_clearance, t_min;            /* smallest c over all check samples, and its trajectory time */
    double p_min[3];                        /* the obstacle voxel centre that attains it (NaN if c == horizon) */
    double t_hit, p_hit[3];                 /* first sample with c < margin and its argmin voxel (t_hit = -1, p_hit NaN if none) */
    int32_t collides, piece_min, sample_min, piece_hit, sample_hit, reserved_;   /* pieces local to the trajectory; -1 = none */
} isdf_clearance_report;
/* B trajectories of N0 pieces concatenated like isdf_eval_discrete's restart batches (T: B*N0, coeffs 6*B*N0 x 3 col-major;
 * isdf_get_batch_trajectories returns exactly this). 1 <= samples_per_piece <= 4096. reports: B. clearance (may be NULL):
 * B*N0*(M+1) doubles, the per-sample c, piece-major. Needs the map and the shape; ignores isdf_set_shard (always the whole
 * trajectory) and the ISDF_WITH_COLLISION flag. Touches no state of the cost paths (work-item schedule, lastTstar).
 * ISDF_ERR_INVALID: bad B / N0 / M, horizon not finite and > 0, margin not finite or > horizon, NULL reports / T / coeffs.
 * ISDF_ERR_STATE: map or shape not set. On ANY failure every report reads min_clearance = NaN, collides = 1 (when reports is
 * given): a caller that ignores the status never reads "safe". */
int isdf_check_collision(isdf_ctx *ctx, int B, int N0, const double *T, const double *coeffs, int samples_per_piece,
                         double margin, double horizon, isdf_clearance_report *reports, double *clearance);
/* device-resident variant: every pointer on ctx's device, asynchronous on cuda_stream (a cudaStream_t, NULL = default stream) */
int isdf_check_collision_device(isdf_ctx *ctx, int B, int N0, const double *d_T, const double *d_coeffs, int samples_per_piece,
                                double margin, double horizon, isdf_clearance_report *d_reports, double *d_clearance,
                                void *cuda_stream);

/* ---- multi-GPU reduction through NVLink / NVSwitch peer memory (optional; ncclAllReduce over the same 19N+1 doubles is the
 * library alternative). One process per GPU. Sequence on every rank:
 *   isdf_set_shard(ctx, rank, world); isdf_peer_export(ctx, world, max_doubles, h) -> all-gather the 64-byte handles ->
 *   isdf_peer_connect(ctx, world, rank, handles, fuse) -> barrier -> evaluations ... -> barrier -> isdf_peer_disconnect(ctx).
 * With fuse != 0 every sharded isdf_eval_discrete* / isdf_eval_swept* call ends with the exchange inside the evaluation's last
 * kernel (discrete: the same CTA that finishes the rank's vector pushes it to the peers), so `d_out` / the accumulated host
 * results are the ALL-RANK sums, added in rank order: bit-identical on every rank. All ranks must issue the same sequence of
 * evaluations. A rank that never arrives makes the others time out (~2 s) and isdf_peer_status() report it; nothing hangs. */
int isdf_peer_export(isdf_ctx *ctx, int world, int max_doubles, unsigned char *handle64);
int isdf_peer_connect(isdf_ctx *ctx, int world, int rank, const unsigned char *handles /* world x 64 */, int fuse_into_eval);
int isdf_peer_allreduce_device(isdf_ctx *ctx, double *d_vec, int n, void *cuda_stream);   /* stand-alone, in place */
int isdf_peer_status(isdf_ctx *ctx);
int isdf_peer_disconnect(isdf_ctx *ctx);

/* ---- front end: attitude-kernel collision checks (SURVEY §8f row 4) -------------------------------------------------------- */
/* BasicShape::initShape's kernel branch (Shape.hpp:405-461): one kernel_size^3 occupancy kernel of the robot per (roll, pitch)
 * attitude, voxel set when getonlySDF(pos, Rx(roll)*Ry(pitch)) <= max(front_end_safeh, occupancy_resolution/2). Returns the
 * attitude grid size (sw_manager.hpp:135-136); at most 128 attitudes, kernel_size odd and <= 29. Call again after changing
 * the shape. */
int isdf_frontend_build_kernels(isdf_ctx *ctx, const isdf_kernel_config *kc, int *xkernel_size, int *ykernel_size);
/* the kernels as booleans, [attitude i*ykernel_size+j][a*ks*ks + b*ks + c] (Shape.hpp:453), n = xk*yk*ks^3 bytes */
int isdf_frontend_get_kernels(isdf_ctx *ctx, uint8_t *out, int n);
/* kernelConv<true> (sw_manager.hpp:821-846) for EVERY voxel and EVERY attitude: masks[4*voxel .. 4*voxel+3] is a 128-bit set,
 * bit i*ykernel_size+j = 1 when attitude (i,j) is collision-free with the robot centred on that voxel (voxel = ix*Y*Z+iy*Z+iz).
 * Cells outside the map count as free, like the reference's inflated map kernel (PCSmap_manager.h:46-78). */
int isdf_frontend_feasibility(isdf_ctx *ctx, uint32_t *masks /* X*Y*Z*4, host */);
int isdf_frontend_feasibility_device(isdf_ctx *ctx, uint32_t *d_masks, void *cuda_stream);
/* checkKernelValue (sw_manager.hpp:914-941) for n queries: voxel index (n x 3), father (roll, pitch) in degrees (n x 2) ->
 * child (roll, pitch) = the first collision-free attitude in visit_kernels_by_distance's order (level pose, then BFS from the
 * father's attitude, sw_manager.hpp:852-913); ok[q] = 0 when no attitude fits (child = father). */
int isdf_frontend_check_batch(isdf_ctx *ctx, int n, const int32_t *ind, const double *father_roll_pitch,
                              double *child_roll_pitch, uint8_t *ok);

/* ---- swept-volume term: addSaftyPenaOnSweptVolumeParallel (hpp:557-649) + getSDFofSweptVolume (swm:710-747) --- */
/* parallel_points (plan_manager.cpp:246-254): P x 3 row-major world-frame voxel centres; resets lastTstar to 0 */
int isdf_set_points(isdf_ctx *ctx, const double *pts, int P);
int isdf_eval_swept(isdf_ctx *ctx, int N, const double *T, const double *coeffs,
                    double *cost, double *gradC, double *gradT);
int isdf_eval_swept_device(isdf_ctx *ctx, int N, const double *d_T, const double *d_coeffs, double *d_out,
                           void *cuda_stream);
/* per-point results of the last swept evaluation: t* (lastTstar, hpp:59), SV-SDF value, g_rel (3 per point); any may be NULL */
int isdf_get_swept_results(isdf_ctx *ctx, double *tstar, double *sdf, double *grel);
/* tier-T1 tail parity: evaluate the chain-rule tail at caller-supplied t*, sdf*, g_rel instead of searching */
int isdf_eval_swept_given(isdf_ctx *ctx, int N, const double *T, const double *coeffs, const double *tstar,
                          const double *sdf, const double *grel, double *cost, double *gradC, double *gradT);

#ifdef __cplusplus
}
#endif
#endif /* ISDF_H */
