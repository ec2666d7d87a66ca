// ORACLE of the whole-body collision check (include/isdf.h, isdf_check_collision) — TEST INFRASTRUCTURE ONLY.
// States the definition directly, on the oracle's own pose pipeline (orc::Traj coefficients + beta basis, orc::Flat quaternion,
// quat_to_R: the pieces pinned to the reference-compiled code by tests/test_reference_pins.py) and its orc::Shape SDFs:
//   for every check sample, every OCCUPIED voxel of the world AABB of the body box inflated by H (x, y, z ascending), the box test
//   |R^T (p_v - x)|_inf <= half_bd + H, the SDF capped at H and the tie rule (first voxel in address order attaining the minimum).
// No bit scan, no culls, no pruning: independent of the device's enumeration. Built by tests/collision_oracle.py with the oracle's flags.
#include "../oracle/oracle_planner.hpp"
#include <cmath>
#include <cstdint>
#include <algorithm>
#include <limits>
#include <vector>

using namespace orc;

extern "C" {

// Same layout as isdf_clearance_report (include/isdf.h; the tests assert it).
struct orc_clearance_report {
    double min_clearance, t_min, p_min[3], t_hit, p_hit[3];
    int32_t collides, piece_min, sample_min, piece_hit, sample_hit, reserved_;
};

// shape: an oracle_lib.Shape handle (its orc::Shape is the handle's first member). occ: X*Y*Z bytes, z fastest.
// T: B*N0, C: 6*B*N0 x 3 column-major. clearance (may be NULL): B*N0*(M+1). unrestricted != 0 drops the box test and scans every
// occupied voxel of the map (the "box changes nothing" property of 1-Lipschitz SDFs).
// Per-sample parameters: bd = kernel_size * occupancy_resolution, flat = {mass, grav, dh, dv, cp, veps}.
int orc_check_collision(const double *flat, double bd, const uint8_t *occ, int X, int Y, int Z, const double *bmin, double res,
                        const void *shape, int B, int N0, const double *T, const double *C, int M, double margin, double H,
                        orc_clearance_report *reports, double *clearance, int unrestricted) {
    const Shape &S_ = *static_cast<const Shape *>(shape);
    Flat F; F.reset(flat[0], flat[1], flat[2], flat[3], flat[4], flat[5]);
    const int N = B * N0;
    Traj tr; tr.N = N; tr.T = T; tr.C = C;
    const double hb = bd / 2 + H;
    const double nan = std::numeric_limits<double>::quiet_NaN();
    const V3 bm(bmin[0], bmin[1], bmin[2]);
    auto centre = [&](long long a, double *p) {
        if (a < 0) { p[0] = p[1] = p[2] = nan; return; }
        const long long yz = (long long)Y * Z;
        const int ix = (int)(a / yz), iy = (int)((a - ix * yz) / Z), iz = (int)(a - ix * yz - (long long)iy * Z);
        const V3 c = V3((ix + 0.5) * res, (iy + 0.5) * res, (iz + 0.5) * res) + bm;   // getGridCubeCenter
        p[0] = c.x; p[1] = c.y; p[2] = c.z;
    };
    // per-sample clearance and argmin voxel: samples are independent (OpenMP over samples changes nothing but the wall time)
    const long long S = (long long)N * (M + 1);
    std::vector<double> val(S);
    std::vector<long long> arg(S);
#pragma omp parallel for schedule(dynamic, 16)
    for (long long s = 0; s < S; s++) {
        const int ig = (int)(s / (M + 1)), j = (int)(s % (M + 1));
        const double step = T[ig] * (1.0 / M);
        double b0[6], b1[6], b2[6], b3[6], b4[6];
        beta_basis(j * step, b0, b1, b2, b3, b4);
        V3 pos, vel, acc, jer;
        for (int ax = 0; ax < 3; ax++)
            for (int k = 0; k < 6; k++) {
                const double ck = tr.c(ig, k, ax);
                pos[ax] += ck * b0[k]; vel[ax] += ck * b1[k]; acc[ax] += ck * b2[k]; jer[ax] += ck * b3[k];
            }
        double q[4];
        F.forward(vel, acc, jer, q);
        const M3 R = quat_to_R(q);
        double best = H;
        long long barg = -1;
        bool finite = std::isfinite(pos.x) && std::isfinite(pos.y) && std::isfinite(pos.z);
        for (int k = 0; k < 9; k++) finite = finite && std::isfinite(R.m[k]);
        if (!finite) best = nan;
        else {
            int lo[3] = {0, 0, 0}, hi[3] = {X - 1, Y - 1, Z - 1};
            if (!unrestricted) {
                const int n[3] = {X, Y, Z};
                for (int a = 0; a < 3; a++) {   // world AABB of the inflated body box, one voxel wider
                    const double e = hb * (std::fabs(R.m[3 * a]) + std::fabs(R.m[3 * a + 1]) + std::fabs(R.m[3 * a + 2]));
                    lo[a] = (int)std::max(0.0, std::floor((pos[a] - e - bmin[a]) / res) - 1.0);
                    hi[a] = (int)std::min((double)(n[a] - 1), std::floor((pos[a] + e - bmin[a]) / res) + 1.0);
                }
            }
            for (int ix = lo[0]; ix <= hi[0]; ix++)
                for (int iy = lo[1]; iy <= hi[1]; iy++)
                    for (int iz = lo[2]; iz <= hi[2]; iz++) {
                        const long long a = ((long long)ix * Y + iy) * Z + iz;
                        if (!occ[a]) continue;
                        const V3 pv = V3((ix + 0.5) * res, (iy + 0.5) * res, (iz + 0.5) * res) + bm;   // getGridCubeCenter
                        const V3 prel = mulT(R, pv - pos);
                        if (!unrestricted && (std::fabs(prel.x) > hb || std::fabs(prel.y) > hb || std::fabs(prel.z) > hb)) continue;
                        const double v = S_.sdf(prel);
                        if (v < best) { best = v; barg = a; }   // ascending address: the first voxel attaining the minimum wins ties
                    }
        }
        val[s] = best; arg[s] = barg;
    }
    if (clearance) std::copy(val.begin(), val.end(), clearance);
    // per trajectory, in (piece, j) order
    for (int b = 0; b < B; b++) {
        orc_clearance_report &r = reports[b];
        r.collides = 0; r.piece_hit = r.sample_hit = -1; r.t_hit = -1.0; r.p_hit[0] = r.p_hit[1] = r.p_hit[2] = nan; r.reserved_ = 0;
        r.min_clearance = nan; r.piece_min = -1;
        long long arg_min = -1, arg_hit = -1;
        double tsum = 0.0;
        for (int i = 0; i < N0; i++) {
            const int ig = b * N0 + i;
            const double step = T[ig] * (1.0 / M);
            for (int j = 0; j <= M; j++) {
                const long long s = (long long)ig * (M + 1) + j;
                const double best = val[s];
                const double t = tsum + j * step;
                // (value, sample) minimum; a NaN sample sorts first
                const bool take = r.piece_min < 0 || (std::isnan(best) && !std::isnan(r.min_clearance)) ||
                                  (!std::isnan(best) && !std::isnan(r.min_clearance) && best < r.min_clearance);
                if (take) { r.min_clearance = best; r.t_min = t; r.piece_min = i; r.sample_min = j; arg_min = arg[s]; }
                if (!r.collides && !(best >= margin)) { r.collides = 1; r.t_hit = t; r.piece_hit = i; r.sample_hit = j; arg_hit = arg[s]; }
            }
            tsum += T[ig];
        }
        centre(arg_min, r.p_min);
        if (r.collides) centre(arg_hit, r.p_hit);
    }
    return 0;
}

}  // extern "C"
