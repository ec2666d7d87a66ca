// Host-side adapter presenting the GPU evaluator behind the reference's optimiser-callback surface:
//   lmbm_evaluate_t : double (*)(void* instance, const double* x, double* g, const int n)            (lmbm/lmbm.h:206-209)
//   lbfgs_evaluate_t: double (*)(void*, const Eigen::VectorXd& x, Eigen::VectorXd& g, double& p_cost) (utils/lbfgs.hpp:213-216)
// BackEnd::costFunctionLmbm restates TrajOptimizer::costFunctionLmbm (back_end_optimizer.hpp:358-430) step for step:
//   x = [tau (N) | xi (3(N-1), waypoint-major)] -> forwardT / forwardP (hpp:175-241) -> MINCO -> energy and its partials ->
//   swept-volume penalty (isdf_eval_swept == addSaftyPenaOnSweptVolumeParallel) -> time-integral penalty (isdf_eval_discrete ==
//   addTimeIntPenaltyParallel) -> propogateGrad -> + rho * sum(T) -> backwardGradT / backwardGradP (hpp:283-330).
// Both device calls ACCUMULATE into cost / gradT / gradC exactly like the reference's reference-arguments.
// On a device error the cost is NaN (see include/isdf.h) so either optimiser driver stops.
// BackEnd::isTrajCollide is the hard verdict the reference's SweptVolumeManager::isTrajCollide (sw_manager.hpp:759-767) only stubs:
// the decision vector the optimiser returned -> the same trajectory costFunctionLmbm evaluates -> isdf_check_collision.
#pragma once
#include "isdf.h"
#include "isdf_minco.hpp"
#include <cmath>
#include <limits>
#include <vector>
#ifdef ISDF_WITH_EIGEN
#include <Eigen/Core>
#endif

namespace isdf_host {

struct BackEnd {
    isdf_ctx *ctx = nullptr;
    int N = 0;                    // pieces; temporalDim = N, spatialDim = 3 (N - 1)  (back_end_optimizer.cpp:24-28)
    double rho = 20.0;            // time weight (hpp:682)
    bool use_swept = true;        // the live collision term (hpp:386-391)
    bool use_time_integral = true;  // hpp:399-405; includes grad_cost_p when ctx was created with ISDF_WITH_COLLISION
    MincoS3 minco;
    std::vector<double> times, points, gradC, gradT, gradPts, gradTimes;
    // per-evaluation diagnostics the reference publishes to its debug monitor (hpp:112-114, 422-424)
    double cost_pos = 0, cost_other = 0, cost_total = 0;
    long cost_iter = 0;
    int last_status = 0;
    int check_samples = 64;       // isTrajCollide: check intervals per piece (the natural choice: the context's integral_intervs)

    void setup(isdf_ctx *c, int pieces, const double *head3x3, const double *tail3x3) {
        ctx = c; N = pieces;
        minco.setConditions(head3x3, tail3x3, N);
        times.assign(N, 0.0); points.assign((size_t)3 * (N - 1), 0.0);
        gradC.assign((size_t)18 * N, 0.0); gradT.assign(N, 0.0); gradPts.assign((size_t)3 * (N - 1), 0.0); gradTimes.assign(N, 0.0);
    }

    // tau -> T diffeomorphism and its pull-back (hpp:214-241, 283-305)
    static void forwardT(const double *tau, double *T, int n) {
        for (int i = 0; i < n; i++) { const double t = tau[i]; T[i] = t > 0.0 ? ((0.5 * t + 1.0) * t + 1.0) : 1.0 / ((0.5 * t - 1.0) * t + 1.0); }
    }
    static void backwardT(const double *T, double *tau, int n) {   // hpp:243-256
        for (int i = 0; i < n; i++) tau[i] = T[i] > 1.0 ? (std::sqrt(2.0 * T[i] - 1.0) - 1.0) : (1.0 - std::sqrt(2.0 / T[i] - 1.0));
    }
    static void backwardGradT(const double *tau, const double *gradT, double *gradTau, int n) {
        for (int i = 0; i < n; i++) {
            if (tau[i] > 0) gradTau[i] = gradT[i] * (tau[i] + 1.0);
            else { const double den = (0.5 * tau[i] - 1.0) * tau[i] + 1.0; gradTau[i] = gradT[i] * (1.0 - tau[i]) / (den * den); }
        }
    }

    // lmbm_evaluate_t
    static double costFunctionLmbm(void *ptr, const double *x, double *g, const int n) {
        BackEnd &o = *static_cast<BackEnd *>(ptr);
        o.cost_iter++;
        const int dimTau = o.N, dimXi = 3 * (o.N - 1);
        if (n != dimTau + dimXi) { o.last_status = ISDF_ERR_INVALID; return std::numeric_limits<double>::quiet_NaN(); }
        forwardT(x, o.times.data(), dimTau);
        for (int k = 0; k < dimXi; k++) o.points[k] = x[dimTau + k];                 // forwardP: column i = xi[3i .. 3i+2]
        o.minco.setParameters(o.points.data(), o.times.data());
        double cost = o.minco.getEnergy();
        o.minco.getEnergyPartialGradByCoeffs(o.gradC.data());
        o.minco.getEnergyPartialGradByTimes(o.gradT.data());
        const double energy_cost = cost;
        const double *coeffs = o.minco.coeffs().data();
        int rc = ISDF_OK;
        if (o.use_swept) rc = isdf_eval_swept(o.ctx, o.N, o.times.data(), coeffs, &cost, o.gradC.data(), o.gradT.data());
        double pos_cost = cost - energy_cost;
        if (rc == ISDF_OK && o.use_time_integral) rc = isdf_eval_discrete(o.ctx, o.N, o.times.data(), coeffs, &cost, o.gradC.data(), o.gradT.data());
        o.last_status = rc;
        if (rc != ISDF_OK) return std::numeric_limits<double>::quiet_NaN();
        o.minco.propagateGrad(o.gradC.data(), o.gradT.data(), o.gradPts.data(), o.gradTimes.data());
        double tsum = 0.0;
        for (int i = 0; i < dimTau; i++) tsum += o.times[i];
        cost += o.rho * tsum;
        for (int i = 0; i < dimTau; i++) o.gradTimes[i] += o.rho;
        o.cost_pos = pos_cost; o.cost_other = cost - pos_cost; o.cost_total = cost;
        backwardGradT(x, o.gradTimes.data(), g, dimTau);
        for (int k = 0; k < dimXi; k++) g[dimTau + k] = o.gradPts[k];               // backwardGradP
        return cost;
    }

    // Does the trajectory of decision vector x (n = N + 3(N-1): what the optimiser returned) collide? Rebuilds the trajectory exactly
    // as costFunctionLmbm does (forwardT, forwardP, MINCO) and checks it at check_samples + 1 samples per piece. Returns true on a hit
    // AND on any error (rep->min_clearance is NaN then, last_status has the code): a failed check never reads "safe". rep may be NULL.
    bool isTrajCollide(const double *x, double margin, double horizon, isdf_clearance_report *rep = nullptr) {
        isdf_clearance_report local;
        if (!rep) rep = &local;
        const int dimTau = N, dimXi = 3 * (N - 1);
        if (!ctx || N < 1 || !x) { last_status = ISDF_ERR_INVALID; rep->min_clearance = std::numeric_limits<double>::quiet_NaN(); rep->collides = 1; return true; }
        forwardT(x, times.data(), dimTau);
        for (int k = 0; k < dimXi; k++) points[k] = x[dimTau + k];
        minco.setParameters(points.data(), times.data());
        last_status = isdf_check_collision(ctx, 1, N, times.data(), minco.coeffs().data(), check_samples, margin, horizon, rep, nullptr);
        return last_status != ISDF_OK || rep->collides != 0;
    }

    // raw twin of lbfgs_evaluate_t (the reference's fork adds the p_cost out-parameter, lbfgs.hpp:213-216)
    static double costFunctionLbfgs(void *ptr, const double *x, double *g, int n, double *p_cost) {
        const double c = costFunctionLmbm(ptr, x, g, n);
        if (p_cost) *p_cost = static_cast<BackEnd *>(ptr)->cost_pos;
        return c;
    }
#ifdef ISDF_WITH_EIGEN
    static double costFunction(void *ptr, const Eigen::VectorXd &x, Eigen::VectorXd &g, double &p_cost) {
        g.resize(x.size());
        return costFunctionLbfgs(ptr, x.data(), g.data(), (int)x.size(), &p_cost);
    }
#endif
};

}  // namespace isdf_host
