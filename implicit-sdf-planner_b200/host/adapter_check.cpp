// Compiles the host-side adapters (syntax + ABI check in build()) and exports flat hooks so the python tests can drive
// them: the MINCO port against the oracle / numpy, and the full LMBM-signature callback on the GPU box.
#include "isdf_shape_adapter.hpp"
#include "isdf_cost_callback.hpp"
#include "isdf_lbfgs.hpp"
#include "isdf_obj.hpp"
#include <algorithm>
#include <cstring>
#include <vector>

using namespace isdf_host;

// the adapters must be assignable to the reference's callback typedefs
typedef double (*lmbm_evaluate_t)(void *instance, const double *x, double *g, const int n);   // lmbm/lmbm.h:206-209
static lmbm_evaluate_t check_lmbm_signature = &BackEnd::costFunctionLmbm;

extern "C" {

int isdf_host_minco_forward(int N, const double *head, const double *tail, const double *inPs, const double *T, double *coeffs,
                            double *energy, double *gradC_energy, double *gradT_energy) {
    MincoS3 m; m.setConditions(head, tail, N); m.setParameters(inPs, T);
    std::memcpy(coeffs, m.coeffs().data(), sizeof(double) * 18 * N);
    if (energy) *energy = m.getEnergy();
    if (gradC_energy) m.getEnergyPartialGradByCoeffs(gradC_energy);
    if (gradT_energy) m.getEnergyPartialGradByTimes(gradT_energy);
    return check_lmbm_signature ? 0 : 1;
}
int isdf_host_minco_backward(int N, const double *head, const double *tail, const double *inPs, const double *T, const double *gradC,
                             const double *gradT, double *gradP, double *gradTout) {
    MincoS3 m; m.setConditions(head, tail, N); m.setParameters(inPs, T);
    m.propagateGrad(gradC, gradT, gradP, gradTout);
    return 0;
}
void *isdf_host_backend_create(isdf_ctx *ctx, int N, const double *head, const double *tail, double rho, int use_swept, int use_time_integral) {
    BackEnd *b = new BackEnd();
    b->setup(ctx, N, head, tail);
    b->rho = rho; b->use_swept = use_swept != 0; b->use_time_integral = use_time_integral != 0;
    return b;
}
double isdf_host_backend_cost(void *be, const double *x, double *g, int n) { return BackEnd::costFunctionLmbm(be, x, g, n); }
void isdf_host_backend_last(void *be, double *cost_pos, double *cost_other, double *cost_total, int *status) {
    BackEnd *b = (BackEnd *)be;
    *cost_pos = b->cost_pos; *cost_other = b->cost_other; *cost_total = b->cost_total; *status = b->last_status;
}
// BackEnd::isTrajCollide on decision vector x (reports into *rep); returns 1 = collides or failed, 0 = collision-free
int isdf_host_backend_collides(void *be, const double *x, int check_samples, double margin, double horizon, isdf_clearance_report *rep, int *status) {
    BackEnd *b = (BackEnd *)be;
    b->check_samples = check_samples;
    const bool hit = b->isTrajCollide(x, margin, horizon, rep);
    if (status) *status = b->last_status;
    return hit ? 1 : 0;
}
void isdf_host_backend_destroy(void *be) { delete (BackEnd *)be; }
void isdf_host_tau_maps(const double *tau, int n, double *T, double *tau_back) { BackEnd::forwardT(tau, T, n); BackEnd::backwardT(T, tau_back, n); }
// OBJ reader (read_triangle_mesh counterpart): returns 0 and the counts; copies up to capV vertices / capF faces when the buffers are given
int isdf_host_read_obj(const char *path, double *V, int capV, int32_t *F, int capF, int *nV, int *nF) {
    std::vector<double> v; std::vector<int32_t> f; std::string err;
    if (!read_obj(path, v, f, err)) return -1;
    *nV = (int)(v.size() / 3); *nF = (int)(f.size() / 3);
    if (V) std::memcpy(V, v.data(), sizeof(double) * 3 * (size_t)std::min(*nV, capV));
    if (F) std::memcpy(F, f.data(), sizeof(int32_t) * 3 * (size_t)std::min(*nF, capF));
    return 0;
}
int isdf_host_set_shape_obj(isdf_ctx *ctx, const char *path, const double *poly_params6) { return set_shape_obj(ctx, path, poly_params6); }
double isdf_host_shape_sdf_grad(isdf_ctx *ctx, const double *p, double *grad) { DeviceShape s(ctx); return s.getSDFwithGrad1(p, grad); }

// L-BFGS on any raw callback (known-answer tests, CPU baseline with the oracle as the callback) ...
int isdf_host_lbfgs_generic(int n, double *x, double *f, lbfgs_eval_raw_t eval, void *instance, int mem_size, int past, double delta,
                            double g_epsilon, int max_iterations, int *iterations, int *evaluations) {
    LbfgsParams pr; pr.mem_size = mem_size; pr.past = past; pr.delta = delta; pr.g_epsilon = g_epsilon; pr.max_iterations = max_iterations;
    pr.min_step = 1.0e-32;                                   // config_CappedCone.yaml:101
    LbfgsStats st; double fx = 0;
    const int r = lbfgs_optimize(n, x, fx, eval, nullptr, nullptr, instance, pr, &st);
    *f = fx; if (iterations) *iterations = st.iterations; if (evaluations) *evaluations = st.evaluations;
    return r;
}
// ... and on the GPU-backed callback (BackEnd::costFunctionLbfgs)
int isdf_host_lbfgs_backend(void *be, double *x, int n, double *f, int mem_size, int past, double delta, double g_epsilon, int max_iterations,
                            int *iterations, int *evaluations) {
    return isdf_host_lbfgs_generic(n, x, f, &BackEnd::costFunctionLbfgs, be, mem_size, past, delta, g_epsilon, max_iterations, iterations, evaluations);
}

// lock-step batched driver on any batched callback (CPU tests: identical to the sequential driver instance by instance) ...
int isdf_host_lbfgs_batch_generic(int B, int n, double *x, double *f, int *ret, lbfgs_eval_batch_t eval, void *instance, int mem_size, int past,
                                  double delta, double g_epsilon, int max_iterations, int *iterations, int *evaluations) {
    LbfgsParams pr; pr.mem_size = mem_size; pr.past = past; pr.delta = delta; pr.g_epsilon = g_epsilon; pr.max_iterations = max_iterations;
    pr.min_step = 1.0e-32;
    if (B < 1 || n < 1 || mem_size < 1) return -1;
    std::vector<LbfgsStats> st(B);
    const int rounds = lbfgs_optimize_batch(B, n, x, f, ret, eval, instance, pr, st.data());
    for (int b = 0; b < B; b++) { if (iterations) iterations[b] = st[b].iterations; if (evaluations) evaluations[b] = st[b].evaluations; }
    return rounds;
}
// ... and on the device callback for B random-restart problems (isdf_callback_batch: MINCO + time-integral/collision term + adjoint)
struct BatchBackEnd { isdf_ctx *ctx; int N0; const double *heads, *tails; double rho; std::vector<double> h, t; int status; };
static void batch_backend_eval(void *inst, int nb, const int *ids, const double *x, double *f, double *g) {
    BatchBackEnd &b = *static_cast<BatchBackEnd *>(inst);
    b.h.resize((size_t)9 * nb); b.t.resize((size_t)9 * nb);
    for (int q = 0; q < nb; q++) {
        std::memcpy(&b.h[(size_t)9 * q], b.heads + (size_t)9 * ids[q], sizeof(double) * 9);
        std::memcpy(&b.t[(size_t)9 * q], b.tails + (size_t)9 * ids[q], sizeof(double) * 9);
    }
    const int r = isdf_callback_batch(b.ctx, nb, b.N0, b.h.data(), b.t.data(), 1, b.rho, x, f, g);   // on failure every f is NaN: the instances stop
    if (r != ISDF_OK) b.status = r;
}
int isdf_host_lbfgs_batch_backend(isdf_ctx *ctx, int B, int N0, const double *heads, const double *tails, double rho, double *x, double *f, int *ret,
                                  int mem_size, int past, double delta, double g_epsilon, int max_iterations, int *iterations, int *evaluations,
                                  int *status) {
    BatchBackEnd be{ctx, N0, heads, tails, rho, {}, {}, 0};
    const int rounds = isdf_host_lbfgs_batch_generic(B, 4 * N0 - 3, x, f, ret, &batch_backend_eval, &be, mem_size, past, delta, g_epsilon, max_iterations,
                                                     iterations, evaluations);
    if (status) *status = be.status;
    return rounds;
}

}  // extern "C"
