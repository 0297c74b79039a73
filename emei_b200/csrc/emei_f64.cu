// float64 / reference-exact mode of every entry point.  MUST be compiled with -fmad=false: the
// expression order in kernels.cuh is then exactly the arithmetic of the reference's python.
#define EMEI_REAL double
#define EMEI_FN(name) name##_f64
#define EMEI_POLICY_ARS  // the precision-independent policy-search kernels (policy.cuh) live here
#include "impl.inc"

extern "C" {
int emei_policy_perturb(const double* theta, double* params, int64_t N, int64_t P, const emei_policy_params* policy, emei_stream_t stream) {
  return emei::policy_perturb(theta, params, N, P, policy, stream);
}

int emei_policy_update(const double* returns, double* theta_io, double* stats, int64_t N, int64_t E, int64_t P,
                       const emei_policy_params* policy, emei_stream_t stream) {
  return emei::policy_update(returns, theta_io, stats, N, E, P, policy, stream);
}
}  // extern "C"
