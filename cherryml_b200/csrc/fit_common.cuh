// Pieces shared by the small-S and large-S fit kernels: the reversible parameterisation
// Q(theta) with its adjoint, the Adam / SGD update, Taylor degree / scaling selection.
//
// Reference semantics (songlab-cal/CherryML v0.2.0):
//   Q(theta)        estimation/_ratelearn/rate.py:167-188 ("pande_reversible"):
//                   s = mask * sym(softplus(upper_diag)), pi = softmax(pi_logits),
//                   M = diag(pi^-1/2) s diag(pi^1/2), Q = M - diag(rowsum(M))
//   optimiser       torch.optim.Adam(lr, betas=(0.9,0.999), eps=1e-8) / SGD(lr),
//                   estimation/_ratelearn/ratelearner.py:123-130
//   parameter order pi logits first, then the S(S-1)/2 upper-diagonal entries in row-major
//                   (triu_indices) order -- the order nn.Module registers them (rate.py:44-53).
#pragma once
#include <cuda_runtime.h>
#include <math.h>

namespace cherry {

// torch.nn.Softplus(beta=1, threshold=20)
__device__ __forceinline__ double softplus_d(double x) { return x > 20.0 ? x : log1p(exp(x)); }
// d softplus / dx (torch uses the same threshold in backward)
__device__ __forceinline__ double softplus_grad_d(double x) {
  if (x > 20.0) return 1.0;
  double e = exp(x);
  return e / (1.0 + e);
}

// index of (i, j), i < j, in the row-major upper triangle of an S x S matrix
__device__ __host__ __forceinline__ int triu_index(int i, int j, int S) {
  return i * S - (i * (i + 1)) / 2 + (j - i - 1);
}

// One Adam (torch semantics, no amsgrad / weight decay) or SGD step on one parameter.
// `step` is the 1-based step count.  A parameter at -inf with zero gradient stays put.
__device__ __forceinline__ void optimizer_step(double& p, double& m, double& v, double g, double lr,
                                               int do_adam, double beta1, double beta2, double eps,
                                               double bc1, double bc2_sqrt) {
  if (do_adam) {
    m = m + (g - m) * (1.0 - beta1);
    v = beta2 * v + (1.0 - beta2) * g * g;
    const double denom = sqrt(v) / bc2_sqrt + eps;
    const double upd = (lr / bc1) * (m / denom);
    if (upd != 0.0) p -= upd;
  } else {
    if (g != 0.0) p -= lr * g;
  }
}

// Taylor degree m (1..kMaxDegree) and squarings s for ||A||_1 = norm: the smallest m whose
// threshold covers the norm, else the maximal degree with s = ceil(log2(norm / theta_max)).
// Thresholds keep the truncation error below 2^-53 * 1e-3 relative to ||A||_1 itself, so
// that small off-diagonal probabilities keep ~13 significant digits before the log.
// Returns false when the norm needs more than kMaxSquarings squarings; s is then clamped to
// kMaxSquarings and the result is outside the accuracy the thresholds promise.  An inf / nan
// norm gets s = 0 and returns true: the nan propagates to the output instead.
constexpr int kMaxDegree = 9;
constexpr int kMaxSquarings = 30;  // covers ||tQ||_1 up to 0.0376 * 2^30 ~ 4e7
__device__ __forceinline__ bool choose_degree(double norm, int& m, int& s) {
  // theta_m solves theta^m / (m+1)! = 1.1e-19
  const double theta[kMaxDegree + 1] = {0.0,      2.2e-19,  8.1e-10, 1.38e-6, 6.0e-5,
                                        6.0e-4,   2.8e-3,   8.4e-3,  0.0195,  0.0376};
  s = 0;
  for (m = 1; m <= kMaxDegree; ++m)
    if (norm <= theta[m]) return true;
  m = kMaxDegree;
  if (!(norm < 1e300)) { s = 0; return true; }  // inf / nan: let it propagate, do not loop
  double r = norm / theta[kMaxDegree];
  s = (int)ceil(log2(r));
  if (s < 0) s = 0;
  if (s > kMaxSquarings) {
    s = kMaxSquarings;
    return false;
  }
  return true;
}

__device__ __forceinline__ double inv_factorial(int j) {
  const double f[kMaxDegree + 1] = {1.0,        1.0,          0.5,           1.0 / 6,      1.0 / 24,
                                    1.0 / 120,  1.0 / 720,    1.0 / 5040,    1.0 / 40320,  1.0 / 362880};
  return f[j];
}

}  // namespace cherry
