// Beta policy on a bounded action interval (Chou, Maturana & Scherer, ICML 2017): the device math shared by the head kernel
// (heads.cu) and the loss / pre-pass kernels (ppo_loss.cu).
//
// Head output row z[0 .. 2A): alpha_j = 1 + softplus(z[j]), beta_j = 1 + softplus(z[A + j]) (torch's F.softplus, beta = 1,
// threshold 20), in fp32.  Everything after the concentrations runs in fp64 and is rounded once.  Each dimension j maps
// Beta(alpha_j, beta_j) on [0, 1] affinely onto [low_j, high_j].
//
// beta_logp is THE log-prob: the head kernel applies it to the action it has just emitted, the loss kernel and the decoupled
// pre-pass kernel call it on the stored action, so equal head outputs and actions give equal bits everywhere.
#pragma once
#include <cuda_runtime.h>

namespace ddrl {

constexpr double kBetaEps = 1e-6;           // x is clamped into [eps, 1 - eps] for the log-prob and the sample
constexpr int kBetaMaxA = 8;                // same limit as the Gaussian head
constexpr int kBetaCfTerms = 1000;          // cap of the incomplete-beta continued fraction (O(sqrt(max(a, b))) terms needed)

// torch.nn.functional.softplus (beta 1, threshold 20) and its derivative as torch's softplus_backward computes it
__device__ __forceinline__ float beta_softplus(float z) { return z > 20.f ? z : log1pf(expf(z)); }
__device__ __forceinline__ float beta_softplus_grad(float z) {
  if (z > 20.f) return 1.f;
  const float e = expf(z);
  return e / (e + 1.f);
}
__device__ __forceinline__ float beta_conc(float z) { return 1.f + beta_softplus(z); }

// NaN stays NaN (fminf / fmaxf would turn it into a bound)
__device__ __forceinline__ double beta_clamp_x(double x) {
  return x < kBetaEps ? kBetaEps : (x > 1.0 - kBetaEps ? 1.0 - kBetaEps : x);
}

// psi(z) for z > 0: recurrence up to z >= 6, then the asymptotic series (error < 1e-13 there)
__device__ __forceinline__ double beta_digamma(double z) {
  double acc = 0.0;
  for (int i = 0; i < 6 && z < 6.0; ++i) { acc -= 1.0 / z; z += 1.0; }
  const double r = 1.0 / z, r2 = r * r;
  return acc + log(z) - 0.5 * r -
         r2 * (1.0 / 12 - r2 * (1.0 / 120 - r2 * (1.0 / 252 - r2 * (1.0 / 240 - r2 * (1.0 / 132)))));
}

// psi'(z) for z > 0, the same way
__device__ __forceinline__ double beta_trigamma(double z) {
  double acc = 0.0;
  for (int i = 0; i < 6 && z < 6.0; ++i) { acc += 1.0 / (z * z); z += 1.0; }
  const double r = 1.0 / z, r2 = r * r;
  return acc + r + 0.5 * r2 + r * r2 * (1.0 / 6 - r2 * (1.0 / 30 - r2 * (1.0 / 42 - r2 * (1.0 / 30))));
}

__device__ __forceinline__ double beta_lbeta(double a, double b) { return lgamma(a) + lgamma(b) - lgamma(a + b); }

// continued fraction of I_x(a, b) (modified Lentz), at most kBetaCfTerms terms
__device__ __forceinline__ double beta_cf(double a, double b, double x) {
  const double tiny = 1e-300, eps = 1e-15;
  const double qab = a + b, qap = a + 1.0, qam = a - 1.0;
  double c = 1.0, d = 1.0 - qab * x / qap;
  if (fabs(d) < tiny) d = tiny;
  d = 1.0 / d;
  double h = d;
  for (int m = 1; m <= kBetaCfTerms; ++m) {
    const int m2 = 2 * m;
    double aa = m * (b - m) * x / ((qam + m2) * (a + m2));
    d = 1.0 + aa * d; if (fabs(d) < tiny) d = tiny;
    c = 1.0 + aa / c; if (fabs(c) < tiny) c = tiny;
    d = 1.0 / d;
    h *= d * c;
    aa = -(a + m) * (qab + m) * x / ((a + m2) * (qap + m2));
    d = 1.0 + aa * d; if (fabs(d) < tiny) d = tiny;
    c = 1.0 + aa / c; if (fabs(c) < tiny) c = tiny;
    d = 1.0 / d;
    const double del = d * c;
    h *= del;
    if (fabs(del - 1.0) < eps) break;
  }
  return h;
}

// regularised incomplete beta I_x(a, b); lb = lbeta(a, b)
__device__ __forceinline__ double beta_inc(double a, double b, double x, double lb) {
  if (x <= 0.0) return 0.0;
  if (x >= 1.0) return 1.0;
  const double bt = exp(a * log(x) + b * log1p(-x) - lb);
  if (x < (a + 1.0) / (a + b + 2.0)) return bt * beta_cf(a, b, x) / a;
  return 1.0 - bt * beta_cf(b, a, 1.0 - x) / b;
}

// x = I^-1_{a,b}(p) for a, b >= 1.  The solve runs in the lower tail (p > 1/2 is solved as 1 - I^-1_{b,a}(1 - p)), so that I
// is never formed as 1 - (something close to 1).  Start: the normal approximation of Abramowitz & Stegun 26.5.22.  Steps:
// Newton on log I_x(a, b) = log p, at most kBetaNewtonSteps.  For a, b >= 1 the density is log-concave, so log I_x is concave
// and increasing in x: after at most one step the iterates approach the root monotonically from the left.  (Newton or Halley
// on I_x itself converge only linearly in the far tail, where I_x behaves like x^a.)  A non-finite a, b or p gives NaN; p <= 0
// gives 0 and p >= 1 gives 1.
constexpr int kBetaNewtonSteps = 16;

__device__ __forceinline__ double beta_inc_inv(double a, double b, double p) {
  if (!(isfinite(a) && isfinite(b) && isfinite(p))) return __longlong_as_double(0x7ff8000000000000LL);
  if (p <= 0.0) return 0.0;
  if (p >= 1.0) return 1.0;
  const bool upper = p > 0.5;
  if (upper) { const double t = a; a = b; b = t; p = 1.0 - p; }
  const double t0 = sqrt(-2.0 * log(p));
  const double y = t0 - (2.30753 + t0 * 0.27061) / (1.0 + t0 * (0.99229 + t0 * 0.04481));
  const double al = (y * y - 3.0) / 6.0;
  const double h = 2.0 / (1.0 / (2.0 * a - 1.0) + 1.0 / (2.0 * b - 1.0));
  const double w = y * sqrt(al + h) / h - (1.0 / (2.0 * b - 1.0) - 1.0 / (2.0 * a - 1.0)) * (al + 5.0 / 6.0 - 2.0 / (3.0 * h));
  double x = a / (a + b * exp(2.0 * w));
  if (!(x > 0.0 && x < 1.0)) x = a / (a + b);             // the start left (0, 1): start from the mean
  const double lb = beta_lbeta(a, b), lp = log(p);
  for (int k = 0; k < kBetaNewtonSteps; ++k) {
    const double v = beta_inc(a, b, x, lb);
    double xn;
    if (v > 0.0) {
      const double dens = exp((a - 1.0) * log(x) + (b - 1.0) * log1p(-x) - lb);
      xn = x - (log(v) - lp) * v / dens;
      if (xn <= 0.0) xn = 0.5 * x;
      if (xn >= 1.0) xn = 0.5 * (x + 1.0);
    } else {
      xn = 0.5 * (x + 1.0);                                 // I_x underflowed: x is far left of the root
    }
    const bool done = fabs(xn - x) <= 1e-13 * xn;
    x = xn;
    if (done) break;
  }
  return upper ? 1.0 - x : x;
}

// log-prob of the action row act[0 .. A) (env units) under the Beta policy of the head row z[0 .. 2A), summed in j order:
//   x = clamp((a - low) / (high - low), eps, 1 - eps)
//   sum_j (alpha-1) log x + (beta-1) log1p(-x) - lbeta(alpha, beta) - log(high - low)
// in fp64, rounded once
__device__ __forceinline__ float beta_logp(const float* __restrict__ z, const float* __restrict__ low,
                                           const float* __restrict__ high, const float* __restrict__ act, int A) {
  double lp = 0.0;
  for (int j = 0; j < A; ++j) {
    const double al = beta_conc(z[j]), be = beta_conc(z[A + j]);
    const double lo = low[j], w = (double)high[j] - lo;
    const double x = beta_clamp_x(((double)act[j] - lo) / w);
    lp += (al - 1.0) * log(x) + (be - 1.0) * log1p(-x) - beta_lbeta(al, be) - log(w);
  }
  return (float)lp;
}

// differential entropy of Beta(a, b) on an interval of width w: H(Beta(a, b)) + log w
__device__ __forceinline__ double beta_entropy(double a, double b, double w) {
  return beta_lbeta(a, b) - (a - 1.0) * beta_digamma(a) - (b - 1.0) * beta_digamma(b) + (a + b - 2.0) * beta_digamma(a + b) +
         log(w);
}

}  // namespace ddrl
