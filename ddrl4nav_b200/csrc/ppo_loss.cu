// K6 -- fused PPO loss, forward + backward, one pass over the minibatch rows.
//
// Replaces USTC_lab/nn/ppo.py:85-108 and the autograd chain from the three loss scalars back to
// the head outputs (actor_linear output and critic_linear output):
//   ratio = exp(logp - old_logp)
//   s     = min(ratio*A, clamp(ratio, 1-c, 1+c)*A)
//   actor = -mean( A>0 ? s : max(s, dual*A) )                  (dual-clip PPO, ppo.py:87-92)
//   v     = mean((R - v)^2)/2  |  smooth_l1(R, v)              (ppo.py:54-57,95)
//   ent   = mean(dist.entropy())                               (ppo.py:106)
//   shared:   d(actor + v_coef*v - ent_coef*ent)               (ppo.py:108-112)
//   unshared: dlogits <- actor only, dv <- v only; entropy only reported (ppo.py:122-123)
// Categorical chain follows torch exactly: softmax -> q = p/sum(p) -> clamp(eps,1-eps) -> log
// -> gather (nn/actor.py:94-101, torch/distributions/categorical.py:70, utils.py probs_to_logits),
// including clamp's zero gradient outside [eps,1-eps] and the 1/2-1/2 tie split of min/max.
// HBM-bound: categorical 8A+24 B/sample, Gaussian 12A+20 B/sample (SURVEY 8d).
//
// Non-reference options (off when both pointers are null; the kernels then compute exactly the reference loss):
//   old_v: clipped value loss, v_c = old_v + clamp(v - old_v, -c, c), loss = max(vloss(R, v), vloss(R, v_c)) per row
//          (clamp passes the gradient on the closed interval, max splits ties 1/2-1/2 as torch.max does).
//   stats: stats[0] += inv_B*((r - 1) - log r) (approx KL), stats[1] += inv_B*[|r - 1| > ppo_clip] (clip fraction), through
//          the same ordered / atomic adds as the loss sums.
//   value_norm (in LossParams): critic 0 learns normalised targets R~ = (R - mean32) * scale32, and old_v is normalised the same
//          way, each operation rounded on its own; the extra critics' value_loss_kernel never normalises.
//   prox (in LossParams, DECOUPLED_PPO): the ratio is taken against the proximal log-prob, r = exp(logp - prox), and the actor
//          term and its gradient are weighted by the behaviour weight w = exp(prox - old_logp) (min(w, is_clip) when is_clip > 0):
//          w * term(r, A) and w * dterm * r.  stats[2] += inv_B*((rho - 1) - log rho), rho = exp(prox - old_logp) untruncated.
//          With prox null, w = 1 and every product by it is exact: the kernels compute exactly the loss without it.
#include "common.cuh"

namespace ddrl {

constexpr float kEpsL = 1.1920928955078125e-07f;
constexpr float kF32Min = -3.4028234663852886e+38f;
constexpr float kLogSqrt2PiL = 0.918938533204672741780329736406f;
constexpr int kMaxAL = 64;

struct LossParams {
  float ppo_clip, dual_clip, v_coef, ent_coef, inv_B, value_clip;
  int smooth_l1, shared;
  const float* value_norm;        // NORM_VALUE: device {mean32, scale32, sigma32} of critic 0's targets, or null
  const float* prox;              // DECOUPLED_PPO: proximal log-probs [B], or null
  float is_clip;                  // DECOUPLED_PPO: truncation of the behaviour weight, <= 0: none
};

// log-prob of the taken action a (clamped into [0, A)) under Categorical(logits = x[0..A)): the softmax -> q = p / sum(p) ->
// clamp(eps, 1 - eps) -> log chain of torch.  Leaves the softmax p[0..A) and s2 = sum(p) for the loss kernel's gradient.  The
// loss kernel and logp_actions_categorical_kernel share it, so equal logits give equal log-prob bits.
__device__ __forceinline__ float categorical_logp(const float* __restrict__ x, int A, float action, float* p, float* s2_out) {
  float m = x[0];
  for (int j = 1; j < A; ++j) m = fmaxf(m, x[j]);
  float s = 0.f;
  for (int j = 0; j < A; ++j) { p[j] = expf(x[j] - m); s += p[j]; }
  float s2 = 0.f;
  for (int j = 0; j < A; ++j) { p[j] = p[j] / s; s2 += p[j]; }
  int a = (int)action;                      // Categorical.log_prob: value.long()
  a = a < 0 ? 0 : (a >= A ? A - 1 : a);     // the reference raises on an action outside [0, A); never read out of bounds
  const float qa = p[a] / s2;
  const float ca = fminf(fmaxf(qa, kEpsL), 1.f - kEpsL);
  *s2_out = s2;
  return logf(ca);
}

// log-prob of the action row act[0..A) under Normal(mu[0..A), exp(log_std)) summed over A (normal.py log_prob); shared by the
// Gaussian loss kernel and logp_actions_gaussian_kernel
__device__ __forceinline__ float gaussian_logp(const float* __restrict__ mu, const float* __restrict__ log_std,
                                               const float* __restrict__ act, int A) {
  float lp = 0.f;
  for (int j = 0; j < A; ++j) {
    const float sd = expf(log_std[j]);
    const float z = act[j] - mu[j];
    lp += -(z * z) / (2.f * (sd * sd)) - logf(sd) - kLogSqrt2PiL;
  }
  return lp;
}

// DECOUPLED_PPO: log r against the proximal log-prob when it is given (else against old_logp), and the behaviour weight w
// (1 without prox); *l_bkl = inv_B * ((rho - 1) - log rho) with rho = exp(prox - old_logp) when stats are on
__device__ __forceinline__ float decoupled_log_ratio(float logp, const float* __restrict__ old_logp, int b, const LossParams& hp,
                                                     bool stats, float* w, float* l_bkl) {
  if (!hp.prox) { *w = 1.f; return logp - old_logp[b]; }
  const float pl = hp.prox[b];
  const float log_rho = pl - old_logp[b];
  const float rho = expf(log_rho);
  *w = hp.is_clip > 0.f ? fminf(rho, hp.is_clip) : rho;
  if (stats) *l_bkl = ((rho - 1.f) - log_rho) * hp.inv_B;
  return logp - pl;
}

// d(term)/d(ratio) of term = A>0 ? s : max(s, dual*A), s = min(ratio*A, clamp(ratio)*A); also returns term
__device__ __forceinline__ float surrogate(float ratio, float A, const LossParams& hp, float* dterm_dratio) {
  const float lo = 1.0f - hp.ppo_clip, hi = 1.0f + hp.ppo_clip;
  const float s1 = ratio * A;
  const float rc = fminf(fmaxf(ratio, lo), hi);
  const float s2 = rc * A;
  const float in_range = (ratio >= lo && ratio <= hi) ? 1.f : 0.f;   // clamp backward mask (closed interval)
  float w1, w2;                                                       // torch.min backward
  if (s1 < s2) { w1 = 1.f; w2 = 0.f; }
  else if (s1 > s2) { w1 = 0.f; w2 = 1.f; }
  else { w1 = 0.5f; w2 = 0.5f; }
  const float s = fminf(s1, s2);
  const float ds = w1 * A + w2 * in_range * A;
  if (A > 0.f) { *dterm_dratio = ds; return s; }
  const float d = hp.dual_clip * A;
  float wm;                                                           // torch.max backward
  if (s > d) wm = 1.f; else if (s < d) wm = 0.f; else wm = 0.5f;
  *dterm_dratio = wm * ds;
  return fmaxf(s, d);
}

__device__ __forceinline__ float value_loss(float R, float v, int smooth_l1, float* dl_dv) {
  const float z = R - v;
  if (!smooth_l1) { *dl_dv = -z; return 0.5f * z * z; }
  const float az = fabsf(z);                 // F.smooth_l1_loss(input=R, target=v), beta=1
  if (az < 1.f) { *dl_dv = -z; return 0.5f * z * z; }
  *dl_dv = z > 0.f ? -1.f : 1.f;
  return az - 0.5f;
}

// value loss of critic 0 and its d/dv, clipped around old_v when old_v is given (c = clip width); with value_norm the target and
// the old value are normalised first
__device__ __forceinline__ float value_loss_clipped(float R, float v, const float* __restrict__ old_v, int b, float c,
                                                    int smooth_l1, const float* __restrict__ value_norm, float* dl_dv) {
  float mean32 = 0.f, scale32 = 0.f;
  if (value_norm) {
    mean32 = value_norm[0];
    scale32 = value_norm[1];
    R = __fmul_rn(__fsub_rn(R, mean32), scale32);
  }
  float dl;
  const float lu = value_loss(R, v, smooth_l1, &dl);
  if (!old_v) { *dl_dv = dl; return lu; }
  const float vo = value_norm ? __fmul_rn(__fsub_rn(old_v[b], mean32), scale32) : old_v[b];
  const float d = v - vo;
  const float vc = vo + fminf(fmaxf(d, -c), c);
  float dlc;
  const float lc = value_loss(R, vc, smooth_l1, &dlc);
  const float in_range = (d >= -c && d <= c) ? 1.f : 0.f;            // clamp backward mask (closed interval)
  float w1, w2;                                                       // torch.max backward
  if (lu > lc) { w1 = 1.f; w2 = 0.f; }
  else if (lu < lc) { w1 = 0.f; w2 = 1.f; }
  else { w1 = 0.5f; w2 = 0.5f; }
  *dl_dv = w1 * dl + w2 * in_range * dlc;
  return fmaxf(lu, lc);
}

__global__ void __launch_bounds__(128) ppo_loss_categorical_kernel(
    const float* __restrict__ logits, int ld, const float* __restrict__ actions, const float* __restrict__ old_logp,
    const float* __restrict__ adv, const float* __restrict__ returns, const float* __restrict__ v, int B, int A,
    LossParams hp, float* __restrict__ dlogits, int ld_d, float* __restrict__ dv, float* __restrict__ loss_sums,
    const float* __restrict__ old_v, float* __restrict__ stats, DetSeq det) {
  __shared__ float scratch[32];
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  float l_actor = 0.f, l_v = 0.f, l_ent = 0.f, l_kl = 0.f, l_cf = 0.f, l_bkl = 0.f;
  if (b < B) {
    const float* x = logits + (size_t)b * ld;
    float p[kMaxAL];
    float s2;
    const float logp = categorical_logp(x, A, actions[b], p, &s2);      // log-prob of the taken action
    int a = (int)actions[b];
    a = a < 0 ? 0 : (a >= A ? A - 1 : a);
    const float Ai = adv[b];
    float w;
    const float log_ratio = decoupled_log_ratio(logp, old_logp, b, hp, stats != nullptr, &w, &l_bkl);
    const float ratio = expf(log_ratio);
    float dterm;
    const float term = surrogate(ratio, Ai, hp, &dterm);
    l_actor = -(w * term) * hp.inv_B;
    if (stats) {
      l_kl = ((ratio - 1.f) - log_ratio) * hp.inv_B;
      l_cf = fabsf(ratio - 1.f) > hp.ppo_clip ? hp.inv_B : 0.f;
    }
    const float w_lp = -hp.inv_B * (w * dterm) * ratio;                 // dLoss/dlogp
    const float w_ent = hp.shared ? -hp.ent_coef * hp.inv_B : 0.f;      // dLoss/dH_b
    // gradient wrt q (normalised probs): gq_j
    float H = 0.f, dot_q = 0.f;
    float gq[kMaxAL];
    for (int j = 0; j < A; ++j) {
      const float q = p[j] / s2;
      const float c = fminf(fmaxf(q, kEpsL), 1.f - kEpsL);
      const float L = fmaxf(logf(c), kF32Min);
      const float inr = (q >= kEpsL && q <= 1.f - kEpsL) ? 1.f : 0.f;
      H -= q * L;
      float g = w_ent * (-(L + inr * q / c));
      if (j == a) g += w_lp * inr / c;
      gq[j] = g;
      dot_q += g * q;
    }
    l_ent = H * hp.inv_B;
    // q = p / s2  ->  gp_k = (gq_k - sum_j gq_j q_j) / s2 ;  softmax: dx_k = p_k (gp_k - sum_j gp_j p_j)
    float dot_p = 0.f;
    for (int j = 0; j < A; ++j) { gq[j] = (gq[j] - dot_q) / s2; dot_p += gq[j] * p[j]; }
    float* dx = dlogits + (size_t)b * ld_d;
    for (int j = 0; j < A; ++j) dx[j] = p[j] * (gq[j] - dot_p);
    float dl;
    l_v = value_loss_clipped(returns[b], v[b], old_v, b, hp.value_clip, hp.smooth_l1, hp.value_norm, &dl) * hp.inv_B;
    dv[b] = dl * hp.inv_B * (hp.shared ? hp.v_coef : 1.f);
  }
  l_actor = block_sum(l_actor, scratch);
  l_v = block_sum(l_v, scratch);
  l_ent = block_sum(l_ent, scratch);
  if (stats) {
    l_kl = block_sum(l_kl, scratch);
    l_cf = block_sum(l_cf, scratch);
    if (hp.prox) l_bkl = block_sum(l_bkl, scratch);
  }
  if (threadIdx.x == 0) {
    if (det.ctr) det_enter(det.ctr, blockIdx.x);         // deterministic mode: the blocks add in block order
    det_add(det.ctr != nullptr, loss_sums + 0, l_actor);
    det_add(det.ctr != nullptr, loss_sums + 1, l_v);
    det_add(det.ctr != nullptr, loss_sums + 2, l_ent);
    if (stats) {
      det_add(det.ctr != nullptr, stats + 0, l_kl);
      det_add(det.ctr != nullptr, stats + 1, l_cf);
      if (hp.prox) det_add(det.ctr != nullptr, stats + 2, l_bkl);
    }
    if (det.ctr) det_leave(det.ctr, blockIdx.x, gridDim.x);
  }
}

__global__ void __launch_bounds__(128) ppo_loss_gaussian_kernel(
    const float* __restrict__ mu, int ld, const float* __restrict__ log_std, const float* __restrict__ actions,
    const float* __restrict__ old_logp, const float* __restrict__ adv, const float* __restrict__ returns,
    const float* __restrict__ v, int B, int A, LossParams hp, float* __restrict__ dmu, int ld_d,
    float* __restrict__ dv, float* __restrict__ dlog_std, float* __restrict__ loss_sums, const float* __restrict__ old_v,
    float* __restrict__ stats, DetSeq det) {
  __shared__ float scratch[32];
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  float l_actor = 0.f, l_v = 0.f, l_ent = 0.f, l_kl = 0.f, l_cf = 0.f, l_bkl = 0.f;
  float dls[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) dls[j] = 0.f;
  if (b < B) {
    const float lp = gaussian_logp(mu + (size_t)b * ld, log_std, actions + (size_t)b * A, A);
    float H = 0.f;
    for (int j = 0; j < A; ++j) H += 0.5f + kLogSqrt2PiL + logf(expf(log_std[j]));      // normal.py:114-115
    const float Ai = adv[b];
    float w;
    const float log_ratio = decoupled_log_ratio(lp, old_logp, b, hp, stats != nullptr, &w, &l_bkl);
    const float ratio = expf(log_ratio);
    float dterm;
    const float term = surrogate(ratio, Ai, hp, &dterm);
    l_actor = -(w * term) * hp.inv_B;
    if (stats) {
      l_kl = ((ratio - 1.f) - log_ratio) * hp.inv_B;
      l_cf = fabsf(ratio - 1.f) > hp.ppo_clip ? hp.inv_B : 0.f;
    }
    l_ent = H * hp.inv_B / (float)A;            // mean over all [B,A] elements
    const float w_lp = -hp.inv_B * (w * dterm) * ratio;
    for (int j = 0; j < A; ++j) {
      const float sd = expf(log_std[j]);
      const float var = sd * sd;
      const float z = actions[(size_t)b * A + j] - mu[(size_t)b * ld + j];
      dmu[(size_t)b * ld_d + j] = w_lp * (z / var);
      float g = w_lp * (z * z / var - 1.f);
      if (hp.shared) g += -hp.ent_coef * hp.inv_B / (float)A;
      if (j < 8) dls[j] = g;
    }
    float dl;
    l_v = value_loss_clipped(returns[b], v[b], old_v, b, hp.value_clip, hp.smooth_l1, hp.value_norm, &dl) * hp.inv_B;
    dv[b] = dl * hp.inv_B * (hp.shared ? hp.v_coef : 1.f);
  }
  l_actor = block_sum(l_actor, scratch);
  l_v = block_sum(l_v, scratch);
  l_ent = block_sum(l_ent, scratch);
  if (stats) {
    l_kl = block_sum(l_kl, scratch);
    l_cf = block_sum(l_cf, scratch);
    if (hp.prox) l_bkl = block_sum(l_bkl, scratch);
  }
  float tls[8];
  for (int j = 0; j < A && j < 8; ++j) tls[j] = block_sum(dls[j], scratch);
  if (threadIdx.x == 0) {
    if (det.ctr) det_enter(det.ctr, blockIdx.x);         // deterministic mode: the blocks add in block order
    det_add(det.ctr != nullptr, loss_sums + 0, l_actor);
    det_add(det.ctr != nullptr, loss_sums + 1, l_v);
    det_add(det.ctr != nullptr, loss_sums + 2, l_ent);
    if (stats) {
      det_add(det.ctr != nullptr, stats + 0, l_kl);
      det_add(det.ctr != nullptr, stats + 1, l_cf);
      if (hp.prox) det_add(det.ctr != nullptr, stats + 2, l_bkl);
    }
    for (int j = 0; j < A && j < 8; ++j) det_add(det.ctr != nullptr, dlog_std + j, tls[j]);
    if (det.ctr) det_leave(det.ctr, blockIdx.x, gridDim.x);
  }
}

// value loss of one extra critic head (nn/ppo.py:97-104)
__global__ void __launch_bounds__(128) value_loss_kernel(const float* __restrict__ returns, const float* __restrict__ v, int B,
                                                         LossParams hp, float* __restrict__ dv, float* __restrict__ loss_sums, DetSeq det) {
  __shared__ float scratch[32];
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  float l_v = 0.f;
  if (b < B) {
    float dl;
    l_v = value_loss(returns[b], v[b], hp.smooth_l1, &dl) * hp.inv_B;
    dv[b] = dl * hp.inv_B * (hp.shared ? hp.v_coef : 1.f);
  }
  l_v = block_sum(l_v, scratch);
  if (threadIdx.x == 0) {
    if (det.ctr) det_enter(det.ctr, blockIdx.x);
    det_add(det.ctr != nullptr, loss_sums + 1, l_v);
    if (det.ctr) det_leave(det.ctr, blockIdx.x, gridDim.x);
  }
}

// DECOUPLED_PPO pre-pass: out_logp[b] = log-prob of the taken action, bit-equal to the loss kernels' on the same logits / means
__global__ void __launch_bounds__(128) logp_actions_categorical_kernel(const float* __restrict__ logits, int ld,
                                                                       const float* __restrict__ actions, int B, int A,
                                                                       float* __restrict__ out_logp) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float p[kMaxAL];
  float s2;
  out_logp[b] = categorical_logp(logits + (size_t)b * ld, A, actions[b], p, &s2);
}

__global__ void __launch_bounds__(128) logp_actions_gaussian_kernel(const float* __restrict__ mu, int ld,
                                                                    const float* __restrict__ log_std,
                                                                    const float* __restrict__ actions, int B, int A,
                                                                    float* __restrict__ out_logp) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  out_logp[b] = gaussian_logp(mu + (size_t)b * ld, log_std, actions + (size_t)b * A, A);
}

static LossParams make_params(const ddrl_ppo_hparams* hp, float inv_B, int shared, const float* value_norm = nullptr,
                              const float* prox = nullptr, float is_clip = 0.f) {
  LossParams p;
  p.ppo_clip = hp->ppo_clip; p.dual_clip = hp->dual_clip; p.v_coef = hp->v_coef; p.ent_coef = hp->ent_coef;
  p.inv_B = inv_B; p.value_clip = hp->value_clip; p.smooth_l1 = hp->smooth_l1; p.shared = shared; p.value_norm = value_norm;
  p.prox = prox; p.is_clip = prox ? is_clip : 0.f;
  return p;
}

}  // namespace ddrl

using namespace ddrl;

// the value clip is on exactly when old_values is given, and then needs a width > 0
static bool value_clip_args_ok(const ddrl_ppo_hparams* hp, const float* old_values) {
  return old_values ? hp->value_clip > 0.f : !(hp->value_clip > 0.f);
}

extern "C" int ddrl_ppo_loss_categorical_dc(const float* logits, int ld, const float* actions, const float* old_logp,
                                            const float* adv, const float* returns, const float* v, int B, int A,
                                            float inv_B_global, const ddrl_ppo_hparams* hp, int shared, float* dlogits,
                                            int ld_d, float* dv, float* loss_sums, const float* old_values, float* stats,
                                            const float* value_norm, const float* prox_logp, float is_clip, void* stream) {
  if (B < 0 || A < 1 || A > kMaxAL || ld < A || ld_d < A || !hp) return DDRL_E_ARG;
  if (!value_clip_args_ok(hp, old_values)) return DDRL_E_ARG;
  if (B == 0) return DDRL_OK;
  if (!logits || !actions || !old_logp || !adv || !returns || !v || !dlogits || !dv || !loss_sums) return DDRL_E_ARG;
  ppo_loss_categorical_kernel<<<ceil_div(B, 128), 128, 0, (cudaStream_t)stream>>>(
      logits, ld, actions, old_logp, adv, returns, v, B, A, make_params(hp, inv_B_global, shared, value_norm, prox_logp, is_clip),
      dlogits, ld_d, dv, loss_sums, old_values, stats, det_seq(1));
  prof_work((8.0 * A + 24.0 + (old_values ? 4.0 : 0.0) + (prox_logp ? 4.0 : 0.0)) * B);
  DDRL_LAUNCHED("ppo_loss_categorical_kernel");
  return DDRL_OK;
}

extern "C" int ddrl_ppo_loss_categorical_vn(const float* logits, int ld, const float* actions, const float* old_logp,
                                            const float* adv, const float* returns, const float* v, int B, int A,
                                            float inv_B_global, const ddrl_ppo_hparams* hp, int shared, float* dlogits,
                                            int ld_d, float* dv, float* loss_sums, const float* old_values, float* stats,
                                            const float* value_norm, void* stream) {
  return ddrl_ppo_loss_categorical_dc(logits, ld, actions, old_logp, adv, returns, v, B, A, inv_B_global, hp, shared, dlogits,
                                      ld_d, dv, loss_sums, old_values, stats, value_norm, nullptr, 0.f, stream);
}

extern "C" int ddrl_ppo_loss_categorical_v(const float* logits, int ld, const float* actions, const float* old_logp,
                                           const float* adv, const float* returns, const float* v, int B, int A,
                                           float inv_B_global, const ddrl_ppo_hparams* hp, int shared, float* dlogits,
                                           int ld_d, float* dv, float* loss_sums, const float* old_values, float* stats,
                                           void* stream) {
  return ddrl_ppo_loss_categorical_vn(logits, ld, actions, old_logp, adv, returns, v, B, A, inv_B_global, hp, shared, dlogits,
                                      ld_d, dv, loss_sums, old_values, stats, nullptr, stream);
}

extern "C" int ddrl_ppo_loss_categorical(const float* logits, int ld, const float* actions, const float* old_logp,
                                         const float* adv, const float* returns, const float* v, int B, int A,
                                         float inv_B_global, const ddrl_ppo_hparams* hp, int shared, float* dlogits,
                                         int ld_d, float* dv, float* loss_sums, void* stream) {
  return ddrl_ppo_loss_categorical_v(logits, ld, actions, old_logp, adv, returns, v, B, A, inv_B_global, hp, shared, dlogits,
                                     ld_d, dv, loss_sums, nullptr, nullptr, stream);
}

extern "C" int ddrl_value_loss(const float* returns, const float* v, int B, float inv_B_global, const ddrl_ppo_hparams* hp,
                               int shared, float* dv, float* loss_sums, void* stream) {
  if (B < 0 || !hp) return DDRL_E_ARG;
  if (B == 0) return DDRL_OK;
  if (!returns || !v || !dv || !loss_sums) return DDRL_E_ARG;
  value_loss_kernel<<<ceil_div(B, 128), 128, 0, (cudaStream_t)stream>>>(returns, v, B, make_params(hp, inv_B_global, shared), dv,
                                                                         loss_sums, det_seq(1));
  prof_work(12.0 * B);
  DDRL_LAUNCHED("value_loss_kernel");
  return DDRL_OK;
}

extern "C" int ddrl_ppo_loss_gaussian_dc(const float* mu, int ld, const float* log_std, const float* actions,
                                         const float* old_logp, const float* adv, const float* returns, const float* v,
                                         int B, int A, float inv_B_global, const ddrl_ppo_hparams* hp, int shared,
                                         float* dmu, int ld_d, float* dv, float* dlog_std, float* loss_sums,
                                         const float* old_values, float* stats, const float* value_norm,
                                         const float* prox_logp, float is_clip, void* stream) {
  if (B < 0 || A < 1 || A > 8 || ld < A || ld_d < A || !hp) return DDRL_E_ARG;
  if (!value_clip_args_ok(hp, old_values)) return DDRL_E_ARG;
  if (B == 0) return DDRL_OK;
  if (!mu || !log_std || !actions || !old_logp || !adv || !returns || !v || !dmu || !dv || !dlog_std || !loss_sums)
    return DDRL_E_ARG;
  ppo_loss_gaussian_kernel<<<ceil_div(B, 128), 128, 0, (cudaStream_t)stream>>>(
      mu, ld, log_std, actions, old_logp, adv, returns, v, B, A, make_params(hp, inv_B_global, shared, value_norm, prox_logp, is_clip),
      dmu, ld_d, dv, dlog_std, loss_sums, old_values, stats, det_seq(1));
  prof_work((12.0 * A + 20.0 + (old_values ? 4.0 : 0.0) + (prox_logp ? 4.0 : 0.0)) * B);
  DDRL_LAUNCHED("ppo_loss_gaussian_kernel");
  return DDRL_OK;
}

extern "C" int ddrl_ppo_loss_gaussian_vn(const float* mu, int ld, const float* log_std, const float* actions,
                                         const float* old_logp, const float* adv, const float* returns, const float* v,
                                         int B, int A, float inv_B_global, const ddrl_ppo_hparams* hp, int shared,
                                         float* dmu, int ld_d, float* dv, float* dlog_std, float* loss_sums,
                                         const float* old_values, float* stats, const float* value_norm, void* stream) {
  return ddrl_ppo_loss_gaussian_dc(mu, ld, log_std, actions, old_logp, adv, returns, v, B, A, inv_B_global, hp, shared, dmu,
                                   ld_d, dv, dlog_std, loss_sums, old_values, stats, value_norm, nullptr, 0.f, stream);
}

extern "C" int ddrl_logp_actions_categorical(const float* logits, int ld, const float* actions, int B, int A, float* out_logp,
                                             void* stream) {
  if (B < 0 || A < 1 || A > kMaxAL || ld < A) return DDRL_E_ARG;
  if (B == 0) return DDRL_OK;
  if (!logits || !actions || !out_logp) return DDRL_E_ARG;
  logp_actions_categorical_kernel<<<ceil_div(B, 128), 128, 0, (cudaStream_t)stream>>>(logits, ld, actions, B, A, out_logp);
  prof_work((4.0 * A + 8.0) * B);
  DDRL_LAUNCHED("logp_actions_categorical_kernel");
  return DDRL_OK;
}

extern "C" int ddrl_logp_actions_gaussian(const float* mu, int ld, const float* log_std, const float* actions, int B, int A,
                                          float* out_logp, void* stream) {
  if (B < 0 || A < 1 || A > 8 || ld < A) return DDRL_E_ARG;
  if (B == 0) return DDRL_OK;
  if (!mu || !log_std || !actions || !out_logp) return DDRL_E_ARG;
  logp_actions_gaussian_kernel<<<ceil_div(B, 128), 128, 0, (cudaStream_t)stream>>>(mu, ld, log_std, actions, B, A, out_logp);
  prof_work((8.0 * A + 4.0) * B);
  DDRL_LAUNCHED("logp_actions_gaussian_kernel");
  return DDRL_OK;
}

extern "C" int ddrl_ppo_loss_gaussian_v(const float* mu, int ld, const float* log_std, const float* actions,
                                        const float* old_logp, const float* adv, const float* returns, const float* v,
                                        int B, int A, float inv_B_global, const ddrl_ppo_hparams* hp, int shared,
                                        float* dmu, int ld_d, float* dv, float* dlog_std, float* loss_sums,
                                        const float* old_values, float* stats, void* stream) {
  return ddrl_ppo_loss_gaussian_vn(mu, ld, log_std, actions, old_logp, adv, returns, v, B, A, inv_B_global, hp, shared, dmu,
                                   ld_d, dv, dlog_std, loss_sums, old_values, stats, nullptr, stream);
}

extern "C" int ddrl_ppo_loss_gaussian(const float* mu, int ld, const float* log_std, const float* actions,
                                      const float* old_logp, const float* adv, const float* returns, const float* v,
                                      int B, int A, float inv_B_global, const ddrl_ppo_hparams* hp, int shared,
                                      float* dmu, int ld_d, float* dv, float* dlog_std, float* loss_sums, void* stream) {
  return ddrl_ppo_loss_gaussian_v(mu, ld, log_std, actions, old_logp, adv, returns, v, B, A, inv_B_global, hp, shared, dmu,
                                  ld_d, dv, dlog_std, loss_sums, nullptr, nullptr, stream);
}
