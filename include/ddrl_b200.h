/* ddrl_b200.h -- C ABI of the B200-native actor-learner hot path for DDRL4NAV.
 *
 * The reference (DRL-Navigation/DDRL4NAV) has no FFI: its "plugin API" for this path is
 * Python duck-typing (SURVEY.md section 8b).  Each entry point below names the reference
 * interface whose arithmetic it replaces (file:line relative to the reference root); the
 * Python mirror in ddrl4nav_b200/ binds them through ctypes and keeps the reference's
 * class / method names.  INTEGRATION.md shows the reference-side stub.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the comment says "host";
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing syncs;
 *   - return value: 0 = DDRL_OK, negative = error code (ddrl_error_string); never throws;
 *   - there is NO CPU fallback: without a CUDA device every compute call returns
 *     DDRL_E_CUDA (and the Python mirror raises).
 */
#ifndef DDRL_B200_H
#define DDRL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DDRL_OK 0
#define DDRL_E_ARG (-1)        /* bad argument (null pointer, shape, enum) */
#define DDRL_E_CUDA (-2)       /* CUDA runtime error (ddrl_last_cuda_error) */
#define DDRL_E_STATE (-3)      /* call order (e.g. learn before bind) */
#define DDRL_E_UNSUPPORTED (-4)
#define DDRL_E_NOMEM (-5)

enum ddrl_arch {               /* encoder family (USTC_lab/nn/__init__.py:12-18) */
  DDRL_ARCH_ATARI = 0,         /* AtariPreNet   nn/atari_encoder.py:11-32 */
  DDRL_ARCH_NAV = 1,           /* NavPreNet     nn/nav_encoder.py:12-43 */
  DDRL_ARCH_NAVPED = 2,        /* NavPedPreNet  nn/nav_encoder.py:46-79 */
  DDRL_ARCH_NAV1D = 3,         /* NavPreNet1D   nn/nav_encoder.py:82-128 */
  DDRL_ARCH_MLP = 4            /* MLPPreNet     nn/mlp_encoder.py:12-29 */
};
enum ddrl_dist { DDRL_DIST_CATEGORICAL = 0, DDRL_DIST_GAUSSIAN = 1 };   /* nn/actor.py:75,43 */
enum ddrl_gemm_mode {
  DDRL_GEMM_SIMT_F32 = 0,      /* CUDA-core fp32 FMA (reference / fallback-free baseline) */
  DDRL_GEMM_TC_3XTF32 = 1,     /* tcgen05 kind::tf32, hi/lo split in shared memory, one tile per CTA (gemm_tc.cu) */
  DDRL_GEMM_TC2_TMEM = 2,      /* same arithmetic; persistent CTAs, activation operand split into TMEM, weights
                                  pre-split per optimiser step (tc2.cu).  Shapes it does not take run on mode 1. */
  DDRL_GEMM_TC3_F16 = 3        /* tcgen05 kind::f16 on scaled fp16 hi / lo splits (22 significant bits, per-tensor power-of-two
                                  scale from a device-resident amax), 64-wide K blocks (tc3.cu).  Shapes it does not take
                                  run on mode 2. */
};

typedef struct ddrl_net ddrl_net;

typedef struct {
  int32_t arch;      /* enum ddrl_arch */
  int32_t in_ch;     /* AtariPreNet num_inputs / Nav* image_channel / MLP input_dim */
  int32_t act_dim;   /* ACTION_OUTPUT_DIM (config/config_nn.py:12-16) */
  int32_t dist;      /* enum ddrl_dist */
  int32_t shared;    /* SHARE_CNN_NET (config_nn.py:57; runner/utils.py:88-135) */
  int32_t feat;      /* AC_INPUT_DIM = 512 (MLP: last_output_dim) */
  int32_t gemm_mode; /* enum ddrl_gemm_mode */
  int32_t laser_ch;  /* DDRL_ARCH_NAV1D: channels of the laser observation; 0 or 1 = the reference's Conv1d(1, 32, 5, 2)
                      * (nn/nav_encoder.py:87); 3 = the non-reference "3 x 960" variant.  Other architectures: 0 */
} ddrl_net_desc;

typedef struct {     /* config/config_nn.py:27-57; torch.optim.Adam defaults */
  float ppo_clip;        /* PPO_CLIP 0.2 */
  float dual_clip;       /* DUEL_PPO_CLIP 3 */
  float v_coef;          /* V_LOSS_THETA 1.0 */
  float ent_coef;        /* ENTROPY_LOSS_THETA 0.05 */
  float max_grad_norm;   /* CLIP_GRID_NUM 0.5 */
  int32_t clip_grad;     /* CLIP_GRID */
  int32_t smooth_l1;     /* SMOOTH_L1_LOSS */
  float lr;              /* LEARNING_RATE (shared mode) */
  float lr_actor;        /* ACTOR_LEARNING_RATE */
  float lr_critic;       /* CRITIC_LEARNING_RATE */
  float beta1, beta2, adam_eps;
  /* non-reference PPO options (0 = off; appended so that a struct built from the fields above stays valid) */
  float value_clip;      /* VALUE_CLIP: clip width c > 0 of critic 0's value loss around the rollout's values (old_values) */
  int32_t ppo_stats;     /* PPO_STATS: the net's loss sums also accumulate the approx KL and the clip fraction */
} ddrl_ppo_hparams;

/* ---- library ------------------------------------------------------------------------- */
int ddrl_version(void);
const char* ddrl_error_string(int code);
const char* ddrl_last_cuda_error(void);
/* number of kernels this library has launched since load / since reset (bench gpu_launches) */
int64_t ddrl_launch_count(void);
void ddrl_launch_count_reset(void);
/* Deterministic mode (also DDRL_DETERMINISTIC=1 in the environment): every cross-block floating-point accumulation of the
 * default (tc3) path -- split-K weight gradients and the bias gradients fused into them, loss sums, the gradient norm, the
 * small-layer weight gradients -- adds its block partials in BLOCK ORDER instead of by unordered atomicAdd, so two runs on
 * the same inputs produce the same bits (the reference's CPU path is run-to-run deterministic, nn/ppo.py:108-129).  Costs a
 * few per cent (shorter reduction grids, serialised final adds).  Returns the previous setting. */
int ddrl_set_deterministic(int on);
/* per-kernel-class device timing for bench.py's roofline line: between start and stop every launch
 * on `stream` is followed by a CUDA event; stop writes "kernel_name ms launches work\n" lines
 * (work = algorithmic flops for GEMMs, bytes for the streaming kernels that declare them). */
int ddrl_prof_start(void* stream);
int ddrl_prof_stop(char* out, int cap);

/* ---- K5: GAE / discounted return scan -------------------------------------------------
 * replaces Agents._accumulate_rewards (USTC_lab/agent/agent.py:124-140).
 * values [T+1, V, N] f32 (row T = bootstrap), rewards [>=T, V, N] f32, dones [>=T, V, N] u8,
 * gamma_host [V] f32 HOST (self.discounts), lambda (self.landa).
 * out: ret [T, V, N] = values + g ; adv [T, N] = g of row v=0.
 * algo: 0 = auto (3, or 1 when T < 8); 1 = sequential per column and 4 = sequential, 2 columns per thread
 *       (both bit-exact with the numpy loop); 3 = single-pass time-parallel warp scan with the widest vector
 *       the shape allows (5 = scalar columns, 7 = 4 columns per thread: needs N % 4 == 0 and 16-byte aligned
 *       pointers, else DDRL_E_UNSUPPORTED); 2 = two-pass chunked warp scan.  2/3/5/7 reassociate only the
 *       carry-in of a time chunk (<= 1e-5 of max|adv|, measured 3e-7). */
int ddrl_gae_f32(const float* values, const float* rewards, const uint8_t* dones,
                 const float* gamma_host, float lambda, int T, int V, int N,
                 float* ret, float* adv, int algo, void* stream);

/* tempo-GAE: replaces Agents._accumulate_tempo_rewards (USTC_lab/agent/agent.py:142-160).
 * Per-step discount table_host[durations[t]] (table = self.tempo_discounts, float64 np.logspace(0,100,101,base=gamma),
 * agent.py:119; durations [>=T] int32 DEVICE = experiences[t].durations[0]).  The np.float64 table entry promotes the
 * reference's recurrence to float64; the kernel computes in float64 with the same operation order (bit-exact).
 * out_f64 != 0: ret [T,V,N] / adv [T,N] are double (the reference's arrays); 0: float (rounded once, what
 * Experience.to_tensor makes of them).  values / rewards / dones as for ddrl_gae_f32; lambda = self.landa. */
int ddrl_gae_tempo(const float* values, const float* rewards, const uint8_t* dones, const int* durations,
                   const double* table_host, int table_len, double lambda, int T, int V, int N,
                   void* ret, void* adv, int out_f64, void* stream);

/* ---- EasyBytes payload decode (SURVEY 8f, row f2) ----------------------------------------
 * replaces the decode half of EasyBytes.decode_forward_states / decode_data (USTC_lab/data/easybytes.py:47-61,114-139)
 * plus the fp32 conversion of the Forward thread (server/forward.py:128-131): slice + concatenate + dtype conversion of
 * the raw Redis payload in one kernel.  payload: the wire bytes on the DEVICE; segs: nseg DEVICE records
 * { uint64 src_off (bytes into payload); uint64 dst_off (floats into dst); uint32 count; uint32 dtype } with dtype the
 * wire code 1 = u8, 2 = f16, 3 = f32, 4 = f64 (easybytes.py:21-26); max_count = largest count (sizes the grid).
 * The host parses only the headers (ddrl4nav_b200/data/easybytes.py).  Conversions are exact / round-to-nearest-even,
 * i.e. bit-identical to numpy's astype(float32). */
int ddrl_easybytes_decode(const uint8_t* payload, const void* segs, int nseg, unsigned int max_count, float* dst,
                          void* stream);

/* Replies of one Forward tick, encoded on the device -- replaces EasyBytes.encode_forward_return_data
 * (USTC_lab/data/easybytes.py:77-109) for [actions, logps, values]: env process j gets the data blocks
 * actions[j*nb:(j+1)*nb] (fp32 [nb] when act_cols == 0, else [nb, act_cols]), logps[...] ([nb]) and
 * values[:, j*nb:(j+1)*nb] ([V, nb, 1]; values is [V, B] row-major).  out = n_env replies of
 * ddrl_easybytes_reply_bytes(nb, act_cols, V) bytes each, back to back (device buffer): one device->host copy, the host
 * cuts it per env process. */
int64_t ddrl_easybytes_reply_bytes(int nb, int act_cols, int V);
int ddrl_easybytes_encode_replies(const float* actions, int act_cols, const float* logps, const float* values, int V, int B,
                                  int n_env, int nb, uint8_t* out, void* stream);

/* ---- K4: action sampling --------------------------------------------------------------
 * replaces random_choice_prob_index / select_action (USTC_lab/server/utils.py:20-47) and the
 * sample/log_prob lines of ForwardThread.run (server/forward.py:137-146).
 * probs [B, A] (row stride ld), u [B] uniforms or NULL => play mode (first-max argmax, logp=0).
 * action[b] = first k with fl32(sum_{j<=k} p_j) > u[b], none => 0;  logp = log(p[b,action]). */
int ddrl_sample_categorical_probs(const float* probs, int ld, const float* u, int B, int A,
                                  float* action, float* logp, void* stream);
/* logits [B, A] (pre-softmax actor_linear output, nn/actor.py:91-98): softmax, Categorical
 * re-normalisation, inverse-CDF sample, logp = log(clamp(p/sum p, eps, 1-eps))[a].
 * probs_out may be NULL. */
int ddrl_categorical_head(const float* logits, int ld, const float* u, int B, int A,
                          float* action, float* logp, float* probs_out, void* stream);
/* Gaussian head (nn/actor.py:58-70): a = mu + exp(log_std)*eps (mul, then add);
 * logp = sum_j Normal(mu,std).log_prob(a); eps NULL => play mode (a = mu, logp = 0). */
int ddrl_gaussian_head(const float* mu, int ld, const float* log_std, const float* eps, int B, int A,
                       float* action, float* logp, void* stream);

/* ---- K6: fused PPO loss forward + backward --------------------------------------------
 * replaces nn/ppo.py:85-108 (+ the head part of autograd).  Per sample: dual-clip surrogate,
 * value loss, entropy; writes d(loss)/d(logits|mu) and d(loss)/d(v); accumulates
 * loss_sums[0..3] += {actor, v, entropy, -} contributions already scaled by inv_B_global and
 * (gaussian) dlog_std[A].  shared=1: gradients are of actor + v_coef*v - ent_coef*ent
 * (ppo.py:108-112); shared=0: dlogits from actor_loss only, dv from v_loss only (ppo.py:122-123).
 * actions are fp32 (categorical: integer-valued).  returns = data.values[0,:]. */
int ddrl_ppo_loss_categorical(const float* logits, int ld, const float* actions, const float* old_logp,
                              const float* adv, const float* returns, const float* v, int B, int A,
                              float inv_B_global, const ddrl_ppo_hparams* hp, int shared,
                              float* dlogits, int ld_d, float* dv, float* loss_sums, void* stream);
int ddrl_ppo_loss_gaussian(const float* mu, int ld, const float* log_std, const float* actions,
                           const float* old_logp, const float* adv, const float* returns, const float* v,
                           int B, int A, float inv_B_global, const ddrl_ppo_hparams* hp, int shared,
                           float* dmu, int ld_d, float* dv, float* dlog_std, float* loss_sums, void* stream);
/* The same with the non-reference options.  old_values [B] (rollout values of critic 0) or NULL: when given, critic 0's value
 * loss is clipped, v_c = old_values + clamp(v - old_values, -hp->value_clip, hp->value_clip) and loss = max(vloss(R, v),
 * vloss(R, v_c)) per row (clamp's gradient passes on the closed interval, ties of max split 1/2-1/2); it must be given exactly
 * when hp->value_clip > 0 (else DDRL_E_ARG).  stats (2 floats) or NULL: stats[0] += inv_B_global * sum((r - 1) - log r)
 * (approx KL) and stats[1] += inv_B_global * #{|r - 1| > hp->ppo_clip} (clip fraction), r = this pass's ratio.  With both
 * NULL these are the calls above, which write nothing past loss_sums[2]. */
int ddrl_ppo_loss_categorical_v(const float* logits, int ld, const float* actions, const float* old_logp,
                                const float* adv, const float* returns, const float* v, int B, int A,
                                float inv_B_global, const ddrl_ppo_hparams* hp, int shared,
                                float* dlogits, int ld_d, float* dv, float* loss_sums, const float* old_values, float* stats,
                                void* stream);
int ddrl_ppo_loss_gaussian_v(const float* mu, int ld, const float* log_std, const float* actions,
                             const float* old_logp, const float* adv, const float* returns, const float* v,
                             int B, int A, float inv_B_global, const ddrl_ppo_hparams* hp, int shared,
                             float* dmu, int ld_d, float* dv, float* dlog_std, float* loss_sums, const float* old_values,
                             float* stats, void* stream);

/* ---- advantage normalisation (non-reference option NORM_ADV) -------------------------------
 * ddrl_adv_moments: m3[0..2] = {n, sum a, sum a^2} of adv[0..n) in fp64 (m3: DEVICE, 3 doubles); a data-parallel learner sums
 * them over the ranks.  ddrl_adv_normalize: out[i] = (adv[i] - mean) / (std + eps) with std the unbiased standard deviation of
 * the moments m3, or of adv[0..n) itself when m3 is NULL (one launch); a moment count <= 1 copies adv unchanged.  Both run as
 * ONE block with a fixed reduction order, so their results are bit-reproducible without deterministic mode, and both can be
 * captured in a graph.  out may be adv. */
int ddrl_adv_moments(const float* adv, int n, double* m3, void* stream);
int ddrl_adv_normalize(const float* adv, int n, const double* m3, float eps, float* out, void* stream);

/* ---- running observation normalisation (non-reference option NORM_OBS) ---------------------
 * ddrl_obs_moments: sums[0..D) = column sums of d = x - shift and sums[D..2D) = column sums of d^2, in fp64, over the row-major
 * fp32 x [B, D] (shift, sums: DEVICE doubles).  Rows are cut into fixed chunks whose partials go to `ws` (at least
 * ddrl_obs_moments_ws_bytes(B, D) bytes; 0 when one chunk covers B, and ws may then be NULL), then a second launch adds them in
 * chunk order: the result depends on (B, D) only, so it is bit-reproducible run to run, rank to rank and device to device.
 * ddrl_obs_rms_update: Chan's merge of the batch {n, mean = shift + S1/n, var = S2/n - (S1/n)^2} into the running {mean [D],
 * var [D], count [1]} (fp64, DEVICE; shift = the running mean the sums were taken around), then the applied form
 * mean32 = fp32(mean), scale32 = fp32(1 / sqrt(var + 1e-8)); n = 0 rewrites only the applied form (sums may be NULL).
 * ddrl_obs_normalize: out = min(max((x - mean32) * scale32, -clip), clip) per column, each operation rounded on its own; clip <= 0
 * means no clamp.  out may be x. */
int64_t ddrl_obs_moments_ws_bytes(int B, int D);
int ddrl_obs_moments(const float* x, int B, int D, const double* shift, double* sums, void* ws, int64_t ws_bytes, void* stream);
int ddrl_obs_rms_update(double* mean, double* var, double* count, const double* sums, double n, int D, float* mean32,
                        float* scale32, void* stream);
int ddrl_obs_normalize(const float* x, int B, int D, const float* mean32, const float* scale32, float clip, float* out,
                       void* stream);

/* Value loss of ONE extra critic head (nn/ppo.py:97-104: rndv_loss / gailv_loss = vlossf(data.values[k], values[k])):
 * dv[b] = d(loss)/d(v[b]) (times v_coef when shared, ppo.py:108), loss_sums[1] += contribution scaled by inv_B_global. */
int ddrl_value_loss(const float* returns, const float* v, int B, float inv_B_global, const ddrl_ppo_hparams* hp,
                    int shared, float* dv, float* loss_sums, void* stream);

/* ---- K7: fused global-norm clip + Adam ------------------------------------------------
 * replaces torch.nn.utils.clip_grad_norm_ (nn/ppo.py:115,126) and torch.optim.Adam.step
 * (ppo.py:117,128-129).  Flat buffers of n floats; segment s covers [seg_begin[s], seg_begin[s+1])
 * with learning rate seg_lr[s] (host arrays, nseg+1 / nseg entries).  step >= 1 (same for all).
 * norm_out (device, 1 float, may be NULL) receives the pre-clip global L2 norm. */
int ddrl_clip_adam(float* params, float* grads, float* m, float* v, int64_t n,
                   const int64_t* seg_begin_host, const float* seg_lr_host, int nseg,
                   int step, const ddrl_ppo_hparams* hp, float* norm_out, void* stream);

/* ---- GEMM building block (exposed for parity tests / roofline benches) ------------------
 * C[M,N] (ldc) = act( A op B + bias ), fp32 in/out.
 *  form 0 "fwd"  : C[m,n] = sum_k A[m*lda+k] * B[n*ldb+k]            (A [M,K], B [N,K])
 *  form 1 "dgrad": C[m,n] = sum_k A[m*lda+k] * B[k*ldb+n]            (A [M,K], B [K,N])
 *  form 2 "wgrad": C[m,n] = sum_k A[k*lda+m] * B[k*ldb+n]            (A [K,M], B [K,N])
 * bias: NULL or [N]; act: 0 none, 1 relu, 2 leaky_relu(0.01); beta: 0 overwrite, 1 accumulate into C.
 * mode: enum ddrl_gemm_mode (mode 2 takes beta = 1 only for form 2 and splits B on the fly). */
int ddrl_gemm_f32(int mode, int form, int M, int N, int K, const float* A, int lda, const float* B, int ldb,
                  float* C, int ldc, const float* bias, int act, int beta, void* stream);

/* ---- convolution building block (implicit GEMM; exposed for parity tests) ----------------
 * The conv layers of the encoders (nn.Conv2d / nn.Conv1d + autograd in nn/atari_encoder.py:16-28,
 * nn/nav_encoder.py:17-31,85-93) on NHWC activations, with the activation operand fetched tap by
 * tap through 4-D TMA boxes (no im2col matrix in memory).  w / dw use the reference's OIHW layout.
 *  op 0: out[B,Ho,Wo,Cout] = act( conv(x[B,H,W,Cin], w) + bias )                act 0/1/2 as ddrl_gemm_f32
 *  op 1: out[B,H,W,Cin]    = conv_transpose(dy[B,Ho,Wo,Cout], w) * act'(mask)   act 0 none, 3 relu', 4 leaky'
 *                            (mask [B,H,W,Cin] = the forward activation whose derivative is applied)
 *  op 2: out[Cout,Cin,KH,KW] = sum_pixels dy (x) x                              (weight gradient)
 * H == 1 && KH == 1 describes a Conv1d over W.  Needs Cin % 32 == 0 (op 0, 2) / Cout % 32 == 0 (op 1);
 * other shapes return DDRL_E_UNSUPPORTED (the engine keeps those layers on explicit im2col). */
typedef struct {
  int32_t B, H, W, Cin, Cout, KH, KW, stride, pad;
} ddrl_conv_desc;
int ddrl_conv_nhwc_f32(int mode /* 1 or 2: enum ddrl_gemm_mode */, int op, const ddrl_conv_desc* d, const float* x, const float* w, const float* bias,
                       const float* dy, int act, const float* mask, float* out, void* stream);

/* ---- the actor-critic net ---------------------------------------------------------------
 * replaces PPO.forward / PPO.learn and the classes they are built from
 * (nn/ppo.py:17-146, nn/actor.py, nn/critic.py, nn/atari_encoder.py, nn/nav_encoder.py,
 * nn/mlp_encoder.py; construction order runner/utils.py:59-170). */
int ddrl_net_create(const ddrl_net_desc* desc, ddrl_net** out);
int ddrl_net_destroy(ddrl_net* net);
/* parameter table in the reference's named_parameters() order */
int ddrl_net_num_tensors(const ddrl_net* net);
int64_t ddrl_net_num_params(const ddrl_net* net);
int ddrl_net_tensor_info(const ddrl_net* net, int i, char* name, int name_cap,
                         int64_t* shape4, int* ndim, int64_t* offset);
/* flat device buffers (reference layout/order).  grads has num_params + 8 floats: the tail
 * [P .. P+3] carries {actor, v, entropy, unused} loss sums so one all-reduce covers both; with hp->ppo_stats the backward
 * passes write [P .. P+4] = {actor, v, entropy, approx-KL, clip-fraction} sums.
 * grads/m/v may be NULL for an inference-only net. */
int ddrl_net_bind(ddrl_net* net, float* params, float* grads, float* adam_m, float* adam_v);
/* Extra value heads (nn/ppo.py:63-64 `add_critic`, :75 `[critic(states) for critic in self._critics]`, :95-105 the V > 1
 * value losses; agent/agent.py:96-108 value_dim_num): `count` (<= 2, "suppose 3 critic net at most", ppo.py:93) Critic
 * heads WITHOUT an encoder of their own (share-CNN mode: runner/utils.py:162 deepcopy(critic)) reading the shared feature.
 * w[k] [feat] and b[k] [1] are device pointers OUTSIDE the flat parameter buffer -- the reference's optimisers are built
 * before add_critic (ppo.py:40-42) and never step them; dw[k] / db[k] receive their gradients (+=, the caller zeroes).
 * While extras are set, ddrl_net_forward writes `values` as [1+count, B] (row stride B) and ddrl_net_backward reads
 * `returns` as [1+count, B_local] (row k = data.values[k]); in_loss[k] != 0 adds vlossf(values[k+1]) to the value loss
 * (gail_critic, ppo.py:101-104) and its gradient to the shared encoder.  Unshared nets: DDRL_E_UNSUPPORTED (an extra critic
 * with its own encoder is a net of its own -- ddrl4nav_b200/nn/ppo.py builds one).  count = 0 clears. */
int ddrl_net_set_extra_critics(ddrl_net* net, int count, const float* const* w, const float* const* b,
                               float* const* dw, float* const* db, const int* in_loss);
/* tell the net the flat params were changed behind its back (load_state_dict, updatenn_by_redis) */
int ddrl_net_params_changed(ddrl_net* net);
/* number of observation slots and per-sample element count of each (for argument checking) */
int ddrl_net_num_obs(const ddrl_net* net);
int64_t ddrl_net_obs_elems(const ddrl_net* net, int slot);

/* Forward module compute body (server/forward.py:128-146): obs[i] fp32 device [B, ...] in the
 * reference's NCHW/state-list order; draw = uniforms [B] (categorical) or N(0,1) [B,A]
 * (gaussian), NULL => play mode.  Outputs: actions [B] or [B,A]; logp [B]; values [B] (the
 * caller views it as [V=1,B,1]); pi_out (optional) probs [B,A] or mu [B,A]. */
int ddrl_net_forward(ddrl_net* net, const float* const* obs, int n_obs, int B, const float* draw,
                     float* actions, float* logp, float* values, float* pi_out, void* stream);

/* Stand-alone encoder forward: features [B, feat] of tower `tower` (0 = prenet / actor.pre, 1 = critic.pre) for the
 * observations obs[] -- replaces AtariPreNet.forward (nn/atari_encoder.py:25-32), NavPreNet / NavPedPreNet.forward
 * (nn/nav_encoder.py:35-43,66-79), NavPreNet1D.forward (nav_encoder.py:115-128), MLPPreNet.forward
 * (nn/mlp_encoder.py:24-29).  out: fp32 device [B, feat]. */
int ddrl_net_encode(ddrl_net* net, const float* const* obs, int n_obs, int B, int tower, float* out, void* stream);

/* One learn iteration, first half (nn/ppo.py:82-123): forward with act=data.actions, fused loss,
 * backward through heads and encoders.  Leaves d(loss)/d(params) for the LOCAL B rows, scaled
 * by 1/B_global, in the flat grads buffer and the loss sums in its tail.  In a data-parallel
 * learner the caller all-reduces grads[0 .. P+4) (sum; [0 .. P+5) with hp->ppo_stats) before ddrl_net_clip_adam.
 * obs_unchanged != 0: the caller guarantees obs[] hold the same bytes as in the previous backward call
 * (iterations 2..10 of PPO.learn); observation-side staging is then reused. */
int ddrl_net_backward(ddrl_net* net, const float* const* obs, int n_obs, int B_local, int B_global,
                      const float* actions, const float* old_logp, const float* adv, const float* returns,
                      const ddrl_ppo_hparams* hp, int obs_unchanged, void* stream);
/* ddrl_net_backward with old_values [B_local] (critic 0's rollout values) for hp->value_clip > 0 (ddrl_ppo_loss_*_v); NULL
 * otherwise.  hp->value_clip > 0 with old_values NULL returns DDRL_E_ARG.  ddrl_net_backward passes NULL. */
int ddrl_net_backward_v(ddrl_net* net, const float* const* obs, int n_obs, int B_local, int B_global,
                        const float* actions, const float* old_logp, const float* adv, const float* returns,
                        const float* old_values, const ddrl_ppo_hparams* hp, int obs_unchanged, void* stream);
/* The same pass in SEGMENTS, for a data-parallel learner that overlaps the gradient all-reduce with the rest of the
 * backward (nn/ppo.py:113-123 runs the actor and the critic backward one after the other; server/backward.py:167 "TODO multi
 * GPU").  Call with segment = 0, 1, ..., *n_segments - 1 in order and the SAME arguments; after segment k returns (stream
 * order), every parameter tensor i with ddrl_net_tensor_segment(net, i) == k holds its final gradient in the flat buffer
 * and may be reduced on another stream while segment k + 1 runs.  A pass that cannot be cut (first iteration of a learn
 * call, micro-batched rows, extra critics) runs whole in segment 0 and reports *n_segments = 1. */
/* The segmented pass takes no old_values: hp->value_clip > 0 returns DDRL_E_ARG. */
int ddrl_net_backward_segment(ddrl_net* net, const float* const* obs, int n_obs, int B_local, int B_global,
                              const float* actions, const float* old_logp, const float* adv, const float* returns,
                              const ddrl_ppo_hparams* hp, int obs_unchanged, int segment, int* n_segments, void* stream);
int ddrl_net_tensor_segment(const ddrl_net* net, int index);
/* Gradient all-reduce (sum) of a data-parallel learner over NVLink / NVSwitch peer memory, as ONE kernel of this library
 * (the reference is single-device: server/backward.py:167 "TODO multi GPU"; nn/ppo.py:113-129 is the step it feeds).
 * peer_bufs[p]: rank p's buffer as mapped into THIS process (peer_bufs[rank] = the local one); multicast_buf: the NVSwitch
 * multicast address of the same buffers, or NULL (plain peer loads / stores); peer_flags[p]: rank p's barrier-flag block
 * (ddrl_peer_allreduce_flag_bytes() bytes, zeroed once, used by nothing else).  Reduces elements [offset, offset + count)
 * (both multiples of 4) in place on every rank: rank r owns slice r, reduces it once and stores the result to all ranks,
 * so replicas hold identical bits.  seq: strictly increasing per call (> 0), identical on all ranks.  Every rank of the
 * group must make the same call; the kernel spins until its peers arrive. */
int ddrl_peer_allreduce_flag_bytes(void);
int ddrl_peer_allreduce_f32(float* const* peer_bufs, float* multicast_buf, void* const* peer_flags, int rank, int world,
                            int64_t offset, int64_t count, uint32_t seq, void* stream);
/* Multi-tensor row gather (minibatch PPO epochs, nn/ppo.py learn with MINI_BATCH_NUM > 1): for every job, dst row i =
 * src row rows[i] (i < n_rows), all jobs in ONE launch.  Strides and row_bytes are in bytes; row_bytes, strides and
 * pointers must be multiples of 4 (16 everywhere selects 16-byte accesses).  Indices outside [0, src_rows) are clamped.
 * rows: device int32 [n_rows].  jobs: HOST array of n_jobs (1..DDRL_GATHER_MAX_JOBS) descriptors, passed to the kernel by
 * value (no host->device copy; the launch can be captured in a CUDA graph). */
#define DDRL_GATHER_MAX_JOBS 12
typedef struct {
  const void* src;
  void* dst;
  int64_t row_bytes;
  int64_t src_stride;
  int64_t dst_stride;
  int64_t src_rows;
} ddrl_gather_job;
int ddrl_gather_rows(const int32_t* rows, int n_rows, const ddrl_gather_job* jobs, int n_jobs, void* stream);
/* ddrl_net_backward for one minibatch of a minibatch epoch: the inputs sit at the same addresses as in an earlier call of
 * this entry point and hold NEW rows.  The pass always restages the observations.  From the second call with the same
 * arguments on, it replays a CUDA graph captured for them (micro-batched rows, extra critics and DDRL_NO_GRAPH=1 run on the
 * stream).  A failed capture here leaves the graphs of ddrl_net_backward / ddrl_net_clip_adam on. */
int ddrl_net_backward_minibatch(ddrl_net* net, const float* const* obs, int n_obs, int B_local, int B_global,
                                const float* actions, const float* old_logp, const float* adv, const float* returns,
                                const ddrl_ppo_hparams* hp, void* stream);
/* ddrl_net_backward_minibatch with old_values, as ddrl_net_backward_v. */
int ddrl_net_backward_minibatch_v(ddrl_net* net, const float* const* obs, int n_obs, int B_local, int B_global,
                                  const float* actions, const float* old_logp, const float* adv, const float* returns,
                                  const float* old_values, const ddrl_ppo_hparams* hp, void* stream);
/* second half (nn/ppo.py:115-129): global-norm clip + the two (or one) Adam steps; then refreshes
 * the packed weights.  loss4_out (device, 4 floats, optional) = {total, actor, v, entropy}; with hp->ppo_stats it must
 * hold 6 floats and receives {total, actor, v, entropy, approx KL, clip fraction}. */
int ddrl_net_clip_adam(ddrl_net* net, int step, const ddrl_ppo_hparams* hp, float* loss4_out, void* stream);
/* bytes of device workspace currently held */
int64_t ddrl_net_workspace_bytes(const ddrl_net* net);

#ifdef __cplusplus
}
#endif
#endif /* DDRL_B200_H */
