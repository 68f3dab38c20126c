"""Tensor-level wrappers over the C ABI (torch is only used for device memory and streams)."""
import ctypes as C
from typing import Optional, Sequence

import torch

from . import _lib
from ._lib import DDRLError, PPOHparams, check, current_stream, ptr, require_cuda


def make_hparams(ppo_clip=0.2, dual_clip=3.0, v_coef=1.0, ent_coef=0.05, max_grad_norm=0.5, clip_grad=True,
                 smooth_l1=False, lr=2e-4, lr_actor=5e-5, lr_critic=1e-3, beta1=0.9, beta2=0.999,
                 adam_eps=1e-8, value_clip=0.0, ppo_stats=False) -> PPOHparams:
    """Defaults = USTC_lab/config/config_nn.py:27-57 and torch.optim.Adam's; value_clip / ppo_stats are the non-reference
    VALUE_CLIP / PPO_STATS options (0 = off)."""
    return PPOHparams(ppo_clip, dual_clip, v_coef, ent_coef, max_grad_norm, int(bool(clip_grad)), int(bool(smooth_l1)),
                      lr, lr_actor, lr_critic, beta1, beta2, adam_eps, value_clip, int(bool(ppo_stats)))


def _f32c(t: torch.Tensor) -> torch.Tensor:
    require_cuda(t)
    if t.dtype != torch.float32 or not t.is_contiguous():
        t = t.to(torch.float32).contiguous()
    return t


def set_deterministic(on: bool = True) -> bool:
    """Run-to-run bit-reproducible gradients / losses on the default engine (ddrl_set_deterministic); returns the previous setting."""
    return bool(_lib.load().ddrl_set_deterministic(1 if on else 0))


def gae(values: torch.Tensor, rewards: torch.Tensor, dones: torch.Tensor, gamma: Sequence[float], lam: float,
        algo: int = 0):
    """values [T+1,V,N] f32, rewards [>=T,V,N] f32, dones [>=T,V,N] u8 -> (returns [T,V,N], advs [T,N]).
    Agents._accumulate_rewards (USTC_lab/agent/agent.py:124-140)."""
    lib = _lib.load()
    values = _f32c(values)
    rewards = _f32c(rewards)
    require_cuda(dones)
    if dones.dtype != torch.uint8 or not dones.is_contiguous():
        dones = dones.to(torch.uint8).contiguous()
    Tp1, V, N = values.shape
    T = Tp1 - 1
    assert rewards.shape[0] >= T and dones.shape[0] >= T and tuple(rewards.shape[1:]) == (V, N)
    ret = torch.empty((T, V, N), dtype=torch.float32, device=values.device)
    adv = torch.empty((T, N), dtype=torch.float32, device=values.device)
    gamma = [float(x) for x in gamma]
    if len(gamma) != V:
        raise DDRLError("gae: %d discounts for %d value rows (agent/agent.py:79 builds one per value row)" % (len(gamma), V))
    g = (C.c_float * V)(*gamma)
    check(lib.ddrl_gae_f32(ptr(values), ptr(rewards), ptr(dones), g, float(lam), T, V, N, ptr(ret), ptr(adv), algo,
                           current_stream()), "ddrl_gae_f32")
    return ret, adv


def gae_tempo(values: torch.Tensor, rewards: torch.Tensor, dones: torch.Tensor, durations: torch.Tensor, table,
              lam: float, out_f64: bool = True):
    """values [T+1,V,N] f32, rewards/dones [>=T,V,N], durations [>=T] int32, table [<=101] float64 (host)
    -> (returns [T,V,N], advs [T,N]) float64 (or float32).  Agents._accumulate_tempo_rewards (agent/agent.py:142-160)."""
    lib = _lib.load()
    values = _f32c(values)
    rewards = _f32c(rewards)
    require_cuda(dones)
    require_cuda(durations)
    if dones.dtype != torch.uint8 or not dones.is_contiguous():
        dones = dones.to(torch.uint8).contiguous()
    if durations.dtype != torch.int32 or not durations.is_contiguous():
        durations = durations.to(torch.int32).contiguous()
    Tp1, V, N = values.shape
    T = Tp1 - 1
    assert rewards.shape[0] >= T and dones.shape[0] >= T and durations.shape[0] >= T and tuple(rewards.shape[1:]) == (V, N)
    tab = [float(x) for x in table]
    assert 1 <= len(tab) <= 101
    if T > 0:
        # the reference indexes the table with the duration and raises IndexError outside it (agent/agent.py:151)
        lo, hi = int(durations[:T].min()), int(durations[:T].max())
        if lo < 0 or hi >= len(tab):
            raise IndexError("gae_tempo: durations span [%d, %d] but the discount table has %d entries" % (lo, hi, len(tab)))
    dt = torch.float64 if out_f64 else torch.float32
    ret = torch.empty((T, V, N), dtype=dt, device=values.device)
    adv = torch.empty((T, N), dtype=dt, device=values.device)
    check(lib.ddrl_gae_tempo(ptr(values), ptr(rewards), ptr(dones), ptr(durations), (C.c_double * len(tab))(*tab), len(tab),
                             C.c_double(float(lam)), T, V, N, ptr(ret), ptr(adv), int(out_f64), current_stream()),
          "ddrl_gae_tempo")
    return ret, adv


def sample_categorical_probs(probs: torch.Tensor, u: Optional[torch.Tensor]):
    """(probs [B,A], u [B] | None) -> (action [B] f32, logp [B] f32); server/utils.py:20-47."""
    lib = _lib.load()
    probs = _f32c(probs)
    B, A = probs.shape
    action = torch.empty(B, dtype=torch.float32, device=probs.device)
    logp = torch.empty(B, dtype=torch.float32, device=probs.device)
    if u is not None:
        u = _f32c(u)
    check(lib.ddrl_sample_categorical_probs(ptr(probs), A, ptr(u), B, A, ptr(action), ptr(logp), current_stream()),
          "ddrl_sample_categorical_probs")
    return action, logp


def categorical_head(logits: torch.Tensor, u: Optional[torch.Tensor], want_probs: bool = True):
    lib = _lib.load()
    logits = _f32c(logits)
    B, A = logits.shape
    action = torch.empty(B, dtype=torch.float32, device=logits.device)
    logp = torch.empty(B, dtype=torch.float32, device=logits.device)
    probs = torch.empty((B, A), dtype=torch.float32, device=logits.device) if want_probs else None
    if u is not None:
        u = _f32c(u)
    check(lib.ddrl_categorical_head(ptr(logits), A, ptr(u), B, A, ptr(action), ptr(logp), ptr(probs), current_stream()),
          "ddrl_categorical_head")
    return action, logp, probs


def categorical_head_m(logits: torch.Tensor, u: Optional[torch.Tensor], mask: Optional[torch.Tensor], want_probs: bool = True):
    """ddrl_categorical_head_m: categorical_head with the action mask [B, A] (any dtype, allowed iff != 0; None: no mask) ->
    (action [B], logp [B], the masked probs [B, A] or None)."""
    lib = _lib.load()
    logits = _f32c(logits)
    B, A = logits.shape
    mask = _mask_f32(mask, B, A)
    action = torch.empty(B, dtype=torch.float32, device=logits.device)
    logp = torch.empty(B, dtype=torch.float32, device=logits.device)
    probs = torch.empty((B, A), dtype=torch.float32, device=logits.device) if want_probs else None
    u = None if u is None else _f32c(u)
    check(lib.ddrl_categorical_head_m(ptr(logits), A, ptr(u), B, A, ptr(action), ptr(logp), ptr(probs), ptr(mask),
                                      current_stream()), "ddrl_categorical_head_m")
    return action, logp, probs


def _mask_f32(mask, B: int, A: int):
    """ACTION_MASK: the mask as the kernels read it, contiguous fp32 [B, A] (None stays None)."""
    if mask is None:
        return None
    mask = _f32c(mask)
    if mask.numel() != B * A:
        raise DDRLError("action mask has shape %s; expected [B=%d, A=%d]" % (tuple(mask.shape), B, A))
    return mask


def gaussian_head(mu: torch.Tensor, log_std: torch.Tensor, eps: Optional[torch.Tensor]):
    lib = _lib.load()
    mu = _f32c(mu)
    log_std = _f32c(log_std)
    B, A = mu.shape
    action = torch.empty((B, A), dtype=torch.float32, device=mu.device)
    logp = torch.empty(B, dtype=torch.float32, device=mu.device)
    if eps is not None:
        eps = _f32c(eps)
    check(lib.ddrl_gaussian_head(ptr(mu), A, ptr(log_std), ptr(eps), B, A, ptr(action), ptr(logp), current_stream()),
          "ddrl_gaussian_head")
    return action, logp


def ppo_loss_categorical(logits, actions, old_logp, adv, returns, v, hp: PPOHparams, shared: bool,
                         b_global: Optional[int] = None):
    """-> (dlogits [B,A], dv [B], loss_sums [4] = {actor, v, entropy, 0}); nn/ppo.py:85-108."""
    lib = _lib.load()
    logits, actions, old_logp, adv, returns, v = map(_f32c, (logits, actions, old_logp, adv, returns, v))
    B, A = logits.shape
    dlogits = torch.empty_like(logits)
    dv = torch.empty(B, dtype=torch.float32, device=logits.device)
    sums = torch.zeros(4, dtype=torch.float32, device=logits.device)
    check(lib.ddrl_ppo_loss_categorical(ptr(logits), A, ptr(actions), ptr(old_logp), ptr(adv), ptr(returns), ptr(v), B, A,
                                        1.0 / float(b_global or B), C.byref(hp), int(shared), ptr(dlogits), A, ptr(dv),
                                        ptr(sums), current_stream()), "ddrl_ppo_loss_categorical")
    return dlogits, dv, sums


def ppo_loss_gaussian(mu, log_std, actions, old_logp, adv, returns, v, hp: PPOHparams, shared: bool,
                      b_global: Optional[int] = None):
    """-> (dmu [B,A], dv [B], dlog_std [A], loss_sums [4])."""
    lib = _lib.load()
    mu, log_std, actions, old_logp, adv, returns, v = map(_f32c, (mu, log_std, actions, old_logp, adv, returns, v))
    B, A = mu.shape
    dmu = torch.empty_like(mu)
    dv = torch.empty(B, dtype=torch.float32, device=mu.device)
    dls = torch.zeros(A, dtype=torch.float32, device=mu.device)
    sums = torch.zeros(4, dtype=torch.float32, device=mu.device)
    check(lib.ddrl_ppo_loss_gaussian(ptr(mu), A, ptr(log_std), ptr(actions), ptr(old_logp), ptr(adv), ptr(returns), ptr(v),
                                     B, A, 1.0 / float(b_global or B), C.byref(hp), int(shared), ptr(dmu), A, ptr(dv),
                                     ptr(dls), ptr(sums), current_stream()), "ddrl_ppo_loss_gaussian")
    return dmu, dv, dls, sums


def ppo_loss_categorical_dc(logits, actions, old_logp, adv, returns, v, hp: PPOHparams, shared: bool, prox_logp=None,
                            is_clip: Optional[float] = None, b_global: Optional[int] = None):
    """The decoupled loss (ddrl_ppo_loss_categorical_dc) with the statistics on -> (dlogits [B,A], dv [B], sums [8]):
    sums[0..3) = {actor, v, entropy}, sums[3..6) = {approx KL, clip fraction, behaviour KL}.  prox_logp None: plain PPO."""
    lib = _lib.load()
    logits, actions, old_logp, adv, returns, v = map(_f32c, (logits, actions, old_logp, adv, returns, v))
    prox_logp = None if prox_logp is None else _f32c(prox_logp)
    B, A = logits.shape
    dlogits = torch.empty_like(logits)
    dv = torch.empty(B, dtype=torch.float32, device=logits.device)
    sums = torch.zeros(8, dtype=torch.float32, device=logits.device)
    check(lib.ddrl_ppo_loss_categorical_dc(ptr(logits), A, ptr(actions), ptr(old_logp), ptr(adv), ptr(returns), ptr(v), B, A,
                                           1.0 / float(b_global or B), C.byref(hp), int(shared), ptr(dlogits), A, ptr(dv),
                                           ptr(sums), None, ptr(sums[3:]), None, ptr(prox_logp), float(is_clip or 0.0),
                                           current_stream()), "ddrl_ppo_loss_categorical_dc")
    return dlogits, dv, sums


def ppo_loss_categorical_m(logits, actions, old_logp, adv, returns, v, hp: PPOHparams, shared: bool, mask=None, old_values=None,
                           value_norm=None, prox_logp=None, is_clip: Optional[float] = None, b_global: Optional[int] = None):
    """ddrl_ppo_loss_categorical_m with the statistics on -> (dlogits [B,A], dv [B], sums [8]), sums as ppo_loss_categorical_dc.
    mask [B, A] (ACTION_MASK; None: no mask), old_values (VALUE_CLIP; needs hp.value_clip > 0), value_norm (device {mean32,
    scale32, sigma32}) and prox_logp (DECOUPLED_PPO) are optional."""
    lib = _lib.load()
    logits, actions, old_logp, adv, returns, v = map(_f32c, (logits, actions, old_logp, adv, returns, v))
    old_values, value_norm, prox_logp = (None if t is None else _f32c(t) for t in (old_values, value_norm, prox_logp))
    B, A = logits.shape
    mask = _mask_f32(mask, B, A)
    dlogits = torch.empty_like(logits)
    dv = torch.empty(B, dtype=torch.float32, device=logits.device)
    sums = torch.zeros(8, dtype=torch.float32, device=logits.device)
    check(lib.ddrl_ppo_loss_categorical_m(ptr(logits), A, ptr(actions), ptr(old_logp), ptr(adv), ptr(returns), ptr(v), B, A,
                                          1.0 / float(b_global or B), C.byref(hp), int(shared), ptr(dlogits), A, ptr(dv),
                                          ptr(sums), ptr(old_values), ptr(sums[3:]), ptr(value_norm), ptr(prox_logp),
                                          float(is_clip or 0.0), ptr(mask), current_stream()), "ddrl_ppo_loss_categorical_m")
    return dlogits, dv, sums


def ppo_loss_gaussian_dc(mu, log_std, actions, old_logp, adv, returns, v, hp: PPOHparams, shared: bool, prox_logp=None,
                         is_clip: Optional[float] = None, b_global: Optional[int] = None):
    """The decoupled loss (ddrl_ppo_loss_gaussian_dc) with the statistics on -> (dmu [B,A], dv [B], dlog_std [A], sums [8]),
    sums as ppo_loss_categorical_dc."""
    lib = _lib.load()
    mu, log_std, actions, old_logp, adv, returns, v = map(_f32c, (mu, log_std, actions, old_logp, adv, returns, v))
    prox_logp = None if prox_logp is None else _f32c(prox_logp)
    B, A = mu.shape
    dmu = torch.empty_like(mu)
    dv = torch.empty(B, dtype=torch.float32, device=mu.device)
    dls = torch.zeros(A, dtype=torch.float32, device=mu.device)
    sums = torch.zeros(8, dtype=torch.float32, device=mu.device)
    check(lib.ddrl_ppo_loss_gaussian_dc(ptr(mu), A, ptr(log_std), ptr(actions), ptr(old_logp), ptr(adv), ptr(returns), ptr(v),
                                        B, A, 1.0 / float(b_global or B), C.byref(hp), int(shared), ptr(dmu), A, ptr(dv),
                                        ptr(dls), ptr(sums), None, ptr(sums[3:]), None, ptr(prox_logp), float(is_clip or 0.0),
                                        current_stream()), "ddrl_ppo_loss_gaussian_dc")
    return dmu, dv, dls, sums


def logp_actions_categorical(logits, actions) -> torch.Tensor:
    """Log-probs [B] of the taken actions under Categorical(logits), bit-equal to the loss kernel's."""
    logits, actions = _f32c(logits), _f32c(actions)
    B, A = logits.shape
    out = torch.empty(B, dtype=torch.float32, device=logits.device)
    check(_lib.load().ddrl_logp_actions_categorical(ptr(logits), A, ptr(actions), B, A, ptr(out), current_stream()),
          "ddrl_logp_actions_categorical")
    return out


def logp_actions_categorical_m(logits, actions, mask=None) -> torch.Tensor:
    """Log-probs [B] of the taken actions under the masked Categorical(logits) (mask [B, A] or None), bit-equal to the loss and
    head kernels'."""
    logits, actions = _f32c(logits), _f32c(actions)
    B, A = logits.shape
    mask = _mask_f32(mask, B, A)
    out = torch.empty(B, dtype=torch.float32, device=logits.device)
    check(_lib.load().ddrl_logp_actions_categorical_m(ptr(logits), A, ptr(actions), B, A, ptr(out), ptr(mask), current_stream()),
          "ddrl_logp_actions_categorical_m")
    return out


def logp_actions_gaussian(mu, log_std, actions) -> torch.Tensor:
    """Log-probs [B] of the action rows under Normal(mu, exp(log_std)) summed over A, bit-equal to the loss kernel's."""
    mu, log_std, actions = _f32c(mu), _f32c(log_std), _f32c(actions)
    B, A = mu.shape
    out = torch.empty(B, dtype=torch.float32, device=mu.device)
    check(_lib.load().ddrl_logp_actions_gaussian(ptr(mu), A, ptr(log_std), ptr(actions), B, A, ptr(out), current_stream()),
          "ddrl_logp_actions_gaussian")
    return out


def beta_head(head, low, high, u: Optional[torch.Tensor], want_conc: bool = True):
    """(head [B, 2A], low [A], high [A] device, u [B, A] uniforms | None = play mode) -> (action [B, A], logp [B], alpha | beta
    [B, 2A] or None); ddrl_beta_head."""
    head, low, high = _f32c(head), _f32c(low), _f32c(high)
    B, A2 = head.shape
    A = A2 // 2
    action = torch.empty((B, A), dtype=torch.float32, device=head.device)
    logp = torch.empty(B, dtype=torch.float32, device=head.device)
    conc = torch.empty((B, A2), dtype=torch.float32, device=head.device) if want_conc else None
    u = None if u is None else _f32c(u)
    check(_lib.load().ddrl_beta_head(ptr(head), A2, ptr(low), ptr(high), ptr(u), B, A, ptr(action), ptr(logp), ptr(conc),
                                     current_stream()), "ddrl_beta_head")
    return action, logp, conc


def ppo_loss_beta(head, low, high, actions, old_logp, adv, returns, v, hp: PPOHparams, shared: bool, old_values=None,
                  value_norm=None, prox_logp=None, is_clip: Optional[float] = None, b_global: Optional[int] = None):
    """ddrl_ppo_loss_beta with the statistics on -> (dhead [B, 2A], dv [B], sums [8]), sums as ppo_loss_categorical_dc.
    old_values (VALUE_CLIP; needs hp.value_clip > 0), value_norm (device {mean32, scale32, sigma32}) and prox_logp
    (DECOUPLED_PPO) are optional."""
    head, low, high, actions, old_logp, adv, returns, v = map(_f32c, (head, low, high, actions, old_logp, adv, returns, v))
    old_values, value_norm, prox_logp = (None if t is None else _f32c(t) for t in (old_values, value_norm, prox_logp))
    B, A2 = head.shape
    dhead = torch.empty_like(head)
    dv = torch.empty(B, dtype=torch.float32, device=head.device)
    sums = torch.zeros(8, dtype=torch.float32, device=head.device)
    check(_lib.load().ddrl_ppo_loss_beta(ptr(head), A2, ptr(low), ptr(high), ptr(actions), ptr(old_logp), ptr(adv), ptr(returns),
                                         ptr(v), B, A2 // 2, 1.0 / float(b_global or B), C.byref(hp), int(shared), ptr(dhead), A2,
                                         ptr(dv), ptr(sums), ptr(old_values), ptr(sums[3:]), ptr(value_norm), ptr(prox_logp),
                                         float(is_clip or 0.0), current_stream()), "ddrl_ppo_loss_beta")
    return dhead, dv, sums


def logp_actions_beta(head, low, high, actions) -> torch.Tensor:
    """Log-probs [B] of the action rows [B, A] under the Beta head [B, 2A], bit-equal to the loss and head kernels'."""
    head, low, high, actions = map(_f32c, (head, low, high, actions))
    B, A2 = head.shape
    out = torch.empty(B, dtype=torch.float32, device=head.device)
    check(_lib.load().ddrl_logp_actions_beta(ptr(head), A2, ptr(low), ptr(high), ptr(actions), B, A2 // 2, ptr(out),
                                             current_stream()), "ddrl_logp_actions_beta")
    return out


def _nvec_arg(nvec):
    """MultiDiscrete branch sizes -> (K, int32 host array); the C entry points validate them."""
    n = [int(x) for x in nvec]
    return len(n), (C.c_int32 * max(len(n), 1))(*n)


def multi_categorical_head(logits, nvec, u: Optional[torch.Tensor], mask=None, want_probs: bool = True):
    """ddrl_multi_categorical_head: (logits [B, sum n], branch sizes nvec, uniforms u [B, K] | None = play mode, mask [B, sum n] |
    None) -> (actions [B, K], logp [B], the per-branch probabilities [B, sum n] or None)."""
    logits = _f32c(logits)
    B, A = logits.shape
    K, arr = _nvec_arg(nvec)
    mask = _mask_f32(mask, B, A)
    action = torch.empty((B, K), dtype=torch.float32, device=logits.device)
    logp = torch.empty(B, dtype=torch.float32, device=logits.device)
    probs = torch.empty((B, A), dtype=torch.float32, device=logits.device) if want_probs else None
    u = None if u is None else _f32c(u)
    check(_lib.load().ddrl_multi_categorical_head(ptr(logits), A, ptr(u), B, K, arr, ptr(action), ptr(logp), ptr(probs), ptr(mask),
                                                  current_stream()), "ddrl_multi_categorical_head")
    return action, logp, probs


def ppo_loss_multi_categorical(logits, nvec, actions, old_logp, adv, returns, v, hp: PPOHparams, shared: bool, mask=None,
                               old_values=None, value_norm=None, prox_logp=None, is_clip: Optional[float] = None,
                               b_global: Optional[int] = None):
    """ddrl_ppo_loss_multi_categorical with the statistics on -> (dlogits [B, sum n], dv [B], sums [8]), sums as
    ppo_loss_categorical_dc; actions [B, K]; the options as ppo_loss_categorical_m."""
    logits, actions, old_logp, adv, returns, v = map(_f32c, (logits, actions, old_logp, adv, returns, v))
    old_values, value_norm, prox_logp = (None if t is None else _f32c(t) for t in (old_values, value_norm, prox_logp))
    B, A = logits.shape
    K, arr = _nvec_arg(nvec)
    mask = _mask_f32(mask, B, A)
    dlogits = torch.empty_like(logits)
    dv = torch.empty(B, dtype=torch.float32, device=logits.device)
    sums = torch.zeros(8, dtype=torch.float32, device=logits.device)
    check(_lib.load().ddrl_ppo_loss_multi_categorical(ptr(logits), A, ptr(actions), ptr(old_logp), ptr(adv), ptr(returns), ptr(v), B,
                                                      K, arr, 1.0 / float(b_global or B), C.byref(hp), int(shared), ptr(dlogits),
                                                      A, ptr(dv), ptr(sums), ptr(old_values), ptr(sums[3:]), ptr(value_norm),
                                                      ptr(prox_logp), float(is_clip or 0.0), ptr(mask), current_stream()),
          "ddrl_ppo_loss_multi_categorical")
    return dlogits, dv, sums


def logp_actions_multi_categorical(logits, nvec, actions, mask=None) -> torch.Tensor:
    """Log-probs [B] of the action rows [B, K] under the MultiDiscrete head (mask [B, sum n] or None), bit-equal to the loss and
    head kernels'."""
    logits, actions = _f32c(logits), _f32c(actions)
    B, A = logits.shape
    K, arr = _nvec_arg(nvec)
    mask = _mask_f32(mask, B, A)
    out = torch.empty(B, dtype=torch.float32, device=logits.device)
    check(_lib.load().ddrl_logp_actions_multi_categorical(ptr(logits), A, ptr(actions), B, K, arr, ptr(out), ptr(mask),
                                                          current_stream()), "ddrl_logp_actions_multi_categorical")
    return out


def net_log_prob(net, states, actions, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """ddrl_net_log_prob: log-probs [B] of `actions` under the current parameters of the PPO module `net`, for `states` as the
    engine takes them (already normalised under NORM_OBS); written into `out` when given."""
    net._ensure_engine()
    keep, arr, n_obs, B = net._obs_ptrs(states)
    actions = _f32c(actions.to(net._flat.device))
    if out is None:
        out = torch.empty(B, dtype=torch.float32, device=net._flat.device)
    check(_lib.load().ddrl_net_log_prob(net._h, arr, n_obs, B, ptr(actions), ptr(out), current_stream()), "ddrl_net_log_prob")
    return out


def clip_adam(params, grads, m, v, seg_begin: Sequence[int], seg_lr: Sequence[float], step: int, hp: PPOHparams):
    """In-place fused clip_grad_norm_ + Adam over flat fp32 buffers; returns the pre-clip norm (device scalar)."""
    lib = _lib.load()
    require_cuda(params, grads, m, v)
    n = params.numel()
    nseg = len(seg_lr)
    sb = (C.c_int64 * (nseg + 1))(*[int(x) for x in seg_begin])
    sl = (C.c_float * nseg)(*[float(x) for x in seg_lr])
    norm = torch.empty(1, dtype=torch.float32, device=params.device)
    check(lib.ddrl_clip_adam(ptr(params), ptr(grads), ptr(m), ptr(v), n, sb, sl, nseg, int(step), C.byref(hp), ptr(norm),
                             current_stream()), "ddrl_clip_adam")
    return norm


def gemm(form: int, A: torch.Tensor, B: torch.Tensor, bias: Optional[torch.Tensor] = None, act: int = 0,
         mode: str = "simt", out: Optional[torch.Tensor] = None, beta: int = 0):
    """form 0: A[M,K] B[N,K] ; form 1: A[M,K] B[K,N] ; form 2: A[K,M] B[K,N]  ->  C[M,N]."""
    lib = _lib.load()
    A, B = _f32c(A), _f32c(B)
    if form == 0:
        M, K = A.shape; N = B.shape[0]; assert B.shape[1] == K
    elif form == 1:
        M, K = A.shape; N = B.shape[1]; assert B.shape[0] == K
    else:
        K, M = A.shape; N = B.shape[1]; assert B.shape[0] == K
    if out is None:
        out = torch.empty((M, N), dtype=torch.float32, device=A.device)
    if bias is not None:
        bias = _f32c(bias)
    check(lib.ddrl_gemm_f32(_lib.GEMM_MODE[mode], form, M, N, K, ptr(A), A.stride(0), ptr(B), B.stride(0), ptr(out),
                            out.stride(0), ptr(bias), act, beta, current_stream()), "ddrl_gemm_f32")
    return out


def conv_nhwc(op: int, x, w, dy=None, bias=None, stride: int = 1, pad: int = 0, act: int = 0, mask=None, mode: str = "tc"):
    """Implicit-GEMM convolution on NHWC activations (ddrl_conv_nhwc_f32).  x [B,H,W,Cin] (or its shape as a tuple for
    op 1), w [Cout,Cin,KH,KW] reference layout.  op 0: forward -> [B,Ho,Wo,Cout]; op 1: data gradient of dy -> [B,H,W,Cin];
    op 2: weight gradient -> [Cout,Cin,KH,KW]."""
    lib = _lib.load()
    w = _f32c(w)
    Cout, Cin, KH, KW = w.shape
    B, H, W = (x.shape if torch.is_tensor(x) else x)[:3]
    conv1d = H == 1 and KH == 1
    Ho = 1 if conv1d else (H + 2 * pad - KH) // stride + 1
    Wo = (W + 2 * pad - KW) // stride + 1
    d = _lib.ConvDesc(B, H, W, Cin, Cout, KH, KW, stride, pad)
    dev = w.device
    if op == 0:
        out = torch.empty((B, Ho, Wo, Cout), dtype=torch.float32, device=dev)
    elif op == 1:
        out = torch.zeros((B, H, W, Cin), dtype=torch.float32, device=dev)
    else:
        out = torch.empty_like(w)
    xx = _f32c(x) if torch.is_tensor(x) else None
    dyy = _f32c(dy) if dy is not None else None
    bb = _f32c(bias) if bias is not None else None
    mm = _f32c(mask) if mask is not None else None
    check(lib.ddrl_conv_nhwc_f32(_lib.GEMM_MODE[mode], op, C.byref(d), ptr(xx), ptr(w), ptr(bb), ptr(dyy), act, ptr(mm), ptr(out), current_stream()),
          "ddrl_conv_nhwc_f32")
    return out


def gather_jobs(pairs, n_rows: int):
    """ddrl_gather_job array for `pairs` [(src, dst), ...]: a row is everything after dim 0 and must be contiguous; dst needs
    >= n_rows rows of the same size and dtype."""
    jobs = (_lib.GatherJob * max(len(pairs), 1))()
    for j, (src, dst) in enumerate(pairs):
        require_cuda(src, dst)
        if src.dtype != dst.dtype or src.device != dst.device:
            raise DDRLError("gather_rows: job %d mixes %s/%s with %s/%s" % (j, src.dtype, src.device, dst.dtype, dst.device))
        row = src[0].numel() if src.dim() > 1 else 1
        drow = dst[0].numel() if dst.dim() > 1 else 1
        contiguous = lambda t: t.dim() <= 1 or t[0:1].is_contiguous()
        if row != drow or dst.shape[0] < n_rows or not (contiguous(src) and contiguous(dst)):
            raise DDRLError("gather_rows: job %d has src %s / dst %s (rows must be contiguous and of one size, dst >= %d rows)"
                            % (j, tuple(src.shape), tuple(dst.shape), n_rows))
        es = src.element_size()
        jobs[j] = _lib.GatherJob(src.data_ptr() or None, dst.data_ptr() or None, row * es, src.stride(0) * es,
                                 dst.stride(0) * es, src.shape[0])
    return jobs


def gather_rows(rows: torch.Tensor, pairs) -> None:
    """dst[i] = src[rows[i]] for every (src, dst) in `pairs`, i < len(rows), in ONE launch (ddrl_gather_rows).  rows: int32
    device tensor; indices outside [0, len(src)) are clamped."""
    require_cuda(rows)
    if rows.dtype != torch.int32 or not rows.is_contiguous():
        raise DDRLError("gather_rows: rows must be a contiguous int32 tensor (got %s)" % rows.dtype)
    n = rows.numel()
    jobs = gather_jobs(pairs, n)
    check(_lib.load().ddrl_gather_rows(ptr(rows), n, jobs, len(pairs), current_stream()), "ddrl_gather_rows")


def adv_moments(adv: torch.Tensor, m3: Optional[torch.Tensor] = None) -> torch.Tensor:
    """{n, sum a, sum a^2} of the fp32 vector `adv` in float64 (ddrl_adv_moments), into `m3` [3] when given."""
    adv = _f32c(adv)
    if m3 is None:
        m3 = torch.empty(3, dtype=torch.float64, device=adv.device)
    if m3.dtype != torch.float64 or m3.numel() != 3 or not m3.is_contiguous() or m3.device != adv.device:
        raise DDRLError("adv_moments: m3 must be a contiguous float64 [3] tensor on %s" % adv.device)
    check(_lib.load().ddrl_adv_moments(ptr(adv), adv.numel(), ptr(m3), current_stream()), "ddrl_adv_moments")
    return m3


def adv_normalize(adv: torch.Tensor, m3: Optional[torch.Tensor] = None, eps: float = 1e-8,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(adv - mean) / (std + eps), std unbiased, over the moments `m3` (adv_moments, possibly summed over ranks) or over adv
    itself when m3 is None (ddrl_adv_normalize, one launch).  out may be adv (in place)."""
    require_cuda(adv)
    if adv.dtype != torch.float32 or not adv.is_contiguous():
        raise DDRLError("adv_normalize: adv must be a contiguous fp32 tensor")
    if out is None:
        out = torch.empty_like(adv)
    if out.dtype != torch.float32 or not out.is_contiguous() or out.numel() != adv.numel() or out.device != adv.device:
        raise DDRLError("adv_normalize: out must be a contiguous fp32 tensor shaped like adv")
    if m3 is not None and (m3.dtype != torch.float64 or m3.numel() != 3 or m3.device != adv.device):
        raise DDRLError("adv_normalize: m3 must be a float64 [3] tensor on %s" % adv.device)
    check(_lib.load().ddrl_adv_normalize(ptr(adv), adv.numel(), ptr(m3), float(eps), ptr(out), current_stream()),
          "ddrl_adv_normalize")
    return out


def _rows_of(x: torch.Tensor, D: int, what: str) -> int:
    """Rows of x read as a row-major [B, D] fp32 block."""
    require_cuda(x)
    if x.dtype != torch.float32 or not x.is_contiguous():
        raise DDRLError("%s: x must be a contiguous fp32 tensor" % what)
    B = x.shape[0] if x.dim() else 1
    if x.numel() != B * D:
        raise DDRLError("%s: x has shape %s; expected [B, %d elements/row]" % (what, tuple(x.shape), D))
    return B


def _f64_vec(t: torch.Tensor, n: int, dev, what: str):
    if t.dtype != torch.float64 or t.numel() != n or not t.is_contiguous() or t.device != dev:
        raise DDRLError("%s must be a contiguous float64 [%d] tensor on %s" % (what, n, dev))


def obs_moments(x: torch.Tensor, shift: torch.Tensor, sums: Optional[torch.Tensor] = None,
                ws: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Column sums {sum (x - shift), sum (x - shift)^2} of x read as [B, D] (D = shift.numel()), in float64, into `sums` [2D]
    (ddrl_obs_moments; bit-reproducible for given (B, D)).  ws: a byte workspace of at least obs_moments_ws_bytes(B, D), else
    one is allocated."""
    D = shift.numel()
    B = _rows_of(x, D, "obs_moments")
    _f64_vec(shift, D, x.device, "obs_moments: shift")
    if sums is None:
        sums = torch.empty(2 * D, dtype=torch.float64, device=x.device)
    _f64_vec(sums, 2 * D, x.device, "obs_moments: sums")
    need = obs_moments_ws_bytes(B, D)
    if need and (ws is None or ws.numel() * ws.element_size() < need):
        ws = torch.empty(need, dtype=torch.uint8, device=x.device)
    nbytes = ws.numel() * ws.element_size() if ws is not None else 0
    check(_lib.load().ddrl_obs_moments(ptr(x), B, D, ptr(shift), ptr(sums), ptr(ws), nbytes, current_stream()),
          "ddrl_obs_moments")
    return sums


def obs_moments_ws_bytes(B: int, D: int) -> int:
    return int(_lib.load().ddrl_obs_moments_ws_bytes(int(B), int(D)))


def obs_rms_update(mean: torch.Tensor, var: torch.Tensor, count: torch.Tensor, sums: Optional[torch.Tensor], n: float,
                   mean32: torch.Tensor, scale32: torch.Tensor) -> None:
    """Merges the batch of `n` rows whose moments (obs_moments around `mean`) are `sums` into the running float64 {mean, var,
    count} in place, then writes the applied form mean32 / scale32 (ddrl_obs_rms_update).  n = 0: the applied form only."""
    D = mean.numel()
    dev = mean.device
    require_cuda(mean)
    for t, k, what in ((mean, D, "mean"), (var, D, "var"), (count, 1, "count")):
        _f64_vec(t, k, dev, "obs_rms_update: " + what)
    if n > 0:
        _f64_vec(sums, 2 * D, dev, "obs_rms_update: sums")
    for t, what in ((mean32, "mean32"), (scale32, "scale32")):
        if t.dtype != torch.float32 or t.numel() != D or not t.is_contiguous() or t.device != dev:
            raise DDRLError("obs_rms_update: %s must be a contiguous fp32 [%d] tensor on %s" % (what, D, dev))
    check(_lib.load().ddrl_obs_rms_update(ptr(mean), ptr(var), ptr(count), ptr(sums) if n > 0 else None, float(n), D,
                                          ptr(mean32), ptr(scale32), current_stream()), "ddrl_obs_rms_update")


def value_norm_update(mean: torch.Tensor, var: torch.Tensor, count: torch.Tensor, sums: Optional[torch.Tensor], n: float,
                      applied: torch.Tensor, head_w: Optional[torch.Tensor] = None, head_b: Optional[torch.Tensor] = None) -> None:
    """NORM_VALUE (ddrl_value_norm_update, one launch): merges the batch of `n` return targets whose moments (obs_moments with
    D = 1 around `mean`) are `sums` into the float64 [1] {mean, var, count} in place, writes applied [3] = {mean32, scale32,
    sigma32}, and, given critic 0's head (fp32 weight [F] and bias [1], e.g. views into the flat parameter buffer), rescales it
    in place so that its unnormalised outputs are kept.  n = 0: the applied form only."""
    dev = mean.device
    require_cuda(mean)
    for t, what in ((mean, "mean"), (var, "var"), (count, "count")):
        _f64_vec(t, 1, dev, "value_norm_update: " + what)
    if n > 0:
        _f64_vec(sums, 2, dev, "value_norm_update: sums")
    if applied.dtype != torch.float32 or applied.numel() != 3 or not applied.is_contiguous() or applied.device != dev:
        raise DDRLError("value_norm_update: applied must be a contiguous fp32 [3] tensor on %s" % dev)
    if (head_w is None) != (head_b is None):
        raise DDRLError("value_norm_update: give both head_w and head_b, or neither")
    F = 0
    if head_w is not None:
        for t, k, what in ((head_w, head_w.numel(), "head_w"), (head_b, 1, "head_b")):
            if t.dtype != torch.float32 or t.numel() != k or k < 1 or not t.is_contiguous() or t.device != dev:
                raise DDRLError("value_norm_update: %s must be a contiguous fp32 tensor on %s (bias: one element)" % (what, dev))
        F = head_w.numel()
    check(_lib.load().ddrl_value_norm_update(ptr(mean), ptr(var), ptr(count), ptr(sums) if n > 0 else None, float(n), ptr(applied),
                                             ptr(head_w), ptr(head_b), F, current_stream()), "ddrl_value_norm_update")


def obs_normalize(x: torch.Tensor, mean32: torch.Tensor, scale32: torch.Tensor, clip: Optional[float],
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """clamp((x - mean32) * scale32, -clip, clip) per column of x read as [B, D] (D = mean32.numel()); clip None: no clamp
    (ddrl_obs_normalize, one launch).  out may be x (in place)."""
    D = mean32.numel()
    B = _rows_of(x, D, "obs_normalize")
    if out is None:
        out = torch.empty_like(x)
    if out.dtype != torch.float32 or not out.is_contiguous() or out.numel() != x.numel() or out.device != x.device:
        raise DDRLError("obs_normalize: out must be a contiguous fp32 tensor shaped like x")
    for t, what in ((mean32, "mean32"), (scale32, "scale32")):
        if t.dtype != torch.float32 or t.numel() != D or not t.is_contiguous() or t.device != x.device:
            raise DDRLError("obs_normalize: %s must be a contiguous fp32 [%d] tensor on %s" % (what, D, x.device))
    check(_lib.load().ddrl_obs_normalize(ptr(x), B, D, ptr(mean32), ptr(scale32), float(clip or 0.0), ptr(out),
                                         current_stream()), "ddrl_obs_normalize")
    return out


def launch_count() -> int:
    return int(_lib.load().ddrl_launch_count())


def launch_count_reset():
    _lib.load().ddrl_launch_count_reset()
