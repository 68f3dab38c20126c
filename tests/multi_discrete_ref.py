"""TEST INFRASTRUCTURE ONLY -- float64 CPU restatement of the MultiDiscrete actor (MultiCategoricalActor), in plain torch on top
of the categorical restatement with the action mask (tests/action_mask_ref.py):

  head      logits [B, sum n]; branch i on the columns [o_i, o_i + n_i), o_i = n_1 + ... + n_{i-1}, with its own mask slice
  log-prob  sum over the branches of the categorical log-prob of the branch's action (actions [B, K])
  entropy   per row, the sum of the branch entropies (the entropy of the product distribution); EntLoss is its mean over rows

The PPO loss is the one of the other actors with every option (tests/beta_ref.losses); gradients come from autograd."""
import numpy as np
import torch
import torch.nn.functional as F

import action_mask_ref as M
import beta_ref as BR
from oracle import restate as R

Tensor = torch.Tensor


def slices(nvec):
    """[(o_i, o_i + n_i)] per branch."""
    out, o = [], 0
    for n in nvec:
        out.append((o, o + n))
        o += n
    return out


def _cut(mask, lo, hi):
    return None if mask is None else torch.as_tensor(mask)[:, lo:hi]


def effective_mask(mask, nvec) -> Tensor:
    """bool [B, sum n]: allowed actions, a branch slice that allows nothing taken as all-ones (per branch, not per row)."""
    return torch.cat([M.effective_mask(_cut(mask, lo, hi)) for lo, hi in slices(nvec)], -1)


def branch_probs(logits: Tensor, mask, nvec) -> Tensor:
    """The per-branch (masked) softmax, [B, sum n]."""
    return torch.cat([M.masked_probs(logits[:, lo:hi], _cut(mask, lo, hi)) for lo, hi in slices(nvec)], -1)


def log_prob(logits: Tensor, mask, actions: Tensor, nvec) -> Tensor:
    out = 0
    for i, (lo, hi) in enumerate(slices(nvec)):
        out = out + M.log_prob(logits[:, lo:hi], _cut(mask, lo, hi), actions[:, i])
    return out


def entropy(logits: Tensor, mask, nvec) -> Tensor:
    out = 0
    for lo, hi in slices(nvec):
        out = out + M.entropy(logits[:, lo:hi], _cut(mask, lo, hi))
    return out


def sample_on_q(q: np.ndarray, u: np.ndarray, mask, nvec) -> np.ndarray:
    """Per branch, the inverse CDF on the kernel's own fp32 q with u[:, i] (action_mask_ref.sample_on_q) -> int [B, K]."""
    B = q.shape[0]
    m = torch.ones(B, sum(nvec), dtype=torch.uint8) if mask is None else torch.as_tensor(mask)
    return np.stack([M.sample_on_q(q[:, lo:hi], u[:, i], m[:, lo:hi]) for i, (lo, hi) in enumerate(slices(nvec))], 1)


def first_max(p: np.ndarray, mask, nvec) -> np.ndarray:
    """Per branch, the first-max argmax over the allowed entries (play mode) -> int [B, K]."""
    eff = effective_mask(mask if mask is not None else torch.ones(p.shape[0], sum(nvec)), nvec).numpy()
    return np.stack([np.argmax(np.where(eff[:, lo:hi], p[:, lo:hi], -1.0), axis=1) for lo, hi in slices(nvec)], 1)


def sample(logits: Tensor, mask, nvec, generator) -> Tensor:
    """Random actions [B, K] (fp32) from the restated distribution."""
    p = branch_probs(logits.double(), mask, nvec)
    return torch.stack([torch.multinomial(p[:, lo:hi], 1, generator=generator).squeeze(-1) for lo, hi in slices(nvec)], 1).float()


def loss_and_grads(logits: Tensor, mask, actions: Tensor, nvec, old: Tensor, adv: Tensor, returns: Tensor, v: Tensor,
                   hp: R.PPOHyper, shared: bool, **options):
    """The fused MultiDiscrete loss kernel restated: ({actor, v, entropy, ApproxKL, ClipFrac[, BehaviourKL]}, d/d logits, d/d v).
    Shared: gradients of actor + v_coef * v - ent_coef * entropy; unshared: the logits' from the actor loss only, v's from the
    value loss only."""
    logits = logits.detach().double().clone().requires_grad_(True)
    v = v.detach().double().clone().requires_grad_(True)
    a, vl, ent, stats = BR.losses(log_prob(logits, mask, actions, nvec), entropy(logits, mask, nvec), v, old, adv, returns, hp,
                                  **options)
    if shared:
        (a + vl * hp.v_coef - ent * hp.ent_coef).backward()
    else:
        a.backward()
        vl.backward()
    out = {"actor": float(a.detach()), "v": float(vl.detach()), "entropy": float(ent.detach()), **stats}
    zero = lambda t: t.grad if t.grad is not None else torch.zeros_like(t)
    return out, zero(logits), zero(v)


def net_grads(spec: R.NetSpec, params, states, mask, actions: Tensor, nvec, old: Tensor, adv: Tensor, returns: Tensor,
              hp: R.PPOHyper = None):
    """Whole-net losses {ActorLoss, VLoss, EntLoss} and raw parameter gradients of one PPO step of a MultiDiscrete net, in
    float64, the encoders from oracle.restate.encoder_forward."""
    hp = hp or R.PPOHyper()
    p = {k: t.detach().double().clone().requires_grad_(True) for k, t in params.items()}
    st = [s.double() for s in states]
    if spec.shared:
        fa = fc = R.encoder_forward(spec.arch, p, "prenet.", st)
    else:
        fa = R.encoder_forward(spec.arch, p, "actor.pre.", st)
        fc = R.encoder_forward(spec.arch, p, "critic.pre.", st)
    logits = F.linear(fa, p["actor.actor_linear.weight"], p["actor.actor_linear.bias"])
    v = F.linear(fc, p["critic.critic_linear.weight"], p["critic.critic_linear.bias"]).squeeze(-1)
    a, vl, ent, _ = BR.losses(log_prob(logits, mask, actions, nvec), entropy(logits, mask, nvec), v, old, adv, returns, hp)
    if spec.shared:
        (a + vl * hp.v_coef - ent * hp.ent_coef).backward()
    else:
        a.backward()
        vl.backward()
    grads = {k: (q.grad if q.grad is not None else torch.zeros_like(q)) for k, q in p.items()}
    return {"ActorLoss": float(a.detach()), "VLoss": float(vl.detach()), "EntLoss": float(ent.detach())}, grads


def random_mask(B: int, nvec, seed: int, p_allowed: float = 0.6, empty_rows: int = 2) -> Tensor:
    """u8 [B, sum n] with ~p_allowed of the actions allowed; in the first `empty_rows` rows branch 0 allows nothing, and in the
    next `empty_rows` rows every branch allows nothing."""
    m = M.random_mask(B, sum(nvec), seed=seed, p_allowed=p_allowed, empty_rows=0)
    lo, hi = slices(nvec)[0]
    m[:empty_rows, lo:hi] = 0
    m[empty_rows:2 * empty_rows] = 0
    return m
