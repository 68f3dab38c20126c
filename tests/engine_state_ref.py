"""References for the engine after parameter updates (tests/test_gpu_engine_state.py, tests/test_gpu_net.py).

* ``grads_match_oracle``: the engine's raw gradients against an oracle pass, within 2e-5 of each tensor's max, a residual
  beyond that explained exactly by ties: pre-activations that are zero to fp32 rounding take either relu branch, and a 2 x 2
  max-pool window whose two largest activations agree to fp32 rounding may send its gradient to either.
* ``clip_adam_step``: one float64 global-norm clip + Adam step (torch.nn.utils.clip_grad_norm_ + torch.optim.Adam,
  capturable=False), with one learning rate per element, so both LR segments of an unshared net are one call.  The betas
  are the fp32 values the engine's hyper-parameter block holds (ddrl_ppo_hparams): 1 - fp32(0.999) is 1.3e-5 away from
  0.001, more than the tolerance on v.
* ``adam_mismatch``: the engine's p, m, v after one step against that reference, in the tolerance form of
  test_gpu_kernels.py::test_clip_adam_vs_torch (fp32 results: a few ulps of each element on top of 1e-5 of the tensor's max).
  Only the m and v checks see a wrong gradient: a gradient off by 1e-3 moves the Adam delta by less than the p tolerance.
"""
import math

import torch
import torch.nn.functional as F

from oracle import restate as R

GRAD_BOUND = 2e-5    # engine gradient vs oracle, of the tensor's max (DESIGN section 3)
TIE_EPS = 1e-6       # an activation with |z| < TIE_EPS * max|z| of its layer is zero to within fp32 rounding: a tie


class PoolRecorder:
    """R.POOL_HOOK: 2 x 2 max pools that record, per window, the gap between the two largest activations, and route the gradient
    of the windows `flips` = {"pool:" + layer: [flat output indices]} to the runner-up (forward value kept)."""

    def __init__(self, flips=None):
        self.gap = {}
        self.flips = flips or {}

    def __call__(self, name, a):
        out, i1 = F.max_pool2d(a, 2, stride=2, return_indices=True)
        masked = a.detach().flatten(2).scatter(2, i1.flatten(2), float("-inf")).view_as(a)
        second, i2 = F.max_pool2d(masked, 2, stride=2, return_indices=True)
        self.gap[name] = (out.detach() - second, float(a.detach().max()))
        idx = self.flips.get("pool:" + name)
        if not idx:
            return out
        sel = torch.zeros(out.numel(), dtype=a.dtype)
        sel[torch.as_tensor(idx, dtype=torch.long)] = 1.0
        runner_up = a.flatten(2).gather(2, i2.flatten(2)).view_as(out)
        # zero-valued term whose gradient moves the selected windows' gradient from the maximum to the runner-up
        return out + sel.view_as(out) * ((runner_up - runner_up.detach()) - (out - out.detach()))


def oracle_pass(fn, flips=None):
    """Runs fn() -- an oracle pass through oracle.restate's encoders -- recording every pre-activation and pool window, with
    the tie elements `flips` = {layer: [flat indices]} (relu) and {"pool:" + layer: [flat indices]} (max pool) decided the
    other way.  Returns (fn(), ties): the candidate ties (key, flat index) -- relu pre-activations with |z| < TIE_EPS max|z|
    of their layer, and live pool windows whose two largest activations differ by less than TIE_EPS of the layer's max
    (exactly equal ones are decided alike: same first-maximum rule on identical values)."""
    rec, pool = R.TieRecorder(flips), PoolRecorder(flips)
    R.TIE_HOOK, R.POOL_HOOK = rec, pool
    try:
        out = fn()
    finally:
        R.TIE_HOOK = R.POOL_HOOK = None
    ties = [(name, int(i)) for name, z in rec.z.items()
            for i in (z.reshape(-1).abs() < TIE_EPS * float(z.abs().max())).nonzero().flatten().tolist()]
    for name, (gap, amax) in pool.gap.items():
        near = (gap > 0) & (gap < TIE_EPS * amax)
        ties += [("pool:" + name, int(i)) for i in near.reshape(-1).nonzero().flatten().tolist()]
    return out, ties


def learn_oracle(spec, params, states, adv, actions, old, ret, hp=None, dtype=torch.float64):
    """oracle(flips) -> ((losses, raw grads), ties) of R.learn_iteration at `params` (no update), in `dtype`."""
    cast = lambda t: t.detach().cpu().to(dtype)
    p = {k: cast(v) for k, v in params.items()}
    st = [cast(s) for s in states]
    a, o, ad, r = cast(actions), cast(old), cast(adv), cast(ret)

    def run():
        losses, raw, _ = R.learn_iteration(R.LearnState(spec, p), st, ad, a, o, r, hp or R.PPOHyper(), apply_update=False)
        return losses, raw
    return lambda flips=None: oracle_pass(run, flips)


def grads_match_oracle(grads, oracle, bound=GRAD_BOUND, label=""):
    """grads {name: engine gradient}; oracle(flips) -> ((losses, {name: gradient}), ties) (learn_oracle, or any oracle pass
    wrapped in oracle_pass).  Asserts every gradient within `bound` of its tensor's max; if the plain comparison fails, the
    residual must be explained EXACTLY by deciding some ties the other way in the oracle.  Returns (worst error
    / max|g|, the oracle's losses)."""
    (losses, raw), ties = oracle()
    grads = {n: g.detach().cpu().double() for n, g in grads.items()}
    scale = {n: max(float(g.abs().max()), 1e-30) for n, g in raw.items()}

    def worst_err(ref):
        return max(float((grads[n] - ref[n].double()).abs().max()) / scale[n] for n in ref)

    worst = worst_err(raw)
    if worst >= bound:
        per = sorted(((float((grads[n] - raw[n].double()).abs().max()) / scale[n], n) for n in raw), reverse=True)[:4]
        assert 0 < len(ties) <= 64, (label, per, len(ties))
        chosen = {}
        for name, i in ties:
            # flipping tie t changes the gradients by D_t; it is part of the explanation iff the residual projects onto D_t
            (_, g1), _ = oracle({name: [i]})
            num = sum(float(((grads[n] - raw[n].double()) * (g1[n] - raw[n]).double()).sum()) / scale[n] ** 2 for n in raw)
            den = sum(float(((g1[n] - raw[n]).double() ** 2).sum()) / scale[n] ** 2 for n in raw)
            if den > 0 and abs(num / den - 1.0) < 0.2:
                chosen.setdefault(name, []).append(i)
        assert chosen, ("gradient mismatch not explained by activation ties", label, per, ties)
        (_, raw2), _ = oracle(chosen)
        worst = worst_err(raw2)
        print(label, "ties decided the other way:", chosen)
    assert worst < bound, (label, worst)
    return worst, losses


def element_lrs(spec, names, sizes, hp=None):
    """Learning rate of every element of the flat parameter buffer (reference order): nn/ppo.py:40-42 -- one Adam over all
    parameters of a shared net, actor.* at lr_actor and critic.* at lr_critic otherwise."""
    hp = hp or R.PPOHyper()
    lr = {"all": hp.lr, "actor": hp.lr_actor, "critic": hp.lr_critic}
    groups = R.param_groups(spec, names)
    return torch.cat([torch.full((n,), lr[groups[k]], dtype=torch.float64) for k, n in zip(names, sizes)])


def fp32(x):
    return float(torch.tensor(x, dtype=torch.float32))


def clip_adam_step(p, g, m, v, step, lr, max_norm=0.5, clip=True, b1=fp32(0.9), b2=fp32(0.999), eps=1e-8):
    """One float64 step of clip_grad_norm_(max_norm) + Adam(betas=(b1, b2), eps) over flat buffers; `lr` is a number or a
    per-element tensor.  The inputs are not written.  Returns (p, m, v, pre-clip norm)."""
    p, g, m, v = (t.detach().cpu().double() for t in (p, g, m, v))
    norm = float(torch.linalg.vector_norm(g))
    if clip:
        g = g * min(max_norm / (norm + 1e-6), 1.0)
    m = m + (1 - b1) * (g - m)                         # exp_avg.lerp_(grad, 1 - beta1)
    v = v * b2 + (1 - b2) * g * g                      # exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
    bc1, bc2 = 1 - b1 ** step, 1 - b2 ** step
    lr = lr.double() if torch.is_tensor(lr) else float(lr)
    p = p - (lr / bc1) * m / (v.sqrt() / math.sqrt(bc2) + eps)
    return p, m, v, norm


def adam_mismatch(p_old, got, ref):
    """Elements of the engine's (p, m, v) after one step outside the tolerance around the float64 reference (p, m, v) stepped
    from p_old: the parameter DELTA within 1e-5 of the largest reference delta + 2 ulp of the parameter (fp32 p resolves the
    update only to ~1 ulp), m and v within 1e-5 of their tensor's max + 4 ulp of the element.  Returns
    {"p" | "m" | "v": (bad count, worst excess)}, empty when all agree."""
    p_old = p_old.detach().cpu().double()
    got = [t.detach().cpu().double() for t in got]
    out = {}
    d_ref = ref[0] - p_old
    checks = (("p", got[0] - p_old, d_ref, 1e-5 * float(d_ref.abs().max()) + 2.4e-7 * (1.0 + p_old.abs())),
              ("m", got[1], ref[1], 1e-5 * float(ref[1].abs().max()) + 4.8e-7 * ref[1].abs()),
              ("v", got[2], ref[2], 1e-5 * float(ref[2].abs().max()) + 4.8e-7 * ref[2].abs()))
    for name, x, r, tol in checks:
        excess = (x - r).abs() - tol
        bad = int((excess > 0).sum())
        if bad:
            out[name] = (bad, float(excess.max()))
    return out
