"""TEST INFRASTRUCTURE ONLY -- float64 restatement of the value-target normalisation of NORM_VALUE (PopArt): gym's
RunningMeanStd of one column (tests/obs_norm_ref.py), the fp32 applied form, the head rescale that keeps the unnormalised
outputs, and critic 0's value loss on normalised targets (the clipped form of tests/ppo_options_ref.py):

  sigma = sqrt(var + 1e-8);  applied = {fp32(mean), fp32(1 / sigma), fp32(sigma)}
  W' = W sigma_old / sigma_new,  b' = (sigma_old b + mean_old - mean_new) / sigma_new
  R~ = (R - mean32) * scale32 (old values alike);  values returned = v * sigma32 + mean32"""
import numpy as np
import torch

import obs_norm_ref as N


class ValueRMS(N.RunningMeanStd):
    def __init__(self):
        super().__init__(1)

    def sigma(self):
        return float(np.sqrt(self.var[0] + 1e-8))


def applied(mean, var):
    sigma = np.sqrt(np.float64(var) + 1e-8)
    return np.array([np.float64(mean), 1.0 / sigma, sigma]).astype(np.float32)


def rescale_head(w, b, old, new):
    """(W', b') in float64 from the statistics (mean, var) before and after the merge."""
    (m0, v0), (m1, v1) = old, new
    s0, s1 = np.sqrt(v0 + 1e-8), np.sqrt(v1 + 1e-8)
    w = np.asarray(w, np.float64)
    return w * s0 / s1, (s0 * np.float64(b) + m0 - m1) / s1


def normalize(x, a):
    """fp32, two roundings: (x - mean32) * scale32."""
    return (torch.as_tensor(x, dtype=torch.float32) - float(a[0])) * float(a[1])


def denormalize(v, a):
    return torch.as_tensor(v, dtype=torch.float32) * float(a[2]) + float(a[0])


def value_loss(v, returns, a, old_values=None, value_clip=None, smooth_l1=False):
    """critic 0's value loss in normalised units, optionally clipped around the normalised old values (float64 autograd)."""
    v = torch.as_tensor(v, dtype=torch.float64)
    R = normalize(returns, a).double()
    rows = (lambda x: torch.nn.functional.smooth_l1_loss(R, x, reduction="none")) if smooth_l1 else (lambda x: (R - x) ** 2 / 2)
    if value_clip is None:
        return torch.mean(rows(v))
    ov = normalize(old_values, a).double()
    vc = ov + torch.clamp(v - ov, -value_clip, value_clip)
    return torch.mean(torch.max(rows(v), rows(vc)))

