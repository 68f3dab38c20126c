"""TEST INFRASTRUCTURE ONLY -- numpy float64 restatement of the running observation statistics of NORM_OBS (gym's
RunningMeanStd: count 1e-4, mean 0, var 1 at the start; Chan's parallel merge of each batch's population moments) and of the
fp32 applied form the learner and the Forward module normalise with:

  mean32 = fp32(mean),  scale32 = fp32(1 / sqrt(var + 1e-8)),  x_hat = clip((x - mean32) * scale32, -clip, clip)"""
import numpy as np


class RunningMeanStd:
    def __init__(self, D):
        self.mean = np.zeros(D, np.float64)
        self.var = np.ones(D, np.float64)
        self.count = 1e-4

    def update(self, x):
        """Folds the rows of x [B, D] in (gym: batch mean, population variance)."""
        x = np.asarray(x, np.float64).reshape(len(x), -1)
        self.update_from_moments(x.mean(axis=0), x.var(axis=0), x.shape[0])

    def update_from_moments(self, batch_mean, batch_var, batch_count):
        delta = batch_mean - self.mean
        tot = self.count + batch_count
        new_mean = self.mean + delta * batch_count / tot
        m2 = self.var * self.count + batch_var * batch_count + np.square(delta) * self.count * batch_count / tot
        self.mean, self.var, self.count = new_mean, m2 / tot, tot

    def update_from_sums(self, s1, s2, n, shift):
        """The same merge from the column sums of d = x - shift and d^2 (what the moments kernel produces)."""
        d = s1 / n
        self.update_from_moments(shift + d, s2 / n - d * d, n)


def shifted_sums(x, shift):
    d = np.asarray(x, np.float64).reshape(len(x), -1) - shift
    return d.sum(axis=0), (d * d).sum(axis=0)


def applied(mean, var):
    return np.asarray(mean, np.float64).astype(np.float32), (1.0 / np.sqrt(np.asarray(var, np.float64) + 1e-8)).astype(np.float32)


def normalize(x, mean32, scale32, clip):
    """fp32: one rounding per operation, as the kernel and torch compute it."""
    x = np.asarray(x, np.float32).reshape(len(x), -1)
    y = (x - mean32) * scale32
    return y if clip is None else np.clip(y, np.float32(-clip), np.float32(clip))
