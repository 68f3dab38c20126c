"""Running observation statistics of the learner and the Forward module (non-reference option NORM_OBS of ``PPO``).

Per normalised observation slot of D elements per row, float64 buffers ``mean_<slot>`` [D], ``var_<slot>`` [D] and
``count_<slot>`` [1] with gym's ``RunningMeanStd`` conventions (start: count 1e-4, mean 0, var 1; a batch is folded in with
Chan's parallel merge of its population moments).  Observations are normalised with the fp32 *applied form*

    mean32 = fp32(mean),  scale32 = fp32(1 / sqrt(var + 1e-8)),  x_hat = clamp((x - mean32) * scale32, -clip, clip)

kept in two non-persistent buffers next to the statistics, so the learner and every predictor that loads the same statistics
compute the same bits.  All arithmetic runs in the CUDA kernels of csrc/obsnorm.cu (kernels.obs_*).

The buffers are created when the owning net's engine is first built, because the slot sizes come from the engine; a
checkpoint loaded before that creates them from its own shapes, and the build checks them.
"""
import re

import numpy as np
import torch

from .. import kernels
from .._lib import DDRLError

_STATE = re.compile(r"(mean|var|count)_(\d+)$")


class ObsRMS(torch.nn.Module):
    def __init__(self, slots, clip):
        """slots: sorted tuple of slot indices, or None for every slot of the net; clip: float > 0 or None (no clamp)."""
        super().__init__()
        self.wanted = slots
        self.clip = clip
        self.slots = None           # the resolved slot tuple once bound to an engine
        self.dims = {}              # slot -> D
        self.sums = None            # float64: the concatenated moments [2 D] of every slot of the current learn call
        self._ws = None             # byte workspace of the two-pass moments
        self._applied = None        # identity of the float64 state the applied form was last computed from

    def state(self, s):
        return getattr(self, "mean_%d" % s), getattr(self, "var_%d" % s), getattr(self, "count_%d" % s)

    def applied(self, s):
        return getattr(self, "mean32_%d" % s), getattr(self, "scale32_%d" % s)

    def bind(self, n_obs, elems, dev):
        """Resolves the slots against an engine with `n_obs` observation slots of elems(s) elements each, and creates (or checks
        and moves) the buffers on `dev`."""
        slots = tuple(range(n_obs)) if self.wanted is None else self.wanted
        bad = [s for s in slots if s >= n_obs]
        if bad:
            raise DDRLError("NORM_OBS slot(s) %s out of range: the net has %d observation slot(s)" % (bad, n_obs))
        dims = {}
        for s in slots:
            D = int(elems(s))
            init = {"mean": lambda: torch.zeros(D, dtype=torch.float64), "var": lambda: torch.ones(D, dtype=torch.float64),
                    "count": lambda: torch.full((1,), 1e-4, dtype=torch.float64)}
            for kind, make in init.items():
                name = "%s_%d" % (kind, s)
                t = self._buffers.get(name)
                want = 1 if kind == "count" else D
                if t is None:
                    t = make()
                elif tuple(t.shape) != (want,):
                    raise DDRLError("NORM_OBS statistics %s have shape %s; slot %d of this net needs (%d,)"
                                    % (name, tuple(t.shape), s, want))
                self.register_buffer(name, t.to(device=dev, dtype=torch.float64).contiguous())
            for name in ("mean32_%d" % s, "scale32_%d" % s):
                self.register_buffer(name, torch.empty(D, dtype=torch.float32, device=dev), persistent=False)
            dims[s] = D
        self.slots, self.dims = slots, dims
        self.sums = torch.zeros(sum(2 * D for D in dims.values()), dtype=torch.float64, device=dev)
        self._ws = None
        self._applied = None

    def _load_from_state_dict(self, state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs):
        for key, t in state_dict.items():
            m = _STATE.match(key[len(prefix):]) if key.startswith(prefix) else None
            if m and key[len(prefix):] not in self._buffers and (self.wanted is None or int(m.group(2)) in self.wanted):
                self.register_buffer(key[len(prefix):], torch.empty(tuple(t.shape), dtype=torch.float64))
        super()._load_from_state_dict(state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs)

    def _key(self):
        return tuple((t.data_ptr(), t._version) for s in self.slots for t in self.state(s))

    def refresh(self):
        """Recomputes the applied form when the float64 state changed outside the kernels (load_state_dict, bind, an edit)."""
        key = self._key()
        if key != self._applied:
            for s in self.slots:
                kernels.obs_rms_update(*self.state(s), None, 0.0, *self.applied(s))
            self._applied = key

    def normalize(self, s, x, out):
        mean32, scale32 = self.applied(s)
        return kernels.obs_normalize(x, mean32, scale32, self.clip, out)

    def _segments(self):
        off = 0
        for s in self.slots:
            D = self.dims[s]
            yield s, self.sums[off:off + 2 * D]
            off += 2 * D

    def moments(self, raw):
        """The moments of the raw rows raw[s] around the current mean of every slot, into self.sums."""
        for s, seg in self._segments():
            x = raw[s]
            need = kernels.obs_moments_ws_bytes(x.shape[0], self.dims[s])
            if need and (self._ws is None or self._ws.numel() < need):
                self._ws = torch.empty(need, dtype=torch.uint8, device=seg.device)
            kernels.obs_moments(x, self.state(s)[0], seg, self._ws)

    def merge(self, n):
        """Folds the batch of `n` rows whose moments are in self.sums into the statistics and rewrites the applied form."""
        for s, seg in self._segments():
            kernels.obs_rms_update(*self.state(s), seg, float(n), *self.applied(s))

    def records(self):
        """Per slot in slot order: mean32 [D], scale32 [D] and the count [1] as fp32 arrays (ONE device-to-host copy)."""
        self.refresh()
        parts = []
        for s in self.slots:
            mean32, scale32 = self.applied(s)
            parts += [mean32, scale32, self.state(s)[2].float()]
        host = torch.cat(parts).cpu().numpy()
        out, off = [], 0
        for s in self.slots:
            D = self.dims[s]
            out += [host[off:off + D], host[off + D:off + 2 * D], host[off + 2 * D:off + 2 * D + 1]]
            off += 2 * D + 1
        return out

    def load_records(self, recs):
        """Sets the applied form of every slot bit-exactly from (mean32, scale32, count) fp32 arrays, and the float64 state to
        (mean32, 1 / scale32^2 - 1e-8, count): an approximation of the learner's state, enough to act with; a learner restores
        from state_dict."""
        dev = self.sums.device
        with torch.no_grad():
            for s, (mean32, scale32, count) in zip(self.slots, recs):
                m32 = torch.from_numpy(np.ascontiguousarray(mean32, dtype=np.float32)).to(dev)
                s32 = torch.from_numpy(np.ascontiguousarray(scale32, dtype=np.float32)).to(dev)
                mean, var, cnt = self.state(s)
                mean.copy_(m32.double())
                var.copy_(1.0 / s32.double() ** 2 - 1e-8)
                cnt.fill_(float(count[0]))
                a_mean, a_scale = self.applied(s)
                a_mean.copy_(m32)
                a_scale.copy_(s32)
        self._applied = self._key()
