"""PPO -- drop-in for USTC_lab/nn/ppo.py:17-146 running on the fused sm_100a engine.

Same constructor, attributes and call contracts as the reference class:
  * ``PPO(actor, critic, prenet, rnd, config, config_nn)``            (runner/utils.py:160)
  * ``net(states, act=None, play_mode=False) -> ((pi, log_p), [values [B,1]])``   (ppo.py:72-75)
  * ``net.learn(Experience)`` -> generator of ``(loss_dict, update_time, last)``   (ppo.py:77-142)
  * ``state_dict()/load_state_dict()/named_parameters()`` names, shapes and order (App. C)
  * ``nn2redis / updatenn_by_redis / updatenn``                         (nn/base.py:60-95)
plus the fused entry point ``net.act(states, draw, play_mode)`` = compute body of
``ForwardThread.run`` (server/forward.py:128-146) with the random draw supplied.

What is different underneath: all parameters live in ONE flat fp32 device buffer (reference
order); ``p.data`` of every ``nn.Parameter`` is a view into it.  Gradients, Adam m and v are flat
buffers of the same layout, so the data-parallel learner all-reduces one buffer and the fused
clip+Adam kernel walks it once.  No autograd graph is ever built.
"""
import copy
import ctypes as C
import functools
import math
import os
import struct
import time

import numpy as np
import torch
from torch.distributions.categorical import Categorical
from torch.distributions.normal import Normal

from .. import _lib, dist, kernels
from .._lib import DDRLError, NetDesc, check, current_stream, ptr
from .base import Basenn
from .obs_rms import ObsRMS, ValueRMS, share_sums


def _on_device(fn):
    """Engine calls run with the NET's device current: the C ABI allocates and launches on the current device, and
    current_stream() is the current device's stream -- a net on cuda:1 must not depend on the caller's set_device."""
    @functools.wraps(fn)
    def wrapped(self, *args, **kwargs):
        p = next(self.parameters(), None)
        if p is None or p.device.type != "cuda":
            return fn(self, *args, **kwargs)
        with torch.cuda.device(p.device):
            return fn(self, *args, **kwargs)
    return wrapped


def _cfg(obj, name, default):
    return getattr(obj, name, default) if obj is not None else default


def _flag_option(config_nn, name):
    v = _cfg(config_nn, name, False)
    if not isinstance(v, (bool, np.bool_)):
        raise DDRLError("%s must be True or False (got %r)" % (name, v))
    return bool(v)


def _positive_option(config_nn, name, default=None):
    v = _cfg(config_nn, name, default)
    if v is None:
        return None
    if isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, float, np.integer, np.floating)) or not math.isfinite(v) or v <= 0:
        raise DDRLError("%s must be a finite number > 0 or None (got %r)" % (name, v))
    return float(v)


def _slots_option(config_nn, name):
    """False (off), True (every observation slot) or a list / tuple of distinct slot indices -> None (off), "all" or a sorted
    tuple.  Indices beyond the net's slots are rejected when the engine is built (ObsRMS.bind)."""
    v = _cfg(config_nn, name, False)
    if isinstance(v, (bool, np.bool_)):
        return "all" if v else None
    ok = isinstance(v, (list, tuple)) and len(v) > 0 and all(
        isinstance(s, (int, np.integer)) and not isinstance(s, (bool, np.bool_)) and s >= 0 for s in v)
    if not ok or len(set(int(s) for s in v)) != len(v):
        raise DDRLError("%s must be True, False or a non-empty list of distinct slot indices >= 0 (got %r)" % (name, v))
    return tuple(sorted(int(s) for s in v))


class PPO(Basenn):
    def __init__(self, actor, critic, prenet=None, rnd=None, config=None, config_nn=None):
        super().__init__(config, config_nn)
        if rnd is not None:
            raise DDRLError("RND is outside the B200 hot path (off by default, config_nn.py:19); use the reference's nn/RND.py")
        self.device = _cfg(config, "DEVICE", "cuda")
        self.prenet = prenet            # registration order = reference (ppo.py:27-29): prenet, actor, critic
        self.actor = actor
        self.critic = critic
        self._critics = [self.critic]
        self.rnd = None
        self.gail_critic = False
        self.share_cnn_net = _cfg(config_nn, "SHARE_CNN_NET", prenet is not None)
        if bool(self.share_cnn_net) != (prenet is not None):
            raise DDRLError("SHARE_CNN_NET=%s but prenet is %s" % (self.share_cnn_net, type(prenet).__name__))
        # PPO training options (non-reference, all off by default): per-step advantage normalisation, clipped value loss of
        # critic 0, approx-KL / clip-fraction statistics, and a KL target that ends the learn call (it implies the statistics)
        self.norm_adv = _flag_option(config_nn, "NORM_ADV")
        self.value_clip = _positive_option(config_nn, "VALUE_CLIP")
        self.target_kl = _positive_option(config_nn, "TARGET_KL")
        self.ppo_stats = _flag_option(config_nn, "PPO_STATS") or self.target_kl is not None
        # running observation normalisation (non-reference, off by default): float64 statistics of the chosen slots in the
        # submodule obs_rms (state_dict keys obs_rms.{mean,var,count}_<slot>), applied by act / forward / encode / learn
        norm_obs = _slots_option(config_nn, "NORM_OBS")
        clip = _positive_option(config_nn, "NORM_OBS_CLIP", 10.0)
        self.obs_rms = None if norm_obs is None else ObsRMS(None if norm_obs == "all" else norm_obs, clip)
        self._obs_act = {}              # NORM_OBS: per slot, the act / encode scratch (grows with B)
        self._obs_learn = {}            # NORM_OBS: per slot, the learner's persistent normalised batch
        self._obs_n = 0                 # NORM_OBS: rows of the global batch of the current learn call
        # value-target normalisation (non-reference, off by default; PopArt): float64 statistics of critic 0's return targets in
        # the submodule value_rms (state_dict keys value_rms.{mean,var,count}); critic 0 learns normalised targets and act /
        # forward return its values denormalised
        self.value_rms = ValueRMS() if _flag_option(config_nn, "NORM_VALUE") else None
        self._norm_sums = None          # NORM_VALUE: the float64 moment sums a data-parallel learner all-reduces (+ NORM_OBS's)
        # decoupled PPO (non-reference, off by default; Hilton, Cobbe & Schulman 2022): the clip is centred on the policy at the
        # start of the learn call (the proximal log-probs) and the actor term is weighted by exp(prox - old), optionally
        # truncated at DECOUPLED_IS_CLIP
        self.decoupled = _flag_option(config_nn, "DECOUPLED_PPO")
        self.decoupled_is_clip = _positive_option(config_nn, "DECOUPLED_IS_CLIP")
        if self.decoupled_is_clip is not None and not self.decoupled:
            raise DDRLError("DECOUPLED_IS_CLIP needs DECOUPLED_PPO=True")
        self.last_prox_logps = None     # DECOUPLED_PPO: the proximal log-probs [B_local] of the last learn call (persistent)
        # invalid-action masking (non-reference, off by default; Huang & Ontanon 2022): one more state slot after the encoder's,
        # [B, A], action j allowed iff != 0; act / forward sample, and learn trains, the masked categorical distribution (per branch
        # for a MultiCategoricalActor, whose mask is [B, sum n])
        self.action_mask = _flag_option(config_nn, "ACTION_MASK")
        if self.action_mask and getattr(actor, "DIST", None) not in ("categorical", "multi_categorical"):
            raise DDRLError("ACTION_MASK needs a CategoricalActor or a MultiCategoricalActor (got %s)" % type(actor).__name__)
        self.hp = kernels.make_hparams(
            ppo_clip=_cfg(config_nn, "PPO_CLIP", 0.2), dual_clip=_cfg(config_nn, "DUEL_PPO_CLIP", 3),
            v_coef=_cfg(config_nn, "V_LOSS_THETA", 1.0), ent_coef=_cfg(config_nn, "ENTROPY_LOSS_THETA", 0.05),
            max_grad_norm=_cfg(config_nn, "CLIP_GRID_NUM", 0.5), clip_grad=_cfg(config_nn, "CLIP_GRID", True),
            smooth_l1=_cfg(config_nn, "SMOOTH_L1_LOSS", False), lr=_cfg(config_nn, "LEARNING_RATE", 2e-4),
            lr_actor=_cfg(config_nn, "ACTOR_LEARNING_RATE", 5e-5), lr_critic=_cfg(config_nn, "CRITIC_LEARNING_RATE", 1e-3),
            value_clip=self.value_clip or 0.0, ppo_stats=self.ppo_stats)
        self.clip_grad = bool(self.hp.clip_grad)
        self.clip_grad_num = self.hp.max_grad_norm
        self.v_loss_theta, self.ent_loss_theta = self.hp.v_coef, self.hp.ent_coef
        self.ppo_clip, self.duel_ppo_clip = self.hp.ppo_clip, self.hp.dual_clip
        self.training_iter_time = _cfg(config_nn, "TRAINING_ITER_TIME", 10)
        # minibatch epochs (non-reference option): every epoch shuffles the batch and takes one optimiser step per chunk
        self.mini_batch_num = _cfg(config_nn, "MINI_BATCH_NUM", 1)
        if isinstance(self.mini_batch_num, bool) or not isinstance(self.mini_batch_num, (int, np.integer)) or self.mini_batch_num < 1:
            raise DDRLError("MINI_BATCH_NUM must be an integer >= 1 (got %r)" % (self.mini_batch_num,))
        self.mini_batch_num = int(self.mini_batch_num)
        seed = _cfg(config_nn, "MINI_BATCH_SEED", None)
        if seed is not None and (isinstance(seed, bool) or not isinstance(seed, (int, np.integer))):
            raise DDRLError("MINI_BATCH_SEED must be an integer or None (got %r)" % (seed,))
        self._mb_seed = None if seed is None else int(seed)
        self._mb_gen = None             # torch.Generator on the net's device (the minibatch shuffles)
        self._mb = None                 # persistent minibatch buffers (_minibatch_buffers)
        self._fb = None                 # persistent full-batch buffers of the PPO options (_full_batch_inputs)
        self._m3 = None                 # float64 [3] advantage moments of a data-parallel NORM_ADV step
        self.last_minibatch_perms = []  # per epoch of the last minibatch learn call: int32 device permutation of the rows
        self.gemm_mode = os.environ.get("DDRL_GEMM_MODE", _cfg(config_nn, "GEMM_MODE", "tc3"))
        self.update_time = 0
        self._adam_step = 0
        self._h = None                  # ddrl_net*
        self._flat = self._grads = self._m = self._v = None
        self._offsets = None
        self._P = 0
        self._versions = None
        self._dp_group = None
        self._dp_world = 1
        self._loss4 = None
        self._extra_key = None          # pointers the engine holds for the extra value heads (shared mode)
        self._extra_scratch = None      # per extra head: this iteration's (dw, db), written by the engine
        self._aux = []                  # one value-only engine per extra critic that owns an encoder (unshared mode)
        self._peer = None               # peer-memory all-reduce state (enable_data_parallel)
        self._peer_error = None
        self._seg_runs = None           # per backward segment: flat gradient ranges final after it (data-parallel overlap)

    # ------------------------------------------------------------------ engine plumbing
    def _encoder(self):
        return self.prenet if self.prenet is not None else self.actor.pre

    def _act_dim(self):
        """Action dimensions A: the Beta head emits alpha | beta pre-activations, 2A columns.  MultiCategoricalActor: the head
        width sum n_i."""
        n = self.actor.actor_linear.out_features
        return n // 2 if self.actor.DIST == "beta" else n

    def _spec(self):
        enc = self._encoder()
        if enc is None or getattr(enc, "ARCH", None) is None:
            raise DDRLError("PPO needs a ddrl4nav_b200 encoder (AtariPreNet / NavPreNet / NavPedPreNet / NavPreNet1D / MLPPreNet)")
        if self.prenet is None and type(self.critic.pre) is not type(enc):
            raise DDRLError("unshared mode needs the same encoder family in actor.pre and critic.pre")
        return dict(arch=enc.ARCH, in_ch=enc.engine_in_ch(), act_dim=self._act_dim(),
                    dist=self.actor.DIST, shared=self.prenet is not None, feat=self.actor.actor_linear.in_features,
                    laser_ch=int(getattr(enc, "laser_channel", 0)))

    def _destroy(self):
        if self._h is not None:
            _lib.load().ddrl_net_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self._destroy()
        except Exception:
            pass

    def _ensure_engine(self):
        """(Re)builds the flat buffers when needed and tells the engine about out-of-band weight edits."""
        plist = list(self.named_parameters())
        dev = plist[0][1].device
        if dev.type != "cuda":
            raise DDRLError("ddrl4nav_b200.nn.PPO needs its parameters on a CUDA device (got %s); there is no CPU "
                            "fallback -- call .to('cuda')" % dev)
        aliased = self._flat is not None and self._flat.device == dev and all(
            p.data_ptr() == self._flat.data_ptr() + 4 * off for (_, p), off in zip(plist, self._offsets))
        if self._h is None or not aliased:
            self._build(plist, dev)
        ver = sum(p._version for _, p in plist)
        if ver != self._versions:
            check(_lib.load().ddrl_net_params_changed(self._h), "ddrl_net_params_changed")
            self._versions = ver
        if len(self._critics) > 1 or self._extra_key is not None:
            self._sync_extra_critics(dev)

    # ------------------------------------------------------------------ extra critics (nn/ppo.py:63-64,75,95-105)
    def _extra_in_loss(self, k):
        """Only the LAST critic's loss is added, and only under gail_critic (ppo.py:101-104); RND (ppo.py:97-100) is out
        of scope and rejected by the constructor."""
        return bool(self.gail_critic) and k == len(self._critics) - 2

    def _sync_extra_critics(self, dev):
        extras = self._critics[1:]
        if self.prenet is None:
            return                      # unshared: every extra critic runs on a value-only engine of its own (self._aux)
        lib = _lib.load()
        key = []
        if self._extra_scratch is None or len(self._extra_scratch) != len(extras):
            self._extra_scratch = [(torch.zeros_like(c.critic_linear.weight, device=dev), torch.zeros_like(c.critic_linear.bias, device=dev))
                                   for c in extras]
        for k, c in enumerate(extras):
            w, b = c.critic_linear.weight, c.critic_linear.bias
            if w.device != dev or not w.is_contiguous() or w.dtype != torch.float32:
                raise DDRLError("extra critic %d must hold contiguous fp32 parameters on %s (call .to(device))" % (k, dev))
            gw, gb = self._extra_scratch[k]
            key.append((w.data_ptr(), b.data_ptr(), gw.data_ptr(), gb.data_ptr(), int(self._extra_in_loss(k))))
        key = tuple(key)
        if key == self._extra_key:
            return
        n = len(key)
        arr = lambda col: (C.c_void_p * max(n, 1))(*[e[col] or None for e in key])
        flags = (C.c_int * max(n, 1))(*[e[4] for e in key])
        check(lib.ddrl_net_set_extra_critics(self._h, n, arr(0), arr(1), arr(2), arr(3), flags), "ddrl_net_set_extra_critics")
        self._extra_key = key if n else None

    def _extra_grads_to_params(self):
        """Adds this iteration's gradients of the extra heads (engine scratch, all-reduced in a data-parallel learner) to
        their `.grad`, which nobody in PPO zeroes -- as with the reference's autograd accumulation."""
        for k, c in enumerate(self._critics[1:]):
            if not self._extra_in_loss(k):
                continue
            for p, g in zip((c.critic_linear.weight, c.critic_linear.bias), self._extra_scratch[k]):
                if self._dp_world > 1:
                    import torch.distributed as tdist
                    tdist.all_reduce(g, group=self._dp_group)
                p.grad = g.clone() if p.grad is None else p.grad.add_(g)
                g.zero_()

    def _aux_net(self, k):
        """Value-only engine of extra critic k in unshared mode: its own encoder + its critic_linear, built as a share-CNN
        net with a throw-away 1-way actor (zero advantage => the actor path contributes exactly nothing)."""
        while len(self._aux) <= k:
            self._aux.append(None)
        c = self._critics[1 + k]
        if self._aux[k] is None or self._aux[k][0] is not c:
            from .actor import CategoricalActor
            from .critic import Critic
            feat = c.critic_linear.in_features
            holder = Critic(last_input_dim=feat, pre=None)
            holder.critic_linear = c.critic_linear               # the SAME parameters: p.data re-points into aux's flat buffer
            actor = CategoricalActor(1, last_input_dim=feat, pre=None)
            aux = PPO(actor, holder, c.pre, None, None, None)      # no config: no Redis connection of its own
            aux.gemm_mode = self.gemm_mode
            aux.hp = kernels.make_hparams(
                ppo_clip=self.hp.ppo_clip, dual_clip=self.hp.dual_clip, v_coef=1.0, ent_coef=0.0,
                max_grad_norm=self.hp.max_grad_norm, clip_grad=self.hp.clip_grad, smooth_l1=self.hp.smooth_l1, lr=0.0,
                lr_actor=0.0, lr_critic=0.0)
            aux.to(self._flat.device)
            self._aux[k] = (c, aux)
        return self._aux[k][1]

    def _build(self, plist, dev):
        lib = _lib.load()
        self._destroy()
        s = self._spec()
        desc = NetDesc(_lib.ARCH[s["arch"]], s["in_ch"], s["act_dim"], _lib.DIST[s["dist"]], int(s["shared"]), s["feat"],
                       _lib.GEMM_MODE[self.gemm_mode], s["laser_ch"])
        h = C.c_void_p()
        check(lib.ddrl_net_create(C.byref(desc), C.byref(h)), "ddrl_net_create")
        self._h = h
        if s["dist"] == "beta":
            A = s["act_dim"]
            check(lib.ddrl_net_set_action_bounds(h, (C.c_float * A)(*self.actor.action_low), (C.c_float * A)(*self.actor.action_high)),
                  "ddrl_net_set_action_bounds")
        if s["dist"] == "multi_categorical":
            nvec = self.actor.nvec
            check(lib.ddrl_net_set_action_branches(h, len(nvec), (C.c_int32 * len(nvec))(*nvec)), "ddrl_net_set_action_branches")
        if self.action_mask:
            check(lib.ddrl_net_set_action_mask(h, 1), "ddrl_net_set_action_mask")
        if self.obs_rms is not None:
            n_obs = lib.ddrl_net_num_obs(h)
            try:
                self.obs_rms.bind(n_obs, lambda i: lib.ddrl_net_obs_elems(h, i), dev, n_obs - 1 if self.action_mask else None)
            except DDRLError:
                self._destroy()
                raise
        if self.value_rms is not None:
            self.value_rms.bind(dev)
            self._norm_sums = self.value_rms.sums if self.obs_rms is None else share_sums(self.obs_rms, self.value_rms)
            check(lib.ddrl_net_set_value_norm(h, ptr(self.value_rms.applied32)), "ddrl_net_set_value_norm")
        nt = lib.ddrl_net_num_tensors(h)
        P = lib.ddrl_net_num_params(h)
        if nt != len(plist):
            raise DDRLError("parameter table mismatch: engine has %d tensors, module has %d" % (nt, len(plist)))
        offsets = []
        name = C.create_string_buffer(128)
        shape = (C.c_int64 * 4)()
        ndim = C.c_int()
        off = C.c_int64()
        for i, (pname, p) in enumerate(plist):
            check(lib.ddrl_net_tensor_info(h, i, name, 128, shape, C.byref(ndim), C.byref(off)), "ddrl_net_tensor_info")
            eshape = tuple(shape[k] for k in range(ndim.value))
            if name.value.decode() != pname or eshape != tuple(p.shape):
                raise DDRLError("parameter %d mismatch: engine %s%s vs module %s%s" %
                                (i, name.value.decode(), eshape, pname, tuple(p.shape)))
            offsets.append(off.value)
        with torch.cuda.device(dev):
            flat = torch.empty(P, dtype=torch.float32, device=dev)
            old_m, old_v = self._m, self._v
            if self._peer is not None and self._peer["grads"].numel() == P + 8 and self._peer["grads"].device == dev:
                self._grads = self._peer["grads"].zero_()      # the symmetric-memory buffer the peer all-reduce works on
            else:
                self._grads = torch.zeros(P + 8, dtype=torch.float32, device=dev)
            self._m = torch.zeros(P, dtype=torch.float32, device=dev)
            self._v = torch.zeros(P, dtype=torch.float32, device=dev)
            if old_m is not None and old_m.numel() == P:       # keep Adam state across a .to()/re-flatten
                self._m.copy_(old_m)
                self._v.copy_(old_v)
            # {total, actor, v, entropy} (+ {approx KL, clip fraction, behaviour KL | -, -} with PPO_STATS): one D2H copy per step
            self._loss4 = torch.zeros(8 if self.ppo_stats else 4, dtype=torch.float32, device=dev)
        with torch.no_grad():
            for (pname, p), o in zip(plist, offsets):
                view = flat[o:o + p.numel()].view(p.shape)
                view.copy_(p.data.to(torch.float32))
                p.data = view
                p.grad = None
        self._flat, self._offsets = flat, offsets
        self._seg_runs = None
        self._P = P
        check(lib.ddrl_net_bind(h, ptr(flat), ptr(self._grads), ptr(self._m), ptr(self._v)), "ddrl_net_bind")
        # stand-alone encoder calls (enc(states) -> [B, 512]) run on this engine's towers
        if self.prenet is not None:
            self.prenet._attach(self, 0)
        else:
            self.actor.pre._attach(self, 0)
            self.critic.pre._attach(self, 1)
        self._versions = sum(p._version for _, p in plist)
        if self.prenet is None:
            self._seg = ([0, offsets[[n for n, _ in plist].index("critic.critic_linear.weight")], P],
                         [self.hp.lr_actor, self.hp.lr_critic])
        else:
            self._seg = ([0, P], [self.hp.lr])

    def _weights_changed(self):
        if self._h is not None:
            check(_lib.load().ddrl_net_params_changed(self._h), "ddrl_net_params_changed")

    def _params_to_host(self):
        if self._flat is None:
            return super()._params_to_host()
        host = self._flat.detach().cpu().numpy()               # ONE D2H copy for the whole model blob
        return [(n, host[o:o + p.numel()].reshape(tuple(p.shape))) for (n, p), o in zip(self.named_parameters(), self._offsets)]

    @_on_device
    def _state_records(self):
        """After the parameters, so that a predictor loading the blob acts with exactly the learner's applied forms:
        NORM_OBS: per normalised slot, in slot order, the records mean32 [D], scale32 [D] and count [1];
        NORM_VALUE: then one record [4] = {mean32, scale32, sigma32, count}."""
        if self.obs_rms is None and self.value_rms is None:
            return []
        self._ensure_engine()
        recs = self.obs_rms.records() if self.obs_rms is not None else []
        return recs + (self.value_rms.records() if self.value_rms is not None else [])

    @_on_device
    def _load_state_records(self, view):
        if self.obs_rms is None and self.value_rms is None:
            return
        self._ensure_engine()
        index = self._load_obs_records(view) if self.obs_rms is not None else 0
        if self.value_rms is not None:
            try:
                wb, _ = self._decode_wb(view[index:])
            except (struct.error, ValueError):
                wb = None
            if wb is None or wb.shape != (4,):
                raise DDRLError("model blob has no NORM_VALUE record [4] after the parameters%s (written by a net without "
                                "NORM_VALUE?)" % (" and the NORM_OBS records" if self.obs_rms is not None else ""))
            self.value_rms.load_records(wb)

    def _load_obs_records(self, view):
        """Reads the NORM_OBS records at the start of `view`; returns the bytes they take."""
        rms, recs, index = self.obs_rms, [], 0
        for s in rms.slots:
            got = []
            for what, n in (("mean32", rms.dims[s]), ("scale32", rms.dims[s]), ("count", 1)):
                try:
                    wb, used = self._decode_wb(view[index:])
                except (struct.error, ValueError):
                    wb, used = None, 0
                if wb is None or wb.shape != (n,):
                    raise DDRLError("model blob has no NORM_OBS %s record [%d] for slot %d after the parameters (written by a net "
                                    "without NORM_OBS, or with other slots?)" % (what, n, s))
                got.append(wb)
                index += used
            recs.append(got)
        rms.load_records(recs)
        return index

    def flat_grads(self):
        """View of the flat gradient buffer (reference parameter order) of the last backward."""
        return self._grads[:self._P]

    def named_grads(self):
        return {n: self._grads[o:o + p.numel()].view(p.shape) for (n, p), o in zip(self.named_parameters(), self._offsets)}

    def _obs_ptrs(self, states, allow_empty=False):
        lib = _lib.load()
        n_obs = lib.ddrl_net_num_obs(self._h)
        if len(states) < n_obs:
            raise DDRLError("expected %d state slots, got %d" % (n_obs, len(states)))
        dev = self._flat.device
        keep, B = [], None
        for i in range(n_obs):
            t = states[i]
            if not torch.is_tensor(t):
                t = torch.as_tensor(np.asarray(t))
            t = t.to(device=dev, dtype=torch.float32).contiguous()
            per = lib.ddrl_net_obs_elems(self._h, i)
            if B is None:
                B = t.shape[0]
            if t.shape[0] != B or ((B or not allow_empty) and (t.numel() // max(B, 1)) != per):
                raise DDRLError("state slot %d has shape %s; expected [B=%d, %d elements/sample]" % (i, tuple(t.shape), B, per))
            keep.append(t)
        arr = (C.c_void_p * n_obs)(*[t.data_ptr() for t in keep])
        return keep, arr, n_obs, B

    def _normalized_obs(self, states, bufs):
        """NORM_OBS: `states` with every normalised slot replaced by its normalised copy in bufs[slot] (the persistent learner
        buffers, or the act scratch, which grows with B); the caller's tensors are never written."""
        rms = self.obs_rms
        rms.refresh()
        dev = self._flat.device
        out = list(states)
        for s in rms.slots:
            if s >= len(out):
                break                   # _obs_ptrs reports the missing slot
            x = out[s] if torch.is_tensor(out[s]) else torch.as_tensor(np.asarray(out[s]))
            x = x.to(device=dev, dtype=torch.float32).contiguous()
            B = x.shape[0] if x.dim() else 0
            if x.dim() == 0 or x.numel() != B * rms.dims[s]:
                raise DDRLError("state slot %d has shape %s; expected [B=%d, %d elements/sample]" % (s, tuple(x.shape), B, rms.dims[s]))
            buf = bufs.get(s)
            if buf is None or buf.shape[0] < B or buf.shape[1:] != x.shape[1:]:
                buf = bufs[s] = torch.empty(x.shape, dtype=torch.float32, device=dev)
            out[s] = rms.normalize(s, x, buf[:B])
        return out

    # ------------------------------------------------------------------ Forward module
    @_on_device
    def act(self, states, draw=None, play_mode=False, want_pi=False):
        """Fused compute body of ForwardThread.run (server/forward.py:128-146).

        draw: uniforms [B] (categorical), standard normals [B,A] (gaussian), uniforms [B,A] (beta) or uniforms [B,K]
        (multi-categorical, K branches); generated on the device when None and not play_mode.  Returns (actions [B] | [B,A] |
        [B,K], logps [B], values [V,B,1][, pi]); V = number of critics (1 unless add_critic was called); pi = probs [B,A], mu
        [B,A], alpha | beta [B,2A] or the per-branch probabilities [B,A] (A = sum n_i)."""
        self._ensure_engine()
        lib = _lib.load()
        if self.obs_rms is not None:
            states = self._normalized_obs(states, self._obs_act)
        if self.value_rms is not None:
            self.value_rms.refresh()
        keep, arr, n_obs, B = self._obs_ptrs(states)
        dev = self._flat.device
        A = self._act_dim()
        dist_name = self.actor.DIST
        if play_mode:
            draw = None
        elif draw is None and dist_name == "categorical":
            draw = torch.rand(B, device=dev)
        elif draw is None and dist_name == "multi_categorical":
            draw = torch.rand(B, len(self.actor.nvec), device=dev)
        elif draw is None:
            draw = (torch.randn if dist_name == "gaussian" else torch.rand)(B, A, device=dev)
        else:
            draw = draw.to(device=dev, dtype=torch.float32).contiguous()
        shape = (B,) if dist_name == "categorical" else ((B, len(self.actor.nvec)) if dist_name == "multi_categorical" else (B, A))
        actions = torch.empty(shape, dtype=torch.float32, device=dev)
        logps = torch.empty(B, dtype=torch.float32, device=dev)
        V = len(self._critics)
        values = torch.empty(V, B, dtype=torch.float32, device=dev)       # shared mode: the engine fills all V rows
        pi = torch.empty((B, 2 * A if dist_name == "beta" else A), dtype=torch.float32, device=dev) if want_pi else None
        check(lib.ddrl_net_forward(self._h, arr, n_obs, B, ptr(draw), ptr(actions), ptr(logps), ptr(values), ptr(pi),
                                   current_stream()), "ddrl_net_forward")
        if V > 1 and self.prenet is None:                                  # unshared: each extra critic on its own engine
            for k in range(V - 1):
                values[1 + k] = self._aux_net(k).act(keep, play_mode=True)[2].view(B)
        out = (actions, logps, values.view(V, B, 1))
        return out + (pi,) if want_pi else out

    @_on_device
    def encode(self, states, tower=0):
        """Features [B, feat] of one encoder tower (0 = prenet / actor.pre, 1 = critic.pre): the stand-alone encoder
        forward of the reference (nn/atari_encoder.py:25-32, nn/nav_encoder.py:35-43,115-128).  NORM_OBS normalises first."""
        self._ensure_engine()
        if self.obs_rms is not None:
            states = self._normalized_obs(states, self._obs_act)
        keep, arr, n_obs, B = self._obs_ptrs(states)
        out = torch.empty(B, self.actor.actor_linear.in_features, dtype=torch.float32, device=self._flat.device)
        check(_lib.load().ddrl_net_encode(self._h, arr, n_obs, B, int(tower), ptr(out), current_stream()), "ddrl_net_encode")
        return out

    def forward(self, states, act=None, play_mode=False):
        """Reference-shaped output: ((pi, log_p), [values [B,1]]) with pi = Categorical / Normal, or the raw
        softmax / mu tensor in play mode (nn/actor.py:58-67,90-98).  BetaActor: the Beta mapped onto the bounds
        (BetaActor.distribution), or the mean action [B,A] in play mode.  MultiCategoricalActor: a MultiCategorical (one
        Categorical per branch), or the per-branch softmax [B, sum n] in play mode.  ACTION_MASK: the engine's softmax is the
        masked one, so the Categorical gives masked actions probability 0."""
        mean, _, values, pi_raw = self.act(states, draw=None, play_mode=True, want_pi=True)
        if self.actor.DIST == "categorical":
            pi = pi_raw if play_mode else Categorical(pi_raw)
        elif self.actor.DIST == "multi_categorical":
            from .actor import MultiCategorical
            pi = pi_raw if play_mode else MultiCategorical(pi_raw, self.actor.nvec)
        elif self.actor.DIST == "beta":
            pi = mean if play_mode else self.actor.distribution(pi_raw)
        else:
            pi = pi_raw if play_mode else Normal(pi_raw, torch.exp(self.actor.log_std.detach()))
        log_p = None
        if act is not None:
            if play_mode:
                raise DDRLError("log-prob of given actions needs play_mode=False (as in the reference)")
            log_p = self.actor.log_prob_from_distribution(pi, act.to(pi_raw.device))
        return (pi, log_p), [values[k].view(-1, 1) for k in range(values.shape[0])]

    # ------------------------------------------------------------------ Backward module
    def enable_data_parallel(self, group=None, collective=None):
        """Shard each full-batch iteration over the ranks of `group` (one process per GPU): local grads are
        pre-scaled by 1/B_global, one all-reduce(sum) of the flat grad buffer (+ loss sums) per iteration, then the
        identical fused clip+Adam on every rank (SURVEY 8e; ddrl4nav_b200/dist.py).

        collective: "peer" (default; DDRL_DP_COLLECTIVE) = this library's own all-reduce kernel over NVLink / NVSwitch peer
        memory (ddrl_peer_allreduce_f32: the gradient buffer moves into symmetric memory; NVSwitch multicast reduces in the
        switch); "nccl" = torch.distributed's all_reduce.  Falls back to "nccl" -- on every rank together -- when symmetric
        memory cannot be set up (CPU groups, no peer access)."""
        import torch.distributed as tdist
        self._dp_group = group if group is not None else tdist.group.WORLD
        self._dp_world = tdist.get_world_size(self._dp_group)
        self._peer = None
        collective = collective or os.environ.get("DDRL_DP_COLLECTIVE", "peer")
        if self._dp_world > 1 and collective == "peer":
            self._setup_peer_allreduce()

    @_on_device
    def _setup_peer_allreduce(self):
        import torch.distributed as tdist
        self._ensure_engine()
        lib = _lib.load()
        dev = self._flat.device
        ok, st = 1, None
        try:
            import torch.distributed._symmetric_memory as symm_mem
            if self._dp_world > 8:
                raise DDRLError("the peer all-reduce covers the GPUs of one box (<= 8 ranks)")
            g = symm_mem.empty(self._P + 8, dtype=torch.float32, device=dev)
            f = symm_mem.empty(lib.ddrl_peer_allreduce_flag_bytes() // 4, dtype=torch.int32, device=dev)
            g.zero_()
            f.zero_()
            hg = symm_mem.rendezvous(g, self._dp_group)
            hf = symm_mem.rendezvous(f, self._dp_group)
            W = self._dp_world
            st = dict(grads=g, flags=f, handles=(hg, hf), rank=int(hg.rank), world=W, seq=0,
                      bufs=(C.c_void_p * W)(*[int(p) for p in hg.buffer_ptrs]),
                      flag_ptrs=(C.c_void_p * W)(*[int(p) for p in hf.buffer_ptrs]),
                      mc=C.c_void_p(int(hg.multicast_ptr)) if int(hg.multicast_ptr or 0) and os.environ.get("DDRL_DP_MULTICAST", "1") != "0" else None)
        except Exception as e:  # noqa: BLE001
            ok, self._peer_error = 0, repr(e)
        # all ranks take the same path: one rank without symmetric memory sends everybody to NCCL
        t = torch.tensor([ok], dtype=torch.int32, device=dev)
        tdist.all_reduce(t, op=tdist.ReduceOp.MIN, group=self._dp_group)       # also orders the zeroed flags before any kernel
        torch.cuda.synchronize(dev)
        if int(t.item()) != 1:
            return
        st["grads"].copy_(self._grads)
        self._grads = st["grads"]
        check(lib.ddrl_net_bind(self._h, ptr(self._flat), ptr(self._grads), ptr(self._m), ptr(self._v)), "ddrl_net_bind")
        self._peer = st

    def _allreduce_grads(self):
        """Sum of grads[0 : P+4] (P+5 with PPO_STATS, P+6 with PPO_STATS and DECOUPLED_PPO) over the ranks, in place: the
        peer-memory kernel when the buffer is symmetric, else NCCL."""
        st = self._peer
        tail = (6 if self.decoupled else 5) if self.ppo_stats else 4
        if st is not None and st["grads"] is self._grads:
            st["seq"] += 1
            count = (self._P + tail + 3) // 4 * 4              # the buffer holds P + 8 floats
            check(_lib.load().ddrl_peer_allreduce_f32(st["bufs"], st["mc"], st["flag_ptrs"], st["rank"], st["world"], 0, count,
                                                      st["seq"], current_stream()), "ddrl_peer_allreduce_f32")
        else:
            dist.allreduce_grads(self._grads, self._P, self._dp_group, tail)

    @_on_device
    def broadcast_parameters(self, src=0):
        self._ensure_engine()
        dist.broadcast_params(self._flat, src=src, group=self._dp_group)
        self._weights_changed()

    def _bwd_args(self, states, advs, actions, old_logps, returns, b_global, obs_unchanged, allow_empty=False):
        """Device-side argument list shared by ddrl_net_backward / ddrl_net_backward_segment (+ the tensors it points into)."""
        keep, arr, n_obs, B = self._obs_ptrs(states, allow_empty)
        dev = self._flat.device
        f = lambda t: t.to(device=dev, dtype=torch.float32).contiguous()
        advs, actions, old_logps, returns = f(advs), f(actions), f(old_logps), f(returns)
        V = len(self._critics)
        rows = returns if returns.dim() == 2 else returns.view(1, -1)
        if V > 1 and self.prenet is not None:
            # the engine reads returns [V, B]: row 0 = data.values[0] (ppo.py:95), last row = data.values[-1] (ppo.py:102)
            ret = torch.empty(V, B, dtype=torch.float32, device=dev)
            ret[:] = rows[0]
            ret[V - 1] = rows[-1]
            returns = ret
        else:
            returns = rows[0].contiguous()     # data.values is [V,B]; the PPO critic uses row 0 (ppo.py:95)
        args = (self._h, arr, n_obs, B, int(b_global or B), ptr(actions), ptr(old_logps), ptr(advs), ptr(returns),
                C.byref(self.hp), int(bool(obs_unchanged)))
        return args, (keep, advs, actions, old_logps, returns, rows), B

    @_on_device
    def backward_only(self, states, advs, actions, old_logps, returns, b_global=None, obs_unchanged=False, minibatch=False,
                      old_values=None, prox_logps=None):
        """forward + fused loss + backward for the local rows; grads (scaled 1/B_global) stay in flat_grads().
        minibatch: the inputs are the persistent minibatch buffers (ddrl_net_backward_minibatch; 0 rows allowed).
        old_values: critic 0's rollout values [B], needed exactly when VALUE_CLIP is set.
        prox_logps: DECOUPLED_PPO's proximal log-probs [B] (device fp32, read in place), or None for the plain PPO loss.
        This is the engine-level pass: with NORM_OBS it takes `states` as given, so they must already be normalised."""
        self._ensure_engine()
        lib = _lib.load()
        if self.value_rms is not None:
            self.value_rms.refresh()
        args, held, B = self._bwd_args(states, advs, actions, old_logps, returns, b_global, obs_unchanged, minibatch)
        keep, rows = held[0], held[-1]
        dev = self._flat.device
        V = len(self._critics)
        if old_values is not None:
            old_values = old_values.to(device=dev, dtype=torch.float32).contiguous()
        if prox_logps is not None and not self.decoupled:
            raise DDRLError("prox_logps needs DECOUPLED_PPO=True")
        # the old-value pointer goes in before the hyper-parameters (ddrl_net_backward_v / _minibatch_v); DECOUPLED_PPO adds
        # the proximal log-probs and the truncation after it (ddrl_net_backward_dc / _minibatch_dc)
        args = args[:9] + (ptr(old_values),) + args[9:]
        if self.decoupled:
            args = args[:10] + (ptr(prox_logps), float(self.decoupled_is_clip or 0.0)) + args[10:]
            if minibatch:
                check(lib.ddrl_net_backward_minibatch_dc(*args[:-1], current_stream()), "ddrl_net_backward_minibatch_dc")
            else:
                check(lib.ddrl_net_backward_dc(*args, current_stream()), "ddrl_net_backward_dc")
        elif minibatch:
            check(lib.ddrl_net_backward_minibatch_v(*args[:-1], current_stream()), "ddrl_net_backward_minibatch_v")
        else:
            check(lib.ddrl_net_backward_v(*args, current_stream()), "ddrl_net_backward_v")
        if V > 1 and self.prenet is not None:
            self._extra_grads_to_params()
        if V > 1 and self.prenet is None and self.gail_critic:
            # unshared: gailv_loss.backward() only reaches the extra critic's own tower (ppo.py:101-104,122-123)
            k = V - 2
            aux = self._aux_net(k)
            # (a minibatch pass keeps its inputs at fixed addresses: the persistent zeros of the minibatch buffers)
            zeros = self._mb["zeros"][:B] if minibatch else torch.zeros(B, dtype=torch.float32, device=dev)
            aux.backward_only(keep, zeros, zeros, zeros, rows[-1].contiguous(), b_global, obs_unchanged, minibatch)
            if self._dp_world > 1:
                dist.allreduce_grads(aux._grads, aux._P, self._dp_group)      # its loss sum rides in the tail, as ours does
            for n, g in aux.named_grads().items():
                if n.startswith("actor."):
                    continue
                p = dict(aux.named_parameters())[n]
                p.grad = g.clone() if p.grad is None else p.grad.add_(g)
            self._grads[self._P + 1] += aux._grads[aux._P + 1] / (self._dp_world if self._dp_world > 1 else 1)
        return B

    # ------------------------------------------------------------------ data-parallel learner: all-reduce under the backward
    def _segment_runs(self, nseg):
        """Per backward segment k: the contiguous [lo, hi) runs of the flat gradient buffer that are final once segment k has
        run (ddrl_net_tensor_segment); the loss sums in the tail travel with the last segment."""
        if self._seg_runs is None or len(self._seg_runs) != nseg:
            lib = _lib.load()
            sizes = [p.numel() for _, p in self.named_parameters()]
            runs = [[] for _ in range(nseg)]
            for i, (o, sz) in enumerate(zip(self._offsets, sizes)):
                k = min(max(lib.ddrl_net_tensor_segment(self._h, i), 0), nseg - 1)
                if runs[k] and runs[k][-1][1] == o:
                    runs[k][-1][1] = o + sz
                else:
                    runs[k].append([o, o + sz])
            last = runs[nseg - 1]
            if last and last[-1][1] == self._P:
                last[-1][1] = self._P + 4
            else:
                last.append([self._P, self._P + 4])
            self._seg_runs = [[(lo, hi) for lo, hi in r] for r in runs]
        return self._seg_runs

    @_on_device
    def _backward_allreduce(self, data, b_global, obs_unchanged):
        """One iteration's backward + gradient all-reduce of a data-parallel learner.

        Default: the whole backward, then ONE launch of the peer-memory all-reduce kernel (_allreduce_grads).
        DDRL_DP_OVERLAP=1: the backward runs as a chain of segments (ddrl_net_backward_segment); the gradient ranges that are
        final after segment k go to NCCL (its own stream) while segment k + 1 computes, so only the last segment's small
        leftovers are reduced in the open.  Measured on 2 B200s (profiles/r2x_*): no gain -- every kernel of this engine is
        one wave of 148 CTAs with statically assigned tiles, so the SMs NCCL's CTAs occupy stretch the kernel they overlap by
        the collective's own duration; kept as an option for boxes where the collective is the larger term."""
        import torch.distributed as tdist
        if len(self._critics) > 1 or os.environ.get("DDRL_DP_OVERLAP", "0") != "1":
            self.backward_only(data.states, data.advs, data.actions, data.old_logps, data.values, b_global, obs_unchanged)
            self._allreduce_grads()
            return
        self._ensure_engine()
        lib = _lib.load()
        args, held, _ = self._bwd_args(data.states, data.advs, data.actions, data.old_logps, data.values, b_global, obs_unchanged)
        nseg = C.c_int(1)
        works = []
        k = 0
        while True:
            check(lib.ddrl_net_backward_segment(*args, k, C.byref(nseg), current_stream()), "ddrl_net_backward_segment")
            if nseg.value <= 1:
                self._allreduce_grads()
                break
            runs = self._segment_runs(nseg.value)[k]
            if k == nseg.value - 1 and len(runs) > 1:
                # the last segment leaves several small ranges: they travel as ONE message
                parts = [self._grads[lo:hi] for lo, hi in runs]
                packed = torch.cat(parts)
                tdist.all_reduce(packed, group=self._dp_group)
                torch._foreach_copy_(parts, list(packed.split([hi - lo for lo, hi in runs])))
            else:
                for lo, hi in runs:
                    works.append(tdist.all_reduce(self._grads[lo:hi], group=self._dp_group, async_op=True))
            k += 1
            if k >= nseg.value:
                break
        for w in works:
            w.wait()
        del held

    @_on_device
    def optimizer_step(self):
        lib = _lib.load()
        self._adam_step += 1
        check(lib.ddrl_net_clip_adam(self._h, self._adam_step, C.byref(self.hp), ptr(self._loss4), current_stream()),
              "ddrl_net_clip_adam")
        return self._loss4

    def learn(self, data):
        """Generator with the reference's contract (nn/ppo.py:77-142): TRAINING_ITER_TIME full-batch iterations
        over `data` (an Experience whose tensors are on the device), yielding
        ({PpoTotalLoss, ActorLoss, VLoss, EntLoss, PpoBackUpTime}, update_time, True) per iteration.
        MINI_BATCH_NUM = M > 1: TRAINING_ITER_TIME shuffled epochs of M minibatches, one optimiser step and one yield
        per minibatch (_learn_minibatch).
        PPO_STATS adds ApproxKL and ClipFrac to every dict; with TARGET_KL the call ends after the first step whose ApproxKL
        exceeds the target (that step is applied and yielded).
        NORM_OBS: every step sees the observations normalised with the statistics held when the call started (those the
        Forward module acted with); the call's batch is folded into the statistics once, before the final step's yield.
        NORM_VALUE: the call's return targets are folded into critic 0's target statistics once, at the start, and the head
        is rescaled to keep its outputs; every step then learns the targets normalised with the new statistics (PopArt).
        DECOUPLED_PPO: the log-probs of the batch under the parameters at the start of the call (after NORM_VALUE's rescale,
        on the NORM_OBS-normalised batch) are the proximal policy every step clips around; the actor term is weighted by
        exp(prox - old_logps), and PPO_STATS adds BehaviourKL, the mean of (rho - 1) - log rho with rho = exp(prox - old)."""
        if self.mini_batch_num > 1:
            yield from self._learn_minibatch(data)
            return
        b_local = len(data.states[0])
        b_global = b_local
        if self._dp_world > 1:
            self._ensure_engine()
            b_global = dist.global_rows(b_local, self._flat.device, self._dp_group)
        if self.obs_rms is not None:
            data = self._obs_norm_begin(data, b_global)
        if self.value_rms is not None:
            self._value_norm_begin(data, b_global)
        prox = self._decoupled_begin(data) if self.decoupled else None
        options = self.norm_adv or self.value_clip is not None or self.ppo_stats or self.value_rms is not None or self.decoupled
        advs, old_values = self._full_batch_inputs(data) if options else (data.advs, None)
        for it in range(self.training_iter_time):
            start_time = time.time()
            if self._dp_world > 1 and not options:
                self._backward_allreduce(data, b_global, obs_unchanged=it > 0)
            else:
                # the options (NORM_VALUE and DECOUPLED_PPO too) take the whole (not the segmented) backward, as extra critics do
                self.backward_only(data.states, advs, data.actions, data.old_logps, data.values, b_global,
                                   obs_unchanged=it > 0, old_values=old_values, prox_logps=prox)
                if self._dp_world > 1:
                    self._allreduce_grads()
            loss_log = self._step_and_log(start_time)
            stop = self._kl_stop(loss_log)
            if self.obs_rms is not None and (stop or it == self.training_iter_time - 1):
                self._obs_norm_end()
            yield loss_log, self.update_time, True
            if stop:
                return

    @_on_device
    def _obs_norm_begin(self, data, n_global):
        """NORM_OBS at the start of a learn call: the moments of the raw batch around the current running mean (summed over
        the ranks of a data-parallel learner: one collective), and the batch normalised with the current statistics into
        the persistent buffers.  Returns a shallow copy of `data` holding the normalised states."""
        self._ensure_engine()
        rms = self.obs_rms
        raw = {}
        for s in rms.slots:
            if s < len(data.states):
                t = data.states[s]
                t = t if torch.is_tensor(t) else torch.as_tensor(np.asarray(t))
                raw[s] = t.to(device=self._flat.device, dtype=torch.float32).contiguous()
        states = self._normalized_obs([raw.get(i, x) for i, x in enumerate(data.states)], self._obs_learn)
        rms.moments(raw)
        if self._dp_world > 1 and self.value_rms is None:        # with NORM_VALUE its collective carries these sums too
            dist.global_obs_sums(rms.sums, self._dp_group)
        self._obs_n = n_global
        out = copy.copy(data)
        out.states = states
        return out

    @_on_device
    def _obs_norm_end(self):
        self.obs_rms.merge(self._obs_n)

    @_on_device
    def _value_norm_begin(self, data, n_global):
        """NORM_VALUE at the start of a learn call: the moments of critic 0's return targets (data.values[0]) around the
        running mean, summed over the ranks of a data-parallel learner (one collective, shared with NORM_OBS's sums), folded
        into the statistics, and critic 0's head rescaled in the flat parameter buffer so that its unnormalised outputs are
        kept.  Every rank merges the same global sums and rescales the same replicated head: the replicas stay identical.
        The engine reads the head from the flat buffer only, so no re-preparation follows."""
        self._ensure_engine()
        self.value_rms.refresh()
        values = data.values if torch.is_tensor(data.values) else torch.as_tensor(np.asarray(data.values))
        values = values.to(device=self._flat.device, dtype=torch.float32)
        self.value_rms.moments({0: (values if values.dim() == 2 else values.view(1, -1))[0].contiguous()})
        if self._dp_world > 1:
            dist.global_obs_sums(self._norm_sums, self._dp_group)
        off = dict(zip((n for n, _ in self.named_parameters()), self._offsets))
        w, b = (self._flat[off["critic.critic_linear." + k]:][:p.numel()]
                for k, p in (("weight", self.critic.critic_linear.weight), ("bias", self.critic.critic_linear.bias)))
        self.value_rms.merge(n_global, w, b)

    @_on_device
    def _decoupled_begin(self, data):
        """DECOUPLED_PPO at the start of a learn call: the log-probs of the local rows' actions under the current parameters
        (ddrl_net_log_prob, the backward's training forward and the loss kernels' log-prob) into the persistent buffer
        last_prox_logps.  Per row: a data-parallel learner needs no collective."""
        self._ensure_engine()
        dev = self._flat.device
        b = len(data.states[0])
        if self.last_prox_logps is None or self.last_prox_logps.numel() != b or self.last_prox_logps.device != dev:
            self.last_prox_logps = torch.empty(b, dtype=torch.float32, device=dev)
        actions = data.actions if torch.is_tensor(data.actions) else torch.as_tensor(np.asarray(data.actions))
        return kernels.net_log_prob(self, data.states, actions, out=self.last_prox_logps)

    def _step_and_log(self, start_time):
        """clip+Adam, then the loss dict of the step from ONE D2H copy (reference: four .item())."""
        loss = self.optimizer_step().tolist()
        self.update_time += 1
        loss_log = {"PpoTotalLoss": loss[0], "ActorLoss": loss[1], "VLoss": loss[2], "EntLoss": loss[3],
                    "PpoBackUpTime": time.time() - start_time}
        if self.ppo_stats:
            loss_log["ApproxKL"] = loss[4]
            loss_log["ClipFrac"] = loss[5]
            if self.decoupled:
                loss_log["BehaviourKL"] = loss[6]
        return loss_log

    def _kl_stop(self, loss_log):
        # every rank of a data-parallel learner holds the same all-reduced ApproxKL, so all of them stop at the same step
        return self.target_kl is not None and loss_log["ApproxKL"] > self.target_kl

    def _old_values(self, data, advs, values):
        """Critic 0's rollout values for VALUE_CLIP: data.old_values when the batch carries them, else values[0] - advs from
        the raw advantages (the GAE of agent/gae.py makes returns = values + g and advs = g[0])."""
        ov = getattr(data, "old_values", None)
        if ov is not None:
            return ov.to(device=self._flat.device, dtype=torch.float32).contiguous()
        return values[0] - advs

    def _normalize_advs(self, adv, out):
        """NORM_ADV: out = (adv - mean) / (std + 1e-8) over the rows of the global step (all ranks' rows)."""
        m3 = None
        if self._dp_world > 1:
            if self._m3 is None or self._m3.device != adv.device:
                self._m3 = torch.zeros(3, dtype=torch.float64, device=adv.device)
            m3 = dist.global_moments(kernels.adv_moments(adv, self._m3), self._dp_group)
        kernels.adv_normalize(adv, m3, 1e-8, out)

    @_on_device
    def _full_batch_inputs(self, data):
        """(advantages, old values) of a full-batch learn call with the PPO options: the advantages normalised once into a
        persistent buffer (the caller's data.advs is never written) and the old values of VALUE_CLIP."""
        self._ensure_engine()
        dev = self._flat.device
        advs = data.advs.to(device=dev, dtype=torch.float32).contiguous()
        old_values = None
        if self.value_clip is not None:
            values = data.values.to(device=dev, dtype=torch.float32)
            old_values = self._old_values(data, advs, values if values.dim() == 2 else values.view(1, -1))
        if self.norm_adv:
            key = (advs.numel(), dev)
            if self._fb is None or self._fb["key"] != key:
                self._fb = dict(key=key, advs=torch.empty(advs.numel(), dtype=torch.float32, device=dev))
            out = self._fb["advs"]
            self._normalize_advs(advs.view(-1), out)
            advs = out
        return advs, old_values

    # ------------------------------------------------------------------ minibatch epochs (non-reference option)
    @staticmethod
    def minibatch_plan(b_local, m):
        """[lo, hi) of each of the m chunks of one shuffled epoch (positions in the permutation); sizes differ by <= 1."""
        return [dist.shard_rows(b_local, k, m) for k in range(m)]

    def _minibatch_sources(self, data):
        """fp32 contiguous device tensors the minibatch rows are gathered from: state slots, actions, old log-probs,
        advantages, the return rows [V, B], and VALUE_CLIP's old values and DECOUPLED_PPO's proximal log-probs."""
        dev = self._flat.device
        f = lambda t: (t if torch.is_tensor(t) else torch.as_tensor(np.asarray(t))).to(device=dev, dtype=torch.float32).contiguous()
        n_obs = _lib.load().ddrl_net_num_obs(self._h)
        if len(data.states) < n_obs:
            raise DDRLError("expected %d state slots, got %d" % (n_obs, len(data.states)))
        values = f(data.values)
        values = values if values.dim() == 2 else values.view(1, -1)
        src = dict(states=[f(data.states[i]) for i in range(n_obs)], actions=f(data.actions), old_logps=f(data.old_logps),
                   advs=f(data.advs), values=values)
        if self.value_clip is not None:
            src["old_values"] = self._old_values(data, src["advs"], values)     # from the raw advantages, once per call
        if self.decoupled:
            src["prox_logps"] = self.last_prox_logps
        if len(src["states"]) + 3 + values.shape[0] + ("old_values" in src) + ("prox_logps" in src) > _lib.GATHER_MAX_JOBS:
            raise DDRLError("minibatch gather: %d return rows exceed the job limit" % values.shape[0])
        return src

    def _minibatch_buffers(self, src, b_local, mb_rows):
        """Persistent buffers of the largest chunk (smaller chunks use the leading rows).  They keep their addresses while
        b_local, M and the shapes stay the same, which is what lets ddrl_net_backward_minibatch replay its graph."""
        dev = self._flat.device
        key = (b_local, self.mini_batch_num, dev, tuple(tuple(t.shape[1:]) for t in src["states"]), tuple(src["actions"].shape[1:]),
               src["values"].shape[0], "old_values" in src, "prox_logps" in src)
        if self._mb is None or self._mb["key"] != key:
            rows = max(mb_rows, 1)
            e = lambda *shape: torch.empty(shape, dtype=torch.float32, device=dev)
            self._mb = dict(key=key, states=[e(rows, *t.shape[1:]) for t in src["states"]],
                            actions=e(rows, *src["actions"].shape[1:]), old_logps=e(rows), advs=e(rows),
                            values=e(src["values"].shape[0] * rows), zeros=torch.zeros(rows, dtype=torch.float32, device=dev))
            for name in ("old_values", "prox_logps"):
                if name in src:
                    self._mb[name] = e(rows)
        return self._mb

    @_on_device
    def _gather_minibatch(self, src, rows):
        """Gathers the rows `rows` (int32 device) of every source into the minibatch buffers in ONE launch, then normalises
        the gathered advantages in place (NORM_ADV); returns the (states, advs, actions, old_logps, returns [V, n],
        old_values | None, prox_logps | None) views backward_only takes."""
        mb, n = self._mb, rows.numel()
        V = src["values"].shape[0]
        ret = mb["values"][:V * n]
        if n:
            pairs = [(s, d) for s, d in zip(src["states"], mb["states"])]
            pairs += [(src["actions"], mb["actions"]), (src["old_logps"], mb["old_logps"]), (src["advs"], mb["advs"])]
            pairs += [(src["values"][v], ret[v * n:(v + 1) * n]) for v in range(V)]
            for name in ("old_values", "prox_logps"):
                if name in src:
                    pairs.append((src[name], mb[name]))
            kernels.gather_rows(rows, pairs)
        if self.norm_adv:
            self._normalize_advs(mb["advs"][:n], mb["advs"][:n])   # in place: the buffers keep their graph-replay addresses
        old_values = mb["old_values"][:n] if "old_values" in src else None
        prox_logps = mb["prox_logps"][:n] if "prox_logps" in src else None
        return ([t[:n] for t in mb["states"]], mb["advs"][:n], mb["actions"][:n], mb["old_logps"][:n], ret.view(V, n), old_values,
                prox_logps)

    def _learn_minibatch(self, data):
        """TRAINING_ITER_TIME epochs; each draws a permutation of the local rows (net-owned generator) and cuts it into
        M chunks; per chunk: gather, backward, all-reduce (data-parallel), clip+Adam, yield.  Data-parallel: global
        minibatch k is chunk k of every rank; its B_global is the sum of the ranks' chunk-k sizes."""
        m = self.mini_batch_num
        b_local = len(data.states[0])
        if self._dp_world == 1 and m > b_local:
            raise DDRLError("MINI_BATCH_NUM=%d exceeds the %d rows of the batch" % (m, b_local))
        self._ensure_engine()
        dev = self._flat.device
        plan = self.minibatch_plan(b_local, m)
        sizes = [hi - lo for lo, hi in plan]
        b_globals = dist.global_chunk_rows(sizes, dev, self._dp_group) if self._dp_world > 1 else sizes
        if self.obs_rms is not None:
            data = self._obs_norm_begin(data, sum(b_globals))       # the gathers then read the normalised batch
        if self.value_rms is not None:
            self._value_norm_begin(data, sum(b_globals))
        if self.decoupled:
            self._decoupled_begin(data)
        src = self._minibatch_sources(data)
        self._minibatch_buffers(src, b_local, max(sizes))
        if self._mb_gen is None or self._mb_gen.device != dev:
            if self._mb_seed is None:           # MINI_BATCH_SEED=None: drawn once from torch's default generator
                self._mb_seed = int(torch.randint(0, 2 ** 62, (1,)).item())
            self._mb_gen = torch.Generator(device=dev)
            self._mb_gen.manual_seed(self._mb_seed)
        self.last_minibatch_perms = []
        for epoch in range(self.training_iter_time):
            perm = torch.randperm(b_local, generator=self._mb_gen, device=dev, dtype=torch.int32)
            self.last_minibatch_perms.append(perm)
            for k, ((lo, hi), b_global) in enumerate(zip(plan, b_globals)):
                start_time = time.time()
                states, advs, actions, old_logps, returns, old_values, prox = self._gather_minibatch(src, perm[lo:hi])
                self.backward_only(states, advs, actions, old_logps, returns, b_global, minibatch=True, old_values=old_values,
                                   prox_logps=prox)
                if self._dp_world > 1:
                    self._allreduce_grads()
                loss_log = self._step_and_log(start_time)
                stop = self._kl_stop(loss_log)
                if self.obs_rms is not None and (stop or (epoch == self.training_iter_time - 1 and k == m - 1)):
                    self._obs_norm_end()
                yield loss_log, self.update_time, True
                if stop:
                    return

    def add_critic(self, critic):
        """nn/ppo.py:63-64.  The extra critic's values come back from forward()/act() as further rows; its value loss joins
        VLoss when `gail_critic` is set (ppo.py:101-104), with the gradient flowing where the reference's autograd sends it:
        through the shared encoder in share-CNN mode, into the critic's own encoder otherwise.  As in the reference, none of
        PPO's optimisers steps the extra critic (they are built before add_critic, ppo.py:40-42): its gradients accumulate
        in `.grad` for whoever owns it (nn/GAIL.py)."""
        if len(self._critics) >= 3:
            raise DDRLError("at most 3 critics (nn/ppo.py:93)")
        if (self.prenet is not None) != (critic.pre is None):
            raise DDRLError("an extra critic carries its own encoder exactly when SHARE_CNN_NET is off (runner/utils.py:162)")
        self._critics.append(critic)
