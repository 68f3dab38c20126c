"""`Basenn` / `PreNet` with the reference's interface (USTC_lab/nn/base.py:23-153).

Weight (de)serialisation keeps the reference's wire format (base.py:38-54): for every
``named_parameters()`` entry, in order, ``>I ndim | >I*ndim shape | raw fp32 bytes``.  Unlike
the reference (one ``.cpu()`` and one ``bytes +=`` per parameter) the blob is produced from a
single device->host copy of the flat parameter buffer.  A subclass may append further records
in the same format after the parameters (``_state_records``): ``PPO`` does so for its NORM_OBS statistics only.
"""
import struct

import numpy as np
import torch
import torch.nn


class Basenn(torch.nn.Module):
    def __init__(self, config, config_nn):
        super().__init__()
        self.conn = self._connect_redis(getattr(config, "MIDDLE_REDIS_HOST", None), getattr(config, "MIDDLE_REDIS_PORT", None))
        self.pipe = self.conn.pipeline() if self.conn is not None else None
        self.model_key = getattr(config, "TASK_NAME", "") + getattr(config, "MODULE_KEY", "MODEL")
        self.device = getattr(config, "DEVICE", "cuda")
        self.model_dtype = getattr(config_nn, "MODULE_NUMPY_DTYPE", np.float32)
        self.model_dtype_bytes = getattr(config_nn, "MODULE_BITS", 32) // 8
        self.model_tensor_dtype = getattr(config_nn, "MODULE_TENSOR_DTYPE", torch.float32)

    def _connect_redis(self, host, port):
        try:
            import redis
        except ImportError:            # no redis client installed: weight sync needs an injected connection
            return None
        return redis.Redis(host=host, port=port)

    # -- wire format (base.py:38-54) --------------------------------------------------------
    def _encode_wb(self, wb_np: np.ndarray) -> bytes:
        shape = wb_np.shape
        return struct.pack(">I", len(shape)) + struct.pack(">%dI" % len(shape), *shape) + wb_np.tobytes()

    def _decode_wb(self, wb_bytes):
        ndim = struct.unpack_from(">I", wb_bytes, 0)[0]
        shape = struct.unpack_from(">%dI" % ndim, wb_bytes, 4)
        count = int(np.prod(shape)) if ndim else 1
        head = 4 + 4 * ndim
        wb = np.frombuffer(wb_bytes, dtype=self.model_dtype, offset=head, count=count).reshape(shape)
        return wb, head + count * self.model_dtype_bytes

    def _params_to_host(self):
        """[(name, np.ndarray)] in named_parameters() order; subclasses with a flat buffer override."""
        return [(k, v.detach().cpu().numpy()) for k, v in self.named_parameters()]

    def _state_records(self):
        """[np.ndarray] written after the parameter records, in the same record format (none here)."""
        return []

    def _load_state_records(self, view):
        """Reads what _state_records wrote from `view`, the bytes after the parameter records (nothing here)."""

    def model_bytes(self) -> bytes:
        return b"".join(self._encode_wb(a) for a in [a for _, a in self._params_to_host()] + self._state_records())

    def nn2redis(self, pipe, update_key, key=None):
        pipe.set(key if key else self.model_key, self.model_bytes())
        pipe.incr(update_key)
        pipe.execute()

    def load_model_bytes(self, model_bytes):
        view = memoryview(model_bytes)
        index = 0
        with torch.no_grad():
            for _, p in self.named_parameters():
                wb, used = self._decode_wb(view[index:])
                index += used
                p.copy_(torch.from_numpy(np.ascontiguousarray(wb)).to(p.device))
        self._load_state_records(view[index:])
        self._weights_changed()

    def updatenn_by_redis(self, conn, key=None):
        self.load_model_bytes(conn.get(key if key else self.model_key))

    def updatenn_by_file(self, file_path: str):
        self.load_state_dict(torch.load(file_path))
        self._weights_changed()

    def updatenn(self, path: str, conn=None):
        if path.startswith("redis"):
            assert conn is not None
            self.updatenn_by_redis(conn, path.split("://")[-1])
        elif path.startswith("file"):
            self.updatenn_by_file(path.split("://")[-1])

    def _weights_changed(self):
        pass

    def states_normalization(self, states):
        pass

    def imitation_learning(self, *args, **kwargs):
        raise NotImplementedError("imitation pre-training is outside the B200 hot path (SURVEY 2 #1: keep the "
                                  "reference's nn/base.py:109-150 for it)")


class PreNet(torch.nn.Module):
    """Encoder base.  Encoders own parameters (names/shapes/init = reference) and a static description of their
    family; the arithmetic runs in the CUDA engine.  ``forward(states) -> [B, 512]`` is the stand-alone encoder call of
    the reference (nn/atari_encoder.py:25-32, nn/nav_encoder.py:35-43,66-79,115-128, nn/mlp_encoder.py:24-29): inside a
    ``PPO`` it runs on that net's engine (``ddrl_net_encode`` on the owning tower), on its own it keeps a private
    inference-only engine fed from its current parameters.  No PyTorch fallback: CPU parameters raise."""
    ARCH = None

    def __init__(self):
        super().__init__()
        object.__setattr__(self, "_owner_ref", None)      # weakref to the PPO whose engine holds this tower
        object.__setattr__(self, "_tower", 0)
        object.__setattr__(self, "_solo", None)           # (handle, flat buffer, [(offset, param)]) of the private engine

    def engine_in_ch(self) -> int:
        raise NotImplementedError

    def _attach(self, owner, tower: int):
        import weakref
        object.__setattr__(self, "_owner_ref", weakref.ref(owner))
        object.__setattr__(self, "_tower", tower)

    def _feat(self) -> int:
        last = [m for m in self.modules() if isinstance(m, torch.nn.Linear)][-1]
        return last.out_features

    def _solo_engine(self, dev):
        import ctypes as C
        from .. import _lib
        from .._lib import DDRLError, NetDesc, check, ptr
        lib = _lib.load()
        plist = list(self.named_parameters())
        if self._solo is not None and self._solo[1].device == dev:
            return self._solo
        if self._solo is not None:
            lib.ddrl_net_destroy(self._solo[0])
        import os
        mode = _lib.GEMM_MODE[os.environ.get("DDRL_GEMM_MODE", "tc3")]
        desc = NetDesc(_lib.ARCH[self.ARCH], self.engine_in_ch(), 1, _lib.DIST["categorical"], 1, self._feat(), mode, 0)
        h = C.c_void_p()
        check(lib.ddrl_net_create(C.byref(desc), C.byref(h)), "ddrl_net_create")
        name, shape, ndim, off = C.create_string_buffer(128), (C.c_int64 * 4)(), C.c_int(), C.c_int64()
        table = []
        for i, (pname, p) in enumerate(plist):                       # shared-mode table starts with "prenet." + our names
            check(lib.ddrl_net_tensor_info(h, i, name, 128, shape, C.byref(ndim), C.byref(off)), "ddrl_net_tensor_info")
            if name.value.decode() != "prenet." + pname or tuple(shape[k] for k in range(ndim.value)) != tuple(p.shape):
                lib.ddrl_net_destroy(h)
                raise DDRLError("encoder parameter %d (%s%s) does not match the engine's table entry %s" %
                                (i, pname, tuple(p.shape), name.value.decode()))
            table.append((off.value, p))
        with torch.cuda.device(dev):
            flat = torch.zeros(lib.ddrl_net_num_params(h), dtype=torch.float32, device=dev)
            check(lib.ddrl_net_bind(h, ptr(flat), None, None, None), "ddrl_net_bind")
        object.__setattr__(self, "_solo", (h, flat, table))
        return self._solo

    def __del__(self):
        try:
            if self._solo is not None:
                from .. import _lib
                _lib.load().ddrl_net_destroy(self._solo[0])
        except Exception:
            pass

    def forward(self, states):
        import ctypes as C
        from .. import _lib
        from .._lib import DDRLError, check, ptr
        owner = self._owner_ref() if self._owner_ref is not None else None
        if owner is not None:
            return owner.encode(states, self._tower)
        p0 = next(self.parameters())
        if p0.device.type != "cuda":
            raise DDRLError("%s.forward needs its parameters on a CUDA device (got %s); there is no PyTorch fallback"
                            % (type(self).__name__, p0.device))
        lib = _lib.load()
        dev = p0.device
        h, flat, table = self._solo_engine(dev)
        with torch.no_grad():
            for off, p in table:
                flat[off:off + p.numel()].copy_(p.detach().reshape(-1))
        check(lib.ddrl_net_params_changed(h), "ddrl_net_params_changed")
        if torch.is_tensor(states):
            states = [states]
        with torch.cuda.device(dev):
            n_obs = lib.ddrl_net_num_obs(h)
            keep = [torch.as_tensor(s).to(device=dev, dtype=torch.float32).contiguous() for s in states[:n_obs]]
            if len(keep) < n_obs:
                raise DDRLError("expected %d state slots, got %d" % (n_obs, len(keep)))
            B = keep[0].shape[0]
            for i, t in enumerate(keep):
                if t.shape[0] != B or t.numel() // max(B, 1) != lib.ddrl_net_obs_elems(h, i):
                    raise DDRLError("state slot %d has shape %s; expected [B=%d, %d elements/sample]" %
                                    (i, tuple(t.shape), B, lib.ddrl_net_obs_elems(h, i)))
            out = torch.empty(B, self._feat(), dtype=torch.float32, device=dev)
            arr = (C.c_void_p * n_obs)(*[t.data_ptr() for t in keep])
            check(lib.ddrl_net_encode(h, arr, n_obs, B, 0, ptr(out), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)),
                  "ddrl_net_encode")
        return out
