"""Host-side mirror of the reference's pixel encoder over librlrep_b200.so's `rlrep_conv_encoder_*` entry points.

`ConvEncoder` stands in for `Encoder` + `RandomShiftsAug` of agent/diffsrdrq/network_arch/drqv2.py:21-57,138-167 (the
same stack is agent/mulvdrq/drqv2.py:19-96): uint8 frame stacks in, flattened 32x35x35 features out, and the backward
pass that autograd would run.  It is the first building block of the pixel agents (kernel K15 of SURVEY.md); the agents
themselves are not assembled yet.  No fallback: without the CUDA library / a device the constructor raises.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib


def _frames_arg(t):
    """A uint8 frame stack as (keep-alive object, pointer).  CUDA tensors -- batches assembled by the device-resident
    replay ring (rlrep_b200.PixelReplayBuffer) -- are handed over by device pointer: the C update recognises device memory
    and copies it device-to-device instead of staging it over PCIe.  Anything else becomes a contiguous host array."""
    if isinstance(t, torch.Tensor) and t.is_cuda:
        t = t.contiguous()
        assert t.dtype == torch.uint8, "frame stacks must be uint8 like the reference's buffers"
        return t, t.data_ptr()
    a = np.ascontiguousarray(torch.as_tensor(t).cpu().numpy())
    assert a.dtype == np.uint8, "frame stacks must be uint8 like the reference's buffers"
    return a, a.ctypes.data


def _obs_batch(obs, obs_shape):
    """Observations [N, *obs_shape] uint8 -- numpy, a CPU tensor or a CUDA tensor -- as (keep-alive, pointer, N).  Wrong
    dtypes and shapes raise ValueError here, before anything reaches the device."""
    t = obs if isinstance(obs, torch.Tensor) else torch.as_tensor(np.asarray(obs))
    if t.dtype != torch.uint8:
        raise ValueError(f"observations must be uint8 frame stacks, got {t.dtype}")
    if t.dim() != 1 + len(obs_shape) or tuple(t.shape[1:]) != tuple(obs_shape) or t.shape[0] == 0:
        raise ValueError(f"observations must have shape [N, {', '.join(map(str, obs_shape))}] with N >= 1, "
                         f"got {tuple(t.shape)}")
    keep, ptr = _frames_arg(t)
    _sync_if_cuda(keep)
    return keep, ptr, int(t.shape[0])


def _act_noise(n, action_dim, sample, explore=False):
    """Host draws of n consecutive single acts, in their order.  Per observation: `torch.normal(zeros(1, A), ones(1, A))`
    when sampling (TruncatedNormal.sample's _standard_normal), then, in muLV-Rep's exploration phase, the `uniform_(-1, 1)`
    of [A] that replaces the action.  One [n, A] draw would consume the generator differently.
    Returns (eps [n, A] float32 or None, uniform [n, A] float32 or None)."""
    eps = np.empty((n, action_dim), dtype=np.float32) if sample else None
    uni = np.empty((n, action_dim), dtype=np.float32) if explore else None
    for i in range(n):
        if sample:
            z = torch.zeros(1, action_dim)
            eps[i] = torch.normal(z, torch.ones_like(z)).numpy()[0]
        if explore:
            uni[i] = torch.empty(action_dim).uniform_(-1.0, 1.0).numpy()
    return eps, uni


def _host_f32(t):
    return np.ascontiguousarray(torch.as_tensor(t).detach().cpu().numpy(), dtype=np.float32).reshape(-1)


def _sync_if_cuda(*ts):
    if any(isinstance(t, torch.Tensor) and t.is_cuda for t in ts):
        torch.cuda.current_stream().synchronize()  # the C library reads the tensors on its own stream


class ConvEncoder:
    LAYERS = ("convnet.0", "convnet.2", "convnet.4", "convnet.6")

    def __init__(self, obs_shape=(9, 84, 84), batch=256, precision="tf32"):
        if not torch.cuda.is_available():
            raise _lib.RlrepError("rlrep_b200.ConvEncoder needs a CUDA device (there is no CPU fallback)")
        c, h, w = obs_shape
        if h != w:
            raise ValueError("square frames only (RandomShiftsAug asserts h == w, drqv2.py:30)")
        self.lib = _lib.load()
        self.obs_shape, self.batch = (int(c), int(h), int(w)), int(batch)
        self._stream = torch.cuda.Stream()
        self._h = C.c_void_p()
        _lib.check(self.lib.rlrep_conv_encoder_create(self.batch, int(c), int(h), _lib.PRECISION[precision],
                                                      self._stream.cuda_stream, C.byref(self._h)))
        d = C.c_int()
        _lib.check(self.lib.rlrep_conv_encoder_feature_dim(self._h, C.byref(d)))
        self.repr_dim = d.value

    def close(self):
        h, self._h = self._h, None
        if h:
            self.lib.rlrep_conv_encoder_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _shape(self, layer, bias):
        cin = self.obs_shape[0] if layer == 0 else 32
        return (32,) if bias else (32, cin, 3, 3)

    def _read(self, layer, what):
        out = np.empty(self._shape(layer, what in (1, 3)), dtype=np.float32)
        _lib.check(self.lib.rlrep_conv_encoder_read(self._h, layer, what, out.ctypes.data))
        return torch.from_numpy(out)

    def state_dict(self):
        sd = {}
        for i, name in enumerate(self.LAYERS):
            sd[name + ".weight"], sd[name + ".bias"] = self._read(i, 0), self._read(i, 1)
        return sd

    def grads(self):
        g = {}
        for i, name in enumerate(self.LAYERS):
            g[name + ".weight"], g[name + ".bias"] = self._read(i, 2), self._read(i, 3)
        return g

    def load_state_dict(self, sd):
        for i, name in enumerate(self.LAYERS):
            for what, key in ((0, ".weight"), (1, ".bias")):
                arr = np.ascontiguousarray(torch.as_tensor(sd[name + key]).detach().cpu().float().numpy())
                if arr.shape != self._shape(i, what == 1):
                    raise ValueError(f"{name + key}: expected {self._shape(i, what == 1)}, got {arr.shape}")
                _lib.check(self.lib.rlrep_conv_encoder_write(self._h, i, what, arr.ctypes.data))

    def _pitch(self, t, name):
        """Row pitch of fp32 CUDA rows [B, repr_dim] with unit column stride (a view with a wider pitch is used in place,
        as the agents pass their wider feature buffers)."""
        if not (t.is_cuda and t.dtype == torch.float32 and t.dim() == 2 and tuple(t.shape) == (self.batch, self.repr_dim)
                and t.stride(1) == 1 and t.stride(0) >= self.repr_dim):
            raise ValueError(f"{name} must be fp32 CUDA rows [{self.batch}, {self.repr_dim}] with unit column stride")
        return t.stride(0)

    def forward(self, obs: torch.Tensor, shifts: torch.Tensor | None = None, out: torch.Tensor | None = None,
                no_grad: bool = False) -> torch.Tensor:
        """obs uint8 [B, C, H, W] on the GPU; shifts int32 [B, 2] = (x, y) in [0, 8] as drawn by RandomShiftsAug's
        `torch.randint(0, 2 * pad + 1, (n, 1, 1, 2))` (drqv2.py:43-47), or None for no augmentation.  The features go
        to `out` [B, repr_dim] (allocated when None; a view with a wider row pitch is written in place, its padding
        columns untouched).  no_grad=True runs the evaluation-only path; backward() must not follow it."""
        assert obs.is_cuda and obs.dtype == torch.uint8 and tuple(obs.shape) == (self.batch, *self.obs_shape)
        obs = obs.contiguous()
        if shifts is not None:
            shifts = shifts.to(device=obs.device, dtype=torch.int32).reshape(self.batch, 2).contiguous()
        if out is None:
            out = torch.empty(self.batch, self.repr_dim, device=obs.device, dtype=torch.float32)
        ld = self._pitch(out, "out")
        cur = torch.cuda.current_stream()
        self._stream.wait_stream(cur)
        _lib.check(self.lib.rlrep_conv_encoder_forward_pitched(
            self._h, obs.data_ptr(), shifts.data_ptr() if shifts is not None else None, out.data_ptr(), ld, int(no_grad)))
        cur.wait_stream(self._stream)
        self._keep = (obs, shifts, out)
        return out

    def backward(self, dfeat: torch.Tensor) -> None:
        """dfeat [B, repr_dim] (a view with a wider row pitch is read in place).  Raises RlrepError unless the last
        forward ran with gradients."""
        assert dfeat.is_cuda and dfeat.dtype == torch.float32 and tuple(dfeat.shape) == (self.batch, self.repr_dim)
        if dfeat.stride(1) != 1 or dfeat.stride(0) < self.repr_dim:
            dfeat = dfeat.contiguous()
        ld = self._pitch(dfeat, "dfeat")
        cur = torch.cuda.current_stream()
        self._stream.wait_stream(cur)
        _lib.check(self.lib.rlrep_conv_encoder_backward_pitched(self._h, dfeat.data_ptr(), ld))
        cur.wait_stream(self._stream)
        self._keep_d = dfeat

    def hw(self, layer: int) -> int:
        """Side of layer `layer`'s output map (41, 39, 37, 35 for 84-pixel frames)."""
        h = (self.obs_shape[1] - 3) // 2 + 1
        return h - 2 * int(layer)

    def read_map(self, which: str, layer: int) -> torch.Tensor:
        """NCHW copy [B, 32, h, h] of an internal map: 'act' = layer `layer`'s post-ReLU output (last forward), 'dact' =
        the gradient with respect to its pre-activation, ReLU mask applied (last backward)."""
        w = {"act": 0, "dact": 1}[which]
        h = self.hw(layer)
        out = torch.empty(self.batch, 32, h, h, device="cuda")
        cur = torch.cuda.current_stream()
        self._stream.wait_stream(cur)
        _lib.check(self.lib.rlrep_conv_encoder_read_map(self._h, w, int(layer), out.data_ptr()))
        cur.wait_stream(self._stream)
        self._keep_m = out
        return out


class ConvDecoder:
    """The pixel decoder on its own (`rlrep_conv_decoder_*`): muLV-Rep's `Decoder` (agent/mulvdrq/drqv2.py:98-117,
    out_kernel=2) or the latent Diff-SR VAE decoder's convolutions (out_kernel=3), x [B, 32*35*35] -> pred [B, 3, 84, 84],
    its two losses and the backward pass, with the handle's internal maps readable for kernel-level tests."""
    LAYERS = ("deconvnet.0", "deconvnet.2", "deconvnet.4", "deconvnet.6", "deconvnet.8")
    MAPS = {"act": 0, "dact": 1, "pred": 2, "dpred": 3}
    IN_DIM = 32 * 35 * 35

    def __init__(self, batch=256, out_kernel=2, precision="tf32"):
        if not torch.cuda.is_available():
            raise _lib.RlrepError("rlrep_b200.ConvDecoder needs a CUDA device (there is no CPU fallback)")
        self.lib = _lib.load()
        self.batch, self.out_kernel = int(batch), int(out_kernel)
        self.hw = (35, 37, 39, 41, 83 if self.out_kernel == 2 else 84)
        self._stream = torch.cuda.Stream()
        self._h = C.c_void_p()
        _lib.check(self.lib.rlrep_conv_decoder_create(self.batch, self.out_kernel, _lib.PRECISION[precision],
                                                      self._stream.cuda_stream, C.byref(self._h)))
        self._loss = torch.zeros(1, device="cuda")

    def close(self):
        h, self._h = self._h, None
        if h:
            self.lib.rlrep_conv_decoder_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _shape(self, layer, bias):
        if layer == 4:
            return (3,) if bias else (3, 32, self.out_kernel, self.out_kernel)
        return (32,) if bias else (32, 32, 3, 3)

    def _read(self, layer, what):
        out = np.empty(self._shape(layer, what in (1, 3)), dtype=np.float32)
        _lib.check(self.lib.rlrep_conv_decoder_read(self._h, layer, what, out.ctypes.data))
        return torch.from_numpy(out)

    def state_dict(self):
        return {f"{n}.{k}": self._read(i, w) for i, n in enumerate(self.LAYERS) for w, k in ((0, "weight"), (1, "bias"))}

    def grads(self):
        return {f"{n}.{k}": self._read(i, w) for i, n in enumerate(self.LAYERS) for w, k in ((2, "weight"), (3, "bias"))}

    def load_state_dict(self, sd):
        for i, name in enumerate(self.LAYERS):
            for what, key in ((0, ".weight"), (1, ".bias")):
                arr = np.ascontiguousarray(torch.as_tensor(sd[name + key]).detach().cpu().float().numpy())
                if arr.shape != self._shape(i, what == 1):
                    raise ValueError(f"{name + key}: expected {self._shape(i, what == 1)}, got {arr.shape}")
                _lib.check(self.lib.rlrep_conv_decoder_write(self._h, i, what, arr.ctypes.data))

    def _call(self, fn, *args, keep=()):
        cur = torch.cuda.current_stream()
        self._stream.wait_stream(cur)
        _lib.check(fn(self._h, *args))
        cur.wait_stream(self._stream)
        self._keep = keep

    def _rows(self, t, name):
        """[B, >= 32*35*35] fp32 CUDA rows with unit column stride (the row pitch is passed on, as the agents do)."""
        if not (t.is_cuda and t.dtype == torch.float32 and t.dim() == 2 and t.shape[0] == self.batch
                and t.shape[1] == self.IN_DIM and t.stride(1) == 1 and t.stride(0) >= self.IN_DIM):
            raise ValueError(f"{name} must be fp32 CUDA rows [{self.batch}, {self.IN_DIM}] with unit column stride")
        return t.stride(0)

    def forward(self, x: torch.Tensor) -> None:
        """x [B, 32*35*35] (a view with a wider row pitch is read in place)."""
        ld = self._rows(x, "x")
        self._call(self.lib.rlrep_conv_decoder_forward, x.data_ptr(), ld, keep=(x,))

    def l1_loss(self, target: torch.Tensor, grad_scale=1.0) -> float:
        assert target.is_cuda and target.dtype == torch.uint8 and tuple(target.shape) == (self.batch, 3, 84, 84)
        target = target.contiguous()
        self._call(self.lib.rlrep_conv_decoder_l1_loss, target.data_ptr(), float(grad_scale), self._loss.data_ptr(),
                   keep=(target,))
        return self._loss.item()

    def mse_sum_loss(self, target: torch.Tensor, shifts: torch.Tensor | None = None, grad_scale=1.0) -> float:
        """shifts int32 [B, 2] = (x, y) in [0, 8] (RandomShiftsAug's draw) or None."""
        assert target.is_cuda and target.dtype == torch.uint8 and tuple(target.shape) == (self.batch, 3, 84, 84)
        target = target.contiguous()
        if shifts is not None:
            shifts = shifts.to(device=target.device, dtype=torch.int32).reshape(self.batch, 2).contiguous()
        self._call(self.lib.rlrep_conv_decoder_mse_sum_loss, target.data_ptr(),
                   shifts.data_ptr() if shifts is not None else None, float(grad_scale), self._loss.data_ptr(),
                   keep=(target, shifts))
        return self._loss.item()

    def backward(self, dx: torch.Tensor | None = None) -> torch.Tensor:
        """Fills the parameter gradients and dx [B, 32*35*35] (allocated when None; a view with a wider row pitch is
        written in place, its padding columns untouched)."""
        if dx is None:
            dx = torch.empty(self.batch, self.IN_DIM, device="cuda")
        ld = self._rows(dx, "dx")
        self._call(self.lib.rlrep_conv_decoder_backward, dx.data_ptr(), ld, keep=(dx,))
        return dx

    def read_map(self, which: str, i: int = 0) -> torch.Tensor:
        """'act' / 'dact' i = 0..4 -> [B, 32, h_i, h_i]; 'pred' / 'dpred' -> [B, 3, 84, 84] (NCHW copies)."""
        w = self.MAPS[which]
        shape = (self.batch, 32, self.hw[i], self.hw[i]) if w < 2 else (self.batch, 3, 84, 84)
        out = torch.empty(shape, device="cuda")
        self._call(self.lib.rlrep_conv_decoder_read_map, w, int(i), out.data_ptr(), keep=(out,))
        return out


class _PixelAgent:
    """What the pixel agents share: the device handle behind `rlrep_<_PREFIX>_*`, created by the first call that needs
    it, its tensor index, the weights and gradients under the reference's module names, and checkpoints.  Subclasses set
    `_PREFIX`, `_ALG` (the checkpoint's `alg`), `_config(batch)` (the ctypes config of the handle), `_kind(name)`, the
    layout class of a tensor name, and `_step` when they keep the reference's host step counter."""
    _PREFIX = None
    _ALG = None
    _step = None
    OUTCONV_SHAPE = None  # reference shape of the decoder's output convolution, if the agent has one

    def __init__(self, precision):
        # construction is lazy like the state-based agents: the device handle is created by the first call that needs
        # it (and raises there without a CUDA device -- there is no CPU fallback)
        self._precision = precision
        self.lib = None
        self._h = None
        self._batch = None
        self._pending = {}

    def _fn(self, name):
        return getattr(self.lib, f"rlrep_{self._PREFIX}_{name}")

    # ---- handle ------------------------------------------------------------------------------------------------
    def _ensure(self, batch):
        if self._h is not None:
            if batch != self._batch:
                raise _lib.RlrepError(f"batch size is fixed per handle (was {self._batch}, got {batch})")
            return
        if not torch.cuda.is_available():
            raise _lib.RlrepError(f"rlrep_b200.{type(self).__name__} needs a CUDA device (there is no CPU fallback)")
        self.lib = _lib.load()
        cfg = self._config(batch)
        hd = C.c_void_p()
        _lib.check(self._fn("create")(C.byref(cfg), None, C.byref(hd)))
        self._h, self._batch = hd, batch
        n = C.c_int()
        _lib.check(self._fn("num_tensors")(hd, C.byref(n)))
        self._index = {}
        for i in range(n.value):
            name, ptr, rows, cols = C.c_char_p(), C.c_void_p(), C.c_int(), C.c_int()
            _lib.check(self._fn("tensor_info")(hd, i, C.byref(name), C.byref(ptr), C.byref(rows), C.byref(cols)))
            self._index[name.value.decode()] = (i, rows.value, cols.value)
        if self._pending:
            sd, self._pending = self._pending, {}
            self.load_state_dict(sd)

    def prepare(self, batch_size):
        """Create the device handle for `batch_size` ahead of the first update."""
        self._ensure(int(batch_size))

    def close(self):
        h, self._h = self._h, None
        if h and self.lib is not None:
            self._fn("destroy")(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- weights under the reference's module names ----------------------------------------------------------------
    def _ref_shape(self, name, rows, cols):
        return {"outconv": self.OUTCONV_SHAPE, "deconv": (32, 32, 3, 3), "conv0": (32, cols // 9, 3, 3),
                "conv": (32, cols // 9, 3, 3), "vec": (rows,), "mat": (rows, cols)}[self._kind(name)]

    def _read_all(self, keep):
        sd = {}
        for name, (i, rows, cols) in self._index.items():
            if not keep(name):
                continue
            out = np.empty(rows * cols, dtype=np.float32)
            _lib.check(self._fn("tensor_read")(self._h, i, out.ctypes.data))
            t, kind = torch.from_numpy(out), self._kind(name)
            if kind == "conv":      # stored [32, (ky, kx, c)] -> reference [32, c, ky, kx]
                t = t.reshape(32, 3, 3, 32).permute(0, 3, 1, 2).contiguous()
            elif kind == "deconv":  # stored [(ky, kx, c_out), c_in] -> reference [c_in, c_out, ky, kx]
                t = t.reshape(3, 3, 32, 32).permute(3, 2, 0, 1).contiguous()
            sd[name] = t.reshape(self._ref_shape(name, rows, cols))
        return sd

    def state_dict(self):
        if self._h is None:
            return dict(self._pending)
        return self._read_all(lambda name: not name.startswith(("grad/", "optim.")))

    def grads(self):
        """Gradients left by the most recent update, under the reference's names."""
        return {k[5:]: v for k, v in self._read_all(lambda name: name.startswith("grad/")).items()}

    def _write(self, k, v):
        i, rows, cols = self._index[k]
        t = torch.as_tensor(v).detach().cpu().float()
        if tuple(t.shape) != self._ref_shape(k, rows, cols):
            raise ValueError(f"{k}: expected {self._ref_shape(k, rows, cols)}, got {tuple(t.shape)}")
        kind = self._kind(k)
        if kind == "conv":
            t = t.permute(0, 2, 3, 1)
        elif kind == "deconv":
            t = t.permute(2, 3, 1, 0)
        arr = np.ascontiguousarray(t.reshape(-1).numpy())
        _lib.check(self._fn("tensor_write")(self._h, i, arr.ctypes.data))

    def load_state_dict(self, sd, sync_targets=None):
        """Targets are copied from the loaded parameters unless `sd` carries them (or `sync_targets` says otherwise)."""
        if self._h is None:
            self._pending.update({k: torch.as_tensor(v).detach().clone() for k, v in sd.items()})
            return
        for k, v in sd.items():
            self._write(k, v)
        if sync_targets or (sync_targets is None and not any("_target." in k for k in sd)):
            _lib.check(self._fn("sync_targets")(self._h))

    # ---- checkpoints ---------------------------------------------------------------------------------------------
    def _need_handle(self, what):
        if self._h is None:
            raise _lib.RlrepError(f"{what} needs the device handle: call prepare(batch_size) or run an update first")

    def optimizer_state_dict(self, step=None):
        """Adam moments of every optimised parameter (`optim.m/<name>`, `optim.v/<name>`: torch.optim.Adam's -- for the
        score network AdamW's -- exp_avg / exp_avg_sq of that parameter, in its reference shape and layout) plus `control`:
        the three Adam step counters and `agent_step`, the host step counter that gates `update_every`.  `step` is only
        used by μLV-Rep, which keeps no such counter (its caller owns the step): it becomes `agent_step`, None when not
        given.  DrQ-v2 and latent Diff-SR save their own `_step` and ignore `step`."""
        self._need_handle("optimizer_state_dict")
        sd = self._read_all(lambda name: name.startswith("optim."))
        st = _lib.OptimState()
        _lib.check(self._fn("get_optim_state")(self._h, C.byref(st)))
        sd["control"] = {"t_feature": st.t_feature, "t_critic": st.t_critic, "t_actor": st.t_actor,
                         "agent_step": self._step if self._step is not None else step}
        return sd

    def load_optimizer_state_dict(self, sd):
        """The inverse of optimizer_state_dict: moments are shape-checked like load_state_dict's weights."""
        self._need_handle("load_optimizer_state_dict")
        for k, v in sd.items():
            if k == "control":
                continue
            if not k.startswith("optim.") or k not in self._index:
                raise ValueError(f"{k}: not an optimiser tensor of this agent")
            self._write(k, v)
        ctl = sd["control"]
        st = _lib.OptimState(t_feature=int(ctl["t_feature"]), t_critic=int(ctl["t_critic"]), t_actor=int(ctl["t_actor"]))
        _lib.check(self._fn("set_optim_state")(self._h, C.byref(st)))
        if self._step is not None:
            self._step = int(ctl["agent_step"])

    def save(self, path, step=None):
        """Checkpoint in the state agents' format (rlrep_b200.agents): a torch.save'd dict with the parameters and Polyak
        targets under the reference's state_dict names and the optimiser state that makes a resumed run continue
        bit-identically.  `step` is saved as μLV-Rep's `agent_step` and ignored by the other agents (see
        optimizer_state_dict)."""
        self._need_handle("save")
        torch.save({"format": "rlrep_b200/1", "alg": self._ALG, "obs_shape": self._observation_shape(),
                    "action_dim": self.action_dim, "batch_size": self._batch, "precision": self._precision,
                    "state_dict": self.state_dict(), "optimizer": self.optimizer_state_dict(step)}, path)

    def load(self, path, load_optimizer=True):
        """Restore a checkpoint written by `save`.  An agent without a handle gets one at the checkpoint's batch size; a
        handle of another batch size is refused (the batch size is fixed per handle).  The precision may differ from the
        saved one, but then the run does not continue bit-identically.  With load_optimizer=False only the parameters and
        their saved targets are written: the handle's moments, step counters and host step counter are left as they are
        (zero on a handle that has not updated yet)."""
        ck = torch.load(path, map_location="cpu", weights_only=True)
        if ck.get("format") != "rlrep_b200/1" or ck.get("alg") != self._ALG:
            raise _lib.RlrepError(f"{path}: not a rlrep_b200 checkpoint of a {self._ALG} agent")
        if (tuple(ck["obs_shape"]), ck["action_dim"]) != (self._observation_shape(), self.action_dim):
            raise _lib.RlrepError(f"{path}: saved for observation shape {tuple(ck['obs_shape'])} and action dimension "
                                  f"{ck['action_dim']}, this agent has {self._observation_shape()} and {self.action_dim}")
        self._ensure(int(ck["batch_size"]))
        self.load_state_dict(ck["state_dict"], sync_targets=False)
        if load_optimizer:
            self.load_optimizer_state_dict(ck["optimizer"])

    def _observation_shape(self):
        return self.obs_dim

    @property
    def gpu_launches_last_update(self):
        v = C.c_int()
        _lib.check(self._fn("last_launches")(self._h, C.byref(v)))
        return v.value

    def _act_batch(self, obs, obs_shape, step, sample, explore=False):
        """The handle's act_batch on uint8 observations [N, *obs_shape], with the noise N single acts would draw.
        Returns (actions [N, A], the exploration phase's uniform draws [N, A] or None)."""
        keep, ptr, n = _obs_batch(obs, obs_shape)
        stddev = float(self.stddev_schedule(step))
        eps, uni = _act_noise(n, self.action_dim, sample=sample, explore=explore)
        out = np.empty((n, self.action_dim), dtype=np.float32)
        _lib.check(self._fn("act_batch")(self._h, ptr, eps.ctypes.data if eps is not None else None, stddev, n,
                                         out.ctypes.data))
        del keep
        return out, uni


class DrqConfig(C.Structure):
    """Mirror of `rlrep_drq_config` (include/rlrep_b200.h)."""
    _fields_ = [("batch_size", C.c_int), ("channels", C.c_int), ("height", C.c_int), ("action_dim", C.c_int),
                ("bn_dim", C.c_int), ("hidden_dim", C.c_int), ("encoder_lr", C.c_double), ("actor_lr", C.c_double),
                ("critic_lr", C.c_double), ("tau", C.c_float), ("stddev_clip", C.c_float), ("precision", C.c_int)]


def _schedule(spec):
    """helper_functions/util.py:142-148 `setup_schedule`."""
    import re
    init, final, duration = [float(g) for g in re.match(r"linear\((.+),(.+),(.+)\)", spec).groups()]

    def fn(step):
        mix = np.clip(step / duration, 0.0, 1.0)
        return (1.0 - mix) * init + mix * final
    return fn


class DrQv2(_PixelAgent):
    """Drop-in for the update path of agent.diffsrdrq.drqv2.DrQv2 (drqv2.py:12-148): same constructor
    (`obs_space`, `action_space`, `args` with tau / update_every / critic_loss / stddev_schedule / stddev_clip / bn_dim /
    actor_hidden_dim / critic_hidden_dim / encoder_lr / actor_lr / critic_lr) and `train_step(replay_iter, step)` with the
    reference's metric keys, plus `select_action(obs, step, deterministic)`.  The batch comes from the caller's replay
    iterator as in the reference (img_stack uint8 [B, 9, 84, 84], action, reward, discount, next_img_stack,
    next_img_step)."""
    _PREFIX = "drq"
    _ALG = "drqv2"

    def __init__(self, obs_space, action_space, args, *, precision="tf32"):
        if getattr(args, "critic_loss", "mse") != "mse":
            raise NotImplementedError("critic_loss='huber' (configs/drqv2.yaml ships 'mse')")
        if args.actor_hidden_dim != args.critic_hidden_dim:
            raise NotImplementedError("actor_hidden_dim != critic_hidden_dim")
        super().__init__(precision)
        self.args = args
        self.obs_dim = tuple(int(x) for x in obs_space.shape)
        self.action_dim = int(action_space.shape[0])
        self.tau, self.update_every = float(args.tau), int(args.update_every)
        self.stddev_schedule, self.stddev_clip = _schedule(args.stddev_schedule), float(args.stddev_clip)
        self.bn_dim, self.hidden_dim = int(args.bn_dim), int(args.actor_hidden_dim)
        self._step = 1

    def _config(self, batch):
        c, h, _ = self.obs_dim
        return DrqConfig(batch_size=batch, channels=c, height=h, action_dim=self.action_dim, bn_dim=self.bn_dim,
                         hidden_dim=self.hidden_dim, encoder_lr=float(self.args.encoder_lr),
                         actor_lr=float(self.args.actor_lr), critic_lr=float(self.args.critic_lr), tau=self.tau,
                         stddev_clip=self.stddev_clip, precision=_lib.PRECISION[self._precision])

    @staticmethod
    def _kind(name):
        if ".convnet." in name and name.endswith("weight"):
            return "conv0" if name.endswith("convnet.0.weight") else "conv"
        if name.endswith("bias") or ".trunk.1." in name:
            return "vec"
        return "mat"

    # ---- reference surface ---------------------------------------------------------------------------------------
    def _draw(self, n):
        """RNG consumption of one updating train_step, in the reference's order (SURVEY.md A.5): RandomShiftsAug's
        `torch.randint(0, 9, (n,1,1,2), dtype=float32)` for img then next_img (network_arch/drqv2.py:43-47), then
        `_standard_normal([n, A])` for the next action and for the actor step (TruncatedNormal.sample, :72-75)."""
        shifts = torch.stack([torch.randint(0, 9, size=(n, 1, 1, 2), dtype=torch.float32).reshape(n, 2) for _ in range(2)])
        z = torch.zeros(n, self.action_dim)
        eps = torch.stack([torch.normal(z, torch.ones_like(z)) for _ in range(2)])
        return shifts.to(torch.int32).numpy(), eps.numpy()

    def select_action(self, obs, step, deterministic=False):
        """drqv2.py:74-82.  `obs` is one uint8 frame stack [C, H, W]; the handle must exist (weights loaded after the
        first train_step, or call `prepare(batch_size)` first)."""
        return self.select_actions(torch.as_tensor(obs).unsqueeze(0), step, deterministic)[0]

    def select_actions(self, obs, step, deterministic=False):
        """`select_action` on N observations at once: obs uint8 [N, C, H, W] (numpy, CPU or CUDA tensor) -> actions
        [N, A].  Row i is bit-identical to `select_action(obs[i])`, and the generator advances exactly as N consecutive
        select_action calls advance it."""
        if self._h is None:
            raise _lib.RlrepError("call prepare(batch_size) or train_step once before select_action")
        return self._act_batch(obs, self.obs_dim, step, sample=not deterministic)[0]

    def train_step(self, replay_iter, step):
        self._step += 1
        if self._step % self.update_every != 0:
            return {}
        batch = next(replay_iter)
        n = batch[0].shape[0]
        (img, p_img), (next_img, p_next) = _frames_arg(batch[0]), _frames_arg(batch[4])
        action, reward, discount = _host_f32(batch[1]), _host_f32(batch[2]), _host_f32(batch[3])
        self._ensure(n)
        shifts, eps = self._draw(n)
        stddev = float(self.stddev_schedule(step))
        m = np.zeros(8, dtype=np.float32)
        shifts, eps = np.ascontiguousarray(shifts), np.ascontiguousarray(eps)
        _sync_if_cuda(img, next_img)
        _lib.check(self.lib.rlrep_drq_update(self._h, p_img, action.ctypes.data, reward.ctypes.data,
                                             discount.ctypes.data, p_next, shifts.ctypes.data,
                                             eps.ctypes.data, stddev, m.ctypes.data))
        return {"loss/actor_loss": float(m[4]), "info/policy_std": stddev, "loss/critic_loss": float(m[0]),
                "info/q_pred": float(m[1]), "info/q_target": float(m[2]), "info/reward": float(m[3])}


class MulvConfig(C.Structure):
    """Mirror of `rlrep_mulv_config` (include/rlrep_b200.h)."""
    _fields_ = [("batch_size", C.c_int), ("channels", C.c_int), ("height", C.c_int), ("action_dim", C.c_int),
                ("feat_dim", C.c_int), ("hidden_dim", C.c_int), ("num_noise", C.c_int), ("lr", C.c_double),
                ("tau", C.c_float), ("stddev_clip", C.c_float), ("vae_w", C.c_float), ("mse_w", C.c_float),
                ("c_noise", C.c_float), ("precision", C.c_int)]


def _cfg_get(cfg, key, default=None):
    """mulv_config.py's `config` is an attribute-access dict; plain namespaces work too."""
    if isinstance(cfg, dict):
        return cfg.get(key, default)
    return getattr(cfg, key, default)


class MuLVDrQv2(_PixelAgent):
    """Drop-in for the update path of agent.mulvdrq.drqv2.DrQV2Agent (drqv2.py:198-461): same constructor
    (`obs_shape`, `action_shape`, `cfg` -- the attribute dict of mulv_config.py) and `update(replay_iter, step)`.  Only
    the shipped configuration path is built (aug, no pre_aug, back_q2feat, tanh heads, ReLU critic, Huber loss,
    c_targ_tau < 1, q_up_n = 1, l2_norm = 0); anything else raises.  The batch comes from the caller's replay iterator
    as in the reference: (img uint8 [B, 9, 84, 84], action, reward, discount, next_img, img_step1)."""

    METRICS = ("critic_loss", "critic_q1", "critic_q2", "critic_target_q", "s_loss", "r_loss", "kl_loss", "actor_loss")
    _PREFIX = "mulv"
    _ALG = "mulvdrq"
    OUTCONV_SHAPE = (3, 32, 2, 2)

    def __init__(self, obs_shape, action_shape, cfg, *, precision="tf32"):
        get = lambda k, d=None: _cfg_get(cfg, k, d)
        unsupported = [k for k, want in (("aug", True), ("pre_aug", False), ("back_q2feat", True), ("tanh", True),
                                         ("both_q", False), ("q_activ", "relu"), ("q_loss", "huber"), ("q_up_n", 1),
                                         ("l2_norm", 0.0)) if get(k, want) != want]
        if unsupported or not float(get("c_targ_tau", 0.01)) < 1.0:
            raise NotImplementedError(f"only mulv_config.py's default path is built (differs in: {unsupported})")
        super().__init__(precision)
        self.cfg = cfg
        self.obs_shape = tuple(int(x) for x in obs_shape)
        self.action_dim = int(action_shape[0])
        self.up_every = int(get("up_every", 2))
        self.stddev_schedule = _schedule(get("stddev_schedule", "linear(1.0,0.1,500000)"))
        self.feat_dim, self.hidden_dim, self.num_noise = int(get("feat_dim", 100)), int(get("hid_dim", 1024)), 20

    def _config(self, batch):
        get = lambda k, d: _cfg_get(self.cfg, k, d)
        c, h, _ = self.obs_shape
        return MulvConfig(batch_size=batch, channels=c, height=h, action_dim=self.action_dim, feat_dim=self.feat_dim,
                          hidden_dim=self.hidden_dim, num_noise=self.num_noise, lr=float(get("lr", 1e-4)),
                          tau=float(get("c_targ_tau", 0.01)), stddev_clip=float(get("stddev_clip", 0.3)),
                          vae_w=float(get("vae_w", 0.5)), mse_w=float(get("mse_w", 1.0)),
                          c_noise=float(get("c_noise", 0.1)), precision=_lib.PRECISION[self._precision])

    def _observation_shape(self):
        return self.obs_shape

    # ---- weights under the reference's module names ----------------------------------------------------------------
    @staticmethod
    def _kind(name):
        if name.endswith("weight"):
            if ".deconvnet.8." in name:
                return "outconv"
            if ".deconvnet." in name:
                return "deconv"
            if ".convnet." in name:
                return "conv0" if name.endswith("convnet.0.weight") else "conv"
            if ".trunk.1." in name or "_linear.1." in name:
                return "vec"
            return "mat"
        return "vec"

    # ---- reference surface ---------------------------------------------------------------------------------------
    def _draw(self, n):
        """RNG consumption of one updating `update`, in the reference's order (SURVEY.md A.5): the two shift draws,
        randn[n, F] (feat_encoder.sample, vae.py:50-58), the next action's normals, randn[20, F] for critic_target and for
        critic (drqv2.py:181), the actor step's normals, randn[20, F] for its critic."""
        F, A, NN = self.feat_dim, self.action_dim, self.num_noise
        shifts = torch.stack([torch.randint(0, 9, size=(n, 1, 1, 2), dtype=torch.float32).reshape(n, 2) for _ in range(2)])
        eps_z = torch.randn(n, F)
        za = torch.zeros(n, A)
        e0 = torch.normal(za, torch.ones_like(za))
        n0 = torch.randn(NN, F)
        n1 = torch.randn(NN, F)
        e1 = torch.normal(za, torch.ones_like(za))
        n2 = torch.randn(NN, F)
        return (shifts.to(torch.int32).numpy(), eps_z.numpy(), torch.stack([e0, e1]).numpy(),
                torch.stack([n0, n1, n2]).numpy())

    def act(self, obs, step, eval_mode):
        """drqv2.py:270-282.  `obs` is one uint8 frame stack [C, H, W]; the handle must exist (`prepare(batch_size)` or one
        `update`).  Exploration (`step < num_expl_steps`, not eval_mode) replaces the sample by U(-1, 1) after drawing it,
        like the reference."""
        return self.act_batch(torch.as_tensor(obs).unsqueeze(0), step, eval_mode)[0]

    def act_batch(self, obs, step, eval_mode):
        """`act` on N observations at once: obs uint8 [N, C, H, W] (numpy, CPU or CUDA tensor) -> actions [N, A].  Row i
        is bit-identical to `act(obs[i])`, and the generator advances exactly as N consecutive act calls advance it."""
        if self._h is None:
            raise _lib.RlrepError("call prepare(batch_size) or update once before act")
        explore = not eval_mode and step < int(_cfg_get(self.cfg, "num_expl_steps", 2000))
        out, uni = self._act_batch(obs, self.obs_shape, step, sample=not eval_mode, explore=explore)
        return uni if explore else out

    def update(self, replay_iter, step):
        if step % self.up_every != 0:
            return {}
        batch = next(replay_iter)
        n = batch[0].shape[0]
        self._ensure(n)
        (img, p_img), (next_img, p_next) = _frames_arg(batch[0]), _frames_arg(batch[4])
        step1, p_step1 = _frames_arg(batch[5][:, -3:, :, :])  # drqv2.py:330: only the newest frame is predicted
        action, reward, discount = _host_f32(batch[1]), _host_f32(batch[2]), _host_f32(batch[3])
        shifts, eps_z, eps_act, noise = (np.ascontiguousarray(a) for a in self._draw(n))
        stddev = float(self.stddev_schedule(step))
        m = np.zeros(8, dtype=np.float32)
        _sync_if_cuda(img, next_img, step1)
        _lib.check(self.lib.rlrep_mulv_update(self._h, p_img, action.ctypes.data, reward.ctypes.data,
                                              discount.ctypes.data, p_next, p_step1,
                                              shifts.ctypes.data, eps_z.ctypes.data, eps_act.ctypes.data,
                                              noise.ctypes.data, stddev, m.ctypes.data))
        return {k: float(v) for k, v in zip(self.METRICS, m)}


class LdiffConfig(C.Structure):
    """Mirror of `rlrep_ldiff_config` (include/rlrep_b200.h)."""
    _fields_ = [("batch_size", C.c_int), ("action_dim", C.c_int), ("latent_dim", C.c_int), ("feature_dim", C.c_int),
                ("bn_dim", C.c_int), ("psi_hidden_dim", C.c_int), ("psi_hidden_depth", C.c_int), ("zeta_hidden_dim", C.c_int),
                ("zeta_hidden_depth", C.c_int), ("hidden_dim", C.c_int), ("ae_lr", C.c_double), ("score_lr", C.c_double),
                ("actor_lr", C.c_double), ("critic_lr", C.c_double), ("weight_decay", C.c_double), ("tau", C.c_float),
                ("kl_coef", C.c_float), ("ae_coef", C.c_float), ("stddev_clip", C.c_float), ("precision", C.c_int)]


class LdiffInputs(C.Structure):
    """Mirror of `rlrep_ldiff_inputs`."""
    _fields_ = [(n, C.c_void_p) for n in ("frames", "next_frames", "shifts", "next_shifts", "action", "reward", "discount",
                                          "eps_post", "alphabar", "temb", "noise", "psi_masks", "zeta_masks", "eps_act")] + \
               [("stddev", C.c_float)]


class LatentDiffSRDrQv2(_PixelAgent):
    """Drop-in for the update path of agent.diffsrdrq.latent_diff_sr.LatentDiffSRDrQv2: same constructor
    (`obs_space`, `action_space`, `args`) and `train_step(replay_iter, step)` with the reference's metric keys.  Only
    configs/latent_diff_sr.yaml's path is built (use_repr_target, back_critic_grad, critic_loss mse, reg_coef 0,
    grad_norm null, extra_repr_step 1, do_scale false, repr_coef 1, ae_lr == score_lr)."""
    _PREFIX = "ldiff"
    _ALG = "ldiffsr"
    OUTCONV_SHAPE = (3, 32, 3, 3)

    def __init__(self, obs_space, action_space, args, *, precision="tf32"):
        a = args
        bad = [k for k, want in (("use_repr_target", True), ("back_critic_grad", True), ("critic_loss", "mse"),
                                 ("reg_coef", 0.0), ("grad_norm", None), ("extra_repr_step", 1), ("do_scale", False),
                                 ("repr_coef", 1.0), ("ae_num_layers", 4), ("ae_num_filters", 32),
                                 ("noise_schedule", "linear")) if getattr(a, k, want) != want]
        if bad or float(a.ae_lr) != float(a.score_lr) or a.bn_dim is None:
            raise NotImplementedError(f"only configs/latent_diff_sr.yaml's path is built (differs in: {bad})")
        super().__init__(precision)
        self.args = a
        self.obs_dim = tuple(int(x) for x in obs_space.shape)
        if self.obs_dim != (9, 84, 84):
            raise NotImplementedError("three stacked 3 x 84 x 84 frames")
        self.action_dim = int(action_space.shape[0])
        self.update_every = int(a.update_every)
        self.stddev_schedule = _schedule(a.stddev_schedule)
        self.L, self.feat = int(a.latent_dim), int(a.feature_dim)
        self.psi = (int(a.psi_hidden_dim), int(a.psi_hidden_depth))
        self.zeta = (int(a.zeta_hidden_dim), int(a.zeta_hidden_depth))
        betas = np.linspace(float(a.noise_param1), float(a.noise_param2), int(a.num_noises))  # util.py:118-134
        self.alphabars = torch.as_tensor(np.cumprod(1 - betas, axis=0), dtype=torch.float32)
        self.num_noises = int(a.num_noises)
        self._step = 1

    def _draw(self, n):
        """RNG consumption of one updating train_step in the reference's order (oracle/ldiffsr_oracle.py header)."""
        L, A, keep = self.L, self.action_dim, 0.9
        shifts = [torch.randint(0, 9, size=(n, 1, 1, 2), dtype=torch.float32).reshape(n, 2) for _ in range(2)]
        eps_post = torch.randn(4 * n, L)
        noise_idx = torch.randint(0, self.num_noises, (n,))
        noise = torch.randn(n, L)
        mask = lambda h: torch.empty(n, h).bernoulli_(keep)  # what F.dropout draws (checked in tests/test_host_logic.py)
        psi_score = [mask(self.psi[0]) for _ in range(self.psi[1])]
        zeta = [mask(self.zeta[0]) for _ in range(self.zeta[1])]
        psi_critic = [mask(self.psi[0]) for _ in range(self.psi[1])]
        za = torch.zeros(n, A)
        eps_act = [torch.normal(za, torch.ones_like(za)) for _ in range(2)]
        half = (L // 2) // 2  # SinusoidalPosEmb(latent_dim // 2), score_mlp.py:94-106
        emb = torch.exp(torch.arange(half) * -(np.log(10000) / (half - 1)))
        emb = noise_idx[..., None] * emb[None, :]
        temb = torch.cat((emb.sin(), emb.cos()), dim=-1)
        return dict(shifts=torch.stack(shifts).to(torch.int32).numpy(), eps_post=eps_post.numpy(),
                    alphabar=self.alphabars[noise_idx].numpy(), temb=temb.float().numpy(), noise=noise.numpy(),
                    psi_masks=torch.stack([torch.cat([s, c]) for s, c in zip(psi_score, psi_critic)]).numpy(),
                    zeta_masks=torch.stack(zeta).numpy(), eps_act=torch.stack(eps_act).numpy())

    def _config(self, batch):
        a = self.args
        return LdiffConfig(batch_size=batch, action_dim=self.action_dim, latent_dim=self.L, feature_dim=self.feat,
                           bn_dim=int(a.bn_dim), psi_hidden_dim=self.psi[0], psi_hidden_depth=self.psi[1],
                           zeta_hidden_dim=self.zeta[0], zeta_hidden_depth=self.zeta[1],
                           hidden_dim=int(a.actor_hidden_dim), ae_lr=float(a.ae_lr), score_lr=float(a.score_lr),
                           actor_lr=float(a.actor_lr), critic_lr=float(a.critic_lr), weight_decay=0.01, tau=float(a.tau),
                           kl_coef=float(a.kl_coef), ae_coef=float(a.ae_coef), stddev_clip=float(a.stddev_clip),
                           precision=_lib.PRECISION[self._precision])

    @staticmethod
    def _kind(name):
        if name.endswith("weight"):
            if ".deconvs.8." in name:
                return "outconv"
            if ".deconvs." in name:
                return "deconv"
            if ".convs." in name:
                return "conv0" if name.endswith("convs.0.weight") else "conv"
            if any(s in name for s in (".ln.", ".layer_norm.", "psi_bottleneck1.1.", "psi_bottleneck2.1.", "trunk.1.")):
                return "vec"
            return "mat"
        return "vec"

    def train_step(self, replay_iter, step):
        self._step += 1
        if self._step % self.update_every != 0:
            return {}
        batch = next(replay_iter)
        n = batch[0].shape[0]
        self._ensure(n)
        d = self._draw(n)
        if all(isinstance(t, torch.Tensor) and t.is_cuda for t in (batch[0], batch[4], batch[5])):
            # a batch assembled on the device (PixelReplayBuffer): the per-frame views are built there as well
            frames = torch.cat([batch[0].reshape(3 * n, 3, 84, 84), batch[5][:, -3:]], dim=0).contiguous()
            next_frames = batch[4].reshape(3 * n, 3, 84, 84).contiguous()
            assert frames.dtype == torch.uint8 and next_frames.dtype == torch.uint8
            p_frames, p_next = frames.data_ptr(), next_frames.data_ptr()
            torch.cuda.current_stream().synchronize()
        else:
            img, next_img, next_step = (np.ascontiguousarray(torch.as_tensor(t).cpu().numpy()) for t in (batch[0], batch[4], batch[5]))
            frames = np.ascontiguousarray(np.concatenate([img.reshape(3 * n, 3, 84, 84), next_step[:, -3:]], axis=0))
            next_frames = np.ascontiguousarray(next_img.reshape(3 * n, 3, 84, 84))
            assert frames.dtype == np.uint8 and next_frames.dtype == np.uint8
            p_frames, p_next = frames.ctypes.data, next_frames.ctypes.data
        action, reward, discount = (torch.as_tensor(t).detach().cpu().numpy() for t in batch[1:4])
        ident = np.full((n, 2), 4, dtype=np.int32)
        shifts = np.ascontiguousarray(np.concatenate([np.repeat(d["shifts"][0], 3, axis=0), ident], axis=0), dtype=np.int32)
        next_shifts = np.ascontiguousarray(np.repeat(d["shifts"][1], 3, axis=0), dtype=np.int32)
        f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)
        keep = dict(shifts=shifts, next_shifts=next_shifts, action=f32(action),
                    reward=f32(reward).reshape(-1), discount=f32(discount).reshape(-1), eps_post=f32(d["eps_post"]),
                    alphabar=f32(d["alphabar"]), temb=f32(d["temb"]), noise=f32(d["noise"]), psi_masks=f32(d["psi_masks"]),
                    zeta_masks=f32(d["zeta_masks"]), eps_act=f32(d["eps_act"]))
        stddev = float(self.stddev_schedule(step))
        inp = LdiffInputs(stddev=stddev, frames=p_frames, next_frames=p_next, **{k: v.ctypes.data for k, v in keep.items()})
        m = np.zeros(8, dtype=np.float32)
        _lib.check(self.lib.rlrep_ldiff_update(self._h, C.byref(inp), m.ctypes.data))
        return {"loss/recon_loss": float(m[0]), "loss/kl_loss": float(m[1]), "loss/score_loss": float(m[2]), "loss/reg_loss": 0.0,
                "loss/critic_loss": float(m[3]), "info/q_pred": float(m[4]), "info/q_target": float(m[5]),
                "info/reward": float(m[6]), "loss/actor_loss": float(m[7]), "info/policy_std": stddev}
