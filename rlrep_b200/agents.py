"""Host-side mirror of the reference's agent classes over the C-ABI handles of librlrep_b200.so.

Same constructors, `train(buffer, batch_size) -> dict` and `select_action(state, explore=False)` as the reference
(agent/sac/sac_agent.py:16-188, agent/ctrlsac/ctrlsac_agent.py:123-362), so the reference's `main.py` drives them
unchanged.  Everything numerical happens in the CUDA library; this file only
  * draws the randomness the way the reference does (np.random.randint for replay indices, torch.randn on the CPU
    generator for every epsilon, in the order of SURVEY.md A.5) and hands it to `rlrep_agent_train`,
  * maps the metrics array back to the reference's info-dict keys,
  * moves weights in and out under the reference's state_dict names.
There is no fallback: without the built library or without a CUDA device the constructors raise.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from . import _lib


def _orthogonal(out_f, in_f, generator=None):
    w = torch.empty(out_f, in_f)
    torch.nn.init.orthogonal_(w, generator=generator)  # utils/util.py:61-66 (weight_init)
    return w


def _default_linear(out_f, in_f, generator=None):
    """nn.Linear's default init (kaiming_uniform(a=sqrt(5)) == U(+-1/sqrt(fan_in)) for weight and bias)."""
    bound = 1.0 / math.sqrt(in_f)
    return ((torch.rand(out_f, in_f, generator=generator) * 2 - 1) * bound,
            (torch.rand(out_f, generator=generator) * 2 - 1) * bound)


class _Handle:
    """Owns one `rlrep_agent*` and exposes tensors / scalars."""

    def __init__(self, cfg: _lib.AgentConfig, comm=None):
        if not torch.cuda.is_available():
            raise _lib.RlrepError("rlrep_b200 agents need a CUDA device (there is no CPU fallback)")
        self.lib = _lib.load()
        self.stream = torch.cuda.current_stream().cuda_stream
        self.device = torch.cuda.current_device()  # the handle lives on the device current at creation
        h = C.c_void_p()
        if comm is None:
            _lib.check(self.lib.rlrep_agent_create(C.byref(cfg), self.stream, C.byref(h)))
        else:  # batch-sharded handle: cfg.batch_size is the rank's share of the global batch
            _lib.check(self.lib.rlrep_agent_create_sharded(C.byref(cfg), comm, self.stream, C.byref(h)))
        self.h = h
        n = C.c_int()
        _lib.check(self.lib.rlrep_agent_num_tensors(self.h, C.byref(n)))
        self.index = {}
        for i in range(n.value):
            name, ptr, rows, cols = C.c_char_p(), C.c_void_p(), C.c_int(), C.c_int()
            _lib.check(self.lib.rlrep_agent_tensor_info(self.h, i, C.byref(name), C.byref(ptr), C.byref(rows), C.byref(cols)))
            self.index[name.value.decode()] = (i, ptr.value, rows.value, cols.value)
        ni, ne, nm = C.c_int(), C.c_int(), C.c_int()
        _lib.check(self.lib.rlrep_agent_train_counts(self.h, C.byref(ni), C.byref(ne), C.byref(nm)))
        self.n_idx, self.n_eps, self.n_metrics = ni.value, ne.value, nm.value
        self.metric_names = [self.lib.rlrep_agent_metric_name(self.h, i).decode() for i in range(self.n_metrics)]
        self._metrics = np.zeros(self.n_metrics, dtype=np.float32)

    def close(self):
        h, self.h = self.h, None
        if h is not None:
            self.lib.rlrep_agent_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # `logical` maps a tensor name to the (rows, cols) the caller sees when the handle was built with hidden widths rounded
    # up to a multiple of 32 (see SACAgent._pad): reads crop to it, writes zero-pad from it.
    logical: dict = {}

    def _logical_shape(self, name, rows, cols):
        base = name.split("/", 1)[1] if name.startswith("optim.") else name
        return self.logical.get(base, (rows, cols))

    def read(self, name) -> torch.Tensor:
        i, _, rows, cols = self.index[name]
        out = np.empty(rows * cols, dtype=np.float32)
        _lib.check(self.lib.rlrep_agent_tensor_read(self.h, i, out.ctypes.data))
        t = torch.from_numpy(out).reshape(rows, cols)
        lr, lc = self._logical_shape(name, rows, cols)
        if (lr, lc) != (rows, cols):
            t = t[:lr, :lc].contiguous()
        return t if not name.endswith(".bias") else t.reshape(lr)

    def write(self, name, value):
        i, _, rows, cols = self.index[name]
        lr, lc = self._logical_shape(name, rows, cols)
        arr = torch.as_tensor(value).detach().cpu().float().reshape(-1)
        if arr.numel() != lr * lc:
            raise ValueError(f"{name}: expected {lr * lc} values, got {arr.numel()}")
        if (lr, lc) != (rows, cols):
            full = torch.zeros(rows, cols)
            full[:lr, :lc] = arr.reshape(lr, lc)
            arr = full.reshape(-1)
        arr = np.ascontiguousarray(arr.numpy())
        _lib.check(self.lib.rlrep_agent_tensor_write(self.h, i, arr.ctypes.data))

    def train(self, ring_handle, idx: np.ndarray, eps) -> np.ndarray:
        """`eps`: float32 numpy array, or a contiguous float32 CUDA tensor (noise drawn on the device: the library copies it
        device to device, rlrep_agent_train accepts either kind of pointer)."""
        if isinstance(eps, torch.Tensor):
            torch.cuda.current_stream(eps.device).synchronize()  # the library works on its own stream
            eps_ptr, n_eps = eps.data_ptr(), eps.numel()
        else:
            eps_ptr, n_eps = eps.ctypes.data, eps.size
        _lib.check(self.lib.rlrep_agent_train(self.h, ring_handle, idx.ctypes.data, idx.size, eps_ptr, n_eps,
                                              self._metrics.ctypes.data, self._metrics.size))
        return self._metrics

    @property
    def log_alpha(self) -> float:
        v = C.c_double()
        _lib.check(self.lib.rlrep_agent_get_log_alpha(self.h, C.byref(v)))
        return v.value

    @log_alpha.setter
    def log_alpha(self, v):
        _lib.check(self.lib.rlrep_agent_set_log_alpha(self.h, float(v)))

    @property
    def optim_state(self) -> dict:
        st = _lib.OptimState()
        _lib.check(self.lib.rlrep_agent_get_optim_state(self.h, C.byref(st)))
        return {k: getattr(st, k) for k, _ in _lib.OptimState._fields_}

    @optim_state.setter
    def optim_state(self, d):
        st = _lib.OptimState()
        _lib.check(self.lib.rlrep_agent_get_optim_state(self.h, C.byref(st)))
        for k, _ in _lib.OptimState._fields_:
            if k in d:
                setattr(st, k, type(getattr(st, k))(d[k]))
        _lib.check(self.lib.rlrep_agent_set_optim_state(self.h, C.byref(st)))

    @property
    def last_launches(self) -> int:
        v = C.c_int()
        _lib.check(self.lib.rlrep_agent_last_launches(self.h, C.byref(v)))
        return v.value

    @property
    def graph_stats(self) -> tuple[int, int]:
        """(kernel nodes, programmatic edges) of the captured train() graph."""
        k, p = C.c_int(), C.c_int()
        _lib.check(self.lib.rlrep_agent_graph_stats(self.h, C.byref(k), C.byref(p)))
        return k.value, p.value


class SACAgent:
    """Drop-in for agent.sac.sac_agent.SACAgent (sac_agent.py:16-188)."""

    alg = "sac"

    def __init__(self, state_dim, action_dim, action_space, lr=3e-4, discount=0.99, target_update_period=2, tau=0.005,
                 alpha=0.1, auto_entropy_tuning=True, hidden_dim=1024, *, precision="tf32", use_cuda_graph=True,
                 noise_device="cpu", generator=None, **extra):
        """`noise_device`: where train() draws its Gaussian noise.  "cpu" (default) uses torch's global CPU generator -- the
        stream the reference consumes when it runs on the CPU, and the one the oracle / golden fixtures are pinned to.
        "cuda" draws the same tensors, in the same order and shapes, with torch's CUDA generator -- the stream the
        reference consumes when it runs with device = cuda (torch.randn_like on CUDA tensors) -- so the noise never exists
        on the host: no host RNG time and no PCIe transfer (4 MB per update for LV-Rep at B = 1024).
        `generator`: a CPU torch.Generator the initial weights are drawn from instead of the global generator (same draws,
        same order)."""
        if noise_device not in ("cpu", "cuda"):
            raise ValueError("noise_device must be 'cpu' or 'cuda'")
        self.noise_device = noise_device
        self.steps = 0
        self.state_dim, self.action_dim = int(state_dim), int(action_dim)
        self.action_range = [float(action_space.low.min()), float(action_space.high.max())]  # sac_agent.py:36-39
        # main.py passes --discount/--tau through argparse without type=, i.e. possibly as strings (SURVEY A.1)
        self.discount, self.tau = float(discount), float(tau)
        self.target_update_period = int(target_update_period)
        self.learnable_temperature = bool(auto_entropy_tuning)
        self.target_entropy = -action_dim
        self._lr, self._alpha0, self._hidden = float(lr), float(alpha), int(hidden_dim)
        self._precision, self._use_graph = precision, bool(use_cuda_graph)
        self._extra = extra
        self._h: _Handle | None = None
        self._batch = None
        self._pending_state = self._initial_state(generator)  # host copy until the handle exists

    # ---- configuration of the C handle (overridden per algorithm) -------------------------------------------
    def _config(self, batch_size) -> _lib.AgentConfig:
        c = _lib.AgentConfig()
        c.alg = _lib.ALG[self.alg]
        c.state_dim, c.action_dim, c.batch_size = self.state_dim, self.action_dim, int(batch_size)
        c.hidden_dim, c.feature_dim, c.actor_hidden_dim = self._pad(self._hidden), 0, self._pad(self._hidden)
        c.feature_steps = 0
        c.lr_critic = c.lr_actor = c.lr_alpha = self._lr
        c.lr_feature = 0.0
        c.discount, c.tau, c.feature_tau = self.discount, self.tau, 0.0
        c.alpha = self._alpha0
        c.target_update_period = self.target_update_period
        c.auto_entropy_tuning = int(self.learnable_temperature)
        c.use_feature_target = 0
        c.precision = _lib.PRECISION[self._precision]
        c.use_cuda_graph = int(self._use_graph)
        return c

    def _layers(self):
        """[(name, out, in, init)] in the reference's construction order."""
        S, A, H = self.state_dim, self.action_dim, self._hidden
        q = [(f"critic.{h}.{i}", o, n, "orth") for h in ("Q1", "Q2") for i, o, n in ((0, H, S + A), (2, H, H), (4, 1, H))]
        return q + self._actor_layers(H)

    def _actor_layers(self, H):
        S, A = self.state_dim, self.action_dim
        return [("actor.trunk.0", H, S, "orth"), ("actor.trunk.2", H, H, "orth"), ("actor.trunk.4", 2 * A, H, "orth")]

    def _initial_state(self, generator=None):
        sd = {}
        for name, out, inp, kind in self._layers():
            if kind == "orth":  # modules that call self.apply(util.weight_init): orthogonal weight, zero bias
                sd[name + ".weight"], sd[name + ".bias"] = _orthogonal(out, inp, generator), torch.zeros(out)
            else:
                sd[name + ".weight"], sd[name + ".bias"] = _default_linear(out, inp, generator)
        return sd

    # ---- handle management --------------------------------------------------------------------------------------
    def _ensure(self, batch_size=None):
        if self._h is not None and (batch_size is None or batch_size == self._batch):
            return self._h
        carried = None
        if self._h is not None:
            # A different batch size (the reference accepts any, per call): activation buffers, TMA descriptors and the
            # captured graph are per batch size, so the handle is rebuilt and EVERYTHING that is state -- weights, targets,
            # Adam moments, step counters, the float64 temperature -- is carried over.
            self._pending_state = self.state_dict()
            self._pending_state.pop("log_alpha", None)
            carried = self.optimizer_state_dict()
            self._h.close()
        self._batch = int(batch_size or 256)
        self._h = self._make_handle(self._batch)
        self.load_state_dict(self._pending_state, strict=False)
        self._pending_state = None
        if carried is not None:
            self.load_optimizer_state_dict(carried)
        return self._h

    @staticmethod
    def _pad(width):
        """Hidden widths the tensor-core path wants as multiples of 32.  A hidden unit whose incoming and outgoing weights
        and bias are zero outputs ELU(0) = ReLU(0) = tanh(0) = sin(0) = 0, receives a zero gradient and gives a zero
        gradient to everything it touches, and Adam keeps zeros at zero: widening a hidden layer with such units is exact.
        The handle is therefore built with the width rounded up, and weights are zero-padded / cropped at the boundary, so
        any `hidden_dim` works like in the reference.  (Feature widths entering a mean -- LV-Rep's KL, Diff-SR's score
        layout -- cannot be padded this way and must be multiples of 32.)"""
        return (int(width) + 31) // 32 * 32

    def _make_handle(self, batch):
        h = _Handle(self._config(batch))
        self._attach_logical(h)
        return h

    def _attach_logical(self, h):
        logical = {}
        for name, out, inp, _ in self._layers():
            logical[name + ".weight"], logical[name + ".bias"] = (out, inp), (out, 1)
        targets = {}
        for k, v in logical.items():  # Polyak copies carry the source module's shapes
            mod = k.split(".", 1)[0]
            targets[mod + "_target." + k.split(".", 1)[1]] = v
        logical.update(targets)
        h.logical = {k: v for k, v in logical.items() if k in h.index and tuple(h.index[k][2:]) != v}

    def state_dict(self):
        """All parameters and Polyak targets under the reference's state_dict names, plus float64 `log_alpha`."""
        if self._h is None:
            return dict(self._pending_state)
        sd = {name: self._h.read(name) for name in self._h.index if not name.startswith("optim.")}
        sd["log_alpha"] = torch.tensor(self._h.log_alpha, dtype=torch.float64)
        return sd

    def optimizer_state_dict(self):
        """Adam moments of every parameter (`optim.m/<name>`, `optim.v/<name>` = torch.optim.Adam's exp_avg / exp_avg_sq)
        plus `control`: the agent's `steps`, the four optimisers' step counters and the temperature's float64 moments."""
        h = self._ensure()
        sd = {name: h.read(name) for name in h.index if name.startswith("optim.")}
        sd["control"] = dict(h.optim_state, agent_steps=self.steps)
        return sd

    def load_optimizer_state_dict(self, sd):
        h = self._ensure()
        for k, v in sd.items():
            if k != "control":
                h.write(k, v)
        ctl = dict(sd.get("control", {}))
        self.steps = int(ctl.pop("agent_steps", self.steps))
        h.optim_state = ctl

    def save(self, path):
        """Checkpoint (the reference parses --save_model but never writes one, main.py:37): a torch.save'd dict with the
        parameters / targets under the reference's state_dict names, so reference modules can load their slices with
        `module.load_state_dict({k[len(prefix):]: v ...})`, plus the optimiser state needed to resume exactly."""
        torch.save({"format": "rlrep_b200/1", "alg": self.alg, "state_dim": self.state_dim, "action_dim": self.action_dim,
                    "batch_size": self._batch, "state_dict": self.state_dict(), "optimizer": self.optimizer_state_dict()},
                   path)

    def load(self, path, load_optimizer=True):
        ck = torch.load(path, map_location="cpu", weights_only=False)
        if ck.get("format") != "rlrep_b200/1" or ck.get("alg") != self.alg:
            raise _lib.RlrepError(f"{path}: not a rlrep_b200 checkpoint of a {self.alg} agent")
        if (ck["state_dim"], ck["action_dim"]) != (self.state_dim, self.action_dim):
            raise _lib.RlrepError(f"{path}: saved for state/action dims {(ck['state_dim'], ck['action_dim'])}")
        self._ensure(ck.get("batch_size") if self._h is None else None)
        self.load_state_dict(ck["state_dict"], strict=False, sync_targets=False)
        if load_optimizer:
            self.load_optimizer_state_dict(ck["optimizer"])

    def load_state_dict(self, sd, strict=True, sync_targets=None):
        """Write weights.  Targets not present in `sd` are re-synchronised from their source networks."""
        if self._h is None:
            self._pending_state.update({k: torch.as_tensor(v).detach().clone() for k, v in sd.items()})
            return
        names = set(self._h.index)
        for k, v in sd.items():
            if k == "log_alpha":
                self._h.log_alpha = float(v)
            elif k in names:
                self._h.write(k, v)
            elif strict:
                raise KeyError(k)
        has_targets = any("_target." in k for k in sd)
        if sync_targets or (sync_targets is None and not has_targets):
            _lib.check(self._h.lib.rlrep_agent_sync_targets(self._h.h))

    @property
    def alpha(self):
        return math.exp(self._h.log_alpha) if self._h is not None else self._alpha0

    @property
    def gpu_launches_last_train(self):
        return self._h.last_launches if self._h is not None else 0

    # ---- reference surface ----------------------------------------------------------------------------------------
    def select_action(self, state, explore=False):  # sac_agent.py:89-96
        h = self._ensure()
        s = np.ascontiguousarray(np.asarray(state, dtype=np.float32).reshape(-1))
        out = np.empty(self.action_dim, dtype=np.float32)
        eps = None
        if explore:
            eps = np.ascontiguousarray(torch.randn(1, self.action_dim).numpy().reshape(-1))
        _lib.check(h.lib.rlrep_agent_act(h.h, s.ctypes.data, eps.ctypes.data if eps is not None else None,
                                         out.ctypes.data))
        return np.clip(out, self.action_range[0], self.action_range[1])

    def select_actions(self, states, explore=False):
        """Batched `select_action`: states [N, state_dim] -> actions [N, action_dim] in one kernel launch per 1024 rows
        (`rlrep_agent_act_batch`).  With explore=True the noise is drawn row by row, torch.randn(1, action_dim) per
        observation from the CPU generator -- exactly what N consecutive select_action(explore=True) calls draw (one
        torch.randn(N, action_dim) call would consume the generator differently)."""
        h = self._ensure()
        s = np.ascontiguousarray(np.asarray(states, dtype=np.float32).reshape(-1, self.state_dim))
        out = np.empty((s.shape[0], self.action_dim), dtype=np.float32)
        eps = None
        if explore:
            eps = np.ascontiguousarray(torch.cat([torch.randn(1, self.action_dim) for _ in range(s.shape[0])]).numpy())
        _lib.check(h.lib.rlrep_agent_act_batch(h.h, s.ctypes.data, eps.ctypes.data if eps is not None else None,
                                               s.shape[0], out.ctypes.data))
        return np.clip(out, self.action_range[0], self.action_range[1])

    def _randn(self, rows, cols, std=None):
        """One [rows, cols] standard-normal draw on `noise_device` (scaled by `std` the way torch.normal(0, std) does)."""
        if self.noise_device == "cpu":
            if std is None:
                return torch.randn(rows, cols)
            return torch.normal(mean=torch.zeros(rows, cols), std=torch.ones(rows, cols) * std)
        dev = torch.device("cuda", self._ensure().device)
        if std is None:
            return torch.randn(rows, cols, device=dev)
        return torch.normal(mean=torch.zeros(rows, cols, device=dev), std=torch.ones(rows, cols, device=dev) * std)

    @staticmethod
    def _pack(parts):
        """The draws of one train() as one flat float32 buffer: numpy on the host, a CUDA tensor on the device."""
        flat = torch.cat([p.reshape(-1) for p in parts])
        return flat if flat.is_cuda else flat.numpy()

    def _draw(self, buffer, batch_size):
        """Indices and noise for one train(), in the reference's RNG order (SURVEY A.5: sac)."""
        idx = np.random.randint(0, buffer.size, size=batch_size)
        eps = [self._randn(batch_size, self.action_dim) for _ in range(2)]  # critic step a', then actor step a
        return idx, self._pack(eps)

    def _info(self, m):
        return self._sac_info(dict(zip(self._h.metric_names, (float(x) for x in m))))

    @staticmethod
    def _sac_info(d):
        # sac_agent.py:131-135: q_loss = mse1 + mse2; 'q2' reports mean(Q1)
        return {"q_loss": float(np.float32(d["q1_loss"]) + np.float32(d["q2_loss"])), "q1": d["q1"], "q2": d["q1"],
                "actor_loss": d["actor_loss"], "alpha_loss": d["alpha_loss"], "alpha": d["alpha"]}

    def train(self, buffer, batch_size):
        """One update (sac_agent.py:169-188).  `buffer` must be an rlrep_b200.ReplayBuffer."""
        h = self._ensure(batch_size)
        buffer.flush()
        self.steps += 1
        idx, eps = self._draw(buffer, batch_size)
        idx = np.ascontiguousarray(idx, dtype=np.int64)
        eps = eps.contiguous() if isinstance(eps, torch.Tensor) else np.ascontiguousarray(eps, dtype=np.float32)
        m = h.train(buffer._h, idx, eps)
        info = self._info(m)
        if not self.learnable_temperature:
            info.pop("alpha_loss", None)
            info.pop("alpha", None)
        return info


class CTRLSACAgent(SACAgent):
    """Drop-in for agent.ctrlsac.ctrlsac_agent.CTRLSACAgent (ctrlsac_agent.py:123-362)."""

    alg = "ctrlsac"

    def __init__(self, state_dim, action_dim, action_space, lr=1e-4, discount=0.99, target_update_period=2, tau=0.005,
                 alpha=0.1, auto_entropy_tuning=True, hidden_dim=1024, feature_tau=0.005, feature_dim=2048,
                 use_feature_target=True, extra_feature_steps=1, **kw):
        self.feature_dim, self.feature_tau = int(feature_dim), float(feature_tau)
        self.use_feature_target, self.extra_feature_steps = bool(use_feature_target), int(extra_feature_steps)
        super().__init__(state_dim, action_dim, action_space, lr=lr, discount=discount,
                         target_update_period=target_update_period, tau=tau, alpha=alpha,
                         auto_entropy_tuning=auto_entropy_tuning, hidden_dim=hidden_dim, **kw)

    def _config(self, batch_size):
        c = super()._config(batch_size)
        # actor hidden fixed at 256, ctrlsac_agent.py:188-194; the feature width may be padded too (zero features are inert:
        # no mean runs over the feature axis in CTRL)
        c.feature_dim, c.actor_hidden_dim = self._pad(self.feature_dim), 256
        c.feature_steps = self.extra_feature_steps + 1
        c.lr_feature = c.lr_critic = self._lr
        c.lr_actor = c.lr_alpha = self._lr / 3  # :195-197
        c.feature_tau = self.feature_tau
        c.use_feature_target = int(self.use_feature_target)
        return c

    def _layers(self):
        S, A, H, D = self.state_dim, self.action_dim, self._hidden, self.feature_dim
        return [("phi.l1", H, S + A, "default"), ("phi.l2", H, H, "default"), ("phi.l3", D, H, "default"),
                ("mu.l1", H, S, "default"), ("mu.l2", H, H, "default"), ("mu.l3", D, H, "default"),
                ("theta.l", 1, D, "default")] + self._actor_layers(256) + \
               [("critic.l1", H, D, "default"), ("critic.l2", 1, H, "default"), ("critic.l4", H, D, "default"),
                ("critic.l5", 1, H, "default")]

    def state_dict(self):
        sd = super().state_dict()
        # frozen_phi / frozen_phi_target are aliases of phi after any train() (ctrlsac_agent.py:344-346)
        for k in [k for k in sd if k.startswith("phi.")]:
            sd["frozen_phi." + k[4:]] = sd[k]
            sd["frozen_phi_target." + k[4:]] = sd[k]
        return sd

    def load_state_dict(self, sd, strict=True, sync_targets=None):
        sd = {k: v for k, v in sd.items() if not k.startswith("frozen_phi")}
        super().load_state_dict(sd, strict=strict, sync_targets=sync_targets)

    def _draw(self, buffer, batch_size):  # SURVEY A.5: K x randint[B] -> randn[B,A] -> randn[B,A]
        K = self.extra_feature_steps + 1
        idx = np.concatenate([np.random.randint(0, buffer.size, size=batch_size) for _ in range(K)])
        eps = [self._randn(batch_size, self.action_dim) for _ in range(2)]
        return idx, self._pack(eps)

    def _info(self, m):
        return dict(zip(self._h.metric_names, (float(x) for x in m)))


class ShardedCTRLSACAgent(CTRLSACAgent):
    """CTRL-SAC with the batch of every train() call split by rows over the ranks of a torch.distributed process group
    (one process per GPU; BASELINE config 4, SURVEY.md 8e).  The reference has no distributed code: this is its update
    on the GLOBAL batch, computed cooperatively -- mu(s') is all-gathered so that every rank owns complete rows of the
    contrastive logits, its gradient is reduce-scattered, parameter gradients and loss sums are all-reduced (NCCL over
    NVLink inside the C library), and every rank applies the same Adam step.

    Every rank must be constructed with the same arguments, load the same weights and run with the same numpy / torch
    seeds: `train(buffer, batch_size)` draws the GLOBAL indices and noise exactly like the reference does and keeps the
    rank's rows; `batch_size` is the global batch and must be divisible by the world size.  The returned info dict is
    global and identical on all ranks."""

    def __init__(self, *args, process_group=None, **kw):
        import torch.distributed as dist
        if not dist.is_initialized():
            raise _lib.RlrepError("ShardedCTRLSACAgent needs an initialised torch.distributed process group")
        self._pg = process_group
        self.rank, self.world = dist.get_rank(process_group), dist.get_world_size(process_group)
        self._comm = None
        kw.setdefault("use_cuda_graph", False)
        super().__init__(*args, **kw)

    def _comm_handle(self):
        """rank 0 creates the NCCL unique id, torch.distributed ships it, every rank joins (rlrep_comm_create)."""
        if self._comm is not None:
            return self._comm
        import torch.distributed as dist
        lib = _lib.load()
        idbuf = (C.c_ubyte * 128)()
        if self.rank == 0:
            _lib.check(lib.rlrep_comm_unique_id(idbuf))
        box = [bytes(idbuf) if self.rank == 0 else None]
        src = dist.get_global_rank(self._pg, 0) if self._pg is not None else 0
        dist.broadcast_object_list(box, src=src, group=self._pg)
        idbuf = (C.c_ubyte * 128).from_buffer_copy(box[0])
        comm = C.c_void_p()
        _lib.check(lib.rlrep_comm_create(idbuf, self.rank, self.world, C.byref(comm)))
        self._comm = comm
        return comm

    def local_batch(self, batch_size):
        if batch_size % self.world != 0:
            raise ValueError(f"global batch {batch_size} is not divisible by the world size {self.world}")
        return batch_size // self.world

    def _make_handle(self, batch):
        return _Handle(self._config(self.local_batch(batch)), comm=self._comm_handle())

    def _draw(self, buffer, batch_size):
        """Global draws in the reference's order (SURVEY A.5), then this rank's rows of each of them."""
        idx, eps = super()._draw(buffer, batch_size)
        K, b = self.extra_feature_steps + 1, self.local_batch(batch_size)
        lo, hi = self.rank * b, (self.rank + 1) * b
        idx = idx.reshape(K, batch_size)[:, lo:hi].reshape(-1)
        eps = eps.reshape(2, batch_size, self.action_dim)[:, lo:hi].reshape(-1)
        return idx, eps

    def close(self):
        if self._h is not None:
            self._h.close()
            self._h = None
        if self._comm is not None:
            _lib.load().rlrep_comm_destroy(self._comm)
            self._comm = None


class VLSACAgent(SACAgent):
    """Drop-in for agent.vlsac.vlsac_agent.VLSACAgent (vlsac_agent.py:66-273, networks/vae.py)."""

    alg = "vlsac"
    NUM_NOISE = 20  # vlsac_agent.py:24

    def __init__(self, state_dim, action_dim, action_space, lr=1e-4, discount=0.99, target_update_period=2, tau=0.005,
                 alpha=0.1, auto_entropy_tuning=True, hidden_dim=256, feature_tau=0.001, feature_dim=256,
                 use_feature_target=True, extra_feature_steps=1, **kw):
        self.feature_dim, self.feature_tau = int(feature_dim), float(feature_tau)
        self.use_feature_target, self.extra_feature_steps = bool(use_feature_target), int(extra_feature_steps)
        super().__init__(state_dim, action_dim, action_space, lr=lr, discount=discount,
                         target_update_period=target_update_period, tau=tau, alpha=alpha,
                         auto_entropy_tuning=auto_entropy_tuning, hidden_dim=hidden_dim, **kw)
        # the critic's fixed noise is drawn once at construction from the global generator (vlsac_agent.py:30-31)
        self._pending_state["critic.noise"] = torch.randn([self.NUM_NOISE, self.feature_dim])

    def _config(self, batch_size):
        c = super()._config(batch_size)
        c.feature_dim = self.feature_dim
        c.feature_steps = self.extra_feature_steps + 1
        c.lr_feature = self._lr          # vlsac_agent.py:113-115; actor / alpha keep SACAgent's optimisers (lr)
        c.feature_tau = self.feature_tau
        c.use_feature_target = int(self.use_feature_target)
        c.num_noise = self.NUM_NOISE
        return c

    def _layers(self):
        S, A, H, D = self.state_dim, self.action_dim, self._hidden, self.feature_dim
        V = 256  # networks/vae.py hidden_dim defaults
        d = "default"
        return [("encoder.l1", V, 2 * S + A, d), ("encoder.l2", V, V, d), ("encoder.mean_linear", D, V, d),
                ("encoder.log_std_linear", D, V, d), ("decoder.l1", V, D, d), ("decoder.state_linear", S, V, d),
                ("decoder.reward_linear", 1, V, d), ("f.l1", V, S + A, d), ("f.l2", V, V, d),
                ("f.mean_linear", D, V, d), ("f.log_std_linear", D, V, d)] + self._actor_layers(H) + \
               [("critic.l1", H, D, d), ("critic.l2", H, H, d), ("critic.l3", 1, H, d), ("critic.l4", H, D, d),
                ("critic.l5", H, H, d), ("critic.l6", 1, H, d)]

    @property
    def critic_noise(self):
        return self.state_dict()["critic.noise"]

    def _draw(self, buffer, batch_size):  # SURVEY A.5: K x (randint[B] -> randn[B,D]) -> randn[B,A] -> randn[B,A]
        K = self.extra_feature_steps + 1
        idx, eps = [], []
        for _ in range(K):
            idx.append(np.random.randint(0, buffer.size, size=batch_size))
            eps.append(self._randn(batch_size, self.feature_dim))
        eps += [self._randn(batch_size, self.action_dim) for _ in range(2)]
        return np.concatenate(idx), self._pack(eps)

    def _info(self, m):
        return dict(zip(self._h.metric_names, (float(x) for x in m)))


def _trunk_layers(prefix, dims, kind="default"):
    """Linear layers of util.mlp / spedersac mlp: Sequential indices 0, 2, 4, ... (utils/util.py:85-96)."""
    return [(f"{prefix}.{2 * i}", dims[i + 1], dims[i], kind) for i in range(len(dims) - 1)]


def _rff_critic_layers(D, H):
    d = "default"
    return [("critic.l1", H, D, d), ("critic.l2", H, H, d), ("critic.l3", 1, H, d), ("critic.l4", H, D, d),
            ("critic.l5", H, H, d), ("critic.l6", 1, H, d)]


class SPEDERSACAgent(SACAgent):
    """Drop-in for agent.spedersac.spedersac_agent.SPEDERSACAgent (spedersac_agent.py:97-322)."""

    alg = "spedersac"

    def __init__(self, state_dim, action_dim, action_space, phi_and_mu_lr=-1, phi_hidden_dim=-1, phi_hidden_depth=-1,
                 mu_hidden_dim=-1, mu_hidden_depth=-1, critic_and_actor_lr=-1, critic_and_actor_hidden_dim=-1,
                 discount=0.99, target_update_period=2, tau=0.005, alpha=0.1, auto_entropy_tuning=True, hidden_dim=1024,
                 feature_tau=0.005, feature_dim=2048, use_feature_target=True, extra_feature_steps=1, **kw):
        if min(phi_and_mu_lr, critic_and_actor_lr) <= 0 or min(phi_hidden_depth, mu_hidden_depth) < 0 or \
                critic_and_actor_hidden_dim <= 0 or (phi_hidden_depth > 0 and phi_hidden_dim <= 0) or \
                (mu_hidden_depth > 0 and mu_hidden_dim <= 0):
            raise ValueError("SPEDERSACAgent needs phi_and_mu_lr, critic_and_actor_lr, the phi / mu trunk sizes and "
                             "critic_and_actor_hidden_dim (the reference's -1 defaults are placeholders, main.py:95-104)")
        self.feature_dim, self.feature_tau = int(feature_dim), float(feature_tau)
        self.use_feature_target, self.extra_feature_steps = bool(use_feature_target), int(extra_feature_steps)
        self._phi = (int(phi_hidden_dim), int(phi_hidden_depth))
        self._mu = (int(mu_hidden_dim), int(mu_hidden_depth))
        self._feat_lr = float(phi_and_mu_lr)
        super().__init__(state_dim, action_dim, action_space, lr=critic_and_actor_lr, discount=discount,
                         target_update_period=target_update_period, tau=tau, alpha=alpha,
                         auto_entropy_tuning=auto_entropy_tuning, hidden_dim=critic_and_actor_hidden_dim, **kw)

    def _config(self, batch_size):
        c = super()._config(batch_size)  # critic / actor / alpha all at critic_and_actor_lr (:168-179)
        c.feature_dim = self._pad(self.feature_dim)  # zero features are inert in SPEDER's losses as well
        c.feature_steps = self.extra_feature_steps + 1
        c.lr_feature = self._feat_lr
        c.feature_tau = self.feature_tau
        c.use_feature_target = int(self.use_feature_target)
        c.phi_hidden_dim, c.phi_hidden_depth = self._pad(self._phi[0]) if self._phi[1] > 0 else self._phi[0], self._phi[1]
        c.mu_hidden_dim, c.mu_hidden_depth = self._pad(self._mu[0]) if self._mu[1] > 0 else self._mu[0], self._mu[1]
        return c

    def _layers(self):
        S, A, H, D = self.state_dim, self.action_dim, self._hidden, self.feature_dim
        (ph, pd), (mh, md) = self._phi, self._mu
        return _trunk_layers("phi.trunk", [S + A] + [ph] * pd + [D]) + _trunk_layers("mu.trunk", [S] + [mh] * md + [D]) + \
            [("theta.l", 1, D, "default")] + self._actor_layers(H) + _rff_critic_layers(D, H)

    def _draw(self, buffer, batch_size):  # SURVEY A.5: K x (randint[B], randint[B]) -> randn[B,A] -> randn[B,A]
        K = self.extra_feature_steps + 1
        idx = np.concatenate([np.random.randint(0, buffer.size, size=batch_size) for _ in range(2 * K)])
        eps = [self._randn(batch_size, self.action_dim) for _ in range(2)]
        return idx, self._pack(eps)

    def _info(self, m):
        return dict(zip(self._h.metric_names, (float(x) for x in m)))


class DIFFSRSACAgent(SACAgent):
    """Drop-in for agent.diffsrsac.diffsrsac_agent.DIFFSRSACAgent (diffsrsac_agent.py:93-343)."""

    alg = "diffsrsac"

    def __init__(self, state_dim, action_dim, action_space, feature_dim=256, phi_and_nabla_mu_lr=0.003,
                 phi_hidden_dim=256, phi_hidden_depth=1, nabla_mu_hidden_dim=512, nabla_mu_hidden_depth=1,
                 critic_and_actor_lr=3e-4, discount=0.99, target_update_period=2, tau=0.005, alpha=0.1,
                 auto_entropy_tuning=True, hidden_dim=256, extra_feature_steps=3, num_noises=1000,
                 critic_elu_layer_regularizer_lambda=0, DARL_noise_a=0.3, DARL_noise_b=0.1, sigma_scale_factor=0.449,
                 **kw):
        if critic_elu_layer_regularizer_lambda != 0:
            # the reference multiplies the regulariser into losses that are never optimised (SURVEY.md A.6 #1): it can
            # only change the reported q_loss_reg.  Not reproduced for lambda != 0.
            raise NotImplementedError("critic_elu_layer_regularizer_lambda != 0")
        self.feature_dim, self.extra_feature_steps = int(feature_dim), int(extra_feature_steps)
        self.num_noises, self.sigma_scale_factor = int(num_noises), float(sigma_scale_factor)
        self._phi = (int(phi_hidden_dim), int(phi_hidden_depth))
        self._nabla = (int(nabla_mu_hidden_dim), int(nabla_mu_hidden_depth))
        self._feat_lr = float(phi_and_nabla_mu_lr)
        self._noise_ab = (float(DARL_noise_a), float(DARL_noise_b))
        super().__init__(state_dim, action_dim, action_space, lr=critic_and_actor_lr, discount=discount,
                         target_update_period=target_update_period, tau=tau, alpha=alpha,
                         auto_entropy_tuning=auto_entropy_tuning, hidden_dim=hidden_dim, **kw)
        self.noise_alphabars = self.generate_alphabars(*self._noise_ab, self.num_noises)
        self._pending_state["alphabars"] = self.noise_alphabars.reshape(1, -1)

    @staticmethod
    def generate_alphabars(a, b, num_alphas):
        """alpha-bar table from the Beta(a, b) CDF, clipped to [raw[-2], raw[1]] (diffsrsac_agent.py:178-203); host-side
        construction-time state, like in the reference."""
        from scipy.stats import beta
        raw = 1.0 - beta.cdf(np.linspace(0, 1, num_alphas), a, b)
        return torch.tensor(np.clip(raw, a_min=raw[-2], a_max=raw[1])).float()

    def _config(self, batch_size):
        c = super()._config(batch_size)
        c.feature_dim = self.feature_dim
        c.feature_steps = self.extra_feature_steps + 1
        c.lr_feature = self._feat_lr
        c.phi_hidden_dim, c.phi_hidden_depth = self._pad(self._phi[0]) if self._phi[1] > 0 else self._phi[0], self._phi[1]
        c.nabla_mu_hidden_dim, c.nabla_mu_hidden_depth = (self._pad(self._nabla[0]) if self._nabla[1] > 0 else self._nabla[0],
                                                          self._nabla[1])
        c.num_noises = self.num_noises
        c.sigma_scale_factor = self.sigma_scale_factor
        return c

    def _layers(self):
        S, A, H, D = self.state_dim, self.action_dim, self._hidden, self.feature_dim
        (ph, pd), (nh, nd) = self._phi, self._nabla
        return _trunk_layers("critic_feed_feature.z_vector", [S + A] + [ph] * pd + [D]) + \
            _trunk_layers("nablamu_net.Mu_z_by_s_layer", [S + 1] + [nh] * nd + [D * S]) + \
            self._actor_layers(H) + _rff_critic_layers(D, H)

    def _draw(self, buffer, batch_size):
        """SURVEY A.5: K x (randint[B] -> torch.randint(0, num_noises, (B,)) -> normal[B,S]) -> randn[B,A] -> randn[B,A].
        Index layout per iteration: B replay rows, then B noise levels."""
        K, B, S = self.extra_feature_steps + 1, batch_size, self.state_dim
        idx, eps = [], []
        for _ in range(K):
            idx.append(np.random.randint(0, buffer.size, size=B))
            idx.append(torch.randint(0, self.num_noises, (B,)).numpy())  # diffsrsac_agent.py:276
            eps.append(self._randn(B, S, std=self.sigma_scale_factor))
        eps += [self._randn(B, self.action_dim) for _ in range(2)]
        return np.concatenate(idx), self._pack(eps)

    def _info(self, m):
        d = dict(zip(self._h.metric_names, (float(x) for x in m)))
        noreg = float(np.float32(d["q1_loss"]) + np.float32(d["q2_loss"]))
        # diffsrsac_agent.py:229-239: the regulariser is lambda = 0; 'q2' reports mean(Q1) (SURVEY.md A.6 #5)
        return {"score_loss": d["score_loss"], "q_loss_reg": noreg, "q_loss_noreg": noreg, "q1": d["q1"], "q2": d["q1"],
                "actor_loss": d["actor_loss"], "alpha_loss": d["alpha_loss"], "alpha": d["alpha"]}


def eval_policy(agent, envs, eval_episodes=10):
    """`utils.util.eval_policy` (utils/util.py:40-57) over a LIST of environment copies stepped in lockstep: all live
    episodes' observations go through one `agent.select_actions` call per step instead of one launch per environment.
    `envs` are gym-style (`reset() -> obs`, `step(a) -> obs, reward, done, info`); returns (average return, all returns)
    over `eval_episodes` episodes, episodes assigned to environments round-robin like the reference's sequential loop."""
    returns, pending = [], int(eval_episodes)
    live = {}
    for k, env in enumerate(envs):
        if pending > 0:
            live[k] = [env.reset(), 0.0]
            pending -= 1
    while live:
        keys = sorted(live)
        actions = agent.select_actions(np.stack([np.asarray(live[k][0], dtype=np.float32) for k in keys]))
        for k, a in zip(keys, actions):
            obs, reward, done, _ = envs[k].step(a)
            live[k][0] = obs
            live[k][1] += float(reward)
            if done:
                returns.append(live[k][1])
                if pending > 0:
                    live[k] = [envs[k].reset(), 0.0]
                    pending -= 1
                else:
                    del live[k]
    return float(np.mean(returns)), returns


AGENTS = {"sac": SACAgent, "ctrlsac": CTRLSACAgent, "vlsac": VLSACAgent, "spedersac": SPEDERSACAgent,
          "diffsrsac": DIFFSRSACAgent}
