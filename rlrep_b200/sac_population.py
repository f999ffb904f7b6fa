"""SAC seed populations: N SAC agents of one configuration, one per seed, trained as ONE batched update on one GPU.

A seed sweep of a SAC baseline is N independent runs.  `Population` runs them as N lone handles on N host threads;
`SACPopulation` holds all N in one library handle (`rlrep_sacpop_*`): every kernel of the update takes the member from a
grid dimension, so one train() is the launch sequence of ONE lone agent's update, with N times the CTAs per launch.

Seed contract: member m reproduces, bit for bit, a lone process that ran

    np.random.seed(seeds[m]); torch.manual_seed(seeds[m])
    agent = SACAgent(state_dim, action_dim, action_space, **kw)
    ... agent.train(buffers[m], batch_size) / agent.select_action(state, explore) ...

because member m draws from its own generators, in the lone agent's order: replay indices from
np.random.RandomState(seeds[m]); initial weights, select_actions noise and (noise_device="cpu") training noise from a CPU
torch.Generator seeded with seeds[m]; training noise from a CUDA torch.Generator seeded with seeds[m] when
noise_device="cuda".  A member's checkpoint (`save_member`) is an ordinary SACAgent checkpoint.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .agents import SACAgent


class _PopHandle:
    """Owns one `rlrep_sacpop*`; tensors are addressed as (member, name)."""

    def __init__(self, cfg: _lib.AgentConfig, members: int):
        if not torch.cuda.is_available():
            raise _lib.RlrepError("rlrep_b200 agents need a CUDA device (there is no CPU fallback)")
        self.lib = _lib.load()
        self.stream = torch.cuda.current_stream().cuda_stream
        self.device = torch.cuda.current_device()
        h = C.c_void_p()
        _lib.check(self.lib.rlrep_sacpop_create(C.byref(cfg), int(members), self.stream, C.byref(h)))
        self.h = h
        self.members = members
        n = C.c_int()
        _lib.check(self.lib.rlrep_sacpop_num_tensors(self.h, C.byref(n)))
        self.index = {}
        for i in range(n.value):
            name, ptr, rows, cols = C.c_char_p(), C.c_void_p(), C.c_int(), C.c_int()
            _lib.check(self.lib.rlrep_sacpop_tensor_info(self.h, 0, i, C.byref(name), C.byref(ptr), C.byref(rows),
                                                         C.byref(cols)))
            self.index[name.value.decode()] = (i, ptr.value, rows.value, cols.value)
        ni, ne, nm = C.c_int(), C.c_int(), C.c_int()
        _lib.check(self.lib.rlrep_sacpop_train_counts(self.h, C.byref(ni), C.byref(ne), C.byref(nm)))
        self.n_idx, self.n_eps, self.n_metrics = ni.value, ne.value, nm.value
        self.metric_names = [self.lib.rlrep_sacpop_metric_name(self.h, i).decode() for i in range(self.n_metrics)]
        self._metrics = np.zeros((members, self.n_metrics), dtype=np.float32)
        self.logical = {}

    def close(self):
        h, self.h = self.h, None
        if h is not None:
            self.lib.rlrep_sacpop_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def read(self, m, name) -> torch.Tensor:
        i, _, rows, cols = self.index[name]
        out = np.empty(rows * cols, dtype=np.float32)
        _lib.check(self.lib.rlrep_sacpop_tensor_read(self.h, m, i, out.ctypes.data))
        t = torch.from_numpy(out).reshape(rows, cols)
        lr, lc = self._logical(name, rows, cols)
        if (lr, lc) != (rows, cols):
            t = t[:lr, :lc].contiguous()
        return t if not name.endswith(".bias") else t.reshape(lr)

    def write(self, m, name, value):
        i, _, rows, cols = self.index[name]
        lr, lc = self._logical(name, rows, cols)
        arr = torch.as_tensor(value).detach().cpu().float().reshape(-1)
        if arr.numel() != lr * lc:
            raise ValueError(f"{name}: expected {lr * lc} values, got {arr.numel()}")
        if (lr, lc) != (rows, cols):
            full = torch.zeros(rows, cols)
            full[:lr, :lc] = arr.reshape(lr, lc)
            arr = full.reshape(-1)
        arr = np.ascontiguousarray(arr.numpy())
        _lib.check(self.lib.rlrep_sacpop_tensor_write(self.h, m, i, arr.ctypes.data))

    def _logical(self, name, rows, cols):
        base = name.split("/", 1)[1] if name.startswith("optim.") else name
        return self.logical.get(base, (rows, cols))

    def get_optim_state(self, m) -> dict:
        st = _lib.OptimState()
        _lib.check(self.lib.rlrep_sacpop_get_optim_state(self.h, m, C.byref(st)))
        return {k: getattr(st, k) for k, _ in _lib.OptimState._fields_}

    def set_optim_state(self, m, d):
        st = _lib.OptimState()
        _lib.check(self.lib.rlrep_sacpop_get_optim_state(self.h, m, C.byref(st)))
        for k, _ in _lib.OptimState._fields_:
            if k in d:
                setattr(st, k, type(getattr(st, k))(d[k]))
        _lib.check(self.lib.rlrep_sacpop_set_optim_state(self.h, m, C.byref(st)))

    @staticmethod
    def rings(buffers):
        return (C.c_void_p * len(buffers))(*[b._h.value for b in buffers])

    def train(self, buffers, idx: np.ndarray, eps) -> np.ndarray:
        if isinstance(eps, torch.Tensor):
            torch.cuda.current_stream(eps.device).synchronize()  # the library works on its own stream
            eps_ptr, n_eps = eps.data_ptr(), eps.numel()
        else:
            eps_ptr, n_eps = eps.ctypes.data, eps.size
        _lib.check(self.lib.rlrep_sacpop_train(self.h, self.rings(buffers), len(buffers), idx.ctypes.data, idx.size,
                                               eps_ptr, n_eps, self._metrics.ctypes.data, self._metrics.size))
        return self._metrics

    @property
    def last_launches(self) -> int:
        v = C.c_int()
        _lib.check(self.lib.rlrep_sacpop_last_launches(self.h, C.byref(v)))
        return v.value


class SACPopulation:
    """len(seeds) SACAgents with the same configuration (SACAgent's keywords, `precision` and `noise_device` included),
    member m seeded with seeds[m] (see the module docstring), trained by one batched update per train() call."""

    alg = "sac"

    def __init__(self, seeds, state_dim, action_dim, action_space, **kw):
        self.seeds = [int(s) for s in seeds]
        if not self.seeds:
            raise ValueError("a population needs at least one seed")
        self._cpu_gen = [torch.Generator().manual_seed(s) for s in self.seeds]
        self._rs = [np.random.RandomState(s) for s in self.seeds]
        self._cuda_gen = None
        # per-member SACAgent shells: configuration, layer shapes and the initial weights, drawn from the member's
        # generator in the lone agent's order; they never create a handle of their own
        self._shells = [SACAgent(state_dim, action_dim, action_space, generator=g, **kw) for g in self._cpu_gen]
        a = self._shells[0]
        self.state_dim, self.action_dim, self.action_range = a.state_dim, a.action_dim, a.action_range
        self.noise_device, self.learnable_temperature = a.noise_device, a.learnable_temperature
        self.steps = [0] * len(self.seeds)
        self._h: _PopHandle | None = None
        self._batch = None

    @property
    def members(self) -> int:
        return len(self.seeds)

    # ---- handle management ----------------------------------------------------------------------------------------
    def _ensure(self, batch_size=None):
        if self._h is not None and (batch_size is None or batch_size == self._batch):
            return self._h
        if self._h is not None:  # a new batch size: rebuild and carry every member's state over (SACAgent._ensure)
            carried = [(self.state_dict(m), self.optimizer_state_dict(m)) for m in range(self.members)]
            self._h.close()
        else:
            carried = [(s._pending_state, None) for s in self._shells]
        self._batch = int(batch_size or 256)
        h = _PopHandle(self._shells[0]._config(self._batch), self.members)
        self._shells[0]._attach_logical(h)
        self._h = h
        for m, (sd, opt) in enumerate(carried):
            self._write_state(m, sd)
            if opt is not None:
                self.load_optimizer_state_dict(m, opt)
        if not any("_target." in k for k in carried[0][0]):
            _lib.check(h.lib.rlrep_sacpop_sync_targets(h.h))
        return h

    def _write_state(self, m, sd):
        h = self._h
        for k, v in sd.items():
            if k == "log_alpha":
                h.set_optim_state(m, {"log_alpha": float(v)})
            elif k in h.index:
                h.write(m, k, v)
            else:
                raise KeyError(k)

    def close(self):
        if self._h is not None:
            self._h.close()
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- per-member state -------------------------------------------------------------------------------------------
    def state_dict(self, m):
        """Member m's parameters and Polyak targets under SACAgent.state_dict()'s names, plus float64 `log_alpha`."""
        h = self._ensure()
        sd = {name: h.read(m, name) for name in h.index if not name.startswith("optim.")}
        sd["log_alpha"] = torch.tensor(h.get_optim_state(m)["log_alpha"], dtype=torch.float64)
        return sd

    def load_state_dict(self, m, sd, sync_targets=None):
        """Write member m's weights; targets not in `sd` are re-synchronised from their source networks (SACAgent)."""
        h = self._ensure()
        self._write_state(m, sd)
        has_targets = any("_target." in k for k in sd)
        if sync_targets or (sync_targets is None and not has_targets):
            for name in h.index:
                if "_target." in name and not name.startswith("optim."):
                    h.write(m, name, h.read(m, name.replace("_target.", ".", 1)))

    def optimizer_state_dict(self, m):
        h = self._ensure()
        sd = {name: h.read(m, name) for name in h.index if name.startswith("optim.")}
        sd["control"] = dict(h.get_optim_state(m), agent_steps=self.steps[m])
        return sd

    def load_optimizer_state_dict(self, m, sd):
        h = self._ensure()
        for k, v in sd.items():
            if k != "control":
                h.write(m, k, v)
        ctl = dict(sd.get("control", {}))
        self.steps[m] = int(ctl.pop("agent_steps", self.steps[m]))
        h.set_optim_state(m, ctl)

    def save_member(self, m, path):
        """Member m as an ordinary SACAgent checkpoint (format rlrep_b200/1): SACAgent.load resumes that seed alone."""
        torch.save({"format": "rlrep_b200/1", "alg": self.alg, "state_dim": self.state_dim, "action_dim": self.action_dim,
                    "batch_size": self._batch, "state_dict": self.state_dict(m),
                    "optimizer": self.optimizer_state_dict(m)}, path)

    def load_member(self, m, path, load_optimizer=True):
        ck = torch.load(path, map_location="cpu", weights_only=False)
        if ck.get("format") != "rlrep_b200/1" or ck.get("alg") != self.alg:
            raise _lib.RlrepError(f"{path}: not a rlrep_b200 checkpoint of a {self.alg} agent")
        if (ck["state_dim"], ck["action_dim"]) != (self.state_dim, self.action_dim):
            raise _lib.RlrepError(f"{path}: saved for state/action dims {(ck['state_dim'], ck['action_dim'])}")
        self._ensure(ck.get("batch_size") if self._h is None else None)
        self.load_state_dict(m, ck["state_dict"], sync_targets=False)
        if load_optimizer:
            self.load_optimizer_state_dict(m, ck["optimizer"])

    @property
    def gpu_launches_last_train(self):
        return self._h.last_launches if self._h is not None else 0

    # ---- training and acting ----------------------------------------------------------------------------------------
    def _randn(self, m, rows, cols):
        if self.noise_device == "cpu":
            return torch.randn(rows, cols, generator=self._cpu_gen[m])
        dev = torch.device("cuda", self._ensure().device)
        if self._cuda_gen is None:
            self._cuda_gen = [torch.Generator(device=dev).manual_seed(s) for s in self.seeds]
        return torch.randn(rows, cols, device=dev, generator=self._cuda_gen[m])

    def _draw(self, buffers, batch_size):
        """Every member's indices and noise for one train(), each from its own generators in SACAgent._draw's order."""
        idx, eps = [], []
        for m, b in enumerate(buffers):
            idx.append(self._rs[m].randint(0, b.size, size=batch_size))
            eps += [self._randn(m, batch_size, self.action_dim) for _ in range(2)]
        return np.ascontiguousarray(np.concatenate(idx), dtype=np.int64), SACAgent._pack(eps)

    def train(self, buffers, batch_size):
        """One update of every member: buffers[m] is member m's rlrep_b200.ReplayBuffer.  Returns one info dict per
        member, with SACAgent.train's keys and value types."""
        if len(buffers) != self.members:
            raise ValueError(f"expected {self.members} buffers, got {len(buffers)}")
        h = self._ensure(batch_size)
        for b in buffers:
            b.flush()
        self.steps = [s + 1 for s in self.steps]
        idx, eps = self._draw(buffers, batch_size)
        eps = eps.contiguous() if isinstance(eps, torch.Tensor) else np.ascontiguousarray(eps, dtype=np.float32)
        metrics = h.train(buffers, idx, eps)
        out = []
        for row in metrics:
            info = SACAgent._sac_info(dict(zip(h.metric_names, (float(x) for x in row))))
            if not self.learnable_temperature:
                info.pop("alpha_loss", None)
                info.pop("alpha", None)
            out.append(info)
        return out

    def select_actions(self, states, explore=False):
        """states [members, state_dim] -> one action per member [members, action_dim] in one kernel launch, clamped like
        SACAgent.select_action; with explore=True member m draws torch.randn(1, action_dim) from its CPU generator, as a
        lone select_action(explore=True) does from the global one."""
        h = self._ensure()
        s = np.ascontiguousarray(np.asarray(states, dtype=np.float32).reshape(self.members, self.state_dim))
        out = np.empty((self.members, self.action_dim), dtype=np.float32)
        eps = None
        if explore:
            eps = np.ascontiguousarray(
                torch.cat([torch.randn(1, self.action_dim, generator=g) for g in self._cpu_gen]).numpy())
        _lib.check(h.lib.rlrep_sacpop_act(h.h, s.ctypes.data, eps.ctypes.data if eps is not None else None,
                                          out.ctypes.data))
        return np.clip(out, self.action_range[0], self.action_range[1])

    def train_resident(self, buffers, idx: np.ndarray, eps: np.ndarray, n_steps: int) -> float:
        """Benchmark aid (rlrep_sacpop_train_resident): n_steps updates of every member with all inputs resident in HBM;
        idx [n_steps, members, batch], eps [n_steps, members, 2 * batch * action_dim].  Returns the CUDA-event time in ms."""
        h = self._ensure(idx.shape[-1])
        for b in buffers:
            b.flush()
        idx = np.ascontiguousarray(idx, dtype=np.int64)
        eps = np.ascontiguousarray(eps, dtype=np.float32)
        ms = C.c_float()
        _lib.check(h.lib.rlrep_sacpop_train_resident(h.h, h.rings(buffers), len(buffers), idx.ctypes.data,
                                                     eps.ctypes.data, int(n_steps), C.byref(ms)))
        return ms.value
