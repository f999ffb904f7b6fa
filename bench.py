#!/usr/bin/env python
"""Benchmark of the rl-rep update step on B200 (contract: see the task statement / DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

One "step" = one `agent.train(buffer, batch_size)` call = K_f feature iterations + critic + actor/alpha + Polyak.
Default workload (BASELINE.json configs[1]): ctrlsac, HalfCheetah shapes (S=17, A=6), batch 256, feature_dim 2048,
hidden 1024, extra_feature_steps 3; synthetic replay ring of 1,000,000 rows (SURVEY.md 8d).

The JSON line (rank 0):
  value        updates/s, whole job, device-timed (CUDA events on the agent's stream), inputs resident in HBM before the
               timed region; the K-step loop is repeated `--repeats` times (default 5) and the MEDIAN repeat is reported
  e2e          updates/s through the public Python API (`agent.train`) with host-drawn indices / noise: H2D of the step's
               inputs and D2H of its metrics inside the timed region (median repeat as well)
  roofline     the kernel with the largest share of the step.  Kernel times come from the CUPTI activity records of
               GRAPH-REPLAYED train() calls (the timed configuration), algorithmic bytes / flops from the launch records;
               `serialized` keeps the one-stream event-timed profile of round 1 for comparison
  fp32         the same workload with precision="fp32" (every GEMM on the IEEE FFMA kernels)
  cpu_baseline the oracle port (plain PyTorch CPU restatement of the reference) on the box's host cores
  sharded      (state workloads) BASELINE configs[3]: ONE CTRL-SAC agent at global batch 16384 sharded by rows over all N
               ranks (N = 1 included, so the per-N lines form a strong-scaling curve) + `sharded_parity`, a small sharded
               update checked against the oracle on the global batch inside this run
--dump-outputs DIR writes what the timed agent produced in its last timed update (see dump_outputs), so that two builds
run with the same arguments, and hence the same inputs, can be compared output for output.
N > 1 (torchrun): `value` is the population reading of the path -- independent agents, one per GPU, no collective in the
data path; time = max over ranks, value = sum of updates / that time.
`--impl reference` times the reference's own CPU implementation of the path (the oracle port with the as-written
[B,B,D] broadcast; /root/reference itself is not available on the GPU box) with all host threads.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys
import tempfile
import threading
import time
import zlib
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

SPEDER_MAIN = dict(extra_feature_steps=5, phi_and_mu_lr=1e-5, phi_hidden_dim=512, phi_hidden_depth=1, mu_hidden_dim=512,
                   mu_hidden_depth=0, critic_and_actor_lr=3e-4, critic_and_actor_hidden_dim=256, feature_dim=2048)

WORKLOADS = {
    # BASELINE.json configs[1] -- the configuration the metric is quoted on
    "ctrlsac_hc_b256": dict(alg="ctrlsac", S=17, A=6, B=256, rows=1_000_000,
                            kw=dict(hidden_dim=1024, feature_dim=2048, extra_feature_steps=3)),
    # BASELINE.json configs[0] (the reference's own CPU-runnable case)
    "sac_hc_b256": dict(alg="sac", S=17, A=6, B=256, rows=1_000_000, kw=dict(hidden_dim=256)),
    # BASELINE.json configs[2]
    "vlsac_hum_b1024": dict(alg="vlsac", S=376, A=17, B=1024, rows=200_000,
                            kw=dict(hidden_dim=256, feature_dim=256, extra_feature_steps=3)),
    # the other two state-based agents at what main.py passes (main.py:93-104)
    "spedersac_hc_b256": dict(alg="spedersac", S=17, A=6, B=256, rows=1_000_000, kw=SPEDER_MAIN),
    "diffsrsac_hc_b256": dict(alg="diffsrsac", S=17, A=6, B=256, rows=1_000_000, kw=dict(hidden_dim=256)),
    # pixel agents (SURVEY.md 8a rows a16 / a17) at their configs' shapes; one replica per GPU at N > 1.  Benched on the
    # TF32 tensor-core path, whose LOSSES meet the north_star TF32 bar at these sizes (tests/test_gpu_mulv.py,
    # test_gpu_drq.py; gradients behind ReLU stacks see ~1e-3 of the masks flip); the strict-fp32 figure (every GEMM and
    # convolution on the FFMA pipes, ~9x slower) rides along under "fp32".
    "drqv2_pixels_b256": dict(alg="drqv2", C=9, A=4, B=256, bn=50, H=1024, rows=0, kw={}),
    "mulvdrq_pixels_b256": dict(alg="mulvdrq", C=9, A=4, B=256, F=100, H=1024, rows=0, kw={}),
    "ldiffsr_pixels_b256": dict(alg="ldiffsr", C=9, A=4, B=256, rows=0, kw={}),
    # BASELINE.json configs[4]: a population of independent pixel agents, `--agents-per-gpu` (default 8) per GPU on their own
    # streams x N GPUs (64 agents at N = 8), no communication; value = sum of the agents' updates per second
    "mulvdrq_population": dict(alg="mulvdrq", C=9, A=4, B=256, F=100, H=1024, rows=0, kw={}, population=True),
    # BASELINE.json configs[3]: large-batch CTRL, GLOBAL batch 16384 split by rows over the ranks (strong scaling:
    # the total work is fixed; 2048 rows per GPU at N = 8), mu(s') all-gathered over NVLink
    "ctrlsac_b16384_sharded": dict(alg="ctrlsac", S=17, A=6, B=16384, rows=1_000_000, sharded=True,
                                   kw=dict(hidden_dim=1024, feature_dim=2048, extra_feature_steps=3)),
}


class Space:
    def __init__(self, A):
        self.low, self.high, self.shape = -np.ones(A, np.float32), np.ones(A, np.float32), (A,)


def config_of(workload, w, n_gpus):
    """The `config` object of the JSON line: identical in both arms (the driver compares them)."""
    c = {"workload": workload, "alg": w["alg"], "B": w["B"], **w["kw"]}
    if "S" in w:
        c.update(S=w["S"], A=w["A"], ring_rows=w["rows"])
    else:
        c.update(obs=[w["C"], 84, 84], A=w["A"])
    if w.get("sharded"):
        c["parallelism"] = (f"one agent, batch sharded by rows over {n_gpus} GPU(s): {w['B'] // n_gpus} rows/GPU, NCCL "
                            f"all-gather of mu(s'), reduce-scatter of d mu, all-reduce of gradients")
    else:
        c["parallelism"] = f"replicas x{n_gpus} (independent agents, no collective)"
    c["l2"] = "no flush between steps: the per-update working set (parameters, gradients, Adam moments, targets) exceeds " \
              "the 126 MB L2 for ctrlsac / pixel agents; smaller agents are L2-resident in both arms' favour (DESIGN.md 5)"
    return c


def module_params(w):
    import bench_data as BD  # layer table only (shapes)
    return {m: sum(o * i + o for _, o, i in layers) for m, layers in BD.layer_table(w["alg"], w["S"], w["A"], w["kw"])}


def algorithmic_bytes(w):
    """HBM bytes one update must move (SURVEY.md 8d / BASELINE.md): Adam 28 B/param (p, g, m, v read; p, m, v
    written), Polyak 12 B/param, plus every fp32 weight streamed once per GEMM that uses it."""
    n = module_params(w)
    alg = w["alg"]
    K = w["kw"].get("extra_feature_steps", {"sac": -1, "diffsrsac": 3}.get(alg, 1)) + 1  # class defaults
    feat = {"ctrlsac": ("phi", "mu", "theta"), "vlsac": ("encoder", "decoder", "f"), "spedersac": ("phi", "mu", "theta"),
            "diffsrsac": ("phi", "nablamu"), "sac": ()}[alg]
    feat_target = {"ctrlsac": "phi", "vlsac": "f", "spedersac": "phi"}.get(alg)
    feat_n = sum(n[m] for m in feat)
    critic_adam = 0 if alg == "diffsrsac" else n["critic"]  # SURVEY.md A.6 #1
    opt = 28 * (K * feat_n + critic_adam + n["actor"]) + 12 * (K * n.get(feat_target, 0) + n["critic"] / 2)
    used = {"ctrlsac": "phi", "vlsac": "f", "spedersac": "phi", "diffsrsac": "phi"}.get(alg)
    used_n = n.get(used, 0)
    stream = 4 * (K * 2 * feat_n + 2 * used_n + 2 * n["critic"] + 2 * used_n + 2 * n["critic"] + 3 * n["actor"])
    return dict(optimizer=opt, weights=stream, total=opt + stream)


# ---------------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index, self.proc, self.path = gpu_index, None, None

    def __enter__(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu_index)], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def summary(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.path or not os.path.exists(self.path):
            return out
        sm, mx, reasons = [], [], set()
        for line in open(self.path):
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


_REAL_STDOUT = None


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


DUMP_BUDGET = 15_000_000  # float32 elements written by --dump-outputs: keeps a dump below 64 MB
DUMP_WHOLE = 65_536  # tensors up to this many elements are always written whole


def dump_outputs(out_dir, metrics, state):
    """--dump-outputs: the metrics the last timed update returned (`metric.<name>.npy`, float64 scalars) and the agent's
    parameters after it (`param.<name>.npy`, float32; float64 for log_alpha).

    The dumped update is the last one of the last timed loop on the benched agent, which runs after the device-resident
    loop that `value` times:
      state agents   the end-to-end loop with noise_device="cuda" (torch's CUDA generator draws the noise; the
                     device-resident loop uses host-drawn noise); the sharded agent: the end-to-end loop with host noise
      pixel agents   the end-to-end loop with the frame stacks resident on the device
    Every input of these loops is seeded, so runs with the same arguments dump the same update.

    When the parameters exceed DUMP_BUDGET, each tensor larger than DUMP_WHOLE is reduced to a sample of its flattened
    elements: the sorted distinct positions of draws from a generator seeded with the tensor's name, the same in every run
    of the same workload."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for k, v in metrics.items():
        np.save(out / f"metric.{k.replace('/', '.')}.npy", np.float64(v))
    arrays = {k: v.detach().cpu().numpy() for k, v in state.items()}
    small = sum(a.size for a in arrays.values() if a.size <= DUMP_WHOLE)
    large = sum(a.size for a in arrays.values() if a.size > DUMP_WHOLE)
    frac = min(1.0, max(0.0, DUMP_BUDGET - small) / max(large, 1))
    for k, a in arrays.items():
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
        if a.size > DUMP_WHOLE and frac < 1.0:
            draws = np.random.default_rng(zlib.crc32(k.encode())).integers(0, a.size, int(a.size * frac))
            a = a.reshape(-1)[np.unique(draws)]
        np.save(out / f"param.{k.replace('/', '.')}.npy", a)


def peaks():
    pk = ROOT / "MEASURED_PEAKS.json"
    if pk.exists():
        return float(json.loads(pk.read_text()).get("hbm_gbs", 6650.0)), "MEASURED_PEAKS.json hbm_gbs"
    return 6650.0, "fallback 6650 GB/s (B200_PROFILING.md)"


def measure_tf32_peak():
    """Dense TF32 tensor-core peak the way MEASURED_PEAKS.json measures bf16: torch.matmul (cuBLAS) on 8192^3, best of
    10 with CUDA events.  Only a roofline denominator -- never on the measured path."""
    import torch
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        a = torch.randn(8192, 8192, device="cuda")
        b = torch.randn(8192, 8192, device="cuda")
        c = torch.empty(8192, 8192, device="cuda")
        for _ in range(3):
            torch.matmul(a, b, out=c)
        best = 1e9
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b, out=c)
            e1.record()
            e1.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return 2 * 8192 ** 3 / (best * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def kernel_label(name):
    """CUPTI kernel name -> the launch label the library records ('..::gemm_tf32_kernel<128, 0, 1>(..)' -> 'gemm_tf32')."""
    m = re.search(r"(\w+?)_kernel\b", name)
    if m:
        return m.group(1)
    if "nccl" in name.lower():
        return "nccl"
    return re.sub(r"[<(].*", "", name).split("::")[-1].strip()


def graph_timeline(step_fn, n_calls):
    """CUPTI activity records (torch.profiler) of `n_calls` graph-replayed updates -> {label: [sum_us, count, union_us]},
    window_us.  `union_us` is the time at least one launch of that kernel was running (branches of the graph overlap)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(n_calls):
            step_fn(i)
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "memcpy" not in e.name.lower()
          and "memset" not in e.name.lower()]
    if not ev:
        return {}, 0.0
    per = {}
    for e in ev:
        per.setdefault(kernel_label(e.name), []).append((e.time_range.start, e.time_range.end))
    out = {}
    for k, iv in per.items():
        iv.sort()
        union, cur_s, cur_e = 0.0, iv[0][0], iv[0][1]
        for s, e in iv[1:]:
            if s > cur_e:
                union += cur_e - cur_s
                cur_s, cur_e = s, e
            else:
                cur_e = max(cur_e, e)
        union += cur_e - cur_s
        out[k] = [sum(e - s for s, e in iv), len(iv), union]
    window = max(e.time_range.end for e in ev) - min(e.time_range.start for e in ev)
    return out, window


# ---------------------------------------------------------------------------------------------------- CPU arm
def make_oracle(w, as_written=True):
    from oracle import rl_oracle as O
    kw = dict(w["kw"])
    init = O.init_state(w["alg"], w["S"], w["A"], kw, seed=0)
    extra = dict(as_written=as_written) if w["alg"] == "ctrlsac" else {}
    if w["alg"] == "vlsac":
        import torch
        extra["critic_noise"] = torch.randn(20, kw.get("feature_dim", 256), generator=torch.Generator().manual_seed(1234))
    agent = O.ORACLES[w["alg"]](w["S"], w["A"], init, discount=0.99, tau=0.005, **kw, **extra)
    ring = O.synthetic_ring(w["S"], w["A"], w["rows"], seed=0)  # the same ring as the GPU arm
    return agent, ring


def time_oracle(w, steps, warmup, as_written=True):
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    agent, ring = make_oracle(w, as_written)
    np.random.seed(1)
    torch.manual_seed(1)
    for _ in range(warmup):
        agent.train(ring, w["B"])
    t0 = time.perf_counter()
    for _ in range(steps):
        agent.train(ring, w["B"])
    dt = time.perf_counter() - t0
    return steps / dt, dt / steps * 1e3, torch.get_num_threads()


def run_reference(args, w, rank, world):
    """--impl reference: the reference's CPU implementation of the path (oracle port, as written) on host cores."""
    if rank != 0:
        return
    as_written = not w.get("sharded")  # the [B,B,D] broadcast needs 2.2 TB at B = 16384: matmul-restated there
    ups, ms, cores = time_oracle(w, args.steps, args.warmup, as_written=as_written)
    sample = f"{args.steps} full train() calls after {args.warmup} warm-up, reference arithmetic " + \
        ("as written ([B,B,D] broadcast logits)" if w["alg"] == "ctrlsac" and as_written else
         "with the logits restated as a matmul (SURVEY.md 8c)" if w["alg"] == "ctrlsac" else "as written")
    line = {
        "impl": "reference", "metric": "agent updates/sec", "value": ups, "unit": "updates/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong" if w.get("sharded") else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_of(args.workload, w, args.gpus),
        "cpu_baseline": {"value": ups, "unit": "updates/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": ups, "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# ---------------------------------------------------------------------------------------------------- pixel arm
def drq_args(w):
    import types
    return types.SimpleNamespace(tau=0.01, update_every=1, critic_loss="mse", stddev_schedule="linear(1.0,0.1,500000)",
                                 stddev_clip=0.3, bn_dim=w["bn"], actor_hidden_dim=w["H"], critic_hidden_dim=w["H"],
                                 encoder_lr=1e-4, actor_lr=1e-4, critic_lr=1e-4)


def ldiff_args():
    """configs/latent_diff_sr.yaml of the reference (agent/diffsrdrq)."""
    import types
    return types.SimpleNamespace(use_repr_target=True, back_critic_grad=True, critic_loss="mse", reg_coef=0.0, grad_norm=None,
                                 extra_repr_step=1, do_scale=False, repr_coef=1.0, ae_num_layers=4, ae_num_filters=32,
                                 noise_schedule="linear", ae_lr=3e-4, score_lr=3e-4, actor_lr=1e-4, critic_lr=1e-4, bn_dim=256,
                                 update_every=1, stddev_schedule="linear(1.0,0.1,500000)", stddev_clip=0.3, latent_dim=256,
                                 feature_dim=512, psi_hidden_dim=512, psi_hidden_depth=2, zeta_hidden_dim=512,
                                 zeta_hidden_depth=4, actor_hidden_dim=1024, critic_hidden_dim=1024, noise_param1=1e-4,
                                 noise_param2=0.02, num_noises=1000, tau=0.01, kl_coef=1.0, ae_coef=1.0)


LDIFF_DIMS = (4, 256, 512, 256, 512, 2, 512, 4, 1024)  # oracle Dims(A, L, feat, bn, psi_h, psi_d, zeta_h, zeta_d, H)


class _Box:
    def __init__(self, shape):
        self.shape = shape


MULV_CFG = dict(aug=True, pre_aug=False, back_q2feat=True, tanh=True, both_q=False, q_activ="relu", q_loss="huber",
                q_up_n=1, l2_norm=0.0, c_targ_tau=0.01, up_every=1, stddev_schedule="linear(1.0,0.1,500000)",
                stddev_clip=0.3, lr=1e-4, vae_w=0.5, mse_w=1.0, c_noise=0.1)


class _PixelArm:
    """The pixel agents behind one face: step(batch, i) = one updating call through the public API with host batches."""

    def __init__(self, w, precision, seed):
        from rlrep_b200 import _lib
        self.w, self.lib_mod = w, _lib
        C_, A = w["C"], w["A"]
        if w["alg"] == "drqv2":
            from oracle import drq_oracle as D  # synthetic batch + deterministic initial weights (data, not arithmetic)
            from rlrep_b200.pixel import DrQv2
            self.agent = DrQv2(_Box((C_, 84, 84)), _Box((A,)), drq_args(w), precision=precision)
            self.agent.load_state_dict(D.init_state(C_, A, w["bn"], w["H"], seed=seed))
            self.step = lambda batch, i: self.agent.train_step(iter([batch]), step=i)
            self.prefix = "rlrep_drq"
            self.h2d = 2 * w["B"] * C_ * 84 * 84 + 4 * (4 * w["B"] + 3 * w["B"] * A + 2 * w["B"])
        elif w["alg"] == "mulvdrq":
            from oracle import mulv_oracle as D
            from rlrep_b200.pixel import MuLVDrQv2
            self.agent = MuLVDrQv2((C_, 84, 84), (A,), dict(MULV_CFG, feat_dim=w["F"], hid_dim=w["H"]), precision=precision)
            self.agent.load_state_dict(D.init_state(C_, A, w["F"], w["H"], seed=seed))
            self.step = lambda batch, i: self.agent.update(iter([batch]), step=i)
            self.prefix = "rlrep_mulv"
            self.h2d = (2 * C_ + 3) * w["B"] * 84 * 84 + 4 * (4 * w["B"] + w["B"] * w["F"] + 3 * w["B"] * A +
                                                              3 * 20 * w["F"] + 2 * w["B"])
        else:
            from oracle import ldiffsr_oracle as D
            from rlrep_b200.pixel import LatentDiffSRDrQv2
            self.agent = LatentDiffSRDrQv2(_Box((C_, 84, 84)), _Box((A,)), ldiff_args(), precision=precision)
            self.agent.load_state_dict(D.init_state(D.Dims(*LDIFF_DIMS), seed=seed))
            self.step = lambda batch, i: self.agent.train_step(iter([batch]), step=i)
            self.prefix = "rlrep_ldiff"
            self.h2d = 2 * w["B"] * C_ * 84 * 84 + 4 * (4 * w["B"] * 256 + 64 * w["B"])
        self.D = D

    def fn(self, name):
        return getattr(self.agent.lib, f"{self.prefix}_{name}", None)

    def make_oracle(self):
        w, D = self.w, self.D
        if w["alg"] == "drqv2":
            o = D.OracleDrQv2(w["A"], D.init_state(w["C"], w["A"], w["bn"], w["H"], seed=0), update_every=1)
            return lambda b: o.train_step(b, 0)
        if w["alg"] == "mulvdrq":
            o = D.OracleMuLVDrQ(w["A"], D.init_state(w["C"], w["A"], w["F"], w["H"], seed=0), up_every=1)
            return lambda b: o.update(b, 0)
        d = D.Dims(*LDIFF_DIMS)
        o = D.OracleLatentDiffSR(d, D.init_state(d, seed=0), update_every=1)
        return lambda b: o.train_step(b, step=0)


def median_of(xs):
    return float(np.median(np.asarray(xs, dtype=np.float64)))


def run_pixels(args, w, rank, world, local_rank):
    """Pixel update (plain DrQ-v2, muLV-Rep DrQ-v2 or latent Diff-SR DrQ-v2): one step = one updating call on a
    [B, 9, 84, 84] uint8 batch (synthetic frames)."""
    import torch
    import torch.distributed as dist
    from rlrep_b200 import _lib
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    C_, A, B = w["C"], w["A"], w["B"]
    precision = args.precision or w.get("precision", "tf32")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def measure(prec, want_profile):
        arm = _PixelArm(w, prec, rank)
        agent, D = arm.agent, arm.D
        batches = [tuple(D.synthetic_pixel_batch(B, C_, 84, A, seed=100 * rank + i)) for i in range(4)]
        torch.manual_seed(1 + rank)
        for i in range(max(args.warmup, 3)):
            arm.step(batches[i % 4], i)
        dev, e2e, clocks, info = [], [], None, None
        resident = arm.fn("update_resident")
        for r in range(args.repeats):
            if resident is not None:  # (1) device-timed on the batch already resident in HBM
                ms = C.c_float()
                barrier()
                with ClockSampler(local_rank) as clk:
                    _lib.check(resident(agent._h, args.steps, 1.0, C.byref(ms)))
                    barrier()
                dev.append(float(ms.value))
                clocks = clocks or clk.summary()
            barrier()
            t0 = time.perf_counter()  # (2) end to end: host batch -> pinned staging -> H2D -> update -> metrics D2H
            for i in range(args.steps):
                info = arm.step(batches[i % 4], i)
            barrier()
            e2e.append((time.perf_counter() - t0) * 1e3)
        if resident is None:  # no resident entry point for this agent: the device-timed figure is the end-to-end loop
            dev = list(e2e)
        # (3) end to end with the frames already in HBM, as rlrep_b200.PixelReplayBuffer (the device-resident
        # EfficientReplayBuffer) hands them over: uint8 frame stacks are CUDA tensors, everything else stays on the host
        e2e_dev = []
        last = info  # what the last timed update returned (--dump-outputs)
        if want_profile:
            is_u8 = lambda x: (isinstance(x, np.ndarray) and x.dtype == np.uint8) or \
                              (isinstance(x, torch.Tensor) and x.dtype == torch.uint8)
            dev_batches = [tuple(torch.as_tensor(x).cuda() if is_u8(x) else x for x in b) for b in batches]
            for i in range(3):
                arm.step(dev_batches[i % 4], i)
            for r in range(min(args.repeats, 3)):
                barrier()
                t0 = time.perf_counter()
                for i in range(args.steps):
                    last = arm.step(dev_batches[i % 4], i)
                barrier()
                e2e_dev.append((time.perf_counter() - t0) * 1e3)
            del dev_batches
        out = dict(dev_ms=median_of(dev), e2e_ms=median_of(e2e), dev_all=dev, e2e_all=e2e, clocks=clocks, info=info, last=last,
                   launches=getattr(agent, "gpu_launches_last_update", 0), arm=arm, batches=batches,
                   e2e_dev_ms=median_of(e2e_dev) if e2e_dev else None)
        return out

    res = measure(precision, True)
    arm, agent, D = res["arm"], res["arm"].agent, res["arm"].D
    if args.dump_outputs and rank == 0:  # before the profiled updates below
        dump_outputs(args.dump_outputs, res["last"], agent.state_dict())
    dev_ms, e2e_ms = res["dev_ms"], res["e2e_ms"]
    launches, clocks, info = res["launches"], res["clocks"], res["info"]
    e2e_dev_ms = res.get("e2e_dev_ms")
    if world > 1:
        t = torch.tensor([dev_ms, e2e_ms, e2e_dev_ms or 0.0], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, e2e_ms, e2e_dev_ms = t.tolist()
        e2e_dev_ms = e2e_dev_ms or None
    roofline, top, cpu, other = None, [], None, None
    if rank == 0:
        hbm_peak, hbm_src = peaks()
        tf32_peak = measure_tf32_peak()
        step_s = dev_ms / args.steps * 1e-3
        prof = arm.fn("profile_update")
        agg = {}
        if prof is not None:
            cap = 4096
            names, kms = (C.c_char_p * cap)(), (C.c_float * cap)()
            kby, kfl, n = (C.c_double * cap)(), (C.c_double * cap)(), C.c_int()
            for _ in range(3):
                _lib.check(prof(agent._h, 1.0, cap, names, kms, kby, kfl, C.byref(n)))
                for i in range(min(n.value, cap)):
                    a = agg.setdefault(names[i].decode(), [0.0, 0, 0.0, 0.0])
                    a[0] += kms[i]; a[1] += 1; a[2] += kby[i]; a[3] += kfl[i]
        # kernel times from the timed configuration (CUPTI), algorithmic work per kernel from the launch records
        tl, window = graph_timeline(lambda i: arm.step(res["batches"][i % 4], i), 3)
        top = sorted(((k, v[0] / 3, v[1] // 3) for k, v in tl.items()), key=lambda x: -x[1])
        if top:
            k0 = top[0][0]
            us, cnt, union = tl[k0]
            by, fl = (agg[k0][2] / 3, agg[k0][3] / 3) if k0 in agg else (0.0, 0.0)
            t0k = us / 3 * 1e-6
            f_h, f_t = by / t0k / 1e9 / hbm_peak, fl / t0k / 1e12 / tf32_peak
            fp32_simt = precision == "fp32"
            roofline = {"kernel": k0, "bound": "hbm" if f_h >= f_t else "tensor",
                        "achieved": by / t0k / 1e9 if f_h >= f_t else fl / t0k / 1e12,
                        "peak": hbm_peak if f_h >= f_t else tf32_peak, "unit": "GB/s" if f_h >= f_t else "TFLOP/s",
                        "frac": max(f_h, f_t), "traffic": None, "share_of_step": union / 3 * 1e-6 / step_s,
                        "launches_per_step": cnt / 3, "avg_launch_us": us / max(cnt, 1),
                        "algorithmic_bytes_per_launch": by / max(cnt / 3, 1), "algorithmic_flops_per_launch": fl / max(cnt / 3, 1),
                        "tf32_peak_tflops": tf32_peak, "timing": "CUPTI activity records of 3 updates through the public API",
                        "peak_source": hbm_src + " / cuBLAS TF32 8192^3 measured in this run" +
                                       ("; fp32 mode runs on the FFMA pipes, the tensor peak is quoted for reference only" if fp32_simt else "")}
        # step roofline against the ALGORITHMIC work of the update (SURVEY.md 8d): conv / linear MACs counted per layer,
        # 28 B per parameter for Adam (+12 B per Polyak-tracked parameter); NOT the column-matrix bytes the lowering moves
        alg = pixel_algorithmic(w)
        roofline = roofline or {}
        roofline["step"] = {"algorithmic_bytes": alg["bytes"], "algorithmic_flops": alg["flops"], "params": alg["params"],
                            "roofline_ms": max(alg["bytes"] / (hbm_peak * 1e9), alg["flops"] / (tf32_peak * 1e12)) * 1e3,
                            "frac": max(alg["bytes"] / (hbm_peak * 1e9), alg["flops"] / (tf32_peak * 1e12)) / step_s,
                            "bound": "hbm" if alg["bytes"] / (hbm_peak * 1e9) >= alg["flops"] / (tf32_peak * 1e12) else "tensor",
                            "how": alg["how"]}
        if world == 1 and not args.no_cpu_baseline:
            torch.set_num_threads(os.cpu_count() or 1)
            oracle_step = arm.make_oracle()
            ob = D.synthetic_pixel_batch(B, C_, 84, A, seed=0)
            oracle_step(ob)
            t1 = time.perf_counter()
            n_cpu = {"drqv2": 20, "mulvdrq": 8}.get(w["alg"], 3)
            for _ in range(n_cpu):
                oracle_step(ob)
            dt = (time.perf_counter() - t1) / n_cpu
            cpu = {"value": 1.0 / dt, "unit": "updates/s", "cores": torch.get_num_threads(), "kind": "port",
                   "sample": f"{n_cpu} updates of the same workload after 1 warm-up ({dt * 1e3:.0f} ms each), reference "
                             f"arithmetic as written (grid_sample augmentation, F.conv2d, autograd, torch.optim.Adam)"}
    del res, arm, agent
    if world == 1 and not args.no_alt_precision:  # the other precision mode, same protocol, fewer repeats
        alt = "tf32" if precision == "fp32" else "fp32"
        keep = (args.repeats, args.steps)
        args.repeats, args.steps = min(args.repeats, 2), min(args.steps, 5)
        r2 = measure(alt, False)
        alt_steps = args.steps
        args.repeats, args.steps = keep
        other = {"precision": alt, "value": alt_steps / (r2["dev_ms"] * 1e-3), "ms_per_step": r2["dev_ms"] / alt_steps,
                 "e2e": alt_steps / (r2["e2e_ms"] * 1e-3), "steps": alt_steps}
        del r2
    if rank == 0:
        line = {"metric": "agent updates/sec", "value": world * args.steps / (dev_ms * 1e-3), "unit": "updates/s",
                "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "tf32" if precision == "tf32" else "f32", "data": "synthetic",
                "config": config_of(args.workload, w, world),
                "e2e": {"value": world * args.steps / (e2e_ms * 1e-3), "unit": "updates/s", "ms_per_step": e2e_ms / args.steps,
                        "h2d_bytes_per_step": arm_h2d(w), "d2h_bytes_per_step": 32},
                "e2e_device_replay": None if not e2e_dev_ms else {
                    "value": world * args.steps / (e2e_dev_ms * 1e-3), "unit": "updates/s",
                    "ms_per_step": e2e_dev_ms / args.steps,
                    "what": "the same public-API loop with the uint8 frame stacks as CUDA tensors, the way "
                            "rlrep_b200.PixelReplayBuffer (device-resident EfficientReplayBuffer) hands batches over: "
                            "no frame upload; actions / rewards / noise still come from the host"},
                "repeats": {"n": args.repeats, "statistic": "median"},
                "gpu_launches": int(launches) * args.steps, "gpu_launches_per_step": int(launches),
                "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "last_info": info,
                ("tf32" if precision == "fp32" else "fp32"): other,
                "top_kernels_us_per_step": [[k, round(v, 1), c] for k, v, c in top[:16]]}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def arm_h2d(w):
    B, C_, A = w["B"], w["C"], w["A"]
    if w["alg"] == "drqv2":
        return 2 * B * C_ * 84 * 84 + 4 * (4 * B + 3 * B * A + 2 * B)
    if w["alg"] == "mulvdrq":
        return (2 * C_ + 3) * B * 84 * 84 + 4 * (4 * B + B * w["F"] + 3 * B * A + 3 * 20 * w["F"] + 2 * B)
    return 2 * B * C_ * 84 * 84 + 4 * (4 * B * 256 + 64 * B)


def pixel_algorithmic(w):
    """Per-layer MAC / parameter count of one pixel update (forward + the backward passes the update needs), so the step
    roofline divides by the work of the ALGORITHM, not by what an im2col lowering moves."""
    B, C_ = w["B"], w["C"]

    def conv_stack(c_in, b):  # 4 x (3x3, 32 ch): stride 2 then stride 1 x3 on 84x84 -> 41, 39, 37, 35
        hw = [41, 39, 37, 35]
        macs = b * (hw[0] ** 2 * 9 * c_in * 32 + sum(h * h * 9 * 32 * 32 for h in hw[1:]))
        return macs, 9 * c_in * 32 + 32 + 3 * (9 * 32 * 32 + 32)

    if w["alg"] == "drqv2":
        enc, enc_p = conv_stack(C_, B)
        H, bn, A = w["H"], w["bn"], w["A"]
        trunk = 39200 * bn
        q = 2 * ((bn + A) * H + H * H + H)
        pi = bn * H + H * H + H * A
        params = enc_p + 2 * (trunk + 2 * bn) + q + pi
        # critic step: encoder fwd x2 (obs, next_obs) + bwd x1; trunk + Q fwd/bwd; target Q fwd; actor step: trunk + pi fwd/bwd + Q fwd + dgrad
        macs = enc * (2 + 2) + B * (3 * (trunk + q) + (trunk + q) + 3 * (trunk + pi) + 2 * q)
        byts = 28 * params + 12 * (q + trunk)
        how = "conv encoder 2 fwd + 1 bwd (2x fwd MACs), trunk/Q/actor MLPs fwd + dgrad + wgrad; Adam 28 B/param + Polyak 12 B/param on the critic"
    elif w["alg"] == "mulvdrq":
        enc, enc_p = conv_stack(C_, B)
        dec = B * (35 * 35 * 9 * 32 * 32 + 37 * 37 * 9 * 32 * 32 + 39 * 39 * 9 * 32 * 32 + 84 * 84 * 9 * 32 * 32 // 4 + 84 * 84 * 4 * 32 * 3)
        F, H, A = w["F"], w["H"], w["A"]
        params = 72_300_000  # SURVEY.md 8a row a16 (encoder 30k, predict_enc 29k, decoder 37k, feat_encoder 15.7M, feat_decoder 41.3M, feat_f 7.8M, actor 5.1M, critic 2.3M)
        lin = 15_681_400 + 41_334_049 + 7_841_400 + 5_077_424 + 20 * 2_308_098
        macs = enc * (3 + 2 * 2) + 3 * dec + B * 3 * lin
        byts = 28 * params + 12 * (30_368 + 2_308_098 + 15_681_400)
        how = "3 encoder passes fwd (+2 bwd), decoder fwd+bwd, wide linears fwd + dgrad + wgrad, 20-noise critic; Adam 28 B/param over 72.3 M params + Polyak"
    else:
        enc, enc_p = conv_stack(3, 4 * B)
        dec = 4 * B * (35 * 35 * 9 * 32 * 32 + 37 * 37 * 9 * 32 * 32 + 39 * 39 * 9 * 32 * 32 + 84 * 84 * 9 * 32 * 32 // 4 + 84 * 84 * 9 * 32 * 3)
        params = 20_300_000 + 285_300_000 + 2_000_000 + 6_300_000  # SURVEY.md 8a row a17
        macs = 3 * enc + 3 * dec + B * 3 * (285_300_000 + 20_000_000 + 8_300_000)
        byts = 28 * params + 12 * (285_300_000 + 20_300_000 + 6_300_000)
        how = "per-frame VAE on 4B frames fwd+bwd, 285 M-parameter score network fwd + dgrad + wgrad, AdamW 28 B/param + three Polyak targets"
    return dict(flops=2.0 * macs, bytes=float(byts), params=params, how=how)


# ---------------------------------------------------------------------------------------------------- population (configs[4])
def run_population(args, w, rank, world, local_rank):
    """`--agents-per-gpu` independent muLV-Rep DrQ-v2 agents per GPU, each with its own handle, stream, weights and data;
    their updates are issued concurrently from one host thread per agent (the C calls release the GIL), so the GPU
    co-schedules kernels of different agents.  No communication.  value = sum of the agents' updates / wall time."""
    import torch
    import torch.distributed as dist
    from rlrep_b200 import _lib
    from rlrep_b200.population import Population
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n_agents = args.agents_per_gpu
    precision = args.precision or w.get("precision", "tf32")
    C_, A, B = w["C"], w["A"], w["B"]
    arms = [_PixelArm(w, precision, seed=rank * n_agents + i) for i in range(n_agents)]
    D = arms[0].D
    batches = [[tuple(D.synthetic_pixel_batch(B, C_, 84, A, seed=1000 * rank + 10 * i + j)) for j in range(2)] for i in range(n_agents)]
    pop = Population([a.agent for a in arms])

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    torch.manual_seed(1 + rank)
    for s in range(max(args.warmup, 3)):  # warm-up one agent at a time (plans, kernel attributes), then together
        for i, a in enumerate(arms):
            a.step(batches[i][s % 2], s)
    pop.map(lambda i, ag: arms[i].step(batches[i][0], 0))

    def resident_all(steps):
        ms = [C.c_float() for _ in arms]
        pop.map(lambda i, ag: _lib.check(arms[i].fn("update_resident")(ag._h, steps, 1.0, C.byref(ms[i]))))
        return [float(m.value) for m in ms]

    # one agent alone on the GPU (the figure the population is compared with)
    ms1 = C.c_float()
    barrier()
    _lib.check(arms[0].fn("update_resident")(arms[0].agent._h, args.steps, 1.0, C.byref(ms1)))
    barrier()
    alone_ms = float(ms1.value) / args.steps
    walls, per_agent, e2e = [], None, []
    for r in range(args.repeats):
        barrier()
        with ClockSampler(local_rank) as clk:
            t0 = time.perf_counter()
            per_agent = resident_all(args.steps)
            torch.cuda.synchronize()
            walls.append((time.perf_counter() - t0) * 1e3)
            barrier()
        clocks = clk.summary()
        barrier()
        t0 = time.perf_counter()  # end to end: every agent's host batch goes through its public update()
        for s in range(args.steps):
            pop.map(lambda i, ag: arms[i].step(batches[i][s % 2], s))
        barrier()
        e2e.append((time.perf_counter() - t0) * 1e3)
    wall_ms, e2e_ms = median_of(walls), median_of(e2e)
    if world > 1:
        t = torch.tensor([wall_ms, e2e_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        wall_ms, e2e_ms = t.tolist()
    if rank == 0:
        total = world * n_agents
        cfg = config_of(args.workload, w, world)
        cfg["parallelism"] = f"population of {total} independent agents: {n_agents} per GPU on their own streams x {world} GPU(s), no collective"
        emit({"metric": "agent updates/sec", "value": total * args.steps / (wall_ms * 1e-3), "unit": "updates/s",
              "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": wall_ms / args.steps,
              "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
              "dtype": "tf32" if precision == "tf32" else "f32", "data": "synthetic", "config": cfg,
              "population": {"agents": total, "agents_per_gpu": n_agents,
                             "one_agent_alone_ms_per_update": alone_ms,
                             "one_agent_alone_updates_per_s_per_gpu": 1e3 / alone_ms,
                             "population_updates_per_s_per_gpu": n_agents * args.steps / (wall_ms * 1e-3),
                             "co_scheduling_gain": (n_agents * args.steps / (wall_ms * 1e-3)) / (1e3 / alone_ms),
                             "per_agent_device_ms_per_update": [round(m / args.steps, 3) for m in per_agent],
                             "timing": "wall clock around the concurrent region, bracketed by device synchronisation "
                                       "(each agent's own CUDA-event time is listed per agent)"},
              "e2e": {"value": total * args.steps / (e2e_ms * 1e-3), "unit": "updates/s", "ms_per_step": e2e_ms / args.steps,
                      "h2d_bytes_per_step": n_agents * arm_h2d(w), "d2h_bytes_per_step": 32 * n_agents},
              "repeats": {"n": args.repeats, "statistic": "median"},
              "gpu_launches": sum(a.agent.gpu_launches_last_update for a in arms) * args.steps,
              "gpu_launches_per_step": sum(a.agent.gpu_launches_last_update for a in arms), "clocks": clocks,
              "roofline": None, "cpu_baseline": None})
    pop.close()
    if world > 1:
        dist.destroy_process_group()


def run_pixel_reference(args, w, rank):
    if rank != 0:
        return
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    arm_oracle = _PixelArm.make_oracle
    if w["alg"] == "drqv2":
        from oracle import drq_oracle as D
    elif w["alg"] == "mulvdrq":
        from oracle import mulv_oracle as D
    else:
        from oracle import ldiffsr_oracle as D
    holder = type("H", (), {"w": w, "D": D})()
    oracle_step = arm_oracle(holder)
    ob = D.synthetic_pixel_batch(w["B"], w["C"], 84, w["A"], seed=0)
    torch.manual_seed(1)
    for _ in range(args.warmup):
        oracle_step(ob)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        oracle_step(ob)
    dt = (time.perf_counter() - t0) / args.steps
    emit({"impl": "reference", "metric": "agent updates/sec", "value": 1.0 / dt, "unit": "updates/s", "n_gpus": args.gpus,
          "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
          "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_of(args.workload, w, args.gpus),
          "cpu_baseline": {"value": 1.0 / dt, "unit": "updates/s", "cores": torch.get_num_threads(), "kind": "port",
                           "sample": f"{args.steps} updates after {args.warmup} warm-up"},
          "e2e": {"value": 1.0 / dt, "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})


# ---------------------------------------------------------------------------------------------------- GPU arm (state agents)
def time_state_agent(args, w, rank, world, local_rank, precision, barrier, repeats, want_clocks=True):
    """Builds the agent + ring of workload `w`, warms up, and times `repeats` x `steps` updates device-resident and end to
    end.  Returns a dict with the agent kept alive for profiling."""
    import torch
    import bench_data as BD  # synthetic ring + deterministic initial weights: data only
    from rlrep_b200 import ReplayBuffer, _lib
    from rlrep_b200.agents import AGENTS
    S, A, B, kw = w["S"], w["A"], w["B"], w["kw"]
    sharded = bool(w.get("sharded"))
    if sharded:
        from rlrep_b200.agents import ShardedCTRLSACAgent
        # one logical agent over all ranks: identical weights, identical seeds, the global batch split by rows
        agent = ShardedCTRLSACAgent(S, A, Space(A), discount=0.99, tau=0.005, precision=precision, **kw)
        seed = 0
    else:
        agent = AGENTS[w["alg"]](S, A, Space(A), discount=0.99, tau=0.005, precision=precision, **kw)
        seed = rank  # independent replicas: own weights, own data, own seeds
    agent.load_state_dict(BD.init_state(w["alg"], S, A, kw, seed=seed))
    ring = BD.synthetic_ring(S, A, w["rows"], seed=seed)
    buf = ReplayBuffer(S, A, max_size=w["rows"])
    buf.load(ring.state, ring.action, ring.next_state, ring.reward, ring.done)
    del ring
    np.random.seed(1 + seed)
    torch.manual_seed(1 + seed)
    for _ in range(max(args.warmup, 3)):  # warm-up through the public API (eager call, graph capture, replays)
        agent.train(buf, B)
    h = agent._h
    dev, e2e, clocks, info = [], [], None, None
    for r in range(repeats):
        # (1) device-timed, inputs resident: all indices / noise uploaded before the timed region
        draws = [agent._draw(buf, B) for _ in range(args.steps)]
        idx_all = np.ascontiguousarray(np.concatenate([d[0] for d in draws]), dtype=np.int64)
        eps_all = np.ascontiguousarray(np.concatenate([d[1] for d in draws]), dtype=np.float32)
        ms = C.c_float()
        barrier()
        with ClockSampler(local_rank) as clk:
            _lib.check(h.lib.rlrep_agent_train_resident(h.h, buf._h, idx_all.ctypes.data, eps_all.ctypes.data, args.steps,
                                                        C.byref(ms)))
            barrier()
        dev.append(float(ms.value))
        if want_clocks and clocks is None:
            clocks = clk.summary()
        # (2) end to end through agent.train(): host RNG draws, H2D of inputs, D2H of metrics, every step
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            info = agent.train(buf, B)
        barrier()
        e2e.append((time.perf_counter() - t0) * 1e3)
    # (3) the same end-to-end loop with the noise drawn by torch's CUDA generator (noise_device="cuda", the stream a
    # reference run on CUDA consumes): no host RNG, only the replay indices cross PCIe
    e2e_dn = []
    last = info  # what the last timed train() call returned (--dump-outputs)
    if not sharded:
        agent.noise_device = "cuda"
        for _ in range(3):
            agent.train(buf, B)
        for r in range(min(repeats, 3)):
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                last = agent.train(buf, B)
            barrier()
            e2e_dn.append((time.perf_counter() - t0) * 1e3)
        agent.noise_device = "cpu"
    return dict(agent=agent, buf=buf, dev_ms=median_of(dev), e2e_ms=median_of(e2e), dev_all=dev, e2e_all=e2e, clocks=clocks,
                info=info, last=last, launches=agent.gpu_launches_last_train, sharded=sharded,
                e2e_device_noise_ms=median_of(e2e_dn) if e2e_dn else None)


def state_roofline(args, w, res, dev_ms):
    """Per-kernel roofline of a state-agent workload on rank 0 (see the module docstring)."""
    from rlrep_b200 import _lib
    agent, buf, B, h = res["agent"], res["buf"], w["B"], res["agent"]._h
    cap = 8192
    names, kms = (C.c_char_p * cap)(), (C.c_float * cap)()
    kby, kfl, n = (C.c_double * cap)(), (C.c_double * cap)(), C.c_int()
    agg, reps = {}, 3
    for _ in range(reps):
        i1, e1 = agent._draw(buf, B)
        i1 = np.ascontiguousarray(i1, dtype=np.int64)
        e1 = np.ascontiguousarray(e1, dtype=np.float32)
        _lib.check(h.lib.rlrep_agent_profile_train(h.h, buf._h, i1.ctypes.data, e1.ctypes.data, cap, names, kms, kby, kfl,
                                                   C.byref(n)))
        for i in range(min(n.value, cap)):
            a = agg.setdefault(names[i].decode(), [0.0, 0, 0.0, 0.0])
            a[0] += kms[i]; a[1] += 1; a[2] += kby[i]; a[3] += kfl[i]
    ser_total = sum(v[0] for v in agg.values())
    hbm_peak, hbm_src = peaks()
    tf32_peak = measure_tf32_peak()  # cuBLAS TF32 8192^3, measured here the way MEASURED_PEAKS.json measures bf16
    traffic = {}
    tp = ROOT / "profiles" / "ncu_traffic.json"  # dram__bytes_read+write per launch from the committed ncu captures
    if tp.exists():
        traffic = json.loads(tp.read_text()).get(args.workload, {})
    step_s = dev_ms / args.steps * 1e-3
    n_tl = 4
    tl, window = graph_timeline(lambda i: agent.train(buf, B), n_tl)  # graph replays: the timed configuration

    def kernel_roofline(name):
        us, count, union = tl[name]
        by, fl = (agg[name][2] / reps * n_tl, agg[name][3] / reps * n_tl) if name in agg else (0.0, 0.0)
        t = us * 1e-6
        gbs, tfs = by / t / 1e9, fl / t / 1e12
        f_hbm, f_tc = gbs / hbm_peak, tfs / tf32_peak
        bound = "hbm" if f_hbm >= f_tc else "tensor"
        out = {"kernel": name, "bound": bound, "achieved": gbs if bound == "hbm" else tfs,
               "peak": hbm_peak if bound == "hbm" else tf32_peak, "unit": "GB/s" if bound == "hbm" else "TFLOP/s",
               "frac": max(f_hbm, f_tc), "traffic": traffic.get(name), "launches_per_step": count / n_tl,
               "avg_launch_us": us / max(count, 1), "algorithmic_bytes_per_launch": by / max(count, 1),
               "algorithmic_flops_per_launch": fl / max(count, 1), "achieved_gbs": gbs, "achieved_tflops": tfs,
               "us_per_step": us / n_tl, "share_of_step": union / n_tl * 1e-6 / step_s}
        if name in agg:  # round 1's method, kept for comparison: every launch alone on one stream, an event behind it
            out["serialized"] = {"avg_launch_us": agg[name][0] / agg[name][1] * 1e3, "share_of_profile": agg[name][0] / ser_total}
        return out

    ranked = sorted(tl, key=lambda k: -tl[k][0])
    top = [(k, tl[k][0] / n_tl, tl[k][1] // n_tl) for k in ranked]
    if not ranked:
        return None, []
    alg_bytes = algorithmic_bytes(w)
    step_flops = sum(v[3] for v in agg.values()) / reps
    t_hbm, t_tc = alg_bytes["total"] / (hbm_peak * 1e9), step_flops / (tf32_peak * 1e12)
    roofline = kernel_roofline(ranked[0])  # the kernel with the largest share of the step
    roofline["peak_source"] = hbm_src if roofline["bound"] == "hbm" else "cuBLAS TF32 8192^3 measured in this run"
    roofline["timing"] = f"CUPTI activity records of {n_tl} graph-replayed train() calls; share_of_step = time at least one " \
                         f"launch of the kernel was running / ms_per_step"
    roofline["tf32_peak_tflops"] = tf32_peak
    roofline["kernels"] = [kernel_roofline(k) for k in ranked[1:6]]
    roofline["graph_window_ms_per_step"] = window / n_tl * 1e-3
    roofline["step"] = {"algorithmic_bytes": alg_bytes["total"], "algorithmic_flops": step_flops,
                        "bound": "hbm" if t_hbm >= t_tc else "tensor",
                        "roofline_ms": max(t_hbm, t_tc) * 1e3, "frac": max(t_hbm, t_tc) / step_s,
                        "achieved_gbs": alg_bytes["total"] / step_s / 1e9,
                        "achieved_tflops": step_flops / step_s / 1e12}
    return roofline, top


def sharded_section(args, rank, world, local_rank, barrier):
    """BASELINE configs[3] inside every run of the default workload: (a) a small sharded update checked against the oracle on
    the GLOBAL batch (the driver's pytest runs on one GPU, so this is where multi-GPU parity becomes visible), (b) the
    batch-16384 update timed over all ranks.  Every rank takes part; rank 0 returns the record."""
    import torch
    import torch.distributed as dist
    import bench_data as BD
    from rlrep_b200 import ReplayBuffer
    from rlrep_b200.agents import ShardedCTRLSACAgent
    out = {}
    # ---- (a) parity: global batch 64 * world, D = 256, H = 128, three updates, TF32 (the benched mode) and fp32
    S, A, rows, n = 17, 6, 4000, 3
    kw = dict(hidden_dim=128, feature_dim=256, extra_feature_steps=2)
    Bp = 64 * world
    init = BD.init_state("ctrlsac", S, A, kw, seed=0)
    oring = BD.synthetic_ring(S, A, rows, seed=0)
    parity = {}
    for prec in ("tf32", "fp32"):
        agent = ShardedCTRLSACAgent(S, A, Space(A), discount=0.99, tau=0.005, precision=prec, **kw)
        agent.load_state_dict(init)
        buf = ReplayBuffer(S, A, max_size=rows)
        buf.load(oring.state, oring.action, oring.next_state, oring.reward, oring.done)
        np.random.seed(1)
        torch.manual_seed(1)
        infos = [agent.train(buf, Bp) for _ in range(n)]
        sd = agent.state_dict()
        digest = float(sum(v.double().abs().sum() for v in sd.values()))
        same = True
        if world > 1:
            t = torch.tensor([digest, -digest], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            same = bool(t[0].item() == digest and -t[1].item() == digest)  # max == min == mine on every rank
        if rank == 0:
            from oracle import rl_oracle as O  # the checker
            oracle = O.ORACLES["ctrlsac"](S, A, init, discount=0.99, tau=0.005, as_written=False, **kw)
            np.random.seed(1)
            torch.manual_seed(1)
            oi = [oracle.train(oring, Bp) for _ in range(n)]
            wi = max(max(0.0, abs(c[k] - o[k]) - 1e-5) / (abs(o[k]) + 1e-12) for c, o in zip(infos, oi) for k in o)
            osd = oracle.state_dict()
            wp = max(((sd[k].double() - v.double()).norm() / (v.double().norm() + 1e-30)).item()
                     for k, v in osd.items() if k != "log_alpha")
            bar = 1e-3 if prec == "tf32" else 1e-5
            parity[prec] = {"info": wi, "param": wp, "bar": bar, "ok": bool(wi < bar and wp < bar),
                            "ranks_bit_identical": same}
        agent.close()
        del agent, buf
    if rank == 0:
        parity["what"] = f"ShardedCTRLSACAgent, global batch {Bp} over {world} rank(s), D=256, H=128, {n} train() calls vs " \
                         f"the CPU oracle on the global batch: worst relative error of any info value / worst per-tensor rel-L2"
        out["sharded_parity"] = parity
    # ---- (b) timing of the batch-16384 update
    w = WORKLOADS["ctrlsac_b16384_sharded"]
    keep_steps = args.steps
    args.steps = max(3, min(args.steps, 10 if world >= 4 else 5))
    res = time_state_agent(args, w, rank, world, local_rank, args.precision or "tf32", barrier, min(args.repeats, 3), False)
    dev_ms, e2e_ms = res["dev_ms"], res["e2e_ms"]
    if world > 1:
        t = torch.tensor([dev_ms, e2e_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, e2e_ms = t.tolist()
    comm_us = None
    # every rank joins the profiled calls (they contain collectives); rank 0 keeps the numbers
    from rlrep_b200 import _lib
    agent, buf, h = res["agent"], res["buf"], res["agent"]._h
    cap = 8192
    names, kms = (C.c_char_p * cap)(), (C.c_float * cap)()
    kby, kfl, n_e = (C.c_double * cap)(), (C.c_double * cap)(), C.c_int()
    i1, e1 = agent._draw(buf, w["B"])
    i1 = np.ascontiguousarray(i1, dtype=np.int64)
    e1 = np.ascontiguousarray(e1, dtype=np.float32)
    _lib.check(h.lib.rlrep_agent_profile_train(h.h, buf._h, i1.ctypes.data, e1.ctypes.data, cap, names, kms, kby, kfl, C.byref(n_e)))
    if rank == 0:
        agg = {}
        for i in range(min(n_e.value, cap)):
            a = agg.setdefault(names[i].decode(), [0.0, 0, 0.0, 0.0])
            a[0] += kms[i]; a[1] += 1; a[2] += kby[i]; a[3] += kfl[i]
        comm_us = {k: round(v[0] * 1e3, 1) for k, v in agg.items() if k.startswith("nccl")}
        flops = sum(v[3] for v in agg.values())
        tf32_peak = measure_tf32_peak()
        step_s = dev_ms / args.steps * 1e-3
        out["sharded"] = {"workload": "ctrlsac_b16384_sharded", "value": args.steps / (dev_ms * 1e-3), "unit": "updates/s",
                          "ms_per_step": dev_ms / args.steps, "steps": args.steps, "scaling": "strong", "n_gpus": world,
                          "rows_per_gpu": w["B"] // world, "e2e_ms_per_step": e2e_ms / args.steps,
                          "gpu_launches_per_step": res["launches"],
                          "comm_us_serialized_per_step": comm_us,
                          "roofline": {"bound": "tensor", "algorithmic_flops_per_gpu": flops, "tf32_peak_tflops": tf32_peak,
                                       "achieved_tflops_per_gpu": flops / step_s / 1e12,
                                       "frac": flops / step_s / 1e12 / tf32_peak},
                          "top_kernels_serialized_us": sorted(([k, round(v[0] * 1e3, 1), v[1]] for k, v in agg.items()),
                                                              key=lambda x: -x[1])[:8]}
    agent.close()
    args.steps = keep_steps
    return out


def run_ours(args, w, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    sharded = bool(w.get("sharded"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:  # the sharded agent at N = 1 still goes through a (single-rank) process group and communicator; an in-process
        #    store instead of a TCP one, so that runs sharing a host never compete for a port
        dist.init_process_group("gloo", store=dist.HashStore(), rank=0, world_size=1)
    precision = args.precision or "tf32"

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    res = time_state_agent(args, w, rank, world, local_rank, precision, barrier, args.repeats)
    dev_ms, e2e_ms = res["dev_ms"], res["e2e_ms"]
    if world > 1:
        t = torch.tensor([dev_ms, e2e_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, e2e_ms = t.tolist()
    h = res["agent"]._h
    ni, ne = h.n_idx, h.n_eps
    if args.dump_outputs and rank == 0:  # before the profiled calls below, which train the agent further
        dump_outputs(args.dump_outputs, res["last"], res["agent"].state_dict())

    roofline, top = None, []
    if sharded and rank != 0:  # the sharded update contains collectives: every rank has to take part in the profiled calls
        from rlrep_b200 import _lib
        for _ in range(3):
            i1, e1 = res["agent"]._draw(res["buf"], w["B"])
            i1 = np.ascontiguousarray(i1, dtype=np.int64)
            e1 = np.ascontiguousarray(e1, dtype=np.float32)
            _lib.check(h.lib.rlrep_agent_profile_train(h.h, res["buf"]._h, i1.ctypes.data, e1.ctypes.data, 0, None, None,
                                                       None, None, C.byref(C.c_int())))
        for _ in range(4):
            res["agent"].train(res["buf"], w["B"])
    if rank == 0:
        roofline, top = state_roofline(args, w, res, dev_ms)
    launches, info, clocks = res["launches"], res["info"], res["clocks"]
    e2e_dn_ms = res.get("e2e_device_noise_ms")
    if world > 1 and e2e_dn_ms is not None:
        t = torch.tensor([e2e_dn_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_dn_ms = t.item()
    if sharded:
        res["agent"].close()
    del res

    # ---- the strict-precision figure next to the TF32 one (rank 0, N = 1)
    fp32 = None
    if world == 1 and not sharded and not args.no_alt_precision and precision == "tf32":
        keep = args.steps
        args.steps = max(5, min(args.steps, 20))
        r32 = time_state_agent(args, w, rank, world, local_rank, "fp32", barrier, min(args.repeats, 3), False)
        fp32 = {"value": args.steps / (r32["dev_ms"] * 1e-3), "unit": "updates/s", "ms_per_step": r32["dev_ms"] / args.steps,
                "e2e": args.steps / (r32["e2e_ms"] * 1e-3), "steps": args.steps,
                "what": 'precision="fp32": every GEMM on the IEEE-fp32 FFMA kernels (parity bar 1e-5)'}
        args.steps = keep
        del r32

    # ---- CPU baseline: the oracle port on this box's host cores (rank 0, N = 1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not sharded:
        n_cpu = {"ctrlsac": 6, "vlsac": 30, "spedersac": 60}.get(w["alg"], 200)  # ~10-30 s of CPU work
        ups, ms_cpu, cores = time_oracle(w, n_cpu, 1, as_written=True)
        cpu = {"value": ups, "unit": "updates/s", "cores": cores, "kind": "port",
               "sample": f"{n_cpu} full train() calls of the same workload after 1 warm-up ({ms_cpu:.0f} ms each), "
                         f"reference arithmetic as written" + (" (broadcast logits)" if w["alg"] == "ctrlsac" else "")}

    # ---- BASELINE configs[3] rides along with the default workload at every N (strong-scaling curve + multi-GPU parity)
    extra = {}
    if args.workload == "ctrlsac_hc_b256" and not args.no_sharded:
        extra = sharded_section(args, rank, world, local_rank, barrier)

    if rank == 0:
        n_agents = 1 if sharded else world  # a sharded run is ONE agent's update, however many GPUs compute it
        line = {
            "metric": "agent updates/sec", "value": n_agents * args.steps / (dev_ms * 1e-3), "unit": "updates/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps,
            "higher_is_better": True, "scaling": "strong" if sharded else "weak", "vs_baseline": None,
            "dtype": "tf32" if precision == "tf32" else "f32", "data": "synthetic",
            "config": config_of(args.workload, w, world),
            "e2e": {"value": n_agents * args.steps / (e2e_ms * 1e-3), "unit": "updates/s", "ms_per_step": e2e_ms / args.steps,
                    "h2d_bytes_per_step": ni * 8 + ne * 4, "d2h_bytes_per_step": 32 * 4},
            "e2e_device_noise": None if e2e_dn_ms is None else {
                "value": n_agents * args.steps / (e2e_dn_ms * 1e-3), "unit": "updates/s",
                "ms_per_step": e2e_dn_ms / args.steps, "h2d_bytes_per_step": ni * 8, "d2h_bytes_per_step": 32 * 4,
                "what": 'agent.train() with noise_device="cuda": the Gaussian noise is drawn by torch\'s CUDA generator '
                        "(what the reference does when run on CUDA) instead of the CPU generator + upload"},
            "repeats": {"n": args.repeats, "statistic": "median",
                        "what": f"the {args.steps}-step timed loop is run {args.repeats} times; value / e2e are the median repeat"},
            "gpu_launches": launches * args.steps,
            "gpu_launches_per_step": launches,
            "clocks": clocks,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "fp32": fp32,
            "top_kernels_us_per_step": [[k, round(v, 1), c] for k, v, c in top[:8]],
            "last_info": info,
        }
        line.update(extra)
        emit(line)
    dist.destroy_process_group()


PIXEL_ALGS = ("drqv2", "mulvdrq", "ldiffsr")


def default_counts(w, impl):
    """(steps, warmup) of a run that does not give --steps / --warmup: 100 / 5, fewer steps where one step is slow.
    An explicit --steps is always used as given, and so is an explicit --warmup, except that the CUDA paths warm up at
    least 3 steps (eager call, graph capture, replay) and report the count they used."""
    pixel = w["alg"] in PIXEL_ALGS
    if impl == "reference":  # bounded samples of CPU work
        if pixel:
            return {"drqv2": 20, "mulvdrq": 8}.get(w["alg"], 3), 2
        if w.get("sharded"):
            return 2, 0  # ~17 TFLOP per update on the host cores
        return (40 if w["alg"] == "ctrlsac" else 100), 5  # ctrlsac: ~0.5-2 s of CPU work per update
    if w.get("population"):
        return 20, 5
    return (50 if pixel else 100), 5


def main():
    # stdout carries the JSON line and nothing else: native libraries (NCCL's version banner ...) write to fd 1 directly,
    # so fd 1 is pointed at stderr for the duration of the run and the JSON line goes to the saved real stdout.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps; default 100, fewer where one step is slow "
                    "(see default_counts)")
    ap.add_argument("--warmup", type=int, default=None, help="warm-up steps; default 5, at least 3 on the CUDA paths (see default_counts)")
    ap.add_argument("--repeats", type=int, default=5, help="the timed K-step loop is repeated this many times; the median is reported")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="ctrlsac_hc_b256", choices=list(WORKLOADS))
    ap.add_argument("--precision", default=None, choices=["tf32", "fp32"], help="default: tf32 (state agents), fp32 (pixel agents)")
    ap.add_argument("--agents-per-gpu", type=int, default=8, help="population workloads: agents (handles / streams) per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-alt-precision", action="store_true", help="skip the second (fp32 / tf32) figure")
    ap.add_argument("--no-sharded", action="store_true", help="skip the configs[3] section of the default workload")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the metrics of the last timed update and the parameters "
                    "after it to DIR/<name>.npy (at most 64 MB; a fixed sample of larger parameter sets; which timed loop "
                    "that is: see dump_outputs)")
    args = ap.parse_args()
    w = WORKLOADS[args.workload]
    steps, warmup = default_counts(w, args.impl)
    args.steps = steps if args.steps is None else args.steps
    args.warmup = warmup if args.warmup is None else args.warmup
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs covers the CUDA implementation (--impl ours)")
    if args.dump_outputs and w.get("population"):
        # the members draw their noise from torch's one CPU generator from concurrent threads: which member receives which
        # draws follows the thread schedule, so no two runs compute the same updates
        ap.error("--dump-outputs: a population's updates differ from run to run, there is nothing to compare")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if w["alg"] in PIXEL_ALGS:
        if args.impl == "reference":
            run_pixel_reference(args, w, rank)
        elif w.get("population"):
            run_population(args, w, rank, world, local_rank)
        else:
            run_pixels(args, w, rank, world, local_rank)
        return
    if args.impl == "reference":
        run_reference(args, w, rank, world)
        return
    run_ours(args, w, rank, world, local_rank)


if __name__ == "__main__":
    main()
