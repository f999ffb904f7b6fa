"""Time the pixel agents' act path: DrQ-v2 (C 9, A 4, bn 50, H 1024) and muLV-Rep (C 9, A 4, feat 100, H 1024), each
on a handle prepared at batch 256, in both precision modes.

* Wall time per call, host clock around the synchronous Python API (median of --calls calls after --warmup), for N = 1
  (`select_action` / `act`) and for N = 8 and 64 (`select_actions` / `act_batch`).
* Device time of every kernel of one N = 1 and one N = 64 call (torch.profiler, CUDA activities, in a pass of its own).
* With --baseline ROOT: the N = 1 timing of another build of this project (a checkout with its library built), run in
  subprocesses that alternate with this tree's, --rounds times each, so both see the same machine state.

Prints the GPU's name and power limit (read-only nvidia-smi query) and writes one JSON file (--out).

    python scripts/pixel_act_timing.py --baseline ../parent --out profiles/pixel_act_b200.json
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
CONFIGS = [(kind, prec) for kind in ("drq", "mulv") for prec in ("fp32", "tf32")]
STEP = 250000  # past muLV-Rep's exploration phase: every call samples TruncatedNormal(mu, stddev)


class _Box:
    def __init__(self, shape):
        self.shape = shape


def _make(kind, precision):
    """(single act, batched act or None) on a handle prepared at batch 256 with init_state(seed=0) weights."""
    import types
    from oracle import drq_oracle as D
    from oracle import mulv_oracle as M
    from rlrep_b200 import pixel
    if kind == "drq":
        args = types.SimpleNamespace(tau=0.01, update_every=2, critic_loss="mse", stddev_schedule="linear(1.0,0.1,500000)",
                                     stddev_clip=0.3, bn_dim=50, actor_hidden_dim=1024, critic_hidden_dim=1024,
                                     encoder_lr=1e-4, actor_lr=1e-4, critic_lr=1e-4)
        a = pixel.DrQv2(_Box((9, 84, 84)), _Box((4,)), args, precision=precision)
        a.load_state_dict(D.init_state(9, 4, 50, 1024, seed=0))
        single = lambda o: a.select_action(o, STEP)
        batched = (lambda o: a.select_actions(o, STEP)) if hasattr(a, "select_actions") else None
    else:
        cfg = dict(feat_dim=100, hid_dim=1024, stddev_schedule="linear(1.0,0.1,500000)", stddev_clip=0.3)
        a = pixel.MuLVDrQv2((9, 84, 84), (4,), cfg, precision=precision)
        a.load_state_dict(M.init_state(9, 4, 100, 1024, seed=0))
        single = lambda o: a.act(o, STEP, False)
        batched = (lambda o: a.act_batch(o, STEP, False)) if hasattr(a, "act_batch") else None
    a.prepare(256)
    return a, single, batched


def _wall_us(fn, calls, warmup):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(calls):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    ts.sort()
    return {"median_us": 1e6 * statistics.median(ts), "p10_us": 1e6 * ts[len(ts) // 10],
            "p90_us": 1e6 * ts[(9 * len(ts)) // 10], "calls": calls}


def _kernels(fn):
    """[(name, device us)] of every kernel and copy of one call, in launch order."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    ev.sort(key=lambda e: e.time_range.start)
    return [{"name": e.name[:160], "us": round(e.time_range.end - e.time_range.start, 2)} for e in ev]


def worker(root, full, calls, warmup):
    """Runs inside `root` (its rlrep_b200 and oracle); prints one JSON line."""
    sys.path.insert(0, str(root))
    import torch
    from oracle import drq_oracle as D
    torch.cuda.init()
    frames = D.synthetic_pixel_batch(64, 9, 84, 4, seed=3).img
    out = {}
    for kind, prec in CONFIGS:
        agent, single, batched = _make(kind, prec)
        torch.manual_seed(0)
        r = {"n1": _wall_us(lambda: single(frames[0]), calls, warmup)}
        if full:
            for n in (8, 64):
                r[f"n{n}"] = _wall_us(lambda: batched(frames[:n]), calls, warmup)
                r[f"n{n}"]["per_obs_us"] = r[f"n{n}"]["median_us"] / n
            r["kernels_n1"] = _kernels(lambda: single(frames[0]))
            r["kernels_n64"] = _kernels(lambda: batched(frames[:64]))
        agent.close()
        out[f"{kind}_{prec}"] = r
    print("RESULT " + json.dumps(out), flush=True)


def _run_worker(root, full, calls, warmup):
    cmd = [sys.executable, str(Path(__file__).resolve()), "--worker", str(root), "--calls", str(calls), "--warmup",
           str(warmup)] + (["--full"] if full else [])
    r = subprocess.run(cmd, cwd=str(root), capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError(f"worker in {root} failed")
    line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")][-1]
    return json.loads(line[len("RESULT "):])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline", type=Path, default=None, help="another built checkout to compare N = 1 against")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--calls", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--out", type=Path, default=ROOT / "profiles" / "pixel_act_b200.json")
    ap.add_argument("--worker", type=Path, default=None)
    ap.add_argument("--full", action="store_true")
    a = ap.parse_args()
    if a.worker is not None:
        worker(a.worker, a.full, a.calls, a.warmup)
        return
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    print(f"GPU: {q}")
    res = {"gpu": q, "step": STEP, "batch": 256, "calls": a.calls, "warmup": a.warmup,
           "configs": {"drq": "C 9, A 4, bn 50, H 1024", "mulv": "C 9, A 4, feat 100, H 1024"}}
    if a.baseline is not None:
        cmp = {k: {"baseline_us": [], "this_us": []} for k in (f"{x}_{y}" for x, y in CONFIGS)}
        for rnd in range(a.rounds):
            for which, root in (("baseline_us", a.baseline.resolve()), ("this_us", ROOT)):
                r = _run_worker(root, False, a.calls, a.warmup)
                for k, v in r.items():
                    cmp[k][which].append(round(v["n1"]["median_us"], 2))
                print(f"round {rnd} {which}: " + ", ".join(f"{k} {v['n1']['median_us']:.1f} us" for k, v in r.items()),
                      flush=True)
        for k, v in cmp.items():
            v["ratio_this_over_baseline"] = round(statistics.median(v["this_us"]) / statistics.median(v["baseline_us"]), 4)
        res["n1_vs_baseline"] = cmp
    full = _run_worker(ROOT, True, a.calls, a.warmup)
    res["this"] = full
    for k, v in full.items():
        print(f"{k}: N=1 {v['n1']['median_us']:.1f} us/call; N=8 {v['n8']['median_us']:.1f} us/call "
              f"({v['n8']['per_obs_us']:.2f} us/obs); N=64 {v['n64']['median_us']:.1f} us/call ({v['n64']['per_obs_us']:.2f} us/obs)")
        for tag in ("kernels_n1", "kernels_n64"):
            print(f"  {tag}: " + "; ".join(f"{e['name'][:40]} {e['us']:.1f}" for e in v[tag]))
    a.out.parent.mkdir(parents=True, exist_ok=True)
    a.out.write_text(json.dumps(res, indent=1) + "\n")
    print(f"wrote {a.out}")


if __name__ == "__main__":
    main()
