"""SAC seed populations on one GPU: aggregate updates/s of N seeds trained three ways (BASELINE config 1 shapes: S = 17,
A = 6, hidden 256, batch 256, TF32).

  (a) SACPopulation: one handle, one batched update for all N members -- device-timed through train_resident (inputs
      resident in HBM, CUDA events) and end to end through train() (host RNG draws, staging, one synchronise per call);
  (b) N lone SACAgent handles under rlrep_b200.Population (one host thread and stream per agent): wall clock over K
      train() rounds, ending in a device synchronise;
  (c) one lone SACAgent: device-timed through train_resident and end to end through train().

The arms run alternately inside every repeat; each figure is the median of the repeats.  The card's name and power limit
are read in the same run and stored with the numbers.

    python scripts/sac_population_timing.py [--out profiles/sac_population_b200.json] [--steps 50] [--repeats 5]
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

S, A, H, B = 17, 6, 256, 256


class Space:
    low, high = -np.ones(A, np.float32), np.ones(A, np.float32)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else ""
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": line}


def buffers(n, rows):
    from rlrep_b200 import ReplayBuffer
    rng = np.random.RandomState(0)
    out = []
    for _ in range(n):
        b = ReplayBuffer(S, A, max_size=rows)
        b.load(rng.randn(rows, S), rng.uniform(-1, 1, (rows, A)), rng.randn(rows, S), rng.randn(rows, 1),
               (rng.rand(rows, 1) < 0.01).astype(np.float64))
        out.append(b)
    return out


def resident_inputs(n, steps, rows):
    rng = np.random.RandomState(1)
    idx = rng.randint(0, rows, size=(steps, n, B)).astype(np.int64)
    eps = rng.randn(steps, n, 2 * B * A).astype(np.float32)
    return idx, eps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "sac_population_b200.json"))
    ap.add_argument("--members", default="1,2,4,8,16,32,64")
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--rows", type=int, default=20000)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "the timing needs a CUDA device"
    from rlrep_b200 import Population, SACAgent, SACPopulation
    K = a.steps
    result = {"workload": {"state_dim": S, "action_dim": A, "hidden_dim": H, "batch_size": B, "precision": "tf32",
                           "steps_per_window": K, "repeats": a.repeats},
              "card": card(), "rows": []}
    for n in [int(x) for x in a.members.split(",")]:
        bufs = buffers(n, a.rows)
        pop = SACPopulation(list(range(n)), S, A, Space(), hidden_dim=H)
        lones = [SACAgent(S, A, Space(), hidden_dim=H) for _ in range(n)]
        threaded = Population(lones)
        idx, eps = resident_inputs(n, K, a.rows)
        for _ in range(3):  # eager call, graph capture, first replay of every handle
            pop.train(bufs, B)
            threaded.map(lambda i, ag: ag.train(bufs[i], B))
        lone = lones[0]
        t = {k: [] for k in ("pop_device", "pop_e2e", "threaded_e2e", "lone_device", "lone_e2e")}
        for _ in range(a.repeats):
            t["pop_device"].append(pop.train_resident(bufs, idx, eps, K) / 1e3)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(K):
                pop.train(bufs, B)
            torch.cuda.synchronize()
            t["pop_e2e"].append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            for _ in range(K):
                threaded.map(lambda i, ag: ag.train(bufs[i], B))
            torch.cuda.synchronize()
            t["threaded_e2e"].append(time.perf_counter() - t0)
            import ctypes as C
            from rlrep_b200 import _lib
            ms = C.c_float()
            li, le = np.ascontiguousarray(idx[:, 0]), np.ascontiguousarray(eps[:, 0])
            _lib.check(lone._h.lib.rlrep_agent_train_resident(lone._h.h, bufs[0]._h, li.ctypes.data, le.ctypes.data, K,
                                                              C.byref(ms)))
            t["lone_device"].append(ms.value / 1e3)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(K):
                lone.train(bufs[0], B)
            torch.cuda.synchronize()
            t["lone_e2e"].append(time.perf_counter() - t0)
        med = {k: statistics.median(v) for k, v in t.items()}
        row = {"members": n,
               "population_device_updates_per_s": n * K / med["pop_device"],
               "population_e2e_updates_per_s": n * K / med["pop_e2e"],
               "threaded_e2e_updates_per_s": n * K / med["threaded_e2e"],
               "lone_device_updates_per_s": K / med["lone_device"],
               "lone_e2e_updates_per_s": K / med["lone_e2e"],
               "population_launches_per_update": pop.gpu_launches_last_train,
               "lone_launches_per_update": lone.gpu_launches_last_train,
               "seconds": {k: v for k, v in t.items()}}
        print(json.dumps({k: (round(v, 1) if isinstance(v, float) else v) for k, v in row.items() if k != "seconds"}),
              flush=True)
        result["rows"].append(row)
        threaded.close()
        pop.close()
        del bufs
        torch.cuda.empty_cache()
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(result, indent=1) + "\n")
    print("wrote", a.out)


if __name__ == "__main__":
    main()
