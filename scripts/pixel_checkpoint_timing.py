"""Save and load one full-size latent Diff-SR checkpoint (configs/latent_diff_sr.yaml sizes: 9 x 84 x 84 observations,
A 4, batch 256, ≈314 M parameters) and report the file size and the wall time of both calls.

The agent makes two updates on synthetic batches first, so the moments and counters are those of a running agent.
`save` is timed from the call to the file being written; `load` into a second agent whose handle is already prepared at
batch 256 (the handle's creation is reported on its own).  The loaded agent's counters and a sample of its tensors are
checked against the saved ones.  The file goes to a temporary directory and is deleted at the end.

Prints the GPU's name and power limit (read-only nvidia-smi query) and writes one JSON file (--out).

    python scripts/pixel_checkpoint_timing.py --out profiles/pixel_checkpoint_b200.json
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--precision", default="tf32", choices=["tf32", "fp32"])
    a = ap.parse_args()
    sys.path.insert(0, str(ROOT))
    import torch
    from bench import LDIFF_DIMS, _Box, ldiff_args
    from oracle import ldiffsr_oracle as O
    from rlrep_b200.pixel import LatentDiffSRDrQv2

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    print(f"GPU: {q}")
    d, B = O.Dims(*LDIFF_DIMS), 256
    agent = LatentDiffSRDrQv2(_Box((9, 84, 84)), _Box((d.A,)), ldiff_args(), precision=a.precision)
    agent.load_state_dict(O.init_state(d, seed=0))
    torch.manual_seed(1)
    for i in range(2):
        agent.train_step(iter([tuple(O.synthetic_pixel_batch(B, 9, 84, d.A, seed=i))]), step=i)
    n_params = sum(t.numel() for k, t in agent.state_dict().items() if "_target." not in k)

    tmp = tempfile.mkdtemp(prefix="rlrep_ckpt_")
    try:
        path = os.path.join(tmp, "ldiffsr.pt")
        t0 = time.perf_counter()
        agent.save(path)
        save_s = time.perf_counter() - t0
        size = os.path.getsize(path)

        other = LatentDiffSRDrQv2(_Box((9, 84, 84)), _Box((d.A,)), ldiff_args(), precision=a.precision)
        t0 = time.perf_counter()
        other.prepare(B)
        prepare_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        other.load(path)
        torch.cuda.synchronize()
        load_s = time.perf_counter() - t0
    finally:
        shutil.rmtree(tmp, ignore_errors=True)

    o1, o2 = agent.optimizer_state_dict(), other.optimizer_state_dict()
    assert o1["control"] == o2["control"], (o1["control"], o2["control"])
    s1, s2 = agent.state_dict(), other.state_dict()
    sample = [k for k in s1 if k.startswith(("score.zeta.fc.", "vae_target.encoder.convs.2.", "critic.", "actor."))]
    assert sample and all(torch.equal(s1[k], s2[k]) for k in sample)
    assert all(torch.equal(o1[k], o2[k]) for k in o1 if k.startswith(("optim.m/score.zeta.", "optim.v/actor.")))

    res = {"gpu": q, "precision": a.precision, "batch": B, "params": n_params, "file_bytes": size,
           "file_gb": size / 1e9, "save_s": save_s, "prepare_s": prepare_s, "load_s": load_s,
           "control": o1["control"], "tmpdir": tempfile.gettempdir(),
           "what": "wall time of agent.save(path) and of agent.load(path) into a handle prepared at batch 256"}
    print(json.dumps(res, indent=1))
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(res, indent=1) + "\n")
    agent.close()
    other.close()


if __name__ == "__main__":
    main()
