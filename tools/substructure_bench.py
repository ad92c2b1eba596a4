"""Kernel time of mmb_jet_substructure (N-subjettiness tau1..tau3 + e2, e3, D2) on the device, and the CPU oracle's rate on the
same jets for context.

    python tools/substructure_bench.py [--out profiles/substructure_bench.json]

Batches of 16 384 and 131 072 jets at N = 128, with JetClass-like multiplicities (normal(45, 18), as the C5 pipeline draws
them) and with every slot used.  Kernel time: CUDA events around `--iters` back-to-back launches after a warm-up (the inputs,
<= 200 MB, are read once per launch; the 16 384-jet batch fits in L2).  The oracle (oracle_substructure, OpenMP over jets,
brute-force clustering) runs on the first `--cpu-jets` jets of each batch.  Prints one JSON line with the card's name and power
limit."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import substructure_oracle as so  # noqa: E402
from multimodal_particles_b200.observables import jet_substructure  # noqa: E402


def batch(B, N, full, seed):
    g = np.random.default_rng(seed)
    mult = np.full(B, N) if full else np.clip(np.rint(g.normal(45, 18, B)), 1, N).astype(int)
    mask = (np.arange(N)[None] < mult[:, None]).astype(np.uint8)
    x = np.empty((B, N, 3), np.float32)
    x[..., 0] = g.exponential(1.0, (B, N)) * 20.0 / (1.0 + np.arange(N)[None] * 0.1) + 0.01
    x[..., 1] = g.normal(0.0, 0.3, (B, N))
    x[..., 2] = g.normal(0.0, 0.3, (B, N))
    return x * mask[..., None], mask, mult


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as exc:   # report, do not guess
        q = f"unavailable ({type(exc).__name__})"
    return name, q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--cpu-jets", type=int, default=4096)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("substructure_bench measures the kernel on a CUDA device; none is visible")
    name, power = card()
    rows = []
    for B in (16384, 131072):
        for full in (False, True):
            x, mask, mult = batch(B, 128, full, B + full)
            xd, md = torch.from_numpy(x).cuda(), torch.from_numpy(mask).cuda()
            out = jet_substructure(xd, md)
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(args.iters):
                out = jet_substructure(xd, md)
            e.record()
            torch.cuda.synchronize()
            ms = s.elapsed_time(e) / args.iters
            nc = min(args.cpu_jets, B)
            t0 = time.perf_counter()
            want, _ = so.jet_substructure(x[:nc], mask[:nc])
            cpu_s = time.perf_counter() - t0
            got = out[:nc].cpu().numpy()
            ok = ~np.isnan(want)
            rows.append({"jets": B, "multiplicity": "all 128" if full else "normal(45, 18) clipped to [1, 128]",
                         "mean_multiplicity": float(mult.mean()), "kernel_ms": ms, "jets_per_s": B / (ms * 1e-3),
                         "oracle_jets": nc, "oracle_threads": so.lib().mmbo_substructure_threads(), "oracle_jets_per_s": nc / cpu_s,
                         "max_rel_err_d2_vs_oracle": float(np.nanmax(np.abs(got[:, 7] - want[:, 7])[ok[:, 7]] /
                                                                     np.abs(want[:, 7])[ok[:, 7]]))})
    rec = {"workload": "mmb_jet_substructure, N = 128, R = 0.8, beta = 1 (one 128-thread block per jet)", "gpu": name,
           "power_limit_and_max_sm_clock": power, "iters": args.iters, "rows": rows}
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
