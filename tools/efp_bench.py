"""Device time of the energy flow polynomials (mmb_energy_flow_polynomials), of FPD and KPD, and of the 1 M-jet C5 run with and
without the EFP pass, in one command.

    python tools/efp_bench.py [--out profiles/efp_bench.json] [--jets 1048576]

- EFP kernel: 16 384-jet batches at N = 128, JetClass-like multiplicities (normal(45, 18) clipped to [1, 128], as the C5 pipeline
  draws them) and every slot used.  CUDA events around `--iters` back-to-back launches after a warm-up.  The numpy fp64 closed
  forms of tests/efp_oracle.py run on the first `--cpu-jets` jets of each batch, for the rate and the largest relative deviation.
- FPD and KPD at their defaults (20 x 10 draws of 20 000-50 000 rows; 10 batches of 5 000) and KPD with batches of 100 000, on the
  five d = 4 EFPs of two independent 131 072-jet JetClass-like batches.  Host clock around each call, which ends in a device
  synchronisation (both read their result on the host).
- The one-GPU C5 run (`pipeline.sharded_generation_run`, 16 384-jet micro-batches) without and with `efp=True`, alternated
  `--repeats` times.
Prints one JSON line per measurement and one summary line, all with the card's name and power limit."""
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
import bench  # noqa: E402
import efp_oracle as eo  # noqa: E402
from multimodal_particles_b200.observables import energy_flow_polynomials, fpd, kpd  # noqa: E402
from multimodal_particles_b200.pipeline import sharded_generation_run  # noqa: E402


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


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--cpu-jets", type=int, default=1024)
    ap.add_argument("--jets", type=int, default=1 << 20)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("efp_bench measures on a CUDA device; none is visible")
    name, power = card()
    lines = []

    def emit(rec):
        rec.update(card=name, power_limit_and_max_sm_clock=power)
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)

    summary = {}
    for full in (False, True):
        x, mask, mult = batch(16384, 128, full, 16384 + full)
        xd, md = torch.from_numpy(x).cuda(), torch.from_numpy(mask).cuda()
        out = energy_flow_polynomials(xd, md)
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(args.iters):
            out = energy_flow_polynomials(xd, md)
        e.record()
        torch.cuda.synchronize()
        ms = s.elapsed_time(e) / args.iters
        nc = args.cpu_jets
        t0 = time.perf_counter()
        want = eo.numpy_batch(x[:nc], mask[:nc])
        cpu_s = time.perf_counter() - t0
        got = out[:nc].cpu().numpy().astype(np.float64)
        rel = float(np.nanmax(np.abs(got - want) / np.maximum(np.abs(want), 1e-300)))
        key = "all_128" if full else "jetclass_like"
        summary[f"efp_jets_per_s_{key}"] = 16384 / (ms * 1e-3)
        emit({"measure": "efp_kernel", "jets": 16384, "multiplicity": "all 128" if full else "normal(45, 18) clipped to [1, 128]",
              "mean_multiplicity": float(mult.mean()), "kernel_ms": ms, "jets_per_s": 16384 / (ms * 1e-3),
              "numpy_jets": nc, "numpy_jets_per_s": nc / cpu_s, "max_rel_dev_vs_numpy_fp64": rel})

    feats = []
    for seed in (1, 2):
        x, mask, _ = batch(131072, 128, False, seed)
        feats.append(energy_flow_polynomials(torch.from_numpy(x).cuda(), torch.from_numpy(mask).cuda())[:, 1:].contiguous())
    real, gen = feats
    fpd(real, gen)                                                  # warm-up: eigh / curve_fit / generator set-up
    (fv, s_fpd) = timed(lambda: fpd(real, gen))
    (kv, s_kpd) = timed(lambda: kpd(real, gen))
    (kv_big, s_kpd_big) = timed(lambda: kpd(real, gen, batch_size=100_000))
    summary.update(fpd_seconds=s_fpd, kpd_seconds=s_kpd, kpd_100k_seconds=s_kpd_big)
    emit({"measure": "fpd_kpd", "rows": [len(real), len(gen)], "features": "efp4_* of two independent JetClass-like batches",
          "fpd": list(fv), "fpd_seconds": s_fpd, "kpd": list(kv), "kpd_seconds": s_kpd, "kpd_batch_100000": list(kv_big),
          "kpd_batch_100000_seconds": s_kpd_big})

    dev = torch.device("cuda", 0)
    cfg, model = bench.build_model(dev)
    runs = {False: [], True: []}
    for _ in range(args.repeats):
        for efp in (False, True):
            rec = sharded_generation_run(model, cfg, args.jets, 0, 1, dev, micro_batch=16384, n_particles=bench.N_PART, efp=efp)
            runs[efp].append(rec["seconds"])
            emit({"measure": "c5_1gpu", "jets": args.jets, "efp": efp, "seconds": rec["seconds"], "jets_per_s": rec["value"],
                  "histogram_sha1": rec["histogram_sha1"]})
    base, with_efp = min(runs[False]), min(runs[True])
    summary.update(c5_seconds_without_efp=runs[False], c5_seconds_with_efp=runs[True], c5_overhead_of_best=with_efp / base - 1.0)
    emit(dict(measure="summary", **summary))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
