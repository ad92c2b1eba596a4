"""Device time and accuracy of every EFP of degree <= 4 (mmb_energy_flow_polynomials_d4) against the JetNet set
(mmb_energy_flow_polynomials), of FPD and KPD on the 36 features, and of the 1 M-jet C5 run with and without ``fpd_reference``,
in one command.

    python tools/efp_d4_bench.py [--out profiles/efp_d4_bench.json] [--jets 1048576] [--reference-jets 131072]

- Kernels: the same 16 384-jet batches at N = 128 as tools/efp_bench.py (JetClass-like multiplicities, normal(45, 18) clipped
  to [1, 128], and every slot used).  CUDA events around `--iters` back-to-back launches of one kernel, the two kernels
  alternated `--rounds` times after a warm-up; the best round of each is reported, with the median.  The numpy fp64 closed forms
  of tests/efp_d4_oracle.py on the first `--cpu-jets` jets give the largest relative deviation of each column set, and the
  shared columns are compared bit for bit.
- FPD and KPD at their defaults on the 36 features (FPD_EFP_COLUMNS) of two independent 131 072-jet JetClass-like batches, and
  for comparison on the five efp4_* columns of the same jets.  Host clock around each call (each ends by reading its result on
  the host), after a warm-up call.
- The one-GPU C5 run (`pipeline.sharded_generation_run`, 16 384-jet micro-batches) without and with `fpd_reference` (built by
  `pipeline.reference_fpd_features`), alternated `--repeats` times; best of each.
Prints one JSON line per measurement and one summary line, all with the card's name and power limit."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
import efp_d4_oracle as do  # noqa: E402
import efp_oracle as eo  # noqa: E402
from efp_bench import batch, card, timed  # noqa: E402
from multimodal_particles_b200.observables import (EFP_COLUMNS, EFP_D4_COLUMNS, energy_flow_polynomials,  # noqa: E402
                                                   energy_flow_polynomials_d4, fpd, jetnet_fpd_features, kpd)
from multimodal_particles_b200.pipeline import reference_fpd_features, sharded_generation_run  # noqa: E402


def kernel_ms(fn, xd, md, iters):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        fn(xd, md)
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / iters


def max_rel(got, want):
    return float(np.nanmax(np.abs(got.astype(np.float64) - want) / np.maximum(np.abs(want), 1e-300)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--cpu-jets", type=int, default=1024)
    ap.add_argument("--jets", type=int, default=1 << 20)
    ap.add_argument("--reference-jets", type=int, default=131072)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("efp_d4_bench measures on a CUDA device; none is visible")
    name, power = card()
    lines = []

    def emit(rec):
        rec.update(card=name, power_limit_and_max_sm_clock=power)
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)

    summary = {}
    shared = [EFP_D4_COLUMNS.index(c) for c in EFP_COLUMNS]
    for full in (False, True):
        x, mask, mult = batch(16384, 128, full, 16384 + full)
        xd, md = torch.from_numpy(x).cuda(), torch.from_numpy(mask).cuda()
        old, new = energy_flow_polynomials(xd, md), energy_flow_polynomials_d4(xd, md)
        torch.cuda.synchronize()
        times = {"jetnet_set": [], "d4": []}
        for _ in range(args.rounds):
            times["jetnet_set"].append(kernel_ms(energy_flow_polynomials, xd, md, args.iters))
            times["d4"].append(kernel_ms(energy_flow_polynomials_d4, xd, md, args.iters))
        nc = args.cpu_jets
        got_old, got_new = old[:nc].cpu().numpy(), new[:nc].cpu().numpy()
        best = {k: min(v) for k, v in times.items()}
        key = "all_128" if full else "jetclass_like"
        summary[f"d4_over_jetnet_set_{key}"] = best["d4"] / best["jetnet_set"]
        summary[f"d4_jets_per_s_{key}"] = 16384 / (best["d4"] * 1e-3)
        emit({"measure": "efp_kernels", "jets": 16384, "multiplicity": "all 128" if full else "normal(45, 18) clipped to [1, 128]",
              "mean_multiplicity": float(mult.mean()), "rounds": args.rounds, "iters_per_round": args.iters,
              "jetnet_set_ms_rounds": times["jetnet_set"], "d4_ms_rounds": times["d4"],
              "jetnet_set_ms_best": best["jetnet_set"], "d4_ms_best": best["d4"],
              "jetnet_set_ms_median": float(np.median(times["jetnet_set"])), "d4_ms_median": float(np.median(times["d4"])),
              "d4_over_jetnet_set_best": best["d4"] / best["jetnet_set"], "d4_jets_per_s": 16384 / (best["d4"] * 1e-3),
              "numpy_jets": nc,
              "max_rel_dev_vs_numpy_fp64_d4": max_rel(got_new, do.numpy_batch(x[:nc], mask[:nc])),
              "max_rel_dev_vs_numpy_fp64_jetnet_set": max_rel(got_old, eo.numpy_batch(x[:nc], mask[:nc])),
              "shared_columns_bit_identical_all_jets": bool(torch.equal(new[:, shared].contiguous(), old))})

    feats = []
    for seed in (1, 2):
        x, mask, _ = batch(131072, 128, False, seed)
        feats.append(jetnet_fpd_features(torch.from_numpy(x).cuda(), torch.from_numpy(mask).cuda()))
    real, gen = feats
    pick = [EFP_D4_COLUMNS.index(c) for c in EFP_COLUMNS[1:]]
    real5, gen5 = real[:, pick].contiguous(), gen[:, pick].contiguous()
    fpd(real, gen)                                                  # warm-up: eigh / curve_fit / generator set-up
    fpd(real5, gen5)
    kpd(real, gen)
    res = {}
    for label, (r, g) in (("36", (real, gen)), ("5", (real5, gen5))):
        res[label] = (timed(lambda: fpd(r, g)), timed(lambda: kpd(r, g)))
    (f36, s_f36), (k36, s_k36) = res["36"]
    (f5, s_f5), (k5, s_k5) = res["5"]
    summary.update(fpd_seconds_36=s_f36, kpd_seconds_36=s_k36, fpd_seconds_5=s_f5, kpd_seconds_5=s_k5)
    emit({"measure": "fpd_kpd", "rows": [len(real), len(gen)], "features": "FPD_EFP_COLUMNS (36) and efp4_* (5) of two independent "
          "JetClass-like batches", "fpd_36": list(f36), "fpd_seconds_36": s_f36, "kpd_36": list(k36), "kpd_seconds_36": s_k36,
          "fpd_5": list(f5), "fpd_seconds_5": s_f5, "kpd_5": list(k5), "kpd_seconds_5": s_k5})

    dev = torch.device("cuda", 0)
    cfg, model = bench.build_model(dev)
    ref = reference_fpd_features(model, cfg, args.reference_jets, dev, n_particles=bench.N_PART)
    runs = {False: [], True: []}
    shas = set()
    for _ in range(args.repeats):
        for with_ref in (False, True):
            rec = sharded_generation_run(model, cfg, args.jets, 0, 1, dev, micro_batch=16384, n_particles=bench.N_PART,
                                         fpd_reference=ref if with_ref else None)
            runs[with_ref].append(rec["seconds"])
            shas.add(rec["histogram_sha1"])
            line = {"measure": "c5_1gpu", "jets": args.jets, "fpd_reference": with_ref, "seconds": rec["seconds"],
                    "jets_per_s": rec["value"], "histogram_sha1": rec["histogram_sha1"]}
            if with_ref:
                line.update({k: rec[k] for k in ("jetnet_fpd", "jetnet_kpd", "jetnet_fpd_reference_jets", "jetnet_fpd_seconds")})
            emit(line)
    base, with_ref = min(runs[False]), min(runs[True])
    summary.update(c5_seconds_without_fpd_reference=runs[False], c5_seconds_with_fpd_reference=runs[True],
                   c5_overhead_of_best=with_ref / base - 1.0, c5_same_histogram_sha1=len(shas) == 1)
    emit(dict(measure="summary", **summary))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
