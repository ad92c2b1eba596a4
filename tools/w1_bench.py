"""Device time of mmb_wasserstein1d (exact 1-D W1 per column) against scipy.stats.wasserstein_distance on the same data.

    python tools/w1_bench.py [--jets 1048576] [--out profiles/w1_bench.json]

Samples come from the C5 generation path (pipeline.reference_observables: source state, solver, observables, substructure), as
two independent samples of --jets jets each (Philox jet offsets 0.. and 2^40..):
  - jet level: the 10 columns of pipeline.w1_columns(substructure=True), generated against reference;
  - particle level: (pt, eta, phi) of every live particle of the same jets (about 45 per jet), generated against reference.
Device time: CUDA events around --iters back-to-back calls after a warm-up call (inputs and workspace exceed the 126 MB L2 at
these sizes).  scipy runs on the same float32 values after the non-finite ones are dropped: all columns at jet level, the pt
column only at particle level.  A torch.profiler pass over one jet-level call splits the device time by kernel.  Prints one JSON
line with the card's name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import scipy.stats
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from multimodal_particles_b200.observables import wasserstein1d  # noqa: E402
from multimodal_particles_b200.pipeline import reference_observables, reference_particles, w1_columns  # noqa: E402

REF_OFFSET = 1 << 40


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as exc:   # report, do not guess
        q = f"unavailable ({type(exc).__name__})"
    return name, q


def particles(model, cfg, n_jets, dev, jet_offset):
    """[live particles, 3] f32 (pt, eta, phi in physical units) of the jets generated as reference_observables makes them."""
    x, m = reference_particles(model, cfg, n_jets, dev, n_particles=bench.N_PART, jet_offset=jet_offset)
    return x[m.bool()]


def device_time(x, y, iters):
    out = wasserstein1d(x, y)
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        out = wasserstein1d(x, y)
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) * 1e-3 / iters, out.cpu().numpy()


def scipy_time(x, y, cols):
    t0 = time.perf_counter()
    vals = []
    for c in cols:
        a, b = x[:, c], y[:, c]
        vals.append(scipy.stats.wasserstein_distance(a[np.isfinite(a)], b[np.isfinite(b)]))
    return time.perf_counter() - t0, np.array(vals)


def kernel_split(x, y):
    from torch.profiler import ProfilerActivity, profile
    wasserstein1d(x, y)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        wasserstein1d(x, y)
        torch.cuda.synchronize()
    split = {}
    for ev in prof.key_averages():
        if ev.device_type.name != "CUDA":
            continue
        key = next((k for k in ("w1_keys", "w1_merge", "w1_final") if k in ev.key), "cub radix sort" if "Radix" in ev.key else "other")
        split[key] = split.get(key, 0.0) + ev.device_time_total * 1e-3   # us -> ms
    return {k: round(v, 4) for k, v in sorted(split.items())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--jets", type=int, default=1 << 20)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("w1_bench measures the kernels on a CUDA device; none is visible")
    name, power = card()
    dev = torch.device("cuda", 0)
    cfg, model = bench.build_model(dev)
    cols = w1_columns(True)
    rows = []

    gen = reference_observables(model, cfg, args.jets, dev, n_particles=bench.N_PART, substructure=True, jet_offset=0)
    ref = reference_observables(model, cfg, args.jets, dev, n_particles=bench.N_PART, substructure=True, jet_offset=REF_OFFSET)
    dev_s, got = device_time(gen, ref, args.iters)
    try:
        split = kernel_split(gen, ref)
    except Exception as exc:   # report, do not guess
        split = f"unavailable ({type(exc).__name__}: {exc})"
    cpu_s, want = scipy_time(gen.cpu().numpy(), ref.cpu().numpy(), range(len(cols)))
    rows.append({"level": "jet", "columns": list(cols), "n": gen.shape[0], "m": ref.shape[0], "device_s": dev_s,
                 "scipy_s": cpu_s, "scipy_columns": len(cols), "scipy_over_device": cpu_s / dev_s,
                 "max_rel_diff_vs_scipy": float(np.max(np.abs(got - want) / np.abs(want))), "w1": dict(zip(cols, got.tolist())),
                 "device_ms_by_kernel": split})
    del gen, ref

    pg, pr = particles(model, cfg, args.jets, dev, 0), particles(model, cfg, args.jets, dev, REF_OFFSET)
    dev_s, got = device_time(pg, pr, args.iters)
    cpu_s, want = scipy_time(pg[:, :1].cpu().numpy(), pr[:, :1].cpu().numpy(), [0])
    rows.append({"level": "particle", "columns": ["pt", "eta", "phi"], "n": pg.shape[0], "m": pr.shape[0], "device_s": dev_s,
                 "scipy_s": cpu_s, "scipy_columns": 1, "scipy_one_column_over_device_three_columns": cpu_s / dev_s,
                 "rel_diff_pt_vs_scipy": float(abs(got[0] - want[0]) / abs(want[0])), "w1": dict(zip(("pt", "eta", "phi"), got.tolist()))})

    rec = {"workload": f"mmb_wasserstein1d: {args.jets} generated jets against {args.jets} independent reference jets (C5 path)",
           "gpu": name, "power_limit_and_max_sm_clock": power, "cpu_threads": os.cpu_count(), "iters": args.iters, "rows": rows}
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
