"""Device time of JetNet's W1-P draws with mmb_wasserstein1d_drawn against the same values composed from existing pieces and
against JetNet's host procedure, the split of its device time by stage, and the 1 M-jet C5 run with and without
``particle_reference``, in one command.

    python tools/jetnet_w1_bench.py [--out profiles/jetnet_w1_bench.json] [--jets 1048576]

- W1-P at JetNet's defaults (5 draws of 50 000 jets from each sample, 3 features) on two independent 131 072-jet samples at
  N = 128, with JetClass-like multiplicities (normal(45, 18) clipped to [1, 128], as the C5 pipeline draws them) and with every
  slot used.  ``wasserstein1d_drawn``: CUDA events around ``--iters`` back-to-back calls after a warm-up call (device time),
  and the host clock around the same calls ending in a device synchronisation.  The composition (per draw: torch gather,
  boolean compaction, one ``wasserstein1d``) waits for the host at every compaction, so it is timed by the host clock only, as
  is JetNet's host procedure (numpy gather, then scipy per draw and feature, on ``--host-draws`` draws).  The composition must
  give the same bits.
- A torch.profiler pass over one ``wasserstein1d_drawn`` call splits its device time by stage.
- The one-GPU C5 run (``pipeline.sharded_generation_run``, 16 384-jet micro-batches) without and with ``particle_reference``
  (``--reference-jets`` reference jets), alternated ``--repeats`` times.
- ``tools/w1_bench.py`` (``mmb_wasserstein1d`` on whole samples, the baseline the drawn path builds on), in a subprocess of the
  same command; its line is passed through.
Prints one JSON line per measurement and one summary line, all with the card's name and power limit."""
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
from multimodal_particles_b200.observables import jetnet_draws, wasserstein1d, wasserstein1d_drawn  # noqa: E402
from multimodal_particles_b200.pipeline import reference_particles, sharded_generation_run  # noqa: E402

N = 128


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as exc:   # report, do not guess
        q = f"unavailable ({type(exc).__name__})"
    return name, q


def sample(n, full, seed, dev):
    g = np.random.default_rng(seed)
    mult = np.full(n, N) if full else np.clip(np.rint(g.normal(45, 18, n)), 1, N).astype(int)
    mask = (np.arange(N)[None] < mult[:, None]).astype(np.uint8)
    x = np.empty((n, N, 3), np.float32)
    x[..., 0] = g.exponential(1.0, (n, N)) * 20.0 / (1.0 + np.arange(N)[None] * 0.1) + 0.01
    x[..., 1] = g.normal(0.0, 0.3, (n, N))
    x[..., 2] = g.normal(0.0, 0.3, (n, N))
    return torch.from_numpy(x * mask[..., None]).to(dev), torch.from_numpy(mask).to(dev)


def composed(x, ix, y, iy, mx, my):
    out = []
    for t in range(ix.shape[0]):
        a = x[ix[t].long()][mx[ix[t].long()].bool()]
        b = y[iy[t].long()][my[iy[t].long()].bool()]
        out.append(wasserstein1d(a, b))
    return torch.stack(out)


def host_jetnet(x, ix, y, iy, mx, my, draws):
    out = []
    for t in range(draws):
        a, b = x[ix[t]][mx[ix[t]].astype(bool)], y[iy[t]][my[iy[t]].astype(bool)]
        out.append([scipy.stats.wasserstein_distance(a[:, c], b[:, c]) for c in range(3)])
    return np.array(out)


def stage_split(x, ix, y, iy, mx, my):
    from torch.profiler import ProfilerActivity, profile
    wasserstein1d_drawn(x, ix, y, iy, mx, my)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        wasserstein1d_drawn(x, ix, y, iy, mx, my)
        torch.cuda.synchronize()
    names = (("w1_drawn_count", "1 count"), ("DeviceScan", "1 scan"), ("w1_drawn_keys", "2 keys"), ("Radix", "3 sort"),
             ("w1_drawn_merge", "4 merge"), ("w1_drawn_final", "4 final"))
    split = {}
    for ev in prof.key_averages():
        if ev.device_type.name != "CUDA":
            continue
        key = next((v for k, v in names if k in ev.key), "memset and other")
        split[key] = split.get(key, 0.0) + ev.device_time_total * 1e-3   # us -> ms
    return {k: round(v, 4) for k, v in sorted(split.items())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--jets", type=int, default=1 << 20)
    ap.add_argument("--sample-jets", type=int, default=131072)
    ap.add_argument("--reference-jets", type=int, default=262144)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--host-draws", type=int, default=1)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("jetnet_w1_bench measures on a CUDA device; none is visible")
    name, power = card()
    dev = torch.device("cuda", 0)
    lines = []

    def emit(rec):
        rec.update(card=name, power_limit_and_max_sm_clock=power)
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)

    summary = {}
    for full in (False, True):
        label = "all 128" if full else "normal(45, 18) clipped to [1, 128]"
        x, mx = sample(args.sample_jets, full, 1, dev)
        y, my = sample(args.sample_jets, full, 2, dev)
        ix, iy = jetnet_draws(len(x), len(y), device=dev)
        out = wasserstein1d_drawn(x, ix, y, iy, mx, my)
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(args.iters):
            out = wasserstein1d_drawn(x, ix, y, iy, mx, my)
        e.record()
        torch.cuda.synchronize()
        drawn_s = s.elapsed_time(e) * 1e-3 / args.iters
        t0 = time.perf_counter()
        for _ in range(args.iters):
            out = wasserstein1d_drawn(x, ix, y, iy, mx, my)
        torch.cuda.synchronize()
        drawn_host_s = (time.perf_counter() - t0) / args.iters
        comp = composed(x, ix, y, iy, mx, my)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.iters):
            comp = composed(x, ix, y, iy, mx, my)
        torch.cuda.synchronize()
        comp_s = (time.perf_counter() - t0) / args.iters
        xh, yh, mxh, myh, ixh, iyh = (t.cpu().numpy() for t in (x, y, mx, my, ix, iy))
        t0 = time.perf_counter()
        host = host_jetnet(xh, ixh, yh, iyh, mxh, myh, args.host_draws)
        host_s = time.perf_counter() - t0
        got = out.cpu().numpy()
        used = int(mx[ix.long()].sum().item())
        emit({"measure": "w1p_draws", "multiplicity": label, "sample_jets": args.sample_jets, "draws": list(ix.shape), "features": 3,
              "used_particles_in_draws_of_one_sample": used, "drawn_device_s": drawn_s, "drawn_host_s": drawn_host_s,
              "composed_host_s": comp_s, "composed_host_over_drawn_host": comp_s / drawn_host_s, "composed_bit_identical": bool(torch.equal(comp.view(torch.int64), out.view(torch.int64))),
              "host_jetnet_draws": args.host_draws, "host_jetnet_s": host_s, "host_jetnet_s_per_draw": host_s / args.host_draws,
              "max_rel_diff_vs_scipy": float(np.max(np.abs(got[:args.host_draws] - host) / np.abs(host))),
              "device_ms_by_stage": stage_split(x, ix, y, iy, mx, my)})
        summary["full" if full else "jetclass"] = {"drawn_device_s": drawn_s, "drawn_host_s": drawn_host_s, "composed_host_s": comp_s, "host_jetnet_s_per_draw": host_s / args.host_draws}
        del x, y, mx, my

    cfg, model = bench.build_model(dev)
    ref = reference_particles(model, cfg, args.reference_jets, dev, n_particles=N)
    base, withp = [], []
    for _ in range(args.repeats):
        for with_particles, acc in ((False, base), (True, withp)):
            rec = sharded_generation_run(model, cfg, args.jets, 0, 1, dev, micro_batch=16384, n_particles=N,
                                         particle_reference=ref if with_particles else None)
            acc.append(rec["seconds"])
            emit({"measure": "c5_1gpu", "jets": args.jets, "particle_reference_jets": args.reference_jets if with_particles else 0,
                  "seconds": rec["seconds"], "jets_per_s": rec["value"], "histogram_sha1": rec["histogram_sha1"],
                  **({k: rec[k] for k in ("w1p", "w1p_features", "jetnet_w1_seconds")} if with_particles else {})})
    w1 = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "w1_bench.py")], capture_output=True, text=True)
    if w1.returncode != 0:
        raise SystemExit(f"tools/w1_bench.py failed:\n{w1.stderr[-3000:]}")
    lines.append(w1.stdout.strip().splitlines()[-1])   # carries the card and power limit itself
    print(lines[-1], flush=True)
    emit({"measure": "summary", **summary, "c5_seconds_without_particle_reference": base, "c5_seconds_with_particle_reference": withp,
          "c5_overhead_of_best": min(withp) / min(base) - 1})
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
