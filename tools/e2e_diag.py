"""End-to-end latency of simulate_dynamics (pinned host state in, host state out) for different numbers of pipeline slices."""
import os, sys, time, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench
from multimodal_particles_b200 import HybridState
dev = torch.device("cuda:0")
cfg, model = bench.build_model(dev)
B = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
batch = bench.source_batch(B, 1234)
pin = lambda t: t.clone().pin_memory()
model.precision = sys.argv[2] if len(sys.argv) > 2 else "auto"
ref = None
for chunks in (1, 2, 4, 0):
    model.pipeline_chunks, model.pipeline_min_jets = chunks, 1
    times, keep = [], []
    for i in range(12):
        st = HybridState(None, pin(batch.source_continuous), pin(batch.source_discrete), pin(batch.source_mask))
        torch.cuda.synchronize(); t0 = time.perf_counter()
        out = model.simulate_dynamics(st, batch, jet_offset=0)
        torch.cuda.synchronize(); times.append((time.perf_counter() - t0) * 1e3)
        keep.append(out)
        keep = keep[-2:]
    if ref is None:
        ref = out
    same = torch.equal(ref.continuous, out.continuous) and torch.equal(ref.discrete, out.discrete)
    t = sorted(times[4:])
    print(f"chunks {chunks}: median {t[len(t)//2]:.3f} ms  min {t[0]:.3f}  -> {B / t[len(t)//2] * 1e3:.0f} jets/s  identical to unsliced: {same}")
