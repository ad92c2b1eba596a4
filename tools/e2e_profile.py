"""Where the host-side microseconds of one simulate_dynamics call (pinned host state in, host state out) go."""
import os, sys, time, gc, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench
from multimodal_particles_b200 import HybridState, _native
dev = torch.device("cuda:0")
cfg, model = bench.build_model(dev)
B = 4096
batch = bench.source_batch(B, 1234)
pin = lambda t: t.clone().pin_memory()
states = [HybridState(None, pin(batch.source_continuous), pin(batch.source_discrete), pin(batch.source_mask)) for _ in range(40)]
for st in states[:8]:
    model.simulate_dynamics(st, batch, jet_offset=0)
torch.cuda.synchronize()
gc.collect(); gc.disable()
tt = lambda: time.perf_counter()
# whole call
ts = []
for st in states[8:24]:
    t0 = tt(); model.simulate_dynamics(st, batch, jet_offset=0); ts.append((tt() - t0) * 1e6)
print("simulate_dynamics: median %.0f us  min %.0f" % (sorted(ts)[len(ts) // 2], min(ts)))
# pieces
nm = model.encoder.native_model(dev)
table = model.step_table()
def med(fn, n=200):
    v = []
    for _ in range(n):
        t0 = tt(); fn(); v.append((tt() - t0) * 1e6)
    return sorted(v)[n // 2]
print("native_model(): %.1f us" % med(lambda: model.encoder.native_model(dev)))
print("step_table(): %.1f us" % med(lambda: model.step_table()))
print("_compute_device: %.1f us" % med(lambda: model._compute_device(states[0])))
print("pinned block alloc: %.1f us" % med(lambda: torch.empty(B * 128 * 20 + 16, dtype=torch.uint8, pin_memory=True)))
print("embedding.context(None): %.1f us" % med(lambda: model.encoder.epic.embedding.context(None, None, "cpu")))
print("HybridState + torch.full: %.1f us" % med(lambda: HybridState(time=torch.full((B, 1), 0.5), continuous=None, discrete=None, absorbing=None)))
st = states[30]
def raw():
    out = nm.generate_host(st.continuous, st.discrete, st.absorbing, table, seed=0, jet_offset=0, chunks=0, precision="auto")
    torch.cuda.current_stream(dev).synchronize()
    return out
v = []
for _ in range(16):
    t0 = tt(); raw(); v.append((tt() - t0) * 1e6)
print("generate_host + sync: median %.0f us" % sorted(v)[8])
def launch_only():
    t0 = tt()
    out = nm.generate_host(st.continuous, st.discrete, st.absorbing, table, seed=0, jet_offset=0, chunks=0, precision="auto")
    t1 = tt()
    torch.cuda.current_stream(dev).synchronize()
    return (t1 - t0) * 1e6
v = [launch_only() for _ in range(16)]
print("generate_host enqueue only: median %.0f us" % sorted(v)[8])
