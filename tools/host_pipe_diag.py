"""Where the end-to-end time of mmb_generate_host goes: wall clock of the bare C call + synchronise (buffers preallocated),
device time between the caller-stream events around it, and the same through simulate_dynamics."""
import os, ctypes, sys, time, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench
from multimodal_particles_b200 import HybridState, _native
from multimodal_particles_b200.steptable import CStepTable
dev = torch.device("cuda:0")
cfg, model = bench.build_model(dev)
B = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
N = 128
batch = bench.source_batch(B, 1234)
native = model.encoder.native_model(dev)
table = model.step_table()
lib = _native.load()
pin = lambda t: t.clone().pin_memory()
x_in, k_in, m_in = pin(batch.source_continuous), pin(batch.source_discrete), pin(batch.source_mask)
x_out = torch.empty((B, N, 3), dtype=torch.float32, pin_memory=True)
k_out = torch.empty((B, N, 1), dtype=torch.int64, pin_memory=True)
flag = torch.empty(1, dtype=torch.int32, pin_memory=True)
ctable = CStepTable.from_table(table)
stream = torch.cuda.current_stream()
for chunks in (0, 2, 4):
    need = lib.mmb_generate_host_workspace_bytes(native._handle, B, N, table.n_steps, chunks, 2)
    ws = torch.empty(need, device=dev, dtype=torch.uint8)
    wall, gpu = [], []
    for i in range(15):
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        s.record(stream)
        _native.check(lib.mmb_generate_host(native._handle, _native._ptr(x_in), _native._ptr(k_in), _native._ptr(m_in), ctypes.byref(ctable), 1, 0, B, N,
                                            _native._ptr(x_out), _native._ptr(k_out), _native._ptr(flag), _native._ptr(ws), ws.numel(), chunks, 2,
                                            _native._stream()))
        t1 = time.perf_counter()
        e.record(stream)
        stream.synchronize()
        t2 = time.perf_counter()
        wall.append(((t1 - t0) * 1e3, (t2 - t0) * 1e3)); gpu.append(s.elapsed_time(e))
    w = sorted(wall[5:], key=lambda p: p[1]); g = sorted(gpu[5:])
    print(f"chunks {chunks}: enqueue {w[len(w)//2][0]:.3f} ms, enqueue+sync {w[len(w)//2][1]:.3f} ms, device time {g[len(g)//2]:.3f} ms")
# device-resident kernel alone for reference
from multimodal_particles_b200.epic import as_u8
x, k, m = batch.source_continuous.to(dev), as_u8(batch.source_discrete.to(dev)), as_u8(batch.source_mask.to(dev))
ts = []
for i in range(10):
    xx, kk = x.clone(), k.clone()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record(); native.generate(xx, kk, m, table, seed=1, jet_offset=0, precision="f16"); e.record(); torch.cuda.synchronize()
    ts.append(s.elapsed_time(e))
print(f"device-resident mmb_generate: {sorted(ts)[len(ts)//2]:.3f} ms")
# PCIe copy rates
big = torch.empty(64 << 20, dtype=torch.uint8, pin_memory=True); dbig = torch.empty(64 << 20, dtype=torch.uint8, device=dev)
for name, fn in (("H2D", lambda: dbig.copy_(big, non_blocking=True)), ("D2H", lambda: big.copy_(dbig, non_blocking=True))):
    fn(); torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record(); fn(); e.record(); torch.cuda.synchronize()
    print(f"{name} 64 MiB pinned: {(64 << 20) / s.elapsed_time(e) / 1e6:.1f} GB/s")
