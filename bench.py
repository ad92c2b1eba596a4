#!/usr/bin/env python
"""bench.py — generated jets/sec of the multimodal bridge generation loop (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--precision auto|f16|bf16|fp32] [--workload c2|c3|c4|c5|wide]

A "step" = one full generation (all 99 solver steps) of one batch of synthetic jets per GPU.
Workload (config.workload) = BASELINE.json configs[1]: EPiC multimodal bridge, JetClass-shaped
synthetic jets (128 particles, 3 continuous + 8 tokens), batch 4096 per GPU, 100 time points.

  value          whole-job jets/s with the source state already resident in HBM (CUDA events on the
                 launch stream, one event pair around the K steps, max over ranks); N>1 includes the
                 exchange of the generated jets and of the validation histograms (copy-engine pushes over NVLink peer
                 memory, or NCCL all-gather + all-reduce: --gather), issued on a
                 side stream under the next step's generation and joined before the end event (SURVEY.md §8e)
  e2e            same metric through the public API MultiModalBridgeMatching.simulate_dynamics with
                 PINNED HOST tensors in and host tensors out (H2D + D2H inside the timed region)
  roofline       dominant kernel of the step (the fused generation kernel): algorithmic FLOPs of the
                 EPiC network (0.819 MFLOP / jet-step, SURVEY.md §8d) / CUDA-event time, against the
                 measured bf16 tensor peak; roofline_update = the standalone fused update kernel
                 (75 B / particle-step) against the measured HBM copy bandwidth
  cpu_baseline   the CPU oracle (C port of the reference algorithm, OpenMP over jets) on a bounded
                 sample of the same workload, rank 0, N=1 only
  roofline_dense the same kernel on a batch whose jets all have 128 live particles (the C2 multiplicities skip dead rows)
  --impl reference   times that CPU port alone (the reference is pure Python and does not travel)
  --dump-outputs DIR c2: after the timed steps, the jets the last timed step generated (all ranks' jets when N > 1) as float32
                 DIR/{continuous,discrete,mask,jet_index}.npy; the inputs depend on the arguments alone, so two builds can be
                 compared output for output
  --workload     c2 (default, the headline) | c3 (one transepic evaluation, B=8192) | c4 (absorbing-flow generation, B=4096) |
                 c5 (1 M jets sharded over the GPUs: source + generation + observables + histograms + gather); with N > 1 the
                 c2 line carries a bounded c5 leg as well (`c5_million_jets`); wide = the C2 loop on an EPiC of the reference's
                 class-default widths (128 hidden units, 6 blocks) on the tcgen05 trunk
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True   # the tree may be read-only: nothing is cached in it
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "generated jets/sec (128 particles, 100 steps)"
WORKLOAD = "C2: EPiC multimodal bridge, JetClass-shape synthetic jets, N=128, Dc=3, S=8, B=4096/GPU, 99 solver steps"
B_PER_GPU, N_PART, N_TIMESTEPS = 4096, 128, 100
# micro-batch of the 1 M-jet run (BASELINE config 5 fixes the total, not the slice): a warp gets about two jets out of a 4096-jet
# call and the kernel ends in a ragged tail (profiles/r02_mma_timeline.md); 16384 jets per call run at 4.45 M jets/s instead of 4.0 M
C5_MICRO_BATCH = 16384
FLOP_PER_JET_STEP = 0.819e6          # SURVEY.md §8d (2*MAC, default widths)
UPDATE_BYTES_PER_PARTICLE = 75       # SURVEY.md §8d / BASELINE.md §4
CPU_SAMPLE_JETS = 16384              # bounded CPU sample: ~15 s on 16 host threads at ~1.1 K jets/s
DUMP_MAX_JETS = 16384                # --dump-outputs: 16384 jets x 128 particles x 5 float32 values = 42 MB (bound: 64 MB)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], bf16=p["bf16_tflops"], bf16_sustained=p.get("bf16_tflops_sustained"), src="measured")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, src="fallback")


class ClockSampler:
    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self._stop = index, [], threading.Event()
        self._thread = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.QUERY}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 6:
                    self.rows.append(parts)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._thread.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


def build_model(device):
    import torch
    from multimodal_particles_b200 import MultiModalBridgeMatching
    from multimodal_particles_b200.config_classes.multimodal_bridge_matching_config import MultimodalBridgeMatchingConfig
    cfg = MultimodalBridgeMatchingConfig()
    cfg.bridge.num_timesteps = N_TIMESTEPS
    cfg.data.max_num_particles = N_PART
    torch.manual_seed(0)
    model = MultiModalBridgeMatching(cfg)
    return cfg, (model.to(device) if device is not None else model)


def source_batch(n_jets, seed):
    import torch
    from multimodal_particles_b200.databatch import jetclass_like_databatch
    return jetclass_like_databatch(n_jets, N_PART, generator=torch.Generator().manual_seed(seed))


def dump_outputs(directory, **arrays):
    """--dump-outputs: one float32 DIR/<name>.npy per array (jet-major), and the jets' indices in jet_index.npy.  Beyond
    DUMP_MAX_JETS jets a fixed, seeded sample of the jets is written."""
    import numpy as np
    import torch
    n = next(iter(arrays.values())).shape[0]
    idx = torch.arange(n)
    if n > DUMP_MAX_JETS:
        idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_MAX_JETS].sort().values
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "jet_index.npy"), idx.numpy().astype(np.float32))
    for name, t in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), t.cpu()[idx].float().numpy())


def host_threads():
    """Threads the CPU arm uses: every core this process may run on.  Set explicitly — torchrun exports OMP_NUM_THREADS=1,
    which would otherwise serialise the OpenMP port (round 1: the reference arm timed out at N = 2, 4, 8)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_port_jets_per_s(n_jets, repeats=1, seed=1234):
    """The oracle port on the host cores, all host threads (OpenMP over jets), same workload distribution."""
    import oracle_lib as ol
    _, model = build_model(None)
    dims, packed = ol.packed_model(model)
    b = source_batch(n_jets, seed)
    tab = model.step_table()
    x, k, m = b.source_continuous.numpy(), b.source_discrete[..., 0].numpy(), b.source_mask[..., 0].numpy()
    best = float("inf")
    for _ in range(repeats):
        t0 = time.perf_counter()
        ol.generate(dims, packed, x, k, m, tab, seed=7, jet_offset=0, nthreads=host_threads())
        best = min(best, time.perf_counter() - t0)
    return n_jets / best, best, host_threads()


def run_reference(args, rank):
    """--impl reference: the CPU implementation of the path (oracle port), rank 0 only."""
    if rank != 0:
        return
    # bounded sample: size each step so that warm-up + K steps stay under ~100 s of CPU work whatever the host is
    rate, _, _ = cpu_port_jets_per_s(256)
    budget_s = 100.0
    sample = int(min(4096, max(64, rate * budget_s / (args.steps + 1))))
    sample -= sample % 64
    for _ in range(max(min(args.warmup, 1), 1)):
        cpu_port_jets_per_s(sample)
    times = []
    for _ in range(args.steps):
        _, dt, cores = cpu_port_jets_per_s(sample)
        times.append(dt)
    total = sum(times)
    value = sample * args.steps / total
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "jets/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample": f"{sample} jets x 99 solver steps per step"},
            "cpu_baseline": {"value": value, "unit": "jets/s", "cores": cores, "kind": "port",
                             "sample": f"{sample} jets x 99 solver steps, OpenMP over jets"},
            "e2e": {"value": value, "unit": "jets/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--precision", default="auto", choices=["auto", "f16", "bf16", "fp32"])
    ap.add_argument("--workload", default="c2", choices=["c2", "c3", "c4", "c5", "wide"])
    ap.add_argument("--gather", default="auto", choices=["auto", "peer", "nccl"],
                    help="N > 1: per-batch exchange of the generated jets (auto: copy-engine push over NVLink peer memory, else NCCL)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the C3 / C4 / C5 side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="c2: write the jets generated by the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl, args.workload) != ("native", "c2"):
        ap.error("--dump-outputs writes the jets of the c2 generation (--impl native --workload c2)")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    from multimodal_particles_b200 import HybridState, _native
    from multimodal_particles_b200.epic import as_u8
    from multimodal_particles_b200 import sharding

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the generation path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    W = max(args.warmup, 3)
    K = args.steps
    B = B_PER_GPU
    pk = peaks()

    if args.workload != "c2":
        line = side_workload_line(args, torch, dist, _native, device, pk, rank, world, W, K)
        if rank == 0:
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    cfg, model = build_model(device)
    native = model.encoder.native_model(device)
    precision = native.generate_precision(N_PART, args.precision)
    table = model.step_table()
    n_steps = table.n_steps
    batch = source_batch(B, 1234 + rank)
    jet_offset = rank * B

    # ---- device-resident arm: fresh source state per iteration (inputs in HBM before timing)
    n_bufs = W + K
    mask = as_u8(batch.source_mask.to(device))
    # the state of every step lives in one packed allocation [x | tokens | mask], so the multi-GPU exchange is one all-gather
    hist = sharding.ValidationHistograms(device, vocab_size=cfg.data.vocab_size_features)
    n_counts = hist.size if world > 1 else 0      # N > 1: the histogram counts of a step ride in the packed allocation
    packs = [sharding.PackedJets(B, N_PART, 3, device, extra_int64=n_counts).load(batch.source_continuous.to(device), as_u8(batch.source_discrete.to(device)), mask)
             for _ in range(n_bufs)]
    xs, ks = [p.x for p in packs], [p.k for p in packs]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)   # > 126 MB L2
    # receive side of the per-batch exchange, two buffers in turn (sharding.PeerGather: copy-engine push over peer memory;
    # --gather nccl: one NCCL all-gather + all-reduce)
    gather_bufs = [sharding.make_gather(B, N_PART, 3, world, device, mode=args.gather, extra_int64=n_counts) for _ in range(2)] if world > 1 else None
    stream = torch.cuda.current_stream()

    side = torch.cuda.Stream(device=device) if world > 1 else None

    def one_step(i):
        """One generation on the launch stream; for N > 1 the histogram kernel, the all-gather of the generated jets and the
        all-reduce of the histograms follow on a side stream, under the next step's generation (SURVEY.md §8e)."""
        native.generate(xs[i], ks[i], mask, table, seed=1, jet_offset=jet_offset + 0, precision=precision)
        if world > 1:
            done = torch.cuda.Event()
            done.record(stream)
            with torch.cuda.stream(side):
                side.wait_event(done)
                counts = hist.accumulate(xs[i], ks[i], mask, out=packs[i].counts)
                gather_bufs[i & 1].gather(packs[i], counts)

    def join():
        if world > 1:
            stream.wait_stream(side)

    t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:   # sampled across warm-up + timed region (the timed region alone is ~10-50 ms)
        for i in range(W):
            one_step(i)
        join()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t_hold = time.perf_counter()
        while len(clocks.rows) < 2 and time.perf_counter() - t_hold < 2.0:   # keep the GPU busy until two samples exist
            native.generate(xs[0], ks[0], mask, table, seed=1, jet_offset=jet_offset, precision=precision)
            torch.cuda.synchronize()
        # L2: one flush before the timed region; every timed step then reads a source state that nothing has touched since
        # (a different buffer per step), so no step finds its inputs in L2 and no flush sits inside the region
        flush.zero_()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t_wall0 = time.perf_counter()
        t_begin.record(stream)
        for i in range(K):
            one_step(W + i)
        join()
        t_end.record(stream)
        torch.cuda.synchronize()
        t_wall = time.perf_counter() - t_wall0
    if args.dump_outputs:
        last = W + K - 1
        if world > 1:   # what a rank holds after a step: the generated jets of every rank, from the exchange
            g = gather_bufs[last & 1]
            x_out, k_out, m_out = (torch.cat([view(r) for r in range(world)]) for view in (g.x, g.k, g.mask))
        else:
            x_out, k_out, m_out = xs[last], ks[last], mask
        if rank == 0:
            dump_outputs(args.dump_outputs, continuous=x_out, discrete=k_out, mask=m_out)
    if world > 1:
        dist.barrier()
    ms = t_begin.elapsed_time(t_end)
    t = torch.tensor([ms], device=device, dtype=torch.float64)
    ms_per_rank = [round(ms, 3)]
    if world > 1:
        every = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(every, t)
        ms_per_rank = [round(float(e.item()), 3) for e in every]   # reported beside the maximum the value is computed from
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = world * B * K / (ms_total * 1e-3)

    # ---- kernel-only timing of the dominant kernel (one mmb_generate call = prologue + generation kernel, same stream)
    def kernel_ms(x_src, k_src, m_dev, reps):
        out = []
        for i in range(reps):
            xs[i].copy_(x_src)
            ks[i].copy_(k_src)
            flush.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(stream)
            native.generate(xs[i], ks[i], m_dev, table, seed=1, jet_offset=jet_offset, precision=precision)
            e.record(stream)
            torch.cuda.synchronize()
            out.append(s.elapsed_time(e))
        return sum(out) / len(out)

    kern = kernel_ms(batch.source_continuous.to(device), as_u8(batch.source_discrete.to(device)), mask, min(K, 5))
    flops = FLOP_PER_JET_STEP * B * n_steps
    achieved_tf = flops / (kern * 1e-3) / 1e12
    kernel_name = {"f16": "mmb::epic_mma_generate_kernel<3,8,8,1> (warp-level mma.sync m16n8k16, fp16 operands, fp32 accumulate)",
                   "bf16": "mmb::epic_tc_kernel<3,8,8,GENERATE> (tcgen05, bf16 operands, fp32 accumulate)",
                   "fp32": "mmb::generate_fp32_kernel (CUDA cores)"}[precision]
    # traffic: dram__bytes_read.sum + dram__bytes_write.sum of one launch from `ncu --set full` (not measurable inside this run):
    # the state lives in registers for all 99 steps, HBM only sees the source state (the result stays in L2 until evicted)
    traffic = {"f16": 3.72e6, "bf16": 3.8e6}.get(precision) if B == 4096 else None
    roofline = {"kernel": kernel_name, "bound": "tensor", "achieved": achieved_tf, "peak": pk["bf16"],
                "unit": "TFLOP/s", "frac": achieved_tf / pk["bf16"], "traffic": traffic,
                "traffic_source": "ncu --set full capture of this kernel at B=4096: profiles/r02_mma_ncu_summary.md" if traffic else None,
                "peak_source": pk["src"], "algorithmic_flops_per_launch": flops, "ms_per_launch": kern,
                "note": "0.819 MFLOP per jet-step counts all 128 slots of every jet; the kernel is bound by issue slots "
                        "(ncu: 58 % issue-active, HMMA pipe 24 %), not by the tensor pipe: K = N = 16 GEMM chains"}
    roofline_dense = None
    if rank == 0:   # worst case for the same kernel: every jet with 128 live particles (no dead rows to skip)
        g = torch.Generator().manual_seed(99)
        xd = torch.randn(B, N_PART, 3, generator=g).to(device)
        kd = torch.randint(0, 8, (B, N_PART), generator=g, dtype=torch.uint8).to(device)
        dense_ms = kernel_ms(xd, kd, torch.ones_like(mask), 3)
        tf = flops / (dense_ms * 1e-3) / 1e12
        roofline_dense = {"workload": "as C2 but all 128 particles of every jet live", "jets_per_s": B / (dense_ms * 1e-3), "ms_per_launch": dense_ms,
                          "bound": "tensor", "achieved": tf, "peak": pk["bf16"], "unit": "TFLOP/s", "frac": tf / pk["bf16"]}

    # ---- standalone fused update kernel at an HBM-scale batch (32768 jets), 75 B / particle
    roofline_update = None
    if rank == 0:
        roofline_update = time_update_kernel(torch, _native, device, pk, flush)

    # ---- end-to-end arm: pinned host tensors -> simulate_dynamics -> host tensors (one mmb_generate_host call per iteration)
    pin = lambda t: t.clone().pin_memory()
    host_states = [HybridState(None, pin(batch.source_continuous), pin(batch.source_discrete), pin(batch.source_mask))
                   for _ in range(3 + K)]
    model.precision = precision
    out = None
    for i in range(3):   # results are held exactly as in the timed loop, so the pinned result buffers reach their steady-state pool
        out = model.simulate_dynamics(host_states[i], batch, jet_offset=jet_offset)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    import gc
    gc.collect()
    gc.disable()          # an iteration is ~1.3 ms: a generation-2 collection inside the loop would show up as an outlier
    t0 = time.perf_counter()
    e2e_iter_ms, t_prev = [], t0
    for i in range(K):
        out = model.simulate_dynamics(host_states[3 + i], batch, jet_offset=jet_offset)
        t_now = time.perf_counter()
        e2e_iter_ms.append(round((t_now - t_prev) * 1e3, 3))
        t_prev = t_now
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    gc.enable()
    te = torch.tensor([e2e_s], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * B * K / float(te.item())
    h2d = B * N_PART * (3 * 4 + 8 + 8)     # fp32 x, int64 tokens, int64 mask (reference layout), from pinned memory
    d2h = B * N_PART * (3 * 4 + 8)         # fp32 x + int64 tokens (widened on the device; the mask is unchanged and stays put)
    assert out.continuous.device.type == "cpu" and out.discrete.dtype == torch.int64

    c5 = None
    if world > 1 and not args.no_secondary:   # BASELINE configs[4] with the same model: 1 M jets over the GPUs of the box
        from multimodal_particles_b200.pipeline import sharded_generation_run
        try:
            c5 = sharded_generation_run(model, cfg, 1 << 20, rank, world, device, micro_batch=C5_MICRO_BATCH, n_particles=N_PART, precision=precision,
                                        gather=args.gather)
        except Exception as exc:
            c5 = {"error": f"{type(exc).__name__}: {exc}"}

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu_port_jets_per_s(256)                                  # warm-up (thread pool, page faults)
            v, dt_cpu, cores = cpu_port_jets_per_s(CPU_SAMPLE_JETS)   # ~10-20 s of CPU work
            cpu = {"value": v, "unit": "jets/s", "cores": cores, "kind": "port",
                   "sample": f"{CPU_SAMPLE_JETS} jets x 99 solver steps of the same workload ({dt_cpu:.1f} s), OpenMP over jets"}
        other = None
        if world == 1 and not args.no_secondary:
            try:
                other = secondary_configs(torch, _native, device, pk)
            except Exception as exc:  # the headline line must not depend on the side measurements
                other = {"error": f"{type(exc).__name__}: {exc}"}
        # kernels of this repo per timed step: bf16 = time-vector prologue + 3 jet-binning kernels + generation kernel;
        # f16 = prologue (time vectors + binning) + generation kernel; (+ histogram kernel for N > 1); NCCL's own kernels not counted
        launches = K * ({"f16": 2, "bf16": 5, "fp32": 1}[precision] + (1 if world > 1 else 0))
        line = {"metric": METRIC, "value": value, "unit": "jets/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": {"f16": "f16", "bf16": "bf16", "fp32": "f32"}[precision], "data": "synthetic",
                "config": {"workload": WORKLOAD, "global_batch": world * B, "precision": precision,
                           "engine": kernel_name,
                           "l2": "256 MiB flush before the timed region; each timed step reads a fresh, never-cached source buffer",
                           "rng": "in-kernel Philox4x32-10", "parallelism": f"jets sharded over {world} GPU(s)",
                           **({"exchange": "per step, on a side stream under the next generation: " + gather_bufs[0].kind
                                           + "; histogram counts travel with the jets (NCCL all-reduce in the all-gather mode)"} if world > 1 else {})},
                "e2e": {"value": e2e_value, "unit": "jets/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "api": "MultiModalBridgeMatching.simulate_dynamics -> mmb_generate_host, direct mode (the kernel reads and writes the pinned host buffers itself)",
                        "ms_per_iteration": e2e_iter_ms},
                "gpu_launches": launches, "roofline": roofline, "roofline_dense": roofline_dense, "roofline_update": roofline_update,
                "cpu_baseline": cpu, "clocks": clocks.summary(), "ms_timed_region_per_rank": ms_per_rank, "wall_s_timed_region": t_wall, "other_configs": other,
                "c5_million_jets": c5}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def side_workload_line(args, torch, dist, _native, device, pk, rank, world, W, K):
    """--workload c3 | c4 | c5: the other BASELINE configs as primary lines (same JSON contract; value = whole-job rate).
    c3 / c4 run one independent batch per rank (jets shard, no collective); c5 is the sharded 1 M-jet run."""
    if args.workload == "c5":
        from multimodal_particles_b200.pipeline import sharded_generation_run
        cfg, model = build_model(device)
        with ClockSampler(device.index or 0) as clocks:   # a step: one timed 1 M-jet run (each after its own 2 warm-up micro-batches)
            recs = [sharded_generation_run(model, cfg, 1 << 20, rank, world, device, micro_batch=C5_MICRO_BATCH, n_particles=N_PART,
                                           precision=args.precision, gather=args.gather) for _ in range(K)]
        if rank != 0:
            return None
        rec, seconds = recs[-1], sum(r["seconds"] for r in recs)
        return {"metric": METRIC, "value": K * (1 << 20) / seconds, "unit": "jets/s", "n_gpus": world, "steps": K, "warmup": 2,
                "ms_per_step": seconds * 1e3 / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": {"f16": "f16", "bf16": "bf16", "fp32": "f32"}[rec["precision"]], "data": "synthetic",
                "config": {"workload": rec["workload"], "global_batch": 1 << 20}, "c5_million_jets": rec, "clocks": clocks.summary(),
                "gpu_launches": K * 5 * ((1 << 20) // B_PER_GPU // world)}
    with ClockSampler(device.index or 0) as clocks:
        rec = secondary_configs(torch, _native, device, pk, only=args.workload, reps=K, warm=max(W, 2))
    key = {"c3": "C3_transepic_evaluation", "c4": "C4_absorbing_generation", "wide": "wide_epic"}[args.workload]
    r = rec[key]
    rate = r["jet_evals_per_s"] if args.workload == "c3" else r["jets_per_s"]
    t = torch.tensor([r["ms"]], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        rate = world * (8192 if args.workload == "c3" else 4096) / (float(t.item()) * 1e-3)
    if rank != 0:
        return None
    metric = "TransdimensionalEPiC evaluations/sec (jets, 128 particles)" if args.workload == "c3" else METRIC
    return {"metric": metric, "value": rate, "unit": "jet-evaluations/s" if args.workload == "c3" else "jets/s", "n_gpus": world,
            "steps": K, "warmup": max(W, 2), "ms_per_step": float(t.item()), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": {"workload": r["workload"]},
            "roofline": r.get("roofline") or r.get("roofline_head"), "clocks": clocks.summary(), "detail": r}


def secondary_configs(torch, _native, device, pk, only=None, reps=None, warm=None):
    """BASELINE configs 3 and 4 on this GPU, reported next to the headline (rank 0, N=1): one C3 transepic evaluation
    (B=8192, N=128; 145.3 MFLOP per jet-evaluation, SURVEY.md §8d) and one C4 absorbing-flow generation (B=4096, 99 steps;
    72.0 MFLOP per jet-step in the rate head).  CUDA events on the launch stream, inputs resident."""

    def timed(fn, reps, warm):
        for _ in range(warm):
            fn()
        ms = []
        for _ in range(reps):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(); fn(); e.record(); torch.cuda.synchronize()
            ms.append(s.elapsed_time(e))
        return sum(ms) / len(ms)

    out = {}
    if only in (None, "c3"):
        out.update(_c3(torch, _native, device, pk, timed, reps or 3, warm or 2))
    if only in (None, "c4"):
        out.update(_c4(torch, _native, device, pk, timed, reps or 2, warm or 1))
    if only in (None, "wide"):
        out.update(_wide(torch, _native, device, pk, timed, reps or 3, warm or 2, gen_reps=reps or 1))
    return out


def _wide(torch, _native, device, pk, timed, reps, warm, gen_reps):
    """The C2 workload on an encoder of the reference's CLASS-DEFAULT widths (EPiCNetwork: num_blocks = 6, dim_hidden_local =
    128, dim_hidden_global = 10; architectures/epic.py:99-101) — the shape where the trunk is GEMM work: 0.415 MFLOP per
    particle and evaluation (12 x 2 x 128 x 128 + local_0 + output layer), all 128 slots of a jet in the reference."""
    from multimodal_particles_b200 import MultiModalBridgeMatching
    from multimodal_particles_b200.config_classes.multimodal_bridge_matching_config import MultimodalBridgeMatchingConfig
    from multimodal_particles_b200.databatch import jetclass_like_databatch
    from multimodal_particles_b200.epic import as_u8
    B = 4096
    cfg = MultimodalBridgeMatchingConfig()
    e = cfg.encoder
    e.dim_hidden_local, e.num_blocks, e.dim_hidden_glob = 128, 6, 10
    cfg.data.max_num_particles, cfg.bridge.num_timesteps = N_PART, N_TIMESTEPS
    torch.manual_seed(0)
    model = MultiModalBridgeMatching(cfg).to(device)
    native = model.encoder.native_model(device)
    b = jetclass_like_databatch(B, N_PART, generator=torch.Generator().manual_seed(1234))
    x, k, m = b.source_continuous.to(device).contiguous(), as_u8(b.source_discrete.to(device)), as_u8(b.source_mask.to(device))
    ones = torch.ones_like(m)
    table = model.step_table()
    temb = table.temb[:1].to(device).contiguous()
    flop_particle = 2 * (12 * 128 * 128 + 16 * 128 + 128 * 11)
    flop_eval = flop_particle * B * N_PART     # the reference's count: every slot goes through the network

    def line(ms_, note):
        tf = flop_eval / (ms_ * 1e-3) / 1e12
        return {"bound": "tensor", "achieved": tf, "peak": pk["bf16"], "unit": "TFLOP/s", "frac": tf / pk["bf16"], "ms_per_launch": ms_, "rows": note}

    def five(mask_):   # five evaluations per event pair, as they follow each other inside a generation (launch gaps overlapped)
        for _ in range(5):
            native.forward(x, k, mask_, temb, precision="bf16")

    ev = timed(lambda: five(m), reps, warm) / 5
    ev_full = timed(lambda: five(ones), reps, warm) / 5
    ev_fp32 = timed(lambda: native.forward(x[:512], k[:512], m[:512], temb, precision="fp32"), 1, 1) * (B / 512)
    gen = timed(lambda: native.generate(x.clone(), k.clone(), m, table, seed=1, jet_offset=0, precision="bf16"), gen_reps, 1)
    live = float(m.float().mean().item())
    return {"wide_epic": {"workload": "EPiC at the class-default widths (H=128, L=6, G=10), B=4096, N=128: one evaluation and a 99-step generation",
                          "ms": gen, "jets_per_s": B / (gen * 1e-3), "evaluation_ms": ev, "jet_evals_per_s": B / (ev * 1e-3),
                          "evaluation_ms_fp32_cuda_cores": ev_fp32, "mean_live_fraction": live,
                          "roofline": line(ev, "JetClass-like mask (mean 45 live of 128), live particles only, one or two jets per 128-row tile"),
                          "roofline_dense": line(ev_full, "all 128 slots live"),
                          "executed_tflops": flop_eval * live / (ev * 1e-3) / 1e12}}


def _c3(torch, _native, device, pk, timed, reps, warm):
    from multimodal_particles_b200.config_classes.transdimensional_unconditional_config import TransdimensionalEpicConfig
    from multimodal_particles_b200.transdimensional import TransdimensionalJumpDiffusion
    out = {}
    B, N, S = 8192, N_PART, 8
    torch.manual_seed(0)
    model = TransdimensionalJumpDiffusion(TransdimensionalEpicConfig()).to(device)
    m = model.net.model
    trunk, heads = m.native_trunk(device), m.native_heads(device)
    fr = model.forward_rate.as_c()

    def evaluation_ms(dims, g):
        mask = (torch.arange(N)[None] < dims[:, None]).float().unsqueeze(-1)
        x = torch.randn(B, N, 3, generator=g) * mask
        x = x - (x.sum(1, keepdim=True) / dims.view(B, 1, 1)) * mask
        oh, ts = torch.randn(B, N, S, generator=g) * mask, torch.rand(B, generator=g) * 0.999 + 1e-3
        near = (torch.rand(B, generator=g) * dims).long()
        x, oh, d32, ts, near = x.to(device), oh.to(device), dims.to(device, torch.int32), ts.to(device), near.to(device, torch.int32)
        return timed(lambda: _native.trans_forward(trunk, heads, x, oh, d32, ts, near, None, fr, precision="bf16", want_auto=False), reps, warm)

    def line(ms, rows):
        tf = 145.33e6 * B / (ms * 1e-3) / 1e12     # the reference's flops: every slot of every jet
        return {"bound": "tensor", "achieved": tf, "peak": pk["bf16"], "unit": "TFLOP/s", "frac": tf / pk["bf16"], "ms_per_evaluation": ms,
                "rows": rows}

    g = torch.Generator().manual_seed(1234)
    ms = evaluation_ms(torch.randint(1, N + 1, (B,), generator=g), g)
    # the multiplicities of the other configs (C2 / C4 / C5): what the network meets when it generates JetClass-like jets
    ms_jc = evaluation_ms((torch.randn(B, generator=g) * 18.0 + 45.0).round().clamp(1, N).long(), g)
    out["C3_transepic_evaluation"] = {"workload": "TransdimensionalEPiC.forward, B=8192, N=128, bf16 stacks", "ms": ms,
                                      "jet_evals_per_s": B / (ms * 1e-3),
                                      "roofline": line(ms, "multiplicities uniform in 1..128 (mean 64.5); padded slots packed to one row per jet"),
                                      "roofline_jetclass_multiplicities": line(ms_jc, "multiplicities ~ N(45, 18) clipped to 1..128, as in C2 / C4 / C5")}
    return out


def _c4(torch, _native, device, pk, timed, reps, warm):
    from multimodal_particles_b200.absorbing_flows import AbsorbingFlow
    from multimodal_particles_b200.config_classes.absorbing_flows_config import AbsorbingConfig
    from multimodal_particles_b200.databatch import jetclass_like_databatch
    from multimodal_particles_b200.epic import as_u8
    out = {}
    B = 4096
    cfg = AbsorbingConfig()
    cfg.data.max_num_particles, cfg.bridge.num_timesteps = N_PART, N_TIMESTEPS
    torch.manual_seed(0)
    flow = AbsorbingFlow(cfg).to(device)
    gen = flow.generator
    b = jetclass_like_databatch(B, N_PART, generator=torch.Generator().manual_seed(1234))
    table = flow.step_table()
    tb = gen.time_bias(table.t)
    trunk, head = gen.native_trunk(device), gen.native_head(device)
    x0, k0, m0 = b.source_continuous.to(device).contiguous(), as_u8(b.source_discrete.to(device)), as_u8(b.source_mask.to(device))

    def run():
        _native.generate_absorbing(trunk, head, x0.clone(), k0.clone(), m0.clone(), table, tb, seed=1, jet_offset=0, precision="bf16")

    ms = timed(run, reps, warm)
    # the rate head alone, on what the trunk hands it: hidden rows of padded slots are zero (epic_tc.cu writes them so), the
    # mask is the source batch's (mean 45 live of 128) — and, beside it, the same head on an all-live batch
    tb1 = tb[:1].to(device)
    hid = torch.randn(B, N_PART, 16, device=device) * m0[..., None]
    ones = torch.ones_like(m0)
    hid_full = torch.randn(B, N_PART, 16, device=device)
    hms = timed(lambda: head.forward(hid, m0, tb1), 5, 3)
    hms_full = timed(lambda: head.forward(hid_full, ones, tb1), 5, 3)

    def line(ms_):
        tf = 72.0e6 * B / (ms_ * 1e-3) / 1e12   # the reference's flops: every one of the 128 slots of a jet goes through the stack
        return {"bound": "tensor", "achieved": tf, "peak": pk["bf16"], "unit": "TFLOP/s", "frac": tf / pk["bf16"], "ms_per_launch": ms_}

    out["C4_absorbing_generation"] = {"workload": "AbsorbingFlow generation, B=4096, N=128, 99 steps", "ms": ms, "jets_per_s": B / (ms * 1e-3),
                                      "roofline_head": dict(line(hms), rows="jetclass-like mask, padded slots packed to one row per jet"),
                                      "roofline_head_dense": dict(line(hms_full), rows="all 128 slots live")}
    return out


def time_update_kernel(torch, _native, device, pk, flush, jets=32768, reps=20):
    B, N, S = jets, N_PART, 8
    g = torch.Generator(device=device).manual_seed(3)
    x = torch.randn(B, N, 3, device=device, generator=g)
    v = torch.randn(B, N, 3, device=device, generator=g)
    lg = torch.randn(B, N, S, device=device, generator=g)
    u = torch.rand(B, N, device=device, generator=g)
    k = torch.randint(0, S, (B, N), device=device, generator=g, dtype=torch.uint8)
    m = torch.ones(B, N, device=device, dtype=torch.uint8)
    stream = torch.cuda.current_stream()
    for _ in range(3):
        _native.bridge_update(x, k, m, v, lg, u, 0.0101, 5.0, 0.4)
    # the working set (315 MB) is larger than L2 (126 MB), so back-to-back launches all stream from HBM; ten launches per
    # event pair keep the host-side launch gap between the two events out of the kernel time
    inner, times = 10, []
    for _ in range(max(reps // inner, 3)):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(stream)
        for _ in range(inner):
            _native.bridge_update(x, k, m, v, lg, u, 0.0101, 5.0, 0.4)
        e.record(stream)
        torch.cuda.synchronize()
        times.append(s.elapsed_time(e) / inner)
    ms = sum(times) / len(times)
    nbytes = UPDATE_BYTES_PER_PARTICLE * B * N
    gbs = nbytes / (ms * 1e-3) / 1e9
    return {"kernel": "mmb::bridge_update_vec_kernel<8,2,5>", "bound": "hbm", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s",
            "frac": gbs / pk["hbm"], "traffic": 269.8e6 if jets == 32768 else None,   # ncu --set full: 260.1 MB read + 9.8 MB written (writes still in L2)
            "traffic_source": "ncu --set full capture at 32768 jets: profiles/r01_update_variants.md" if jets == 32768 else None,
            "peak_source": pk["src"], "jets": jets,
            "l2": "working set 315 MB > 126 MB L2; 10 launches per event pair",
            "algorithmic_bytes_per_launch": nbytes, "ms_per_launch": ms}


if __name__ == "__main__":
    main()
