"""Time one training step's loss and gradient work of MultiModalBridgeMatching on the GPU: ``bridge_matching_losses`` plus
``backward()`` (native fp32 kernels, epic_grad.cu) beside torch eager autograd of the float32 restatement (tests/grad_lib.py) on
the same GPU and batches, with the largest gradient difference between the two.  CUDA-event times after warm-up, N = 128 and
JetClass-like masks (bench.source_batch's distribution).  Writes one JSON file (default profiles/epic_grad_bench.json)."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench  # noqa: E402
import grad_lib  # noqa: E402
from multimodal_particles_b200 import HybridState, MultiModalBridgeMatching, _native  # noqa: E402
from multimodal_particles_b200.config_classes.multimodal_bridge_matching_config import MultimodalBridgeMatchingConfig  # noqa: E402

CASES = [("c2", {}, 1024), ("c2", {}, 4096), ("class_default", dict(dim_hidden_local=128, num_blocks=6, dim_hidden_glob=10), 1024)]
N = 128


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def timed(fn, warmup, iters):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / iters


def run_case(name, tweak, B, warmup, iters, dev):
    cfg = MultimodalBridgeMatchingConfig()
    for key, val in tweak.items():
        setattr(cfg.encoder, key, val)
    torch.manual_seed(0)
    model = MultiModalBridgeMatching(cfg).to(dev)
    src = bench.source_batch(B, 1234)
    g = torch.Generator().manual_seed(5)
    mask = src.source_mask
    batch = type("Batch", (), {})()
    batch.source_continuous, batch.target_continuous = src.source_continuous, torch.randn(B, N, 3, generator=g) * mask
    batch.target_discrete = torch.randint(0, 8, (B, N, 1), generator=g) * mask
    state = HybridState(torch.rand(B, 1, 1, generator=g), (torch.randn(B, N, 3, generator=g) * mask).to(dev),
                        (torch.randint(0, 8, (B, N, 1), generator=g) * mask).to(dev), mask.to(dev))
    params = [p for n, p in model.named_parameters() if n.startswith("encoder.")]

    def native():
        model.zero_grad(set_to_none=True)
        l0, l1 = model.bridge_matching_losses(state, batch)
        (l0 + l1).backward()

    ref = grad_lib.Restatement(model, torch.float32, dev)
    ref_params = list(ref.encoder_parameters().values())

    def eager():
        for p in ref_params:
            p.grad = None
        r0, r1 = ref.bridge_matching_losses(state, batch)
        (r0 + r1).backward()

    ms_native = timed(native, warmup, iters)
    ms_eager = timed(eager, warmup, iters)
    native()
    eager()
    worst_abs = max(float((p.grad - q.grad).abs().max()) for p, q in zip(params, ref_params))
    worst_rel = max(float((p.grad - q.grad).abs().max()) / max(float(q.grad.abs().max()), 1e-30) for p, q in zip(params, ref_params))
    lib = _native.load()
    head = model.encoder.fc_layer
    dims = model.encoder.epic.epic_dims(head[0].out_features)
    blob_bytes = 4 * lib.mmb_epic_packed_floats(ctypes.byref(dims))
    ws_bytes = lib.mmb_epic_loss_grad_workspace_bytes(ctypes.byref(dims), B, N)
    return {"case": name, "B": B, "N": N, "live_particles": int(mask.sum()), "native_ms": ms_native, "torch_eager_fp32_autograd_ms": ms_eager,
            "max_abs_grad_difference": worst_abs, "max_grad_difference_over_max_eager_grad": worst_rel,
            "weight_blob_bytes": blob_bytes, "workspace_bytes": ws_bytes}


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "epic_grad_bench.json"))
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("epic_grad_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    rows = [run_case(name, tweak, B, args.warmup, args.iters, dev) for name, tweak, B in CASES]
    out = {"what": "bridge_matching_losses + backward(), CUDA events per call after warm-up", "card": card(), "cases": rows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
