"""BASELINE config 5: a 1 M-jet generation run sharded over the GPUs of one box (multimodal_particles_b200/pipeline.py).

    python tools/million_jets.py [--jets 1048576] [--substructure]                           # one GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 tools/million_jets.py

Prints one JSON line on rank 0 (device time by CUDA events, max over ranks; `histogram_sha1` is the same for every GPU count)."""
import argparse
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench  # noqa: E402
from multimodal_particles_b200.pipeline import sharded_generation_run  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--jets", type=int, default=1 << 20)
    ap.add_argument("--micro-batch", type=int, default=16384)
    ap.add_argument("--precision", default="auto")
    ap.add_argument("--substructure", action="store_true", help="also histogram tau21, tau32 and D2 of every jet on the device")
    args = ap.parse_args()
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg, model = bench.build_model(dev)
    rec = sharded_generation_run(model, cfg, args.jets, rank, world, dev, micro_batch=args.micro_batch, n_particles=bench.N_PART,
                                 precision=args.precision, substructure=args.substructure)
    if rank == 0:
        print(json.dumps(rec))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
