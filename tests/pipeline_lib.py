"""Scaffolding of the tests of the sharded generation run (pipeline.sharded_generation_run): the one-GPU run and a two-rank run
over NCCL whose record the tests compare with it (test infrastructure only)."""
import json
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

DEV = "cuda:0"


def one_gpu_run(model, cfg, total, micro_batch, **kw):
    """The run of ``total`` jets on cuda:0 alone, one warm-up micro-batch."""
    import bench
    from multimodal_particles_b200.pipeline import sharded_generation_run
    return sharded_generation_run(model, cfg, total, 0, 1, torch.device(DEV), micro_batch=micro_batch, n_particles=bench.N_PART,
                                  warmup_batches=1, **kw)


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _two_gpu_worker(rank, world, port, out_path, total, make_kwargs, keys):
    import bench
    from multimodal_particles_b200.pipeline import sharded_generation_run
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        cfg, model = bench.build_model(dev)
        rec = sharded_generation_run(model, cfg, total, rank, world, dev, micro_batch=16384, n_particles=bench.N_PART,
                                     warmup_batches=1, **make_kwargs(model, cfg, dev))
        if rank == 0:
            with open(out_path, "w") as f:
                json.dump({k: rec[k] for k in keys}, f)
    finally:
        dist.destroy_process_group()


def two_gpu_run(tmp_path, total, make_kwargs, keys):
    """The record entries ``keys`` (through JSON) of a run of ``total`` jets on cuda:0 and cuda:1, micro-batch 16384.  Each rank
    passes ``make_kwargs(model, cfg, device)`` (references included) to the run; it must be a top-level function of the test
    module, so that the spawned ranks can unpickle it."""
    out = str(tmp_path / "two_gpu.json")
    mp.spawn(_two_gpu_worker, args=(2, free_port(), out, total, make_kwargs, keys), nprocs=2, join=True)
    with open(out) as f:
        return json.load(f)
