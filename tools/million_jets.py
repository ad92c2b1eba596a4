"""BASELINE config 5: a 1 M-jet generation run sharded over the GPUs of one box (multimodal_particles_b200/pipeline.py).

    python tools/million_jets.py [--jets 1048576] [--substructure] [--efp] [--w1-reference-jets M | --w1-reference FILE.npz]
                                 [--w1p-reference-jets M] [--fpd-reference-jets M] [--out F]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 tools/million_jets.py

Prints one JSON line on rank 0 (device time by CUDA events, max over ranks; `histogram_sha1` is the same for every GPU count).
With a W1 reference — M jets built by `pipeline.reference_observables` from disjoint Philox streams, or one array per column
of `pipeline.w1_columns` in an .npz file — the record also holds the W1 of every column against it (`w1`, `w1_seconds`), and with
`--efp` also W1-EFP (the efp4_* entries of `w1`), `fpd` and `kpd` of the five d = 4 EFPs.  With `--w1p-reference-jets M` the
particles of M reference jets (`pipeline.reference_particles`) score JetNet's W1-P (`w1p`, `w1p_features`), and with a W1
reference also its W1-M (`w1m`) and, with `--efp`, W1-EFP (`w1efp`): mean and std over JetNet's draws.  With
`--fpd-reference-jets M` every EFP of degree <= 4 of M reference jets (`pipeline.reference_fpd_features`) scores FPD and KPD on
JetNet's feature set (`jetnet_fpd`, `jetnet_kpd`)."""
import argparse
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench  # noqa: E402
from multimodal_particles_b200.pipeline import (reference_fpd_features, reference_observables, reference_particles,  # noqa: E402
                                                sharded_generation_run, w1_columns)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--jets", type=int, default=1 << 20)
    ap.add_argument("--micro-batch", type=int, default=16384)
    ap.add_argument("--precision", default="auto")
    ap.add_argument("--substructure", action="store_true", help="also histogram tau21, tau32 and D2 of every jet on the device")
    ap.add_argument("--efp", action="store_true", help="also compute the energy flow polynomials of every jet (W1-EFP, FPD, KPD)")
    ap.add_argument("--w1-reference-jets", type=int, default=0, help="score W1 against an independent reference sample of this size")
    ap.add_argument("--w1-reference", default=None, help="score W1 against this .npz (one array per column name)")
    ap.add_argument("--w1p-reference-jets", type=int, default=0,
                    help="score JetNet's W1-P (and W1-M / W1-EFP with a W1 reference) against the particles of this many reference jets")
    ap.add_argument("--fpd-reference-jets", type=int, default=0,
                    help="score FPD and KPD on every EFP of degree <= 4 (JetNet's feature set) against this many reference jets")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg, model = bench.build_model(dev)
    reference = None
    if args.w1_reference:
        with np.load(args.w1_reference) as f:
            reference = torch.from_numpy(np.stack([f[c].astype(np.float32).reshape(-1) for c in w1_columns(args.substructure, args.efp)], 1)).to(dev)
    elif args.w1_reference_jets > 0:
        reference = reference_observables(model, cfg, args.w1_reference_jets, dev, n_particles=bench.N_PART,
                                          substructure=args.substructure, micro_batch=args.micro_batch, precision=args.precision,
                                          efp=args.efp)
    particles = None
    if args.w1p_reference_jets > 0:
        particles = reference_particles(model, cfg, args.w1p_reference_jets, dev, n_particles=bench.N_PART, micro_batch=args.micro_batch,
                                        precision=args.precision)
    fpd_reference = None
    if args.fpd_reference_jets > 0:
        fpd_reference = reference_fpd_features(model, cfg, args.fpd_reference_jets, dev, n_particles=bench.N_PART,
                                               micro_batch=args.micro_batch, precision=args.precision)
    rec = sharded_generation_run(model, cfg, args.jets, rank, world, dev, micro_batch=args.micro_batch, n_particles=bench.N_PART,
                                 precision=args.precision, substructure=args.substructure, w1_reference=reference,
                                 efp=args.efp, particle_reference=particles, fpd_reference=fpd_reference)
    if rank == 0:
        line = json.dumps(rec)
        print(line)
        if args.out:
            with open(args.out, "w") as f:
                f.write(line + "\n")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
