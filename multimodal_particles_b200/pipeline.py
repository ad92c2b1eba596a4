"""BASELINE config 5: a generation run of many jets sharded over the GPUs of one box, entirely on the device.

Each rank owns a contiguous slice of the jets (``sharding.shard_range``; its start is the Philox jet offset, so the jets — and
therefore every histogram count — do not depend on the number of GPUs) and walks it in micro-batches: source state on the
device (``mmb_sample_source``; reference ``sample_noise`` / ``sample_masks``, mp/data/particle_clouds/utils.py:222-286), the
fused solver loop (``mmb_generate``; mbm.py:199-216), post-processing + jet observables (``mmb_jet_observables``;
particles.py:85-89,124-156, jets.py:90-107) and the validation histograms (``mmb_validation_histograms``) accumulated into
per-GPU int64 counts.  Exchanges (SURVEY.md §8e): the packed micro-batch (1 792 B / jet) goes to every rank once per micro-batch,
on a side stream under the next micro-batch's generation — pushed over NVLink peer memory by the copy engines
(``sharding.PeerGather``; one NCCL all-gather where peer memory is unavailable) — and one all-reduce of the histograms and of the
jet-observable sums at the end.  ``_jet_features`` runs the per-jet kernels of a micro-batch for the side stream and the
reference builders alike; its outputs feed additive sums (zeroed after the warm-up and all-reduced in the timed window as one
list), one per-jet row buffer in jet order (gathered after the window by ``_gather_rows``) or the particle draw buffers.  With
``substructure=True`` the side stream also runs ``mmb_jet_substructure`` on every micro-batch and histograms tau21, tau32 and D2
into int64 counts of their own (SUBSTRUCTURE_BINS).  With ``w1_reference`` the row buffer holds the W1_COLUMNS of every jet;
after the timed window they are scored against the reference with ``mmb_wasserstein1d`` (``reference_observables`` builds an
independent reference sample).  With ``efp=True`` the side stream also runs ``mmb_energy_flow_polynomials``; their columns join
the W1 columns, and with a reference the five d = 4 EFPs are also scored by FPD and KPD (``observables.fpd`` / ``kpd``) after the
timed window.  With ``particle_reference`` the side stream copies the post-processed particles of the jets JetNet's W1-P draws
(``observables.jetnet_draws``, made before the window) into one buffer; after the window the buffers of the ranks are summed and
scored with ``observables.w1p`` (``reference_particles`` builds the reference), and with ``w1_reference`` W1-M and W1-EFP are
scored from the gathered jet columns.  With ``fpd_reference`` the side stream also runs ``mmb_energy_flow_polynomials_d4`` and
JetNet's FPD / KPD features (``observables.jetnet_fpd_features``, every EFP of degree <= 4) of every jet follow the W1 columns in
the row buffer; after the window they are scored with ``fpd`` and ``kpd`` (``reference_fpd_features`` builds the reference).  The
reference has no multi-GPU code (SURVEY.md §2.1); ``tools/million_jets.py`` and the multi-GPU arms of ``bench.py`` call this.
"""
import hashlib

import numpy as np
import torch
import torch.distributed as dist

from . import sharding
from .observables import (EFP_COLUMNS, FPD_EFP_COLUMNS, JET_COLUMNS, PARTICLE_COLUMNS, SUBSTRUCTURE_COLUMNS, energy_flow_polynomials, fpd,
                          jet_observables, jet_substructure, jetnet_draws, jetnet_fpd_features, kpd, w1_summary, w1efp, w1m, wasserstein1d,
                          wasserstein1d_drawn)
from .source import sample_source_state

STATS = {"mean": [1.2, 0.0, 0.0], "std": [0.35, 0.2, 0.2]}   # de-standardisation to a jet-like scale (pT > 0)
# substructure histograms: (column, lo, hi) with 100 bins each, out-of-range values in the edge bins, then one count of the jets
# where the observable is undefined (NaN); counts layout [3][101]
SUBSTRUCTURE_HISTS = (("tau21", 0.0, 1.0), ("tau32", 0.0, 1.0), ("d2", 0.0, 10.0))
SUBSTRUCTURE_BINS = 100
# jet-level columns scored by W1 against a reference sample; with substructure, W1_SUBSTRUCTURE_COLUMNS follow, then with efp
# EFP_COLUMNS (FPD and KPD score EFP_COLUMNS[1:], the five d = 4 EFPs)
W1_COLUMNS = ("pt", "m", "eta", "phi", "multiplicity", "Q_total", "Q_jet")
W1_SUBSTRUCTURE_COLUMNS = ("tau21", "tau32", "d2")


def w1_columns(substructure=False, efp=False):
    return W1_COLUMNS + (W1_SUBSTRUCTURE_COLUMNS if substructure else ()) + (EFP_COLUMNS if efp else ())


def _w1_index(device):
    """Device index tensors of W1_COLUMNS in jet_observables rows and of W1_SUBSTRUCTURE_COLUMNS in jet_substructure rows (made
    once, so that picking the columns of a micro-batch copies nothing from the host)."""
    return (torch.tensor([JET_COLUMNS.index(c) for c in W1_COLUMNS], device=device),
            torch.tensor([SUBSTRUCTURE_COLUMNS.index(c) for c in W1_SUBSTRUCTURE_COLUMNS], device=device))


def _jet_features(x, k, m, stats, particles=False, substructure=False, efp=False, fpd=False):
    """The per-jet kernels on one micro-batch, each only when wanted: (x_phys [B,N,3] | None, jets [B,11], sub [B,8] | None,
    efps [B,6] | None, fpd [B, len(FPD_EFP_COLUMNS)] | None) from ``jet_observables`` (post-processed particles with
    ``particles``), ``jet_substructure``, ``energy_flow_polynomials`` and ``jetnet_fpd_features``."""
    x_phys, _, jets = jet_observables(x, k, m, stats, want_particles=particles)
    return (x_phys, jets, jet_substructure(x, m, stats) if substructure else None, energy_flow_polynomials(x, m, stats) if efp else None,
            jetnet_fpd_features(x, m, stats) if fpd else None)


def _rows(features, index, w1=True):
    """[B, K] f32: one micro-batch's per-jet rows from its ``_jet_features``: with ``w1`` the W1 columns (those computed of
    ``w1_columns``), then FPD_EFP_COLUMNS when they were computed."""
    _, jets, sub, efps, fpd_features = features
    rows = []
    if w1:
        rows += [jets.index_select(1, index[0])] + ([sub.index_select(1, index[1])] if sub is not None else []) + ([efps] if efps is not None else [])
    if fpd_features is not None:
        rows.append(fpd_features)
    return rows[0] if len(rows) == 1 else torch.cat(rows, 1)


def _target_multiplicity(N):
    return np.clip(np.rint(np.random.default_rng(0).normal(45, 18, 20000)), 1, N).astype(int)     # JetClass-like multiplicities


class SubstructureHistograms:
    """int64 counts [3 * 101] and sums of the defined values [3] (f64) of tau21, tau32 and D2; integer scatter-adds only, so
    the counts do not depend on the batching or on the order of the jets."""

    def __init__(self, device):
        nb = SUBSTRUCTURE_BINS
        self.cols = [SUBSTRUCTURE_COLUMNS.index(c) for c, _, _ in SUBSTRUCTURE_HISTS]
        self.lo = torch.tensor([h[1] for h in SUBSTRUCTURE_HISTS], dtype=torch.float32, device=device)
        self.scale = torch.tensor([nb / (h[2] - h[1]) for h in SUBSTRUCTURE_HISTS], dtype=torch.float32, device=device)
        self.offset = torch.arange(3, device=device) * (nb + 1)
        self.counts = torch.zeros(3 * (nb + 1), dtype=torch.int64, device=device)
        self.sums = torch.zeros(3, dtype=torch.float64, device=device)

    def add(self, sub):
        """Adds one batch of ``jet_substructure`` rows [B, 8]."""
        nb = SUBSTRUCTURE_BINS
        v = sub[:, self.cols]
        undefined = torch.isnan(v)
        b = ((v - self.lo) * self.scale).floor().clamp_(0, nb - 1)
        b = torch.where(undefined, float(nb), b).long() + self.offset
        self.counts.scatter_add_(0, b.reshape(-1), torch.ones(b.numel(), dtype=torch.int64, device=sub.device))
        self.sums.add_(torch.where(undefined, 0.0, v).double().sum(0))


def sharded_generation_run(model, cfg, total_jets, rank, world, device, micro_batch=4096, n_particles=128, precision="auto",
                           warmup_batches=2, gather="auto", substructure=False, w1_reference=None, efp=False, particle_reference=None,
                           fpd_reference=None):
    """-> dict (rank 0: the C5 record; other ranks: None).  Device time by CUDA events around the whole slice incl. the final
    all-reduce, max over ranks.  ``substructure``: also histogram tau21, tau32 and D2 of every jet (``substructure_sha1``,
    ``substructure_counts`` and the means of the defined values join the record).  ``w1_reference``: [m, K] f32 device tensor
    of reference values of ``w1_columns(substructure)``; after the timed window the generated values of every jet are gathered
    in jet order and ``w1`` ({column: W1}), ``w1_used`` ({column: [finite generated, finite reference]}),
    ``w1_reference_jets`` and ``w1_seconds`` (CUDA events around the W1 call) join the record.  ``efp``: also compute the
    energy flow polynomials of every jet (the means of the defined values join the record as ``mean_efp1`` ...); their
    columns follow in ``w1_columns(substructure, efp)``, and with a reference ``fpd`` and ``kpd`` ([value, error] of the five
    d = 4 EFPs against the reference's) and ``jet_metrics_seconds`` (CUDA events around both) join the record too.
    ``particle_reference``: (x [m, N, 3] f32, mask [m, N] u8) device tensors of post-processed reference particles
    (``reference_particles``); ``w1p`` ([mean, std]), ``w1p_features`` ({column: [mean, std]}), with ``w1_reference`` also ``w1m``
    and with ``efp`` ``w1efp`` (JetNet's defaults, ``observables.w1p`` / ``w1m`` / ``w1efp``), and ``jetnet_w1_seconds`` (CUDA
    events around the whole scoring, so it includes its host waits for the per-draw values) join the record.
    ``fpd_reference``: [m, len(FPD_EFP_COLUMNS)] f32 device tensor of reference ``observables.jetnet_fpd_features``
    (``reference_fpd_features``); the side stream keeps those features of every jet (144 B per jet), and after the timed window
    they are gathered in jet order and ``jetnet_fpd`` and ``jetnet_kpd`` ([value, error] of ``fpd`` / ``kpd`` at their
    defaults), ``jetnet_fpd_reference_jets`` and ``jetnet_fpd_seconds`` (CUDA events around both calls) join the record."""
    native = model.encoder.native_model(device)
    table = model.step_table()
    lo, hi = sharding.shard_range(total_jets, rank, world)
    MB, N = micro_batch, n_particles
    mult_hist = _target_multiplicity(N)
    hist = sharding.ValidationHistograms(device, vocab_size=cfg.data.vocab_size_features)
    counts = torch.zeros(hist.size, dtype=torch.int64, device=device)
    jet_sums = torch.zeros(11, dtype=torch.float64, device=device)
    sub_hist = SubstructureHistograms(device) if substructure else None
    efp_sums = torch.zeros(len(EFP_COLUMNS) + 1, dtype=torch.float64, device=device) if efp else None   # sums, then defined jets
    # the additive accumulators: zeroed after the warm-up, all-reduced inside the timed window
    additive = [counts, jet_sums] + ([sub_hist.counts, sub_hist.sums] if substructure else []) + ([efp_sums] if efp else [])
    w1_cols = w1_columns(substructure, efp)
    n_w1 = len(w1_cols) if w1_reference is not None else 0
    if w1_reference is not None and (w1_reference.dim() != 2 or w1_reference.shape[1] != len(w1_cols)):
        raise ValueError(f"w1_reference must be [m, {len(w1_cols)}] ({', '.join(w1_cols)}), got {tuple(w1_reference.shape)}")
    if particle_reference is not None:
        p_ref_x, p_ref_m = particle_reference
        if p_ref_x.dim() != 3 or tuple(p_ref_x.shape[1:]) != (N, 3) or p_ref_m.shape[:2] != p_ref_x.shape[:2]:
            raise ValueError(f"particle_reference must be (x [m, {N}, 3], mask [m, {N}]), got {tuple(p_ref_x.shape)}, {tuple(p_ref_m.shape)}")
        p_plan = _particle_plan(len(p_ref_x), total_jets, lo, hi, MB, device)
        p_x = torch.zeros(p_plan["slots"], N, 3, dtype=torch.float32, device=device)   # the drawn jets' particles, by draw slot
        p_m = torch.zeros(p_plan["slots"], N, dtype=torch.uint8, device=device)
    if fpd_reference is not None:
        if fpd_reference.dim() != 2 or fpd_reference.shape[1] != len(FPD_EFP_COLUMNS):
            raise ValueError(f"fpd_reference must be [m, {len(FPD_EFP_COLUMNS)}] (FPD_EFP_COLUMNS), got {tuple(fpd_reference.shape)}")
    # per-jet rows of this rank's jets in jet order: the W1 columns (with w1_reference), then FPD_EFP_COLUMNS (with fpd_reference)
    n_rows = n_w1 + (len(FPD_EFP_COLUMNS) if fpd_reference is not None else 0)
    rows = torch.empty(hi - lo, n_rows, dtype=torch.float32, device=device) if n_rows else None
    w1_index = _w1_index(device)
    want = dict(particles=particle_reference is not None, substructure=substructure, efp=efp, fpd=fpd_reference is not None)
    packs = [sharding.PackedJets(MB, N, 3, device) for _ in range(3)]      # state of a micro-batch: [x | tokens | mask], one allocation
    recv = [sharding.make_gather(MB, N, 3, world, device, mode=gather) for _ in range(2)] if world > 1 else None
    side = torch.cuda.Stream(device=device)
    main_s = torch.cuda.current_stream(device)

    def run(n_from, n_to):
        # launch stream: source state + solver loop of micro-batch i, back to back; side stream: observables, histograms and the
        # exchange of micro-batch i under the generation of i + 1 (their small kernels find room in its tail).  A packed buffer
        # is refilled only after the side stream is done with it.
        free = [None] * len(packs)
        for i, start in enumerate(range(n_from, n_to, MB)):
            B = min(MB, n_to - start)
            pk = packs[i % 3]
            if free[i % 3] is not None:
                main_s.wait_event(free[i % 3])
            out = (pk.x, pk.k, pk.mask) if B == MB else None
            x, k, m = sample_source_state(B, N, target_multiplicity=mult_hist, min_num_particles=0, device=device, seed=7, jet_offset=start,
                                          compact=True, out=out)
            native.generate(x, k, m, table, seed=11, jet_offset=start, precision=precision)
            ev = torch.cuda.Event()
            ev.record(main_s)
            with torch.cuda.stream(side):
                side.wait_event(ev)
                features = _jet_features(x, k, m, STATS, **want)
                x_phys, jets, sub, efps, _ = features
                counts.add_(hist.accumulate(x, k, m))
                jet_sums.add_(torch.nan_to_num(jets.double()).sum(0))
                if substructure:
                    sub_hist.add(sub)
                if efp:
                    defined = ~torch.isnan(efps[:, :1])
                    efp_sums.add_(torch.cat([torch.where(defined, efps, 0.0).double().sum(0), defined.double().sum(0)]))
                if rows is not None:
                    rows[start - lo:start - lo + B].copy_(_rows(features, w1_index, w1=w1_reference is not None))
                if particle_reference is not None:
                    a, b = p_plan["ranges"][start]
                    if b > a:   # the draw slots of this micro-batch's jets (ranges made on the host before the window)
                        sel, jet = p_plan["slot"][a:b], p_plan["jet"][a:b] - start
                        p_x.index_copy_(0, sel, x_phys.index_select(0, jet))
                        p_m.index_copy_(0, sel, m.index_select(0, jet))
                if world > 1 and B == MB:
                    recv[i & 1].gather(pk)          # the packed micro-batch to every rank (copy-engine push, or one all-gather)
                for t in (x, k, m):
                    t.record_stream(side)
                free[i % 3] = torch.cuda.Event()
                free[i % 3].record(side)
        main_s.wait_stream(side)

    run(lo, min(hi, lo + warmup_batches * MB))       # warm-up, then reset the accumulators
    for acc in additive:
        acc.zero_()
    torch.cuda.synchronize(device)
    if world > 1:
        dist.barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record(main_s)
    run(lo, hi)
    if world > 1:
        for acc in additive:
            dist.all_reduce(acc)
    e.record(main_s)
    torch.cuda.synchronize(device)
    t = torch.tensor([s.elapsed_time(e)], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    all_rows = _gather_rows(rows, total_jets, world, device) if rows is not None and world > 1 else rows
    if particle_reference is not None and world > 1:   # every draw slot has one owner; the other ranks hold zeros
        dist.all_reduce(p_x)
        dist.all_reduce(p_m)
    if rank != 0:
        return None
    ms = float(t.item())
    off = 3 * hist.bins + cfg.data.vocab_size_features
    host_counts = counts.cpu().numpy()
    mult = host_counts[off:]
    rec = {"workload": f"C5: {total_jets} jets, N={N}, {table.n_steps} solver steps; source + generation + observables + histograms on "
                        f"the device, per-micro-batch all-gather of the jets + final all-reduce of the histograms",
            "n_gpus": world, "micro_batch": MB, "exchange": recv[0].kind if recv else "none", "seconds": ms * 1e-3, "value": total_jets / (ms * 1e-3), "unit": "jets/s",
            "precision": native.generate_precision(N, precision),
            "jets_in_histogram": int(mult.sum()), "mean_multiplicity": float((mult * np.arange(len(mult))).sum() / max(mult.sum(), 1)),
            "mean_jet_pt": float(jet_sums[4].item() / total_jets), "mean_jet_mass": float(jet_sums[5].item() / total_jets),
            "token_counts": host_counts[3 * hist.bins:off].tolist(),
            # integer counts of jets keyed by their GLOBAL index: identical for every number of GPUs
            "histogram_sha1": hashlib.sha1(host_counts.astype(np.int64).tobytes()).hexdigest()}
    if substructure:
        sc = sub_hist.counts.cpu().numpy().astype(np.int64)
        per = sc.reshape(3, SUBSTRUCTURE_BINS + 1)
        sums = sub_hist.sums.cpu().numpy()
        rec["substructure_counts"] = {name: per[i].tolist() for i, (name, _, _) in enumerate(SUBSTRUCTURE_HISTS)}
        for i, (name, _, _) in enumerate(SUBSTRUCTURE_HISTS):
            defined = int(per[i, :SUBSTRUCTURE_BINS].sum())
            rec[f"mean_{name}"] = float(sums[i] / defined) if defined else float("nan")
        rec["substructure_sha1"] = hashlib.sha1(sc.tobytes()).hexdigest()
    if efp:
        es = efp_sums.tolist()
        for name, v in zip(EFP_COLUMNS, es):
            rec[f"mean_{name}"] = v / es[-1] if es[-1] else float("nan")
    w1_all, w1_ref = None, None
    if w1_reference is not None:
        w1_all, w1_ref = all_rows[:, :n_w1], w1_reference.to(device, torch.float32)
        rec.update(_score_w1(w1_all, w1_ref, w1_cols))
        if efp:   # the five d = 4 EFPs
            pick = [w1_cols.index(c) for c in EFP_COLUMNS[1:]]
            rec.update(_score_fpd_kpd(w1_all[:, pick], w1_ref[:, pick], "fpd", "kpd", "jet_metrics_seconds"))
    if particle_reference is not None:
        rec.update(_score_jetnet_w1(p_ref_x.to(device, torch.float32), p_ref_m.to(device), p_x, p_m, p_plan["idx_real"], w1_all, w1_ref,
                                    w1_cols, efp))
    if fpd_reference is not None:
        rec.update(_score_fpd_kpd(all_rows[:, n_w1:], fpd_reference.to(device, torch.float32), "jetnet_fpd", "jetnet_kpd",
                                  "jetnet_fpd_seconds"))
        rec["jetnet_fpd_reference_jets"] = int(fpd_reference.shape[0])
    return rec


def _particle_plan(n_reference, total, lo, hi, micro_batch, device):
    """JetNet's W1-P draws over the global jets [0, total) (``jetnet_draws``: the same on every rank), sorted by jet, and the
    range of that order each micro-batch of this rank's [lo, hi) owns (one host read, before the timed window)."""
    idx_real, idx_gen = jetnet_draws(n_reference, total, device=device)
    jet, slot = torch.sort(idx_gen.reshape(-1).long(), stable=True)
    starts = torch.arange(lo, hi + micro_batch, micro_batch, device=device).clamp_(max=hi)
    cut = torch.searchsorted(jet, starts).tolist()
    return {"idx_real": idx_real, "slots": idx_gen.numel(), "jet": jet, "slot": slot,
            "ranges": {int(a): (cut[i], cut[i + 1]) for i, a in enumerate(starts[:-1].tolist())}}


def _timed(device, fn):
    """(fn(), seconds between CUDA events recorded on the current stream around it); ends in a synchronise."""
    stream = torch.cuda.current_stream(device)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record(stream)
    out = fn()
    e.record(stream)
    torch.cuda.synchronize(device)
    return out, s.elapsed_time(e) * 1e-3


def _score_jetnet_w1(ref_x, ref_m, gen_x, gen_m, idx_real, jet_values, jet_reference, cols, efp):
    """W1-P of the gathered draw slots against the reference particles (``observables.w1p`` with the run's draws), and with jet
    columns W1-M and W1-EFP (``observables.w1m`` / ``w1efp``).  The CUDA events span all of them, including the host reading
    each call's per-draw values and the numpy aggregation between the calls, so the time is that of the whole scoring."""
    def score():
        slots = torch.arange(gen_x.shape[0], dtype=torch.int32, device=gen_x.device).reshape(idx_real.shape)
        vals = wasserstein1d_drawn(ref_x, idx_real, gen_x, slots, ref_m, gen_m).cpu().numpy()
        rec = {"w1p": list(w1_summary(vals)),
               "w1p_features": {c: [float(a), float(b)] for c, a, b in zip(PARTICLE_COLUMNS, *w1_summary(vals, average=False))}}
        if jet_values is not None:
            m = cols.index("m")
            rec["w1m"] = list(w1m(jet_reference[:, m], jet_values[:, m]))
            if efp:
                pick = [cols.index(c) for c in EFP_COLUMNS[1:]]
                rec["w1efp"] = list(w1efp(jet_reference[:, pick], jet_values[:, pick]))
        return rec

    rec, seconds = _timed(gen_x.device, score)
    return dict(rec, jetnet_w1_seconds=seconds)


def _gather_rows(buf, total, world, device):
    """Every rank's [hi - lo, K] rows -> [total, K] in rank (= jet) order: padded to the largest shard, all-gathered, trimmed."""
    sizes = [b - a for a, b in (sharding.shard_range(total, r, world) for r in range(world))]
    S = max(sizes)
    padded = torch.zeros(S, buf.shape[1], dtype=buf.dtype, device=device)
    padded[:buf.shape[0]].copy_(buf)
    out = torch.empty(world * S, buf.shape[1], dtype=buf.dtype, device=device)
    dist.all_gather_into_tensor(out, padded)
    return torch.cat([out[r * S:r * S + sizes[r]] for r in range(world)])


def _score_w1(values, reference, cols):
    (w1, used), seconds = _timed(values.device, lambda: wasserstein1d(values, reference, return_counts=True))
    w1, used = w1.tolist(), used.tolist()
    return {"w1": dict(zip(cols, w1)), "w1_used": {c: [used[0][i], used[1][i]] for i, c in enumerate(cols)},
            "w1_reference_jets": int(reference.shape[0]), "w1_seconds": seconds}


def _score_fpd_kpd(values, reference, fpd_key, kpd_key, seconds_key):
    """FPD and KPD (observables.fpd / kpd at their defaults) of the gathered rows against the reference's, timed by CUDA events
    around both."""
    (f, k), seconds = _timed(values.device, lambda: (fpd(reference, values), kpd(reference, values)))
    return {fpd_key: list(f), kpd_key: list(k), seconds_key: seconds}


def _reference_jets(model, n_jets, device, N, jet_offset, micro_batch, precision):
    """Yields (start, x, k, mask) of the micro-batches of ``n_jets`` generated jets made as ``sharded_generation_run`` makes them
    (same model, source, solver) from the Philox jet offsets ``jet_offset + start + j``."""
    native = model.encoder.native_model(device)
    table = model.step_table()
    mult_hist = _target_multiplicity(N)
    for start in range(0, n_jets, micro_batch):
        B = min(micro_batch, n_jets - start)
        x, k, m = sample_source_state(B, N, target_multiplicity=mult_hist, min_num_particles=0, device=device, seed=7,
                                      jet_offset=jet_offset + start, compact=True)
        native.generate(x, k, m, table, seed=11, jet_offset=jet_offset + start, precision=precision)
        yield start, x, k, m


def _reference(model, n_jets, device, n_particles, jet_offset, micro_batch, precision, stats, outs, pick, **want):
    """Fills ``outs`` ([n_jets, ...] tensors) in jet order with ``pick(features, mask)`` of each micro-batch of ``_reference_jets``,
    ``features`` being its ``_jet_features(**want)``, so that a reference is made as the run makes its own values."""
    for start, x, k, m in _reference_jets(model, n_jets, device, n_particles, jet_offset, micro_batch, precision):
        for out, v in zip(outs, pick(_jet_features(x, k, m, stats, **want), m)):
            out[start:start + x.shape[0]] = v
    return outs


def reference_observables(model, cfg, n_jets, device, n_particles=128, substructure=False, jet_offset=1 << 40, micro_batch=16384,
                          precision="auto", stats=STATS, efp=False):
    """[n_jets, K] f32 on ``device``: the ``w1_columns(substructure, efp)`` of ``n_jets`` jets made as ``sharded_generation_run`` makes
    them (same model, source, solver, observables) but from the Philox jet offsets ``jet_offset + j``, disjoint from any run's
    [0, total), so the sample is independent of it.  W1 between two such samples is the seed-to-seed noise floor.  ``stats``:
    the de-standardisation of the observables."""
    out = torch.empty(n_jets, len(w1_columns(substructure, efp)), dtype=torch.float32, device=device)
    index = _w1_index(device)
    _reference(model, n_jets, device, n_particles, jet_offset, micro_batch, precision, stats, [out], lambda f, m: [_rows(f, index)],
               substructure=substructure, efp=efp)
    return out


def reference_particles(model, cfg, n_jets, device, n_particles=128, jet_offset=1 << 40, micro_batch=16384, precision="auto", stats=STATS):
    """(x [n_jets, N, 3] f32, mask [n_jets, N] u8) on ``device``: the post-processed particles (PARTICLE_COLUMNS) and masks of
    ``n_jets`` jets made as ``reference_observables`` makes them (same model, source, solver, post-processing, Philox jet offsets
    ``jet_offset + j``); the particle reference of ``sharded_generation_run(particle_reference=...)``.  ``jet_offset=0``
    reproduces the run's own jets."""
    N = n_particles
    outs = [torch.empty(n_jets, N, 3, dtype=torch.float32, device=device), torch.empty(n_jets, N, dtype=torch.uint8, device=device)]
    return tuple(_reference(model, n_jets, device, N, jet_offset, micro_batch, precision, stats, outs, lambda f, m: [f[0], m],
                            particles=True))


def reference_fpd_features(model, cfg, n_jets, device, n_particles=128, jet_offset=1 << 40, micro_batch=16384, precision="auto",
                           stats=STATS):
    """[n_jets, len(FPD_EFP_COLUMNS)] f32 on ``device``: ``observables.jetnet_fpd_features`` of ``n_jets`` jets made as
    ``reference_observables`` makes them (Philox jet offsets ``jet_offset + j``); the reference of
    ``sharded_generation_run(fpd_reference=...)``.  ``jet_offset=0`` reproduces the run's own jets."""
    out = torch.empty(n_jets, len(FPD_EFP_COLUMNS), dtype=torch.float32, device=device)
    _reference(model, n_jets, device, n_particles, jet_offset, micro_batch, precision, stats, [out], lambda f, m: [f[4]], fpd=True)
    return out
