"""Cost of the genome-wide budget against the per-chromosome search, on the same device-resident scores.

Scores: synthetic hg38 @ 50 bp x 10 samples, scored on the device (rocco_b200.synth).  Legs, timed with CUDA events after a
warm-up, median of --reps:
  * per_chromosome: the batched per-chromosome search with the HG_PARAMS budgets and gammas (pipeline.solve_packed);
  * genome: the genome-wide search (pipeline.solve_genome_packed) at the bin-weighted mean of those budgets;
  * allreduce: one torch.distributed.all_reduce of 2^L + 1 doubles (L = 2), the per-round collective of the genome search.
Run on one GPU as `python tools/genome_budget.py`, and sharded over ranks (chromosomes by LPT, pipeline.lpt_partition) as
`torchrun --nproc-per-node 8 tools/genome_budget.py`.  Rank 0 prints one JSON line, with the card name and power limit read in
the same run (and appends it to --out when given).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np
import torch


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def timed(fn, reps):
    out, ms = None, []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return out, float(np.median(ms)), ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=10)
    ap.add_argument("--step", type=int, default=50)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    args = ap.parse_args()

    import torch.distributed as dist
    from rocco_b200 import pipeline
    from rocco_b200.synth import HG_PARAMS, HG38_SIZES, chrom_bins, chrom_matrix_torch, chrom_seed

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    names = list(HG38_SIZES)
    bins = [chrom_bins(c, args.step) for c in names]
    mine = pipeline.lpt_partition(bins, world)[rank]
    lengths = [bins[k] for k in mine]
    offsets, total = pipeline.layout_offsets(lengths)
    d_scores = torch.zeros(total, dtype=torch.float64, device=dev)
    prm = pipeline.score_params(prior_df=6.0)
    for k, off, n in zip(mine, offsets, lengths):
        x = chrom_matrix_torch(args.samples, n, chrom_seed(names[k]), dev)
        pipeline.score_loci_wls_device(x, out_scores=d_scores[off:off + n], params=prm)
        del x
    torch.cuda.synchronize()
    budgets = [HG_PARAMS[names[k]][0] for k in mine]
    gammas = [HG_PARAMS[names[k]][1] for k in mine]
    genome_budget = float(sum(HG_PARAMS[c][0] * b for c, b in zip(names, bins)) / sum(bins))
    d_masks = torch.zeros(total, dtype=torch.uint8, device=dev)

    rec = {"card": card(), "ranks": world, "samples": args.samples, "step": args.step, "genome_bins": int(sum(bins)),
           "genome_budget": genome_budget, "reps": args.reps}
    # warm-up of both searches
    pipeline.solve_packed(d_scores, offsets, lengths, budgets, gammas, d_masks=d_masks)
    pipeline.solve_genome_packed(d_scores, offsets, lengths, genome_budget, gammas, d_masks=d_masks)
    if world > 1:
        dist.barrier()
    (_, per), ms_per, _ = timed(lambda: pipeline.solve_packed(d_scores, offsets, lengths, budgets, gammas, d_masks=d_masks),
                                args.reps)
    if world > 1:
        dist.barrier()
    (_, genome, _), ms_gen, all_gen = timed(
        lambda: pipeline.solve_genome_packed(d_scores, offsets, lengths, genome_budget, gammas, d_masks=d_masks), args.reps)
    rec["per_chromosome"] = {"ms": ms_per, "rounds_max": max([r["search_rounds"] for r in per], default=0)}
    rec["genome"] = {"ms": ms_gen, "ms_all": all_gen, "rounds": genome["search_rounds"], "dp_passes": genome["dp_passes"],
                     "selection_penalty": genome["selection_penalty"], "selected_count": genome["selected_count"],
                     "target_count": genome["target_count"]}
    if world > 1:
        buf = torch.zeros(5, dtype=torch.float64, device=dev)
        for _ in range(20):
            dist.all_reduce(buf)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(200):
            dist.all_reduce(buf)
        b.record()
        torch.cuda.synchronize()
        rec["allreduce_us"] = a.elapsed_time(b) * 1000.0 / 200
        ms = torch.tensor([ms_per, ms_gen], dtype=torch.float64, device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        rec["slowest_rank_ms"] = {"per_chromosome": float(ms[0]), "genome": float(ms[1])}
    if rank == 0:
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
