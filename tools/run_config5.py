"""BASELINE.json config 5 at full size: hg38 @ 20 bp (154.4 M bins) x 1000 samples stored float32 (617.7 GB), SAMPLES sharded
over the ranks (125 per GPU at 8), one all-reduce of the four per-bin accumulators per chromosome, then a 256-multiplier sweep
per chromosome on the rank that owns it (LPT).  Chromosomes are generated, scored and dropped one at a time, so a rank never
holds more than one chromosome's matrix + scratch (~35 GB).

    torchrun --nproc-per-node 8 tools/run_config5.py [--samples 1000] [--step-bp 20] [--chroms chr1,chr2] [--budget-null]
                                                      [--random-streams numpy] [--central-tendency median]

--budget-null replaces the sweep by the default CLI flow on the same layout: per chromosome the sharded scoring keeps each
rank's centred rows, the wild-bootstrap budget null runs with the samples still sharded (2n column sums all-reduced per
scoring pass), the fractions go through the empirical-Bayes budgets and the automatic gamma (host, identical on every
rank), and the owner rank solves each chromosome at its budget: pipeline.run_sample_sharded_defaults.
--random-streams numpy draws the null's innovations from the reference's own NumPy streams, each rank generating the rows
of its samples.
"""
import argparse, json, math, os, sys, time
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rocco_b200 import pipeline, _lib
from rocco_b200.synth import HG38_SIZES, HG_PARAMS, chrom_matrix_torch, chrom_seed

ap = argparse.ArgumentParser()
ap.add_argument("--samples", type=int, default=1000)
ap.add_argument("--step-bp", type=int, default=20)
ap.add_argument("--chroms", default="")
ap.add_argument("--multipliers", type=int, default=256)
ap.add_argument("--budget-null", action="store_true", help="budget null + EB budgets + solve instead of the sweep")
ap.add_argument("--null-draws", type=int, default=25)
ap.add_argument("--random-streams", choices=("philox", "numpy"), default="philox", help="with --budget-null: the null's innovations")
ap.add_argument("--central-tendency", default="", help="score each chromosome by this column statistic of the sharded "
                "samples (median, mean, tmean, quantile, ...) instead of the WLS score")
args = ap.parse_args()
rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
local = int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if world > 1:
    dist.init_process_group("nccl", device_id=dev)
names = [c for c in HG38_SIZES if not args.chroms or c in args.chroms.split(",")]
bins = [int(math.ceil(HG38_SIZES[c] / args.step_bp)) for c in names]
m_local = args.samples // world
owner = {}
for r, part in enumerate(pipeline.lpt_partition(bins, world)):
    for k in part:
        owner[k] = r
prm = pipeline.score_params(prior_df=6.0)
ev = lambda: torch.cuda.Event(enable_timing=True)


def budget_null_run():
    """pipeline.run_sample_sharded_defaults on the config-5 layout, chromosomes generated just in time; its mark hook
    records the per-chromosome events and, after each null, times the collective alone at the estimator's size."""
    per_chrom, events = {}, {}

    def chroms():
        for c, n in zip(names, bins):
            x = chrom_matrix_torch(m_local, n, chrom_seed(c), dev, torch.float32, sample_stream=rank + 1)
            if world > 1:
                dist.barrier()
            yield c, x
            del x

    def mark(label):
        e = ev()
        e.record()
        events[label] = e
        if label.startswith("done:"):
            # the collective alone, at the estimator's size (2n sums + 4 status slots), timed after the call
            n = bins[names.index(label[5:])]
            buf = torch.zeros(2 * n + 4, dtype=torch.float64, device=dev)
            r = [ev() for _ in range(2)]
            if world > 1:
                dist.all_reduce(buf)
            r[0].record()
            for _ in range(5):
                if world > 1:
                    dist.all_reduce(buf)
            r[1].record()
            torch.cuda.synchronize()
            per_chrom[label[5:]] = {"all_reduce_ms": r[0].elapsed_time(r[1]) / 5}

    out = pipeline.run_sample_sharded_defaults(chroms(), m_local * world, prm, mark=mark,
                                              default_args={"num_null_draws": args.null_draws,
                                                            "random_streams": args.random_streams})
    torch.cuda.synchronize()
    for c, n in zip(names, bins):
        det = out["defaults"]["null"][c]
        passes = 2 + int(det["num_null_draws"])
        null_ms = events[f"null:{c}"].elapsed_time(events[f"done:{c}"])
        per_chrom[c].update({"bins": n, "score_ms": events[f"score:{c}"].elapsed_time(events[f"null:{c}"]),
                             "budget_null_ms": null_ms, "passes": passes, "ms_per_pass": null_ms / passes,
                             "nonnull_fraction": det["nonnull_fraction"]})
    t_solve = events["solve"].elapsed_time(events["end"])
    solved = {c: int(r["selected_count"]) for c, r in zip(out["my_names"], out["results"])}
    budgets, gammas = out["budgets"], out["gammas"]
    keys = ("score_ms", "budget_null_ms", "ms_per_pass", "all_reduce_ms")
    t = torch.tensor([[per_chrom[c][q] for q in keys] + [per_chrom[c]["passes"]] for c in names], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    gathered = [None] * world
    if world > 1:
        dist.all_gather_object(gathered, solved)
    else:
        gathered = [solved]
    if rank == 0:
        mx = t.tolist()
        print(json.dumps({
            "config": f"hg38 @ {args.step_bp} bp x {m_local * world} samples f32, sample-sharded over {world} GPUs, budget null + "
                      f"EB budgets + auto gamma + solve ({args.random_streams} streams)", "gpu": torch.cuda.get_device_name(dev),
            "chroms": {c: {"bins": per_chrom[c]["bins"], "budget": budgets[c], "gamma": gammas[c],
                           "nonnull_fraction": per_chrom[c]["nonnull_fraction"],
                           "ms_max_over_ranks": dict(zip(keys, mx[i][:4])), "passes_max_over_ranks": int(mx[i][4]),
                           "selected": next((g[c] for g in gathered if c in g), None)} for i, c in enumerate(names)},
            "solve_ms_rank0": t_solve}))


def central_tendency_run():
    """bigWig-style scoring on the config-5 layout: per chromosome the column statistic of the sample-sharded matrix (one
    all-to-all of the rows by bin range, the kernel on the owned range, one all-gather of the track), then the sweep on
    the chromosome's owner.  The exchange and the kernel are timed apart: the exchange alone is rerun at the call's size."""
    per = {}
    for k, (c, n) in enumerate(zip(names, bins)):
        x = chrom_matrix_torch(m_local, n, chrom_seed(c), dev, torch.float32, sample_stream=rank + 1)
        if world > 1:
            dist.barrier()
        e = [ev() for _ in range(3)]
        e[0].record()
        scores = pipeline.column_stat_sample_sharded(x, m_local * world, args.central_tendency)
        e[1].record()
        if owner[k] == rank:
            srt = torch.sort(scores).values
            lo, hi = float(srt[int(0.50 * (n - 1))]), float(srt[int(0.999 * (n - 1))])
            pipeline.sweep_multipliers(scores, HG_PARAMS[c][1], np.linspace(max(lo, 0.0), max(hi, lo), args.multipliers))
        e[2].record()
        torch.cuda.synchronize()
        # the pieces: pack + all-to-all, then the kernel on the owned range of m_total rows
        ranges = pipeline.column_bin_ranges(n, world)
        lo_b, hi_b = ranges[rank]
        t = [ev() for _ in range(4)]
        t[0].record()
        send = pipeline.column_pack_ranges(x, ranges)
        recv = torch.empty(m_local * world * (hi_b - lo_b), dtype=x.dtype, device=dev)
        t[1].record()
        if world > 1:
            dist.all_to_all_single(recv, send, [m_local * (hi_b - lo_b)] * world, [m_local * (b - a) for a, b in ranges])
        t[2].record()
        del send
        if hi_b > lo_b:
            pipeline.column_stat_device(recv.view(m_local * world, hi_b - lo_b), args.central_tendency)
        t[3].record()
        torch.cuda.synchronize()
        per[c] = [n, e[0].elapsed_time(e[1]), e[1].elapsed_time(e[2]), t[0].elapsed_time(t[1]), t[1].elapsed_time(t[2]),
                  t[2].elapsed_time(t[3])]
        del x, recv, scores
    keys = ("sharded_stat_ms", "sweep_ms(owner)", "pack_ms", "all_to_all_ms", "kernel_ms")
    t = torch.tensor([per[c][1:] for c in names], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        mx = t.tolist()
        tot = [sum(r[i] for r in mx) for i in range(len(keys))]
        print(json.dumps({"config": f"hg38 @ {args.step_bp} bp x {m_local * world} samples f32, sample-sharded over {world} "
                                    f"GPUs, column statistic {args.central_tendency!r} + {args.multipliers}-multiplier sweep",
                          "gpu": torch.cuda.get_device_name(dev), "bins": sum(bins),
                          "ms_max_over_ranks_total": dict(zip(keys, tot)),
                          "chroms": {c: dict(zip(("bins",) + keys, [per[c][0]] + mx[i])) for i, c in enumerate(names)}}))


if args.central_tendency:
    central_tendency_run()
    if world > 1:
        dist.destroy_process_group()
    sys.exit(0)
if args.budget_null:
    budget_null_run()
    if world > 1:
        dist.destroy_process_group()
    sys.exit(0)
t_score = t_reduce = t_final = t_sweep = 0.0
gen = 0.0
selected = {}
for k, (c, n) in enumerate(zip(names, bins)):
    g0 = time.perf_counter()
    x = chrom_matrix_torch(m_local, n, chrom_seed(c), dev, torch.float32, sample_stream=rank + 1)
    torch.cuda.synchronize(); gen += time.perf_counter() - g0
    if world > 1:
        dist.barrier()
    e = [ev() for _ in range(5)]
    e[0].record()
    acc = pipeline.score_partial_device(x, prm)
    e[1].record()
    if world > 1:
        dist.all_reduce(acc)
    e[2].record()
    scores = pipeline.score_finalize_device(acc, m_local * world, prm)
    e[3].record()
    if owner[k] == rank:
        srt = torch.sort(scores).values
        lo, hi = float(srt[int(0.50 * (n - 1))]), float(srt[int(0.999 * (n - 1))])
        lam = np.linspace(max(lo, 0.0), hi, args.multipliers)
        counts, pen, obj = pipeline.sweep_multipliers(scores, HG_PARAMS[c][1], lam)
        selected[c] = (int(counts[0]), int(counts[-1]))
    e[4].record()
    torch.cuda.synchronize()
    t_score += e[0].elapsed_time(e[1]); t_reduce += e[1].elapsed_time(e[2]); t_final += e[2].elapsed_time(e[3])
    t_sweep += e[3].elapsed_time(e[4])
    del x, acc, scores
t = torch.tensor([t_score, t_reduce, t_final, t_sweep, t_score + t_reduce + t_final + t_sweep, gen * 1e3], dtype=torch.float64, device=dev)
if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
if rank == 0:
    tot_bins = sum(bins)
    ms = t.tolist()
    print(json.dumps({"config": f"hg38 @ {args.step_bp} bp x {m_local * world} samples f32, sample-sharded over {world} GPUs, "
                                f"{args.multipliers}-multiplier sweep", "bins": tot_bins, "input_GB": tot_bins * m_local * world * 4 / 1e9,
                      "ms_max_over_ranks": {"score_partial": ms[0], "all_reduce_4xn_f64": ms[1], "finalize": ms[2],
                                            "sort+sweep (owner rank)": ms[3], "total": ms[4], "synthetic_generation(untimed)": ms[5]},
                      "bins_per_s": tot_bins / (ms[4] / 1e3), "sample_bins_per_s": tot_bins * m_local * world / (ms[4] / 1e3),
                      "allreduce_bytes": tot_bins * 32, "sweep_counts_first_last(rank0 chroms)": selected}))
if world > 1:
    dist.destroy_process_group()
