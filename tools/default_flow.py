"""ROCCO's default flow (budget null -> EB budgets -> automatic gamma -> solve) on the synthetic config-4 genome, timed by
phase, next to the fixed-parameter step on the same matrices.

    python tools/default_flow.py [--samples 100] [--step-bp 50] [--chroms chr1,chr21] [--draws 25] [--random-streams numpy]
    torchrun --nproc-per-node 8 tools/default_flow.py

hg38 @ 50 bp x 100 samples float64, the chromosomes LPT-packed over the ranks and resident in HBM (as bench.py lays them
out).  pipeline.run_shard(budgets=None, gammas=None) runs once untimed, then once with its `mark` hook recording a CUDA
event at each phase boundary; the genome BED is written by distributed.write_genome_bed.  Phase times are the maximum
over ranks.  The fixed-parameter step (HG_PARAMS budgets and gammas, run_shard + genome BED) is timed on the same
matrices in the same process: median of --fixed-steps after one warm-up.  --random-streams picks the null's innovations:
Philox (default) or the reference's own NumPy streams generated on the device.  One JSON line on rank 0's stdout.
"""
import argparse, json, math, os, shutil, subprocess, sys, tempfile, time
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rocco_b200 import pipeline, distributed as rdist
from rocco_b200.synth import HG38_SIZES, HG_PARAMS, chrom_matrix_torch, chrom_seed

ap = argparse.ArgumentParser()
ap.add_argument("--samples", type=int, default=100)
ap.add_argument("--step-bp", type=int, default=50)
ap.add_argument("--chroms", default="")
ap.add_argument("--draws", type=int, default=25, help="num_null_draws (the reference's default is 25)")
ap.add_argument("--fixed-steps", type=int, default=3)
ap.add_argument("--random-streams", choices=("philox", "numpy"), default="philox",
                help="the budget null's innovations: Philox, or the reference's NumPy PCG64 streams")
args = ap.parse_args()
rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
local = int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if world > 1:
    dist.init_process_group("nccl", device_id=dev)


def gpu_card():
    """Name and power limit of this rank's GPU, read in the run that is measured."""
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power}
    except (OSError, ValueError, subprocess.SubprocessError):
        return {"name": torch.cuda.get_device_name(dev), "power_limit": "not read"}


names = [c for c in HG38_SIZES if not args.chroms or c in args.chroms.split(",")]
bins = [int(math.ceil(HG38_SIZES[c] / args.step_bp)) for c in names]
mine = pipeline.lpt_partition(bins, world)[rank]
my_names = [names[k] for k in mine]
d_mats = [chrom_matrix_torch(args.samples, bins[k], chrom_seed(names[k]), dev, torch.float64) for k in mine]
prm = pipeline.score_params(prior_df=6.0)
lex = sorted(names)
tmp = [tempfile.mkdtemp(prefix="rocco_b200_default_flow_") if rank == 0 else None]
if world > 1:
    dist.broadcast_object_list(tmp, src=0)
bed_path = os.path.join(tmp[0], "genome.bed")
empty = (np.zeros(0, np.int32), np.zeros(0, np.int64), np.zeros(0, np.int64))


def barrier():
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()


def write_bed(out):
    sel = sum(r["selected_count"] for r in out["results"])
    return rdist.write_genome_bed(bed_path, lex, my_names, out["runs"] if my_names else empty, args.step_bp,
                                  extras=(sel, sum(bins[k] for k in mine)), device=dev if world > 1 else None)


def default_flow(events=None):
    def mark(label):
        if events is not None:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            events.append((label, e))
    out = pipeline.run_shard(d_mats, None, None, params=prm, chrom_names=my_names, genome_names=names,
                             default_args={"num_null_draws": args.draws, "random_streams": args.random_streams}, mark=mark)
    mark("bed")
    t0 = time.perf_counter()
    tot = write_bed(out)
    mark("bed_end")
    torch.cuda.synchronize()
    return out, tot, 1e3 * (time.perf_counter() - t0)


default_flow()                                             # warm-up: modules, allocator, every kernel of the flow
barrier()
events = []
out, tot, bed_host_ms = default_flow(events)
barrier()
labels = [lab for lab, _ in events]
ms = [events[i][1].elapsed_time(events[i + 1][1]) for i in range(len(events) - 1)]     # phase i: label i -> label i+1
phase = {"score": 0.0, "null": 0.0, "agree": 0.0, "solve": 0.0, "runs": 0.0, "bed": 0.0}
null_by = {c: 0.0 for c in names}
for lab, t in zip(labels, ms):
    kind, _, chrom = lab.partition(":")
    if kind in ("score", "null"):
        phase[kind] += t
        if kind == "null":
            null_by[chrom] = t
    elif kind in phase:
        phase[kind] += t
phase["total"] = events[0][1].elapsed_time(events[-1][1])
phase["bed"] = max(phase["bed"], bed_host_ms)               # host-side text formatting and writes

# the fixed-parameter step on the same matrices
budgets = [HG_PARAMS[c][0] for c in my_names]
gammas = [HG_PARAMS[c][1] for c in my_names]


def fixed_step():
    o = pipeline.run_shard(d_mats, budgets, gammas, params=prm) if my_names else {"results": [], "runs": empty}
    write_bed(o)


fixed_step()
fixed = []
for _ in range(args.fixed_steps):
    barrier()
    t0 = time.perf_counter()
    fixed_step()
    torch.cuda.synchronize()
    fixed.append(1e3 * (time.perf_counter() - t0))
fixed_ms = float(np.median(fixed))

keys = list(phase)
vec = torch.tensor([phase[k] for k in keys] + [null_by[c] for c in names] + [fixed_ms], dtype=torch.float64, device=dev)
if world > 1:
    dist.all_reduce(vec, op=dist.ReduceOp.MAX)
vec = vec.tolist()
mine_info = {c: {"budget": b, "gamma": g, "draws": int(d["num_null_draws"]), "selected": int(r["selected_count"]),
                 "bins": int(n)}
             for c, b, g, d, r, n in zip(my_names, out["budgets"], out["gammas"], out["defaults"]["null"], out["results"],
                                         out["lengths"])}
every = [None] * world
if world > 1:
    dist.all_gather_object(every, {"card": gpu_card(), "chroms": mine_info})
else:
    every = [{"card": gpu_card(), "chroms": mine_info}]
if rank == 0:
    chroms = {}
    for e in every:
        chroms.update(e["chroms"])
    nb = len(keys)
    line = {
        "config": f"hg38 @ {args.step_bp} bp x {args.samples} samples f64 resident, chromosomes LPT-sharded over {world} GPU(s), "
                  f"ROCCO default flow (budget null with up to {args.draws} draws -> EB budgets -> automatic gamma -> solve)",
        "random_streams": args.random_streams,
        "gpus": [e["card"] for e in every], "bins": int(sum(bins)),
        "default_flow_ms_max_over_ranks": dict(zip(keys, vec[:nb])),
        "null_ms_by_chrom_max_over_ranks": dict(zip(names, vec[nb:nb + len(names)])),
        "fixed_param_step_ms_max_over_ranks": vec[-1],
        "default_over_fixed": vec[nb - 1] / vec[-1] if vec[-1] > 0 else None,
        "selected_bins": int(tot[0]), "chroms": {c: chroms[c] for c in names},
    }
    sys.stdout.write(json.dumps(line) + "\n")
    sys.stdout.flush()
barrier()
if rank == 0:
    shutil.rmtree(tmp[0], ignore_errors=True)
if world > 1:
    dist.destroy_process_group()
