"""Column statistics at large sample counts: the per-thread list kernels (automatic mode below the crossover) against the
shared-memory tile kernel (rocco_b200_colstat_set_mode(1)), per (m, statistic, dtype).  Prints one JSON line with ms,
algorithmic GB/s (m * bytes_in + 8 per bin) and bins/s for each, the GPU's name and its power limit.  Inputs are sized
past L2; each timing is the median of CUDA-event timed launches after warm-up.  A kernel that refuses a size (the list
kernels above 768 / ~1600 samples) is reported as null.

    python tools/colstat_large.py [--ms 100,300,768,1000,4096,16384] [--stats median,mad,tmean,mean] [--reps 5]
"""
import argparse, json, os, subprocess, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rocco_b200 import _lib, pipeline
from rocco_b200.synth import chrom_matrix_torch

ap = argparse.ArgumentParser()
ap.add_argument("--ms", default="100,300,768,1000,4096,16384")
ap.add_argument("--stats", default="median,quantile,mad,iqr,tmean,tstd,mean")
ap.add_argument("--dtypes", default="float32,float64")
ap.add_argument("--bytes", type=float, default=2e9, help="input size per case (L2 is 126 MB)")
ap.add_argument("--reps", type=int, default=5)
args = ap.parse_args()
lib = _lib.load()
dev = torch.device("cuda", 0)


def power_limit():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return q.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        return None


def timed(fn):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(args.reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return sorted(ts)[len(ts) // 2]


rows = []
for dt in args.dtypes.split(","):
    dtype = getattr(torch, dt)
    esize = torch.tensor([], dtype=dtype).element_size()
    for m in [int(v) for v in args.ms.split(",")]:
        n = max(4096, int(args.bytes / (m * esize)))
        x = chrom_matrix_torch(m, n, 1234, dev, dtype)
        out = torch.empty(n, dtype=torch.float64, device=dev)
        nbytes = m * n * esize + 8 * n
        for stat in args.stats.split(","):
            row = {"m": m, "n": n, "dtype": dt, "stat": stat}
            res = {}
            for name, mode in (("lists", 0), ("tile", 1)):
                prev = lib.rocco_b200_colstat_set_mode(mode)
                try:
                    ms = timed(lambda: pipeline.column_stat_device(x, stat, out=out))
                    row[name] = {"ms": ms, "GBps": nbytes / 1e9 / (ms / 1e3), "bins_per_s": n / (ms / 1e3)}
                    res[name] = out.clone()
                except ValueError:
                    row[name] = None
                finally:
                    lib.rocco_b200_colstat_set_mode(prev)
            if len(res) == 2:
                row["same_values"] = bool(torch.equal(res["lists"], res["tile"]) or
                                          torch.equal(torch.nan_to_num(res["lists"], 7.0), torch.nan_to_num(res["tile"], 7.0)))
            rows.append(row)
            print(json.dumps(row), file=sys.stderr, flush=True)
        del x, out
        torch.cuda.empty_cache()
print(json.dumps({"gpu": torch.cuda.get_device_name(dev), "power_limit": power_limit(), "rows": rows}))
