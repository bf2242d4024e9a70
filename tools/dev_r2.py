"""Round-2 development probes (run on the GPU box): A/B checks and timings of the reworked kernels.

    python tools/dev_r2.py scopes      # per-scope times of one chromosome set (profile scopes)

Results go to stdout and gpurun_out/dev_<cmd>.json.
"""
import json
import os
import sys
import time

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from rocco_b200 import _lib, pipeline  # noqa: E402
from rocco_b200.synth import HG38_SIZES, HG_PARAMS, chrom_bins, chrom_matrix_numpy, chrom_matrix_torch, chrom_seed  # noqa: E402

DEV = torch.device("cuda", 0)
OUT = os.path.join(REPO, "gpurun_out")
os.makedirs(OUT, exist_ok=True)


def scopes_of(fn, reps=3):
    fn()
    torch.cuda.synchronize()
    _lib.profile_enable(True)
    _lib.profile_report()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    rep = _lib.profile_report()
    _lib.profile_enable(False)
    return {k: {"ms": v[0] / reps, "GBps": (v[2] / 1e9) / (v[0] / 1e3) if v[0] > 0 else 0.0} for k, v in rep.items()}


def cmd_scopes():
    names = sys.argv[2].split(",") if len(sys.argv) > 2 else ["chr21"]
    m = int(sys.argv[3]) if len(sys.argv) > 3 else 100
    mats = [chrom_matrix_torch(m, chrom_bins(c), chrom_seed(c), DEV, torch.float64) for c in names]
    budgets = [HG_PARAMS[c][0] for c in names]
    gammas = [HG_PARAMS[c][1] for c in names]
    prm = pipeline.score_params(prior_df=6.0)
    sp = scopes_of(lambda: pipeline.run_shard(mats, budgets, gammas, params=prm))
    tot = sum(v["ms"] for v in sp.values())
    for k, v in sorted(sp.items(), key=lambda kv: -kv[1]["ms"]):
        print(f"{k:28s} {v['ms']:9.3f} ms  {v['GBps']:8.1f} GB/s")
    print("total profiled", tot)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(3):
        pipeline.run_shard(mats, budgets, gammas, params=prm)
    torch.cuda.synchronize()
    print("wall per step ms", 1e3 * (time.perf_counter() - t0) / 3)
    json.dump(sp, open(os.path.join(OUT, "dev_scopes.json"), "w"), indent=1)




def cmd_fallback():
    """which rows of a chromosome take the sort fallback, and why"""
    import ctypes
    name = sys.argv[2] if len(sys.argv) > 2 else "chr1"
    m = int(sys.argv[3]) if len(sys.argv) > 3 else 100
    x = chrom_matrix_torch(m, chrom_bins(name), chrom_seed(name), DEV, torch.float64)
    lib = _lib.load()
    r0 = (ctypes.c_longlong * 8)(); r1 = (ctypes.c_longlong * 8)()
    lib.rocco_b200_trend_fallback_reasons(r0)
    f0 = lib.rocco_b200_trend_fallback_rows()
    pipeline.score_loci_wls_device(x, params=pipeline.score_params(prior_df=6.0))
    lib.rocco_b200_trend_fallback_reasons(r1)
    print(name, "fallback rows", lib.rocco_b200_trend_fallback_rows() - f0, "reasons [xslot,xcount,ytotal,yslot,ycount]", [r1[k] - r0[k] for k in range(5)])


def cmd_timeline():
    """device-side gaps between the profile scopes of one run_shard call"""
    names = sys.argv[2].split(",") if len(sys.argv) > 2 else ["chr21"]
    m = int(sys.argv[3]) if len(sys.argv) > 3 else 100
    mats = [chrom_matrix_torch(m, chrom_bins(c), chrom_seed(c), DEV, torch.float64) for c in names]
    budgets = [HG_PARAMS[c][0] for c in names]
    gammas = [HG_PARAMS[c][1] for c in names]
    prm = pipeline.score_params(prior_df=6.0)
    for _ in range(2):
        pipeline.run_shard(mats, budgets, gammas, params=prm)
    torch.cuda.synchronize()
    _lib.profile_enable(True)
    _lib.profile_report()
    pipeline.run_shard(mats, budgets, gammas, params=prm)
    torch.cuda.synchronize()
    tl = _lib.profile_timeline()
    _lib.profile_enable(False)
    _lib.profile_report()
    end_prev, gaps = None, {}
    busy = 0.0
    for name, t0, ms in tl:
        if end_prev is not None:
            key = f"{prev_name}->{name}"
            g = gaps.setdefault(key, [0, 0.0])
            g[0] += 1; g[1] += t0 - end_prev
        end_prev, prev_name = t0 + ms, name
        busy += ms
    span = tl[-1][1] + tl[-1][2] - tl[0][1]
    print("search rounds ms:", " ".join(f"{ms:.3f}" for name, t0, ms in tl if name == "chain_search_round"))
    print(f"span {span:.3f} ms, inside scopes {busy:.3f} ms, gaps {span - busy:.3f} ms over {len(tl)} scopes")
    for k, (c, g) in sorted(gaps.items(), key=lambda kv: -kv[1][1])[:25]:
        print(f"{k:55s} n={c:4d} gap {g:8.3f} ms ({1e3 * g / c:7.1f} us each)")


if __name__ == "__main__":
    {"scopes": cmd_scopes, "fallback": cmd_fallback, "timeline": cmd_timeline}[sys.argv[1]]()
