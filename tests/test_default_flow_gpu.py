"""ROCCO's default budgets and gamma on the device path: ``pipeline.run_shard`` with ``budgets`` / ``gammas`` None and
``pipeline.run_sample_sharded_defaults``.  Pinned to the hand composition of the existing pieces (scoring, budget null,
``_resolve_budgets``, ``_resolve_chrom_gamma``, the fixed-parameter ``run_shard``) and to their own one-rank result when
the chromosomes or the samples are spread over two ranks."""
import hashlib
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from rocco_b200.synth import chrom_matrix_numpy

pytestmark = pytest.mark.gpu

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GENOME = ["chrA", "chrB", "chrC", "chrD"]
SIZES = [60_001, 131_072, 250_000, 90_017]
SAMPLES = 10


def genome_matrices(samples=SAMPLES):
    """The synthetic genome as NumPy float64 matrices, in genome order."""
    return [chrom_matrix_numpy(samples, n, seed=101 + k) for k, n in enumerate(SIZES)]


def digest(mask) -> str:
    return hashlib.sha256(np.ascontiguousarray(mask).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def mats():
    import torch
    return [torch.from_numpy(x).cuda() for x in genome_matrices()]


def hand_composition(mats, names, genome, args, budgets=None, gammas=None):
    """score_loci_wls_device -> budget_null_device (resolved window) -> _resolve_budgets over the cache in genome order ->
    _resolve_chrom_gamma -> run_shard with those budgets and gammas."""
    from rocco_b200 import pipeline
    from rocco_b200.inference import _resolve_local_baseline_window
    from rocco_b200.rocco import _resolve_budgets, _resolve_chrom_gamma
    prm = pipeline.score_params(prior_df=6.0)
    full = pipeline._default_flow_args(args)
    nulls = {}
    for c, x in zip(names, mats):
        scores, extra = pipeline.score_loci_wls_device(x, params=prm, details=True)
        window = _resolve_local_baseline_window(x.shape[1], 101)
        assert window == extra["local_baseline_window"]
        _, nulls[c] = pipeline.budget_null_device(extra["centered_matrix"], scores, params=prm, dependence_lag_hint=window,
                                                  num_null_draws=full["num_null_draws"], random_seed=full["random_seed"])
    if budgets is None:
        cache = {c: {"budget_count_hat": nulls[c]["effective_count"], "total_count": nulls[c]["effective_total_count"]}
                 for c in genome}
        eb, _ = _resolve_budgets(cache, full)
        budgets = [eb[c] for c in names]
    if gammas is None:
        gammas = [_resolve_chrom_gamma(c, {"gamma": None}, None, nulls[c])[0] for c in names]
    out = pipeline.run_shard(mats, budgets, gammas, params=prm)
    return out, budgets, gammas, [nulls[c] for c in names]


@pytest.mark.parametrize("case", ["defaults", "target_scaled", "fixed_gamma", "explicit_budgets", "out_of_order"])
def test_one_rank_equals_the_hand_composition(mats, case):
    import torch
    from rocco_b200 import pipeline
    args = {"budget": 0.03, "scale_chrom_budgets": 1.25, "budget_posterior_quantile": 0.05} if case == "target_scaled" else {}
    names, use = list(GENOME), list(mats)
    if case == "out_of_order":
        order = [2, 0, 3, 1]
        names, use = [GENOME[k] for k in order], [mats[k] for k in order]
    budgets = [0.02, 0.03, 0.015, 0.04] if case == "explicit_budgets" else None
    gammas = [1.0, 2.5, 0.0, 6.0] if case == "fixed_gamma" else None
    want, want_b, want_g, want_nulls = hand_composition(use, names, GENOME, args, budgets, gammas)
    got = pipeline.run_shard(use, budgets, gammas, params=pipeline.score_params(prior_df=6.0), chrom_names=names,
                             genome_names=GENOME, default_args=args or None)
    assert got["budgets"] == want_b and got["gammas"] == want_g
    assert got["defaults"]["null"] == want_nulls                     # every key of every details dict, bit for bit
    assert torch.equal(got["d_scores"], want["d_scores"]) and torch.equal(got["d_masks"], want["d_masks"])
    assert got["results"] == want["results"]
    assert all(np.array_equal(a, b) for a, b in zip(got["runs"], want["runs"]))
    meta = got["defaults"]
    assert (meta["budget_meta"] is None) == (budgets is not None)
    assert all((m is None) == (gammas is not None) for m in meta["gamma_meta"])
    if gammas is None:
        assert [m["gamma_clipped"] for m in meta["gamma_meta"]] == got["gammas"]


def test_rejections(mats):
    from rocco_b200 import pipeline
    two = mats[:2]
    with pytest.raises(ValueError, match="genome_budget"):
        pipeline.run_shard(two, None, None, genome_budget=0.02)
    with pytest.raises(ValueError, match="genome_budget"):
        pipeline.run_shard(two, None, [1.0, 1.0], genome_budget=0.02, default_args={"num_null_draws": 8})
    with pytest.raises(ValueError, match="score_streams"):
        pipeline.run_shard(two, None, None, chrom_names=GENOME[:2], score_streams=2)
    with pytest.raises(ValueError, match="chrom_names"):
        pipeline.run_shard(two, None, None, chrom_names=GENOME[:3])
    with pytest.raises(ValueError, match="chrom_names"):
        pipeline.run_shard(two, None, None)
    with pytest.raises(ValueError, match="no rank holds"):
        pipeline.run_shard(two, None, None, chrom_names=GENOME[:2], genome_names=GENOME)
    for extra in ({"default_args": {"num_null_draws": 8}}, {"chrom_names": GENOME[:2]}, {"genome_names": GENOME},
                  {"mark": print}):
        with pytest.raises(ValueError, match="default flow"):                # explicit budgets and gammas: not ignored
            pipeline.run_shard(two, [0.02, 0.02], [1.0, 1.0], **extra)


def test_centered_out_matches_the_details(mats):
    import torch
    from rocco_b200 import pipeline
    x = mats[0]
    prm = pipeline.score_params(prior_df=6.0)
    s, extra = pipeline.score_loci_wls_device(x, params=prm, details=True)
    cent = torch.empty(tuple(x.shape), dtype=torch.float64, device=x.device)
    s2 = pipeline.score_loci_wls_device(x, params=prm, centered_out=cent)
    assert torch.equal(s, s2) and torch.equal(cent, extra["centered_matrix"])
    with pytest.raises(ValueError):
        pipeline.score_loci_wls_device(x, params=prm, centered_out=cent[:, 1:])


# ------------------------------------------------------------------ chromosomes over two ranks
WORKER = r'''
import hashlib, json, os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["ROCCO_B200_REPO"])
sys.path.insert(0, os.environ["ROCCO_B200_TESTS"])
from rocco_b200 import pipeline, distributed as rdist
from test_default_flow_gpu import GENOME, genome_matrices, digest

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
backend = os.environ["ROCCO_B200_BACKEND"]
local = int(os.environ["LOCAL_RANK"]) % torch.cuda.device_count()     # gloo: both ranks may share one device
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
tmp = os.environ["ROCCO_B200_TMP"]
prm = pipeline.score_params(prior_df=6.0)
mats = [torch.from_numpy(x).to(dev) for x in genome_matrices()]
lex = sorted(GENOME)

def summary(out, names, bed):
    return {"budgets": dict(zip(names, out["budgets"])), "gammas": dict(zip(names, out["gammas"])),
            "masks": {c: digest(out["d_masks"][o:o + n].cpu().numpy()) for c, o, n in zip(names, out["offsets"], out["lengths"])},
            "bed": hashlib.sha256(open(bed, "rb").read()).hexdigest() if bed else None}

# the one-rank run of the whole genome, before the process group exists
whole = pipeline.run_shard(mats, None, None, params=prm, chrom_names=GENOME)
bed = os.path.join(tmp, f"whole_{rank}.bed")
rdist.write_genome_bed(bed, lex, GENOME, whole["runs"], 50)
result = {"rank": rank, "whole": summary(whole, GENOME, bed)}
if backend == "nccl":
    dist.init_process_group("nccl", device_id=dev)
else:
    dist.init_process_group("gloo")
splits = {"uneven": (["chrC"], ["chrD", "chrA", "chrB"]), "empty_rank": ([], GENOME[::-1])}
for name, parts in splits.items():
    mine = parts[rank]
    out = pipeline.run_shard([mats[GENOME.index(c)] for c in mine], None, None, params=prm, chrom_names=mine,
                             genome_names=GENOME)
    bed = os.path.join(tmp, f"{name}.bed")
    rdist.write_genome_bed(bed, lex, mine, out["runs"], 50, device=dev if backend == "nccl" else None)
    torch.cuda.synchronize()
    dist.barrier()
    result[name] = summary(out, mine, bed)
    dist.barrier()
bad = [mats[GENOME.index(c)].clone() for c in splits["uneven"][rank]]
if rank == 1:
    bad[1][3, 777] = float("nan")
try:
    pipeline.run_shard(bad, None, None, params=prm, chrom_names=splits["uneven"][rank], genome_names=GENOME)
    result["nonfinite"] = "no error"
except ValueError as exc:
    result["nonfinite"] = str(exc)
sys.stdout.write("RESULT " + json.dumps(result) + "\n")
sys.stdout.flush()
dist.destroy_process_group()
'''


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _torchrun(tmp_path, script_text, env_extra, timeout=900):
    script = tmp_path / "worker.py"
    script.write_text(script_text)
    env = dict(os.environ, ROCCO_B200_REPO=REPO, ROCCO_B200_TESTS=os.path.join(REPO, "tests"), ROCCO_B200_TMP=str(tmp_path),
               **env_extra)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), str(script)]
    res = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=timeout)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    rows = sorted((json.loads(ln.split("RESULT ", 1)[1]) for ln in res.stdout.splitlines() if "RESULT " in ln),
                  key=lambda r: r["rank"])
    assert len(rows) == 2
    return rows


@pytest.mark.parametrize("backend", ["nccl", "gloo"])
def test_two_ranks_equal_one_rank(tmp_path, backend):
    """nccl: one GPU per rank; gloo: both ranks allowed on one GPU, the gather going through the host."""
    import torch
    if backend == "nccl" and torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    rows = _torchrun(tmp_path, WORKER, {"ROCCO_B200_BACKEND": backend})
    whole = rows[0]["whole"]
    assert rows[1]["whole"] == whole
    for name in ("uneven", "empty_rank"):
        merged = {k: {} for k in ("budgets", "gammas", "masks")}
        for r in rows:
            for k in merged:
                merged[k].update(r[name][k])
        for k in merged:
            assert merged[k] == whole[k], (name, k)
        assert rows[0][name]["bed"] == whole["bed"], name
    assert "another rank" in rows[0]["nonfinite"], rows[0]["nonfinite"]
    assert "chrA" in rows[1]["nonfinite"] and "another rank" not in rows[1]["nonfinite"], rows[1]["nonfinite"]


# ------------------------------------------------------------------ samples over ranks
def test_sample_sharded_one_process_equals_the_hand_composition(mats):
    import torch
    from rocco_b200 import pipeline
    from rocco_b200.rocco import _resolve_budgets, _resolve_chrom_gamma
    prm = pipeline.score_params(prior_df=6.0)
    got = pipeline.run_sample_sharded_defaults(iter(zip(GENOME, mats)), SAMPLES, prm)
    nulls, scores = {}, []
    for c, x in zip(GENOME, mats):
        s, cent, window = pipeline.score_loci_wls_sample_sharded(x, SAMPLES, prm, keep_centered=True)
        _, nulls[c] = pipeline.budget_null_sample_sharded(cent, s, params=prm, dependence_lag_hint=window)
        scores.append(s)
    budgets, meta = _resolve_budgets({c: {"budget_count_hat": nulls[c]["effective_count"],
                                          "total_count": nulls[c]["effective_total_count"]} for c in GENOME},
                                     pipeline.DEFAULT_FLOW_ARGS)
    gammas = {c: _resolve_chrom_gamma(c, {"gamma": None}, None, nulls[c])[0] for c in GENOME}
    assert got["defaults"]["null"] == nulls and got["budgets"] == budgets and got["gammas"] == gammas
    assert got["defaults"]["budget_meta"] == meta
    assert got["my_names"] == GENOME
    res = pipeline.solve_chromosomes(scores, [budgets[c] for c in GENOME], [gammas[c] for c in GENOME])
    for r, want, o, n in zip(got["results"], res, got["offsets"], SIZES):
        assert np.array_equal(got["d_masks"][o:o + n].cpu().numpy(), want.pop("solution"))
        assert r == want


SAMPLE_WORKER = r'''
import json, os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["ROCCO_B200_REPO"])
sys.path.insert(0, os.environ["ROCCO_B200_TESTS"])
from rocco_b200 import pipeline
from test_default_flow_gpu import GENOME, SAMPLES, genome_matrices, digest

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
backend = os.environ["ROCCO_B200_BACKEND"]
local = int(os.environ["LOCAL_RANK"]) % torch.cuda.device_count()     # gloo: both ranks may share one device
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
prm = pipeline.score_params(prior_df=6.0)
xs = genome_matrices()
# the unsharded flow on the same samples, before the process group exists
whole = pipeline.run_shard([torch.from_numpy(x).to(dev) for x in xs], None, None, params=prm, chrom_names=GENOME)
if backend == "nccl":
    dist.init_process_group("nccl", device_id=dev)
else:
    dist.init_process_group("gloo")
lo, hi = (0, 4) if rank == 0 else (4, SAMPLES)
out = pipeline.run_sample_sharded_defaults(((c, torch.from_numpy(x[lo:hi]).to(dev)) for c, x in zip(GENOME, xs)), SAMPLES, prm)
# a NaN in rank 1's rows of the second chromosome: the scoring fails there, before the accumulator all-reduce
def poisoned():
    for k, (c, x) in enumerate(zip(GENOME, xs)):
        rows = torch.from_numpy(x[lo:hi]).to(dev)
        if rank == 1 and k == 1:
            rows[0, 99] = float("nan")
        yield c, rows
try:
    pipeline.run_sample_sharded_defaults(poisoned(), SAMPLES, prm)
    nonfinite = "no error"
except ValueError as exc:
    nonfinite = str(exc)
result = {"rank": rank, "nonfinite": nonfinite, "budgets": out["budgets"], "gammas": out["gammas"], "null": out["defaults"]["null"],
          "masks": {c: digest(out["d_masks"][o:o + n].cpu().numpy()) for c, o, n in
                    zip(out["my_names"], out["offsets"], [out["lengths"][GENOME.index(c)] for c in out["my_names"]])},
          "whole": {"budgets": dict(zip(GENOME, whole["budgets"])), "gammas": dict(zip(GENOME, whole["gammas"])),
                    "null": dict(zip(GENOME, whole["defaults"]["null"])),
                    "masks": {c: digest(whole["d_masks"][o:o + n].cpu().numpy())
                              for c, o, n in zip(GENOME, whole["offsets"], whole["lengths"])}}}
sys.stdout.write("RESULT " + json.dumps(result) + "\n")
sys.stdout.flush()
dist.destroy_process_group()
'''


@pytest.mark.parametrize("backend", ["nccl", "gloo"])
def test_sample_sharded_two_ranks(tmp_path, backend):
    """nccl: one GPU per rank; gloo: both ranks allowed on one GPU, the collectives going through the host."""
    import torch
    if backend == "nccl" and torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from rocco_b200.pipeline import target_count_for_budget
    from tests.test_budget_sharded_gpu import SHARD_REL_TOL, assert_close_details
    rows = _torchrun(tmp_path, SAMPLE_WORKER, {"ROCCO_B200_BACKEND": backend})
    for k in ("budgets", "gammas", "null"):
        assert rows[0][k] == rows[1][k], k
    whole = rows[0]["whole"]
    masks = {**rows[0]["masks"], **rows[1]["masks"]}
    assert sorted(masks) == sorted(GENOME)
    for c, n in zip(GENOME, SIZES):
        assert_close_details(rows[0]["null"][c], whole["null"][c], n, what=c)
        for k in ("budgets", "gammas"):
            assert abs(rows[0][k][c] - whole[k][c]) <= SHARD_REL_TOL * abs(whole[k][c]), (c, k, rows[0][k][c], whole[k][c])
        if target_count_for_budget(n, rows[0]["budgets"][c]) == target_count_for_budget(n, whole["budgets"][c]):
            assert masks[c] == whole["masks"][c], c
    assert "chrB" in rows[1]["nonfinite"] and "another rank" not in rows[1]["nonfinite"], rows[1]["nonfinite"]
    assert "chrB failed on another rank" in rows[0]["nonfinite"], rows[0]["nonfinite"]
