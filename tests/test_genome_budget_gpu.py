"""Genome-wide budget: one multiplier searched over every chromosome (pipeline.solve_genome / rocco_b200_chain_solve_genome_dev).

The oracle below is the definition itself: the reference's search (dp.py:89-164) on the CONCATENATED chain S = s_1 || s_2 ..,
C = c_1 || 0 || c_2 || 0 .., with the bracket built from the correctly rounded sum of C, solved by
oracle.solve_penalized_chain on the whole concatenation.  That the chromosomes decouple at zero-cost junctions is therefore
tested here, not assumed.
"""
import json
import math
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZES = [1, 2, 257, 4096, 4097, 70_001, 300_001]
GAMMAS = [0.0, 1.0, 6.86]


def _scores(n, seed, peak_frac=0.03):
    rng = np.random.default_rng(seed)
    return rng.normal(size=n) - 0.8 + 4.0 * (rng.random(n) < peak_frac) * rng.random(n)


def _genome(seed=0):
    scores = [_scores(n, seed * 100 + k) for k, n in enumerate(SIZES)]
    gammas = [GAMMAS[k % len(GAMMAS)] for k in range(len(SIZES))]
    return scores, gammas


def _kind(orc):
    return "reference" if orc.reference_available() else "port"


def oracle_genome(orc, scores, costs, budget, max_iter=60):
    """(lambda, per-chromosome masks, genome count, DP passes) of the definition."""
    s = np.concatenate(scores)
    c = np.concatenate([np.append(np.asarray(x, dtype=np.float64), 0.0) for x in costs])[:-1]
    n = s.shape[0]
    kind = _kind(orc)
    target = int(max(0, min(int(np.floor(n * float(budget))), n)))
    passes = 0

    def run(lam):
        nonlocal passes
        passes += 1
        return orc.solve_penalized_chain(s, c, lam, kind=kind)

    if target == n:
        sol, _, cnt = run(0.0)
    else:
        csum = math.fsum(c.tolist())
        lo = float(np.min(s) - csum - 1.0)
        hi = float(np.max(s) + csum + 1.0)
        cnt_lo = run(lo)[2]
        while cnt_lo <= target:
            lo -= max(1.0, abs(lo))
            cnt_lo = run(lo)[2]
        best = run(hi)
        while best[2] > target:
            hi += max(1.0, abs(hi))
            best = run(hi)
        for _ in range(max_iter):
            mid = (lo + hi) / 2.0
            got = run(mid)
            if got[2] > target:
                lo = mid
            else:
                hi, best = mid, got
        sol, cnt = best[0], best[2]
    lam = 0.0 if target == n else hi
    bounds = np.cumsum([0] + [len(x) for x in scores])
    return lam, [sol[bounds[k]:bounds[k + 1]] for k in range(len(scores))], int(cnt), passes, target


@pytest.fixture(scope="module")
def pipeline():
    from rocco_b200 import pipeline
    return pipeline


def _costs_of(scores, gammas):
    return [np.full(max(len(s) - 1, 0), g) for s, g in zip(scores, gammas)]


def _check_against_oracle(orc, scores, costs, budget, masks, genome, results):
    lam, want, cnt, passes, target = oracle_genome(orc, scores, costs, budget)
    for k, (m, w) in enumerate(zip(masks, want)):
        assert np.array_equal(m, w), (budget, k, len(w), int(np.sum(m != w)))
    assert genome["selected_count"] == cnt and cnt <= target
    assert genome["selected_count"] == sum(r["selected_count"] for r in results)
    assert genome["target_count"] == target
    assert abs(genome["selection_penalty"] - lam) <= 1e-9, (genome["selection_penalty"], lam)
    assert genome["dp_passes"] == passes
    for s, c, w, r in zip(scores, costs, want, results):
        obj = orc.objective_value(w, s, c)
        assert abs(r["objective"] - obj) <= 1e-6 * max(1.0, abs(obj))
        assert r["selection_penalty"] == genome["selection_penalty"]
    return lam


@pytest.mark.parametrize("budget", [0.0, 0.02, 0.3, 1.0])
def test_mixed_genome_matches_concatenated_oracle(pipeline, oracle, budget):
    scores, gammas = _genome(seed=1)
    masks, genome, results = pipeline.solve_genome(scores, budget, gammas)
    _check_against_oracle(oracle, scores, _costs_of(scores, gammas), budget, masks, genome, results)
    if budget < 1.0:
        assert genome["dp_passes"] == 62
        # every chromosome solved at the returned multiplier by the fixed-multiplier path: the same masks
        fixed = pipeline.solve_chromosomes(scores, [None] * len(scores), gammas,
                                           selection_penalties=[genome["selection_penalty"]] * len(scores))
        for m, r in zip(masks, fixed):
            assert np.array_equal(m, r["solution"])


def test_vector_costs_genome_matches_concatenated_oracle(pipeline, oracle):
    scores, _ = _genome(seed=2)
    rng = np.random.default_rng(9)
    costs = [rng.uniform(0.0, 2.5, size=max(len(s) - 1, 0)) for s in scores]
    masks, genome, results = pipeline.solve_genome(scores, 0.02, None, switch_costs_list=costs)
    _check_against_oracle(oracle, scores, costs, 0.02, masks, genome, results)
    assert genome["dp_passes"] == 62


def test_identical_bits_across_depths_freezing_and_runs(pipeline):
    from rocco_b200 import _lib
    scores, gammas = _genome(seed=3)
    base = pipeline.solve_genome(scores, 0.02, gammas)

    def same(got):
        assert got[1]["selection_penalty"] == base[1]["selection_penalty"]
        assert got[1]["selected_count"] == base[1]["selected_count"]
        for a, b in zip(got[0], base[0]):
            assert np.array_equal(a, b)
        for a, b in zip(got[2], base[2]):
            assert {k: v for k, v in a.items() if k != "search_rounds"} == {k: v for k, v in b.items() if k != "search_rounds"}

    same(pipeline.solve_genome(scores, 0.02, gammas))
    for levels in (1, 2, 3, 4):
        same(pipeline.solve_genome(scores, 0.02, gammas, levels_per_round=levels))
    prev = _lib.load().rocco_b200_chain_set_tile_freezing(0)
    try:
        same(pipeline.solve_genome(scores, 0.02, gammas))
    finally:
        _lib.load().rocco_b200_chain_set_tile_freezing(prev)


def test_one_chromosome_genome_equals_per_chromosome_search(pipeline):
    s = _scores(70_001, seed=44)
    masks, genome, _ = pipeline.solve_genome([s], 0.02, [1.0])
    ref = pipeline.solve_chromosomes([s], [0.02], [1.0])[0]
    assert np.array_equal(masks[0], ref["solution"])
    assert genome["selected_count"] == ref["selected_count"]
    assert abs(genome["selection_penalty"] - ref["selection_penalty"]) <= 1e-9


def test_rejections(pipeline):
    from rocco_b200 import _lib
    s = _scores(5000, seed=3)
    prev = _lib.load().rocco_b200_chain_set_exact_search(1)
    try:
        with pytest.raises(ValueError):
            pipeline.solve_genome([s], 0.02, [1.0])
    finally:
        _lib.load().rocco_b200_chain_set_exact_search(prev)
    with pytest.raises(ValueError):
        pipeline.solve_genome([], 0.02, [])
    with pytest.raises(ValueError):
        pipeline.solve_genome([s, np.zeros(0)], 0.02, [1.0, 1.0])
    with pytest.raises(ValueError):
        pipeline.solve_genome([s], 0.02, [-1.0])
    bad = s.copy()
    bad[17] = np.nan
    with pytest.raises(ValueError):
        pipeline.solve_genome([bad], 0.02, [1.0])


def test_run_shard_genome_budget(pipeline):
    import torch
    from rocco_b200.synth import chrom_matrix_numpy
    mats = [torch.from_numpy(chrom_matrix_numpy(6, n, seed=n)).cuda() for n in (9000, 30_000)]
    with pytest.raises(ValueError):
        pipeline.run_shard(mats, [0.02, 0.02], [1.0, 1.0], genome_budget=0.02)
    out = pipeline.run_shard(mats, None, [1.0, 1.0], genome_budget=0.02)
    scores = [out["d_scores"][o:o + n].cpu().numpy() for o, n in zip(out["offsets"], out["lengths"])]
    masks, genome, _ = pipeline.solve_genome(scores, 0.02, [1.0, 1.0])
    assert out["genome"] == genome
    for m, o, n in zip(masks, out["offsets"], out["lengths"]):
        assert np.array_equal(out["d_masks"][o:o + n].cpu().numpy(), m)


# ------------------------------------------------------------------ two ranks
WORKER = r'''
import hashlib, json, os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["ROCCO_B200_REPO"])
sys.path.insert(0, os.environ["ROCCO_B200_TESTS"])
from rocco_b200 import pipeline
from test_genome_budget_gpu import _genome

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
backend = os.environ["ROCCO_B200_BACKEND"]
local = int(os.environ["LOCAL_RANK"]) % torch.cuda.device_count()     # gloo: both ranks may share one device
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
scores, gammas = _genome(seed=5)
# single-process run of the whole genome, before the process group exists
whole = pipeline.solve_genome(scores, 0.02, gammas)
if backend == "nccl":
    dist.init_process_group("nccl", device_id=dev)
else:
    dist.init_process_group("gloo")

def digest(masks):
    return hashlib.sha256(b"".join(m.tobytes() for m in masks)).hexdigest()

out = {"rank": rank}
small = [k for k, s in enumerate(scores) if len(s) <= 4096]
large = [k for k in range(len(scores)) if k not in small]
for name, mine in (("uneven", small if rank == 0 else large), ("empty_rank", [] if rank == 0 else list(range(len(scores))))):
    masks, genome, res = pipeline.solve_genome([scores[k] for k in mine], 0.02, [gammas[k] for k in mine])
    out[name] = {"lam": float(genome["selection_penalty"]).hex(), "count": genome["selected_count"],
                 "counts": [r["selected_count"] for r in res],
                 "masks_equal_whole": all(np.array_equal(m, whole[0][k]) for m, k in zip(masks, mine)),
                 "whole_counts": [whole[2][k]["selected_count"] for k in mine]}
out["whole"] = {"lam": float(whole[1]["selection_penalty"]).hex(), "count": whole[1]["selected_count"]}
bad = [scores[k].copy() for k in (small if rank == 0 else large)]
if rank == 1:
    bad[0][5] = np.nan
try:
    pipeline.solve_genome(bad, 0.02, [gammas[k] for k in (small if rank == 0 else large)])
    out["nonfinite"] = "no error"
except ValueError as exc:
    out["nonfinite"] = "ValueError"
# one write of the whole line (well under PIPE_BUF): print() writes the text and the newline separately, so the two
# ranks' lines could interleave on the shared pipe
sys.stdout.write("RESULT " + json.dumps(out) + "\n")
sys.stdout.flush()
dist.destroy_process_group()
'''


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("backend", ["nccl", "gloo"])
def test_two_rank_genome_budget(tmp_path, backend):
    """nccl: one GPU per rank; gloo: the same protocol with both ranks allowed on one GPU (CUDA tensors reduced through
    the host), so the sharded search is also exercised where only one GPU is visible."""
    import torch
    if backend == "nccl" and torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, ROCCO_B200_REPO=REPO, ROCCO_B200_TESTS=os.path.join(REPO, "tests"), ROCCO_B200_BACKEND=backend)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), str(script)]
    res = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    rows = [json.loads(ln.split("RESULT ", 1)[1]) for ln in res.stdout.splitlines() if "RESULT " in ln]
    assert len(rows) == 2
    for r in rows:
        for name in ("uneven", "empty_rank"):
            got = r[name]
            assert got["lam"] == r["whole"]["lam"] and got["count"] == r["whole"]["count"], (name, r)
            assert got["masks_equal_whole"] and got["counts"] == got["whole_counts"], (name, r)
        assert r["nonfinite"] == "ValueError", r
    assert rows[0]["whole"] == rows[1]["whole"]
