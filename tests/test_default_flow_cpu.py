"""World-size-2 gloo test (CPU) of the default flow's agreement step: ``pipeline.agree_chromosome_names`` and
``pipeline.gather_budget_estimates`` with plain numbers in place of the budget null's estimates.  Chromosomes split over
the ranks and listed out of genome order must give every rank the genome-ordered cache of one process, and every
rejection must reach both ranks."""
import json
import os
import socket

import numpy as np
import pytest

GENOME = ["chr1", "chr2", "chr10", "chrX", "chr21", "chr19"]
ARGS = {"budget": None, "scale_chrom_budgets": 1.0, "budget_posterior_quantile": 0.01}


def _estimates():
    """(effective_count, effective_total_count) per chromosome: dispersed rates, so the EB fit is the beta-binomial MLE."""
    rng = np.random.default_rng(31)
    totals = rng.integers(300_000, 2_000_000, size=len(GENOME)).astype(np.float64)
    counts = np.round(totals * rng.uniform(0.01, 0.05, size=len(GENOME)) * 8.0) / 8.0
    return {c: (float(k), float(t)) for c, k, t in zip(GENOME, counts, totals)}


def _single_process_cache():
    est = _estimates()
    return {c: {"budget_count_hat": est[c][0], "total_count": est[c][1]} for c in GENOME}


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _attempt(fn):
    try:
        return {"ok": fn()}
    except ValueError as exc:
        return {"error": str(exc)}


def _worker(rank, size, port, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=size)
    try:
        from rocco_b200 import pipeline
        from rocco_b200.rocco import _resolve_budgets
        est = _estimates()

        def flow(mine, genome=GENOME, status=None, failure=None, agreed=None, problem=None):
            slots = pipeline.agree_chromosome_names(mine, genome, problem=problem, agreed=agreed)
            rows = [est[c] + ((status or {}).get(c, 0),) for c in mine]
            cache = pipeline.gather_budget_estimates(mine, genome, rows, slots, failure=failure)
            budgets, meta = _resolve_budgets(cache, ARGS)
            return {"cache": list(cache.items()), "budgets": list(budgets.items()), "alpha": meta["alpha"]}

        out = {}
        # uneven split, each rank's list out of genome order
        out["uneven"] = _attempt(lambda: flow(["chrX", "chr1"] if rank == 0 else ["chr19", "chr21", "chr10", "chr2"]))
        # one rank holds nothing
        out["empty_rank"] = _attempt(lambda: flow([] if rank == 0 else GENOME[::-1]))
        # a failed chromosome on rank 1
        out["status"] = _attempt(lambda: flow(["chr1", "chr2", "chr10"] if rank == 0 else ["chrX", "chr21", "chr19"],
                                              status={"chr21": 1} if rank == 1 else None,
                                              failure="chr21: boom" if rank == 1 else None))
        # a failure on a rank that holds no chromosome (its own status row carries it)
        out["empty_rank_failure"] = _attempt(lambda: flow([] if rank == 0 else GENOME,
                                                          failure="setup boom" if rank == 0 else None))
        # names: unknown, duplicate, unowned, differing genome lists, disagreeing arguments, a rank-local problem
        halves = (GENOME[:3], GENOME[3:])
        out["unknown"] = _attempt(lambda: flow(halves[rank] + (["chrZ"] if rank == 0 else [])))
        out["duplicate"] = _attempt(lambda: flow(halves[rank] + (["chr1"] if rank == 1 else [])))
        out["unowned"] = _attempt(lambda: flow(halves[rank] if rank == 0 else ["chrX", "chr19"]))
        out["duplicate_in_genome"] = _attempt(lambda: flow(halves[rank], genome=GENOME + ["chr2"]))
        out["genome_differs"] = _attempt(lambda: flow(halves[rank], genome=GENOME if rank == 0 else GENOME[::-1]))
        out["agreed_differs"] = _attempt(lambda: flow(halves[rank], agreed=("draws", 25 if rank == 0 else 8)))
        out["problem"] = _attempt(lambda: flow(halves[rank], problem="bad local argument" if rank == 0 else None))
        # the group still works after every rejection: the next collective pairs up
        out["after"] = _attempt(lambda: flow(halves[rank]))
        with open(os.path.join(out_dir, f"rank{rank}.json"), "w") as fh:
            json.dump(out, fh)
    finally:
        dist.destroy_process_group()


@pytest.fixture(scope="module")
def two_ranks(tmp_path_factory):
    import torch.multiprocessing as mp
    out = tmp_path_factory.mktemp("default_flow")
    mp.spawn(_worker, args=(2, _free_port(), str(out)), nprocs=2, join=True)
    return [json.load(open(out / f"rank{r}.json")) for r in range(2)]


def _single_process_result():
    from rocco_b200.rocco import _resolve_budgets
    cache = _single_process_cache()
    budgets, meta = _resolve_budgets(cache, ARGS)
    return {"cache": [list(kv) for kv in cache.items()], "budgets": [list(kv) for kv in budgets.items()], "alpha": meta["alpha"]}


@pytest.mark.parametrize("case", ["uneven", "empty_rank", "after"])
def test_both_ranks_get_the_single_process_cache_and_budgets(two_ranks, case):
    want = _single_process_result()
    for r in two_ranks:
        assert r[case] == {"ok": want}, (case, r[case])       # genome order, and the same doubles


def test_a_status_on_one_rank_raises_on_both(two_ranks):
    assert two_ranks[1]["status"] == {"error": "chr21: boom"}
    assert "chr21" in two_ranks[0]["status"]["error"] and "another rank" in two_ranks[0]["status"]["error"]
    assert two_ranks[0]["empty_rank_failure"] == {"error": "setup boom"}
    assert "another rank" in two_ranks[1]["empty_rank_failure"]["error"]


@pytest.mark.parametrize("case,text", [("unknown", "missing from `genome_names`"), ("duplicate", "more than once"),
                                       ("unowned", "no rank holds"), ("duplicate_in_genome", "more than once"),
                                       ("genome_differs", "same `genome_names`"), ("agreed_differs", "same default")])
def test_name_problems_raise_the_same_error_on_both_ranks(two_ranks, case, text):
    errors = [r[case].get("error") for r in two_ranks]
    assert errors[0] is not None and errors[0] == errors[1], (case, errors)
    assert text in errors[0], (case, errors[0])


def test_a_local_problem_reaches_the_other_rank(two_ranks):
    assert two_ranks[0]["problem"] == {"error": "bad local argument"}
    assert "another rank" in two_ranks[1]["problem"]["error"] and "bad local argument" in two_ranks[1]["problem"]["error"]


def test_one_process():
    """Without a process group the helpers run the same checks and build the same cache."""
    from rocco_b200 import pipeline
    est = _estimates()
    mine = GENOME[::-1]
    slots = pipeline.agree_chromosome_names(mine, GENOME)
    assert slots == len(GENOME)
    cache = pipeline.gather_budget_estimates(mine, GENOME, [est[c] + (0,) for c in mine], slots)
    assert list(cache.items()) == list(_single_process_cache().items())
    with pytest.raises(ValueError, match="no rank holds"):
        pipeline.agree_chromosome_names(GENOME[1:], GENOME)
    with pytest.raises(ValueError, match="missing"):
        pipeline.agree_chromosome_names(GENOME + ["chrZ"], GENOME)
    with pytest.raises(ValueError, match="boom"):
        pipeline.gather_budget_estimates(mine, GENOME, [est[c] + (0,) for c in mine], slots, failure="boom")
    with pytest.raises(ValueError, match="failed"):
        pipeline.gather_budget_estimates(mine, GENOME, [est[c] + (int(c == "chr2"),) for c in mine], slots)
    with pytest.raises(ValueError, match="unknown `default_args`"):
        pipeline._default_flow_args({"gamma": 1.0})
