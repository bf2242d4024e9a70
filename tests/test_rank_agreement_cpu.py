"""Cross-rank plumbing of ``rocco_b200.distributed`` on a world-size-2 gloo group (CPU): ``agree``, ``world`` and
``collective_device``; and the builders of the native parameter structs against the library's own defaults."""
import ctypes
import json
import os
import socket

import pytest


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
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=size)
    try:
        from rocco_b200 import distributed as rd
        singles = [dist.new_group([0]), dist.new_group([1])]
        out = {"world": list(rd.world()), "world_group": list(rd.world(dist.group.WORLD)),
               "world_single": list(rd.world(singles[rank])),
               "device": str(rd.collective_device(None)), "device_given": str(rd.collective_device(None, torch.device("cuda", 0)))}
        # facts of different sizes per rank come back in rank order
        out["facts"] = _attempt(lambda: rd.agree(None, {"rank": rank, "items": list(range(rank + 2))}, None, "test"))
        out["problem"] = _attempt(lambda: rd.agree("bad thing on rank 1" if rank == 1 else None, {"rank": rank}, None, "test"))
        # a one-rank group: no collective, whatever the other rank does
        out["single"] = _attempt(lambda: rd.agree(None, {"rank": rank}, singles[rank], "test"))
        # the group still pairs up after a rejection
        out["after"] = _attempt(lambda: rd.agree(None, {"rank": rank}, None, "test"))
        with open(os.path.join(out_dir, f"rank{rank}.json"), "w") as fh:
            json.dump(out, fh)
    finally:
        dist.destroy_process_group()


@pytest.fixture(scope="module")
def two_ranks(tmp_path_factory):
    import torch.multiprocessing as mp
    out = tmp_path_factory.mktemp("rank_agreement")
    mp.spawn(_worker, args=(2, _free_port(), str(out)), nprocs=2, join=True)
    return [json.load(open(out / f"rank{r}.json")) for r in range(2)]


def test_world_with_a_group(two_ranks):
    for rank, r in enumerate(two_ranks):
        assert r["world"] == [rank, 2] and r["world_group"] == [rank, 2]
        assert r["world_single"] == [0, 1]


def test_collective_device_is_the_cpu_on_gloo(two_ranks):
    for r in two_ranks:
        assert r["device"] == "cpu" and r["device_given"] == "cpu"


def test_agree_returns_the_facts_in_rank_order(two_ranks):
    want = [{"rank": 0, "items": [0, 1]}, {"rank": 1, "items": [0, 1, 2]}]
    for r in two_ranks:
        assert r["facts"] == {"ok": want}
        assert r["after"] == {"ok": [{"rank": 0}, {"rank": 1}]}
    assert two_ranks[0]["single"] == {"ok": [{"rank": 0}]} and two_ranks[1]["single"] == {"ok": [{"rank": 1}]}


def test_a_problem_raises_on_both_ranks(two_ranks):
    assert two_ranks[1]["problem"] == {"error": "bad thing on rank 1"}
    assert two_ranks[0]["problem"] == {"error": "test: another rank rejected its arguments: bad thing on rank 1"}


def test_one_process_runs_no_collective(monkeypatch):
    import torch.distributed as dist
    from rocco_b200 import distributed as rd

    def no_collective(*args, **kwargs):
        raise AssertionError("a collective ran")

    monkeypatch.setattr(dist, "all_gather_object", no_collective)
    assert rd.world() == (0, 1)
    assert rd.agree(None, {"x": 1}, None, "test") == [{"x": 1}]
    with pytest.raises(ValueError, match="^mine$"):
        rd.agree("mine", {"x": 1}, None, "test")


# ------------------------------------------------------------------ parameter builders
def test_default_builders_give_the_library_defaults():
    from rocco_b200 import _lib, pipeline
    from rocco_b200.inference import budget_params
    score = _lib.ScoreParams()
    _lib.load().rocco_b200_default_score_params(ctypes.byref(score))
    assert bytes(pipeline.score_params()) == bytes(score)
    budget = _lib.BudgetParams()
    _lib.load().rocco_b200_default_budget_params(ctypes.byref(budget))
    assert bytes(budget_params(pipeline.score_params())) == bytes(budget)


def test_budget_params_fields():
    import torch
    from rocco_b200 import pipeline
    from rocco_b200.inference import budget_params
    inn = torch.zeros(4, dtype=torch.float64)
    prm = budget_params(pipeline.score_params(prior_df=6.0, min_effect=0.5), dependence_lag_hint=-3, num_null_draws=0,
                        min_null_draws=0, stability_abs_tol=1e-3, stability_rel_tol=2e-2, random_seed=-1,
                        sample_offset=7, d_innovations=inn)
    assert prm.score.prior_df == 6.0 and prm.score.use_min_effect == 1 and prm.score.min_effect == 0.5
    assert prm.dependence_lag_hint == 1 and prm.num_null_draws == 1 and prm.min_null_draws == 1
    assert prm.stability_abs_tol == 1e-3 and prm.stability_rel_tol == 2e-2
    assert prm.random_seed == 2**64 - 1 and prm.random_streams == 0
    assert prm.sample_offset == 7 and prm.d_innovations == inn.data_ptr()
    prm = budget_params(pipeline.score_params(), dependence_lag_hint=40, random_seed=2**64 + 3)
    assert prm.dependence_lag_hint == 40 and prm.random_seed == 3
    assert prm.sample_offset == 0 and prm.d_innovations is None
    assert budget_params(pipeline.score_params(), random_seed=9, random_streams="numpy").random_streams == 1
    with pytest.raises(ValueError):
        budget_params(pipeline.score_params(), random_streams="numpy", d_innovations=inn)
    with pytest.raises(ValueError):
        budget_params(pipeline.score_params(), random_streams="pcg")
