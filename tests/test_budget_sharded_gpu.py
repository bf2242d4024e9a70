"""Budget null with the samples sharded over ranks (pipeline.budget_null_sample_sharded, the config-5 layout).

Most of the evidence comes from one GPU: the sharded C entry is driven from host threads, one per emulated rank, each on
its own stream, with an in-process reducer (a threading.Barrier that synchronises the streams and sums the buffers).  A
protocol mistake -- a rank that leaves while the other still waits in a reduce -- then shows up as a barrier timeout on
the host, never as a stuck collective.  The NCCL test at the end runs two real ranks when two GPUs are visible.
"""
import json
import os
import socket
import subprocess
import sys
import threading

import numpy as np
import pytest

from rocco_b200.synth import chrom_matrix_numpy

pytestmark = pytest.mark.gpu

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INDICATOR_KEYS = {"observed_positive_fraction", "observed_negative_fraction", "null_positive_fraction",
                  "observed_tail_occupancy", "null_tail_occupancy", "nonnull_fraction", "negative_fraction"}
COUNT_KEYS = {"negative_support_size", "effective_count", "positive_score_count"}
SHARD_REL_TOL = 1e-9          # sharded vs unsharded: the column sums are added in another order (~1e-16 relative)


def reference_innovations(seed, draws, m, n, taps):
    """The reference's own streams (inference.py:653-662): default_rng(seed + 104729 (draw + 1)), samples in order."""
    out = np.empty((draws, m, n + taps - 1))
    for d in range(draws):
        rng = np.random.default_rng(int(seed) + 104729 * (d + 1))
        for i in range(m):
            out[d, i] = rng.standard_normal(n + taps - 1)
    return out


def assert_close_details(got, want, n, rel=SHARD_REL_TOL, what=""):
    assert set(got) == set(want), what
    for k, v in want.items():
        if isinstance(v, (str, bool)):
            assert got[k] == v, (what, k)
        elif k in INDICATOR_KEYS:
            assert abs(got[k] - v) <= 2.0 / n + 1e-12, (what, k, got[k], v)
        elif k in COUNT_KEYS:
            assert abs(got[k] - v) <= 2.0 + rel * abs(v), (what, k, got[k], v)
        else:
            assert abs(got[k] - v) <= rel * max(1.0, abs(v)), (what, k, got[k], v)


def run_shards(parts, **kw):
    """Run pipeline._budget_null_sharded for every (rows, sample_offset, innovations) of `parts` from its own host thread
    and stream, summing the reduce buffers in process.  Returns per shard ("ok", (fraction, details)) or
    ("err", exception, last_error text)."""
    import torch
    from rocco_b200 import _lib, pipeline
    k_shards = len(parts)
    m_total = sum(int(p[0].shape[0]) for p in parts)
    barrier = threading.Barrier(k_shards, timeout=120)
    bufs = [None] * k_shards
    total = [None]

    def reducer(k):
        def fn(buf):
            torch.cuda.current_stream().synchronize()
            bufs[k] = buf
            barrier.wait()
            if k == 0:
                acc = bufs[0].clone()
                for b in bufs[1:]:
                    acc += b
                torch.cuda.current_stream().synchronize()
                total[0] = acc
            barrier.wait()
            buf.copy_(total[0])
            torch.cuda.current_stream().synchronize()
            barrier.wait()                    # nobody starts the next reduce before every rank has its copy
        return fn

    out = [None] * k_shards

    def worker(k):
        rows, offset, inn = parts[k]
        stream = torch.cuda.Stream()
        try:
            with torch.cuda.stream(stream):
                out[k] = ("ok", pipeline._budget_null_sharded(rows, m_total, offset, reducer(k), innovations=inn, **kw))
        except Exception as exc:              # noqa: BLE001 - reported to the test
            out[k] = ("err", exc, _lib.last_error())

    torch.cuda.synchronize()
    threads = [threading.Thread(target=worker, args=(k,)) for k in range(k_shards)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(timeout=900)
    assert not any(t.is_alive() for t in threads), "a shard never returned"
    return out


@pytest.fixture(scope="module")
def case():
    """7 samples x 60k bins: centred rows and observed scores on the device."""
    import torch
    from rocco_b200 import pipeline
    x = chrom_matrix_numpy(7, 60_000, seed=17)
    prm = pipeline.score_params(prior_df=6.0)
    scores, det = pipeline.score_loci_wls_device(torch.from_numpy(x).cuda(), params=prm, details=True)
    return {"centered": det["centered_matrix"], "scores": scores, "params": prm, "hint": det["local_baseline_window"]}


def test_one_shard_is_the_unsharded_path(case):
    import torch
    from rocco_b200 import pipeline
    c, s, prm = case["centered"], case["scores"], case["params"]
    m, n = c.shape
    noop = lambda buf: None                                                           # noqa: E731
    common = dict(params=prm, dependence_lag_hint=case["hint"], num_null_draws=12, random_seed=5)
    want = pipeline.budget_null_device(c, s, **common)
    got = pipeline._budget_null_sharded(c, m, 0, noop, d_observed_scores=s, **common)
    assert got == want                                                                # every key bit for bit
    alone = pipeline.budget_null_sample_sharded(c, s, **common)                       # no process group: one rank
    assert alone == want
    # supplied innovations: the reduce-and-finalise passes against the unsharded C path
    bw = int(want[1]["wild_bandwidth"])
    inn = torch.from_numpy(np.random.default_rng(8).standard_normal((4, m, n + 2 * bw))).cuda()
    kw = dict(params=prm, dependence_lag_hint=case["hint"], num_null_draws=4, innovations=inn)
    want_i = pipeline._budget_null_sharded(c, m, 0, None, d_observed_scores=s, **kw)
    got_i = pipeline._budget_null_sharded(c, m, 0, noop, d_observed_scores=s, **kw)
    assert got_i == want_i
    assert want_i[1]["num_null_draws"] == 4.0


def test_two_shards_on_one_gpu_match_the_unsharded_estimator(case):
    from rocco_b200 import pipeline
    c, s, prm = case["centered"], case["scores"], case["params"]
    n = c.shape[1]
    common = dict(params=prm, dependence_lag_hint=case["hint"], num_null_draws=10, min_null_draws=10, random_seed=21)
    want_frac, want = pipeline.budget_null_device(c, s, **common)
    # 3 + 4 rows: the second shard's offset (3) is not rank * m_local (4)
    out = run_shards([(c[:3].contiguous(), 0, None), (c[3:].contiguous(), 3, None)], d_observed_scores=s, **common)
    assert [o[0] for o in out] == ["ok", "ok"], out
    (f0, d0), (f1, d1) = out[0][1], out[1][1]
    assert d0 == d1 and f0 == f1                                                      # both ranks: the same bits
    assert d0["num_null_draws"] == 10.0
    assert abs(f0 - want_frac) <= 2.0 / n
    assert_close_details(d0, want, n, what="3+4 shards")
    # the fit's scores (no observed track given) come out of the reduce too
    out2 = run_shards([(c[:3].contiguous(), 0, None), (c[3:].contiguous(), 3, None)], **common)
    assert out2[0][0] == "ok" and out2[0][1] == out2[1][1]
    assert_close_details(out2[0][1][1], pipeline.budget_null_device(c, None, **common)[1], n, what="fit scores")


def test_two_shards_reproduce_the_reference_replay():
    """The goldens of the real reference (tests/test_budget_gpu.py::test_budget_estimator_replays_reference) with the rows
    split over two emulated ranks and the replayed innovations sliced by sample."""
    import torch
    from rocco_b200 import pipeline
    from rocco_b200.inference import _resolve_budget_bootstrap_bandwidth
    g = np.load(os.path.join(REPO, "tests", "golden", "reference_budget_v1_11_0.npz"))
    for tag in ("ref_test", "synth_a", "synth_b"):
        kw = json.loads(str(g[f"{tag}_kwargs"]))
        want = json.loads(str(g[f"{tag}_meta"]))
        centered, scores = g[f"{tag}_centered"], g[f"{tag}_scores"]
        m, n = centered.shape
        bw = _resolve_budget_bootstrap_bandwidth(n, kw.get("dependence_lag_hint"))
        inn = reference_innovations(kw.get("random_seed", 0), kw["num_null_draws"], m, n, 2 * bw + 1)
        h = m // 2
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()             # noqa: E731
        out = run_shards([(dev(centered[:h]), 0, dev(inn[:, :h])), (dev(centered[h:]), h, dev(inn[:, h:]))],
                         d_observed_scores=dev(scores), params=pipeline.score_params(prior_df=kw.get("prior_df", 5.0)),
                         dependence_lag_hint=kw.get("dependence_lag_hint"), num_null_draws=kw["num_null_draws"],
                         random_seed=kw.get("random_seed", 0))
        assert [o[0] for o in out] == ["ok", "ok"], (tag, out)
        frac, meta = out[0][1]
        assert out[1][1] == out[0][1], tag
        for k, v in want.items():
            if isinstance(v, (str, bool)):
                assert meta[k] == v, (tag, k)
            elif k in INDICATOR_KEYS:
                assert abs(meta[k] - v) <= 2.0 / n + 1e-12, (tag, k, meta[k], v)
            elif k in COUNT_KEYS:
                assert abs(meta[k] - v) <= 2.0 + 1e-6 * abs(v), (tag, k, meta[k], v)
            else:
                assert abs(meta[k] - v) <= 1e-6 * max(1.0, abs(v)), (tag, k, meta[k], v)
        assert abs(frac - float(g[f"{tag}_fraction"])) <= 2.0 / n, tag


def test_a_local_failure_ends_every_shard_with_the_same_status(case):
    import torch
    from rocco_b200 import pipeline
    c, s, prm = case["centered"], case["scores"], case["params"]
    m, n = c.shape
    bw = pipeline._lib.load().rocco_b200_budget_bandwidth(n, case["hint"])
    inn = np.random.default_rng(4).standard_normal((3, m, n + 2 * bw))
    inn[0, 5] *= 1e-13                 # sample 5 (row 2 of the second shard): multiplier s.d. ~1e-13 < 1e-8 in draw 0
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()                 # noqa: E731
    kw = dict(d_observed_scores=s, params=prm, dependence_lag_hint=case["hint"], num_null_draws=3)
    out = run_shards([(c[:3].contiguous(), 0, dev(inn[:, :3])), (c[3:].contiguous(), 3, dev(inn[:, 3:]))], **kw)
    assert [o[0] for o in out] == ["err", "err"], out
    assert all(isinstance(o[1], ValueError) for o in out), out                      # non-finite status on both, no timeout
    assert "degenerate multiplier field" in out[1][2] and "another rank" in out[0][2], (out[0][2], out[1][2])
    with pytest.raises(ValueError):                                                   # the unsharded estimator agrees
        pipeline._budget_null_sharded(c, m, 0, None, innovations=dev(inn), **kw)


def test_sharded_arguments_are_checked():
    import torch
    from rocco_b200 import pipeline
    with pytest.raises(ValueError):
        pipeline.budget_null_sample_sharded(torch.zeros((2, 100), dtype=torch.float32, device="cuda"))
    with pytest.raises(ValueError):
        pipeline.budget_null_sample_sharded(torch.zeros((2, 100), dtype=torch.float64, device="cuda"),
                                            torch.zeros(99, dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        pipeline.budget_null_sample_sharded(torch.zeros((2, 100), dtype=torch.float64, device="cuda"), num_null_draws=2,
                                            innovations=torch.zeros((2, 2, 100), dtype=torch.float64, device="cuda"))


WORKER = r'''
import json, os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["ROCCO_B200_REPO"])
from rocco_b200 import pipeline
from rocco_b200.synth import chrom_matrix_numpy

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
backend = os.environ["ROCCO_B200_BACKEND"]
local = int(os.environ["LOCAL_RANK"]) % torch.cuda.device_count()     # gloo: both ranks may share one device
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if backend == "nccl":
    dist.init_process_group("nccl", device_id=dev)
else:
    dist.init_process_group("gloo")
m, n = 8, 120_001
x = chrom_matrix_numpy(m, n, seed=23)
prm = pipeline.score_params(prior_df=6.0)
lo, hi = (0, 3) if rank == 0 else (3, m)
out = {"rank": rank, "runs": []}
for dtype, draws, min_draws in ((np.float64, 8, 8), (np.float32, 8, 8), (np.float64, 25, None)):
    xs = x.astype(dtype)
    scores, cent, window = pipeline.score_loci_wls_sample_sharded(torch.from_numpy(xs[lo:hi]).to(dev), m, prm, keep_centered=True)
    kw = dict(params=prm, dependence_lag_hint=window, num_null_draws=draws, min_null_draws=min_draws, random_seed=7)
    frac, det = pipeline.budget_null_sample_sharded(cent, scores, **kw)
    w_scores, extra = pipeline.score_loci_wls_device(torch.from_numpy(xs).to(dev), params=prm, details=True)
    w_frac, w_det = pipeline.budget_null_device(extra["centered_matrix"], w_scores, **kw)
    every = [None] * world
    dist.all_gather_object(every, (frac, det))
    out["runs"].append({"dtype": np.dtype(dtype).name, "fixed_draws": min_draws is not None, "window": window,
                        "window_unsharded": extra["local_baseline_window"], "identical_across_ranks": all(e == every[0] for e in every),
                        "frac": frac, "det": det, "unsharded_frac": w_frac, "unsharded": w_det})
# a rank-local argument problem (float32 rows on rank 1) raises on both ranks before any reduce
try:
    pipeline.budget_null_sample_sharded(cent.float() if rank == 1 else cent, scores, **kw)
    out["local_problem"] = "no error"
except ValueError as exc:
    out["local_problem"] = str(exc)
sys.stdout.write("RESULT " + json.dumps(out) + "\n")
sys.stdout.flush()
dist.destroy_process_group()
'''


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_two_rank_nccl_sample_sharded_budget_null(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    _two_rank_sample_sharded_budget_null(tmp_path, "nccl")


def test_two_rank_gloo_sample_sharded_budget_null(tmp_path):
    """Both ranks may share one GPU: the reduces of CUDA tensors go through the host."""
    _two_rank_sample_sharded_budget_null(tmp_path, "gloo")


def _two_rank_sample_sharded_budget_null(tmp_path, backend):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, ROCCO_B200_REPO=REPO, ROCCO_B200_BACKEND=backend)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), str(script)]
    res = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    rows = [json.loads(ln.split("RESULT ", 1)[1]) for ln in res.stdout.splitlines() if "RESULT " in ln]
    assert len(rows) == 2
    for r in rows:
        for run in r["runs"]:
            assert run["identical_across_ranks"], run["dtype"]
            assert run["window"] == run["window_unsharded"]
            assert run["det"]["num_null_draws"] == rows[0]["runs"][r["runs"].index(run)]["det"]["num_null_draws"]
            if run["fixed_draws"]:
                n = run["det"]["num_loci"]
                assert abs(run["frac"] - run["unsharded_frac"]) <= 2.0 / n
                assert_close_details(run["det"], run["unsharded"], n, what=run["dtype"])
    by_rank = {r["rank"]: r["local_problem"] for r in rows}
    assert "float64" in by_rank[1] and "another rank" not in by_rank[1], by_rank
    assert "another rank" in by_rank[0] and by_rank[1] in by_rank[0], by_rank
