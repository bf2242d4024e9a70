"""Column statistics with the samples sharded over ranks (pipeline.column_stat_sample_sharded): every column reaches its
owner complete and in global sample order, so the result has the bits of the unsharded column_stat_device call."""
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
METHODS = (dict(method="median"), dict(method="quantile", quantile=0.75), dict(method="tmean", tprop=0.05),
           dict(method="mean"), dict(method="mad"), dict(method="iqr", rng=(10, 90)), dict(method="std"),
           dict(method="tstd", tprop=0.1), dict(method="quantile", quantile=0.5, power=0.5))


def _emulated(pipeline, shards, **kw):
    """The exchange of column_stat_sample_sharded played out in one process: every shard packs its ranges, each range's
    owner concatenates what it would receive (ranks in order) and reduces it; the owners' parts make the track."""
    import torch
    rows = [s.shape[0] for s in shards]
    n = shards[0].shape[1]
    ranges = pipeline.column_bin_ranges(n, len(shards))
    sends = [pipeline.column_pack_ranges(s, ranges) for s in shards]
    parts = []
    for q, (lo, hi) in enumerate(ranges):
        pieces = []
        for p, send in enumerate(sends):
            start = sum(rows[p] * (b - a) for a, b in ranges[:q])
            pieces.append(send[start: start + rows[p] * (hi - lo)])
        recv = torch.cat(pieces).view(sum(rows), hi - lo)
        if hi > lo:
            parts.append(pipeline.column_stat_device(recv, **kw))
    return torch.cat(parts)


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("m,n", [(1000, 1001), (37, 31), (900, 4099)])
def test_one_gpu_emulation_equals_unsharded(dtype, m, n):
    import torch
    from rocco_b200 import pipeline
    x = torch.from_numpy(chrom_matrix_numpy(m, n, seed=m + n)).to(getattr(torch, dtype)).cuda()
    cut = [0, m // 5, m // 5 + m // 2, m]                        # three uneven shards
    shards = [x[cut[k]: cut[k + 1]].contiguous() for k in range(3)]
    for kw in METHODS:
        want = pipeline.column_stat_device(x, **kw)
        assert torch.equal(_emulated(pipeline, shards, **kw), want), kw
    # a world of one rank is the unsharded call
    assert torch.equal(pipeline.column_stat_sample_sharded(x, m, "median"), pipeline.column_stat_device(x, "median"))
    with pytest.raises(ValueError):
        pipeline.column_stat_sample_sharded(x, m + 1, "median")
    with pytest.raises(ValueError):
        pipeline.column_stat_sample_sharded(x, m, "nope")


def test_bin_ranges():
    from rocco_b200 import pipeline
    for n, r in ((1, 2), (31, 2), (32, 2), (1001, 3), (12_450_000, 8), (5, 8)):
        ranges = pipeline.column_bin_ranges(n, r)
        assert len(ranges) == r and ranges[0][0] == 0 and ranges[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(ranges, ranges[1:]))
        last = max(q for q in range(r) if ranges[q][1] > ranges[q][0])
        assert all((hi - lo) % 16 == 0 for lo, hi in ranges[:last])


WORKER = r'''
import hashlib, json, os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["ROCCO_B200_REPO"])
sys.path.insert(0, os.environ["ROCCO_B200_TESTS"])
from rocco_b200 import pipeline
from rocco_b200.synth import chrom_matrix_numpy
from test_colstats_sharded_gpu import METHODS

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
backend = os.environ["ROCCO_B200_BACKEND"]
local = int(os.environ["LOCAL_RANK"]) % torch.cuda.device_count()     # gloo: both ranks may share one device
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if backend == "nccl":
    dist.init_process_group("nccl", device_id=dev)
else:
    dist.init_process_group("gloo")
out = {"rank": rank, "cases": {}}
m = 1000
split = 377                                                            # uneven shards
for n in (1001, 13):                                                   # odd n; n <= 16: rank 1 owns no bins
    x = torch.from_numpy(chrom_matrix_numpy(m, n, seed=n)).to(torch.float32).to(dev)
    mine = x[:split] if rank == 0 else x[split:]
    mine = mine.contiguous()
    for k, kw in enumerate(METHODS):
        got = pipeline.column_stat_sample_sharded(mine, m, **kw)
        want = pipeline.column_stat_device(x, **kw)
        out["cases"][f"{n}:{k}"] = {"equal": bool(torch.equal(got, want)),
                                    "digest": hashlib.sha256(got.cpu().numpy().tobytes()).hexdigest()}
try:
    bad = torch.zeros((10, 51 if rank == 1 else 50), dtype=torch.float32, device=dev)
    pipeline.column_stat_sample_sharded(bad, 20, "median")
    out["mismatch"] = "no error"
except ValueError:
    out["mismatch"] = "ValueError"
sys.stdout.write("RESULT " + json.dumps(out) + "\n")
sys.stdout.flush()
dist.destroy_process_group()
'''


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("backend", ["nccl", "gloo"])
def test_two_ranks(tmp_path, backend):
    """nccl: one GPU per rank; gloo: both ranks may share one GPU, the collectives going through host memory."""
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
        assert all(c["equal"] for c in r["cases"].values()), r["rank"]
        assert r["mismatch"] == "ValueError", r
    assert {k: v["digest"] for k, v in rows[0]["cases"].items()} == {k: v["digest"] for k, v in rows[1]["cases"].items()}
