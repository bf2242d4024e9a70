"""Multi-GPU plumbing: one process per GPU, chromosomes sharded across ranks (SURVEY.md section 8e).

Every chromosome is scored, budgeted and solved independently in the reference (rocco.py:948-1098,
1157-1182), so the data path has NO collective.  The only exchange is a single all-reduce of
[selected bins, bins] for the genome-wide selected fraction (reporting) and a gather of the per-rank
BED shards to rank 0, which then sorts/merges them exactly like combine_chrom_results.
Works with NCCL (GPUs) and gloo (CPU tests) alike; with world size 1 nothing is initialised.
"""
from __future__ import annotations

import contextlib
from typing import Sequence

from . import _lib
from .pipeline import lpt_partition
from .rocco import _merge_bed_records


def _dist():
    import torch.distributed as dist
    return dist


def world(group=None) -> tuple[int, int]:
    """(rank, size) of this process in ``group`` (default: the whole world); (0, 1) without an initialised process group."""
    dist = _dist()
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


def collective_device(group, device=None):
    """Where the tensors of a collective on ``group`` live: the CPU for gloo, otherwise ``device`` (default: the current
    CUDA device)."""
    import torch
    if _dist().get_backend(group) == "gloo":
        return torch.device("cpu")
    return device if device is not None else torch.device("cuda", torch.cuda.current_device())


def agree(problem, facts: dict, group, what: str) -> list:
    """Every rank's ``facts`` in rank order, from one ``all_gather_object`` of ``{"problem": problem, **facts}`` over
    ``group`` (with one rank: ``[facts]`` and no collective).  ``problem`` is this rank's own argument error, or None.
    A rank with a problem raises ``ValueError(problem)`` and every other rank a ``ValueError`` that names it, so all
    ranks leave together instead of some entering a collective that the others never reach.  Checks across the
    gathered facts are the caller's."""
    size = world(group)[1]
    if size <= 1:
        if problem is not None:
            raise ValueError(problem)
        return [facts]
    every = [None] * size
    _dist().all_gather_object(every, {"problem": problem, **facts}, group=group)
    if problem is not None:
        raise ValueError(problem)
    bad = next((r["problem"] for r in every if r["problem"] is not None), None)
    if bad is not None:
        raise ValueError(f"{what}: another rank rejected its arguments: {bad}")
    return [{k: v for k, v in r.items() if k != "problem"} for r in every]


class _DeviceBuffer:
    """A raw float64 device buffer as a torch tensor (``__cuda_array_interface__``, no copy)."""

    def __init__(self, ptr: int, count: int):
        self.__cuda_array_interface__ = {"shape": (int(count),), "typestr": "<f8", "data": (int(ptr), False),
                                          "strides": None, "version": 2}


@contextlib.contextmanager
def allreduce_callback(reduce_fn, device, what: str):
    """``reduce_fn(buf)`` as the native ``rocco_b200_allreduce_fn`` (None when ``reduce_fn`` is None), for one native
    call made inside the ``with`` block.  ``buf`` is the library's float64 buffer as a tensor on ``device``.  An
    exception in ``reduce_fn`` fails the callback instead of unwinding through the C frames, and leaving the block raises
    it as ``RuntimeError`` -- before the caller looks at the native status, which then only reports the failed reduce."""
    import torch
    failure = []

    def call(ptr, count, _stream, _user):
        try:
            reduce_fn(torch.as_tensor(_DeviceBuffer(ptr, count), device=device))
            return 0
        except BaseException as exc:
            failure.append(exc)
            return 1

    yield None if reduce_fn is None else _lib.ALLREDUCE_FN(call)
    if failure:
        raise RuntimeError(f"{what}: the all-reduce failed: {failure[0]!r}") from failure[0]


def workspace_allreduce(workspace, group):
    """A ``reduce_fn`` for ``allreduce_callback``: sums ``buf`` over ``group`` in place through ``workspace``, a float64
    CUDA tensor at least as long as any ``buf``, allocated by the caller before the ranks agree (so that its failure is
    reported to every rank)."""
    dist = _dist()

    def reduce_fn(buf):
        w = workspace[: buf.numel()]
        w.copy_(buf)
        dist.all_reduce(w, group=group)
        buf.copy_(w)
    return reduce_fn


def shard_chromosomes(bin_counts: Sequence[int]) -> list[int]:
    """Indices of the chromosomes this rank owns (LPT packing by bin count, identical on every rank)."""
    rank, size = world()
    return lpt_partition(bin_counts, size)[rank]


def allreduce_selected(selected: int, bins: int, device=None) -> tuple[int, int]:
    """Genome-wide (selected bins, bins): the path's single cross-rank exchange."""
    import torch
    dist = _dist()
    rank, size = world()
    if size == 1:
        return int(selected), int(bins)
    t = torch.tensor([int(selected), int(bins)], dtype=torch.int64, device=device or "cpu")
    dist.all_reduce(t)
    return int(t[0].item()), int(t[1].item())


def gather_bed_records(records: list[tuple[str, int, int]]):
    """Rank 0 receives every rank's records and returns them merged in combine_chrom_results order
    (chromosome string, start, end); other ranks return None."""
    dist = _dist()
    rank, size = world()
    if size == 1:
        return _merge_bed_records(records)
    gathered = [None] * size if rank == 0 else None
    dist.gather_object(records, gathered, dst=0)
    if rank != 0:
        return None
    flat = [r for part in gathered for r in part]
    return _merge_bed_records(flat)


def gather_runs(chrom_index, starts, ends, device=None):
    """All ranks' runs (global chromosome index, first bin, last bin + 1) on rank 0, as three int64 arrays ordered by
    (chromosome index, start); other ranks get None.  Tensor collectives only (one all-gather of the counts, one of the
    padded records), so it runs on NCCL with CUDA tensors and on gloo with CPU tensors alike."""
    import numpy as np
    import torch
    dist = _dist()
    rank, size = world()
    rec = np.stack([np.asarray(chrom_index, dtype=np.int64), np.asarray(starts, dtype=np.int64),
                    np.asarray(ends, dtype=np.int64)]) if len(starts) else np.zeros((3, 0), dtype=np.int64)
    if size > 1:
        dev = device or "cpu"
        cnt = torch.tensor([rec.shape[1]], dtype=torch.int64, device=dev)
        counts = [torch.zeros_like(cnt) for _ in range(size)]
        dist.all_gather(counts, cnt)
        counts = [int(c.item()) for c in counts]
        kmax = max(max(counts), 1)
        pad = torch.zeros((3, kmax), dtype=torch.int64, device=dev)
        pad[:, :rec.shape[1]] = torch.from_numpy(rec).to(dev)
        parts = [torch.zeros_like(pad) for _ in range(size)]
        dist.all_gather(parts, pad)
        if rank != 0:
            return None
        rec = np.concatenate([p[:, :k].cpu().numpy() for p, k in zip(parts, counts)], axis=1)
    order = np.lexsort((rec[1], rec[0]))
    return rec[0][order], rec[1][order], rec[2][order]


def write_genome_bed(path: str, genome_names, my_names, runs, step: int, extras=(), device=None, first_start: int = 0):
    """ONE BED file for the genome, written by all ranks together without a gather pass.

    `genome_names`: every chromosome of the genome in the file's record order (the reference's combined BED sorts by the
    chromosome STRING, rocco.py:74-95); `my_names`: this rank's chromosomes, `runs` their (local chromosome index, first
    bin, last bin + 1) arrays as `pipeline.masks_to_runs` returns them.  One all-gather carries every rank's per-chromosome
    text sizes (plus the integers in `extras`, which come back summed over ranks: e.g. selected bins and bins); each
    rank then writes its chromosomes at their byte offsets (`pipeline.write_genome_bed_part`) and rank 0 fixes the file
    length.  The file is complete once every rank has returned (callers synchronise before reading it).
    Returns the list of summed extras."""
    import numpy as np
    import torch
    from . import pipeline
    dist = _dist()
    rank, size = world()
    genome_names = list(genome_names)
    pos = np.array([genome_names.index(c) for c in my_names], dtype=np.int64)
    sizes = np.zeros(len(genome_names), dtype=np.int64)
    if len(my_names):
        sizes[pos] = pipeline.bed_text_sizes(my_names, runs, step, first_start)
    msg = np.concatenate([np.asarray(list(extras), dtype=np.int64), sizes])
    if size > 1:
        dev = device or "cpu"
        mine = torch.from_numpy(msg).to(dev)
        parts = [torch.zeros_like(mine) for _ in range(size)]
        dist.all_gather(parts, mine)
        allv = torch.stack(parts).cpu().numpy()
    else:
        allv = msg[None, :]
    k = len(list(extras))
    total_sizes = allv[:, k:].sum(axis=0)                      # one rank owns each chromosome
    offsets = np.concatenate([[0], np.cumsum(total_sizes)[:-1]])
    if len(my_names):
        pipeline.write_genome_bed_part(path, list(my_names), runs, step, offsets[pos], first_start)
    if rank == 0:
        with open(path, "ab") as fh:                           # exact length, whatever an earlier file left behind
            fh.truncate(int(total_sizes.sum()))
    return [int(v) for v in allv[:, :k].sum(axis=0)]
