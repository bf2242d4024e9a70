"""Device-resident driver of the hot path for MANY chromosomes at once.

The reference walks chromosomes one by one (rocco.py:948) and solves them in a fork pool of <= 4
processes (rocco.py:1146-1184).  Here every chromosome of a rank's shard is laid out in one device
buffer and each stage is a single batched launch set: scores [sum n_c] float64, masks [sum n_c]
uint8, chromosome c at ``offset_c`` (offsets padded to 16 elements so 128-bit accesses stay aligned).
PyTorch is used for device memory and streams only.
"""
from __future__ import annotations

import ctypes
import threading
from typing import Optional, Sequence

import numpy as np

from . import _lib

ALIGN = 16


def _torch():
    import torch
    return torch


def _stream_ptr(device) -> int:
    torch = _torch()
    return int(torch.cuda.current_stream(device).cuda_stream)


def layout_offsets(lengths: Sequence[int]) -> tuple[list[int], int]:
    offsets, cur = [], 0
    for n in lengths:
        offsets.append(cur)
        cur += (int(n) + ALIGN - 1) // ALIGN * ALIGN
    return offsets, max(cur, ALIGN)


def target_count_for_budget(n: int, budget: float) -> int:
    """dp.py:197 -- computed on the host in float64 exactly as the reference does."""
    return int(np.floor(int(n) * float(budget)))


def pack_scores(scores_list, device=None):
    """Concatenate per-chromosome score vectors (NumPy or CUDA tensors) into one float64 device buffer."""
    torch = _torch()
    if device is None:
        device = next((s.device for s in scores_list if isinstance(s, torch.Tensor) and s.is_cuda),
                      torch.device("cuda", torch.cuda.current_device()))
    lengths = [int(s.shape[0]) for s in scores_list]
    offsets, total = layout_offsets(lengths)
    buf = torch.zeros(total, dtype=torch.float64, device=device)
    for s, off, n in zip(scores_list, offsets, lengths):
        if isinstance(s, torch.Tensor):
            if s.dim() != 1:
                raise ValueError("`scores` must be a one-dimensional array")
            buf[off:off + n].copy_(s.to(dtype=torch.float64), non_blocking=True)
        else:
            a = np.ascontiguousarray(s, dtype=np.float64)
            if a.ndim != 1:
                raise ValueError("`scores` must be a one-dimensional array")
            buf[off:off + n].copy_(torch.from_numpy(a), non_blocking=False)
    return buf, offsets, lengths


def solve_packed(d_scores, offsets, lengths, budgets, gammas, selection_penalties=None, max_iter: int = 60,
                 levels_per_round: int = 0, d_masks=None):
    """Run the batched chain solve on an already packed device buffer.

    Returns (d_masks uint8 tensor, list of ChainResult-like dicts).  No host copy of the masks."""
    torch = _torch()
    lib = _lib.load()
    _lib.require_device()
    nchrom = len(lengths)
    if selection_penalties is None:
        selection_penalties = [None] * nchrom
    tasks = (_lib.ChainTask * nchrom)()
    for c in range(nchrom):
        n = int(lengths[c])
        if n <= 0:
            raise ValueError("`scores` cannot be empty")
        g = float(gammas[c])
        t = tasks[c]
        t.offset, t.n, t.gamma = int(offsets[c]), n, g
        t.cost_sum = _lib.numpy_sum_const(g, n - 1) if n > 1 else 0.0
        t.max_iter = int(max_iter)
        if selection_penalties[c] is not None:
            t.mode, t.selection_penalty, t.target_count = 0, float(selection_penalties[c]), 0
        elif budgets[c] is None:
            t.mode, t.selection_penalty, t.target_count = 0, 0.0, 0
        else:
            t.mode, t.selection_penalty = 1, 0.0
            t.target_count = target_count_for_budget(n, budgets[c])
    if d_masks is None:
        d_masks = torch.zeros(d_scores.shape[0], dtype=torch.uint8, device=d_scores.device)
    results = (_lib.ChainResult * nchrom)()
    with torch.cuda.device(d_scores.device):
        st = lib.rocco_b200_chain_solve_batch_dev(
            ctypes.c_void_p(d_scores.data_ptr()), None, tasks, nchrom,
            ctypes.c_void_p(d_masks.data_ptr()), results, int(levels_per_round),
            ctypes.c_void_p(_stream_ptr(d_scores.device)))
    _lib.check(st, "solve_chrom_exact")
    return d_masks, [_chain_result_dict(results[c]) for c in range(nchrom)]


def _chain_result_dict(r) -> dict:
    return {
        "selection_penalty": float(r.selection_penalty),
        "penalized_objective": float(r.penalized_objective),
        "objective": float(r.objective),
        "selected_count": int(r.selected_count),
        "switch_count": int(r.switch_count),
        "exact_tie_bins": int(r.exact_tie_bins),
        "near_tie_bins": int(r.near_tie_bins),
        "dp_passes": int(r.dp_passes),
        "search_rounds": int(r.search_rounds),
    }


def solve_chromosomes(scores_list, budgets, gammas, selection_penalties=None, max_iter: int = 60,
                      levels_per_round: int = 0):
    """solve_chrom_exact for a list of chromosomes in one batched launch set; NumPy masks returned."""
    torch = _torch()
    if any(isinstance(s, torch.Tensor) and s.is_cuda for s in scores_list):
        d_scores, offsets, lengths = pack_scores(scores_list)
        d_masks, res = solve_packed(d_scores, offsets, lengths, budgets, gammas, selection_penalties,
                                    max_iter=max_iter, levels_per_round=levels_per_round)
        h_masks = d_masks.cpu().numpy()
    else:
        # Host inputs: run on this thread's own high-priority stream with pinned staging.  The solve is a chain of short
        # launches; on the shared default stream (or at normal priority) it queues behind whatever bulk scoring kernels
        # and 256 MB copies other host threads have in flight, and a pageable upload is cut into many small DMA commands
        # each of which waits for one of those copies.
        _lib.require_device()
        dev = torch.device("cuda", torch.cuda.current_device())
        arrays = []
        for s in scores_list:
            a = np.ascontiguousarray(s, dtype=np.float64)
            if a.ndim != 1:
                raise ValueError("`scores` must be a one-dimensional array")
            arrays.append(a)
        lengths = [int(a.shape[0]) for a in arrays]
        offsets, total = layout_offsets(lengths)
        with _StageLease(total * 9) as stage, _UrgentStream(dev) as stream:
            h_scores = stage[: total * 8].view(torch.float64)
            h_scores.zero_()
            for a, off, n in zip(arrays, offsets, lengths):
                h_scores[off:off + n].copy_(torch.from_numpy(a))
            with torch.cuda.stream(stream):
                d_scores = torch.empty(total, dtype=torch.float64, device=dev)
                # kernel-driven upload: a DMA command would wait for every bulk copy already queued (see runtime.cu)
                _lib.check(_lib.load().rocco_b200_pull_pinned(ctypes.c_void_p(d_scores.data_ptr()), ctypes.c_void_p(h_scores.data_ptr()),
                                                              total * 8, ctypes.c_void_p(stream.cuda_stream)), "upload")
                d_masks, res = solve_packed(d_scores, offsets, lengths, budgets, gammas, selection_penalties,
                                            max_iter=max_iter, levels_per_round=levels_per_round)
                h_m = stage[total * 8: total * 9]
                h_m.copy_(d_masks, non_blocking=True)
                stream.synchronize()
            h_masks = h_m.numpy().copy()
    for r, off, n in zip(res, offsets, lengths):
        r["solution"] = h_masks[off:off + n].copy()
    return res


# ------------------------------------------------------------------ genome-wide budget: one multiplier for every chromosome
# Opt-in, and not a behaviour of the reference (which searches one multiplier per chromosome, dp.py:197-207): the search of
# dp.py:89-164 on the concatenated chain S = s_1 || s_2 || ... with zero switch cost at the junctions (include/rocco_b200.h).
def genome_cost_sum(lengths, gammas) -> float:
    """Correctly rounded sum of gamma_c * (n_c - 1): the switch costs of the concatenated chain.  Summed exactly (rationals),
    so the bracket does not depend on the order of the chromosomes or on how they are spread over ranks."""
    from fractions import Fraction
    return float(sum((Fraction(float(g)) * max(int(n) - 1, 0) for n, g in zip(lengths, gammas)), Fraction(0)))


def _genome_cost_max(lengths, gammas) -> float:
    return max([float(g) for n, g in zip(lengths, gammas) if int(n) >= 2], default=0.0)


def _exact_search_on() -> bool:
    lib = _lib.load()
    prev = lib.rocco_b200_chain_set_exact_search(0)
    lib.rocco_b200_chain_set_exact_search(prev)
    return bool(prev)


def _genome_problem(d_scores, offsets, lengths, gammas, genome_budget):
    """This rank's own argument errors, or None."""
    torch = _torch()
    if not isinstance(d_scores, torch.Tensor) or not d_scores.is_cuda or d_scores.dtype != torch.float64 or d_scores.dim() != 1:
        return "`d_scores` must be a one-dimensional float64 CUDA tensor"
    if len(offsets) != len(lengths) or len(gammas) != len(lengths):
        return "`offsets`, `lengths` and `gammas` must have one entry per chromosome"
    if any(int(n) <= 0 for n in lengths):
        return "`scores` cannot be empty"
    if any(not (float(g) >= 0.0) or not np.isfinite(float(g)) for g in gammas):
        return "switch costs (`gammas`) must be finite and >= 0"
    if any(int(o) < 0 or int(o) + int(n) > d_scores.shape[0] for o, n in zip(offsets, lengths)):
        return "a chromosome lies outside `d_scores`"
    if not np.isfinite(float(genome_budget)):
        return "`genome_budget` must be finite"
    if _exact_search_on():
        return "exact search replays one chromosome's recurrence and has no meaning for a genome-wide budget; turn it off"
    return None


def _score_extremes(d_scores, offsets, lengths):
    """(min, max) over this rank's chromosomes, None without chromosomes; raises on a non-finite score."""
    torch = _torch()
    if not lengths:
        return None
    parts = [d_scores[int(o):int(o) + int(n)] for o, n in zip(offsets, lengths)]
    ext = torch.stack([torch.stack([p.min(), p.max(), torch.isfinite(p).all().to(torch.float64)]) for p in parts]).cpu()
    if not bool((ext[:, 2] > 0).all()):
        return "non-finite"
    return float(ext[:, 0].min()), float(ext[:, 1].max())


def _solve_genome(d_scores, d_costs, offsets, lengths, gammas, search, levels_per_round, d_masks, reduce_fn):
    """One rank's call of rocco_b200_chain_solve_genome_dev with the search fields already agreed.  ``reduce_fn(buf)`` sums
    the float64 CUDA tensor ``buf`` over the ranks in place on torch's current stream (None: this call holds the genome)."""
    from .distributed import allreduce_callback
    torch = _torch()
    lib = _lib.load()
    dev = d_scores.device
    nchrom = len(lengths)
    tasks = (_lib.ChainTask * max(nchrom, 1))()
    for c in range(nchrom):
        t = tasks[c]
        t.offset, t.n, t.gamma, t.max_iter = int(offsets[c]), int(lengths[c]), float(gammas[c]), int(search.max_iter)
    if d_masks is None:
        d_masks = torch.zeros(d_scores.shape[0], dtype=torch.uint8, device=dev)
    results = (_lib.ChainResult * max(nchrom, 1))()
    genome = _lib.GenomeResult()
    with torch.cuda.device(dev), allreduce_callback(reduce_fn, dev, "genome budget") as cb:
        st = lib.rocco_b200_chain_solve_genome_dev(
            ctypes.c_void_p(d_scores.data_ptr()), None if d_costs is None else ctypes.c_void_p(d_costs.data_ptr()),
            tasks, nchrom, ctypes.byref(search), cb, None, ctypes.c_void_p(d_masks.data_ptr()), results,
            ctypes.byref(genome), int(levels_per_round), ctypes.c_void_p(_stream_ptr(dev)))
    if st == _lib.ST_INVALID and _lib.last_error().startswith("genome budget"):
        raise ValueError(_lib.last_error())
    _lib.check(st, "genome budget")
    out = {"selection_penalty": float(genome.selection_penalty), "selected_count": int(genome.selected_count),
           "total_bins": int(search.total_bins), "target_count": int(search.target_count),
           "dp_passes": int(genome.dp_passes), "search_rounds": int(genome.search_rounds)}
    return d_masks, out, [_chain_result_dict(results[c]) for c in range(nchrom)]


def solve_genome_packed(d_scores, offsets, lengths, genome_budget, gammas, max_iter: int = 60, levels_per_round: int = 0,
                        d_masks=None, group=None):
    """One multiplier for the whole genome: the chromosomes packed in ``d_scores`` (as ``solve_packed``) and, when ``group``
    has more than one rank, those of every other rank of it (a rank may hold none).  target = floor(N * genome_budget) over
    all N bins; each search round's counts are summed over the ranks with one ``torch.distributed.all_reduce`` of at most
    2^L + 1 doubles.  Returns ``(d_masks, genome, results)``: ``genome`` holds the multiplier, the genome's selected count,
    N, the target, the DP passes and the rounds; ``results`` the per-chromosome dicts of ``solve_packed``."""
    from .distributed import agree, workspace_allreduce, world
    torch = _torch()
    _lib.require_device()
    problem = _genome_problem(d_scores, offsets, lengths, gammas, genome_budget)
    nan = float("nan")
    if world(group)[1] <= 1:
        if problem:
            raise ValueError(problem)
        total = sum(int(n) for n in lengths)
        if total == 0:
            raise ValueError("the genome has no chromosome")
        search = _lib.GenomeSearch(total, target_count_for_budget(total, genome_budget), genome_cost_sum(lengths, gammas),
                                   _genome_cost_max(lengths, gammas), nan, nan, int(max_iter), 0)
        return _solve_genome(d_scores, None, offsets, lengths, gammas, search, levels_per_round, d_masks, None)

    dev = d_scores.device if isinstance(d_scores, torch.Tensor) and d_scores.is_cuda else torch.device("cuda", torch.cuda.current_device())
    # the reduce workspace (2^8 - 1 counts + 2 slots at most) is allocated before the ranks compare notes, so that its
    # failure is one more problem reported to all of them
    workspace = None
    extremes = None
    if problem is None:
        try:
            workspace = torch.empty(257, dtype=torch.float64, device=dev)
            extremes = _score_extremes(d_scores, offsets, lengths)
        except RuntimeError as exc:
            problem = f"genome budget: {exc}"
        if extremes == "non-finite":
            problem = "genome budget: non-finite values in `d_scores`"
    mine = {} if problem else {"n": [int(n) for n in lengths], "gamma": [float(g) for g in gammas], "extremes": extremes,
                               "agreed": (float(genome_budget), int(max_iter), int(levels_per_round))}
    every = agree(problem, mine, group, "genome budget")
    if any(r["agreed"] != mine["agreed"] for r in every):
        raise ValueError("genome budget: every rank must pass the same genome_budget, max_iter and levels_per_round")
    all_n = [n for r in every for n in r["n"]]
    all_g = [g for r in every for g in r["gamma"]]
    total = sum(all_n)
    if total == 0:
        raise ValueError("the genome has no chromosome")
    ext = [r["extremes"] for r in every if r["extremes"] is not None]
    search = _lib.GenomeSearch(total, target_count_for_budget(total, genome_budget), genome_cost_sum(all_n, all_g),
                               _genome_cost_max(all_n, all_g), min(e[0] for e in ext), max(e[1] for e in ext),
                               int(max_iter), 0)
    return _solve_genome(d_scores, None, offsets, lengths, gammas, search, levels_per_round, d_masks,
                         workspace_allreduce(workspace, group))


def solve_genome(scores_list, genome_budget, gammas, switch_costs_list=None, max_iter: int = 60, levels_per_round: int = 0,
                 group=None):
    """``solve_genome_packed`` for a list of NumPy arrays or tensors; returns ``(masks, genome, results)`` with the masks as
    NumPy arrays.  ``switch_costs_list`` (single process only; ``gammas`` is then ignored) gives each chromosome its own
    n_c - 1 switch costs; their genome sum is ``math.fsum`` of all of them."""
    import math
    from .distributed import world
    torch = _torch()
    if switch_costs_list is None:
        d_scores, offsets, lengths = pack_scores(scores_list)
        d_masks, genome, results = solve_genome_packed(d_scores, offsets, lengths, genome_budget, gammas, max_iter=max_iter,
                                                       levels_per_round=levels_per_round, group=group)
    else:
        if world(group)[1] > 1:
            raise ValueError("`switch_costs_list` is supported in a single process only")
        _lib.require_device()
        if len(switch_costs_list) != len(scores_list):
            raise ValueError("`switch_costs_list` must have one vector per chromosome")
        d_scores, offsets, lengths = pack_scores(scores_list)
        costs = [np.ascontiguousarray(c, dtype=np.float64).reshape(-1) for c in switch_costs_list]
        for c, n in zip(costs, lengths):
            if c.shape[0] != max(n - 1, 0):
                raise ValueError("each switch-cost vector must have n - 1 entries")
            if c.size and not (np.all(np.isfinite(c)) and np.all(c >= 0.0)):
                raise ValueError("switch costs must be finite and >= 0")
        zeros = [0.0] * len(lengths)
        problem = _genome_problem(d_scores, offsets, lengths, zeros, genome_budget)
        if problem:
            raise ValueError(problem)
        total = sum(lengths)
        if total == 0:
            raise ValueError("the genome has no chromosome")
        d_costs = torch.zeros_like(d_scores)
        for c, off in zip(costs, offsets):
            if c.size:
                d_costs[off:off + c.shape[0]].copy_(torch.from_numpy(c))
        flat = [float(x) for c in costs for x in c]
        search = _lib.GenomeSearch(total, target_count_for_budget(total, genome_budget), math.fsum(flat), max(flat, default=0.0),
                                   float("nan"), float("nan"), int(max_iter), 0)
        d_masks, genome, results = _solve_genome(d_scores, d_costs, offsets, lengths, zeros, search, levels_per_round, None, None)
    h_masks = d_masks.cpu().numpy()
    return [h_masks[off:off + n].copy() for off, n in zip(offsets, lengths)], genome, results


_URGENT: dict = {}


class _UrgentStream:
    """Borrow a highest-priority stream of `dev` from a process-wide free list (returned on exit).  The set of streams
    stays as small as the peak number of concurrent host threads, so torch's per-stream caching allocator reaches a steady
    state instead of seeing a fresh stream -- and a fresh cudaMalloc -- for every short-lived worker thread."""

    def __init__(self, dev):
        self.key = (dev.type, dev.index)
        self.dev = dev
        self.stream = None

    def __enter__(self):
        torch = _torch()
        with _STAGES_LOCK:
            free = _URGENT.setdefault(self.key, [])
            self.stream = free.pop() if free else None
        if self.stream is None:
            self.stream = torch.cuda.Stream(device=self.dev, priority=-1)
        return self.stream

    def __exit__(self, *exc):
        with _STAGES_LOCK:
            _URGENT[self.key].append(self.stream)
        self.stream = None
        return False


_STAGES: list = []
_STAGES_LOCK = threading.Lock()


class _StageLease:
    """A pinned staging buffer (uint8) borrowed from a process-wide free list and returned on exit.  Buffers are sized in
    64 MB steps and never freed: allocating or freeing pinned memory synchronises the device, which would stall the bulk
    copies and kernels of every other host thread."""

    def __init__(self, nbytes: int):
        self.nbytes = int(nbytes)
        self.buf = None

    def __enter__(self):
        torch = _torch()
        with _STAGES_LOCK:
            fit = [k for k, b in enumerate(_STAGES) if b.numel() >= self.nbytes]
            if fit:
                self.buf = _STAGES.pop(min(fit, key=lambda k: _STAGES[k].numel()))
        if self.buf is None:
            step = 64 << 20
            self.buf = torch.empty(((self.nbytes + step - 1) // step) * step or step, dtype=torch.uint8, pin_memory=True)
        return self.buf

    def __exit__(self, *exc):
        with _STAGES_LOCK:
            _STAGES.append(self.buf)
        self.buf = None
        return False


def masks_to_runs(d_masks, offsets, lengths):
    """All maximal runs of selected bins (last bin of each chromosome dropped), one batched pass.

    Returns (chrom_index int32[k], start_bin int64[k], end_bin int64[k]) with end exclusive."""
    torch = _torch()
    lib = _lib.load()
    nchrom = len(lengths)
    cap = int(sum((int(n) + 1) // 2 for n in lengths)) + 1
    starts = np.empty(cap, dtype=np.int64)
    ends = np.empty(cap, dtype=np.int64)
    chrom = np.empty(cap, dtype=np.int32)
    offs = np.asarray(offsets, dtype=np.uint64)
    lens = np.asarray(lengths, dtype=np.uint64)
    with torch.cuda.device(d_masks.device):
        k = lib.rocco_b200_mask_to_runs_batch_dev(
            ctypes.c_void_p(d_masks.data_ptr()), _lib.np_ptr(offs), _lib.np_ptr(lens), nchrom,
            _lib.np_ptr(starts), _lib.np_ptr(ends), _lib.np_ptr(chrom), cap,
            ctypes.c_void_p(_stream_ptr(d_masks.device)))
    if k < 0:
        _lib.check(int(k), "mask_to_runs")
    return chrom[:k].copy(), starts[:k].copy(), ends[:k].copy()


# ---------------------------------------------------------------------------------------------
# scoring on device-resident matrices
# ---------------------------------------------------------------------------------------------
def score_params(lower_bound_z=1.0, prior_df=5.0, min_effect=None, precision_floor_ratio=0.01,
                 spatial_window=31, baseline_window=101, exact_pilot=False):
    lib = _lib.load()
    prm = _lib.ScoreParams()
    lib.rocco_b200_default_score_params(ctypes.byref(prm))
    prm.lower_bound_z = float(lower_bound_z)
    prm.prior_df = float(prior_df)
    prm.use_min_effect = 0 if min_effect is None else 1
    prm.min_effect = 0.0 if min_effect is None else max(float(min_effect), 0.0)
    prm.precision_floor_ratio = float(max(precision_floor_ratio, 0.0))
    prm.spatial_window = int(spatial_window)
    prm.baseline_window = int(baseline_window)
    prm.pilot_mode = 1 if exact_pilot else 0          # exact np.median row offsets for any row length (validation mode)
    return prm


def score_loci_wls_device(d_matrix, out_scores=None, params=None, details: bool = False, centered_out=None):
    """score_loci_wls on a CUDA tensor [samples, bins] (float64 or float32, C-contiguous).

    Writes the scores into ``out_scores`` (a float64 CUDA tensor/view of length bins) or a new
    tensor; with ``details`` also returns the per-locus detail tensors.  ``centered_out`` (a contiguous float64 CUDA
    tensor shaped like the matrix) receives the centred rows -- the input of ``budget_null_device`` -- without the
    detail vectors being allocated.  Nothing leaves the device."""
    torch = _torch()
    lib = _lib.load()
    if d_matrix.dim() != 2 or not d_matrix.is_cuda or not d_matrix.is_contiguous():
        raise ValueError("`d_matrix` must be a contiguous two-dimensional CUDA tensor")
    if d_matrix.dtype not in (torch.float64, torch.float32):
        raise ValueError("`d_matrix` must be float64 or float32")
    m, n = d_matrix.shape
    if m == 0 or n == 0:
        raise ValueError("`chrom_matrix` must be non-empty")
    dev = d_matrix.device
    if centered_out is not None and (tuple(centered_out.shape) != (m, n) or centered_out.dtype != torch.float64
                                     or centered_out.device != dev or not centered_out.is_contiguous()):
        raise ValueError("`centered_out` must be a contiguous float64 tensor shaped like `d_matrix` on its device")
    if out_scores is None:
        out_scores = torch.empty(n, dtype=torch.float64, device=dev)
    out = _lib.ScoreOutputs()
    out.scores = out_scores.data_ptr()
    extra = {}
    if details:
        for k in ("mean", "raw_variance", "prior_variance", "moderated_variance", "standard_error"):
            extra[k] = torch.empty(n, dtype=torch.float64, device=dev)
            setattr(out, k, extra[k].data_ptr())
        extra["centered_matrix"] = torch.empty((m, n), dtype=torch.float64, device=dev) if centered_out is None else centered_out
    elif centered_out is not None:
        extra["centered_matrix"] = centered_out
    if "centered_matrix" in extra:
        out.centered_matrix = extra["centered_matrix"].data_ptr()
    prm = params if params is not None else score_params()
    with torch.cuda.device(dev):
        st = lib.rocco_b200_score_loci_wls_dev(
            ctypes.c_void_p(d_matrix.data_ptr()), 1 if d_matrix.dtype == torch.float32 else 0, m, n,
            ctypes.byref(prm), ctypes.byref(out), ctypes.c_void_p(_stream_ptr(dev)))
    if st == _lib.ST_NONFINITE:
        raise ValueError("Locus scoring produced non-finite values (or `chrom_matrix` contains non-finite values)")
    _lib.check(st, "score_loci_wls")
    if not details:
        return out_scores
    extra["total_df"] = float(out.total_df)
    extra["prior_spatial_window"] = int(out.resolved_spatial_window)
    extra["local_baseline_window"] = int(out.baseline_window)
    extra["local_baseline_lambda"] = float(out.baseline_lambda)
    return out_scores, extra


def lpt_partition(weights: Sequence[int], parts: int) -> list[list[int]]:
    """Longest-processing-time greedy packing of chromosomes onto ranks by bin count (SURVEY.md 8e)."""
    order = sorted(range(len(weights)), key=lambda i: (-int(weights[i]), i))
    loads = [0] * parts
    out: list[list[int]] = [[] for _ in range(parts)]
    for i in order:
        r = min(range(parts), key=lambda k: (loads[k], k))
        out[r].append(i)
        loads[r] += int(weights[i])
    for r in range(parts):
        out[r].sort()
    return out


_SCORE_STREAMS: dict = {}


def _score_streams(dev, count: int):
    torch = _torch()
    key = (dev.index, count)
    if key not in _SCORE_STREAMS:
        _SCORE_STREAMS[key] = [torch.cuda.Stream(device=dev) for _ in range(count)]
    return _SCORE_STREAMS[key]


# ------------------------------------------------------------------ ROCCO's default budgets and gamma (rocco.py:1023-1143)
# The reference's CLI without --gamma: per chromosome, score, run the wild-bootstrap budget null on the centred rows, then
# feed every chromosome's (effective_count, effective_total_count) to the empirical-Bayes budgets and set the automatic
# gamma from the null's autocorrelation time and the median positive score.
# "random_streams": the budget null's innovations, "philox" or "numpy" (the reference's own streams: see
# inference.random_streams_code).
DEFAULT_FLOW_ARGS = {"budget": None, "scale_chrom_budgets": 1.0, "budget_posterior_quantile": 0.01, "num_null_draws": 25,
                     "random_seed": 0, "random_streams": "philox"}


def _default_flow_args(default_args) -> dict:
    """The reference's CLI keys with their defaults, overridden by ``default_args``."""
    args = dict(DEFAULT_FLOW_ARGS)
    unknown = sorted(set(default_args or {}) - set(args))
    if unknown:
        raise ValueError(f"unknown `default_args` keys {unknown}; known: {sorted(args)}")
    args.update(default_args or {})
    if args["random_streams"] not in ("philox", "numpy"):
        raise ValueError(f"`random_streams` must be 'philox' or 'numpy', got {args['random_streams']!r}")
    return args


def _chromosome_name_problem(every) -> Optional[str]:
    """The first disagreement in the gathered ``{"names", "genome", "agreed"}`` of every rank, or None."""
    genome = every[0]["genome"]
    if any(r["genome"] != genome for r in every):
        return "default flow: every rank must pass the same `genome_names`"
    if any(r["agreed"] != every[0]["agreed"] for r in every):
        return "default flow: every rank must pass the same default arguments and the same budget and gamma modes"
    if len(set(genome)) != len(genome):
        return f"default flow: `genome_names` lists {sorted({c for c in genome if genome.count(c) > 1})} more than once"
    known = set(genome)
    for rank, r in enumerate(every):
        unknown = [c for c in r["names"] if c not in known]
        if unknown:
            return f"default flow: rank {rank} holds chromosomes missing from `genome_names`: {unknown}"
    held = [c for r in every for c in r["names"]]
    twice = sorted({c for c in held if held.count(c) > 1})
    if twice:
        return f"default flow: chromosomes held more than once: {twice}"
    unowned = [c for c in genome if c not in set(held)]
    if unowned:
        return f"default flow: no rank holds {unowned}"
    if not genome:
        return "default flow: the genome has no chromosome"
    return None


def agree_chromosome_names(chrom_names, genome_names, group=None, problem=None, agreed=None) -> int:
    """Check, on every rank of ``group`` at once, that the chromosomes the ranks hold are the genome: every name of
    ``chrom_names`` is in ``genome_names``, no name is held twice, no name of the genome is held by nobody, and every rank
    passed the same ``genome_names`` and ``agreed`` value.  ``problem`` is this rank's own argument error (or None).  One
    ``all_gather_object``; every rank raises the same ``ValueError``, except that a rank with a ``problem`` raises its own.
    Returns the number of chromosome slots of ``gather_budget_estimates``: the most any rank holds."""
    from .distributed import agree
    mine = {"names": [str(c) for c in chrom_names], "genome": None if genome_names is None else [str(c) for c in genome_names],
            "agreed": agreed}
    every = agree(problem, mine, group, "default flow")
    if any(r["genome"] is None for r in every):
        raise ValueError("default flow: `genome_names` is required when the chromosomes are spread over several ranks")
    msg = _chromosome_name_problem(every)
    if msg:
        raise ValueError(msg)
    return max(len(r["names"]) for r in every)


def gather_budget_estimates(chrom_names, genome_names, rows, slots: int, group=None, failure=None, device=None) -> dict:
    """The empirical-Bayes cache of the whole genome, in ``genome_names`` order, on every rank of ``group``.

    ``rows`` holds one ``(effective_count, effective_total_count, status)`` per chromosome of ``chrom_names`` (status 0:
    estimated; anything else: failed or not run); ``slots`` is what ``agree_chromosome_names`` returned.  One
    ``all_gather`` of ``slots + 1`` float64 rows ``[genome index, effective_count, effective_total_count, status]`` per
    rank (padding rows carry index -1; the last row is the rank's own status, set when it passes ``failure``, so that a
    rank without chromosomes can report one), on the CPU for gloo and on ``device`` (default: the current CUDA device)
    otherwise.  A status on any rank raises ``ValueError`` on every rank; the rank passing ``failure`` (its own message)
    raises that.
    Returns ``{name: {"budget_count_hat": effective_count, "total_count": effective_total_count}}`` in genome order, the
    cache ``rocco._resolve_budgets`` takes: the order is data, as the optimiser's path depends on the summation order."""
    from .distributed import collective_device, world
    torch = _torch()
    genome = [str(c) for c in genome_names]
    index = {c: g for g, c in enumerate(genome)}
    if len(rows) != len(chrom_names) or len(chrom_names) > int(slots):
        raise ValueError("`rows` must hold one entry per chromosome, and at most `slots`")
    table = np.zeros((int(slots) + 1, 4), dtype=np.float64)
    table[:, 0] = -1.0
    for k, (c, (count, total, status)) in enumerate(zip(chrom_names, rows)):
        table[k] = (index[str(c)], float(count), float(total), float(status))
    table[int(slots), 3] = 0.0 if failure is None else 1.0
    size = world(group)[1]
    if size <= 1:
        every = table
    else:
        import torch.distributed as dist
        mine = torch.from_numpy(table).to(collective_device(group, device))
        parts = [torch.empty_like(mine) for _ in range(size)]
        dist.all_gather(parts, mine, group=group)
        every = torch.cat(parts).cpu().numpy()
    if failure is not None:
        raise ValueError(failure)
    failed = every[(every[:, 0] >= 0) & (every[:, 3] != 0)]
    if failed.shape[0] or np.any(every[every[:, 0] < 0, 3] != 0):
        where = [genome[int(g)] for g in failed[:, 0]]
        raise ValueError("default flow: another rank failed" + (f" on {where}" if where else ""))
    by_index = {int(r[0]): r for r in every if r[0] >= 0}
    if sorted(by_index) != list(range(len(genome))):
        raise ValueError("default flow: the ranks' chromosomes do not cover `genome_names` exactly once")
    return {c: {"budget_count_hat": float(by_index[g][1]), "total_count": float(by_index[g][2])} for g, c in enumerate(genome)}


def _run_shard_defaults(d_matrices, budgets, gammas, params, levels_per_round, want_runs, score_streams, group,
                        chrom_names, genome_names, default_args, mark):
    """``run_shard`` with ROCCO's default budgets (``budgets`` None) and/or automatic gamma (``gammas`` None)."""
    from .distributed import world
    from .inference import _resolve_local_baseline_window
    from .rocco import _resolve_budgets, _resolve_chrom_gamma
    torch = _torch()
    mark = mark or (lambda label: None)
    nchrom = len(d_matrices)
    # this rank's own argument errors: the name agreement reports them to every rank
    problem = None
    try:
        args = _default_flow_args(default_args)
    except ValueError as exc:
        problem, args = str(exc), dict(DEFAULT_FLOW_ARGS)
    names = [] if chrom_names is None else [str(c) for c in chrom_names]
    if problem is None and score_streams > 1:
        problem = "the default flow scores one chromosome at a time: `score_streams` must be 1"
    if problem is None and (chrom_names is None or len(names) != nchrom):
        problem = "`chrom_names` must name each matrix of `d_matrices`, in the same order"
    if problem is None and any(v is not None and len(v) != nchrom for v in (budgets, gammas)):
        problem = "`budgets` and `gammas` must have one entry per matrix of `d_matrices`"
    if problem is None and any(not isinstance(x, torch.Tensor) or x.dim() != 2 or not x.is_cuda for x in d_matrices):
        problem = "every matrix of `d_matrices` must be a two-dimensional CUDA tensor"
    if genome_names is None and world(group)[1] <= 1:
        genome_names = names
    agreed = (tuple((k, args[k]) for k in sorted(args)), budgets is None, gammas is None)
    slots = agree_chromosome_names(names, genome_names, group=group, problem=problem, agreed=agreed)

    lengths = [int(x.shape[1]) for x in d_matrices]
    offsets, total = layout_offsets(lengths)
    # from here until the gather, every error of this rank goes into its status rows, so no rank is left in a collective
    nulls, rows, failure, dev, d_scores = [], [], None, None, None
    try:
        dev = d_matrices[0].device if nchrom else torch.device("cuda", torch.cuda.current_device())
        d_scores = torch.zeros(total, dtype=torch.float64, device=dev)
        prm = params if params is not None else score_params()
    except (ValueError, RuntimeError) as exc:
        failure = f"default flow: setting up the scores failed: {exc}"
    # one chromosome at a time: its centred rows live only until its null has run
    for name, x, off, n in zip(names, d_matrices, offsets, lengths):
        if failure is not None:
            break
        centered = None
        try:
            mark(f"score:{name}")
            centered = torch.empty(tuple(x.shape), dtype=torch.float64, device=dev)
            scores = score_loci_wls_device(x, out_scores=d_scores[off:off + n], params=prm, centered_out=centered)
            window = _resolve_local_baseline_window(n, prm.baseline_window if prm.baseline_window > 0 else 101)
            mark(f"null:{name}")
            _, det = budget_null_device(centered, scores, params=prm, dependence_lag_hint=window,
                                        num_null_draws=args["num_null_draws"], random_seed=args["random_seed"],
                                        random_streams=args["random_streams"])
        except (ValueError, RuntimeError) as exc:
            failure = f"default flow: {name}: {exc}"
            break
        finally:
            del centered
        nulls.append(det)
        rows.append((det["effective_count"], det["effective_total_count"], 0))
    rows += [(0.0, 0.0, 1)] * (nchrom - len(rows))
    mark("agree")
    cache = gather_budget_estimates(names, genome_names, rows, slots, group=group, failure=failure, device=dev)
    budget_meta = None
    if budgets is None:
        eb, budget_meta = _resolve_budgets(cache, args)
        budgets = [eb[c] for c in names]
    pairs = [_resolve_chrom_gamma(c, {"gamma": None if gammas is None else gammas[k]}, None, det)
             for k, (c, det) in enumerate(zip(names, nulls))]
    gammas = [g for g, _ in pairs]
    mark("solve")
    if nchrom:
        d_masks, results = solve_packed(d_scores, offsets, lengths, budgets, gammas, levels_per_round=levels_per_round)
    else:
        d_masks, results = torch.zeros(total, dtype=torch.uint8, device=dev), []
    mark("runs")
    runs = None
    if want_runs:
        runs = masks_to_runs(d_masks, offsets, lengths) if nchrom else \
            (np.zeros(0, np.int32), np.zeros(0, np.int64), np.zeros(0, np.int64))
    mark("end")
    return {"d_scores": d_scores, "d_masks": d_masks, "offsets": offsets, "lengths": lengths, "results": results,
            "runs": runs, "budgets": list(budgets), "gammas": gammas,
            "defaults": {"null": nulls, "gamma_meta": [m for _, m in pairs], "budget_meta": budget_meta}}


def run_shard(d_matrices, budgets, gammas, params=None, levels_per_round: int = 0, want_runs: bool = True,
              score_streams: int = 1, genome_budget=None, group=None, chrom_names=None, genome_names=None,
              default_args=None, mark=None):
    """The hot path for one rank's chromosomes, device-resident end to end:
    score every chromosome -> one batched budget search + solve -> one batched mask->runs pass.

    With `score_streams` > 1 chromosomes are scored from that many host threads, each on its own CUDA stream
    (measured on B200: no gain at 100 samples -- the streaming kernels already fill the device -- so the default is 1).
    With `genome_budget` (and `budgets` None) the search is the genome-wide one of `solve_genome_packed`: one multiplier
    for the chromosomes of every rank of `group`, and the result gains "genome".
    Returns dict(d_scores, d_masks, offsets, lengths, results, runs).

    ROCCO's defaults (its CLI without --gamma, rocco.py:1023-1143): `budgets` None (without `genome_budget`) gives the
    empirical-Bayes budgets, `gammas` None the automatic gamma; either needs the wild-bootstrap budget null of every
    chromosome.  Each chromosome is scored with its centred rows kept, its null runs on them (the Whittaker window is the
    dependence hint), and the rows are freed before the next chromosome; `score_streams` must be 1.  `chrom_names` names
    the matrices; `genome_names` lists every chromosome of every rank of `group` in genome order (ROCCO's chromosome
    order; default with one rank: `chrom_names`), the order in which the budgets are fitted.  `default_args` overrides
    the CLI keys of `DEFAULT_FLOW_ARGS`.  The ranks first agree on the names (`agree_chromosome_names`), then exchange
    their estimates in one all-gather (`gather_budget_estimates`); a failure on any rank raises ValueError on all of
    them.  The result gains "budgets" and "gammas" (lists in `d_matrices` order) and "defaults": the null's details
    ("null"), the gamma meta ("gamma_meta", None for a fixed gamma), both per chromosome, and the EB "budget_meta" (None
    for explicit budgets).  A rank without chromosomes passes `d_matrices=[]` and takes part all the same.
    `mark(label)`, when given, is called on the host as each phase begins ("score:<name>", "null:<name>", "agree",
    "solve", "runs") and at the "end": a hook for timing with CUDA events."""
    if genome_budget is not None and budgets is not None:
        raise ValueError("pass either per-chromosome `budgets` or one `genome_budget`, not both")
    if genome_budget is not None and (gammas is None or default_args is not None):
        raise ValueError("`genome_budget` takes explicit `gammas`; it does not combine with the default budgets or gamma")
    if gammas is None or (budgets is None and genome_budget is None):
        return _run_shard_defaults(d_matrices, budgets, gammas, params, levels_per_round, want_runs, score_streams, group,
                                   chrom_names, genome_names, default_args, mark)
    if any(v is not None for v in (chrom_names, genome_names, default_args, mark)):
        raise ValueError("`chrom_names`, `genome_names`, `default_args` and `mark` belong to the default flow "
                         "(`budgets` or `gammas` None); with explicit budgets and gammas they would be ignored")
    torch = _torch()
    lengths = [int(x.shape[1]) for x in d_matrices]
    offsets, total = layout_offsets(lengths)
    dev = d_matrices[0].device
    d_scores = torch.zeros(total, dtype=torch.float64, device=dev)
    if score_streams <= 1 or len(d_matrices) == 1:
        for x, off, n in zip(d_matrices, offsets, lengths):
            score_loci_wls_device(x, out_scores=d_scores[off:off + n], params=params)
    else:
        from concurrent.futures import ThreadPoolExecutor
        streams = _score_streams(dev, score_streams)
        main = torch.cuda.current_stream(dev)
        ready = torch.cuda.Event()
        ready.record(main)
        # largest chromosomes first, alternating streams
        order = sorted(range(len(d_matrices)), key=lambda i: -lengths[i])

        def work(slot):
            st = streams[slot]
            st.wait_event(ready)
            with torch.cuda.device(dev), torch.cuda.stream(st):
                for i in order[slot::score_streams]:
                    score_loci_wls_device(d_matrices[i], out_scores=d_scores[offsets[i]:offsets[i] + lengths[i]], params=params)
            ev = torch.cuda.Event()
            ev.record(st)
            return ev

        with ThreadPoolExecutor(max_workers=score_streams) as pool:
            for ev in pool.map(work, range(score_streams)):
                main.wait_event(ev)
    genome = None
    if genome_budget is None:
        d_masks, results = solve_packed(d_scores, offsets, lengths, budgets, gammas, levels_per_round=levels_per_round)
    else:
        d_masks, genome, results = solve_genome_packed(d_scores, offsets, lengths, genome_budget, gammas,
                                                       levels_per_round=levels_per_round, group=group)
    runs = masks_to_runs(d_masks, offsets, lengths) if want_runs else None
    out = {"d_scores": d_scores, "d_masks": d_masks, "offsets": offsets, "lengths": lengths,
           "results": results, "runs": runs}
    if genome is not None:
        out["genome"] = genome
    return out


def runs_to_bed_file(path: str, chrom_names, runs, step: int, first_start: int = 0) -> str:
    """Write all runs as BED3 (chromosomes in the given order; coordinates = first_start + bin*step) with the native
    formatter -- no per-record Python work."""
    chrom, starts, ends = runs
    return _lib.write_bed_arrays(path, list(chrom_names), chrom, first_start + starts * step, first_start + ends * step)


_POW10 = np.array([10 ** k for k in range(1, 19)], dtype=np.int64)


def bed_text_sizes(chrom_names, runs, step: int, first_start: int = 0) -> np.ndarray:
    """Bytes of BED3 text each chromosome of `runs` will take (name, two tabs, newline, the digits of both coordinates) --
    what a rank announces to the others before a genome BED is assembled with positioned writes (`write_genome_bed_part`)."""
    chrom, starts, ends = runs
    k = len(chrom_names)
    if chrom.shape[0] == 0:
        return np.zeros(k, dtype=np.int64)
    s = first_start + starts * step
    e = first_start + ends * step
    if int(s.min(initial=0)) < 0:
        raise ValueError("negative coordinates")
    digits = (np.searchsorted(_POW10, s, side="right") + 1) + (np.searchsorted(_POW10, e, side="right") + 1)
    name_len = np.array([len(str(c).encode("utf-8")) for c in chrom_names], dtype=np.int64)
    per_chrom_digits = np.bincount(chrom, weights=digits, minlength=k).astype(np.int64)
    counts = np.bincount(chrom, minlength=k).astype(np.int64)
    return per_chrom_digits + counts * (name_len + 3)


def write_genome_bed_part(path: str, chrom_names, runs, step: int, offsets, first_start: int = 0) -> int:
    """This rank's chromosomes written into the shared genome BED at their byte offsets (`offsets[c]` for chromosome index c
    of `chrom_names`; chromosomes without records are skipped).  Returns the bytes written."""
    chrom, starts, ends = runs
    bounds = np.searchsorted(chrom, np.arange(len(chrom_names) + 1))
    total = 0
    for c, name in enumerate(chrom_names):
        a, b = int(bounds[c]), int(bounds[c + 1])
        if b > a:
            total += _lib.write_bed_arrays_at(path, int(offsets[c]), [name], None, first_start + starts[a:b] * step,
                                              first_start + ends[a:b] * step)
    return total


def reorder_runs(runs, chrom_order):
    """Runs regrouped so that chromosome index `chrom_order[0]` comes first, then `chrom_order[1]`, ...  The runs of a
    shard arrive grouped by chromosome and sorted by start inside each group (`mask_to_runs`), so putting a genome into
    the reference's record order (rocco.py:74-95: chromosome STRINGS ascending, then start) is a permutation of
    blocks -- no sort.  Returns (position in chrom_order as int32, starts, ends)."""
    chrom, starts, ends = runs
    order = np.asarray(chrom_order, dtype=np.int64)
    bounds = np.searchsorted(chrom, np.arange(int(order.max(initial=-1)) + 2))
    take = np.concatenate([np.arange(bounds[c], bounds[c + 1]) for c in order] or [np.zeros(0, np.int64)])
    sizes = bounds[order + 1] - bounds[order]
    return np.repeat(np.arange(order.shape[0], dtype=np.int32), sizes), starts[take], ends[take]


def runs_to_bed_text(chrom_names, runs, step: int, first_start: int = 0) -> str:
    """BED3 text of all runs (per chromosome in the given order; coordinates = first_start + bin*step)."""
    chrom, starts, ends = runs
    s = first_start + starts * step
    e = first_start + ends * step
    names = np.asarray(chrom_names, dtype=object)[chrom]
    return "".join(f"{c}\t{a}\t{b}\n" for c, a, b in zip(names.tolist(), s.tolist(), e.tolist()))


def sweep_multipliers(scores, gamma: float, lambdas):
    """Selected count, penalized objective and objective of one chromosome for MANY multipliers
    (BASELINE.json config 5: a 256-multiplier budget sweep) -- up to 256 per launch set, the scores
    read once per tile whatever the number of multipliers.  Returns three NumPy arrays."""
    torch = _torch()
    lib = _lib.load()
    _lib.require_device()
    if isinstance(scores, torch.Tensor):
        d_scores = scores.to(dtype=torch.float64).contiguous()
        if not d_scores.is_cuda:
            d_scores = d_scores.cuda()
    else:
        d_scores = torch.from_numpy(np.ascontiguousarray(scores, dtype=np.float64)).cuda()
    if d_scores.dim() != 1 or d_scores.shape[0] == 0:
        raise ValueError("`scores` must be a non-empty one-dimensional array")
    lam = np.ascontiguousarray(lambdas, dtype=np.float64)
    k = lam.shape[0]
    counts = np.zeros(k, dtype=np.int64)
    pen = np.zeros(k, dtype=np.float64)
    obj = np.zeros(k, dtype=np.float64)
    with torch.cuda.device(d_scores.device):
        st = lib.rocco_b200_chain_sweep_dev(
            ctypes.c_void_p(d_scores.data_ptr()), int(d_scores.shape[0]), float(gamma), _lib.np_ptr(lam), int(k),
            _lib.np_ptr(counts), _lib.np_ptr(pen), _lib.np_ptr(obj), ctypes.c_void_p(_stream_ptr(d_scores.device)))
    _lib.check(st, "sweep_multipliers")
    return counts, pen, obj


def score_partial_device(d_matrix_local, params=None, centered_out=None):
    """Per-sample stages of this rank's rows -> the four per-bin accumulators, a [4, bins] float64 CUDA tensor.
    ``centered_out`` (a contiguous float64 CUDA tensor shaped like the rows) also receives the rows' centred values."""
    torch = _torch()
    lib = _lib.load()
    if d_matrix_local.dim() != 2 or not d_matrix_local.is_cuda or not d_matrix_local.is_contiguous():
        raise ValueError("`d_matrix_local` must be a contiguous two-dimensional CUDA tensor")
    m, n = d_matrix_local.shape
    if centered_out is not None and (tuple(centered_out.shape) != (m, n) or centered_out.dtype != torch.float64
                                     or centered_out.device != d_matrix_local.device or not centered_out.is_contiguous()):
        raise ValueError("`centered_out` must be a contiguous float64 tensor shaped like `d_matrix_local` on its device")
    acc = torch.empty((4, n), dtype=torch.float64, device=d_matrix_local.device)
    prm = params if params is not None else score_params()
    with torch.cuda.device(d_matrix_local.device):
        st = lib.rocco_b200_score_partial_ex_dev(
            ctypes.c_void_p(d_matrix_local.data_ptr()), 1 if d_matrix_local.dtype == torch.float32 else 0, m, n,
            ctypes.byref(prm), None if centered_out is None else ctypes.c_void_p(centered_out.data_ptr()),
            ctypes.c_void_p(acc.data_ptr()), ctypes.c_void_p(_stream_ptr(d_matrix_local.device)))
    if st == _lib.ST_NONFINITE:
        raise ValueError("Locus scoring produced non-finite values (or `chrom_matrix` contains non-finite values)")
    _lib.check(st, "score_partial")
    return acc


def score_finalize_device(acc, m_total: int, params=None, details: bool = False):
    torch = _torch()
    lib = _lib.load()
    n = acc.shape[1]
    out = _lib.ScoreOutputs()
    res = {"scores": torch.empty(n, dtype=torch.float64, device=acc.device)}
    if details:
        for k in ("mean", "raw_variance", "prior_variance", "moderated_variance", "standard_error"):
            res[k] = torch.empty(n, dtype=torch.float64, device=acc.device)
    for k, v in res.items():
        setattr(out, k, v.data_ptr())
    prm = params if params is not None else score_params()
    with torch.cuda.device(acc.device):
        st = lib.rocco_b200_score_finalize_dev(ctypes.c_void_p(acc.data_ptr()), int(m_total), n, ctypes.byref(prm),
                                               ctypes.byref(out), ctypes.c_void_p(_stream_ptr(acc.device)))
    if st == _lib.ST_NONFINITE:
        raise ValueError("Locus scoring produced non-finite values")
    _lib.check(st, "score_finalize")
    return res if details else res["scores"]


def score_loci_wls_sample_sharded(d_matrix_local, m_total: int, params=None, group=None, details: bool = False,
                                  keep_centered: bool = False):
    """score_loci_wls with the SAMPLES sharded over ranks (every rank holds [m_local, bins] of the same bins):
    per-sample stages stay local; one all-reduce(sum, float64) of the [4, bins] accumulators; every rank then
    finishes the per-bin combine (SURVEY.md section 8e(2)).

    With ``keep_centered`` returns ``(result, d_centered_local, baseline_window)``: this rank's centred rows (float64,
    the input of ``budget_null_sample_sharded``) and the resolved Whittaker window, which is the
    ``dependence_lag_hint`` the reference's CLI hands the budget null (rocco.py:1035)."""
    import torch.distributed as dist
    from .distributed import world
    torch = _torch()
    centered = None
    if keep_centered:
        centered = torch.empty(tuple(d_matrix_local.shape), dtype=torch.float64, device=d_matrix_local.device)
    acc = score_partial_device(d_matrix_local, params, centered_out=centered)
    if world(group)[1] > 1:
        dist.all_reduce(acc, group=group)
    result = score_finalize_device(acc, m_total, params, details=details)
    if not keep_centered:
        return result
    from .inference import _resolve_local_baseline_window
    prm = params if params is not None else score_params()
    window = _resolve_local_baseline_window(d_matrix_local.shape[1], prm.baseline_window if prm.baseline_window > 0 else 101)
    return result, centered, window


# ------------------------------------------------------------------ budget null on device tensors (SURVEY.md 8(f) rank 1)
def budget_null_device(d_centered, d_observed_scores=None, params=None, dependence_lag_hint=None, num_null_draws=25,
                       random_seed=0, min_null_draws=None, stability_abs_tol=5.0e-3, stability_rel_tol=5.0e-2,
                       random_streams="philox"):
    """``estimate_budget_nonnull_fraction_from_wild_bootstrap_null`` (inference.py:988-1148) on CUDA tensors: the centred
    matrix [samples, bins] (float64, as ``score_loci_wls_device(..., details=True)`` returns it) and optionally the observed
    scores stay on the device; returns ``(nonnull_fraction, details)`` with the reference's keys plus the positive-score
    median/count that ``rocco._resolve_chrom_gamma`` needs.  ``random_streams``: "philox" (default) or "numpy", the
    reference's own streams generated on the device (``inference.random_streams_code``)."""
    from .inference import _budget_details, budget_params
    torch = _torch()
    lib = _lib.load()
    problem = _budget_null_problem(d_centered, d_observed_scores, None, num_null_draws, dependence_lag_hint, random_seed,
                                   random_streams)
    if problem:
        raise ValueError(problem)
    m, n = d_centered.shape
    prm = budget_params(params if params is not None else score_params(), dependence_lag_hint, num_null_draws,
                        min_null_draws, stability_abs_tol, stability_rel_tol, random_seed, random_streams)
    res = _lib.BudgetResult()
    dev = d_centered.device
    with torch.cuda.device(dev):
        st = lib.rocco_b200_budget_nonnull_fraction_dev(
            ctypes.c_void_p(d_centered.data_ptr()), m, n,
            None if d_observed_scores is None else ctypes.c_void_p(d_observed_scores.data_ptr()),
            ctypes.byref(prm), ctypes.byref(res), ctypes.c_void_p(_stream_ptr(dev)))
    if st == _lib.ST_NONFINITE:
        raise ValueError("Budget initialization produced non-finite values")
    _lib.check(st, "budget null")
    return float(res.nonnull_fraction), _budget_details(res)


# ------------------------------------------------------------------ budget null with the samples sharded over ranks
def _budget_null_sharded(d_centered_local, m_total: int, sample_offset: int, reduce_fn, d_observed_scores=None, params=None,
                         dependence_lag_hint=None, num_null_draws=25, random_seed=0, min_null_draws=None,
                         stability_abs_tol=5.0e-3, stability_rel_tol=5.0e-2, innovations=None, random_streams="philox"):
    """One rank's part of the sample-sharded estimator, shapes already agreed between the ranks.  ``reduce_fn(buf)`` sums
    the float64 CUDA tensor ``buf`` over all ranks in place, ordered on torch's current stream; it is called with the same
    length on every rank, 2 + (draws used) times.  An exception in it becomes a failed call on this rank.  ``reduce_fn=None``
    (one rank holding every sample) is the unsharded estimator.  ``random_streams`` as for ``budget_null_device``: with
    "numpy", row r of this rank takes the normals of global sample ``sample_offset + r``, so the field is the same
    whatever the sharding."""
    from .distributed import allreduce_callback
    from .inference import _budget_details, budget_params
    torch = _torch()
    lib = _lib.load()
    prm = budget_params(params if params is not None else score_params(), dependence_lag_hint, num_null_draws,
                        min_null_draws, stability_abs_tol, stability_rel_tol, random_seed, random_streams,
                        sample_offset=sample_offset, d_innovations=innovations)
    m, n = d_centered_local.shape
    dev = d_centered_local.device
    res = _lib.BudgetResult()
    with torch.cuda.device(dev), allreduce_callback(reduce_fn, dev, "budget null") as cb:
        st = lib.rocco_b200_budget_nonnull_fraction_sharded_dev(
            ctypes.c_void_p(d_centered_local.data_ptr()), m, n, int(m_total),
            None if d_observed_scores is None else ctypes.c_void_p(d_observed_scores.data_ptr()),
            ctypes.byref(prm), cb, None, ctypes.byref(res), ctypes.c_void_p(_stream_ptr(dev)))
    if st == _lib.ST_NONFINITE:
        raise ValueError("Budget initialization produced non-finite values")
    _lib.check(st, "budget null")
    return float(res.nonnull_fraction), _budget_details(res)


def _budget_null_problem(d_centered, d_observed_scores, innovations, num_null_draws, dependence_lag_hint, random_seed,
                         random_streams):
    """The argument errors of ``budget_null_device`` and of one rank of ``budget_null_sample_sharded`` (checked there
    before the ranks compare shapes), or None."""
    from .inference import _resolve_budget_bootstrap_bandwidth, random_streams_code
    torch = _torch()
    try:
        random_streams_code(random_streams, random_seed, innovations)
    except ValueError as exc:
        return str(exc)
    x = d_centered
    if x.dim() != 2 or not x.is_cuda or not x.is_contiguous() or x.dtype != torch.float64:
        return "the centred rows must be a contiguous two-dimensional float64 CUDA tensor"
    m, n = x.shape
    if m == 0 or n == 0:
        return "`centered_matrix` must contain at least one sample and one locus"
    for name, t, shape in (("observed_scores", d_observed_scores, (n,)),
                           ("innovations", innovations, (int(max(1, num_null_draws)), m,
                                                         n + 2 * _resolve_budget_bootstrap_bandwidth(n, dependence_lag_hint)))):
        if t is not None and (tuple(t.shape) != shape or t.dtype != torch.float64 or t.device != x.device or not t.is_contiguous()):
            return f"`{name}` must be a contiguous float64 tensor of shape {shape} on the device of the centred rows"
    return None


def budget_null_sample_sharded(d_centered_local, d_observed_scores=None, params=None, group=None, dependence_lag_hint=None,
                               num_null_draws=25, random_seed=0, min_null_draws=None, stability_abs_tol=5.0e-3,
                               stability_rel_tol=5.0e-2, innovations=None, random_streams="philox"):
    """``budget_null_device`` with the SAMPLES sharded over the ranks of ``group`` (BASELINE.json config 5): every rank
    passes its centred rows ``[m_local, bins]`` (e.g. from ``score_loci_wls_sample_sharded(..., keep_centered=True)``, ranks
    in sample order) and the same observed scores and arguments.  Each scoring pass all-reduces 2 x bins float64 column
    sums (plus four status slots); every rank returns the same ``(nonnull_fraction, details)``, with the keys of
    ``budget_null_device``, and raises the same exception.  ``innovations``: this rank's rows,
    ``[draws, m_local, bins + 2*bandwidth]`` float64 on the device.  ``random_streams``: as for ``budget_null_device``;
    with "numpy" every rank generates the rows of its own samples, so the result equals the unsharded call's streams."""
    from .distributed import agree, workspace_allreduce, world
    torch = _torch()
    problem = _budget_null_problem(d_centered_local, d_observed_scores, innovations, num_null_draws, dependence_lag_hint,
                                   random_seed, random_streams)
    rank, size = world(group)
    if size <= 1:
        if problem:
            raise ValueError(problem)
        m = d_centered_local.shape[0]
        return _budget_null_sharded(d_centered_local, m, 0, None, d_observed_scores, params, dependence_lag_hint,
                                    num_null_draws, random_seed, min_null_draws, stability_abs_tol, stability_rel_tol, innovations,
                                    random_streams)
    dev = d_centered_local.device if d_centered_local.is_cuda else torch.device("cuda", torch.cuda.current_device())
    m, n = (d_centered_local.shape if d_centered_local.dim() == 2 else (0, 0))
    # the reduce workspace is allocated before the ranks compare notes, so that its failure is one more problem reported
    workspace = None
    if problem is None:
        try:
            workspace = torch.empty(2 * n + 4, dtype=torch.float64, device=dev)
        except RuntimeError as exc:
            problem = f"could not allocate the reduce workspace: {exc}"
    rows = agree(problem, {"m": int(m), "n": int(n)}, group, "budget null")
    if any(r["n"] != n for r in rows):
        raise ValueError(f"budget null: every rank must hold the same loci, got bins {[r['n'] for r in rows]}")
    offset, m_total = sum(r["m"] for r in rows[:rank]), sum(r["m"] for r in rows)
    return _budget_null_sharded(d_centered_local, m_total, offset, workspace_allreduce(workspace, group), d_observed_scores,
                                params, dependence_lag_hint, num_null_draws, random_seed, min_null_draws, stability_abs_tol,
                                stability_rel_tol, innovations, random_streams)


def _score_sample_sharded_agreed(x, m_total: int, prm, group, name: str):
    """``score_loci_wls_sample_sharded(..., keep_centered=True)`` with the ranks agreeing on success first: one
    all-reduce(MAX) of ``[failed, bins, -bins]`` comes before the accumulator all-reduce, so a rank whose per-sample stages
    fail (non-finite rows, allocation) or whose bins differ makes every rank raise ``ValueError`` instead of leaving the
    others waiting in the accumulator all-reduce.  Same calls and bits as ``score_loci_wls_sample_sharded`` otherwise."""
    from .distributed import collective_device, world
    from .inference import _resolve_local_baseline_window
    torch = _torch()
    failure, acc, centered, n = None, None, None, -1
    try:
        n = int(x.shape[1])
        centered = torch.empty(tuple(x.shape), dtype=torch.float64, device=x.device)
        acc = score_partial_device(x, prm, centered_out=centered)
    except (ValueError, RuntimeError) as exc:
        failure = f"default flow: {name}: {exc}"
    if world(group)[1] > 1:
        import torch.distributed as dist
        flag = torch.tensor([0.0 if failure is None else 1.0, float(n), -float(n)], dtype=torch.float64,
                            device=collective_device(group, x.device if isinstance(x, torch.Tensor) and x.is_cuda else None))
        dist.all_reduce(flag, op=dist.ReduceOp.MAX, group=group)
        failed, n_max, n_min = flag[0].item(), flag[1].item(), -flag[2].item()
        if failure is None and failed:
            failure = f"default flow: {name} failed on another rank"
        elif failure is None and n_max != n_min:
            failure = f"default flow: {name}: every rank must hold the same bins, got {int(n_min)} to {int(n_max)}"
        if failure is None:
            dist.all_reduce(acc, group=group)
    if failure is not None:
        raise ValueError(failure)
    scores = score_finalize_device(acc, m_total, prm)
    return scores, centered, _resolve_local_baseline_window(n, prm.baseline_window if prm.baseline_window > 0 else 101)


def run_sample_sharded_defaults(chroms, m_total: int, params=None, default_args=None, group=None, levels_per_round: int = 0,
                                mark=None):
    """ROCCO's default flow (EB budgets, automatic gamma) with the SAMPLES sharded over the ranks of ``group`` (config 5).

    ``chroms`` yields ``(name, d_rows_local)`` in genome order, the same chromosomes on every rank, each rank's rows of
    the chromosome (ranks in sample order); it is consumed one chromosome at a time, so the caller can generate or load
    each just in time.  Per chromosome: the scoring of ``score_loci_wls_sample_sharded(..., keep_centered=True)``, then
    ``budget_null_sample_sharded`` on the centred rows with the Whittaker window as the dependence hint; the rows are
    dropped before the next chromosome is drawn.  A failure on one rank raises ``ValueError`` on every rank: the scoring
    agrees on success before its all-reduce (``_score_sample_sharded_agreed``) and the null carries its own status.  Every rank then holds every chromosome's details, so the EB budgets and
    the gammas are computed on every rank from the same doubles, with no further exchange.  Each chromosome is solved on
    its ``lpt_partition`` owner; the scores are kept on every rank until then (8 B per bin).  ``default_args``: as for
    ``run_shard``.  ``mark(label)`` is called on the host at "score:<name>", "null:<name>", "done:<name>", "solve" and
    "end".  Returns dict(names, lengths, budgets, gammas (dicts by name), defaults (null details and gamma meta by name,
    budget_meta), my_names (this rank's chromosomes, genome order), d_masks, offsets, results, runs): ``my_names`` and
    ``runs`` go straight to ``distributed.write_genome_bed``."""
    from .distributed import world
    from .rocco import _resolve_budgets, _resolve_chrom_gamma
    args = _default_flow_args(default_args)
    mark = mark or (lambda label: None)
    prm = params if params is not None else score_params()
    names, lengths, scores, nulls = [], [], [], {}
    for name, x in chroms:
        name = str(name)
        if name in nulls:
            raise ValueError(f"default flow: {name} comes twice")
        mark(f"score:{name}")
        s, centered, window = _score_sample_sharded_agreed(x, m_total, prm, group, name)
        del x
        mark(f"null:{name}")
        _, det = budget_null_sample_sharded(centered, s, params=prm, group=group, dependence_lag_hint=window,
                                            num_null_draws=args["num_null_draws"], random_seed=args["random_seed"],
                                            random_streams=args["random_streams"])
        del centered
        mark(f"done:{name}")
        names.append(name)
        lengths.append(int(s.shape[0]))
        scores.append(s)
        nulls[name] = det
    if not names:
        raise ValueError("default flow: the genome has no chromosome")
    cache = {c: {"budget_count_hat": nulls[c]["effective_count"], "total_count": nulls[c]["effective_total_count"]}
             for c in names}
    budgets, budget_meta = _resolve_budgets(cache, args)
    pairs = {c: _resolve_chrom_gamma(c, {"gamma": None}, None, nulls[c]) for c in names}
    gammas = {c: g for c, (g, _) in pairs.items()}
    mark("solve")
    rank, size = world(group)
    mine = lpt_partition(lengths, size)[rank]
    mine_scores = [scores[k] for k in mine]
    del scores
    my_names = [names[k] for k in mine]
    out = {"names": names, "lengths": lengths, "budgets": budgets, "gammas": gammas, "my_names": my_names,
           "defaults": {"null": nulls, "gamma_meta": {c: m for c, (_, m) in pairs.items()}, "budget_meta": budget_meta},
           "d_masks": None, "offsets": [], "results": [],
           "runs": (np.zeros(0, np.int32), np.zeros(0, np.int64), np.zeros(0, np.int64))}
    if my_names:
        d_scores, offsets, my_lengths = pack_scores(mine_scores)
        del mine_scores
        d_masks, results = solve_packed(d_scores, offsets, my_lengths, [budgets[c] for c in my_names],
                                        [gammas[c] for c in my_names], levels_per_round=levels_per_round)
        out.update(d_masks=d_masks, offsets=offsets, results=results, runs=masks_to_runs(d_masks, offsets, my_lengths))
    mark("end")
    return out


# ------------------------------------------------------------------ column statistics on device tensors
_DISPERSION_METHODS = ("mad", "iqr", "std", "tstd")


def _column_stat_spec(method, quantile=0.50, tprop=0.05, rng=(25, 75)) -> tuple[int, float, float, bool]:
    """(stat code, arg0, arg1, dispersion) of a method of ``score_central_tendency_chrom`` or ``score_dispersion_chrom``
    (``median`` = quantile 0.5), normalised as those functions do."""
    from .rocco import _STAT, _central_tendency_stat, _dispersion_stat, _normalize_method
    method_ = _normalize_method(method)
    if method_ in _DISPERSION_METHODS:
        stat, arg0, arg1 = _dispersion_stat(method, rng, tprop)
        return _STAT[stat], float(arg0), float(arg1), True
    stat, arg0, arg1 = _central_tendency_stat("quantile" if method_ == "median" else method,
                                              0.50 if method_ == "median" else quantile, tprop)
    return _STAT[stat], float(arg0), float(arg1), False


def _column_stat_launch(d_matrix, code: int, arg0: float, arg1: float, power: float, out):
    torch = _torch()
    lib = _lib.load()
    m, n = d_matrix.shape
    with torch.cuda.device(d_matrix.device):
        st = lib.rocco_b200_column_stat_dev(
            ctypes.c_void_p(d_matrix.data_ptr()), 1 if d_matrix.dtype == torch.float32 else 0, int(m), int(n), int(code),
            float(arg0), float(arg1), float(power), ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(_stream_ptr(d_matrix.device)))
    _lib.check(st, "column statistic")
    return out


def _column_matrix_problem(x) -> Optional[str]:
    torch = _torch()
    if not isinstance(x, torch.Tensor) or x.dim() != 2 or not x.is_cuda or not x.is_contiguous() \
            or x.dtype not in (torch.float32, torch.float64):
        return "the matrix must be a contiguous two-dimensional float32 or float64 CUDA tensor"
    return None


def column_stat_device(d_matrix, method="quantile", quantile=0.50, tprop=0.05, rng=(25, 75), power=1.0, out=None):
    """``score_central_tendency_chrom`` / ``score_dispersion_chrom`` (by ``method``: quantile, median, tmean, mean, mad,
    iqr, std, tstd) of a [samples, bins] float32 or float64 CUDA tensor; returns the [bins] float64 CUDA tensor (``out``
    when given).  Inputs must be finite."""
    torch = _torch()
    problem = _column_matrix_problem(d_matrix)
    if problem:
        raise ValueError(f"`d_matrix`: {problem}")
    code, arg0, arg1, _ = _column_stat_spec(method, quantile, tprop, rng)
    m, n = d_matrix.shape
    if m == 0:
        raise ValueError("`d_matrix` must hold at least one sample")
    if out is None:
        out = torch.empty(n, dtype=torch.float64, device=d_matrix.device)
    elif tuple(out.shape) != (n,) or out.dtype != torch.float64 or out.device != d_matrix.device or not out.is_contiguous():
        raise ValueError("`out` must be a contiguous float64 tensor of one value per bin on the device of `d_matrix`")
    if n == 0:
        return out
    return _column_stat_launch(d_matrix, code, arg0, arg1, power, out)


def column_bin_ranges(n: int, ranks: int) -> list[tuple[int, int]]:
    """The contiguous bin range [lo, hi) each rank owns in ``column_stat_sample_sharded``: equal widths rounded up to a
    multiple of 16 bins, so only the last non-empty range is shorter; ranks past it own nothing."""
    width = -(-(-(-int(n) // int(ranks))) // ALIGN) * ALIGN
    return [(min(q * width, n), min((q + 1) * width, n)) for q in range(ranks)]


def column_pack_ranges(d_rows, ranges):
    """The send buffer of ``column_stat_sample_sharded``: the rows' [m, hi - lo] block of every bin range, row-major,
    one after the other (one strided device copy per range)."""
    torch = _torch()
    m, n = d_rows.shape
    send = torch.empty(m * n, dtype=d_rows.dtype, device=d_rows.device)
    off = 0
    for a, b in ranges:
        if b > a and m > 0:
            send[off: off + m * (b - a)].view(m, b - a).copy_(d_rows[:, a:b])
        off += m * (b - a)
    return send


def column_stat_sample_sharded(d_rows_local, m_total: int, method="quantile", quantile=0.50, tprop=0.05, rng=(25, 75),
                               power=1.0, group=None):
    """``column_stat_device`` with the SAMPLES sharded over the ranks of ``group``: every rank passes its rows
    ``[m_local, bins]`` (ranks in sample order, as ``score_loci_wls_sample_sharded`` takes them) and the same method and
    arguments, and every rank returns the full [bins] float64 track.

    The bins are split into one contiguous range per rank (``column_bin_ranges``).  One ``all_to_all_single`` sends each
    rank's rows of every range to the range's owner, which then holds the complete columns ``[m_total, |range|]`` in global
    sample order, runs the column kernel on them, and one ``all_gather_into_tensor`` hands the track to every rank.  Every
    column is therefore reduced exactly as by the unsharded call, sums included: the result has the same bits.  With the
    gloo backend the two collectives go through host memory."""
    import torch.distributed as dist
    from .distributed import agree, collective_device, world
    torch = _torch()
    x = d_rows_local
    problem = _column_matrix_problem(x)
    problem = f"`d_rows_local`: {problem}" if problem else None
    try:
        code, arg0, arg1, _ = _column_stat_spec(method, quantile, tprop, rng)
    except ValueError as exc:
        problem, code, arg0, arg1 = problem or str(exc), -1, 0.0, 0.0
    rank, size = world(group)
    if size <= 1:
        if problem:
            raise ValueError(problem)
        if x.shape[0] != int(m_total):
            raise ValueError(f"`m_total` ({m_total}) must equal the number of rows ({x.shape[0]}) on a single rank")
        return column_stat_device(x, method, quantile, tprop, rng, power)
    m, n = (int(x.shape[0]), int(x.shape[1])) if problem is None else (0, 0)
    mine = {"m": m, "n": n, "dtype": str(x.dtype) if problem is None else "",
            "agreed": (int(m_total), int(code), float(arg0), float(arg1), float(power))}
    every = agree(problem, mine, group, "column statistic")
    if any(r["agreed"] != mine["agreed"] for r in every):
        raise ValueError("column statistic: every rank must pass the same m_total, method and arguments")
    if any(r["n"] != n or r["dtype"] != mine["dtype"] for r in every):
        raise ValueError(f"column statistic: every rank must hold the same bins and dtype, got "
                         f"{[(r['n'], r['dtype']) for r in every]}")
    rows = [r["m"] for r in every]
    if sum(rows) != int(m_total) or int(m_total) == 0:
        raise ValueError(f"column statistic: the ranks hold {sum(rows)} samples, `m_total` is {m_total}")
    dev = x.device
    ranges = column_bin_ranges(n, size)
    width = max(b - a for a, b in ranges)
    lo, hi = ranges[rank]
    cdev = collective_device(group, dev)
    # send: this rank's [m, |B_q|] block of every range q, back to back; receive: [m_total, |B_rank|] in sample order
    send = column_pack_ranges(x, ranges)
    recv = torch.empty(int(m_total) * (hi - lo), dtype=x.dtype, device=cdev)
    dist.all_to_all_single(recv, send.to(cdev), output_split_sizes=[r * (hi - lo) for r in rows],
                           input_split_sizes=[m * (b - a) for a, b in ranges], group=group)
    del send
    # this rank's range, padded to the common width, and one status slot: a failure is raised on every rank
    part = torch.zeros(width + 1, dtype=torch.float64, device=dev)
    failure = None
    if hi > lo:
        try:
            cols = recv.to(dev).view(int(m_total), hi - lo)
            _column_stat_launch(cols, code, arg0, arg1, power, part[: hi - lo])
            del cols
        except (RuntimeError, ValueError) as exc:
            failure = exc
            part[width] = 1.0
    del recv
    full = torch.empty(size * (width + 1), dtype=torch.float64, device=cdev)
    dist.all_gather_into_tensor(full, part.to(cdev), group=group)
    full = full.view(size, width + 1).to(dev)
    if failure is not None:
        raise failure
    if bool((full[:, width] != 0).any()):
        raise RuntimeError("column statistic: the kernel failed on another rank")
    return full[:, :width].reshape(-1)[:n].contiguous()
