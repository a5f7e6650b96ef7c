"""Multi-GPU plumbing: one process per GPU, points sharded by contiguous index range, ONE all-reduce
(sum) of the partial normal equations before the replicated solve (SURVEY 8e).  Evaluation shards the
queries the same way and needs no communication.

The only collective on the path is `torch.distributed.all_reduce` of the handle's partial buffer
[G in stencil storage | g | node histogram | totlwt | nrows] -- NCCL over NVLink on GPUs; the same
host logic runs over gloo with CPU tensors in the tests.
"""
from __future__ import annotations

import numpy as np


def shard_range(n: int, rank: int, world: int):
    """Contiguous slice [lo, hi) of n items owned by `rank` (remainder spread over the first ranks)."""
    base, rem = divmod(int(n), int(world))
    lo = rank * base + min(rank, rem)
    hi = lo + base + (1 if rank < rem else 0)
    return lo, hi


def partial_layout(ndim: int, nodes, gcv=False):
    """Offsets of the fields inside the partial buffer (float64 counts).  gcv: the handle called enable_gcv, which adds
    the ywy = sum (w y)^2 slot at the end."""
    ncol = int(np.prod(np.asarray(nodes, dtype=np.int64)[:ndim]))
    nst = 4 ** ndim
    off = {"S": (0, ncol * nst), "g": (ncol * nst, ncol * nst + ncol),
           "cnt": (ncol * nst + ncol, ncol * nst + 2 * ncol),
           "totlwt": (ncol * nst + 2 * ncol, ncol * nst + 2 * ncol + 1),
           "nrows": (ncol * nst + 2 * ncol + 1, ncol * nst + 2 * ncol + 2)}
    total = ncol * nst + 2 * ncol + 2
    if gcv:
        off["ywy"] = (total, total + 1)
        total += 1
    return off, total


def allreduce_partials(buf, group=None):
    """In-place sum of the partial buffer across ranks (no-op for a single process)."""
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
    return buf


def _on_handle_stream(handle, fn, stream=None):
    """Run the collective `fn()` ordered against the handle's private stream (on which assembly, compute and refine
    run).  Default: issue it ON that stream.  A caller-chosen `stream` is fenced with events on both sides."""
    import torch

    hs = torch.cuda.ExternalStream(handle.stream())
    if stream is None or getattr(stream, "cuda_stream", None) == hs.cuda_stream:
        with torch.cuda.stream(hs):
            fn()
        return
    before, after = torch.cuda.Event(), torch.cuda.Event()
    before.record(hs)
    stream.wait_event(before)
    with torch.cuda.stream(stream):
        fn()
    after.record(stream)
    hs.wait_event(after)


def fit_sharded(handle, x, y, w, weighted=True, device_resident=False, l1x=None, n=None, group=None, stream=None,
                broadcast_coef=False, select_smoothing=None, prepare_variance=False, criterion="gcv"):
    """Every rank adds ITS shard to `handle`, the partial sums are all-reduced, every rank solves.
    Returns (coef, ierror).  The all-reduce is ordered against the handle's stream (see _on_handle_stream), so no
    host synchronisation is needed around it.  The replicated solves see identical inputs (the all-reduce hands every
    rank the same sums), add their constraint rows through order-independent integer limbs and solve deterministically,
    so the coefficients are bitwise identical on all ranks (tests/test_gpu_multi.py); `broadcast_coef` additionally
    broadcasts rank 0's coefficients (8*ncol bytes) for hosts that want to rule out any divergence, e.g. mixed GPU types.
    `select_smoothing` (a penalty name; the handle must have called enable_gcv): after the all-reduce every rank
    selects lambda by `criterion` ("gcv" or "reml") on the summed buffer -- bit-identical inputs, so every rank selects
    the same lambda -- and the solve is the selected fit.  `prepare_variance`: after the selection (if any) and before the solve, every rank
    builds the posterior-variance tables from the same summed buffer -- bit-identical on every rank, so the queries of
    handle.variance / variance_device then shard without communication.  A refusal raises SplpakError."""
    import torch
    import torch.distributed as dist

    if device_resident:
        rc = handle.add_points_device(x, l1x, y, w, n, weighted)
    else:
        rc = handle.add_points(x, y, w, weighted=weighted)
    if rc != 0:
        return None, rc
    part = handle.partial_tensor()
    _on_handle_stream(handle, lambda: allreduce_partials(part, group), stream)
    if select_smoothing is not None:
        handle.select_smoothing(select_smoothing, criterion=criterion)
    if prepare_variance:
        handle.prepare_variance()
    coef, ierr = handle.compute()
    if broadcast_coef and dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        t = torch.from_numpy(np.ascontiguousarray(coef, dtype=np.float64)).cuda()
        dist.broadcast(t, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        coef = t.cpu().numpy().astype(coef.dtype, copy=False)
    return coef, ierr
