"""Multi-GPU bulk scoring: shard the pair axis, all-reduce three scalars.

The path shards naturally (SURVEY 8e): pairs are independent, so each rank scores a
contiguous block of (batch x n-best) pairs with no data-path communication; the only
exchange is one ``all_reduce(sum)`` of ``[sum(err), sum(ref_tokens), #pairs]`` (fp64,
24 bytes), the pattern of the reference's ``training.py:887-908`` applied to the
accumulation of ``command_line.py:1135-1147``.  With the NCCL backend the buffer never
leaves the device and the collective is enqueued behind the scoring kernels.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
import torch.distributed as dist

from . import _ops
from . import functional as F


def bind_host_to_gpu(device_index: int) -> Optional[int]:
    """Pin this process (one per GPU) to the CPUs of the NUMA node its GPU hangs off, so that
    the page-locked staging buffers of the host-tensor path are allocated next to the PCIe root
    they are copied through.  With 8 ranks copying 212 MB each per step, buffers on the far
    socket cross the inter-socket link and cap the aggregate H2D rate.  Returns the node, or
    None when the topology is not exposed (single socket, containers without sysfs)."""
    import os

    try:
        props = torch.cuda.get_device_properties(device_index)
        bus = "{:04x}:{:02x}:{:02x}.0".format(props.pci_domain_id, props.pci_bus_id,
                                              props.pci_device_id)
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return node
    except (OSError, ValueError, AttributeError):
        return None


def shard_bounds(num_items: int, rank: int, world_size: int, group: int = 1) -> Tuple[int, int]:
    """Contiguous block ``[lo, hi)`` of ``num_items`` for ``rank``; block edges are
    multiples of ``group`` so an n-best group never straddles two ranks (the softmax
    and mean of _string.py:1463-1465 are per group)."""
    if num_items % group:
        raise ValueError(f"{num_items} items are not a multiple of the group size {group}")
    units = num_items // group
    base, rem = divmod(units, world_size)
    lo = rank * base + min(rank, rem)
    hi = lo + base + (1 if rank < rem else 0)
    return lo * group, hi * group


def bulk_error_rate(ref: torch.Tensor, hyp: torch.Tensor, eos: Optional[int] = None,
                    include_eos: bool = False, batch_first: bool = False, ins_cost: float = 1.0,
                    del_cost: float = 1.0, sub_cost: float = 1.0, distances: bool = False,
                    process_group=None, warn: bool = False):
    """Score this rank's pairs and reduce the totals over the process group.

    ``ref`` / ``hyp`` are the LOCAL shard (see :func:`shard_bounds`).  Returns
    ``(per_pair, totals)`` where ``totals = [sum(err), sum(ref_tokens), #pairs]`` is the
    globally reduced fp64 tensor; the corpus-level rate of
    ``compute-torch-token-data-dir-error-rates`` (command_line.py:1141-1147) is
    ``totals[0] / totals[1]`` (or ``/ totals[2]`` with ``distances``).
    """
    # (the plain function: the registered op `b200lev::error_sums` is the same call behind the
    # dispatcher, which costs a strongly scaled step more than its kernel)
    er, acc, flags = _ops.error_sums_impl(ref, hyp, eos, include_eos, batch_first,
                                          float(ins_cost), float(del_cost), float(sub_cost), False,
                                          not distances, 1)
    if warn:
        F._warn_flags(flags, eos, include_eos, False, False)
    if dist.is_available() and dist.is_initialized():
        if dist.get_backend(process_group) == "gloo" and acc.is_cuda:
            host = acc.cpu()
            dist.all_reduce(host, op=dist.ReduceOp.SUM, group=process_group)
            acc = host.to(acc.device)
        else:
            dist.all_reduce(acc, op=dist.ReduceOp.SUM, group=process_group)
    return er, acc


def bulk_error_counts(ref: torch.Tensor, hyp: torch.Tensor, eos: Optional[int] = None,
                      include_eos: bool = False, batch_first: bool = False, ins_cost: float = 1.0,
                      del_cost: float = 1.0, sub_cost: float = 1.0, process_group=None,
                      warn: bool = False):
    """:func:`bulk_error_rate` with the breakdown: score this rank's pairs and reduce the
    counts over the process group.

    Returns ``(per_pair, totals)``: ``per_pair`` is this rank's ``(N, 4)`` int64
    ``(C, S, D, I)`` (:func:`b200lev.functional.error_counts`) and ``totals`` its column sums,
    int64[4], summed over the ranks.  The corpus WER is ``(S + D + I) / (C + S + D)``."""
    per_pair, flags = _ops.error_counts_impl(ref, hyp, eos, include_eos, batch_first,
                                             float(ins_cost), float(del_cost), float(sub_cost))
    if warn:
        F._warn_flags(flags, eos, include_eos, False, False)
    totals = per_pair.sum(0)
    if dist.is_available() and dist.is_initialized():
        if dist.get_backend(process_group) == "gloo" and totals.is_cuda:
            host = totals.cpu()
            dist.all_reduce(host, op=dist.ReduceOp.SUM, group=process_group)
            totals = host.to(totals.device)
        else:
            dist.all_reduce(totals, op=dist.ReduceOp.SUM, group=process_group)
    return per_pair, totals


def score_corpora_sharded(ref, hyp, process_group=None, **score_kwargs):
    """``scoring.score_corpora`` over the ranks of a process group: the aligned corpora are cut
    into contiguous blocks of utterances (:func:`shard_bounds`), every rank scores its block on
    its own GPU, and ONE ``all_reduce(sum)`` of ``[sum(err), sum(ref_tokens), #utterances]``
    (fp64) gives every rank the corpus totals that ``compute-torch-token-data-dir-error-rates``
    prints (command_line.py:1135-1147).

    Returns ``(lo, hi, errors[lo:hi], ref_lens[lo:hi], totals)``.  The token-to-code map is built
    per rank from its block only: the edit distance depends on token equality inside a pair,
    so the blocks do not have to agree on the codes."""
    import numpy as np

    from . import scoring as S

    if ref.utt_ids != hyp.utt_ids:
        raise ValueError("corpora are not aligned (see align_utterances)")
    if dist.is_available() and dist.is_initialized():
        rank, world = dist.get_rank(process_group), dist.get_world_size(process_group)
    else:
        rank, world = 0, 1
    lo, hi = shard_bounds(len(ref), rank, world)
    keep = np.arange(lo, hi, dtype=np.int64)
    errors, rlens = S.score_corpora(ref.select(keep), hyp.select(keep), **score_kwargs)
    totals = torch.tensor([float(errors.astype(np.float64).sum()), float(rlens.sum()), float(hi - lo)],
                          dtype=torch.float64)
    if world > 1:
        if dist.get_backend(process_group) != "gloo":
            totals = totals.to(torch.device("cuda", torch.cuda.current_device()))
        dist.all_reduce(totals, op=dist.ReduceOp.SUM, group=process_group)
    return lo, hi, errors, rlens, totals.cpu()
