"""The functionals of the reference's string-matching family, same signatures.

Mirrors ``pydrobert.torch.functional`` (functional.py:49-58 of the reference) for the
names backed by ``pydrobert/torch/_string.py`` ("SM" below): argument meaning,
defaults, shapes, dtypes, error messages and the three data-dependent warnings are
the reference's; the numbers come from the sm_100a kernels behind ``torch.ops.b200lev``.

Every function here compiles under ``torch.jit.script`` (the reference scripts its
modules, tests/conftest.py:166-174) and is wrapped in ``torch.jit.script_if_tracing`` as
the reference's are (_compat.py:189,300), so a traced module keeps its shape checks,
group sizes and warnings dynamic instead of baking the example's into the graph.  The
body is therefore TorchScript: no closures, no dict globals, one ``torch.ops.b200lev``
call per step.  In plain eager mode the ``if not torch.jit.is_scripting()`` branches call
the op bodies directly (no dispatcher round trip).

Host tensors: the reference runs wherever its inputs live.  Here a CPU tensor is copied
to the current CUDA device inside the op, the kernels run there and the result is copied
back (``_host.py``).  Without a CUDA device the call raises; there is no CPU
implementation.
"""

import warnings
from typing import Any, Optional, Tuple

import torch

from . import _ops, config

__all__ = [
    "alignment_positions",
    "edit_distance",
    "error_alignment",
    "error_counts",
    "error_rate",
    "fill_after_eos",
    "hard_optimal_completion_distillation_loss",
    "infix_edit_distance",
    "infix_matches",
    "minimum_bayes_risk",
    "minimum_error_rate_loss",
    "optimal_completion",
    "pairwise_edit_distances",
    "pairwise_error_rates",
    "prefix_edit_distances",
    "prefix_error_rates",
    "sequence_log_probs",
    "ctc_greedy_search",
    "beam_search_advance",
    "random_walk_advance",
]

script = torch.jit.script_if_tracing


def _reduction_code(reduction: str) -> int:
    """SM:1250, 1471: the message of a bad ``reduction``; the codes are the C ABI's."""
    if reduction == "none":
        return 0
    elif reduction == "mean":
        return 1
    elif reduction == "sum":
        return 2
    raise RuntimeError(f"'{reduction}' is not a valid value for reduction")


def _warn_flags(flags: torch.Tensor, eos: Optional[int], include_eos: bool, norm: bool,
                prefix: bool) -> None:
    """The data-dependent warnings of SM:202-217, 361-366, 398-404 (one 4-byte read of the
    flag word the kernels wrote: bit 0/1 = a ref/hyp sequence without eos, bit 2 = an empty
    reference)."""
    f = int(flags.item())
    if eos is not None and include_eos:
        if (f & 1) != 0:
            warnings.warn(
                "include_eos=True, but a transcription in ref did not "
                "contain the eos symbol ({}). To suppress this "
                "warning, set warn=False".format(eos)
            )
        if (f & 2) != 0:
            warnings.warn(
                "include_eos=True, but a transcription in hyp did not "
                "contain the eos symbol ({}). To suppress this "
                "warning, set warn=False".format(eos)
            )
    if norm and (f & 4) != 0:
        if prefix:
            warnings.warn(
                "ref contains empty transcripts. Error rates will be "
                "0 for prefixes of length 0, 1 otherwise. To suppress "
                "this warning, set warn=False"
            )
        else:
            warnings.warn(
                "ref contains empty transcripts. Error rates for entries "
                "will be 1 if any insertion and 0 otherwise. To suppress "
                "this warning, set warn=False"
            )


def _string_matching(
    ref: torch.Tensor,
    hyp: torch.Tensor,
    eos: Optional[int],
    include_eos: bool,
    batch_first: bool,
    ins_cost: float,
    del_cost: float,
    sub_cost: float,
    warn: bool,
    norm: bool = False,
    return_prf_dsts: bool = False,
    exclude_last: bool = False,
    padding: int = config.INDEX_PAD_VALUE,
    return_mistakes: bool = False,
    ref_group: int = 1,
) -> torch.Tensor:
    """SM:146-406 for the final and prefix modes (the mask mode is folded into
    :func:`optimal_completion`)."""
    if ref.dim() != 2 or hyp.dim() != 2:
        raise RuntimeError("ref and hyp must be 2 dimensional")
    uniform = (ins_cost == del_cost) and (del_cost == sub_cost) and (sub_cost > 0.0)
    if not uniform and return_mistakes and warn:  # SM:175-180
        warnings.warn(
            "The behaviour for non-uniform error rates has changed after v0.3.0. "
            "Please switch to edit_distance functions for old behaviour. Set "
            "warn=False to suppress this warning"
        )
    if not torch.jit.is_scripting():
        if not _ops.needs_dispatcher():
            out, flags = _ops.string_matching_impl(
                ref, hyp, eos, include_eos, batch_first, float(ins_cost), float(del_cost),
                float(sub_cost), norm, return_prf_dsts, exclude_last, int(padding),
                return_mistakes, ref_group)
            if warn:
                _warn_flags(flags, eos, include_eos, norm, return_prf_dsts)
            return out
    out, flags = torch.ops.b200lev.string_matching(
        ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, norm,
        return_prf_dsts, exclude_last, padding, return_mistakes, ref_group)
    if warn:
        _warn_flags(flags, eos, include_eos, norm, return_prf_dsts)
    return out


@script
def error_rate(
    ref: torch.Tensor,
    hyp: torch.Tensor,
    eos: Optional[int] = None,
    include_eos: bool = False,
    norm: bool = True,
    batch_first: bool = False,
    ins_cost: float = config.DEFT_INS_COST,
    del_cost: float = config.DEFT_DEL_COST,
    sub_cost: float = config.DEFT_SUB_COST,
    warn: bool = True,
) -> torch.Tensor:
    """Functional version of ErrorRate (SM:409-434)."""
    return _string_matching(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost,
                            sub_cost, warn, norm, False, False, config.INDEX_PAD_VALUE, True, 1)


@script
def edit_distance(
    ref: torch.Tensor,
    hyp: torch.Tensor,
    eos: Optional[int] = None,
    include_eos: bool = False,
    norm: bool = False,
    batch_first: bool = False,
    ins_cost: float = config.DEFT_INS_COST,
    del_cost: float = config.DEFT_DEL_COST,
    sub_cost: float = config.DEFT_SUB_COST,
    warn: bool = True,
) -> torch.Tensor:
    """Functional version of EditDistance (SM:437-461)."""
    return _string_matching(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost,
                            sub_cost, warn, norm, False, False, config.INDEX_PAD_VALUE, False, 1)


@script
def prefix_error_rates(
    ref: torch.Tensor,
    hyp: torch.Tensor,
    eos: Optional[int] = None,
    include_eos: bool = True,
    norm: bool = True,
    batch_first: bool = False,
    ins_cost: float = config.DEFT_INS_COST,
    del_cost: float = config.DEFT_DEL_COST,
    sub_cost: float = config.DEFT_SUB_COST,
    padding: int = config.INDEX_PAD_VALUE,
    exclude_last: bool = False,
    warn: bool = True,
) -> torch.Tensor:
    """Functional version of PrefixErrorRates (SM:520-550)."""
    return _string_matching(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost,
                            sub_cost, warn, norm, True, exclude_last, padding, True, 1)


@script
def prefix_edit_distances(
    ref: torch.Tensor,
    hyp: torch.Tensor,
    eos: Optional[int] = None,
    include_eos: bool = True,
    norm: bool = False,
    batch_first: bool = False,
    ins_cost: float = config.DEFT_INS_COST,
    del_cost: float = config.DEFT_DEL_COST,
    sub_cost: float = config.DEFT_SUB_COST,
    padding: int = config.INDEX_PAD_VALUE,
    exclude_last: bool = False,
    warn: bool = True,
) -> torch.Tensor:
    """Functional version of PrefixEditDistances (SM:553-583)."""
    return _string_matching(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost,
                            sub_cost, warn, norm, True, exclude_last, padding, False, 1)


def _error_path(
    ref: torch.Tensor,
    hyp: torch.Tensor,
    eos: Optional[int],
    include_eos: bool,
    batch_first: bool,
    ins_cost: float,
    del_cost: float,
    sub_cost: float,
    warn: bool,
    align: bool,
) -> torch.Tensor:
    """:func:`error_alignment` if ``align`` else :func:`error_counts`."""
    if ref.dim() != 2 or hyp.dim() != 2:
        raise RuntimeError("ref and hyp must be 2 dimensional")
    if not torch.jit.is_scripting():
        if not _ops.needs_dispatcher():
            out, flags = _ops.error_path_impl(ref, hyp, eos, include_eos, batch_first,
                                              float(ins_cost), float(del_cost), float(sub_cost), align)
            if warn:
                _warn_flags(flags, eos, include_eos, False, False)
            return out
    if align:
        out, flags = torch.ops.b200lev.error_alignment(ref, hyp, eos, include_eos, batch_first,
                                                       ins_cost, del_cost, sub_cost)
    else:
        out, flags = torch.ops.b200lev.error_counts(ref, hyp, eos, include_eos, batch_first,
                                                    ins_cost, del_cost, sub_cost)
    if warn:
        _warn_flags(flags, eos, include_eos, False, False)
    return out


@script
def error_counts(
    ref: torch.Tensor,
    hyp: torch.Tensor,
    eos: Optional[int] = None,
    include_eos: bool = False,
    batch_first: bool = False,
    ins_cost: float = config.DEFT_INS_COST,
    del_cost: float = config.DEFT_DEL_COST,
    sub_cost: float = config.DEFT_SUB_COST,
    warn: bool = True,
) -> torch.Tensor:
    """Per pair the correct, substitution, deletion and insertion counts (sclite's C/S/D/I):
    ``(N, 4)`` long, columns in that order.

    They are the op counts along the path that :func:`error_rate` counts its errors on
    (SM:292-314: every cell takes the substitution candidate unless the insertion candidate is
    smaller, then the deletion candidate only if it is smaller still), also for uniform costs.
    Lengths follow ``eos`` / ``include_eos`` as in :func:`error_rate`, so ``C + S + D`` is the
    reference length, ``C + S + I`` the hypothesis length and ``S + D + I`` equals
    ``error_rate(..., norm=False)`` with the same costs.  ``warn`` covers the two missing-eos
    warnings."""
    return _error_path(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, warn,
                       False)


@script
def error_alignment(
    ref: torch.Tensor,
    hyp: torch.Tensor,
    eos: Optional[int] = None,
    include_eos: bool = False,
    batch_first: bool = False,
    ins_cost: float = config.DEFT_INS_COST,
    del_cost: float = config.DEFT_DEL_COST,
    sub_cost: float = config.DEFT_SUB_COST,
    warn: bool = True,
) -> torch.Tensor:
    """Per pair the edit operations along the path :func:`error_counts` counts: int8
    ``(R + H, N)``, or ``(N, R + H)`` with ``batch_first``, where R and H are the padded lengths.

    Step ``k`` of a pair is 0 (correct), 1 (substitution), 2 (deletion) or 3 (insertion), in
    forward order from the start of both sequences; steps from the path length ``r + I`` on hold
    -1.  Per pair the histogram of the ops equals :func:`error_counts` with the same arguments.
    Arguments, lengths and warnings are those of :func:`error_counts`.  The output's shape
    depends on the input shapes only, so the call reads nothing back to the host (with
    ``warn=False``).  :func:`alignment_positions` maps the steps to token positions."""
    return _error_path(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, warn,
                       True)


def _infix(
    ref: torch.Tensor,
    hyp: torch.Tensor,
    eos: Optional[int],
    include_eos: bool,
    norm: bool,
    batch_first: bool,
    ins_cost: float,
    del_cost: float,
    sub_cost: float,
    warn: bool,
    spans: bool,
) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """:func:`infix_matches` if ``spans`` else :func:`infix_edit_distance` (empty bounds)."""
    if ref.dim() != 2 or hyp.dim() != 2:
        raise RuntimeError("ref and hyp must be 2 dimensional")
    if not torch.jit.is_scripting():
        if not _ops.needs_dispatcher():
            dist, start, end, flags = _ops.infix_impl(ref, hyp, eos, include_eos, batch_first, float(ins_cost),
                                                      float(del_cost), float(sub_cost), norm, spans)
            if warn:
                _warn_flags(flags, eos, include_eos, norm, False)
            return dist, start, end
    dist, start, end, flags = torch.ops.b200lev.infix(ref, hyp, eos, include_eos, batch_first, ins_cost,
                                                      del_cost, sub_cost, norm, spans)
    if warn:
        _warn_flags(flags, eos, include_eos, norm, False)
    return dist, start, end


@script
def infix_edit_distance(
    ref: torch.Tensor,
    hyp: torch.Tensor,
    eos: Optional[int] = None,
    include_eos: bool = False,
    norm: bool = False,
    batch_first: bool = False,
    ins_cost: float = config.DEFT_INS_COST,
    del_cost: float = config.DEFT_DEL_COST,
    sub_cost: float = config.DEFT_SUB_COST,
    warn: bool = True,
) -> torch.Tensor:
    """The cheapest alignment of each whole reference against any contiguous stretch
    ``hyp[s:e]`` of its hypothesis: fp32 ``(N,)``.  Leading and trailing hypothesis tokens cost
    nothing (edlib's "HW" mode).

    The value is the minimum over ``0 <= s <= e <= h`` of :func:`edit_distance` of the reference
    against ``hyp[s:e]``, bit for bit.  Arguments, lengths, costs and warnings are those of
    :func:`edit_distance`; ``norm`` divides by the reference length as it does there, and an
    empty reference has distance 0.  For free ends on the reference side instead, swap ``ref``
    and ``hyp`` and swap ``ins_cost`` with ``del_cost``.  The output's shape depends on the input
    shapes only, so the call reads nothing back to the host (with ``warn=False``)."""
    return _infix(ref, hyp, eos, include_eos, norm, batch_first, ins_cost, del_cost, sub_cost, warn,
                  False)[0]


@script
def infix_matches(
    ref: torch.Tensor,
    hyp: torch.Tensor,
    eos: Optional[int] = None,
    include_eos: bool = False,
    batch_first: bool = False,
    ins_cost: float = config.DEFT_INS_COST,
    del_cost: float = config.DEFT_DEL_COST,
    sub_cost: float = config.DEFT_SUB_COST,
    warn: bool = True,
) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """Where each reference matches inside its hypothesis: ``(dist, start, end)``, fp32 and two
    int64 ``(N,)``.

    ``dist`` is :func:`infix_edit_distance` (``norm=False``) and the match is
    ``hyp[start:end]``: :func:`edit_distance` of the reference against it equals ``dist``.
    ``end`` is the first hypothesis position at which the minimum is reached and ``start`` the
    latest start of an optimal alignment ending there.  An empty reference gives ``(0, 0, 0)``,
    an empty hypothesis ``(r * del_cost, 0, 0)``.  Arguments, lengths and warnings are those of
    :func:`infix_edit_distance`."""
    return _infix(ref, hyp, eos, include_eos, False, batch_first, ins_cost, del_cost, sub_cost, warn,
                  True)


@script
def alignment_positions(ops: torch.Tensor, batch_first: bool = False) -> Tuple[torch.Tensor, torch.Tensor]:
    """The token positions the steps of :func:`error_alignment` consume: ``(ref_pos, hyp_pos)``,
    int64, shaped like ``ops``.

    ``ref_pos[k]`` is the index of the reference token step ``k`` consumes (correct,
    substitution or deletion), -1 for an insertion and for padding; ``hyp_pos[k]`` the index of
    the hypothesis token (correct, substitution or insertion), -1 for a deletion and for
    padding.  Gathering the tokens at both turns the ops into confusion pairs or display
    columns."""
    dim = 1 if batch_first else 0
    on_ref = (ops >= 0) & (ops != 3)
    on_hyp = (ops >= 0) & (ops != 2)
    ref_pos = (on_ref.long().cumsum(dim) - 1).masked_fill(~on_ref, -1)
    hyp_pos = (on_hyp.long().cumsum(dim) - 1).masked_fill(~on_hyp, -1)
    return ref_pos, hyp_pos


def _pairwise(
    ref: torch.Tensor,
    hyp: torch.Tensor,
    eos: Optional[int],
    include_eos: bool,
    norm: bool,
    batch_first: bool,
    ins_cost: float,
    del_cost: float,
    sub_cost: float,
    warn: bool,
    return_mistakes: bool,
) -> torch.Tensor:
    if ref.dim() != 3 or hyp.dim() != 3:
        raise RuntimeError("ref and hyp must be 3 dimensional")
    if ref.size(0 if batch_first else 1) != hyp.size(0 if batch_first else 1):
        raise RuntimeError("ref and hyp group dimensions must match")
    uniform = (ins_cost == del_cost) and (del_cost == sub_cost) and (sub_cost > 0.0)
    if not uniform and return_mistakes and warn:  # SM:175-180
        warnings.warn(
            "The behaviour for non-uniform error rates has changed after v0.3.0. "
            "Please switch to edit_distance functions for old behaviour. Set "
            "warn=False to suppress this warning"
        )
    if not torch.jit.is_scripting():
        if not _ops.needs_dispatcher():
            out, flags = _ops.pairwise_impl(ref, hyp, eos, include_eos, batch_first, float(ins_cost),
                                            float(del_cost), float(sub_cost), norm, return_mistakes)
            if warn:
                _warn_flags(flags, eos, include_eos, norm, False)
            return out
    out, flags = torch.ops.b200lev.pairwise(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost,
                                            sub_cost, norm, return_mistakes)
    if warn:
        _warn_flags(flags, eos, include_eos, norm, False)
    return out


@script
def pairwise_error_rates(
    ref: torch.Tensor,
    hyp: torch.Tensor,
    eos: Optional[int] = None,
    include_eos: bool = False,
    norm: bool = True,
    batch_first: bool = False,
    ins_cost: float = config.DEFT_INS_COST,
    del_cost: float = config.DEFT_DEL_COST,
    sub_cost: float = config.DEFT_SUB_COST,
    warn: bool = True,
) -> torch.Tensor:
    """Every reference of a group against every hypothesis of it: fp32 ``(G, A, B)``.

    ``ref`` is ``(R, G, A)`` and ``hyp`` ``(H, G, B)`` (``(G, A, R)`` and ``(G, B, H)`` with
    ``batch_first``).  ``out[g, a, b]`` is, bit for bit, :func:`error_rate` of reference
    ``(g, a)`` against hypothesis ``(g, b)`` with the same arguments, without the ``G·A·B`` pairs
    being materialised.  Lengths, costs and warnings are those of :func:`error_rate`.  The output's
    shape depends on the input shapes only, so the call reads nothing back to the host (with
    ``warn=False``)."""
    return _pairwise(ref, hyp, eos, include_eos, norm, batch_first, ins_cost, del_cost, sub_cost,
                     warn, True)


@script
def pairwise_edit_distances(
    ref: torch.Tensor,
    hyp: torch.Tensor,
    eos: Optional[int] = None,
    include_eos: bool = False,
    norm: bool = False,
    batch_first: bool = False,
    ins_cost: float = config.DEFT_INS_COST,
    del_cost: float = config.DEFT_DEL_COST,
    sub_cost: float = config.DEFT_SUB_COST,
    warn: bool = True,
) -> torch.Tensor:
    """:func:`pairwise_error_rates` with :func:`edit_distance` in place of :func:`error_rate`:
    ``out[g, a, b]`` is, bit for bit, :func:`edit_distance` of reference ``(g, a)`` against
    hypothesis ``(g, b)``."""
    return _pairwise(ref, hyp, eos, include_eos, norm, batch_first, ins_cost, del_cost, sub_cost,
                     warn, False)


@script
def minimum_bayes_risk(
    log_probs: torch.Tensor,
    hyp: torch.Tensor,
    eos: Optional[int] = None,
    include_eos: bool = True,
    batch_first: bool = False,
    norm: bool = True,
    ins_cost: float = config.DEFT_INS_COST,
    del_cost: float = config.DEFT_DEL_COST,
    sub_cost: float = config.DEFT_SUB_COST,
    warn: bool = True,
) -> Tuple[torch.Tensor, torch.Tensor]:
    """Minimum-Bayes-risk selection from n-best lists: ``(best, risk)``.

    ``hyp`` is ``(H, N, M)`` (``(N, M, H)`` with ``batch_first``): N lists of M hypotheses, with
    model scores ``log_probs`` ``(N, M)``.  Each hypothesis is scored against every other one of
    its list, which stands in for the reference::

        risk[n, i] = sum_j softmax(log_probs[n])_j * er(ref=hyp[n, j], hyp=hyp[n, i])

    where ``er`` is :func:`pairwise_error_rates` with these arguments (with ``norm=False``,
    :func:`pairwise_edit_distances`).  ``best`` (int64 ``(N,)``) is the arg min of ``risk``, equal
    risks going to the lowest index.  ``risk`` has the dtype of ``log_probs`` and is accumulated
    in fp32 (fp64 for fp64 ``log_probs``); identical hypotheses get identical risks.  A ``-inf``
    log-probability gives its hypothesis zero weight.  The defaults are those of
    :func:`minimum_error_rate_loss`.

    For decoding only: neither output carries a gradient."""
    if log_probs.dim() != 2:
        raise RuntimeError("log_probs must be 2 dimensional")
    if hyp.dim() != 3:
        raise RuntimeError("hyp must be 3 dimensional")
    if batch_first:
        batch_size, samples = hyp.size(0), hyp.size(1)
    else:
        batch_size, samples = hyp.size(1), hyp.size(2)
    if log_probs.size(0) != batch_size or log_probs.size(1) != samples:
        raise RuntimeError("ref and hyp batch_size and sample dimensions must match")
    if samples < 1:
        raise RuntimeError(f"Batch must have at least one sample, got {samples}")
    uniform = (ins_cost == del_cost) and (del_cost == sub_cost) and (sub_cost > 0.0)
    if not uniform and norm and warn:  # SM:175-180 (the error-rate form)
        warnings.warn(
            "The behaviour for non-uniform error rates has changed after v0.3.0. "
            "Please switch to edit_distance functions for old behaviour. Set "
            "warn=False to suppress this warning"
        )
    lp = log_probs.detach()
    if not torch.jit.is_scripting():
        if not _ops.needs_dispatcher():
            best, risk, flags = _ops.minimum_bayes_risk_impl(lp, hyp, eos, include_eos, batch_first, norm,
                                                             float(ins_cost), float(del_cost),
                                                             float(sub_cost))
            if warn:
                _warn_flags(flags, eos, include_eos, norm, False)
            return best, risk
    best, risk, flags = torch.ops.b200lev.minimum_bayes_risk(lp, hyp, eos, include_eos, batch_first, norm,
                                                             ins_cost, del_cost, sub_cost)
    if warn:
        _warn_flags(flags, eos, include_eos, norm, False)
    return best, risk


def _optimal_completion(
    ref: torch.Tensor,
    hyp: torch.Tensor,
    eos: Optional[int],
    include_eos: bool,
    batch_first: bool,
    ins_cost: float,
    del_cost: float,
    sub_cost: float,
    padding: int,
    exclude_last: bool,
    warn: bool,
) -> torch.Tensor:
    if ref.dim() != 2 or hyp.dim() != 2:
        raise RuntimeError("ref and hyp must be 2 dimensional")
    if not torch.jit.is_scripting():
        if not _ops.needs_dispatcher():
            out, flags = _ops.optimal_completion_impl(
                ref, hyp, eos, include_eos, batch_first, float(ins_cost), float(del_cost),
                float(sub_cost), int(padding), exclude_last)
            if warn:
                _warn_flags(flags, eos, include_eos, False, False)
            return out
    out, flags = torch.ops.b200lev.optimal_completion(
        ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, padding,
        exclude_last)
    if warn:
        _warn_flags(flags, eos, include_eos, False, False)
    return out


@script
def optimal_completion(
    ref: torch.Tensor,
    hyp: torch.Tensor,
    eos: Optional[int] = None,
    include_eos: bool = True,
    batch_first: bool = False,
    ins_cost: float = config.DEFT_INS_COST,
    del_cost: float = config.DEFT_DEL_COST,
    sub_cost: float = config.DEFT_SUB_COST,
    padding: int = config.INDEX_PAD_VALUE,
    exclude_last: bool = False,
    warn: bool = True,
) -> torch.Tensor:
    """Functional version of OptimalCompletion (SM:464-517)."""
    return _optimal_completion(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost,
                               sub_cost, padding, exclude_last, warn)


@script
def hard_optimal_completion_distillation_loss(
    logits: torch.Tensor,
    ref: torch.Tensor,
    hyp: torch.Tensor,
    eos: Optional[int] = None,
    include_eos: bool = True,
    batch_first: bool = False,
    ins_cost: float = config.DEFT_INS_COST,
    del_cost: float = config.DEFT_DEL_COST,
    sub_cost: float = config.DEFT_SUB_COST,
    weight: Optional[torch.Tensor] = None,
    reduction: str = "mean",
    ignore_index: int = -2,
    warn: bool = True,
) -> torch.Tensor:
    """Functional version of HardOptimalCompletionDistillationLoss (SM:1188-1251)."""
    if logits.dim() != 3:
        raise RuntimeError("logits must be 3 dimensional")
    if logits.shape[:-1] != hyp.shape:
        raise RuntimeError("first two dims of logits must match hyp shape")
    if include_eos:
        if eos is not None and ((eos < 0) or (eos >= logits.size(-1))):
            raise RuntimeError(f"If include_eos=True, eos ({eos}) must be a class idx")
        if eos is not None and eos == ignore_index:
            raise RuntimeError(f"If include_eos=True, eos cannot equal ignore_index ({eos}")
    code = _reduction_code(reduction)
    optimals = _optimal_completion(ref, hyp, eos, include_eos, batch_first, ins_cost, del_cost,
                                   sub_cost, ignore_index, True, warn)  # SM:1216-1228
    if not torch.jit.is_scripting():
        if not _ops.needs_dispatcher():
            return _ops.ocd_loss_eager(logits, optimals, weight, ignore_index, code, 1 if batch_first else 0)
    loss, _, _ = torch.ops.b200lev.ocd_loss(logits, optimals, weight, ignore_index, code,
                                            1 if batch_first else 0)
    return loss


@script
def minimum_error_rate_loss(
    log_probs: torch.Tensor,
    ref: torch.Tensor,
    hyp: torch.Tensor,
    eos: Optional[int] = None,
    include_eos: bool = True,
    sub_avg: bool = True,
    batch_first: bool = False,
    norm: bool = True,
    ins_cost: float = config.DEFT_INS_COST,
    del_cost: float = config.DEFT_DEL_COST,
    sub_cost: float = config.DEFT_SUB_COST,
    reduction: str = "mean",
    warn: bool = True,
) -> torch.Tensor:
    """Functional version of MinimumErrorRateLoss (SM:1400-1472).

    A 2-D ``ref`` is NOT physically repeated over the samples (SM:1426, 1439): the
    kernels read reference column ``pair // samples`` instead."""
    if log_probs.dim() != 2:
        raise RuntimeError("log_probs must be 2 dimensional")
    if hyp.dim() != 3:
        raise RuntimeError("hyp must be 3 dimensional")
    if ref.dim() != 2 and ref.dim() != 3:
        raise RuntimeError("ref must be 2 or 3 dimensional")
    if batch_first:
        batch_size, samples, max_hyp_steps = hyp.size(0), hyp.size(1), hyp.size(2)
        ref_batch = ref.size(0)
        ref_samples = ref.size(1) if ref.dim() == 3 else samples
    else:
        max_hyp_steps, batch_size, samples = hyp.size(0), hyp.size(1), hyp.size(2)
        ref_batch = ref.size(1)
        ref_samples = ref.size(2) if ref.dim() == 3 else samples
    if (ref_batch != batch_size or ref_samples != samples or log_probs.size(0) != batch_size
            or log_probs.size(1) != samples):
        raise RuntimeError("ref and hyp batch_size and sample dimensions must match")
    if samples < 2:
        raise RuntimeError(f"Batch must have at least two samples, got {samples}")
    code = _reduction_code(reduction)
    group = samples if ref.dim() == 2 else 1
    if batch_first:
        hyp2 = hyp.reshape(-1, max_hyp_steps)
        ref2 = ref if ref.dim() == 2 else ref.reshape(-1, ref.size(-1))
    else:
        hyp2 = hyp.reshape(max_hyp_steps, -1)
        ref2 = ref if ref.dim() == 2 else ref.reshape(ref.size(0), -1)
    er = _string_matching(ref2, hyp2, eos, include_eos, batch_first, ins_cost, del_cost, sub_cost,
                          warn, norm, False, False, 0, True, group)  # SM:1451-1462
    if not torch.jit.is_scripting():
        if not _ops.needs_dispatcher():
            return _ops.mwer_loss_eager(er, log_probs, sub_avg, code)
    return torch.ops.b200lev.mwer_loss(er, log_probs, sub_avg, code)


@script
def fill_after_eos(
    tokens: torch.Tensor,
    eos: int,
    dim: int = 0,
    fill: Optional[float] = None,
    value: Optional[torch.Tensor] = None,
) -> torch.Tensor:
    """Functional version of FillAfterEndOfSequence (SM:30-42)."""
    out = tokens if value is None else value
    fill_ = float(eos) if fill is None else fill
    fill_mask = torch.ops.b200lev.after_eos_mask(tokens, eos, dim)
    return out.masked_fill(fill_mask, fill_)


def _prod(sizes: Tuple[int, ...]) -> int:
    n = 1
    for s in sizes:
        n *= s
    return n


@script
def _sequence_log_probs_tensor(logits: torch.Tensor, hyp: torch.Tensor, dim: int,
                               eos: Optional[int]) -> torch.Tensor:
    """_decoding.py:1516-1548"""
    hyp_dim = hyp.dim()
    if dim < -hyp_dim or dim > hyp_dim - 1:  # _decoding.py:1521-1525
        raise RuntimeError(
            "Dimension out of range (expected to be in range of [{}, {}], but "
            "got {})".format(-hyp_dim, hyp_dim - 1, dim)
        )
    dim = (hyp_dim + dim) % hyp_dim
    if logits.dim() != hyp_dim + 1 or logits.shape[:-1] != hyp.shape:
        raise RuntimeError(
            "logits must have the shape of hyp plus a class axis: got {} and {}".format(
                logits.shape, hyp.shape))
    if not logits.is_floating_point():
        raise RuntimeError("logits must be floating point")
    outer, inner = 1, 1
    for i in range(dim):
        outer *= hyp.size(i)
    for i in range(dim + 1, hyp_dim):
        inner *= hyp.size(i)
    T, V = hyp.size(dim), logits.size(-1)
    out_shape = hyp.shape[:dim] + hyp.shape[dim + 1:]
    logits4 = logits.contiguous().view(outer, T, inner, V)
    hyp3 = hyp.to(torch.long).contiguous().view(outer, T, inner)
    if not torch.jit.is_scripting():
        if not (_ops.needs_dispatcher() or _ops.wants_grad(logits)):
            out, _, _ = _ops.sequence_log_probs_impl(logits4, hyp3, eos)
            return out.view(out_shape)
    out, _, _ = torch.ops.b200lev.sequence_log_probs(logits4, hyp3, eos)
    return out.view(out_shape)


@script
def _sequence_log_probs_packed(
        logits: Tuple[torch.Tensor, torch.Tensor, Optional[torch.Tensor], Optional[torch.Tensor]],
        hyp: torch.Tensor, dim: int) -> torch.Tensor:
    """_decoding.py:1551-1586: ``logits`` is a PackedSequence (data ``(sum(lens), V)``, batch
    sizes per step, sorting permutations) of per-step distributions and ``hyp`` the ``(T, N)``
    (``dim == 0``) or ``(N, T)`` (``dim == 1``) token matrix of the same sequences in their
    original order.

    The packed data is a ragged view of a padded ``(T, N, V)`` tensor: a step that a sequence
    does not have contributes nothing.  That is exactly what the tensor kernel does with a
    token outside ``[0, V)``, so the packed rows are gathered into the padded layout (one
    ``index_select``: its backward scatters the padded gradient back), the steps beyond a
    sequence's length get token -1, and the tensor path does the rest."""
    hyp_dim = hyp.dim()
    if dim < -hyp_dim or dim > hyp_dim - 1:
        raise RuntimeError(
            "Dimension out of range (expected to be in range of [{}, {}], but "
            "got {})".format(-hyp_dim, hyp_dim - 1, dim)
        )
    if hyp_dim != 2:
        raise RuntimeError("hyp must be 2 dimensional when logits is a PackedSequence")
    dim = (hyp_dim + dim) % hyp_dim
    data, batch_sizes, sidxs, uidxs = logits
    dev = data.device
    bs = batch_sizes.to(device=dev, dtype=torch.long)  # (T,) sequences alive at step t, descending
    T = bs.size(0)
    N = hyp.size(1 - dim)
    if T == 0 or N == 0:
        return torch.zeros(N, dtype=data.dtype, device=dev)
    # row of `data` that holds step t of the n-th LONGEST sequence (clamped where it has none)
    first = torch.cumsum(bs, 0) - bs
    n_idx = torch.arange(N, device=dev)
    alive = n_idx.unsqueeze(0) < bs.unsqueeze(1)  # (T, N)
    rows = first.unsqueeze(1) + torch.min(n_idx.unsqueeze(0), (bs - 1).clamp_min(0).unsqueeze(1))
    padded = data.index_select(0, rows.flatten()).view(T, N, data.size(1))
    # the hypotheses in the same (sorted) order, steps x sequences, -1 beyond a sequence's length
    h = hyp.to(dev)
    if dim == 1:
        h = h.t()
    if sidxs is not None:
        h = h.index_select(1, sidxs.to(dev))
    if h.size(0) >= T:
        h = h[:T]
    else:
        h = torch.cat([h, h.new_full((T - h.size(0), N), -1)], 0)
    h = h.masked_fill(~alive, -1)
    out = _sequence_log_probs_tensor(padded, h, 0, None)
    if uidxs is not None:
        out = out.index_select(0, uidxs.to(dev))
    return out


@script
def sequence_log_probs(logits: Any, hyp: torch.Tensor, dim: int = 0, eos: Optional[int] = None
                       ) -> torch.Tensor:
    """Functional version of SequenceLogProbabilities (_decoding.py:1516-1633): joint
    log-probability of the token sequences in ``hyp`` (``(A*, T, B*)``, step axis ``dim``) under
    the categorical distributions ``logits`` (``(A*, T, B*, V)``, or a PackedSequence of
    ``(T, N)`` / ``(N, T)`` sequences).  Tokens outside ``[0, V)`` are padding; with ``eos`` the
    first eos step is the last one counted (tensor ``logits`` only, as in the reference).
    Differentiable with respect to ``logits``."""
    if isinstance(logits, torch.Tensor):
        return _sequence_log_probs_tensor(logits, hyp, dim, eos)
    elif torch.jit.isinstance(
            logits, Tuple[torch.Tensor, torch.Tensor, Optional[torch.Tensor], Optional[torch.Tensor]]):
        return _sequence_log_probs_packed(logits, hyp, dim)
    raise RuntimeError("logits must be either a Tensor or PackedSequence")


@script
def ctc_greedy_search(logits: torch.Tensor, in_lens: Optional[torch.Tensor] = None, blank_idx: int = -1,
                      batch_first: bool = False, is_probs: bool = False
                      ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """Functional version of CTCGreedySearch (_decoding.py:507-560): per step the most likely
    class of ``logits`` (``(T, N, V)``, or ``(N, T, V)`` if ``batch_first``); returns the path
    score ``max_ (N,)`` (sum of the chosen log-probabilities; product of the chosen
    probabilities with ``is_probs``), ``paths`` (``(T, N)`` / ``(N, T)`` long: blanks and repeats
    removed, compacted to the front) and ``out_lens (N,)``.  Equal maxima resolve to the lowest
    class index.  ``max_`` is differentiable w.r.t. ``logits``."""
    if logits.dim() != 3:
        raise RuntimeError("logits must be 3-dimensional")
    V = logits.size(2)
    if blank_idx < -V or blank_idx > (V - 1):
        raise RuntimeError(
            "Blank index out of range (expected to be in the range of "
            f"[-{V},{V-1}], but got {blank_idx})"
        )
    if not logits.is_floating_point():
        raise RuntimeError("logits must be floating point")
    blank = (blank_idx + V) % V
    N = logits.size(0) if batch_first else logits.size(1)
    T = logits.size(1) if batch_first else logits.size(0)
    if in_lens is not None:
        if in_lens.dim() != 1 or in_lens.size(0) != N:
            raise RuntimeError(f"in_lens must have shape ({N},)")
    outer = N if batch_first else 1
    inner = 1 if batch_first else N
    logits4 = logits.contiguous().view(outer, T, inner, V)
    if not torch.jit.is_scripting():
        if not (_ops.needs_dispatcher() or _ops.wants_grad(logits)):
            max_, paths, out_lens, _, _, _ = _ops.ctc_greedy_search_impl(logits4, in_lens, blank, is_probs)
            if batch_first:
                return max_.view(N), paths.view(N, T), out_lens.view(N)
            return max_.view(N), paths.view(T, N), out_lens.view(N)
    max_, paths, out_lens, _, _, _ = torch.ops.b200lev.ctc_greedy_search(logits4, in_lens, blank, is_probs)
    if batch_first:
        return max_.view(N), paths.view(N, T), out_lens.view(N)
    return max_.view(N), paths.view(T, N), out_lens.view(N)


@script
def beam_search_advance(
    log_probs_t: torch.Tensor,
    width: int,
    log_probs_prev: torch.Tensor,
    y_prev: torch.Tensor,
    y_prev_lens: Optional[torch.Tensor] = None,
) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """Beam search step function (_decoding.py:41-155): the ``width`` best extensions of the
    ``old_width`` prefixes ``y_prev`` (``(S, N, old_width)``) by one token of ``log_probs_t``
    (``(N, old_width, V)``).  Returns ``(y_next, y_next_lens, log_probs_next, next_src)``.
    Equal candidate scores resolve to the lower ``old_width * V`` index (the reference leaves
    that order to ``torch.topk``); paths beyond ``old_width * V`` get ``-inf``, length 0 and
    source 0, their tokens are zeros (uninitialised in the reference)."""
    if log_probs_t.dim() != 3:
        raise RuntimeError("log_probs_t must be 3 dimensional")
    N, Kp, V = log_probs_t.shape
    if width < 1:
        raise RuntimeError(f"Expected width to be >= 1, got {width}")
    if log_probs_prev.dim() != 2 or log_probs_prev.size(0) != N or log_probs_prev.size(1) != Kp:
        raise RuntimeError(
            f"Expected log_probs_prev to be of shape {(N, Kp)}, got "
            f"{log_probs_prev.shape}"
        )
    if y_prev.dim() != 3:
        raise RuntimeError("y_prev must be 3 dimensional")
    if y_prev.size(1) != N or y_prev.size(2) != Kp:
        raise RuntimeError(
            f"Expected the last two dimensions of y_prev to be {(N, Kp)}, "
            f"got {y_prev.shape[1:]}"
        )
    if y_prev_lens is not None and (y_prev_lens.dim() != 2 or y_prev_lens.size(0) != N
                                    or y_prev_lens.size(1) != Kp):
        raise RuntimeError(
            f"Expected y_prev_lens to have shape {(N, Kp)}, got {y_prev_lens.shape}"
        )
    return torch.ops.b200lev.beam_search_advance(log_probs_t, width, log_probs_prev, y_prev, y_prev_lens)


@script
def random_walk_advance(
    log_probs_t: torch.Tensor,
    log_probs_prev: torch.Tensor,
    y_prev: torch.Tensor,
    y_prev_lens: Optional[torch.Tensor] = None,
) -> Tuple[torch.Tensor, torch.Tensor]:
    """Random walk step function (_decoding.py:1207-1283): one token per path drawn from
    ``exp(log_probs_t)`` (``(N, V)``), appended to ``y_prev`` (``(S, N)``).  Returns
    ``(y_next, log_probs_next)``."""
    if log_probs_t.dim() != 2:
        raise RuntimeError("log_probs_t must be 2-dimensional")
    N, V = log_probs_t.shape
    if log_probs_prev.dim() != 1 or log_probs_prev.size(0) != N:
        raise RuntimeError(
            f"Expected log_probs_prev to be of shape {(N,)}, got {log_probs_prev.shape}"
        )
    if y_prev.dim() != 2:
        raise RuntimeError("y_prev must be 2-dimensional")
    if y_prev.size(1) != N:
        raise RuntimeError(f"Expected dim 1 of y_prev to be {N}, got {y_prev.size(-1)}")
    if y_prev_lens is not None and (y_prev_lens.dim() != 1 or y_prev_lens.size(0) != N):
        raise RuntimeError(
            f"Expected y_prev_lens to have shape {(N,)}, got {y_prev_lens.shape}"
        )
    return torch.ops.b200lev.random_walk_advance(log_probs_t, log_probs_prev, y_prev, y_prev_lens)
