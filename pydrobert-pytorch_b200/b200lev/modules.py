"""The eight ``nn.Module`` shells of the reference's string-matching family.

Same constructor signatures, validation (``argcheck``), ``__constants__``,
``extra_repr`` and forward arguments as ``pydrobert.torch.modules`` (modules.py:115-124
of the reference; classes at _string.py:45-134, 680-1166, 1254-1378, 1475-1646).  Each
forward calls the functional of the same name, which dispatches to the sm_100a kernels.
"""

import abc
from typing import Any, Optional, Tuple

import torch

from . import argcheck, config
from . import functional as F

__all__ = [
    "EditDistance",
    "ErrorAlignment",
    "ErrorCounts",
    "ErrorRate",
    "FillAfterEndOfSequence",
    "HardOptimalCompletionDistillationLoss",
    "InfixEditDistance",
    "InfixMatches",
    "MinimumBayesRisk",
    "MinimumErrorRateLoss",
    "OptimalCompletion",
    "PairwiseEditDistances",
    "PairwiseErrorRates",
    "PrefixEditDistances",
    "PrefixErrorRates",
    "SequenceLogProbabilities",
    "CTCGreedySearch",
]

_REDUCTIONS = ("mean", "sum", "none")


class FillAfterEndOfSequence(torch.nn.Module):
    """Fill after the first end-of-sequence token with a value (_string.py:45-134)"""

    __constants__ = "eos", "dim", "fill"

    eos: int
    dim: int
    fill: float

    def __init__(self, eos: int, dim: int = 0, fill: Optional[float] = None) -> None:
        eos = argcheck.is_int(eos, "eos")
        dim = argcheck.is_int(dim, "dim")
        fill = float(eos) if fill is None else argcheck.is_float(fill, "fill")
        super().__init__()
        self.eos, self.dim, self.fill = eos, dim, fill

    def extra_repr(self) -> str:
        return ", ".join(f"{x}={getattr(self, x)}" for x in self.__constants__)

    def forward(self, tokens: torch.Tensor, value: Optional[torch.Tensor] = None) -> torch.Tensor:
        return F.fill_after_eos(tokens, self.eos, self.dim, self.fill, value)


class _StringMatching(torch.nn.Module, metaclass=abc.ABCMeta):
    """_string.py:680-719"""

    __constants__ = ("eos", "include_eos", "batch_first", "ins_cost", "del_cost", "sub_cost", "warn")

    eos: Optional[int]
    include_eos: bool
    batch_first: bool
    ins_cost: float
    del_cost: float
    sub_cost: float
    warn: bool

    def __init__(self, eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, warn):
        eos = argcheck.is_int(eos, "eos", True)
        include_eos = argcheck.is_bool(include_eos, "include_eos")
        batch_first = argcheck.is_bool(batch_first, "batch_first")
        ins_cost = argcheck.is_float(ins_cost, "ins_cost")
        del_cost = argcheck.is_float(del_cost, "del_cost")
        sub_cost = argcheck.is_float(sub_cost, "sub_cost")
        warn = argcheck.is_bool(warn, "warn")
        super().__init__()
        self.eos, self.include_eos, self.batch_first = eos, include_eos, batch_first
        self.ins_cost, self.del_cost, self.sub_cost = ins_cost, del_cost, sub_cost
        self.warn = warn

    def extra_repr(self) -> str:
        return ", ".join(f"{x}={getattr(self, x)}" for x in self.__constants__)

    @abc.abstractmethod
    def forward(self, ref: torch.Tensor, hyp: torch.Tensor) -> torch.Tensor:
        raise NotImplementedError


class EditDistance(_StringMatching):
    """Compute an edit distance over a batch of references and hypotheses
    (_string.py:722-797)"""

    __constants__ = ("eos", "include_eos", "norm", "batch_first", "ins_cost", "del_cost",
                     "sub_cost", "warn")
    norm: bool

    def __init__(self, eos: Optional[int] = None, include_eos: bool = False, norm: bool = False,
                 batch_first: bool = False, ins_cost: float = config.DEFT_INS_COST,
                 del_cost: float = config.DEFT_DEL_COST, sub_cost: float = config.DEFT_SUB_COST,
                 warn: bool = True):
        norm = argcheck.is_bool(norm, "norm")
        super().__init__(eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, warn)
        self.norm = norm

    def forward(self, ref: torch.Tensor, hyp: torch.Tensor) -> torch.Tensor:
        return F.edit_distance(ref, hyp, self.eos, self.include_eos, self.norm, self.batch_first,
                               self.ins_cost, self.del_cost, self.sub_cost, self.warn)


class ErrorAlignment(_StringMatching):
    """The edit operations per pair along the path ErrorCounts counts: int8 ``(R + H, N)``, or
    ``(N, R + H)`` with ``batch_first`` (see :func:`b200lev.functional.error_alignment`)"""

    def __init__(self, eos: Optional[int] = None, include_eos: bool = False, batch_first: bool = False,
                 ins_cost: float = config.DEFT_INS_COST, del_cost: float = config.DEFT_DEL_COST,
                 sub_cost: float = config.DEFT_SUB_COST, warn: bool = True):
        super().__init__(eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, warn)

    def forward(self, ref: torch.Tensor, hyp: torch.Tensor) -> torch.Tensor:
        return F.error_alignment(ref, hyp, self.eos, self.include_eos, self.batch_first, self.ins_cost,
                                 self.del_cost, self.sub_cost, self.warn)


class ErrorCounts(_StringMatching):
    """Correct, substitution, deletion and insertion counts (sclite's C/S/D/I) per pair along
    the path ErrorRate counts its errors on: ``(N, 4)`` long (see
    :func:`b200lev.functional.error_counts`)"""

    def __init__(self, eos: Optional[int] = None, include_eos: bool = False, batch_first: bool = False,
                 ins_cost: float = config.DEFT_INS_COST, del_cost: float = config.DEFT_DEL_COST,
                 sub_cost: float = config.DEFT_SUB_COST, warn: bool = True):
        super().__init__(eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, warn)

    def forward(self, ref: torch.Tensor, hyp: torch.Tensor) -> torch.Tensor:
        return F.error_counts(ref, hyp, self.eos, self.include_eos, self.batch_first, self.ins_cost,
                              self.del_cost, self.sub_cost, self.warn)


class InfixEditDistance(_StringMatching):
    """The cheapest match of each reference anywhere inside its hypothesis: fp32 ``(N,)`` (see
    :func:`b200lev.functional.infix_edit_distance`)"""

    __constants__ = EditDistance.__constants__
    norm: bool

    def __init__(self, eos: Optional[int] = None, include_eos: bool = False, norm: bool = False,
                 batch_first: bool = False, ins_cost: float = config.DEFT_INS_COST,
                 del_cost: float = config.DEFT_DEL_COST, sub_cost: float = config.DEFT_SUB_COST,
                 warn: bool = True):
        norm = argcheck.is_bool(norm, "norm")
        super().__init__(eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, warn)
        self.norm = norm

    def forward(self, ref: torch.Tensor, hyp: torch.Tensor) -> torch.Tensor:
        return F.infix_edit_distance(ref, hyp, self.eos, self.include_eos, self.norm, self.batch_first,
                                     self.ins_cost, self.del_cost, self.sub_cost, self.warn)


class InfixMatches(_StringMatching):
    """Where each reference matches inside its hypothesis: ``(dist, start, end)`` (see
    :func:`b200lev.functional.infix_matches`)"""

    def __init__(self, eos: Optional[int] = None, include_eos: bool = False, batch_first: bool = False,
                 ins_cost: float = config.DEFT_INS_COST, del_cost: float = config.DEFT_DEL_COST,
                 sub_cost: float = config.DEFT_SUB_COST, warn: bool = True):
        super().__init__(eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, warn)

    def forward(self, ref: torch.Tensor, hyp: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        return F.infix_matches(ref, hyp, self.eos, self.include_eos, self.batch_first, self.ins_cost,
                               self.del_cost, self.sub_cost, self.warn)


class ErrorRate(_StringMatching):
    """Calculate error rates over a batch of references and hypotheses
    (_string.py:888-967)"""

    __constants__ = EditDistance.__constants__
    norm: bool

    def __init__(self, eos: Optional[int] = None, include_eos: bool = False, norm: bool = True,
                 batch_first: bool = False, ins_cost: float = config.DEFT_INS_COST,
                 del_cost: float = config.DEFT_DEL_COST, sub_cost: float = config.DEFT_SUB_COST,
                 warn: bool = True):
        norm = argcheck.is_bool(norm, "norm")
        super().__init__(eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, warn)
        self.norm = norm

    def forward(self, ref: torch.Tensor, hyp: torch.Tensor) -> torch.Tensor:
        return F.error_rate(ref, hyp, self.eos, self.include_eos, self.norm, self.batch_first,
                            self.ins_cost, self.del_cost, self.sub_cost, self.warn)


class PairwiseEditDistances(_StringMatching):
    """Every reference of a group against every hypothesis of it, as EditDistance: ``(G, A, B)``
    (see :func:`b200lev.functional.pairwise_edit_distances`)"""

    __constants__ = EditDistance.__constants__
    norm: bool

    def __init__(self, eos: Optional[int] = None, include_eos: bool = False, norm: bool = False,
                 batch_first: bool = False, ins_cost: float = config.DEFT_INS_COST,
                 del_cost: float = config.DEFT_DEL_COST, sub_cost: float = config.DEFT_SUB_COST,
                 warn: bool = True):
        norm = argcheck.is_bool(norm, "norm")
        super().__init__(eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, warn)
        self.norm = norm

    def forward(self, ref: torch.Tensor, hyp: torch.Tensor) -> torch.Tensor:
        return F.pairwise_edit_distances(ref, hyp, self.eos, self.include_eos, self.norm, self.batch_first,
                                         self.ins_cost, self.del_cost, self.sub_cost, self.warn)


class PairwiseErrorRates(_StringMatching):
    """Every reference of a group against every hypothesis of it, as ErrorRate: ``(G, A, B)``
    (see :func:`b200lev.functional.pairwise_error_rates`)"""

    __constants__ = EditDistance.__constants__
    norm: bool

    def __init__(self, eos: Optional[int] = None, include_eos: bool = False, norm: bool = True,
                 batch_first: bool = False, ins_cost: float = config.DEFT_INS_COST,
                 del_cost: float = config.DEFT_DEL_COST, sub_cost: float = config.DEFT_SUB_COST,
                 warn: bool = True):
        norm = argcheck.is_bool(norm, "norm")
        super().__init__(eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, warn)
        self.norm = norm

    def forward(self, ref: torch.Tensor, hyp: torch.Tensor) -> torch.Tensor:
        return F.pairwise_error_rates(ref, hyp, self.eos, self.include_eos, self.norm, self.batch_first,
                                      self.ins_cost, self.del_cost, self.sub_cost, self.warn)


class MinimumBayesRisk(_StringMatching):
    """Minimum-Bayes-risk selection from n-best lists: ``(best, risk)`` for ``log_probs`` ``(N, M)``
    and ``hyp`` ``(H, N, M)`` (see :func:`b200lev.functional.minimum_bayes_risk`; decoding only,
    no gradient)"""

    __constants__ = EditDistance.__constants__
    norm: bool

    def __init__(self, eos: Optional[int] = None, include_eos: bool = True, batch_first: bool = False,
                 norm: bool = True, ins_cost: float = config.DEFT_INS_COST,
                 del_cost: float = config.DEFT_DEL_COST, sub_cost: float = config.DEFT_SUB_COST,
                 warn: bool = True):
        norm = argcheck.is_bool(norm, "norm")
        super().__init__(eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, warn)
        self.norm = norm

    def forward(self, log_probs: torch.Tensor, hyp: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        return F.minimum_bayes_risk(log_probs, hyp, self.eos, self.include_eos, self.batch_first, self.norm,
                                    self.ins_cost, self.del_cost, self.sub_cost, self.warn)


class _Prefix(_StringMatching):
    __constants__ = ("eos", "include_eos", "norm", "batch_first", "ins_cost", "del_cost",
                     "sub_cost", "padding", "exclude_last", "warn")
    norm: bool
    padding: int
    exclude_last: bool

    def _init(self, eos, include_eos, norm, batch_first, ins_cost, del_cost, sub_cost, padding,
              exclude_last, warn):
        norm = argcheck.is_bool(norm, "norm")
        padding = argcheck.is_int(padding, "padding")
        exclude_last = argcheck.is_bool(exclude_last, "exclude_last")
        _StringMatching.__init__(self, eos, include_eos, batch_first, ins_cost, del_cost,
                                 sub_cost, warn)
        self.norm, self.padding, self.exclude_last = norm, padding, exclude_last


class PrefixEditDistances(_Prefix):
    """Compute the edit distance between ref and each prefix of hyp (_string.py:800-885)"""

    def __init__(self, eos: Optional[int] = None, include_eos: bool = True, norm: bool = False,
                 batch_first: bool = False, ins_cost: float = config.DEFT_INS_COST,
                 del_cost: float = config.DEFT_DEL_COST, sub_cost: float = config.DEFT_SUB_COST,
                 padding: int = config.INDEX_PAD_VALUE, exclude_last: bool = False,
                 warn: bool = True):
        self._init(eos, include_eos, norm, batch_first, ins_cost, del_cost, sub_cost, padding,
                   exclude_last, warn)

    def forward(self, ref: torch.Tensor, hyp: torch.Tensor) -> torch.Tensor:
        return F.prefix_edit_distances(ref, hyp, self.eos, self.include_eos, self.norm,
                                       self.batch_first, self.ins_cost, self.del_cost,
                                       self.sub_cost, self.padding, self.exclude_last, self.warn)


class PrefixErrorRates(_Prefix):
    """Compute the error rate between ref and each prefix of hyp (_string.py:970-1049)"""

    def __init__(self, eos: Optional[int] = None, include_eos: bool = True, norm: bool = True,
                 batch_first: bool = False, ins_cost: float = config.DEFT_INS_COST,
                 del_cost: float = config.DEFT_DEL_COST, sub_cost: float = config.DEFT_SUB_COST,
                 padding: int = config.INDEX_PAD_VALUE, exclude_last: bool = False,
                 warn: bool = True):
        self._init(eos, include_eos, norm, batch_first, ins_cost, del_cost, sub_cost, padding,
                   exclude_last, warn)

    def forward(self, ref: torch.Tensor, hyp: torch.Tensor) -> torch.Tensor:
        return F.prefix_error_rates(ref, hyp, self.eos, self.include_eos, self.norm,
                                    self.batch_first, self.ins_cost, self.del_cost,
                                    self.sub_cost, self.padding, self.exclude_last, self.warn)


class OptimalCompletion(_StringMatching):
    """Return a mask of next tokens of a minimum edit distance prefix
    (_string.py:1052-1166)"""

    __constants__ = ("eos", "include_eos", "batch_first", "ins_cost", "del_cost", "sub_cost",
                     "padding", "exclude_last", "warn")
    padding: int
    exclude_last: bool

    def __init__(self, eos: Optional[int] = None, include_eos: bool = True,
                 batch_first: bool = False, ins_cost: float = config.DEFT_INS_COST,
                 del_cost: float = config.DEFT_DEL_COST, sub_cost: float = config.DEFT_SUB_COST,
                 padding: int = config.INDEX_PAD_VALUE, exclude_last: bool = False,
                 warn: bool = True):
        padding = argcheck.is_int(padding, "padding")
        exclude_last = argcheck.is_bool(exclude_last, "exclude_last")
        super().__init__(eos, include_eos, batch_first, ins_cost, del_cost, sub_cost, warn)
        self.padding, self.exclude_last = padding, exclude_last

    def forward(self, ref: torch.Tensor, hyp: torch.Tensor) -> torch.Tensor:
        return F.optimal_completion(ref, hyp, self.eos, self.include_eos, self.batch_first,
                                    self.ins_cost, self.del_cost, self.sub_cost, self.padding,
                                    self.exclude_last, self.warn)


class HardOptimalCompletionDistillationLoss(torch.nn.Module):
    """A categorical loss function over optimal next tokens (_string.py:1254-1378)"""

    __constants__ = ("eos", "include_eos", "batch_first", "ins_cost", "del_cost", "sub_cost",
                     "reduction", "ignore_index")

    eos: Optional[int]
    include_eos: bool
    batch_first: bool
    ins_cost: float
    del_cost: float
    sub_cost: float
    reduction: str
    ignore_index: int

    def __init__(self, eos: Optional[int] = None, include_eos: bool = True,
                 batch_first: bool = False, ins_cost: float = config.DEFT_INS_COST,
                 del_cost: float = config.DEFT_DEL_COST, sub_cost: float = config.DEFT_SUB_COST,
                 weight: Optional[torch.Tensor] = None, reduction: str = "mean",
                 ignore_index: int = config.INDEX_PAD_VALUE):
        eos = argcheck.is_int(eos, "eos", True)
        include_eos = argcheck.is_bool(include_eos, "include_eos")
        batch_first = argcheck.is_bool(batch_first, "batch_first")
        ins_cost = argcheck.is_float(ins_cost, "ins_cost")
        del_cost = argcheck.is_float(del_cost, "del_cost")
        sub_cost = argcheck.is_float(sub_cost, "sub_cost")
        weight = argcheck.is_tensor(weight, "weight", True)
        reduction = argcheck.is_in(reduction, _REDUCTIONS, "reduction")
        ignore_index = argcheck.is_int(ignore_index, "ignore_index")
        super().__init__()
        self.eos, self.include_eos, self.batch_first = eos, include_eos, batch_first
        self.ins_cost, self.del_cost, self.sub_cost = ins_cost, del_cost, sub_cost
        self.reduction, self.ignore_index = reduction, ignore_index
        self.register_buffer("weight", weight)

    def extra_repr(self) -> str:
        return ", ".join(f"{x}={getattr(self, x)}" for x in self.__constants__)

    def forward(self, logits: torch.Tensor, ref: torch.Tensor, hyp: torch.Tensor,
                warn: bool = True) -> torch.Tensor:
        return F.hard_optimal_completion_distillation_loss(
            logits, ref, hyp, self.eos, self.include_eos, self.batch_first, self.ins_cost,
            self.del_cost, self.sub_cost, self.weight, self.reduction, self.ignore_index, warn)


class MinimumErrorRateLoss(torch.nn.Module):
    """Error rate expectation normalized over some number of transcripts
    (_string.py:1475-1646)"""

    __constants__ = ("eos", "include_eos", "sub_avg", "batch_first", "norm", "ins_cost",
                     "del_cost", "sub_cost", "reduction")

    eos: Optional[int]
    include_eos: bool
    sub_avg: bool
    batch_first: bool
    norm: bool
    ins_cost: float
    del_cost: float
    sub_cost: float
    reduction: str

    def __init__(self, eos: Optional[int] = None, include_eos: bool = True, sub_avg: bool = True,
                 batch_first: bool = False, norm: bool = True,
                 ins_cost: float = config.DEFT_INS_COST, del_cost: float = config.DEFT_DEL_COST,
                 sub_cost: float = config.DEFT_SUB_COST, reduction: str = "mean"):
        eos = argcheck.is_int(eos, "eos", True)
        include_eos = argcheck.is_bool(include_eos, "include_eos")
        sub_avg = argcheck.is_bool(sub_avg, "sub_avg")
        batch_first = argcheck.is_bool(batch_first, "batch_first")
        norm = argcheck.is_bool(norm, "norm")
        ins_cost = argcheck.is_float(ins_cost, "ins_cost")
        del_cost = argcheck.is_float(del_cost, "del_cost")
        sub_cost = argcheck.is_float(sub_cost, "sub_cost")
        reduction = argcheck.is_in(reduction, _REDUCTIONS, "reduction")
        super().__init__()
        self.eos, self.include_eos, self.sub_avg = eos, include_eos, sub_avg
        self.batch_first, self.norm, self.reduction = batch_first, norm, reduction
        self.ins_cost, self.del_cost, self.sub_cost = ins_cost, del_cost, sub_cost

    def extra_repr(self) -> str:
        return ", ".join(f"{x}={getattr(self, x)}" for x in self.__constants__)

    def forward(self, log_probs: torch.Tensor, ref: torch.Tensor, hyp: torch.Tensor,
                warn: bool = True) -> torch.Tensor:
        return F.minimum_error_rate_loss(
            log_probs, ref, hyp, self.eos, self.include_eos, self.sub_avg, self.batch_first,
            self.norm, self.ins_cost, self.del_cost, self.sub_cost, self.reduction, warn)


class SequenceLogProbabilities(torch.nn.Module):
    """Calculate joint log probability of sequences (_decoding.py:1636-1721); `logits` is a
    tensor or a PackedSequence"""

    __constants__ = "dim", "eos"
    dim: int
    eos: Optional[int]

    def __init__(self, dim: int = 0, eos: Optional[int] = None):
        dim = argcheck.is_int(dim, "dim")
        if eos is not None:
            eos = argcheck.is_int(eos, "eos")
        super().__init__()
        self.dim = dim
        self.eos = eos

    def extra_repr(self) -> str:
        s = f"dim={self.dim}"
        if self.eos is not None:
            s += f", eos={self.eos}"
        return s

    def forward(self, logits: Any, hyp: torch.Tensor) -> torch.Tensor:
        return F.sequence_log_probs(logits, hyp, self.dim, self.eos)


class CTCGreedySearch(torch.nn.Module):
    """CTC greedy search (_decoding.py:563-633): the most likely class per step with blanks and
    repeats removed, and the (log-)probability of that path"""

    __constants__ = "blank_idx", "batch_first", "is_probs"
    blank_idx: int
    batch_first: bool
    is_probs: bool

    def __init__(self, blank_idx: int = -1, batch_first: bool = False, is_probs: bool = False):
        blank_idx = argcheck.is_int(blank_idx, "blank_idx")
        batch_first = argcheck.is_bool(batch_first, "batch_first")
        is_probs = argcheck.is_bool(is_probs, "is_probs")
        super().__init__()
        self.blank_idx = blank_idx
        self.batch_first = batch_first
        self.is_probs = is_probs

    def extra_repr(self) -> str:
        return ", ".join(f"{x}={getattr(self, x)}" for x in self.__constants__)

    def forward(self, logits: torch.Tensor, in_lens: Optional[torch.Tensor] = None
                ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        return F.ctc_greedy_search(logits, in_lens, self.blank_idx, self.batch_first, self.is_probs)
