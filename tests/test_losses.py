"""The two training losses in every dtype their kernels are instantiated for (fp32, fp64, fp16, bf16):
hard OCD (K5, lev_ocd_{fwd,reduce,bwd}_kernel) and MWER (K6, lev_mwer_{fwd,bwd}_kernel) against the
float64 oracle, on the SIMT emulator (tests/emu) and on the device.

The referee is oracle.oracle fed the exact values the kernels see: the inputs rounded to the test dtype
(class weights to the accumulation dtype), then widened to float64.  Shapes put a partial last warp
stride on the vocabulary / group axis (V, M in {31, 33, 1037, 70}) and a partly empty last 256-thread
block on the row axis (rows not a multiple of 8).
"""
import numpy as np
import pytest
import torch

import parity_cases as PC
from oracle import oracle as O

DTYPES = [torch.float32, torch.float64, torch.float16, torch.bfloat16]
# one unit in the last place of a 16-bit output: the kernels accumulate in fp32 and round once
ULP16 = {torch.float16: 2.0 ** -10, torch.bfloat16: 2.0 ** -7}
REDUCTIONS = ["mean", "sum", "none"]
OCD_V = [2, 31, 32, 33, 1037]
MWER_M = [2, 31, 32, 33, 70]


def _acc(dtype):
    return torch.float64 if dtype == torch.float64 else torch.float32


def _fmax(a):
    """Largest finite magnitude (0 if there is none)."""
    a = np.abs(np.asarray(a, np.float64))
    a = a[np.isfinite(a)]
    return float(a.max()) if a.size else 0.0


def _assert_close(act, exp, rtol, atol, what):
    """|act - exp| <= atol + rtol |exp| elementwise (atol may be an array); infinities and NaNs must
    sit exactly where the referee has them."""
    act, exp = np.asarray(act, np.float64), np.asarray(exp, np.float64)
    assert act.shape == exp.shape, (what, act.shape, exp.shape)
    same = (act == exp) | (np.isnan(act) & np.isnan(exp))
    with np.errstate(invalid="ignore"):
        err = np.where(same, 0.0, np.abs(act - exp))
        bound = np.broadcast_to(atol + rtol * np.where(same, 0.0, np.abs(exp)), err.shape)
        ok = err <= bound
    if not ok.all():
        ratio = np.where(ok, 0.0, np.where(np.isnan(err), np.inf, err / np.maximum(bound, 1e-300)))
        i = np.unravel_index(np.argmax(ratio), ratio.shape)
        raise AssertionError(f"{what}: {int((~ok).sum())} of {ok.size} outside the bar; worst at {i}: got "
                             f"{act[i]!r}, want {exp[i]!r}, bar {bound[i]:.3g}")


def _check_loss(act, exp, dtype, scale, what, slack=0.0):
    """A loss against the referee.  `scale` is the size of the largest term (fp64, fp32) or the sum of
    the term magnitudes that each carry their own 16-bit rounding (fp16, bf16)."""
    if dtype == torch.float64:
        # float64 throughout: a few ulps of the largest term, summed over at most a few thousand terms
        _assert_close(act, exp, 1e-12, 1e-12 * scale + slack, what)
    elif dtype == torch.float32:
        # the fp32 bars of parity_cases.check_golden_losses: two fp32 log-sum-exps differ by a few ulps
        _assert_close(act, exp, 2e-6, 2e-6 * max(1.0, _fmax(exp)) + slack, what)
    else:
        # fp32 accumulation rounded once to 16 bits: one unit in the last place of the terms
        _assert_close(act, exp, 0.0, ULP16[dtype] * scale + slack, what)


def _check_grad(act, exp, dtype, what, slack=0.0):
    scale = _fmax(exp)
    if dtype == torch.float64:
        # as for the loss: every element is a softmax term minus the target term, in float64
        _assert_close(act, exp, 1e-12, 1e-12 * scale + slack, what)
    elif dtype == torch.float32:
        _assert_close(act, exp, 2e-5, 1e-6 * max(1.0, scale) + slack, what)  # check_golden_losses
    else:
        # fp32 arithmetic, one rounding to 16 bits per element: one ulp of the largest element
        _assert_close(act, exp, 0.0, ULP16[dtype] * scale + slack, what)


# ---- hard OCD ---------------------------------------------------------------------------------
def _ocd_batch(rng, R, H, N, V, eos=0, all_classes=False):
    """(ref (R, N), hyp (H, N)) tokens; with `all_classes` every token, padding included, is a class."""
    if all_classes:
        return rng.integers(0, V, (R, N)), rng.integers(0, V, (H, N))
    return (PC.random_tokens(rng, R, N, V, eos, -2, R // 3), PC.random_tokens(rng, H, N, V, eos, -3, H // 3))


def check_ocd(F, dev, dtype, ref, hyp, logits, *, weight=None, reduction="mean", eos=0, include_eos=True,
              batch_first=False, ignore_index=-2, grad_seed=0, view=None, what=""):
    """One call of hard_optimal_completion_distillation_loss, forward and backward, against the oracle.
    ref / hyp / logits are numpy arrays in the layout `batch_first` names; `view` maps the logits
    tensor (already on `dev`, in `dtype`) to the tensor that is passed."""
    what = f"ocd {dtype} V={logits.shape[-1]} {reduction} bf={batch_first} w={weight is not None} {what}"
    x = torch.from_numpy(logits).to(dtype)
    x64 = x.double()
    w = None if weight is None else torch.from_numpy(weight).to(_acc(dtype))
    exp_go = None
    go = None
    if reduction == "none":
        go = torch.from_numpy(np.random.default_rng(grad_seed).standard_normal(logits.shape[:2])).to(dtype)
        exp_go = go.double().numpy()
    exp_loss, exp_grad = O.hard_optimal_completion_distillation_loss(
        x64, ref, hyp, eos=eos, include_eos=include_eos, batch_first=batch_first,
        weight=None if w is None else w.double(), reduction=reduction, ignore_index=ignore_index,
        grad_output=exp_go)
    xd = x.to(dev)
    if view is not None:
        xd = view(xd)
    xd.requires_grad_(True)
    loss = F.hard_optimal_completion_distillation_loss(
        xd, torch.from_numpy(ref).to(dev), torch.from_numpy(hyp).to(dev), eos=eos, include_eos=include_eos,
        batch_first=batch_first, weight=None if w is None else w.to(dev), reduction=reduction,
        ignore_index=ignore_index, warn=False)
    assert loss.dtype == dtype and loss.device == xd.device, what  # the logits' dtype
    (grad,) = torch.autograd.grad([loss], [xd], None if go is None else [go.to(dev)])
    assert grad.dtype == dtype and grad.shape == xd.shape, what
    # the per-step terms w_t (lse - z_t) / |S| are >= 0 (weights >= 0): no cancellation, so the
    # largest value is the scale of the terms
    _check_loss(loss.detach().double().cpu().numpy(), exp_loss, dtype, _fmax(exp_loss), what + " loss")
    _check_grad(grad.double().cpu().numpy(), exp_grad, dtype, what + " grad")
    return exp_loss


def _weight(rng, V):
    w = rng.uniform(0.25, 2.0, V)
    w[1::4] = 0.0  # classes with weight 0
    return w


def run_ocd_matrix(F, dev, dtype, V, H=13, N=7, R=10):
    """reductions x layouts x (no weight, weight): rows H * N = 91 leave the last block part empty."""
    rng = np.random.default_rng(V * 7 + DTYPES.index(dtype))
    ref, hyp = _ocd_batch(rng, R, H, N, V)
    ref[0, 0] = hyp[0, 1] = 0  # an empty reference and an empty hypothesis
    logits = rng.standard_normal((H, N, V)) * 3.0
    w = _weight(rng, V)
    for reduction in REDUCTIONS:
        for bf in (False, True):
            r, h, lg = (ref.T.copy(), hyp.T.copy(), logits.transpose(1, 0, 2).copy()) if bf else (ref, hyp, logits)
            for weight in (None, w):
                check_ocd(F, dev, dtype, r, h, lg, weight=weight, reduction=reduction, batch_first=bf)


def run_ocd_edges(F, dev, dtype, V=11, H=13, N=7, R=10):
    rng = np.random.default_rng(100 + DTYPES.index(dtype))
    ref, hyp = _ocd_batch(rng, R, H, N, 7)  # tokens < 7: classes 7..10 are never targets
    ref[0, ::3] = 0  # empty references
    hyp[0, 1::3] = 0  # empty hypotheses
    ref[0, 2::5] = hyp[0, 2::5] = 0  # both
    logits = rng.standard_normal((H, N, V)) * 3.0
    w = _weight(rng, V)
    masked = logits.copy()
    masked[rng.random((H, N)) < 0.5, 7:] = -np.inf  # masked classes, none of them a target
    masked[rng.random((H, N, V)) < 0.1] = -np.inf
    masked = np.where(np.isin(np.arange(V), np.unique(ref[ref >= 0])), logits, masked)
    tg = O.optimal_completion(ref, hyp, eos=0, padding=-2, exclude_last=True)  # (H, N, U)
    a, b = np.argwhere((tg >= 0).any(2))[3]
    neg_target = logits.copy()
    neg_target[a, b, tg[a, b][tg[a, b] >= 0][0]] = -np.inf  # a target whose logit is -inf: the loss is inf
    all_ref, all_hyp = _ocd_batch(rng, R, H, N, V, all_classes=True)
    cases = [
        ("empty", ref, hyp, logits, {}),
        ("include_eos=False", ref, hyp, logits, dict(include_eos=False)),
        ("eos=None", all_ref, all_hyp, logits, dict(eos=None)),
        ("ignore_index=-100", ref, hyp, logits, dict(ignore_index=-100)),
        ("ignore_index=V+5", ref, hyp, logits, dict(ignore_index=V + 5)),
        ("eos=None ignore_index=V+5", all_ref, all_hyp, logits, dict(eos=None, ignore_index=V + 5)),
        ("masked classes", ref, hyp, masked, {}),
        ("-inf target", ref, hyp, neg_target, {}),
    ]
    for name, r, h, lg, kw in cases:
        for reduction in REDUCTIONS:
            for bf in (False, True):
                args = (r.T.copy(), h.T.copy(), lg.transpose(1, 0, 2).copy()) if bf else (r, h, lg)
                weight = w if reduction == "sum" else None
                exp = check_ocd(F, dev, dtype, *args, weight=weight, reduction=reduction, batch_first=bf,
                                what=name, **kw)
                if name == "-inf target" and reduction != "none":
                    assert not np.isfinite(exp)  # inf, or NaN where that target has weight 0


def run_ocd_long_sequence_axis(F, dev, dtype):
    """37 sequences (two blocks of 32 in lev_ocd_reduce_kernel) of 131 steps (past the 128 steps a
    warp's four loads cover), in both layouts: rows 4847."""
    rng = np.random.default_rng(7)
    H, N, V = 131, 37, 33
    ref, hyp = _ocd_batch(rng, 12, H, N, V)
    ref[0, 5] = hyp[0, 6] = 0
    logits = rng.standard_normal((H, N, V))
    for reduction in ("mean", "sum"):
        check_ocd(F, dev, dtype, ref, hyp, logits, reduction=reduction)
        check_ocd(F, dev, dtype, ref.T.copy(), hyp.T.copy(), logits.transpose(1, 0, 2).copy(),
                  weight=_weight(rng, V), reduction=reduction, batch_first=True)


def run_ocd_permuted_logits(F, dev, dtype):
    """Logits (T, N, V) as a permuted view of an (N, T, V) tensor: ls_a = V < ls_b = T * V."""
    rng = np.random.default_rng(8)
    H, N, V = 11, 9, 33
    ref, hyp = _ocd_batch(rng, 9, H, N, V)
    logits = rng.standard_normal((H, N, V))
    for reduction in REDUCTIONS:
        check_ocd(F, dev, dtype, ref, hyp, logits, weight=_weight(rng, V), reduction=reduction,
                  view=lambda x: x.permute(1, 0, 2).contiguous().permute(1, 0, 2), what="permuted")


def run_ocd_errors(F, dev):
    """What cross_entropy rejects, the library rejects with torch's messages."""
    rng = np.random.default_rng(9)
    H, N, V = 7, 4, 9
    ref, hyp = _ocd_batch(rng, 6, H, N, V)
    ref[:, 2] = [3, 12, 5, 0, -2, -2]  # reference token 12 is not a class
    lg = torch.randn(H, N, V, device=dev)
    with pytest.raises(IndexError, match=r"Target 12 is out of bounds\."):
        F.hard_optimal_completion_distillation_loss(lg, torch.from_numpy(ref).to(dev),
                                                    torch.from_numpy(hyp).to(dev), eos=0, warn=False)
    # eos=None: the padding -1 of a reference is a target, and not ignore_index
    ref2 = rng.integers(0, V, (6, N))
    ref2[4:, 1] = -1
    with pytest.raises(IndexError, match=r"Target -1 is out of bounds\."):
        F.hard_optimal_completion_distillation_loss(lg, torch.from_numpy(ref2).to(dev),
                                                    torch.from_numpy(hyp).to(dev), eos=None, warn=False)
    ref[1, 2] = 4
    for w in (torch.ones(V - 4), torch.ones(V + 1), torch.ones(1, V)):
        with pytest.raises(RuntimeError, match=rf"weight tensor should be defined either for all {V} classes "
                                               rf"or no classes but got weight tensor of shape: \[{', '.join(map(str, w.shape))}\]"):
            F.hard_optimal_completion_distillation_loss(lg, torch.from_numpy(ref).to(dev),
                                                        torch.from_numpy(hyp).to(dev), eos=0,
                                                        weight=w.to(dev), warn=False)


# ---- MWER ---------------------------------------------------------------------------------------
def _mwer_batch(rng, T, N, M, V=9):
    ref = PC.random_tokens(rng, T, N, V, 0, -2, 2)
    hyp = PC.random_tokens(rng, T, N * M, V, 0, -3, 1).reshape(T, N, M)
    return ref, hyp


def check_mwer(F, dev, dtype, ref, hyp, lp, *, sub_avg, reduction, batch_first=False, grad_seed=0,
               view=None, what=""):
    """One call of minimum_error_rate_loss, forward and backward, against the oracle.  `lp` is (N, M)
    numpy; `view` maps the log-prob tensor (on `dev`, in `dtype`) to the tensor that is passed."""
    N, M = lp.shape
    what = f"mwer {dtype} M={M} {reduction} sub_avg={sub_avg} bf={batch_first} {what}"
    x = torch.from_numpy(lp).to(dtype)
    x64 = x.double()
    out_dtype = _acc(dtype)  # fp32 for fp16 / bf16 / fp32 inputs, fp64 for fp64
    go = exp_go = None
    if reduction == "none":
        go = torch.from_numpy(np.random.default_rng(grad_seed).standard_normal((N, M))).to(out_dtype)
        exp_go = go.double().numpy()
    kw = dict(eos=0, include_eos=True, sub_avg=sub_avg, batch_first=batch_first, norm=True)
    exp_loss, exp_grad = O.minimum_error_rate_loss(x64, ref, hyp, reduction=reduction, grad_output=exp_go, **kw)
    # the terms e_nm p_nm of the loss, for the bars (and, rounded as the forward rounds p, the 16-bit
    # referee): e from the oracle's fp32 error rates, minus their mean in float64 as the oracle does
    if batch_first:
        er = O.error_rate(np.repeat(ref, M, 0), hyp.reshape(N * M, -1), 0, True, True, True)
    else:
        er = O.error_rate(np.repeat(ref, M, 1), hyp.reshape(hyp.shape[0], N * M), 0, True, True, False)
    er = er.astype(np.float64).reshape(N, M)
    e = er - er.mean(1, keepdims=True) if sub_avg else er
    with np.errstate(invalid="ignore"):
        p = torch.softmax(x64, 1).numpy()
        terms = e * p
        np.testing.assert_allclose({"mean": terms.mean(), "sum": terms.sum(), "none": terms}[reduction],
                                   exp_loss, rtol=1e-13, atol=1e-15)  # the terms are the oracle's
        if dtype in ULP16:
            # lev_mwer_fwd_kernel rounds the softmax to the dtype of log_probs before the product, as
            # torch's 16-bit softmax output is
            terms = e * torch.from_numpy(p).to(dtype).double().numpy()
            exp_loss = {"mean": terms.mean(), "sum": terms.sum(), "none": terms}[reduction]
    div = N * M if reduction == "mean" else 1
    # fp64: the largest term; 16-bit: every term carries its own rounding of p
    scale = (_fmax(terms) if dtype not in ULP16 or reduction == "none" else np.nansum(np.abs(terms))) / div
    slack_l = slack_g = 0.0
    if dtype == torch.float64 and sub_avg:
        # e is (er - mean) taken in fp32, as the reference takes it (its mean over up to 70 fp32 values
        # in the kernel's summation order, then the difference): a few units of 2^-24 max|er| per term
        # (1.1 seen), against the oracle's float64 subtraction
        d = 4 * 2.0 ** -24 * np.abs(er).max(1, keepdims=True) * np.nan_to_num(p)
        slack_l = {"mean": d.sum() / div, "sum": d.sum(), "none": d}[reduction]
        gmax = (np.abs(exp_go).max(1, keepdims=True) if reduction == "none" else 1.0 / div)
        slack_g = 2 * d * gmax  # d grad_m = p_m (go_m de_m - sum_k p_k go_k de_k)
    xd = x.to(dev)
    if view is not None:
        xd = view(xd)
    xd.requires_grad_(True)
    loss = F.minimum_error_rate_loss(xd, torch.from_numpy(ref).to(dev), torch.from_numpy(hyp).to(dev),
                                     reduction=reduction, warn=False, **kw)
    assert loss.dtype == out_dtype and loss.device == xd.device, what
    (grad,) = torch.autograd.grad([loss], [xd], None if go is None else [go.to(dev)])
    assert grad.dtype == dtype and grad.shape == (N, M), what
    _check_loss(loss.detach().double().cpu().numpy(), exp_loss, dtype, scale, what + " loss", slack_l)
    # the backward takes the unrounded softmax: the oracle's gradient
    _check_grad(grad.double().cpu().numpy(), exp_grad, dtype, what + " grad", slack_g)
    return exp_loss, exp_grad


def run_mwer_matrix(F, dev, dtype, M, N=13, T=8):
    """reductions x sub_avg x layouts; N = 13 groups leave the last 256-thread block part empty."""
    rng = np.random.default_rng(M * 5 + DTYPES.index(dtype))
    ref, hyp = _mwer_batch(rng, T, N, M)
    lp = rng.standard_normal((N, M)) * 2.0
    for reduction in REDUCTIONS:
        for sub_avg in (True, False):
            check_mwer(F, dev, dtype, ref, hyp, lp, sub_avg=sub_avg, reduction=reduction)
            check_mwer(F, dev, dtype, ref.T.copy(), hyp.transpose(1, 2, 0).copy(), lp, sub_avg=sub_avg,
                       reduction=reduction, batch_first=True)


def run_mwer_views(F, dev, dtype):
    """log_probs as a column block of a wider tensor (stride (M + 5, 1)) and as a transposed view
    (stride (1, N))."""
    rng = np.random.default_rng(11)
    N, M, T = 9, 33, 7
    ref, hyp = _mwer_batch(rng, T, N, M)
    lp = rng.standard_normal((N, M))
    col = lambda x: torch.cat([x[:, :3], x, x[:, :2]], 1)[:, 3:3 + M]  # noqa: E731
    tr = lambda x: x.t().contiguous().t()  # noqa: E731
    for name, view in (("column view", col), ("transposed view", tr)):
        for reduction in REDUCTIONS:
            check_mwer(F, dev, dtype, ref, hyp, lp, sub_avg=True, reduction=reduction, view=view, what=name)


def run_mwer_neg_inf(F, dev, dtype):
    """Pruned beam slots (-inf log-probs, as beam_search_advance emits them): zero weight, and NaN
    exactly where the oracle has it (a group with no live slot)."""
    rng = np.random.default_rng(12)
    N, M, T = 9, 33, 7
    ref, hyp = _mwer_batch(rng, T, N, M)
    lp = rng.standard_normal((N, M))
    lp[rng.random((N, M)) < 0.3] = -np.inf
    lp[:, 0] = 0.5
    for reduction in REDUCTIONS:
        check_mwer(F, dev, dtype, ref, hyp, lp, sub_avg=True, reduction=reduction, what="-inf")
    lp[4] = -np.inf
    exp_loss, exp_grad = check_mwer(F, dev, dtype, ref, hyp, lp, sub_avg=False, reduction="none",
                                    what="-inf group")
    assert np.isnan(exp_loss[4]).all() and np.isfinite(np.delete(exp_loss, 4, 0)).all()


# ---- the library on the SIMT emulator ---------------------------------------------------------
@pytest.fixture(scope="module")
def F():
    from emu_backend import emulated_kernels

    with emulated_kernels():
        import b200lev.functional as F_

        yield F_


CPU = torch.device("cpu")


@pytest.mark.parametrize("V", OCD_V)
@pytest.mark.parametrize("dtype", DTYPES, ids=str)
def test_ocd_vs_oracle(F, dtype, V):
    run_ocd_matrix(F, CPU, dtype, V)


@pytest.mark.parametrize("dtype", DTYPES, ids=str)
def test_ocd_edges(F, dtype):
    run_ocd_edges(F, CPU, dtype)


@pytest.mark.parametrize("dtype", [torch.float64, torch.bfloat16], ids=str)
def test_ocd_long_sequence_axis(F, dtype):
    run_ocd_long_sequence_axis(F, CPU, dtype)


@pytest.mark.parametrize("dtype", DTYPES, ids=str)
def test_ocd_permuted_logits(F, dtype):
    run_ocd_permuted_logits(F, CPU, dtype)


def test_ocd_fp64_weight_is_not_narrowed(F):
    """Weights that fp32 cannot hold: an fp64 weight reaches the fp64 kernels unrounded."""
    rng = np.random.default_rng(13)
    ref, hyp = _ocd_batch(rng, 8, 9, 5, 31)
    w = 1.0 + rng.random(31) * 1e-3  # every weight has bits below fp32's 24
    for reduction in REDUCTIONS:
        check_ocd(F, CPU, torch.float64, ref, hyp, rng.standard_normal((9, 5, 31)), weight=w, reduction=reduction)


def test_ocd_empty_batch_mean_is_nan(F):
    """No sequences: the mean over them is NaN, as torch's mean of an empty tensor is."""
    for dtype in (torch.float32, torch.float64):
        lg = torch.zeros(5, 0, 7, dtype=dtype, requires_grad=True)
        loss = F.hard_optimal_completion_distillation_loss(lg, torch.zeros(4, 0, dtype=torch.long),
                                                           torch.zeros(5, 0, dtype=torch.long), eos=0, warn=False)
        assert loss.dtype == dtype and torch.isnan(loss)
        (g,) = torch.autograd.grad([loss], [lg])
        assert g.shape == (5, 0, 7)


def test_ocd_errors(F):
    run_ocd_errors(F, CPU)


@pytest.mark.parametrize("M", MWER_M)
@pytest.mark.parametrize("dtype", DTYPES, ids=str)
def test_mwer_vs_oracle(F, dtype, M):
    run_mwer_matrix(F, CPU, dtype, M)


@pytest.mark.parametrize("dtype", DTYPES, ids=str)
def test_mwer_strided_log_probs(F, dtype):
    run_mwer_views(F, CPU, dtype)


@pytest.mark.parametrize("dtype", DTYPES, ids=str)
def test_mwer_neg_inf_log_probs(F, dtype):
    run_mwer_neg_inf(F, CPU, dtype)


# ---- the device ---------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def FG():
    import b200lev.functional as F_

    return F_


CUDA = torch.device("cuda")


@pytest.mark.gpu
@pytest.mark.parametrize("V", OCD_V)
@pytest.mark.parametrize("dtype", DTYPES, ids=str)
def test_gpu_ocd_vs_oracle(FG, dtype, V):
    run_ocd_matrix(FG, CUDA, dtype, V)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=str)
def test_gpu_ocd_edges_and_views(FG, dtype):
    run_ocd_edges(FG, CUDA, dtype)
    run_ocd_long_sequence_axis(FG, CUDA, dtype)
    run_ocd_permuted_logits(FG, CUDA, dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=str)
def test_gpu_ocd_cfg3(FG, dtype):
    """The cfg3 shape: 128 character sequences, T = 201, V = 32."""
    rng = np.random.default_rng(3)
    N, T, V = 128, 201, 32
    ref = PC.random_tokens(rng, T, N, V, 0, 0, min_len=99)
    hyp = PC.random_tokens(rng, T, N, V, 0, 0, min_len=99)
    for n in range(0, N, 2):  # noisy copies: realistic (sparse) target sets
        hyp[:, n] = np.where(rng.random(T) > 0.1, ref[:, n], hyp[:, n])
    logits = rng.standard_normal((T, N, V))
    for reduction in ("mean", "none"):
        check_ocd(FG, CUDA, dtype, ref, hyp, logits, reduction=reduction, ignore_index=-100)


@pytest.mark.gpu
def test_gpu_ocd_large_vocabulary_bf16(FG):
    rng = np.random.default_rng(10)
    H, N, V = 21, 15, 10_000
    ref, hyp = _ocd_batch(rng, 18, H, N, V)
    logits = rng.standard_normal((H, N, V)) * 2.0
    for reduction in REDUCTIONS:
        check_ocd(FG, CUDA, torch.bfloat16, ref, hyp, logits, weight=_weight(rng, V), reduction=reduction)


@pytest.mark.gpu
def test_gpu_ocd_errors(FG):
    run_ocd_errors(FG, CUDA)


@pytest.mark.gpu
@pytest.mark.parametrize("M", MWER_M)
@pytest.mark.parametrize("dtype", DTYPES, ids=str)
def test_gpu_mwer_vs_oracle(FG, dtype, M):
    run_mwer_matrix(FG, CUDA, dtype, M)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=str)
def test_gpu_mwer_views_and_neg_inf(FG, dtype):
    run_mwer_views(FG, CUDA, dtype)
    run_mwer_neg_inf(FG, CUDA, dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.bfloat16], ids=str)
def test_gpu_host_tensors_in_and_out(FG, dtype):
    """Host tensors in, host tensors out (the library stages them through the device)."""
    rng = np.random.default_rng(14)
    ref, hyp = _ocd_batch(rng, 10, 13, 7, 33)
    for reduction in ("mean", "none"):
        check_ocd(FG, CPU, dtype, ref, hyp, rng.standard_normal((13, 7, 33)), weight=_weight(rng, 33),
                  reduction=reduction)
    mref, mhyp = _mwer_batch(rng, 8, 13, 33)
    for reduction in ("sum", "none"):
        check_mwer(FG, CPU, dtype, mref, mhyp, rng.standard_normal((13, 33)), sub_avg=True, reduction=reduction)
