"""Kernel-logic + host-logic tests on a GPU-less box.

The CUDA sources under pydrobert-pytorch_b200/csrc are compiled against the SIMT
emulator of tests/emu (every CUDA thread a cooperative fiber; see emu_cuda.h) and the
unmodified Python host layer drives them through the same C ABI.  What this pins:
index arithmetic, wavefront skew, strip hand-off, epilogues, flags, the compaction and
the losses -- against the reference's golden outputs and the oracle.  What it cannot
pin (memory-model effects, real launch limits) is left to the `-m gpu` suite, which is
the parity gate proper.
"""
import numpy as np
import pytest
import torch

import parity_cases as PC
from emu_backend import emulated_kernels


@pytest.fixture(scope="module")
def F():
    with emulated_kernels():
        import b200lev.functional as F_

        yield F_


DEV = torch.device("cpu")


def test_golden_small_cases(F, golden_sm):
    names = [n for n in golden_sm.params if n.startswith("s")]
    assert PC.check_golden_string_matching(F, DEV, golden_sm, names) >= 300


@pytest.mark.parametrize("name", ["cfg1", "cfg2r", "cfg3r", "cfg4r", "cfg5r", "cfg5f", "wide", "tall"])
def test_golden_config_shaped_cases(F, golden_sm, name):
    assert PC.check_golden_string_matching(F, DEV, golden_sm, [name]) >= 4


def test_golden_losses(F, golden_loss):
    assert PC.check_golden_losses(F, DEV, golden_loss) == 72


@pytest.mark.parametrize("costs", [(1, 1, 1), (3, 3, 4), (1, 2, 3), (0.5, 1.0, 0.25), (0.7, 1.1, 1.3)])
@pytest.mark.parametrize("shape", [(40, 45, 6), (70, 30, 5), (130, 20, 3), (300, 40, 2)])
@pytest.mark.parametrize("cta", ["0", "1"], ids=["warp_kernel", "cta_kernel"])
def test_random_vs_oracle_strips(F, costs, shape, cta, monkeypatch):
    """Reference lengths on both sides of every strip-width boundary (32/64/128/256
    columns) so the multi-strip hand-off and every C variant are exercised, on both the
    warp-per-pair kernel (lev_dp.cu) and the CTA-per-pair kernel (lev_cta.cu)."""
    monkeypatch.setenv("B200LEV_CTA_KERNEL", cta)
    R, H, N = shape
    PC.check_vs_oracle(F, DEV, seed=R * 1000 + H, R=R, H=H, N=N, V=6, costs=costs,
                       include_eos=True, norm=True, exclude_last=False, min_frac=0.5)


@pytest.mark.parametrize("flags", [
    dict(include_eos=False, norm=False, batch_first=True, exclude_last=True),
    dict(include_eos=True, norm=True, batch_first=True, exclude_last=False, no_eos_frac=0.3),
    dict(include_eos=False, norm=True, batch_first=False, exclude_last=True, eos=None),
])
def test_random_vs_oracle_flags(F, flags):
    for seed, costs in enumerate([(1, 1, 1), (2, 1, 3), (2, 2, 2)]):
        PC.check_vs_oracle(F, DEV, seed=seed, R=37, H=33, N=7, V=4, costs=costs, min_frac=0.0,
                           padding=-7, **flags)


@pytest.mark.parametrize("dtype", [torch.int32, torch.int16, torch.int8])
def test_token_dtypes(F, dtype):
    PC.check_vs_oracle(F, DEV, seed=5, R=20, H=22, N=5, V=9, costs=(1, 1, 1), eos=-1,
                       include_eos=False, dtype=dtype)


def test_n_best_shared_reference(F):
    """MWER's 2-D ref (SM:1426/1439) is read through ref_group, never repeated."""
    rng = np.random.default_rng(3)
    R, H, N, M = 12, 14, 4, 3
    ref = PC.random_tokens(rng, R, N, 7, 0, -1)
    hyp = PC.random_tokens(rng, H, N * M, 7, 0, -1).reshape(H, N, M)
    lp = rng.standard_normal((N, M)).astype(np.float32)
    from oracle import oracle as O

    exp_loss, exp_grad = O.minimum_error_rate_loss(lp, ref, hyp, eos=0)
    x = torch.from_numpy(lp).requires_grad_(True)
    loss = F.minimum_error_rate_loss(x, torch.from_numpy(ref), torch.from_numpy(hyp), eos=0,
                                     warn=False)
    loss.backward()
    np.testing.assert_allclose(loss.item(), exp_loss, rtol=2e-6, atol=1e-7)
    np.testing.assert_allclose(x.grad.numpy(), exp_grad, rtol=2e-5, atol=1e-7)


def test_grouped_references_take_the_fused_kernel(F, monkeypatch):
    PC.check_grouped_references(F, DEV)
    monkeypatch.setenv("B200LEV_BITVEC", "0")  # the same batches through the wavefront kernels
    PC.check_grouped_references(F, DEV, seed=1)


def test_warnings(F):
    PC.check_warnings(F, DEV)


def test_errors(F):
    PC.check_errors(F, DEV)


def test_sclite(F, golden_sclite):
    z = golden_sclite
    ers = F.error_rate(torch.from_numpy(z["ref"]), torch.from_numpy(z["hyp"]), eos=-1,
                       include_eos=False, norm=False, ins_cost=3.0, del_cost=3.0, sub_cost=4.0,
                       warn=False).numpy()
    assert np.array_equal(ers, z["errs"])
    assert f"{ers.sum() / z['ref_lens'].sum():.03f}" == f"{float(z['total']):.03f}"


def test_fill_after_eos(F):
    PC.check_fill_after_eos(F, DEV)


@pytest.mark.parametrize("jit_type", ["nojit", "trace", "script"])
def test_modules_jit(F, jit_type):
    import b200lev.modules as M

    PC.check_modules(F, M, DEV, jit_type)


def test_modules_match_functionals(F):
    import b200lev.modules as M

    rng = np.random.default_rng(1)
    ref = torch.from_numpy(PC.random_tokens(rng, 9, 4, 5, 0, -1))
    hyp = torch.from_numpy(PC.random_tokens(rng, 8, 4, 5, 0, -1))
    assert torch.equal(M.ErrorRate(eos=0, warn=False)(ref, hyp), F.error_rate(ref, hyp, eos=0, warn=False))
    assert torch.equal(M.EditDistance(eos=0)(ref, hyp), F.edit_distance(ref, hyp, eos=0))
    assert torch.equal(M.PrefixErrorRates(eos=0, warn=False)(ref, hyp),
                       F.prefix_error_rates(ref, hyp, eos=0, warn=False))
    assert torch.equal(M.PrefixEditDistances(eos=0, padding=-3)(ref, hyp),
                       F.prefix_edit_distances(ref, hyp, eos=0, padding=-3))
    assert torch.equal(M.OptimalCompletion(eos=0)(ref, hyp), F.optimal_completion(ref, hyp, eos=0))
    assert "eos=0" in repr(M.ErrorRate(eos=0))
    with pytest.raises(ValueError, match="eos .* is not an int"):
        M.ErrorRate(eos="a")
    with pytest.raises(ValueError, match="is not one of"):
        M.MinimumErrorRateLoss(reduction="bad")
    logits = torch.randn(8, 4, 5, requires_grad=True)
    loss = M.HardOptimalCompletionDistillationLoss(eos=0)(logits, ref, hyp)
    loss.backward()
    assert torch.isfinite(loss) and logits.grad.abs().sum() > 0


def test_wide_tokens(F):
    PC.check_wide_tokens(F, DEV)


@pytest.mark.parametrize("shape", [(20, 25, 70), (31, 30, 90), (45, 50, 40), (101, 101, 40),
                                   (201, 60, 12), (420, 40, 6), (800, 30, 3)])
@pytest.mark.parametrize("costs", [(1, 1, 1), (3, 3, 4)])
def test_group_kernel_vs_oracle(F, shape, costs, monkeypatch):
    """The length-bucketed group kernel (lev_group.cu), forced on for small batches:
    every lane-group width G = 1..32, cost-only and (cost, count) paths, final and
    prefix outputs, ragged lengths incl. empty sequences."""
    monkeypatch.setenv("B200LEV_GROUP_MIN_PAIRS", "1")
    R, H, N = shape
    for flags in (dict(include_eos=True, norm=True, exclude_last=False, min_frac=0.0),
                  dict(include_eos=False, norm=False, exclude_last=True, min_frac=0.4,
                       batch_first=True)):
        # spread=1: tokens fit 16 bits -> packed 2 x int16 DPX path; 70001: 32-bit path
        for spread in (1, 70001):
            PC.check_vs_oracle(F, DEV, seed=R + H, R=R, H=H, N=N, V=5, costs=costs, do_mask=False,
                               padding=-3, spread=spread, **flags)


@pytest.fixture(params=["fused", "short"])
def bv_form(request, monkeypatch):
    """The two kernels of the unit-cost bit-vector path: the fused kernel (lev_bvfused.cu, the
    default for R > 64, here for every R) and the lane-per-pair short-reference kernel
    (lev_bvshort.cu, R <= 64; larger shapes of a "short" run fall through to the fused kernel)."""
    if request.param == "short":
        monkeypatch.setenv("B200LEV_BVSHORT_MIN_PAIRS", "1")
    else:
        monkeypatch.setenv("B200LEV_BV_SHORT", "0")
    return request.param


@pytest.mark.parametrize("costs", [(1, 1, 1), (3, 3, 4)])
@pytest.mark.parametrize("group", [1, 3])
def test_final_sums_every_kernel_form(F, bv_form, costs, group, monkeypatch):
    """b200lev_final_sums (the bulk-scoring step, command_line.py:1124-1147): the fp64 totals are
    the same whether the short-reference kernel accumulates them itself or lev_err_sum_kernel follows
    the fused / wavefront kernels -- odd pair counts (lanes shadowing the last pair), references
    shared by `group` hypotheses, normalised and raw values."""
    from b200lev import _ops

    monkeypatch.setenv("B200LEV_BITVEC", "1")
    monkeypatch.setenv("B200LEV_BITVEC_MIN_PAIRS", "1")
    monkeypatch.setenv("B200LEV_BVS_CTAS", "2")  # several blocks of pairs per warp
    rng = np.random.default_rng(11)
    for R, H, n_ref in ((20, 25, 37), (30, 9, 1100), (64, 30, 45), (90, 40, 33)):
        ref = PC.random_tokens(rng, R, n_ref, 12, -1, -2, min_len=0)
        hyp = PC.random_tokens(rng, H, n_ref * group, 12, -1, -2, min_len=0)
        for norm in (False, True):
            exp = PC.O.error_rate(np.repeat(ref, group, axis=1), hyp, eos=-1, include_eos=False,
                                  norm=norm, ins_cost=costs[0], del_cost=costs[1], sub_cost=costs[2])
            er, acc, _ = _ops.error_sums(torch.from_numpy(ref), torch.from_numpy(hyp), -1, False, False,
                                         float(costs[0]), float(costs[1]), float(costs[2]), norm, True,
                                         group)
            PC.assert_same(er, exp, True, f"sums {R}x{H} norm={norm}")
            ref_lens = np.where((ref == -1).any(0), (ref == -1).argmax(0), R)
            got = acc.tolist()
            assert got[1:] == [float(ref_lens.sum() * group), float(n_ref * group)]
            if norm:  # fp64 sums of rounded quotients: order-dependent in the last bits
                assert abs(got[0] - float(exp.astype(np.float64).sum())) < 1e-9
            else:
                assert got[0] == float(exp.astype(np.float64).sum())


@pytest.mark.parametrize("shape", [(1, 9, 33), (20, 25, 70), (32, 40, 64), (33, 30, 31), (64, 70, 40),
                                   (65, 20, 45), (96, 101, 35), (101, 101, 40), (128, 60, 34)])
@pytest.mark.parametrize("costs", [(1, 1, 1), (3, 3, 3), (0.5, 0.5, 0.5)])
def test_bitvec_kernels_vs_oracle(F, bv_form, shape, costs, monkeypatch):
    """The unit-cost bit-vector path (lev_bitvec.cu), forced on for small batches: every
    word count W = 1..4 with reference lengths on both sides of the word boundaries,
    final and prefix outputs, ragged lengths incl. empty sequences, missing eos, the uniform
    cost multiplier, narrow and >16-bit token ranges."""
    monkeypatch.setenv("B200LEV_BITVEC", "1")
    monkeypatch.setenv("B200LEV_BITVEC_MIN_PAIRS", "1")
    R, H, N = shape
    for flags in (dict(include_eos=True, norm=True, exclude_last=False, min_frac=0.0),
                  dict(include_eos=False, norm=False, exclude_last=True, min_frac=0.4),
                  dict(include_eos=True, norm=True, exclude_last=True, min_frac=0.2, no_eos_frac=0.3),
                  dict(include_eos=False, norm=True, exclude_last=False, min_frac=0.0, eos=None)):
        # V=3000: mostly distinct tokens, so hash buckets fill up and builds are retried
        for spread, V in ((1, 5), (70001, 40), (1, 3000)):
            PC.check_vs_oracle(F, DEV, seed=R + H, R=R, H=H, N=N, V=V, costs=costs, do_mask=False,
                               padding=-3, spread=spread, **flags)


@pytest.mark.parametrize("dtype", [torch.int32, torch.int16, torch.int8])
def test_bitvec_token_dtypes_nbest_and_wide(F, bv_form, dtype, monkeypatch):
    monkeypatch.setenv("B200LEV_BITVEC", "1")
    monkeypatch.setenv("B200LEV_BITVEC_MIN_PAIRS", "1")
    PC.check_vs_oracle(F, DEV, seed=5, R=40, H=45, N=37, V=9, costs=(1, 1, 1), do_mask=False,
                       dtype=dtype, norm=True)
    test_n_best_shared_reference(F)
    PC.check_wide_tokens(F, DEV)
    PC.check_warnings(F, DEV)


@pytest.mark.parametrize("shared", [True, False], ids=["nbest", "unrelated_refs"])
@pytest.mark.parametrize("shape", [(30, 33, 12, 8), (101, 101, 9, 8), (64, 40, 5, 16), (90, 70, 20, 4)])
def test_bitvec_device_selected(F, bv_form, shape, shared, monkeypatch):
    """Default mode: the bit-vector kernels are enqueued ahead of the wavefront path and decide
    on the device -- they take n-best shaped batches (<= 4 distinct references per 32 pairs)
    and veto the others, whose work the group kernels then do.  Same numbers either way."""
    monkeypatch.delenv("B200LEV_BITVEC", raising=False)
    monkeypatch.setenv("B200LEV_BITVEC_MIN_PAIRS", "1")
    monkeypatch.setenv("B200LEV_GROUP_MIN_PAIRS", "1")
    R, H, n_utts, nbest = shape
    PC.check_nbest_batch(F, DEV, seed=R + H, R=R, H=H, n_utts=n_utts, nbest=nbest, shared=shared)
    # a reference token outside int32: vetoed on the device, the 64-bit wavefront kernel answers
    PC.check_nbest_batch(F, DEV, seed=R + H, R=R, H=H, n_utts=n_utts, nbest=nbest, shared=shared,
                         wide=True)


@pytest.mark.parametrize("shared", [True, False], ids=["nbest", "unrelated_refs"])
def test_fused_kernel_claims_blocks_from_the_counter(F, shared, monkeypatch):
    """Big batches: a warp of the fused kernel takes the block of its own index, then claims further
    blocks of 32 pairs from a global counter (forced here with a one-CTA grid: 12 blocks, 4 warps),
    in the forced mode (the counter zeroed by a memset) and the device-selected one (by the probe)."""
    monkeypatch.setenv("B200LEV_BV_SHORT", "0")
    monkeypatch.setenv("B200LEV_BVF_CTAS", "1")
    monkeypatch.setenv("B200LEV_BITVEC_MIN_PAIRS", "1")
    monkeypatch.setenv("B200LEV_GROUP_MIN_PAIRS", "1")
    for mode in ("1", None):
        if mode is None:
            monkeypatch.delenv("B200LEV_BITVEC", raising=False)
        else:
            monkeypatch.setenv("B200LEV_BITVEC", mode)
        PC.check_nbest_batch(F, DEV, seed=5, R=70, H=45, n_utts=47, nbest=8, shared=shared)


def test_bitvec_degenerate_shapes(F, bv_form, monkeypatch):
    """Forced bit-vector path on the shapes the reference's tests poke at: empty hypotheses,
    one-token references, batches that are not a multiple of 32, all-eos columns."""
    monkeypatch.setenv("B200LEV_BITVEC", "1")
    monkeypatch.setenv("B200LEV_BITVEC_MIN_PAIRS", "1")
    from oracle import oracle as O

    h = torch.tensor([[1, 2, 3], [2, 2, 2]])
    z = torch.zeros((0, 3), dtype=torch.long)
    assert F.edit_distance(h, z).tolist() == [2.0, 2.0, 2.0]  # empty hyp: all deletions
    assert F.prefix_edit_distances(h, z).shape == (1, 3)
    assert F.prefix_edit_distances(h, z).tolist() == [[2.0, 2.0, 2.0]]
    rng = np.random.default_rng(2)
    for R, H, N in ((1, 1, 1), (1, 40, 33), (128, 1, 31), (7, 3, 65)):
        ref = rng.integers(0, 3, size=(R, N))
        hyp = rng.integers(0, 3, size=(H, N))
        ref[:, 0] = 0  # eos everywhere: an empty reference (norm: SM:360-366)
        for kw in (dict(eos=0, include_eos=False, norm=True), dict(eos=0, include_eos=True, norm=False),
                   dict(eos=None, norm=True)):
            exp = O.prefix_error_rates(ref, hyp, padding=-5, **kw)
            act = F.prefix_error_rates(torch.from_numpy(ref), torch.from_numpy(hyp), padding=-5,
                                       warn=False, **kw)
            PC.assert_same(act, exp, True, f"degenerate {R}x{H}x{N} {kw}")
            exp = O.error_rate(ref, hyp, **kw)
            act = F.error_rate(torch.from_numpy(ref), torch.from_numpy(hyp), warn=False, **kw)
            PC.assert_same(act, exp, True, f"degenerate final {R}x{H}x{N} {kw}")


def test_bitvec_golden(F, bv_form, golden_sm, monkeypatch):
    monkeypatch.setenv("B200LEV_BITVEC", "1")
    monkeypatch.setenv("B200LEV_BITVEC_MIN_PAIRS", "1")
    names = [n for n in golden_sm.params if n.startswith("s")] + ["cfg1", "cfg2r", "cfg4r", "wide"]
    assert PC.check_golden_string_matching(F, DEV, golden_sm, names) >= 300


def test_pack_persistent_ctas_and_cta_histogram(F, monkeypatch):
    """Big batches: a pack CTA walks many blocks of 32 sequences and collects the (class,
    length) histogram in shared memory (forced here with a 2-CTA grid)."""
    monkeypatch.setenv("B200LEV_GROUP_MIN_PAIRS", "1")
    monkeypatch.setenv("B200LEV_PACK_CTAS", "2")
    monkeypatch.setenv("B200LEV_BITVEC", "0")
    for R, H, N in ((31, 31, 700), (70, 40, 530)):
        PC.check_vs_oracle(F, DEV, seed=R + N, R=R, H=H, N=N, V=6, costs=(1, 1, 1), do_mask=False,
                           include_eos=True, norm=True, min_frac=0.1)


@pytest.mark.parametrize("want", ["592", "5"])
def test_pack_split_along_the_sequence_axis(F, want, monkeypatch):
    """Few, long sequences: several pack CTAs share a block of 32 sequences, each taking a range
    of positions; first-eos positions meet in the workspace, the CTA with the last ticket writes
    the lengths (eos early / late / missing, tokens outside int32, N over two blocks)."""
    monkeypatch.setenv("B200LEV_PACK_SPLIT", want)
    monkeypatch.setenv("B200LEV_BITVEC", "0")
    for R, H, N in ((300, 390, 3), (390, 260, 34)):
        for include_eos in (True, False):
            PC.check_vs_oracle(F, DEV, seed=R + N, R=R, H=H, N=N, V=7, costs=(1, 2, 3), do_mask=False,
                               include_eos=include_eos, norm=True, min_frac=0.05)
    PC.check_wide_tokens(F, DEV, R=260, H=130, N=3)


def test_group_kernel_n_best_and_wide(F, monkeypatch):
    monkeypatch.setenv("B200LEV_GROUP_MIN_PAIRS", "1")
    test_n_best_shared_reference(F)
    PC.check_wide_tokens(F, DEV)


@pytest.mark.parametrize("shape", [(60, 70, 5), (130, 40, 4), (300, 90, 3), (700, 45, 2)])
@pytest.mark.parametrize("costs", [(1, 1, 1), (3, 3, 4), (0.5, 1.0, 0.25), (0.7, 1.1, 1.3)])
def test_cta_kernel_vs_oracle(F, shape, costs, monkeypatch):
    """lev_cta.cu: one CTA per pair, strips pipelined across warps, tokens staged by (emulated)
    TMA bulk copies; every C variant, cost / count / float channels, final + prefix."""
    monkeypatch.setenv("B200LEV_CTA_KERNEL", "1")
    R, H, N = shape
    for flags in (dict(include_eos=True, norm=True, exclude_last=False, min_frac=0.0),
                  dict(include_eos=False, norm=False, exclude_last=True, min_frac=0.5,
                       batch_first=True)):
        PC.check_vs_oracle(F, DEV, seed=R * 7 + H, R=R, H=H, N=N, V=5, costs=costs, do_mask=False,
                           padding=-3, **flags)


def test_warp_kernel_when_cta_disabled(F, monkeypatch):
    monkeypatch.setenv("B200LEV_CTA_KERNEL", "0")
    PC.check_vs_oracle(F, DEV, seed=3, R=130, H=40, N=4, V=5, costs=(1, 2, 3), do_mask=False)


def test_seqlp_golden(F, golden_seqlp):
    assert PC.check_golden_seqlp(F, DEV, golden_seqlp) == 84


@pytest.mark.parametrize("case", [((7, 5), 0, 33, 2), ((3, 6, 4), 1, 264, None), ((2, 4, 3, 2), -1, 9, 0),
                                  ((40,), 0, 1000, 5), ((5, 0), 0, 7, None), ((0, 5), 0, 7, 1)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_seqlp_vs_oracle(F, case, dtype):
    """Vector (16-byte) and scalar row paths (V a multiple of the vector width or not), all
    step axes, empty axes."""
    shape, dim, V, eos = case
    PC.check_seqlp_vs_oracle(F, DEV, seed=V, shape=shape, dim=dim, V=V, eos=eos, dtype=dtype)


def test_seqlp_errors_and_module(F):
    import b200lev.modules as M

    lg, hyp = torch.randn(4, 3, 5), torch.randint(0, 5, (4, 3))
    with pytest.raises(RuntimeError, match="Dimension out of range"):
        F.sequence_log_probs(lg, hyp, 2)
    with pytest.raises(RuntimeError, match="class axis"):
        F.sequence_log_probs(lg[:, :2], hyp, 0)
    m = M.SequenceLogProbabilities(1, eos=2)
    assert "dim=1, eos=2" in repr(m)
    assert torch.equal(m(lg, hyp), F.sequence_log_probs(lg, hyp, 1, 2))
    with pytest.raises(ValueError):
        M.SequenceLogProbabilities("x")


# ---- bulk-scoring front end (SURVEY 8f next #2) ---------------------------------------------
@pytest.fixture(scope="module")
def scoring(F):
    import b200lev.scoring as S

    return S


def test_scoring_golden_command_outputs(scoring, golden_scoring, tmp_path):
    """Every option set the reference command was run on: same text, same exceptions."""
    assert PC.check_golden_scoring(scoring, golden_scoring, tmp_path) == 30


def test_scoring_batches_by_cell_budget(scoring, golden_scoring):
    """A tiny budget splits the corpus into many length-sorted calls: same numbers."""
    A = golden_scoring["corpora"]["A"]
    utts = sorted(A)
    ref = scoring.TokenCorpus.from_sequences(utts, [A[u]["ref"] for u in utts], "r")
    hyp = scoring.TokenCorpus.from_sequences(utts, [A[u]["hyp"] for u in utts], "h")
    one, rl1 = scoring.score_corpora(ref, hyp, quiet=True)
    many, rl2 = scoring.score_corpora(ref, hyp, quiet=True, cell_budget=64)
    np.testing.assert_array_equal(one, many)
    np.testing.assert_array_equal(rl1, rl2)
    from oracle import oracle as O

    for k, u in enumerate(utts):  # unit costs, no eos: the plain Levenshtein distance
        r, h = np.array(A[u]["ref"], dtype=np.int64), np.array(A[u]["hyp"], dtype=np.int64)
        if h.size:
            exp = np.asarray(O.edit_distance(r[:, None], h[:, None]))[0]
        else:
            exp = r.size
        assert one[k] == exp and rl1[k] == r.size, u


def test_scoring_corpus_helpers(scoring):
    c = scoring.TokenCorpus.from_sequences(["a", "b", "c", "d"], [[1, 2, 3], [], [4], [5, 6]], "x")
    s = c.select(np.array([0, 2, 3]))
    assert s.utt_ids == ["a", "c", "d"] and s.tokens.tolist() == [1, 2, 3, 4, 5, 6]
    assert s.offsets.tolist() == [0, 3, 4, 6]
    e = c.select(np.array([1]))
    assert e.tokens.shape == (0,) and e.offsets.tolist() == [0, 0]
    with pytest.raises(ValueError, match="not aligned"):
        scoring.score_corpora(c, s)
    with pytest.raises(ValueError, match="offsets"):
        scoring.TokenCorpus(["a"], np.arange(3), np.array([0, 2]))


def test_scoring_recode_paths_agree(scoring, golden_scoring, monkeypatch):
    """Plain shift, dense table and sort-based ranking of the ids give the same errors,
    for ids that are negative, sparse or wider than 32 bits."""
    A = golden_scoring["corpora"]["A"]
    utts = sorted(A)
    base_r, base_h = [A[u]["ref"] for u in utts], [A[u]["hyp"] for u in utts]

    def corpora(f):
        return (scoring.TokenCorpus.from_sequences(utts, [[f(t) for t in s] for s in base_r], "r"),
                scoring.TokenCorpus.from_sequences(utts, [[f(t) for t in s] for s in base_h], "h"))

    want, lens = scoring.score_corpora(*corpora(lambda t: t), quiet=True)
    monkeypatch.setattr(scoring, "_CHUNK", 16)  # the threaded host passes, many small tasks
    np.testing.assert_array_equal(scoring.score_corpora(*corpora(lambda t: t), quiet=True)[0], want)
    rep, ign = {3: 5, 9: 100}, {0, -2}
    want_ri, lens_ri = scoring.score_corpora(*corpora(lambda t: t), replace=rep, ignore=ign, quiet=True)
    assert (lens_ri < lens).any()
    for f in (lambda t: t * 1000 - 7, lambda t: t * (1 << 40) - 5, lambda t: t + (1 << 33)):
        got, _ = scoring.score_corpora(*corpora(f), quiet=True)
        np.testing.assert_array_equal(got, want)
        for span in (1 << 26, 4):  # dense table / np.unique
            monkeypatch.setattr(scoring, "_DENSE_SPAN", span)
            got, gl = scoring.score_corpora(*corpora(f), replace={f(k): f(v) for k, v in rep.items()},
                                            ignore={f(t) for t in ign}, quiet=True)
            np.testing.assert_array_equal(got, want_ri)
            np.testing.assert_array_equal(gl, lens_ri)


def test_ragged_to_padded(F):
    assert PC.check_ragged_to_padded(DEV) == 36


# ---- ctc_greedy_search (SURVEY 8f next #4) -----------------------------------------------------
def test_ctc_golden(F, golden_ctc):
    assert PC.check_golden_ctc(F, DEV, golden_ctc) == 106


@pytest.mark.parametrize("batch_first", [False, True])
@pytest.mark.parametrize("shape", [(9, 4, 5), (40, 3, 37), (5, 2, 300), (70, 2, 3)])
def test_ctc_vs_oracle_with_gradient(F, shape, batch_first):
    PC.check_ctc_vs_oracle(F, DEV, seed=sum(shape), T=shape[0], N=shape[1], V=shape[2], batch_first=batch_first)
    PC.check_ctc_vs_oracle(F, DEV, seed=1 + sum(shape), T=shape[0], N=shape[1], V=shape[2],
                           batch_first=batch_first, dtype=torch.float64, with_lens=False)


def test_ctc_low_precision_ties_and_errors(F):
    """bf16 rows with many equal maxima: the lowest class index wins (as the oracle's arg max)."""
    from b200lev import _abi

    rng = np.random.default_rng(5)
    x = torch.tensor(rng.integers(-2, 3, (30, 4, 9)).astype(np.float32)).to(torch.bfloat16)
    max_, paths, out_lens = F.ctc_greedy_search(x, None, 0)
    e_max, e_paths, e_lens = PC.O.ctc_greedy_search(x.float().numpy(), None, 0)
    np.testing.assert_array_equal(paths.numpy(), e_paths)
    np.testing.assert_array_equal(out_lens.numpy(), e_lens)
    np.testing.assert_allclose(max_.float().numpy(), e_max, rtol=2e-2)
    with pytest.raises(RuntimeError, match="3-dimensional"):
        F.ctc_greedy_search(torch.zeros(3, 4))
    with pytest.raises(RuntimeError, match=r"Blank index out of range \(expected to be in the range of \[-5,4\], but got 5\)"):
        F.ctc_greedy_search(torch.zeros(3, 4, 5), None, 5)
    with pytest.raises(RuntimeError, match="in_lens must have shape"):
        F.ctc_greedy_search(torch.zeros(3, 4, 5), torch.zeros(3, dtype=torch.long))
    p = torch.full((3, 2, 4), 0.25, requires_grad=True)
    m, _, _ = F.ctc_greedy_search(p, None, -1, False, True)
    m.sum().backward()  # (is_probs=True: the product's gradient, check_ctc_probs_gradient)
    assert torch.allclose(p.grad[:, :, 0], torch.full((3, 2), 0.0625)) and float(p.grad[:, :, 1:].abs().sum()) == 0.0
    m, paths, lens = F.ctc_greedy_search(torch.zeros(0, 2, 4))
    assert m.tolist() == [0.0, 0.0] and paths.shape == (0, 2) and lens.tolist() == [0, 0]
    import b200lev.modules as M

    mod = M.CTCGreedySearch(blank_idx=0, batch_first=True)
    assert "blank_idx=0, batch_first=True, is_probs=False" == mod.extra_repr()
    assert mod(torch.zeros(2, 3, 4))[2].tolist() == [0, 0]


@pytest.mark.parametrize("N,batch_first", [(70, False), (33, True), (64, False)])
def test_completion_fill_staged_rows(F, N, batch_first):
    """Enough pairs that whole warps of the fill kernel own 32 adjacent output rows (the
    shared-memory staged path), plus the ragged last warp and rows that straddle two prefixes."""
    PC.check_vs_oracle(F, DEV, seed=N, R=11, H=9, N=N, V=5, costs=(1, 1, 1), include_eos=True,
                       batch_first=batch_first, exclude_last=False, min_frac=0.3)
    PC.check_vs_oracle(F, DEV, seed=N + 1, R=14, H=6, N=N, V=3, costs=(1, 2, 3), include_eos=False,
                       batch_first=batch_first, exclude_last=True, min_frac=0.0, padding=-7)


def test_ctc_probs_gradient(F):
    PC.check_ctc_probs_gradient(F, DEV)


def test_ctc_masked_classes(F):
    PC.check_ctc_masked_classes(F, DEV)


def test_decode_steps_golden_and_oracle(F, golden_decode):
    """SURVEY 8f #3: beam_search_advance / random_walk_advance against the reference's outputs
    and the oracle."""
    assert PC.check_golden_decode(F, DEV, golden_decode) == 26
    PC.check_decode_vs_oracle(F, DEV)


def test_completion_many_distinct_tokens(F):
    """Mask mode with more than 32 distinct reference tokens (bitmaps of several words, the
    atomic equality pass) next to the one-word chained pass (few distinct tokens), single- and
    multi-strip references."""
    for R, H, N, V in ((40, 45, 7, 1000), (300, 40, 3, 2000), (70, 30, 5, 40), (300, 35, 2, 20)):
        PC.check_vs_oracle(F, DEV, seed=R + V, R=R, H=H, N=N, V=V, costs=(1, 1, 1), include_eos=True,
                           norm=False, exclude_last=False, min_frac=0.5)


@pytest.mark.parametrize("costs", [(1, 1, 1), (2, 3, 4)])
def test_completion_packed_mask_kernel(F, costs, monkeypatch):
    """lev_mask16.cu forced on for small batches: every column count C (r + 1 <= 64 / 128 / 256),
    odd batch sizes (a duo with one pair), rows beyond the 64-row ring of the equality sheet,
    pairs of very different lengths sharing a warp, exclude_last, mixed batches where references
    with more than 32 distinct tokens stay on lev_warp_kernel, and tokens spread beyond one 16-bit
    window (the whole batch stays there)."""
    monkeypatch.setenv("B200LEV_MASK16_MIN_PAIRS", "1")
    for R, H, N, V, spread in ((20, 25, 7, 6, 1), (63, 100, 5, 20, 1), (64, 70, 4, 30, 1), (127, 40, 3, 25, 1),
                               (200, 150, 5, 30, 1), (255, 140, 2, 12, 1), (60, 70, 9, 45, 1),
                               (50, 40, 5, 10, 70001)):
        for excl in (False, True):
            PC.check_vs_oracle(F, DEV, seed=R + H, R=R, H=H, N=N, V=V, costs=costs, include_eos=not excl,
                               norm=False, exclude_last=excl, min_frac=0.0, spread=spread)


def test_completion_small_alphabets(F, monkeypatch):
    PC.check_completion_small_alphabets(F, DEV)
    monkeypatch.setenv("B200LEV_MASK16_MIN_PAIRS", "1")
    PC.check_completion_small_alphabets(F, DEV, seed=1)


def test_sequence_log_probs_packed(F, golden_seqlp_packed):
    assert PC.check_golden_seqlp_packed(F, DEV, golden_seqlp_packed) == 6
