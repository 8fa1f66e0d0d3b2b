"""Parity tests proper: the sm_100a kernels, called through the C ABI by the product
host code, against the reference's golden outputs and the CPU oracle.

Bars (stated again at the asserts in parity_cases.py): bit-exact for integer / dyadic
costs -- distances, counts, prefix tables, completion targets; rtol 1e-6 for
non-dyadic costs; 2e-6 / 2e-5 relative (with an absolute floor of 1e-6 x scale) for
fp32 losses / gradients.  Nothing here reads /root/reference.
"""
import sys

import numpy as np
import pytest
import torch

import parity_cases as PC
from oracle import oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def F():
    import b200lev.functional as F_
    from b200lev import _abi

    eb = sys.modules.get("emu_backend")  # (imported by the CPU test modules at collection)
    assert eb is None or not eb.ACTIVE, "the GPU suite must never run on the emulator seam"
    _abi.lib()  # fail loudly if the CUDA library is missing
    return F_


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda", 0)


def test_library_is_the_cuda_build(F):
    from b200lev import _abi

    from b200lev import _host

    assert _abi.lib().b200lev_device_count() >= 1
    assert _abi.lib()._name == _abi.LIB_PATH
    # host tensors compute on the GPU (and come back); devices that are neither raise
    assert _host.compute_device(torch.device("cpu")).type == "cuda"
    with pytest.raises(_abi.B200LevError, match="no CPU fallback"):
        _host.compute_device(torch.device("meta"))


def test_golden_string_matching(F, dev, golden_sm):
    assert PC.check_golden_string_matching(F, dev, golden_sm) >= 340


def test_golden_losses(F, dev, golden_loss):
    assert PC.check_golden_losses(F, dev, golden_loss) == 72


def test_sclite(F, dev, golden_sclite):
    z = golden_sclite
    ers = F.error_rate(torch.from_numpy(z["ref"]).to(dev), torch.from_numpy(z["hyp"]).to(dev),
                       eos=-1, include_eos=False, norm=False, ins_cost=3.0, del_cost=3.0,
                       sub_cost=4.0, warn=False).cpu().numpy()
    assert np.array_equal(ers, z["errs"])
    assert f"{ers.sum() / z['ref_lens'].sum():.03f}" == f"{float(z['total']):.03f}"


@pytest.mark.parametrize("costs", [(1, 1, 1), (3, 3, 4), (1, 2, 3), (0.5, 1.0, 0.25), (0.7, 1.1, 1.3)])
@pytest.mark.parametrize("shape", [(31, 33, 40), (40, 45, 33), (70, 30, 17), (130, 100, 9),
                                   (300, 260, 5), (700, 90, 3)])
@pytest.mark.parametrize("cta", ["0", "1"], ids=["warp_kernel", "cta_kernel"])
def test_random_vs_oracle(F, dev, costs, shape, cta, monkeypatch):
    """Both the warp-per-pair kernel (lev_dp.cu) and the CTA-per-pair kernel with TMA-staged
    tokens (lev_cta.cu), forced through B200LEV_CTA_KERNEL."""
    monkeypatch.setenv("B200LEV_CTA_KERNEL", cta)
    R, H, N = shape
    PC.check_vs_oracle(F, dev, seed=R * 1000 + H, R=R, H=H, N=N, V=6, costs=costs,
                       include_eos=True, norm=True, min_frac=0.4)


@pytest.mark.parametrize("flags", [
    dict(include_eos=False, norm=False, batch_first=True, exclude_last=True),
    dict(include_eos=True, norm=True, batch_first=True, exclude_last=False, no_eos_frac=0.3),
    dict(include_eos=False, norm=True, batch_first=False, exclude_last=True, eos=None),
    dict(include_eos=True, norm=False, batch_first=False, exclude_last=True, eos=-1),
])
def test_random_vs_oracle_flags(F, dev, flags):
    for seed, costs in enumerate([(1, 1, 1), (2, 1, 3), (2, 2, 2), (0.25, 0.5, 0.5)]):
        PC.check_vs_oracle(F, dev, seed=seed, R=37, H=33, N=65, V=4, costs=costs, min_frac=0.0,
                           padding=-7, **flags)


@pytest.mark.parametrize("dtype", [torch.int32, torch.int16, torch.int8])
def test_token_dtypes(F, dev, dtype):
    PC.check_vs_oracle(F, dev, seed=5, R=20, H=22, N=50, V=9, costs=(1, 1, 1), eos=-1,
                       include_eos=False, dtype=dtype)


def test_empty_and_degenerate_shapes(F, dev):
    z = torch.zeros((0, 3), dtype=torch.long, device=dev)
    h = torch.tensor([[1, 2, 3], [2, 2, 2]], device=dev)
    assert F.edit_distance(z, h).tolist() == [2.0, 2.0, 2.0]       # empty ref: all insertions
    assert F.edit_distance(h, z).tolist() == [2.0, 2.0, 2.0]       # empty hyp: all deletions
    assert F.error_rate(z, h, warn=False).tolist() == [1.0, 1.0, 1.0]  # SM:405
    assert F.error_rate(z, z, warn=False).tolist() == [0.0, 0.0, 0.0]
    assert F.prefix_edit_distances(h, z).shape == (1, 3)
    assert F.edit_distance(h[:, :0], h[:, :0]).shape == (0,)
    oc = F.optimal_completion(h, z)
    assert oc.shape[:2] == (1, 3) and oc[0, :, 0].tolist() == [1, 2, 3]


def test_cfg1_error_rate(F, dev):
    """BASELINE config 1: batch 32, T~50, vocab 30, eos-padded, unit costs."""
    rng = np.random.default_rng(1)
    ref = PC.random_tokens(rng, 51, 32, 30, 0, 0, min_len=24)
    hyp = PC.random_tokens(rng, 51, 32, 30, 0, 0, min_len=24)
    exp = O.error_rate(ref, hyp, eos=0)
    act = F.error_rate(torch.from_numpy(ref).to(dev), torch.from_numpy(hyp).to(dev), eos=0, warn=False)
    PC.assert_same(act, exp, True, "cfg1")


def test_cfg2_prefix_and_mwer(F, dev):
    """BASELINE config 2: 64 x 8-best word hyps, T=100, vocab 10k, bf16 log-probs."""
    rng = np.random.default_rng(2)
    N, M, T, V = 64, 8, 101, 10000
    ref = PC.random_tokens(rng, T, N, V, 0, 0, min_len=49)
    hyp = PC.random_tokens(rng, T, N * M, V, 0, 0, min_len=49)
    # make the hyps noisy copies of the refs half of the time so that distances vary
    for n in range(0, N * M, 2):
        r = ref[:, n // M]
        keep = rng.random(T) > 0.1
        hyp[:, n] = np.where(keep, r, hyp[:, n])
    refx = np.repeat(ref, M, axis=1)
    exp = O.prefix_error_rates(refx, hyp, eos=0)
    act = F.prefix_error_rates(torch.from_numpy(refx).to(dev), torch.from_numpy(hyp).to(dev), eos=0,
                               warn=False)
    PC.assert_same(act, exp, True, "cfg2 prefix_error_rates")
    lp = rng.standard_normal((N, M)).astype(np.float32)
    exp_loss, exp_grad = O.minimum_error_rate_loss(lp, ref, hyp.reshape(T, N, M), eos=0)
    for dtype, rtol in ((torch.float32, 2e-6), (torch.bfloat16, 2e-2)):
        x = torch.from_numpy(lp).to(dev).to(dtype).requires_grad_(True)
        if dtype != torch.float32:
            exp_loss, exp_grad = O.minimum_error_rate_loss(x.detach().float().cpu().numpy(), ref,
                                                           hyp.reshape(T, N, M), eos=0)
        loss = F.minimum_error_rate_loss(x, torch.from_numpy(ref).to(dev),
                                         torch.from_numpy(hyp.reshape(T, N, M)).to(dev), eos=0,
                                         warn=False)
        assert loss.dtype == torch.float32  # fp32 for fp32/bf16 inputs (SURVEY a8)
        loss.backward()
        assert x.grad.dtype == dtype
        np.testing.assert_allclose(loss.item(), exp_loss, rtol=rtol, atol=rtol * 1e-1)
        np.testing.assert_allclose(x.grad.float().cpu().numpy(), exp_grad, rtol=rtol * 10,
                                   atol=rtol * float(np.abs(exp_grad).max()))


def test_cfg3_completion_and_ocd(F, dev):
    """BASELINE config 3: batch 128 char seqs, T=200, V=32, include_eos."""
    rng = np.random.default_rng(3)
    N, T, V = 128, 201, 32
    ref = PC.random_tokens(rng, T, N, V, 0, 0, min_len=99)
    hyp = PC.random_tokens(rng, T, N, V, 0, 0, min_len=99)
    for n in range(0, N, 2):  # noisy copies: realistic (sparse) target sets
        keep = rng.random(T) > 0.1
        hyp[:, n] = np.where(keep, ref[:, n], hyp[:, n])
    exp = O.optimal_completion(ref, hyp, eos=0)
    tr, th = torch.from_numpy(ref).to(dev), torch.from_numpy(hyp).to(dev)
    act = F.optimal_completion(tr, th, eos=0, warn=False)
    PC.assert_same(act, exp, True, "cfg3 optimal_completion")
    logits = rng.standard_normal((T, N, V)).astype(np.float32)
    for reduction in ("mean", "none"):
        exp_loss, exp_grad = O.hard_optimal_completion_distillation_loss(
            logits, ref, hyp, eos=0, reduction=reduction, ignore_index=-100)
        x = torch.from_numpy(logits).to(dev).requires_grad_(True)
        loss = F.hard_optimal_completion_distillation_loss(x, tr, th, eos=0, reduction=reduction,
                                                           ignore_index=-100, warn=False)
        (g,) = torch.autograd.grad([loss.sum()], [x])
        np.testing.assert_allclose(loss.detach().cpu().numpy(), exp_loss, rtol=2e-6, atol=2e-6)
        np.testing.assert_allclose(g.cpu().numpy(), exp_grad, rtol=2e-5,
                                   atol=1e-6 * float(np.abs(exp_grad).max()))


def test_cfg4_bulk_slice_and_sums(F, dev):
    """BASELINE config 4 on a 100k-pair slice, plus the fp64 device accumulators."""
    from b200lev import dist as D

    rng = np.random.default_rng(4)
    P, T, V = 100_003, 31, 10000  # (not a multiple of 32: the last warp shadows the last pair)
    ref = PC.random_tokens(rng, T, P, V, -1, -2, min_len=9)
    hyp = PC.random_tokens(rng, T, P, V, -1, -2, min_len=9)
    exp = O.error_rate(ref, hyp, eos=-1, include_eos=False, norm=False)
    er, acc = D.bulk_error_rate(torch.from_numpy(ref).to(dev), torch.from_numpy(hyp).to(dev), eos=-1)
    PC.assert_same(er, exp, True, "cfg4 slice")
    ref_lens = (ref == -1).argmax(0)
    assert acc.tolist() == [float(exp.astype(np.float64).sum()), float(ref_lens.sum()), float(P)]


def test_cfg5_long_nonunit_costs(F, dev):
    """BASELINE config 5 shape (T=2000, ragged, NIST costs 3/3/4) on 24 pairs, and the
    secondary float-cost run at 1e-6."""
    rng = np.random.default_rng(5)
    N, T, V = 24, 2001, 64
    ref = PC.random_tokens(rng, T, N, V, 0, 0, min_len=199)
    hyp = PC.random_tokens(rng, T, N, V, 0, 0, min_len=199)
    tr, th = torch.from_numpy(ref).to(dev), torch.from_numpy(hyp).to(dev)
    for func in ("prefix_edit_distances", "prefix_error_rates"):
        exp = getattr(O, func)(ref, hyp, eos=0, ins_cost=3, del_cost=3, sub_cost=4)
        act = getattr(F, func)(tr, th, eos=0, ins_cost=3, del_cost=3, sub_cost=4, warn=False)
        PC.assert_same(act, exp, True, func)
    exp = O.prefix_edit_distances(ref[:600, :6], hyp[:600, :6], eos=0, ins_cost=0.7, del_cost=1.1,
                                  sub_cost=1.3)
    act = F.prefix_edit_distances(tr[:600, :6], th[:600, :6], eos=0, ins_cost=0.7, del_cost=1.1,
                                  sub_cost=1.3)
    PC.assert_same(act, exp, False, "cfg5 float costs")


def test_full_size_properties(F, dev):
    """1M pairs (config 4 size): size-independent properties instead of the oracle."""
    g = torch.Generator(device="cpu").manual_seed(9)
    P, T, V = 1_000_000, 31, 10000
    lens = torch.randint(10, 31, (P,), generator=g)
    tok = torch.randint(1, V, (T, P), generator=g)
    pos = torch.arange(T).unsqueeze(1)
    ref = torch.where(pos < lens, tok, torch.where(pos == lens, -1, -2)).to(dev)
    perm = torch.randperm(P, generator=g).to(dev)
    hyp = ref[:, perm]
    # identity: d(x, x) = 0
    assert F.edit_distance(ref, ref, eos=-1).abs().sum().item() == 0
    d_rh = F.edit_distance(ref, hyp, eos=-1, ins_cost=1, del_cost=2, sub_cost=2)
    # duality: swapping the roles of ref and hyp swaps insertions and deletions
    d_hr = F.edit_distance(hyp, ref, eos=-1, ins_cost=2, del_cost=1, sub_cost=2)
    assert torch.equal(d_rh, d_hr)
    # bounds: | |r| - |h| | * min(ins,del)  <=  d  <=  sub*min + ...; and the last valid
    # prefix row equals the final distance
    pe = F.prefix_edit_distances(ref, hyp, eos=-1, include_eos=False, ins_cost=1, del_cost=2,
                                 sub_cost=2)
    hl = (lens.to(dev))[perm]
    last = pe.gather(0, hl.unsqueeze(0)).squeeze(0)
    assert torch.equal(last, d_rh)
    assert (pe[0] == 2.0 * lens.to(dev)).all()
    # checksum against the oracle on a strided sample
    idx = torch.arange(0, P, 997, device=dev)
    exp = O.edit_distance(ref[:, idx].cpu().numpy(), hyp[:, idx].cpu().numpy(), eos=-1, ins_cost=1,
                          del_cost=2, sub_cost=2)
    assert np.array_equal(d_rh[idx].cpu().numpy(), exp)


def test_host_tensors_and_views(F, dev):
    rng = np.random.default_rng(7)
    ref = PC.random_tokens(rng, 30, 64, 9, 0, -1)
    hyp = PC.random_tokens(rng, 28, 64, 9, 0, -1)
    exp = O.error_rate(ref, hyp, eos=0)
    # host tensors in, host tensor out (the e2e path)
    out = F.error_rate(torch.from_numpy(ref).pin_memory(), torch.from_numpy(hyp).pin_memory(),
                       eos=0, warn=False)
    assert out.device.type == "cpu" and np.array_equal(out.numpy(), exp)
    # non-contiguous views + a side stream
    big = torch.zeros((60, 128), dtype=torch.long, device=dev)
    big[::2, ::2] = torch.from_numpy(ref).to(dev)
    s = torch.cuda.Stream(dev)
    s.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(s):
        out = F.error_rate(big[::2, ::2], torch.from_numpy(hyp).to(dev), eos=0, warn=False)
    s.synchronize()
    assert np.array_equal(out.cpu().numpy(), exp)


@pytest.mark.parametrize("batch_first", [False, True], ids=["seq_first", "batch_first"])
@pytest.mark.parametrize("pinned", [True, False], ids=["pinned", "pageable"])
def test_host_pipeline_matches_single_call(F, dev, batch_first, pinned, monkeypatch):
    """Large host batches flow through the three-stream block pipeline (functional.py); the
    numbers, the host-side result layout and the warnings are those of one call."""
    from b200lev import _host as Fm
    monkeypatch.setattr(Fm, "PIPE_MIN_BYTES", 1 << 16)
    rng = np.random.default_rng(11)
    n = 2000 + 37  # not a multiple of the block size
    ref = PC.random_tokens(rng, 40, n, 50, 0, -1)
    hyp = PC.random_tokens(rng, 45, n, 50, 0, -1)
    ref[:, 5] = 3  # a reference without eos: the warning must survive the blocks
    assert Fm.block_plan(torch.from_numpy(ref), torch.from_numpy(hyp), False, 1) is not None
    rt, ht = torch.from_numpy(ref), torch.from_numpy(hyp)
    if batch_first:
        rt, ht = rt.t().contiguous(), ht.t().contiguous()
    if pinned:
        rt, ht = rt.pin_memory(), ht.pin_memory()
    for fn, kw in ((F.prefix_error_rates, dict(eos=0, include_eos=True)),
                   (F.prefix_edit_distances, dict(eos=0, include_eos=False, exclude_last=True)),
                   (F.error_rate, dict(eos=0, include_eos=True)),
                   (F.edit_distance, dict(eos=0, ins_cost=1.0, del_cost=2.0, sub_cost=3.0))):
        want = fn(rt.to(dev), ht.to(dev), batch_first=batch_first, warn=False, **kw).cpu()
        got = fn(rt, ht, batch_first=batch_first, warn=False, **kw)
        assert got.device.type == "cpu" and got.shape == want.shape
        assert torch.equal(got, want), fn.__name__
    with pytest.warns(UserWarning, match="transcription in ref did not"):
        F.error_rate(rt, ht, eos=0, include_eos=True, batch_first=batch_first)
    # column views of a wider host matrix (pitch != width)
    if not batch_first:
        wide = torch.zeros((40, n + 100), dtype=torch.long)
        wide[:, 50:50 + n] = torch.from_numpy(ref)
        got = F.error_rate(wide[:, 50:50 + n], ht, eos=0, warn=False)
        assert torch.equal(got, F.error_rate(rt.to(dev), ht.to(dev), eos=0, warn=False).cpu())


def test_warnings_and_errors(F, dev):
    PC.check_warnings(F, dev)
    PC.check_errors(F, dev)


@pytest.mark.parametrize("jit_type", ["nojit", "trace", "script"])
def test_modules_jit(F, dev, jit_type):
    """Every module, plain / traced / scripted (the reference's tests do all three,
    conftest.py:166-174), on shapes other than the trace examples'."""
    import b200lev.modules as M

    PC.check_modules(F, M, dev, jit_type)


def test_fill_after_eos(F, dev):
    PC.check_fill_after_eos(F, dev)


def test_modules_host_tensors(F, dev):
    """Host tensors through the modules: computed on the GPU, returned on the host."""
    import b200lev.modules as M

    PC.check_modules(F, M, torch.device("cpu"), "script")
    PC.check_fill_after_eos(F, torch.device("cpu"))


def test_wide_tokens(F, dev):
    PC.check_wide_tokens(F, dev)


@pytest.mark.parametrize("shape", [(20, 25, 300), (31, 30, 500), (45, 50, 300), (101, 101, 4200),
                                   (201, 60, 100), (420, 40, 40), (800, 30, 20)])
@pytest.mark.parametrize("costs", [(1, 1, 1), (3, 3, 4)])
def test_group_kernel_vs_oracle(F, dev, shape, costs, monkeypatch):
    """lev_group.cu (length-bucketed lane groups) at every group width G = 1..32."""
    monkeypatch.setenv("B200LEV_GROUP_MIN_PAIRS", "1")
    R, H, N = shape
    for flags in (dict(include_eos=True, norm=True, exclude_last=False, min_frac=0.0),
                  dict(include_eos=False, norm=False, exclude_last=True, min_frac=0.4,
                       batch_first=True)):
        # spread=1: tokens fit 16 bits -> packed 2 x int16 DPX path; 70001: 32-bit path
        for spread in (1, 70001):
            PC.check_vs_oracle(F, dev, seed=R + H, R=R, H=H, N=N, V=5, costs=costs, do_mask=False,
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


@pytest.mark.parametrize("shape", [(20, 25, 300), (33, 30, 500), (64, 50, 300), (101, 101, 4200),
                                   (128, 60, 700)])
def test_bitvec_path_vs_oracle(F, bv_form, dev, shape, monkeypatch):
    """The experimental unit-cost bit-vector path (lev_bitvec.cu, B200LEV_BITVEC=1): every word
    count, final + prefix, ragged lengths, narrow and wide token ranges, uniform multiplier."""
    monkeypatch.setenv("B200LEV_BITVEC", "1")
    monkeypatch.setenv("B200LEV_BITVEC_MIN_PAIRS", "1")
    R, H, N = shape
    for costs in ((1, 1, 1), (0.5, 0.5, 0.5)):
        for flags in (dict(include_eos=True, norm=True, exclude_last=False, min_frac=0.0),
                      dict(include_eos=False, norm=False, exclude_last=True, min_frac=0.4, no_eos_frac=0.2)):
            for spread, V in ((1, 50), (70001, 50), (1, 3000)):
                PC.check_vs_oracle(F, dev, seed=R + H, R=R, H=H, N=N, V=V, costs=costs, do_mask=False,
                                   padding=-3, spread=spread, **flags)
    PC.check_wide_tokens(F, dev)


@pytest.mark.parametrize("shared", [True, False], ids=["nbest", "unrelated_refs"])
def test_bitvec_device_selected(F, bv_form, dev, shared):
    """Default mode at sizes where both paths are eligible: n-best shaped batches are taken by
    the bit-vector kernels, unrelated references (and references with tokens outside int32)
    are vetoed on the device and answered by the wavefront kernels.  Same numbers."""
    for R, H, n_utts, nbest in ((101, 101, 600, 8), (40, 60, 300, 16), (128, 30, 1100, 4),
                                (100, 600, 520, 8), (1, 50, 600, 8), (33, 1, 520, 8)):
        PC.check_nbest_batch(F, dev, seed=R, R=R, H=H, n_utts=n_utts, nbest=nbest, shared=shared)
        PC.check_nbest_batch(F, dev, seed=R, R=R, H=H, n_utts=n_utts, nbest=nbest, shared=shared,
                             wide=True)


def test_group_kernel_wide_tokens(F, dev, monkeypatch):
    monkeypatch.setenv("B200LEV_GROUP_MIN_PAIRS", "1")
    PC.check_wide_tokens(F, dev)


def test_cfg5_full_batch_properties(F, dev):
    """BASELINE config 5 at full size (256 pairs, T=2000, NIST costs) on the CTA-per-pair
    kernel: the last valid prefix row equals the final distance; identical pairs cost 0;
    a strided sample is checked against the oracle."""
    rng = np.random.default_rng(55)
    N, T, V = 256, 2001, 64
    ref = PC.random_tokens(rng, T, N, V, 0, 0, min_len=199)
    hyp = PC.random_tokens(rng, T, N, V, 0, 0, min_len=199)
    tr, th = torch.from_numpy(ref).to(dev), torch.from_numpy(hyp).to(dev)
    kw = dict(eos=0, ins_cost=3, del_cost=3, sub_cost=4)
    pe = F.prefix_edit_distances(tr, th, **kw)
    ed = F.edit_distance(tr, th, include_eos=True, **kw)
    hl = torch.from_numpy((hyp == 0).argmax(0) + 1).to(dev)
    assert torch.equal(pe.gather(0, hl.unsqueeze(0)).squeeze(0), ed)
    assert F.edit_distance(tr, tr, include_eos=True, **kw).abs().sum().item() == 0
    idx = np.arange(0, N, 37)
    exp = O.prefix_error_rates(ref[:, idx], hyp[:, idx], **kw)
    act = F.prefix_error_rates(tr[:, idx], th[:, idx], warn=False, **kw)
    PC.assert_same(act, exp, True, "cfg5 sample")


# ---- sequence_log_probs ("next #1", _decoding.py:1516-1548) --------------------------------
def test_seqlp_golden(F, dev, golden_seqlp):
    assert PC.check_golden_seqlp(F, dev, golden_seqlp) == 84


@pytest.mark.parametrize("case", [((7, 5), 0, 33, 2), ((3, 6, 4), 1, 264, None), ((2, 4, 3, 2), -1, 9, 0),
                                  ((40,), 0, 1000, 5), ((5, 0), 0, 7, None), ((64, 33), 0, 1001, 3)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16, torch.float64])
def test_seqlp_vs_oracle(F, dev, case, dtype):
    shape, dim, V, eos = case
    PC.check_seqlp_vs_oracle(F, dev, seed=V, shape=shape, dim=dim, V=V, eos=eos, dtype=dtype)


def _seqlp_torch(logits, hyp, dim, eos):
    """The same sum written with stock torch ops on the GPU (a float reference for sizes the
    oracle is too slow for): masked gather of a log_softmax."""
    V = logits.shape[-1]
    lp = torch.log_softmax(logits, -1)
    bad = (hyp < 0) | (hyp >= V)
    if eos is not None:
        is_eos = hyp == eos
        bad |= (is_eos.cumsum(dim) - is_eos.long()) > 0
    picked = lp.gather(-1, hyp.masked_fill(bad, 0).unsqueeze(-1)).squeeze(-1).masked_fill(bad, 0.0)
    return picked.sum(dim)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_seqlp_full_size_cfg2(F, dev, dtype):
    """cfg2's MWER front end: (T=100, 64 x 8 = 512, V=10000) logits (1 GB in bf16), ragged
    eos-terminated hypotheses; forward and gradient against stock torch ops."""
    g = torch.Generator(device="cpu").manual_seed(5)
    T, N, V = 100, 512, 10000
    hyp = torch.randint(1, V, (T, N), generator=g)
    lens = torch.randint(50, T + 1, (N,), generator=g)
    hyp[torch.arange(T)[:, None] >= (lens - 1)[None, :]] = 0
    hyp[3, 7] = -5  # a padding token
    hyp = hyp.to(dev)
    logits = (torch.randn(T, N, V, generator=g) * 2).to(dtype).to(dev).requires_grad_(True)
    go = torch.randn(N, generator=g).to(dtype).to(dev)
    out = F.sequence_log_probs(logits, hyp, 0, eos=0)
    (out * go).sum().backward()
    grad = logits.grad.clone()
    logits.grad = None
    exp = _seqlp_torch(logits, hyp, 0, 0)
    (exp * go).sum().backward()
    rtol, atol = PC.SEQLP_TOL[str(dtype).split(".")[-1]]
    torch.testing.assert_close(out.float(), exp.float(), rtol=rtol, atol=atol * 50)
    # compare gradients where they are not both exactly zero (skipped rows) in fp32
    torch.testing.assert_close(grad.float(), logits.grad.float(), rtol=rtol * 4, atol=atol)
    skipped = torch.arange(T, device=dev)[:, None] >= lens.to(dev)[None, :]
    assert float(grad[skipped].abs().max()) == 0.0


# ---- bulk-scoring front end (SURVEY 8f next #2) ---------------------------------------------
def test_scoring_golden_command_outputs(F, golden_scoring, tmp_path):
    import b200lev.scoring as S

    assert PC.check_golden_scoring(S, golden_scoring, tmp_path) == 30


def test_scoring_large_corpus_matches_direct_call(F, dev):
    """200 k utterances from flat arrays (int16 codes, length-sorted batches, host pipeline)
    against error_rate on the padded int64 matrices built the plain way."""
    import b200lev.scoring as S

    rng = np.random.default_rng(11)
    N, T, V = 200_000, 31, 5000
    rl = rng.integers(1, T + 1, N)
    hl = rng.integers(0, T + 1, N)
    ref = np.full((T + 1, N), -2, dtype=np.int64)
    hyp = np.full((T + 1, N), -2, dtype=np.int64)
    rt = rng.integers(0, V, (T, N))
    ht = np.where(rng.random((T, N)) < 0.7, rt, rng.integers(0, V, (T, N)))
    rows = np.arange(T)[:, None]
    ref[:T][rows < rl] = rt[rows < rl]
    hyp[:T][rows < hl] = ht[rows < hl]
    ref[rl, np.arange(N)] = -1
    hyp[hl, np.arange(N)] = -1
    exp = F.error_rate(torch.from_numpy(ref).to(dev), torch.from_numpy(hyp).to(dev), eos=-1, norm=False)
    ids = [f"u{i:07d}" for i in range(N)]
    rc = S.TokenCorpus(ids, ref[:T].T[(rows < rl).T], np.concatenate([[0], np.cumsum(rl)]), "r")
    hc = S.TokenCorpus(ids, hyp[:T].T[(rows < hl).T], np.concatenate([[0], np.cumsum(hl)]), "h")
    for budget in (S._CELL_BUDGET, 1 << 21):
        got, lens = S.score_corpora(rc, hc, quiet=True, cell_budget=budget)
        np.testing.assert_array_equal(got, exp.cpu().numpy())
        np.testing.assert_array_equal(lens, rl)


def test_ragged_to_padded(F, dev):
    assert PC.check_ragged_to_padded(dev) == 36


# ---- ctc_greedy_search (SURVEY 8f next #4) -----------------------------------------------------
def test_ctc_golden(F, dev, golden_ctc):
    assert PC.check_golden_ctc(F, dev, golden_ctc) == 106


@pytest.mark.parametrize("batch_first", [False, True])
@pytest.mark.parametrize("shape", [(9, 4, 5), (40, 3, 37), (5, 2, 300), (70, 2, 3), (120, 7, 1003)])
def test_ctc_vs_oracle_with_gradient(F, dev, shape, batch_first):
    PC.check_ctc_vs_oracle(F, dev, seed=sum(shape), T=shape[0], N=shape[1], V=shape[2], batch_first=batch_first)
    PC.check_ctc_vs_oracle(F, dev, seed=1 + sum(shape), T=shape[0], N=shape[1], V=shape[2],
                           batch_first=batch_first, dtype=torch.float64, with_lens=False)


def test_ctc_full_size_against_torch_ops(F, dev):
    """cfg2-sized logits (100, 512, 10 000) bf16: paths, lengths and score against the same
    computation written with stock torch ops on the device (fp32 log-softmax of the bf16 values)."""
    g = torch.Generator(device="cpu").manual_seed(3)
    T, N, V = 100, 512, 10_000
    x = (torch.randn((T, N, V), generator=g, dtype=torch.float32) * 2).to(torch.bfloat16).to(dev)
    lens = torch.randint(0, T + 1, (N,), generator=g).to(dev)
    max_, paths, out_lens = F.ctc_greedy_search(x, lens, 0)
    lp = x.float().log_softmax(2)
    val, arg = lp.max(2)
    valid = torch.arange(T, device=dev)[:, None] < lens[None, :]
    keep = (arg != 0) & valid
    keep[1:] &= arg[1:] != arg[:-1]
    assert torch.equal(out_lens, keep.sum(0))
    for n in range(0, N, 37):
        assert torch.equal(paths[: int(out_lens[n]), n], arg[:, n][keep[:, n]])
    exp = torch.where(valid, val, torch.zeros_like(val)).sum(0)
    torch.testing.assert_close(max_.float(), exp, rtol=2e-2, atol=1e-2)


@pytest.mark.parametrize("N,batch_first", [(70, False), (33, True), (1000, False)])
def test_completion_fill_staged_rows(F, dev, N, batch_first):
    PC.check_vs_oracle(F, dev, seed=N, R=31, H=29, N=N, V=7, costs=(1, 1, 1), include_eos=True,
                       batch_first=batch_first, exclude_last=False, min_frac=0.3)
    PC.check_vs_oracle(F, dev, seed=N + 1, R=14, H=6, N=N, V=3, costs=(1, 2, 3), include_eos=False,
                       batch_first=batch_first, exclude_last=True, min_frac=0.0, padding=-7)


def test_ctc_probs_gradient(F, dev):
    PC.check_ctc_probs_gradient(F, dev)


def test_ctc_masked_classes(F, dev):
    PC.check_ctc_masked_classes(F, dev)


def test_bench_batch_all_dp_paths_agree(F, dev, monkeypatch):
    """bench.py's own batch (cfg2 shape x 131 072 pairs): the device-selected default, the
    forced bit-vector kernels and the wavefront kernels are three independent routes to the same
    numbers -- bit-identical prefix rates and final rates; plus the oracle on a strided sample
    and d(x, x) = 0 through the n-best (shared reference) layout."""
    import bench

    ref_np, hyp_np, _ = bench.make_batch(16384, seed=0)
    ref = torch.from_numpy(np.repeat(ref_np, bench.NBEST, axis=1)).to(dev)
    hyp = torch.from_numpy(hyp_np).to(dev)
    outs = {}
    for mode in ("2", "1", "0"):
        monkeypatch.setenv("B200LEV_BITVEC", mode)
        outs[mode] = (F.prefix_error_rates(ref, hyp, eos=0, warn=False),
                      F.error_rate(ref, hyp, eos=0, include_eos=True, warn=False))
    for mode in ("1", "0"):
        assert torch.equal(outs["2"][0], outs[mode][0]), f"prefix rates differ: default vs BITVEC={mode}"
        assert torch.equal(outs["2"][1], outs[mode][1]), f"final rates differ: default vs BITVEC={mode}"
    monkeypatch.setenv("B200LEV_BITVEC", "2")
    idx = torch.arange(0, hyp.shape[1], 1013, device=dev)
    exp = O.prefix_error_rates(ref[:, idx].cpu().numpy(), hyp[:, idx].cpu().numpy(), eos=0)
    assert np.array_equal(outs["2"][0][:, idx].cpu().numpy(), np.asarray(exp, dtype=np.float32))
    assert F.error_rate(ref, ref, eos=0, include_eos=True, warn=False).abs().sum().item() == 0


def test_device_selected_fork_ordering(F, dev, monkeypatch):
    """The stand-by chain runs on a side stream beside the bit-vector kernel: back-to-back
    calls on a non-default stream, alternating batches the bit-vector kernels take (n-best) and
    veto (unrelated references), no synchronisation in between -- every result equals the
    wavefront kernels' (B200LEV_BITVEC=0) result of the same batch on the default stream."""
    import bench

    ref_np, hyp_np, _ = bench.make_batch(1024, seed=5)
    hyp = torch.from_numpy(hyp_np).to(dev)
    shared = torch.from_numpy(np.repeat(ref_np, bench.NBEST, axis=1)).to(dev)
    unrelated = torch.from_numpy(bench.make_batch(1024, seed=6)[1]).to(dev)
    monkeypatch.setenv("B200LEV_BITVEC", "0")
    want = [F.prefix_error_rates(r, hyp, eos=0, warn=False) for r in (shared, unrelated)]
    want_f = [F.error_rate(r, hyp, eos=0, warn=False) for r in (shared, unrelated)]
    torch.cuda.synchronize()
    monkeypatch.delenv("B200LEV_BITVEC")
    s = torch.cuda.Stream(dev)
    got = []
    with torch.cuda.stream(s):
        for k in range(12):
            r = (shared, unrelated)[k % 2]
            got.append((k % 2, F.prefix_error_rates(r, hyp, eos=0, warn=False),
                        F.error_rate(r, hyp, eos=0, warn=False)))
    s.synchronize()
    for which, pe, er in got:
        assert torch.equal(pe, want[which]) and torch.equal(er, want_f[which])


@pytest.mark.parametrize("which", ["nbest", "unrelated_refs"])
def test_device_selected_call_in_cuda_graph(F, dev, which):
    """The fork/join of the device-selected mode is a capturable pattern: the public call,
    captured into a CUDA graph after a warm-up call and replayed on fresh inputs copied into the
    captured buffers, gives the eager result."""
    import bench

    ref_np, hyp_np, _ = bench.make_batch(1024, seed=8)
    hyp = torch.from_numpy(hyp_np).to(dev)
    if which == "nbest":
        ref = torch.from_numpy(np.repeat(ref_np, bench.NBEST, axis=1)).to(dev)
    else:
        ref = torch.from_numpy(bench.make_batch(1024, seed=9)[1]).to(dev)
    want = F.prefix_error_rates(ref, hyp, eos=0, warn=False)  # (also the warm-up call)
    s = torch.cuda.Stream(dev)
    s.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(s):
        F.prefix_error_rates(ref, hyp, eos=0, warn=False)
    torch.cuda.current_stream(dev).wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = F.prefix_error_rates(ref, hyp, eos=0, warn=False)
    out.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, want)
    # new data through the same graph
    hyp2 = torch.from_numpy(bench.make_batch(1024, seed=10)[1]).to(dev)
    want2 = F.prefix_error_rates(ref, hyp2, eos=0, warn=False)
    hyp.copy_(hyp2)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, want2)


def test_decode_steps_golden_and_oracle(F, dev, golden_decode):
    """SURVEY 8f #3: beam_search_advance / random_walk_advance against the reference's outputs
    and the oracle, device and host tensors."""
    assert PC.check_golden_decode(F, dev, golden_decode) == 26
    PC.check_decode_vs_oracle(F, dev)
    assert PC.check_golden_decode(F, torch.device("cpu"), golden_decode) == 26


def test_completion_many_distinct_tokens(F, dev):
    """Mask mode with more than 32 distinct reference tokens (bitmaps of several words, the
    atomic equality pass) next to the one-word chained pass (few distinct tokens), single- and
    multi-strip references."""
    for R, H, N, V in ((40, 45, 7, 1000), (300, 40, 3, 2000), (70, 30, 5, 40), (300, 35, 2, 20)):
        PC.check_vs_oracle(F, dev, seed=R + V, R=R, H=H, N=N, V=V, costs=(1, 1, 1), include_eos=True,
                           norm=False, exclude_last=False, min_frac=0.5)


@pytest.mark.parametrize("costs", [(1, 1, 1), (2, 3, 4)])
def test_completion_packed_mask_kernel(F, dev, costs, monkeypatch):
    """lev_mask16.cu (two pairs per warp, 16-bit DPX) forced on for small batches -- see the
    emulator test of the same name -- and on a batch large enough to take it by default."""
    monkeypatch.setenv("B200LEV_MASK16_MIN_PAIRS", "1")
    for R, H, N, V, spread in ((20, 25, 7, 6, 1), (63, 100, 5, 20, 1), (64, 70, 4, 30, 1), (127, 40, 3, 25, 1),
                               (200, 150, 5, 30, 1), (255, 140, 2, 12, 1), (60, 70, 9, 45, 1),
                               (50, 40, 5, 10, 70001)):
        for excl in (False, True):
            PC.check_vs_oracle(F, dev, seed=R + H, R=R, H=H, N=N, V=V, costs=costs, include_eos=not excl,
                               norm=False, exclude_last=excl, min_frac=0.0, spread=spread)
    monkeypatch.delenv("B200LEV_MASK16_MIN_PAIRS")
    PC.check_vs_oracle(F, dev, seed=3, R=40, H=36, N=2500, V=24, costs=costs, include_eos=True, norm=False,
                       exclude_last=False, min_frac=0.2)


def test_grouped_references_take_the_fused_kernel(F, dev, monkeypatch):
    PC.check_grouped_references(F, dev)
    monkeypatch.setenv("B200LEV_BITVEC", "0")  # the same batches through the wavefront kernels
    PC.check_grouped_references(F, dev, seed=1)


def test_completion_small_alphabets(F, dev, monkeypatch):
    PC.check_completion_small_alphabets(F, dev)
    monkeypatch.setenv("B200LEV_MASK16_MIN_PAIRS", "1")
    PC.check_completion_small_alphabets(F, dev, seed=1)


@pytest.mark.parametrize("N", [33, 37, 64, 65, 97])
def test_completion_target_writer_alignment(F, dev, N):
    """The target writer stores 16 bytes per lane where a warp's run of 32 rows starts on an even
    element, and 8 bytes where it does not (odd set size x odd batch size): both must be exact."""
    for V in (3, 4, 7):
        PC.check_vs_oracle(F, dev, seed=N + V, R=21, H=19, N=N, V=V, costs=(1, 1, 1), include_eos=True,
                           norm=False, exclude_last=False, min_frac=0.3)


def test_sequence_log_probs_packed(F, dev, golden_seqlp_packed):
    assert PC.check_golden_seqlp_packed(F, dev, golden_seqlp_packed) == 6
