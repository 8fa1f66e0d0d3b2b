"""The fused bit-vector kernel's hash keys (lev_bitvec.cuh): a way holds (x << s) | position with
x = token * multiplier, a free way the all-ones residual and the position R.  These cases aim at
that format -- tokens whose residual is the free ways', tokens that share a residual or agree
mod 2^(32 - s), INT32_MIN, 64-bit tokens whose low word is a reference token, full tables -- and
check the fused kernel bit for bit against the oracle, on the emulator and on the device."""
import sys

import numpy as np
import pytest
import torch

import parity_cases as PC
from oracle import oracle as O

SEED0_MULT = 0x9E3779B1  # lev_bv_mult(0): the multiplier of a build that needs no retry
INT32_MIN = -(2**31)


@pytest.fixture(scope="module", params=["emu", pytest.param("gpu", marks=pytest.mark.gpu)])
def backend(request):
    if request.param == "emu":
        from emu_backend import emulated_kernels

        with emulated_kernels():
            import b200lev.functional as F_

            yield F_, torch.device("cpu")
    else:
        import b200lev.functional as F_
        from b200lev import _abi

        eb = sys.modules.get("emu_backend")
        assert eb is None or not eb.ACTIVE, "the GPU cases must not run on the emulator seam"
        _abi.lib()
        yield F_, torch.device("cuda", 0)


@pytest.fixture(autouse=True)
def fused_kernel(monkeypatch):
    monkeypatch.setenv("B200LEV_BITVEC", "1")
    monkeypatch.setenv("B200LEV_BITVEC_MIN_PAIRS", "1")
    monkeypatch.setenv("B200LEV_BV_SHORT", "0")


def slots_log2(R):
    s = 4
    while (1 << s) <= R:
        s += 1
    return s


def token_of(x):
    """The int32 token whose product with the seed-0 multiplier is x (mod 2^32)."""
    v = (x * pow(SEED0_MULT, -1, 1 << 32)) % (1 << 32)
    return v - (1 << 32) if v >= 1 << 31 else v


def batch(rng, R, H, n_ref, pool_ref, pool_hyp, nbest=8):
    """n_ref references of R tokens drawn from pool_ref, nbest hypotheses of H tokens each drawn
    from pool_hyp; eos 0 at a random place in most columns."""
    ref = rng.choice(np.asarray(pool_ref, dtype=np.int64), size=(R, n_ref))
    hyp = rng.choice(np.asarray(pool_hyp, dtype=np.int64), size=(H, n_ref * nbest))
    for a in (ref, hyp):
        for n in range(a.shape[1]):
            if rng.random() < 0.8:
                a[rng.integers(0, a.shape[0]), n] = 0
    return np.repeat(ref, nbest, axis=1), hyp


def check(F, dev, ref, hyp, what, dtype=torch.int64):
    r = torch.from_numpy(ref).to(dtype).to(dev)
    h = torch.from_numpy(hyp).to(dtype).to(dev)
    for kw in (dict(eos=0), dict(eos=0, include_eos=False, norm=False), dict(eos=None)):
        exp = O.prefix_error_rates(ref, hyp, padding=-2, **kw)
        PC.assert_same(F.prefix_error_rates(r, h, padding=-2, warn=False, **kw), exp, True, f"{what} prefix {kw}")
        exp = O.error_rate(ref, hyp, **kw)
        PC.assert_same(F.error_rate(r, h, warn=False, **kw), exp, True, f"{what} final {kw}")


@pytest.mark.parametrize("R", [101, 127, 128, 64])
def test_tokens_with_the_free_way_residual(backend, R):
    """Tokens whose residual is all ones -- what a free way holds -- in several buckets, absent from
    some references and present in others, among common tokens."""
    F, dev = backend
    s = slots_log2(R)
    ones = (1 << (32 - s)) - 1
    special = [token_of((b << (32 - s)) | ones) for b in (0, 1, 5, (1 << s) // 3, (1 << s) - 1)]
    rng = np.random.default_rng(R)
    common = list(range(1, 12))
    ref, hyp = batch(rng, R, R - 7, 9, common + special[:3], common + special)
    check(F, dev, ref, hyp, f"free-way residual R={R}")
    check(F, dev, ref, hyp, f"free-way residual R={R} int32", torch.int32)


@pytest.mark.parametrize("R", [101, 128])
def test_tokens_sharing_a_residual(backend, R):
    """Tokens with one residual in different buckets, and tokens equal mod 2^(32 - s): the
    residual alone or the low bits alone must not make a match."""
    F, dev = backend
    s = slots_log2(R)
    res = 0x2A5 & ((1 << (32 - s)) - 1)
    same_res = [token_of((b << (32 - s)) | res) for b in (3, 4, 9, (1 << s) - 2)]
    base = [7, 123456, -98765]
    same_low = [v + k * (1 << (32 - s)) for v in base for k in (1, 2, -1)]
    rng = np.random.default_rng(3)
    ref, hyp = batch(rng, R, R, 9, [1, 2, 3] + same_res[:2] + base, [1, 2, 3] + same_res + base + same_low)
    check(F, dev, ref, hyp, f"shared residual R={R}")
    check(F, dev, ref, hyp, f"shared residual R={R} int32", torch.int32)


def test_int32_min_token(backend):
    F, dev = backend
    rng = np.random.default_rng(4)
    ref, hyp = batch(rng, 101, 90, 9, [1, 2, 3, INT32_MIN], [1, 2, 3, 4, INT32_MIN, INT32_MIN + 1])
    check(F, dev, ref, hyp, "INT32_MIN")
    check(F, dev, ref, hyp, "INT32_MIN int32", torch.int32)


def test_full_tables(backend):
    """A reference of R = 128 distinct tokens (every bucket of 4 ways busy, retried builds), R = 127
    and R = 128 with a small alphabet."""
    F, dev = backend
    rng = np.random.default_rng(5)
    for R in (127, 128):
        ref = np.stack([rng.permutation(np.arange(1, 5000))[:R] for _ in range(6)], axis=1)
        ref = np.repeat(ref, 8, axis=1)
        hyp = np.where(rng.random((R, 48)) < 0.7, ref, rng.integers(1, 5000, (R, 48)))
        hyp[rng.integers(0, R, 48), np.arange(48)] = 0
        check(F, dev, ref, hyp, f"distinct R={R}")
        ref, hyp = batch(rng, R, 70, 7, list(range(1, 6)), list(range(1, 7)))
        check(F, dev, ref, hyp, f"small alphabet R={R}")


def test_wide_hypothesis_tokens_with_a_reference_low_word(backend):
    """64-bit hypothesis tokens whose low word is a reference token: no match."""
    F, dev = backend
    rng = np.random.default_rng(6)
    common = [1, 2, 3, 77, -5]
    wide = [v + (k << 32) for v in common for k in (1, -1, 3)]
    ref, hyp = batch(rng, 101, 101, 9, common, common + wide)
    check(F, dev, ref, hyp, "wide hypothesis tokens")
