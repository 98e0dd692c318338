"""Every launch path of the GAE reverse scan (gae_reverse_scan in csrc/carenv_kernels.cu) bit-exact against
oracle.carenv_port.gae_port, the float32 restatement pinned to the reference's golden vectors:

  k_gae<8>, one column per thread        T < 512 with N < 100,000, and T >= 512 while N fits one resident wave
  k_gae<8>, >= 2 columns per thread      T >= 512 and N above the resident threads of one wave
  k_gae<16>                              T < 512 and N >= 100,000

at shapes around the unroll depths (tails of 0..15 steps), for several (gamma, lambda) pairs, and the input forms the
wrapper accepts.  Also the wrapper's checks of caller-provided output buffers.
"""
import numpy as np
import pytest
import torch

import ppo_car_b200
from oracle.carenv_port import gae_port

pytestmark = pytest.mark.gpu

# (0.9, 0.8): gamma * lambda evaluated in double and rounded (0.72) differs from the float32 product (0.71999997)
GAMMA_LAMBDA = [(0.99, 0.95), (0.9, 0.8), (1.0, 1.0), (0.99, 0.0)]


def _inputs(T, N, seed):
    """rew, val, term, trunc [T, N] and last_val, last_term, last_trunc [N] on the GPU; term and trunc are 0/1 with
    steps where both are set, and the last flags are set for some columns."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    u = lambda *s: torch.rand(s, generator=g, device="cuda")
    rew = u(T, N) * 1.4 - 0.3
    val = torch.randn((T, N), generator=g, device="cuda")
    term = (u(T, N) < 0.05).float()
    trunc = (u(T, N) < 0.05).float()
    both = u(T, N) < 0.01
    term[both] = 1.0
    trunc[both] = 1.0
    lv = torch.randn(N, generator=g, device="cuda")
    lt, lu = (u(N) < 0.1).float(), (u(N) < 0.1).float()
    return rew, val, term, trunc, lv, lt, lu


def _check(inputs, pairs=GAMMA_LAMBDA):
    host = [t.cpu().numpy() for t in inputs]
    for gamma, lam in pairs:
        adv, ret = ppo_car_b200.gae_reverse_scan(*inputs, gamma=gamma, gae_lambda=lam)
        ra, rr = gae_port(*host, gamma=gamma, gae_lambda=lam)
        assert np.array_equal(adv.cpu().numpy(), ra), (gamma, lam)
        assert np.array_equal(ret.cpu().numpy(), rr), (gamma, lam)


def test_the_gamma_lambda_pairs_discriminate():
    """For (0.9, 0.8) forming gamma * lambda in float32 gives another value than rounding the double product, so a
    kernel that does the former fails the bit-exact comparisons below."""
    assert np.float32(0.9 * 0.8) != np.float32(np.float32(0.9) * np.float32(0.8))
    assert np.float32(0.99 * 0.95) == np.float32(np.float32(0.99) * np.float32(0.95))


@pytest.mark.parametrize("N", [1, 63, 65, 4099])
@pytest.mark.parametrize("T", [1, 7, 8, 9, 63, 511])
def test_unroll8_one_column_per_thread(T, N):
    _check(_inputs(T, N, seed=T * 10007 + N))


@pytest.mark.parametrize("T,N", [(512, 1), (512, 97), (513, 65), (1031, 4099)])
def test_unroll8_one_wave_with_one_column_per_thread(T, N):
    _check(_inputs(T, N, seed=T * 10007 + N))


@pytest.mark.parametrize("T", [512, 519])
def test_unroll8_several_columns_per_thread(T):
    """N = 310,001 is more than the device can hold resident (SMs x 2,048 threads), so every thread of the one-wave
    grid walks at least two columns."""
    N = 310_001
    props = torch.cuda.get_device_properties(0)
    assert N > props.multi_processor_count * props.max_threads_per_multi_processor
    _check(_inputs(T, N, seed=T), pairs=[(0.99, 0.95), (0.9, 0.8)])


@pytest.mark.parametrize("N", [100_000, 100_003])
@pytest.mark.parametrize("T", [1, 15, 16, 17, 37, 511])
def test_unroll16_wide(T, N):
    _check(_inputs(T, N, seed=T * 7 + N), pairs=[(0.99, 0.95), (0.9, 0.8)] if T > 40 else GAMMA_LAMBDA)


def test_unroll16_wide_multiple_of_the_unroll():
    _check(_inputs(128, 262_147, seed=5), pairs=[(0.99, 0.95), (0.9, 0.8)])


def test_input_forms():
    """A transposed (non-contiguous) rew, bool and int term / trunc, last_* as (N,) and as (1, N), all give the
    port's result; T = 0 or N = 0 gives empty outputs."""
    T, N = 77, 300
    rew, val, term, trunc, lv, lt, lu = _inputs(T, N, seed=3)
    want = gae_port(*(t.cpu().numpy() for t in (rew, val, term, trunc, lv, lt, lu)))
    rew_t = rew.t().contiguous().t()                               # same values, column-major storage
    assert not rew_t.is_contiguous()
    forms = [
        (rew_t, val, term, trunc, lv, lt, lu),
        (rew, val, term.bool(), trunc.bool(), lv, lt.bool(), lu.bool()),
        (rew, val, term.to(torch.int32), trunc.to(torch.int64), lv, lt.to(torch.int32), lu.to(torch.uint8)),
        (rew, val, term, trunc, lv.reshape(1, N), lt.reshape(1, N), lu.reshape(1, N)),
    ]
    for form in forms:
        adv, ret = ppo_car_b200.gae_reverse_scan(*form)
        assert np.array_equal(adv.cpu().numpy(), want[0]) and np.array_equal(ret.cpu().numpy(), want[1])
    for T0, N0 in ((0, 5), (5, 0)):
        z, last = torch.zeros((T0, N0), device="cuda"), torch.zeros(N0, device="cuda")
        adv, ret = ppo_car_b200.gae_reverse_scan(z, z, z, z, last, last, last)
        assert adv.shape == (T0, N0) and ret.shape == (T0, N0)


def test_output_buffers_are_checked_before_the_launch():
    """adv_out / ret_out must be contiguous float32 (T, N) tensors on rew's device: a larger buffer, a float64 one and
    a transposed view of an (N, T) tensor are refused with ValueError and left untouched; a right one is filled."""
    T, N = 40, 70
    inputs = _inputs(T, N, seed=4)
    want = gae_port(*(t.cpu().numpy() for t in inputs))
    good = lambda: torch.full((T, N), 7.0, device="cuda")
    wrong = [torch.full((T + 1, N), 7.0, device="cuda"), torch.full((T, N + 1), 7.0, device="cuda"),
             torch.full((T * N + 8,), 7.0, device="cuda"), torch.full((T, N), 7.0, device="cuda", dtype=torch.float64),
             torch.full((N, T), 7.0, device="cuda").t()]
    for bad in wrong:
        for kw in (dict(adv_out=bad, ret_out=good()), dict(adv_out=good(), ret_out=bad)):
            with pytest.raises(ValueError):
                ppo_car_b200.gae_reverse_scan(*inputs, **kw)
            torch.cuda.synchronize()
            assert bool((kw["adv_out"] == 7.0).all()) and bool((kw["ret_out"] == 7.0).all())
    adv_out, ret_out = good(), good()
    adv, ret = ppo_car_b200.gae_reverse_scan(*inputs, adv_out=adv_out, ret_out=ret_out)
    assert adv is adv_out and ret is ret_out
    assert np.array_equal(adv.cpu().numpy(), want[0]) and np.array_equal(ret.cpu().numpy(), want[1])
