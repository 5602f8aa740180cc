"""compressor / expander on the GPU through the C ABI vs the CPU oracle and the reference golden.

Tolerance (north star): 1e-4 relative fp32, judged per item against the fp64 arbiter with the
SURVEY.md 8c rule err(new) <= max(1e-4, err(ref fp32))."""
import numpy as np
import pytest
import torch

import oracle
from conftest import load_golden
from helpers import COMP_RANGES, SR, denorm, param_grad_err, peak_err, run_with_grads

pytestmark = pytest.mark.gpu
TOL = 1e-4


def _inputs(bs, chs, n, seed, attack_max01=1.0):
    g = torch.Generator().manual_seed(seed)
    level = torch.rand(bs, 1, 1, generator=g)
    x = (torch.rand(bs, chs, n, generator=g) * 2 - 1) * level
    p01 = torch.rand(bs, 6, generator=g)
    p01[:, 4] = p01[:, 4].clamp(min=0.05)        # knee > 0 (W == 0 gives NaN grads in the reference too)
    p01[:, 2] *= attack_max01
    return x, p01


def _check(cuda_device, fn_gpu, fn_orc, x, params, grads=True, extra=None):
    extra = extra or {}
    y, dx, dp = run_with_grads(lambda xx, p: fn_gpu(xx, SR, *p, **extra), x, params, torch.float32, cuda_device)
    y64, dx64, dp64 = run_with_grads(lambda xx, p: fn_orc(xx, SR, *p, **extra), x, params, torch.float64, "cpu")
    y32, dx32, dp32 = run_with_grads(lambda xx, p: fn_orc(xx, SR, *p, **extra), x, params, torch.float32, "cpu")
    e, e32 = peak_err(y, y64), peak_err(y32, y64)
    assert (e <= torch.clamp(e32, min=TOL)).all(), (e, e32)
    if grads:
        e, e32 = peak_err(dx, dx64), peak_err(dx32, dx64)
        assert (e <= torch.clamp(e32, min=TOL)).all(), ("dx", e, e32)
        assert dp[3] is None and dp64[3] is None                      # release_ms: no gradient
        e, e32 = param_grad_err(dp, dp64), param_grad_err(dp32, dp64)
        assert (e <= torch.clamp(e32, min=TOL)).all(), ("dparam", e, e32)


def test_compressor_golden(cuda_device):
    import dasp_pytorch_b200 as D
    g = load_golden("compressor.npz")
    names = [str(s) for s in g["names"]]
    s = int(g["t_stride"])         # per-sample reference arrays are stored at every s-th time index
    params = denorm(g["p01"], COMP_RANGES)
    y, dx, dp = run_with_grads(lambda xx, p: D.compressor(xx, SR, *p), g["x"], params, torch.float32, cuda_device)
    # item 0 has a 90 ms attack at N=4096: the reference time-aliases there (tests/test_oracle_golden.py)
    assert peak_err(y[..., ::s], g["comp_y64"])[1:].max() < TOL
    assert peak_err(dx[..., ::s], g["comp_dx64"])[1:].max() < TOL
    ref = [None if n == "release_ms" else torch.as_tensor(g[f"comp_d_{n}"]) for n in names]
    assert param_grad_err(dp, ref)[1:].max() < TOL
    y7 = D.compressor(torch.as_tensor(g["x"]).to(cuda_device), SR, *[p.to(cuda_device) for p in params],
                      lookahead_samples=7).cpu()
    assert peak_err(y7[..., ::s], g["comp_la7_y64"])[1:].max() < TOL


@pytest.mark.parametrize("bs,chs,n", [(8, 2, 48000), (3, 1, 48000), (2, 3, 20000)])
def test_compressor_full_ranges_vs_oracle(cuda_device, bs, chs, n):
    import dasp_pytorch_b200 as D
    x, p01 = _inputs(bs, chs, n, seed=5)
    _check(cuda_device, D.compressor, oracle.compressor, x, denorm(p01, COMP_RANGES))


def _ragged_check(cuda_device, bs, chs, n, seed):
    import dasp_pytorch_b200 as D
    x, p01 = _inputs(bs, chs, n, seed=seed)
    params = denorm(p01, COMP_RANGES)
    y, dx, dp = run_with_grads(lambda xx, p: D.compressor(xx, SR, *p), x, params, torch.float32, cuda_device)
    y64, dx64, dp64 = run_with_grads(lambda xx, p: oracle.compressor(xx, SR, *p, fsm_tail=1 << 16), x, params,
                                     torch.float64, "cpu")
    yt = oracle.compressor(x.double(), SR, *[p.double() for p in params], smoother="recursion")
    assert (peak_err(y64, yt) < 1e-9).all()          # enlarged grid == recursion
    assert (peak_err(y, y64) < TOL).all()
    assert (peak_err(dx, dx64) < TOL).all()
    assert (param_grad_err(dp, dp64) < 10 * TOL).all()


@pytest.mark.parametrize("bs,chs,n", [(2, 2, 4097), (3, 2, 100), (2, 1, 1), (2, 2, 224 * 8 + 4), (5, 3, 3000)])
def test_compressor_ragged_shapes(cuda_device, bs, chs, n):
    """unaligned N (scalar path), N smaller than a tile, 3 channels.  At these small N the reference's FFT grid
    time-aliases the smoother tail, so the arbiter here is the oracle with an enlarged grid (fsm_tail:
    alias-free == true recursion, still differentiable)."""
    _ragged_check(cuda_device, bs, chs, n, seed=6)


@pytest.mark.parametrize("warps", [1, 2, 4, 8, 16])
def test_compressor_every_warps_per_item_variant(cuda_device, warps):
    """pin each warps-per-item kernel variant (test hook) on a small batch with several tiles + a ragged tail"""
    from dasp_pytorch_b200 import _abi
    _abi.lib().dasp_debug_force_warps(warps)
    try:
        _ragged_check(cuda_device, 3, 2, 224 * 8 * 2 + 36, seed=16 + warps)
    finally:
        _abi.lib().dasp_debug_force_warps(0)


def test_compressor_lookahead_grads(cuda_device):
    import dasp_pytorch_b200 as D
    x, p01 = _inputs(4, 2, 30000, seed=7)
    _check(cuda_device, D.compressor, oracle.compressor, x, denorm(p01, COMP_RANGES), extra={"lookahead_samples": 33})


def test_expander_vs_oracle(cuda_device):
    import dasp_pytorch_b200 as D
    x, p01 = _inputs(6, 2, 40000, seed=8)
    params = denorm(p01, COMP_RANGES)
    params[1] = params[1].clamp(max=4.0)     # expansion ratio 1..4 keeps the gain in float range
    _check(cuda_device, D.expander, oracle.expander, x, params)


def test_compressor_identity_below_threshold_full_size(cuda_device):
    """BASELINE config-3 size (512 x 2 x 48000): below T - W/2 the compressor is a pure makeup gain
    (functional.py:352), whatever the smoother does; and the op is 1-homogeneous in nothing else."""
    import dasp_pytorch_b200 as D
    torch.manual_seed(0)
    bs = 512
    x = (torch.rand(bs, 2, 48000, device=cuda_device) * 2 - 1) * 1e-3     # peak -54 dBFS (sum of 2 ch)
    one = torch.ones(bs, device=cuda_device)
    mk = torch.linspace(0, 12, bs, device=cuda_device)
    y = D.compressor(x, SR, -20 * one, 4 * one, 10 * one, 10 * one, 6 * one, mk)
    expect = x * (10 ** (mk / 20)).view(bs, 1, 1)
    assert torch.allclose(y, expect, rtol=3e-6, atol=0)
    # ratio 1 is the identity for any level
    x1 = torch.rand(bs, 2, 48000, device=cuda_device) * 2 - 1
    y1 = D.compressor(x1, SR, -30 * one, one, 10 * one, 10 * one, 6 * one, 0 * one)
    assert torch.allclose(y1, x1, rtol=3e-6, atol=0)


def test_dynamics_param_contract(cuda_device):
    import dasp_pytorch_b200 as D
    x = torch.rand(3, 2, 2000, device=cuda_device) - 0.5
    p = [torch.full((3,), v, device=cuda_device) for v in (-20.0, 4.0, 10.0, 50.0, 6.0, 3.0)]
    y0 = D.compressor(x, SR, *p)
    y1 = D.compressor(x, SR, *[q.view(3, 1) for q in p])            # any shape with bs elements
    y2 = D.compressor(x, SR, threshold_db=p[0], ratio=p[1], attack_ms=p[2], release_ms=p[3] * 0 + 5, knee_db=p[4],
                      makeup_gain_db=p[5])                          # keyword names are ABI; release ignored
    assert torch.equal(y0, y1) and torch.equal(y0, y2)
    with pytest.raises(RuntimeError):
        D.compressor(x, SR, p[0][:2], *p[1:])


@pytest.mark.parametrize("n,attack_ms", [(1024, 100.0), (8192, 100.0), (8192, 5.0), (48000, 100.0)])
def test_compressor_gap_to_the_frequency_sampling_reference(cuda_device, n, attack_ms):
    """The kernels run the TRUE zero-state recursion of the attack smoother; the reference evaluates it by frequency
    sampling on an n_fft = 2^ceil(log2(2n-1)) grid (signal.py:95-133), which time-aliases the smoother's tail: the wrapped
    contribution is ~ alpha^(n_fft - n) of the gain curve (alpha = exp(-ln 9 / (sr * attack)): 100 ms at 44.1 kHz and
    n = 1024 -> alpha^1024 = 0.60; n = 8192 -> 1.7e-2; n = 48000 -> 1e-18).  This test TRACKS that gap instead of
    hiding it: the distance of the GPU result from the reference-faithful oracle (fsm_tail = 0) must equal the distance
    of the alias-free oracle from it (to 1e-4 in the per-item peak metric) -- i.e. the only difference to the reference IS
    the documented aliasing term, which is large at small n (the wrapped dB values go through 10^(dB/20)) -- and at the
    BASELINE length the gap itself is below 1e-4."""
    import dasp_pytorch_b200 as D
    bs = 3
    x, p01 = _inputs(bs, 2, n, seed=n)
    params = denorm(p01, COMP_RANGES)
    params[2] = torch.full((bs,), attack_ms)
    xs = x.to(cuda_device)
    y = D.compressor(xs, SR, *[p.to(cuda_device) for p in params]).cpu().double()
    ref = oracle.compressor(x.double(), SR, *[p.double() for p in params])                        # reference arithmetic
    truth = oracle.compressor(x.double(), SR, *[p.double() for p in params], fsm_tail=1 << 18)    # no wrap-around
    gap_gpu, gap_truth = peak_err(y, ref), peak_err(truth, ref)
    assert (peak_err(y, truth) < TOL).all()
    # triangle inequality in the per-item peak metric: the two gaps can differ by at most err(y, truth) * max|truth| / max|ref|
    scale = truth.reshape(bs, -1).abs().amax(1) / ref.reshape(bs, -1).abs().amax(1)
    assert ((gap_gpu - gap_truth).abs() <= TOL * torch.clamp(scale, min=1.0)).all(), (gap_gpu, gap_truth)
    alpha = float(torch.exp(-torch.log(torch.tensor(9.0)) / (SR * attack_ms * 1e-3)))
    n_fft = 1 << (2 * n - 1 - 1).bit_length()
    wrapped = alpha ** (n_fft - n)                 # share of the gain curve (in dB) that wraps around: 0.60 / 1.7e-2 / 3.5e-36 / 1e-18
    if wrapped < 1e-6:
        assert gap_truth.max() < TOL               # BASELINE length, or a short attack: the reference IS the recursion
    else:
        assert gap_truth.max() > 1e-3              # the reference itself is visibly aliased here (recorded, not hidden)
