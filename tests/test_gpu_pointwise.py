"""gain / distortion on the GPU through the C ABI vs the CPU oracle and the reference golden."""
import numpy as np
import pytest
import torch

import oracle
from conftest import load_golden
from helpers import SR, peak_err, run_with_grads

pytestmark = pytest.mark.gpu


def test_distortion_golden(cuda_device):
    import dasp_pytorch_b200 as D
    g = load_golden("pointwise.npz")
    s = int(g["t_stride"])         # per-sample reference arrays are stored at every s-th time index
    y, dx, dp = run_with_grads(lambda x, p: D.distortion(x, 16000, p[0]), g["dist_x"], [g["dist_db"]],
                               torch.float32, cuda_device)
    assert peak_err(y[..., ::s], g["dist_y64"]).max() < 1e-5        # tolerance: 1e-4 rel fp32 (north star); observed ~1e-7
    assert peak_err(y[..., ::s], g["dist_y32"]).max() < 1e-5
    assert peak_err(dx[..., ::s], g["dist_dx64"]).max() < 1e-5
    assert np.allclose(dp[0].numpy(), g["dist_d_drive_db"], rtol=1e-4, atol=1e-9)
    # stereo: one drive per (item, channel) row
    y, dx, dp = run_with_grads(lambda x, p: D.distortion(x, SR, p[0]), g["dist2_x"], [g["dist2_db"]],
                               torch.float32, cuda_device)
    assert peak_err(y[..., ::s], g["dist2_y64"]).max() < 1e-5
    assert np.allclose(dp[0].numpy(), g["dist2_d_drive_db"], rtol=1e-4, atol=1e-9)


def test_gain_golden(cuda_device):
    import dasp_pytorch_b200 as D
    g = load_golden("pointwise.npz")
    s = int(g["t_stride"])
    y, dx, dp = run_with_grads(lambda x, p: D.gain(x, SR, p[0]), g["gain_x"], [g["gain_db"]], torch.float32,
                               cuda_device)
    assert peak_err(y[..., ::s], g["gain_y64"]).max() < 1e-5
    assert peak_err(dx[..., ::s], g["gain_dx64"]).max() < 1e-5
    assert np.allclose(dp[0].numpy(), g["gain_d_gain_db"], rtol=1e-4, atol=1e-9)


@pytest.mark.parametrize("shape", [(3, 2, 48000), (2, 1, 4097), (5, 3, 1), (1, 1, 3), (2, 2, 12290)])
def test_pointwise_shapes_vs_oracle(cuda_device, shape):
    """ragged / unaligned / tiny lengths (scalar path when N % 4 != 0)"""
    import dasp_pytorch_b200 as D
    torch.manual_seed(1)
    bs, chs, n = shape
    x = torch.rand(shape) * 2 - 1
    drive = torch.rand(bs * chs) * 24
    gdb = torch.rand(bs) * 48 - 24
    for fn_g, fn_o, p in ((D.distortion, oracle.distortion, drive), (D.gain, oracle.gain, gdb)):
        y, dx, dp = run_with_grads(lambda xx, q: fn_g(xx, SR, q[0]), x, [p], torch.float32, cuda_device)
        yo, dxo, dpo = run_with_grads(lambda xx, q: fn_o(xx, SR, q[0]), x, [p], torch.float64, "cpu")
        assert peak_err(y, yo).max() < 1e-5
        assert (dx.double() - dxo).abs().max() <= 1e-5 * dxo.abs().max() + 1e-12
        assert (dp[0].double() - dpo[0]).abs().max() <= 1e-4 * dpo[0].abs().max() + 1e-12


def test_pointwise_param_shapes_and_errors(cuda_device):
    import dasp_pytorch_b200 as D
    x = torch.rand(4, 1, 256, device=cuda_device)
    d = torch.rand(4, device=cuda_device)
    y0 = D.distortion(x, SR, d)
    for shp in [(4, 1), (4, 1, 1), (1, 4)]:
        assert torch.equal(D.distortion(x, SR, d.view(shp)), y0)
    # README quickstart: 0-dim drive with bs = chs = 1
    y = D.distortion(x[:1], SR, torch.tensor(16.0, device=cuda_device))
    assert y.shape == (1, 1, 256)
    with pytest.raises(RuntimeError):
        D.distortion(torch.rand(2, 2, 16, device=cuda_device), SR, torch.rand(2, device=cuda_device))
    with pytest.raises(RuntimeError):
        D.gain(x, SR, torch.rand(3, device=cuda_device))
    with pytest.raises(D.functional.DaspError):
        D.gain(x.cpu(), SR, d.cpu())
    # fp64 in -> fp64 out (computed in fp32)
    y64 = D.gain(x.double(), SR, d.double())
    assert y64.dtype == torch.float64
    # empty batch / empty time axis
    assert D.gain(x[:0], SR, d[:0]).shape == (0, 1, 256)
    assert D.distortion(x[:, :, :0], SR, d).shape == (4, 1, 0)


def test_pointwise_full_size_properties(cuda_device):
    """BASELINE config-5 shape: size-independent properties instead of an oracle run."""
    import dasp_pytorch_b200 as D
    torch.manual_seed(0)
    x = (torch.rand(1024, 2, 48000, device=cuda_device) * 2 - 1)
    zero = torch.zeros(1024, device=cuda_device)
    assert torch.equal(D.gain(x, SR, zero), x)                      # 0 dB == identity, bit exact
    g6 = D.gain(x, SR, zero + 20.0)
    assert torch.allclose(g6, x * 10.0, rtol=2e-6, atol=0)
    d = D.distortion(x, SR, torch.zeros(2048, device=cuda_device))
    assert torch.allclose(d, torch.tanh(x), rtol=0, atol=2e-7)      # odd symmetry + torch.tanh agreement
    assert torch.equal(D.distortion(-x, SR, torch.zeros(2048, device=cuda_device)), -d)
