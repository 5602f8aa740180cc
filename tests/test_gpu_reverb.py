"""noise_shaped_reverberation on the GPU through the C ABI vs the CPU oracle and the reference golden.
Tolerance: 1e-4 relative fp32 (north star), per item, against the fp64 arbiter fed the SAME noise tensor."""
import numpy as np
import pytest
import torch

import oracle
from conftest import load_golden
from helpers import SR, param_grad_err, peak_err, run_with_grads

pytestmark = pytest.mark.gpu
TOL = 1e-4


def _params01(bs, seed):
    g = torch.Generator().manual_seed(seed)
    p = torch.rand(bs, 25, generator=g)
    return [p[:, i].clone() for i in range(25)]


def _check(cuda_device, x, params, L, taps, seed, sr=SR):
    import dasp_pytorch_b200 as D
    bs = x.shape[0]
    noise = oracle.reverb_noise(bs, L, taps, seed)
    nz = noise.to(cuda_device)
    y, dx, dp = run_with_grads(
        lambda xx, p: D.noise_shaped_reverberation(xx, sr, *p, num_samples=L, num_bandpass_taps=taps, noise=nz),
        x, params, torch.float32, cuda_device)
    y64, dx64, dp64 = run_with_grads(
        lambda xx, p: oracle.noise_shaped_reverberation(xx, sr, *p, num_samples=L, num_bandpass_taps=taps, noise=noise),
        x, params, torch.float64, "cpu")
    assert y.shape == y64.shape
    assert peak_err(y, y64).max() < TOL, peak_err(y, y64)
    assert peak_err(dx, dx64).max() < TOL, peak_err(dx, dx64)
    assert param_grad_err(dp, dp64).max() < TOL, param_grad_err(dp, dp64)


@pytest.mark.parametrize("tag", ["st", "mono"])
def test_reverb_golden(cuda_device, tag):
    import dasp_pytorch_b200 as D
    g = load_golden("reverb.npz")
    L, taps, seed = int(g["L"]), int(g["taps"]), int(g[f"{tag}_seed"])
    names = [str(s) for s in g["names"]]
    x = g[f"{tag}_x"]
    noise = oracle.reverb_noise(x.shape[0], L, taps, seed).to(cuda_device)
    params = [torch.as_tensor(g[f"{tag}_p01"])[:, i] for i in range(25)]
    y, dx, dp = run_with_grads(
        lambda xx, p: D.noise_shaped_reverberation(xx, SR, *p, num_samples=L, num_bandpass_taps=taps, noise=noise),
        x, params, torch.float32, cuda_device)
    assert y.shape == (x.shape[0], 2, x.shape[2])                      # mono in -> stereo out
    assert peak_err(y, g[f"{tag}_y64"]).max() < TOL
    assert peak_err(y, g[f"{tag}_y32"]).max() < TOL
    assert peak_err(dx, g[f"{tag}_dx64"]).max() < TOL
    ref = [torch.as_tensor(g[f"{tag}_d_{n}"]) for n in names]
    assert param_grad_err(dp, ref).max() < TOL


@pytest.mark.parametrize("bs,chs,n,L,taps", [(3, 2, 20000, 30000, 1023), (5, 1, 6000, 9000, 255), (6, 2, 3001, 5000, 31),
                                             (1, 2, 100, 16, 3), (9, 2, 4096, 8192, 1023)])
def test_reverb_vs_oracle(cuda_device, bs, chs, n, L, taps):
    """chunk remainders (bs % 4 != 0), mono, ragged lengths, tiny IR, several block counts"""
    g = torch.Generator().manual_seed(bs * 7 + chs)
    x = torch.rand(bs, chs, n, generator=g) * 2 - 1
    _check(cuda_device, x, _params01(bs, 100 + bs), L, taps, seed=bs)


def test_reverb_config4_shape(cuda_device):
    """BASELINE config-4 geometry (N=48000, IR=96000, 1023 taps) on a few items, same noise as the oracle"""
    g = torch.Generator().manual_seed(4)
    x = torch.rand(4, 2, 48000, generator=g) * 2 - 1
    _check(cuda_device, x, _params01(4, 44), 96000, 1023, seed=40)


def test_reverb_device_noise_properties(cuda_device):
    """default path (Philox noise on the device): mix=0 is the identity, seeding is reproducible, and the
    synthesised IR has the statistics of the reference construction (checked via its energy)."""
    import dasp_pytorch_b200 as D
    bs, n, L, taps = 8, 16000, 24000, 1023
    x = torch.zeros(bs, 2, n, device=cuda_device)
    x[:, :, 0] = 1.0                                        # impulse -> the wet path outputs the IR itself
    p = [q.to(cuda_device) for q in _params01(bs, 5)]
    p[24] = torch.zeros(bs, device=cuda_device)
    xr = torch.rand(bs, 2, n, device=cuda_device)
    assert torch.equal(D.noise_shaped_reverberation(xr, SR, *p, num_samples=L, num_bandpass_taps=taps), xr)
    p[24] = torch.ones(bs, device=cuda_device)
    torch.manual_seed(123)
    a = D.noise_shaped_reverberation(x, SR, *p, num_samples=L, num_bandpass_taps=taps)
    torch.manual_seed(123)
    b = D.noise_shaped_reverberation(x, SR, *p, num_samples=L, num_bandpass_taps=taps)
    c = D.noise_shaped_reverberation(x, SR, *p, num_samples=L, num_bandpass_taps=taps)
    assert torch.equal(a, b) and not torch.equal(a, c)
    # energy of the IR vs the oracle's with independent reference-style noise: same distribution => ratio ~ 1
    ir = a.cpu().double()
    noise = oracle.reverb_noise(bs, L, taps, 9)
    ref = oracle.noise_shaped_reverberation(x.cpu().double(), SR, *[q.cpu().double() for q in p], num_samples=L,
                                            num_bandpass_taps=taps, noise=noise)
    e_new = ir.pow(2).sum(dim=(1, 2))
    e_ref = ref.pow(2).sum(dim=(1, 2))
    ratio = (e_new / e_ref)
    assert ((ratio > 0.6) & (ratio < 1.6)).all(), ratio
    assert abs(float(ratio.log().mean())) < 0.2
    # left/right IRs are independent draws, not copies
    assert (ir[:, 0] - ir[:, 1]).abs().max() > 1e-4


def test_reverb_device_noise_band_statistics(cuda_device):
    """spectral synthesis (device noise) must produce an IR with the same second-order statistics as the
    reference construction: compare octave-band energies of the IR, averaged over 24 items x 2 channels,
    with the oracle fed reference-style time-domain noise."""
    import dasp_pytorch_b200 as D
    bs, n, L, taps = 24, 48000, 96000, 1023            # BASELINE geometry: leff = 48000, polyphase factor 6
    x = torch.zeros(bs, 2, n, device=cuda_device)
    x[:, :, 0] = 1.0
    ones = torch.ones(bs, device=cuda_device)
    p = [ones * 1.0] * 12 + [ones * 0.3] * 12 + [ones]
    torch.manual_seed(7)
    ir = D.noise_shaped_reverberation(x, SR, *p, num_samples=L, num_bandpass_taps=taps).cpu().double()
    nref = 6
    noise = oracle.reverb_noise(nref, L, taps, 11)
    ref = oracle.noise_shaped_reverberation(x[:nref].cpu().double(), SR, *[q[:nref].cpu().double() for q in p],
                                            num_samples=L, num_bandpass_taps=taps, noise=noise)
    edges = [0, 22, 45, 90, 180, 355, 710, 1400, 2800, 5600, 11200, 17000, 22050]
    freqs = torch.fft.rfftfreq(n, 1 / SR)

    def band_energy(sig):
        pw = torch.fft.rfft(sig, dim=-1).abs().pow(2).mean(dim=(0, 1))
        return torch.stack([pw[(freqs >= lo) & (freqs < hi)].sum() for lo, hi in zip(edges[:-1], edges[1:])])

    e_new, e_ref = band_energy(ir), band_energy(ref)
    ratio = e_new / e_ref
    assert ((ratio > 0.55) & (ratio < 1.8)).all(), ratio        # few independent draws in the lowest bands
    assert abs(float(ratio[4:].log().mean())) < 0.12, ratio     # well-averaged bands agree within ~10 %
    # envelope: energy of the last quarter relative to the first quarter follows exp(-2 (10*0.3+1) t)
    q = n // 4
    dec_new = ir[..., -q:].pow(2).sum() / ir[..., :q].pow(2).sum()
    dec_ref = ref[..., -q:].pow(2).sum() / ref[..., :q].pow(2).sum()
    assert 0.7 < float(dec_new / dec_ref) < 1.4


def test_reverb_long_audio_and_long_filters(cuda_device):
    """examples/demo.py-like length (N >> IR): 49 audio blocks x 16 IR partitions takes the generic
    (non register-cached) multiply path and a polyphase factor of 9; plus a 4095-tap filter bank (32768-pt blocks)."""
    import dasp_pytorch_b200 as D
    g = torch.Generator().manual_seed(12)
    x = torch.rand(1, 2, 200000, generator=g) * 2 - 1
    _check(cuda_device, x, _params01(1, 77), 65536, 1023, seed=5)
    x2 = torch.rand(2, 1, 30000, generator=g) * 2 - 1
    _check(cuda_device, x2, _params01(2, 78), 20000, 4095, seed=6)
    # device-noise path on the same geometries: finite, stereo, right shape
    xs = x.to(cuda_device)
    p = [q.to(cuda_device) for q in _params01(1, 77)]
    y = D.noise_shaped_reverberation(xs, SR, *p)                       # reference defaults: 65536 samples, 1023 taps
    assert y.shape == (1, 2, 200000) and bool(torch.isfinite(y).all())


def test_reverb_contract(cuda_device):
    import dasp_pytorch_b200 as D
    x = torch.rand(2, 2, 512, device=cuda_device)
    p = [q.to(cuda_device) for q in _params01(2, 3)]
    with pytest.raises(AssertionError):
        D.noise_shaped_reverberation(x, SR, *p, num_samples=256, num_bandpass_taps=30)       # even taps
    with pytest.raises(AssertionError):
        D.noise_shaped_reverberation(torch.rand(2, 3, 512, device=cuda_device), SR, *p, num_samples=256,
                                     num_bandpass_taps=31)                                   # > 2 channels
    with pytest.raises(D.functional.DaspError):
        D.noise_shaped_reverberation(x, 16000, *p, num_samples=256, num_bandpass_taps=31)    # 18 kHz > sr/2
    y = D.noise_shaped_reverberation(x, SR, *[q.view(2, 1) for q in p], num_samples=256, num_bandpass_taps=31)
    assert y.shape == (2, 2, 512)
    names = [f"band{i}_gain" for i in range(12)] + [f"band{i}_decay" for i in range(12)] + ["mix"]
    torch.manual_seed(1)
    y1 = D.noise_shaped_reverberation(x, SR, **dict(zip(names, p)), num_samples=256, num_bandpass_taps=31)
    torch.manual_seed(1)
    y2 = D.noise_shaped_reverberation(x, SR, *p, num_samples=256, num_bandpass_taps=31)
    assert torch.equal(y1, y2)


def test_reverb_chunking_is_invisible(cuda_device, monkeypatch):
    """The pipeline processes the batch in chunks (default: one item per SM); the Philox stream is keyed by the
    absolute item index, so any chunk size -- including one that leaves a remainder chunk -- gives the same result."""
    import dasp_pytorch_b200 as D
    from dasp_pytorch_b200 import functional as F
    bs, n, L, taps = 5, 8000, 12000, 255
    g = torch.Generator().manual_seed(3)
    x = (torch.rand(bs, 2, n, generator=g) * 2 - 1).to(cuda_device)
    p = [q.to(cuda_device) for q in _params01(bs, 8)]

    def run(chunk):
        monkeypatch.setattr(F, "REVERB_CHUNK_ITEMS", chunk)
        torch.manual_seed(5)
        xx = x.clone().requires_grad_(True)
        pp = [q.clone().requires_grad_(True) for q in p]
        y = D.noise_shaped_reverberation(xx, SR, *pp, num_samples=L, num_bandpass_taps=taps)
        y.square().sum().backward()
        return y.detach(), xx.grad, torch.stack([q.grad for q in pp], 1)

    ref = run(0)                                    # automatic: the whole batch in one chunk
    for chunk in (1, 2, 3):
        got = run(chunk)
        for a, b in zip(got, ref):              # (cuFFT may pick another kernel for another batch size: rounding only)
            assert float((a - b).abs().max() / b.abs().max()) < 2e-6, chunk


@pytest.mark.parametrize("n,L,taps,want_r", [(6000, 4000, 255, 1), (12000, 30000, 1023, 2), (20000, 20000, 1023, 3),
                                             (30000, 40000, 1023, 4), (36000, 36000, 1023, 5), (48000, 48000, 1023, 6),
                                             (48000, 96000, 1023, 6), (50000, 50000, 1023, 7), (60000, 60000, 1023, 8),
                                             (70000, 66000, 1023, 9), (20000, 20000, 2047, 2), (6001, 9000, 255, 1)])
def test_reverb_device_noise_path_pinned_to_oracle(cuda_device, n, L, taps, want_r):
    """DETERMINISTIC parity of the device-noise path against the fp64 oracle, for polyphase factors R = 1 ... 9:
    spectral_gen_kernel -> ifft_shape_kernel (8192-point blocks) or -> batched cuFFT -> shape_ir_pp_kernel (2047 taps:
    16384-point blocks), then the partitioned convolution (own FFT, or cuFFT for the unaligned n = 6001), and the
    backward incl. ir_grad_pp_kernel.

    The generator draws, per (item, band, channel), a white PERIODIC sequence w of length n1 = R*nb in the frequency
    domain and filters it circularly: f[t] = sum_m h[m] w[(t-m) mod n1].  With the test hook
    dasp_debug_reverb_flat_filterbank the filters are unit impulses, so the f buffer kept for the backward is w itself.
    The reference-style noise tensor  noise[t'] = w[(t' - P) mod n1]  (P = taps-1, h symmetric) then makes the
    reference's valid cross-correlation (functional.py:551-556) produce exactly the same f for every t < min(L, n)
    (n1 >= min(L, n) + P: no wrap-around inside the window), so y, dL/dx and all 25 parameter gradients of the default
    call must equal oracle.noise_shaped_reverberation(noise=...) to 1e-4 -- a wrong Hermitian pairing, twiddle,
    s_half/s_full scaling or polyphase index anywhere in these kernels fails this test."""
    import dasp_pytorch_b200 as D
    from dasp_pytorch_b200 import _abi
    lib = _abi.lib()
    bs, P = 2, taps - 1
    geom = _abi.ReverbGeom()
    assert lib.dasp_reverb_geometry(0, n, L, taps, 0, geom) == 0
    nb, R = geom.nb, geom.rpp
    assert R == want_r
    want_path = 0 if taps == 2047 else 2        # 2047 taps need 16384-point blocks: the cuFFT polyphase synthesis
    assert nb == (16384 if want_path == 0 else 8192)
    n1 = R * nb
    g = torch.Generator().manual_seed(n + L)
    x = (torch.rand(bs, 2, n, generator=g) * 2 - 1)
    params = _params01(bs, 5 + want_r)
    kw = dict(num_samples=L, num_bandpass_taps=taps)

    # 1) the white sequences: same seed, unit-impulse filter bank, read f_save from the autograd node
    lib.dasp_debug_reverb_flat_filterbank(1)
    try:
        torch.manual_seed(1234)
        xq = x.to(cuda_device).requires_grad_(True)
        yq = D.noise_shaped_reverberation(xq, SR, *[p.to(cuda_device) for p in params], **kw)
        fsave = yq.grad_fn.saved_tensors[3]
    finally:
        lib.dasp_debug_reverb_flat_filterbank(0)
    assert lib.dasp_debug_reverb_last_path() == want_path
    w = torch.view_as_complex(fsave[: bs * 12 * R * nb * 2].reshape(bs, 12, R, nb, 2).contiguous())   # [.., b, a] = w[R a + b]
    w = w.permute(0, 1, 3, 2).reshape(bs, 12, n1).cpu()               # (item, band, t), real = left, imag = right
    assert abs(float(w.real.std()) - 1.0) < 0.02 and abs(float(w.imag.std()) - 1.0) < 0.02      # white, unit variance
    idx = (torch.arange(L + P) - P) % n1
    noise = torch.stack([w.real[:, :, idx], w.imag[:, :, idx]], 1).reshape(bs * 2, 12, L + P).double()

    # 2) the default call with the same seed vs the oracle fed that noise
    def run_default(xx, p):
        torch.manual_seed(1234)
        return D.noise_shaped_reverberation(xx, SR, *p, **kw)

    y, dx, dp = run_with_grads(run_default, x, params, torch.float32, cuda_device)
    assert lib.dasp_debug_reverb_last_path() == want_path
    y64, dx64, dp64 = run_with_grads(
        lambda xx, p: oracle.noise_shaped_reverberation(xx, SR, *p, noise=noise, method="fft", **kw),
        x, params, torch.float64, "cpu")
    assert peak_err(y, y64).max() < TOL, peak_err(y, y64)
    assert peak_err(dx, dx64).max() < TOL, peak_err(dx, dx64)
    assert param_grad_err(dp, dp64).max() < TOL, param_grad_err(dp, dp64)

    # 3) a forward that keeps nothing for a backward computes the same bits
    with torch.no_grad():
        y_inf = run_default(x.to(cuda_device), [p.to(cuda_device) for p in params])
    assert torch.equal(y_inf.cpu(), y)
