"""Generate tests/golden/*.npz by running the UNMODIFIED reference on CPU.

Run in the authoring container only (needs /root/reference, which does not exist on
the GPU box):

    python oracle/make_golden.py

Each fixture stores seeded inputs, the reference outputs in fp32 and fp64, and the
reference's autograd gradients (loss = mean(y^2)) in fp64.  The oracle
(oracle/dasp_oracle.py) is pinned against these in tests/test_oracle_golden.py; the CUDA
path is checked against them in the ``-m gpu`` tests.  Sizes are kept small so the
fixtures stay a few MB in total and every file under 1 MB: where the full-length outputs
would not fit, the per-sample arrays (outputs and dL/dx) keep every ``t_stride``-th time
index while the inputs and the parameter gradients are stored whole.
"""

from __future__ import annotations

import os
import sys

import numpy as np
import torch

REF = os.environ.get("DASP_REFERENCE", "/root/reference")
sys.path.insert(0, REF)
import dasp_pytorch  # noqa: E402  (the reference)
import dasp_pytorch.functional as RF  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden")
# Time stride of the per-sample arrays in pointwise/parametric_eq/compressor.npz.  Odd, so the
# sample still reaches every lane of the kernels' power-of-two vector widths.
T_STRIDE = 3


def denorm(proc, p01):
    d = proc.denormalize_param_dict(proc.extract_param_dict(p01))
    return d


def run_with_grads(fn, x, params: dict, dtype, extra=None):
    """returns y, dx, {name: dparam} for loss = mean(y^2)."""
    extra = extra or {}
    xx = x.to(dtype).clone().requires_grad_(True)
    pp = {k: v.to(dtype).clone().requires_grad_(True) for k, v in params.items()}
    y = fn(xx, **pp, **extra)
    loss = y.pow(2).mean()
    loss.backward()
    grads = {k: (v.grad if v.grad is not None else None) for k, v in pp.items()}
    return y.detach(), xx.grad.detach(), grads


def pack(prefix, y32, y64, dx64, grads64, store, stride=1):
    store[f"{prefix}_y32"] = y32[..., ::stride].numpy()
    store[f"{prefix}_y64"] = y64[..., ::stride].numpy()
    store[f"{prefix}_dx64"] = dx64[..., ::stride].numpy()
    for k, g in grads64.items():
        if g is not None:
            store[f"{prefix}_d_{k}"] = g.numpy()


def main():
    os.makedirs(OUT, exist_ok=True)
    sr = 44100

    # ---------------- gain / distortion ----------------
    g = torch.Generator().manual_seed(11)
    st = {"t_stride": np.array(T_STRIDE)}
    x = torch.rand(3, 2, 1024, generator=g) * 2 - 1
    gd = torch.rand(3, generator=g) * 48 - 24
    st["gain_x"], st["gain_db"] = x.numpy(), gd.numpy()
    f = lambda xx, gain_db: RF.gain(xx, sr, gain_db)
    y32, _, _ = run_with_grads(f, x, {"gain_db": gd}, torch.float32)
    y64, dx, gr = run_with_grads(f, x, {"gain_db": gd}, torch.float64)
    pack("gain", y32, y64, dx, gr, st, T_STRIDE)

    x = torch.rand(4, 1, 16000, generator=g) * 2 - 1          # BASELINE config 1 shape
    dd = torch.rand(4, generator=g) * 24
    st["dist_x"], st["dist_db"] = x.numpy(), dd.numpy()
    f = lambda xx, drive_db: RF.distortion(xx, 16000, drive_db)
    y32, _, _ = run_with_grads(f, x, {"drive_db": dd}, torch.float32)
    y64, dx, gr = run_with_grads(f, x, {"drive_db": dd}, torch.float64)
    pack("dist", y32, y64, dx, gr, st, T_STRIDE)

    x = torch.rand(2, 2, 512, generator=g) * 2 - 1            # stereo: one drive per row
    dd = torch.rand(4, generator=g) * 24
    st["dist2_x"], st["dist2_db"] = x.numpy(), dd.numpy()
    f = lambda xx, drive_db: RF.distortion(xx, sr, drive_db)
    y32, _, _ = run_with_grads(f, x, {"drive_db": dd}, torch.float32)
    y64, dx, gr = run_with_grads(f, x, {"drive_db": dd}, torch.float64)
    pack("dist2", y32, y64, dx, gr, st, T_STRIDE)
    np.savez_compressed(os.path.join(OUT, "pointwise.npz"), **st)

    # ---------------- parametric EQ ----------------
    g = torch.Generator().manual_seed(22)
    st = {"t_stride": np.array(T_STRIDE)}
    bs, chs, n = 6, 2, 4096
    x = torch.rand(bs, chs, n, generator=g) * 2 - 1
    p01 = torch.rand(bs, 18, generator=g)
    p01[0, 1] = 0.0      # low-shelf cutoff at 20 Hz: the ill-conditioned corner (SURVEY fact 3)
    p01[1, 1] = 0.01
    proc = dasp_pytorch.ParametricEQ(sr)
    params = denorm(proc, p01)
    st["x"], st["p01"] = x.numpy(), p01.numpy()
    st["names"] = np.array(list(params.keys()))
    f = lambda xx, **kw: RF.parametric_eq(xx, sr, **kw)
    y32, _, _ = run_with_grads(f, x, params, torch.float32)
    y64, dx, gr = run_with_grads(f, x, params, torch.float64)
    pack("eq", y32, y64, dx, gr, st, T_STRIDE)
    np.savez_compressed(os.path.join(OUT, "parametric_eq.npz"), **st)

    # ---------------- compressor ----------------
    g = torch.Generator().manual_seed(33)
    st = {"t_stride": np.array(T_STRIDE)}
    bs, chs, n = 6, 2, 4096
    level = torch.rand(bs, 1, 1, generator=g)
    x = (torch.rand(bs, chs, n, generator=g) * 2 - 1) * level
    p01 = torch.rand(bs, 6, generator=g)
    p01[:, 4] = p01[:, 4].clamp(min=0.05)     # knee_db > 0 (W == 0 gives NaN grads upstream)
    # attack <= 12.6 ms for items 1..5 so the smoother's impulse response has died out inside
    # n_fft - N = 4096 samples (frequency sampling == recursion); item 0 keeps a long attack
    # on purpose: it pins the oracle's reproduction of the reference's time aliasing.
    p01[1:, 2] *= 0.08
    p01[0, 2] = 0.9
    proc = dasp_pytorch.Compressor(sr)
    params = denorm(proc, p01)
    st["x"], st["p01"] = x.numpy(), p01.numpy()
    st["names"] = np.array(list(params.keys()))
    f = lambda xx, **kw: RF.compressor(xx, sr, **kw)
    y32, _, _ = run_with_grads(f, x, params, torch.float32)
    y64, dx, gr = run_with_grads(f, x, params, torch.float64)
    pack("comp", y32, y64, dx, gr, st, T_STRIDE)
    y64la, _, _ = run_with_grads(f, x, params, torch.float64, extra={"lookahead_samples": 7})
    st["comp_la7_y64"] = y64la[..., ::T_STRIDE].numpy()
    np.savez_compressed(os.path.join(OUT, "compressor.npz"), **st)

    # ---------------- reverb ----------------
    st = {}
    g = torch.Generator().manual_seed(44)
    bs, n, L, taps = 2, 2048, 3000, 255
    proc = dasp_pytorch.NoiseShapedReverb(sr)
    for tag, chs, seed in (("st", 2, 7), ("mono", 1, 8)):
        x = torch.rand(bs, chs, n, generator=g) * 2 - 1
        p01 = torch.rand(bs, 25, generator=g)
        params = denorm(proc, p01)
        st[f"{tag}_x"], st[f"{tag}_p01"] = x.numpy(), p01.numpy()
        st[f"{tag}_seed"] = np.array(seed)

        def f(xx, **kw):
            torch.manual_seed(seed)      # the reference draws its noise right after this
            return RF.noise_shaped_reverberation(xx, sr, **kw, num_samples=L,
                                                 num_bandpass_taps=taps)

        y32, _, _ = run_with_grads(f, x, params, torch.float32)
        y64, dx, gr = run_with_grads(f, x, params, torch.float64)
        pack(f"{tag}", y32, y64, dx, gr, st)
    st["names"] = np.array(list(params.keys()))
    st["L"], st["taps"] = np.array(L), np.array(taps)
    torch.manual_seed(7)
    st["noise_seed7_head"] = torch.randn(bs * 2, 12, L + taps - 1)[0, 0, :16].numpy()
    fb = dasp_pytorch.signal.octave_band_filterbank(taps, sr)
    st["filterbank"] = fb.squeeze(1).numpy()
    np.savez_compressed(os.path.join(OUT, "reverb.npz"), **st)

    # ---------------- stereo widener / panner / bus ----------------
    g = torch.Generator().manual_seed(55)
    st = {}
    x = torch.rand(3, 2, 700, generator=g) * 2 - 1
    w = torch.rand(3, 1, generator=g)
    st["wid_x"], st["wid_w"] = x.numpy(), w.numpy()
    f = lambda xx, width: RF.stereo_widener(xx.clone(), sr, width)
    y32, _, _ = run_with_grads(f, x, {"width": w}, torch.float32)
    y64, dx, gr = run_with_grads(f, x, {"width": w}, torch.float64)
    pack("wid", y32, y64, dx, gr, st)
    x = torch.rand(3, 4, 500, generator=g) * 2 - 1
    pn = torch.rand(3, 4, generator=g) * 0.9 + 0.05
    st["pan_x"], st["pan_p"] = x.numpy(), pn.numpy()
    f = lambda xx, pan: RF.stereo_panner(xx, sr, pan)
    y32, _, _ = run_with_grads(f, x, {"pan": pn}, torch.float32)
    y64, dx, gr = run_with_grads(f, x, {"pan": pn}, torch.float64)
    pack("pan", y32, y64, dx, gr, st)
    x = torch.rand(3, 2, 5, 400, generator=g) * 2 - 1
    sd = torch.rand(3, 5, 1, generator=g) * 24 - 18
    st["bus_x"], st["bus_s"] = x.numpy(), sd.numpy()
    f = lambda xx, send_db: RF.stereo_bus(xx, sr, send_db)
    y32, _, _ = run_with_grads(f, x, {"send_db": sd}, torch.float32)
    y64, dx, gr = run_with_grads(f, x, {"send_db": sd}, torch.float64)
    pack("bus", y32, y64, dx, gr, st)
    np.savez_compressed(os.path.join(OUT, "stereo.npz"), **st)

    for fn in sorted(os.listdir(OUT)):
        print(fn, os.path.getsize(os.path.join(OUT, fn)) // 1024, "KiB")


if __name__ == "__main__":
    main()
