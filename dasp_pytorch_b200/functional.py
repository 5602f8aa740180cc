"""B200-native drop-in for ``dasp_pytorch.functional``'s audio-processor hot path.

Same function names, argument order, keyword names, defaults and
``(batch, channels, samples)`` tensor contract as the reference
(``dasp_pytorch/functional.py`` @ c9ae0126), so that
``Processor.process_normalized`` -> ``process_fn(x, sample_rate, **params)``
(reference ``modules.py:45-49``) and direct calls keep working unchanged.  Every
op is a ``torch.autograd.Function`` whose forward and backward call hand-written
sm_100a kernels through the C ABI in ``include/dasp_b200.h``; there is no PyTorch,
Triton or CPU fallback -- non-CUDA inputs raise ``DaspError``.

Arithmetic is fp32 (coefficient design in fp64 inside the kernels).  Inputs in
another floating dtype are computed in fp32 and returned in the input dtype.
"""
from __future__ import annotations

from typing import Optional

import torch

from dasp_pytorch_b200 import _abi
from dasp_pytorch_b200._abi import DaspError, check, ptr, stream_ptr

__all__ = [
    "gain",
    "distortion",
    "stereo_widener",
    "stereo_panner",
    "stereo_bus",
    "parametric_eq",
    "compressor",
    "expander",
    "noise_shaped_reverberation",
]


# --------------------------------------------------------------------------------------
# helpers
# --------------------------------------------------------------------------------------


def _audio(x: torch.Tensor, name: str = "x"):
    """validate the (bs, chs, n) audio tensor -> (fp32 contiguous tensor, original dtype)"""
    if not torch.is_tensor(x) or x.dim() != 3:
        raise ValueError(f"{name} must be a tensor of shape (batch, channels, samples)")
    if not x.is_cuda:
        raise DaspError(
            f"{name} is on {x.device}: dasp_pytorch_b200 only runs on CUDA (B200) tensors and has no CPU path"
        )
    if not x.is_floating_point():
        raise DaspError(f"{name} must be a floating-point tensor, got {x.dtype}")
    return x.to(torch.float32).contiguous(), x.dtype


def _param(p, n_expected: int, like: torch.Tensor, name: str, allow_broadcast: bool = False) -> torch.Tensor:
    """flatten a parameter to fp32 ``(n_expected,)`` on x's device, keeping autograd history.

    The reference reshapes parameters with ``.view(bs, 1, 1)`` and friends, i.e. it accepts
    any shape holding the right number of elements (SURVEY.md 8b); integer tensors are
    promoted (examples/demo.py:44 passes int64 cut-offs).
    """
    if not torch.is_tensor(p):
        p = torch.as_tensor(p)
    if p.device != like.device:
        if p.numel() == 1 and not p.requires_grad:
            p = p.to(like.device)
        else:
            raise DaspError(f"{name} is on {p.device} but x is on {like.device}")
    p = p.reshape(-1).to(torch.float32)
    if p.numel() != n_expected:
        if allow_broadcast and p.numel() == 1:
            p = p.expand(n_expected)
        else:
            raise RuntimeError(
                f"{name}: expected {n_expected} element(s) (one per batch item), got {p.numel()}"
            )
    return p


def _ws(n_floats: int, device) -> torch.Tensor:
    return torch.empty(max(int(n_floats), 1), dtype=torch.float32, device=device)


# bench.py sets this to a list to collect (stage, start_event, end_event) around every C-ABI call
STAGE_TIMING = None


class _timed:
    """CUDA events on the launching stream around one C-ABI call (active only while benchmarking)."""

    def __init__(self, name, device):
        self.name, self.device = name, device

    def __enter__(self):
        if STAGE_TIMING is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.a.record(torch.cuda.current_stream(self.device))
        return self

    def __exit__(self, *exc):
        if STAGE_TIMING is not None:
            self.b.record(torch.cuda.current_stream(self.device))
            STAGE_TIMING.append((self.name, self.a, self.b))
        return False


# --------------------------------------------------------------------------------------
# gain / distortion
# --------------------------------------------------------------------------------------


class _PointwiseFn(torch.autograd.Function):
    """y = f(x * 10^(p_db/20)) with one p_db per row; f = identity (gain) or tanh (distortion)."""

    @staticmethod
    def forward(ctx, x, p_db, kind: str, rows: int, n: int):
        lib = _abi.lib()
        y = torch.empty_like(x)
        with torch.cuda.device(x.device), _timed("dist_fwd", x.device):
            st = stream_ptr(x.device)
            if kind == "gain":
                check(lib.dasp_gain_fwd(ptr(x), ptr(p_db), ptr(y), rows, 1, n, st), "dasp_gain_fwd")
            else:
                check(lib.dasp_distortion_fwd(ptr(x), ptr(p_db), ptr(y), rows, n, st), "dasp_distortion_fwd")
        ctx.save_for_backward(x, p_db)
        ctx.kind, ctx.rows, ctx.n = kind, rows, n
        return y

    @staticmethod
    def backward(ctx, gy):
        lib = _abi.lib()
        x, p_db = ctx.saved_tensors
        rows, n = ctx.rows, ctx.n
        gy = gy.contiguous()
        gx = torch.empty_like(x)
        gp = torch.empty_like(p_db)
        nws = lib.dasp_pointwise_bwd_workspace_floats(rows, n)
        ws = _ws(nws, x.device)
        with torch.cuda.device(x.device), _timed("dist_bwd", x.device):
            st = stream_ptr(x.device)
            if ctx.kind == "gain":
                check(lib.dasp_gain_bwd(ptr(gy), ptr(x), ptr(p_db), ptr(gx), ptr(gp), ptr(ws), nws, rows, 1, n, st),
                      "dasp_gain_bwd")
            else:
                check(lib.dasp_distortion_bwd(ptr(gy), ptr(x), ptr(p_db), ptr(gx), ptr(gp), ptr(ws), nws, rows, n,
                                              st), "dasp_distortion_bwd")
        return gx, gp, None, None, None


def gain(x: torch.Tensor, sample_rate: int, gain_db: torch.Tensor):
    """Apply a per-item gain in dB (reference ``functional.py:10-29``).

    Args:
        x: audio ``(bs, chs, seq_len)``.
        sample_rate: unused (kept for the common processor signature).
        gain_db: ``bs`` elements, any shape.
    """
    xf, dt = _audio(x)
    bs, chs, n = xf.shape
    g = _param(gain_db, bs, xf, "gain_db")
    y = _PointwiseFn.apply(xf, g.contiguous(), "gain", bs, chs * n)
    return y.to(dt)


def distortion(x: torch.Tensor, sample_rate: int, drive_db: torch.Tensor):
    """tanh soft clipper with drive in dB (reference ``functional.py:65-78``).

    Like the reference's ``drive_db.view(bs, chs, -1)``, the drive needs one element per
    (item, channel) row -- i.e. ``bs`` elements for mono input, ``bs*chs`` for multichannel.
    """
    xf, dt = _audio(x)
    bs, chs, n = xf.shape
    d = _param(drive_db, bs * chs, xf, "drive_db")
    y = _PointwiseFn.apply(xf, d.contiguous(), "distortion", bs * chs, n)
    return y.to(dt)


# --------------------------------------------------------------------------------------
# stereo mixing processors
# --------------------------------------------------------------------------------------


class _StereoFn(torch.autograd.Function):
    """kind: 'widener' | 'panner' | 'bus' -- streaming mixes with one scalar parameter per row."""

    @staticmethod
    def forward(ctx, x, p, kind):
        lib = _abi.lib()
        dev = x.device
        with torch.cuda.device(dev):
            st = stream_ptr(dev)
            if kind == "widener":
                bs, _, n = x.shape
                y = torch.empty_like(x)
                check(lib.dasp_widener_fwd(ptr(x), ptr(p), ptr(y), bs, n, st), "dasp_widener_fwd")
            elif kind == "panner":
                bs, tracks, n = x.shape
                y = torch.empty(bs, 2, tracks, n, dtype=torch.float32, device=dev)
                check(lib.dasp_panner_fwd(ptr(x), ptr(p), ptr(y), bs, tracks, n, st), "dasp_panner_fwd")
            else:
                bs, _, tracks, n = x.shape
                y = torch.empty(bs, 2, n, dtype=torch.float32, device=dev)
                check(lib.dasp_bus_fwd(ptr(x), ptr(p), ptr(y), bs, tracks, n, st), "dasp_bus_fwd")
        ctx.save_for_backward(x, p)
        ctx.kind = kind
        return y

    @staticmethod
    def backward(ctx, gy):
        lib = _abi.lib()
        x, p = ctx.saved_tensors
        dev = x.device
        gy = gy.contiguous()
        gx = torch.empty_like(x)
        gp = torch.empty_like(p)
        with torch.cuda.device(dev):
            st = stream_ptr(dev)
            if ctx.kind == "widener":
                bs, _, n = x.shape
                nws = lib.dasp_stereo_bwd_workspace_floats(bs, n)
                ws = _ws(nws, dev)
                check(lib.dasp_widener_bwd(ptr(gy), ptr(x), ptr(p), ptr(gx), ptr(gp), ptr(ws), nws, bs, n, st),
                      "dasp_widener_bwd")
            elif ctx.kind == "panner":
                bs, tracks, n = x.shape
                nws = lib.dasp_stereo_bwd_workspace_floats(bs * tracks, n)
                ws = _ws(nws, dev)
                check(lib.dasp_panner_bwd(ptr(gy), ptr(x), ptr(p), ptr(gx), ptr(gp), ptr(ws), nws, bs, tracks, n, st),
                      "dasp_panner_bwd")
            else:
                bs, _, tracks, n = x.shape
                nws = lib.dasp_stereo_bwd_workspace_floats(bs * 2 * tracks, n)
                ws = _ws(nws, dev)
                check(lib.dasp_bus_bwd(ptr(gy), ptr(x), ptr(p), ptr(gx), ptr(gp), ptr(ws), nws, bs, tracks, n, st),
                      "dasp_bus_bwd")
        return gx, gp, None


def _audio_nd(x, ndim, name="x"):
    if not torch.is_tensor(x) or x.dim() != ndim:
        raise ValueError(f"{name} must be a {ndim}-dimensional tensor")
    if not x.is_cuda:
        raise DaspError(f"{name} is on {x.device}: dasp_pytorch_b200 only runs on CUDA (B200) tensors and has no CPU path")
    if not x.is_floating_point():
        raise DaspError(f"{name} must be a floating-point tensor, got {x.dtype}")
    return x.to(torch.float32).contiguous(), x.dtype


def stereo_widener(x: torch.Tensor, sample_rate: float, width: torch.Tensor):
    """Mid/side stereo widener (reference ``functional.py:580-604``).

    ``x`` is ``(bs, 2, seq_len)``, ``width`` holds ``bs`` elements (0 = mono sum, 0.5 = unchanged,
    1 = side only).  mid = (L+R)/sqrt2 scaled by 2(1-width), side = (L-R)/sqrt2 scaled by 2 width.
    """
    xf, dt = _audio_nd(x, 3)
    bs, chs, _ = xf.shape
    assert chs == 2, "Input tensor must have shape (bs, 2, seq_len)"
    w = _param(width, bs, xf, "width").contiguous()
    return _StereoFn.apply(xf, w, "widener").to(dt)


def stereo_panner(x: torch.Tensor, sample_rate: float, pan: torch.Tensor):
    """Pan mono tracks across the stereo field (reference ``functional.py:607-636``).

    ``x`` is ``(bs, num_tracks, seq_len)``, ``pan`` in ``[0, 1]`` holds ``bs*num_tracks`` elements; returns
    ``(bs, 2, num_tracks, seq_len)`` -- the layout the reference's code produces (its docstring says
    ``(bs, num_tracks, 2, seq_len)``, its ``unsqueeze(1).repeat(1, 2, 1, 1)`` does not).
    """
    xf, dt = _audio_nd(x, 3)
    bs, tracks, _ = xf.shape
    pn = _param(pan, bs * tracks, xf, "pan").contiguous()
    return _StereoFn.apply(xf, pn, "panner").to(dt)


def stereo_bus(x: torch.Tensor, sample_rate: int, send_db: torch.Tensor):
    """Sum stereo tracks to a stereo bus with per-track send levels in dB (reference ``functional.py:32-62``).

    ``x`` is ``(bs, 2, tracks, seq_len)``, ``send_db`` holds ``bs*tracks`` elements; returns ``(bs, 2, seq_len)``.
    """
    xf, dt = _audio_nd(x, 4)
    bs, chs, tracks, _ = xf.shape
    assert chs == 2, "Input tensor must have shape (bs, 2, tracks, seq_len)"
    sd = _param(send_db, bs * tracks, xf, "send_db").contiguous()
    return _StereoFn.apply(xf, sd, "bus").to(dt)


# --------------------------------------------------------------------------------------
# compressor / expander
# --------------------------------------------------------------------------------------


class _DynamicsFn(torch.autograd.Function):
    """Feed-forward dynamics processor: kind 0 = compressor, 1 = expander."""

    @staticmethod
    def forward(ctx, x, threshold, ratio, attack, knee, makeup, kind, sample_rate, eps, lookahead):
        lib = _abi.lib()
        bs, chs, n = x.shape
        y = torch.empty_like(x)
        need_bwd = any(ctx.needs_input_grad[:6])
        ckpt = None
        with torch.cuda.device(x.device):
            if need_bwd:
                tile = lib.dasp_dynamics_tile_len(bs, chs)     # depends on the device's SM count
                if tile <= 0:
                    raise DaspError(f"dynamics: unsupported channel count {chs}")
                ckpt = torch.empty(bs * max(1, -(-n // tile)), dtype=torch.float32, device=x.device)
            with _timed("comp_fwd", x.device):
                check(lib.dasp_dynamics_fwd(kind, ptr(x), ptr(threshold), ptr(ratio), ptr(attack), ptr(knee),
                                            ptr(makeup), ptr(y), ptr(ckpt), bs, chs, n, float(sample_rate),
                                            float(eps), int(lookahead), stream_ptr(x.device)), "dasp_dynamics_fwd")
        if need_bwd:
            ctx.save_for_backward(x, threshold, ratio, attack, knee, makeup, ckpt)
        ctx.cfg = (kind, float(sample_rate), float(eps), int(lookahead))
        return y

    @staticmethod
    def backward(ctx, gy):
        lib = _abi.lib()
        x, threshold, ratio, attack, knee, makeup, ckpt = ctx.saved_tensors
        kind, sample_rate, eps, lookahead = ctx.cfg
        bs, chs, n = x.shape
        gy = gy.contiguous()
        gx = torch.empty_like(x)
        gp = torch.empty(bs, 6, dtype=torch.float32, device=x.device)
        scratch = torch.empty(bs * n, dtype=torch.float32, device=x.device) if lookahead > 0 else None
        with torch.cuda.device(x.device), _timed("comp_bwd", x.device):
            check(lib.dasp_dynamics_bwd(kind, ptr(gy), ptr(x), ptr(threshold), ptr(ratio), ptr(attack), ptr(knee),
                                        ptr(makeup), ptr(ckpt), ptr(gx), ptr(gp), ptr(scratch), bs, chs, n,
                                        sample_rate, eps, lookahead, stream_ptr(x.device)), "dasp_dynamics_bwd")
        return gx, gp[:, 0], gp[:, 1], gp[:, 2], gp[:, 4], gp[:, 5], None, None, None, None


def _dynamics(kind, x, sample_rate, threshold_db, ratio, attack_ms, release_ms, knee_db, makeup_gain_db, eps,
              lookahead_samples):
    xf, dt = _audio(x)
    bs = xf.shape[0]
    ps = [
        _param(p, bs, xf, name, allow_broadcast=True).contiguous()
        for p, name in (
            (threshold_db, "threshold_db"),
            (ratio, "ratio"),
            (attack_ms, "attack_ms"),
            (knee_db, "knee_db"),
            (makeup_gain_db, "makeup_gain_db"),
        )
    ]
    # release_ms is validated for shape only: the reference accepts and ignores it
    # (functional.py:333,343-344), so it receives no gradient here either.
    _param(release_ms, bs, xf, "release_ms", allow_broadcast=True)
    y = _DynamicsFn.apply(xf, *ps, kind, sample_rate, eps, int(lookahead_samples))
    return y.to(dt)


def dynamics_packed(kind: int, x: torch.Tensor, sample_rate: float, params: torch.Tensor, eps: float = 1e-8,
                    lookahead_samples: int = 0):
    """compressor (kind 0) / expander (kind 1) with the six parameters stacked as ``(bs, 6)`` in signature order
    (threshold, ratio, attack, release, knee, makeup).  One transpose instead of six column copies."""
    xf, dt = _audio(x)
    pt = _packed(params, xf.shape[0], 6, xf, "params").t().contiguous()        # (6, bs): rows are contiguous
    y = _DynamicsFn.apply(xf, pt[0], pt[1], pt[2], pt[4], pt[5], kind, sample_rate, eps, int(lookahead_samples))
    return y.to(dt)


def compressor(
    x: torch.Tensor,
    sample_rate: float,
    threshold_db: torch.Tensor,
    ratio: torch.Tensor,
    attack_ms: torch.Tensor,
    release_ms: torch.Tensor,
    knee_db: torch.Tensor,
    makeup_gain_db: torch.Tensor,
    eps: float = 1e-8,
    lookahead_samples: int = 0,
):
    """Feed-forward dynamic range compressor (reference ``functional.py:275-399``).

    Side chain = sum of the channels, soft-knee static curve, one-pole *attack* smoothing of the
    gain-reduction curve (``release_ms`` is accepted and ignored exactly like the reference),
    makeup gain, optional look-ahead delay of the audio path.  The smoother is evaluated as
    the true zero-state recursion; the reference's frequency-sampling evaluation on
    ``n_fft = 2**ceil(log2(2n-1))`` points is identical up to the time-aliased tail of the smoother's
    impulse response, whose size is ``alpha**(n_fft - n)`` of the gain curve with
    ``alpha = exp(-ln 9 / (sample_rate * attack_ms / 1e3))``: < 1e-15 at the BASELINE length
    (n = 48000), 1.7e-2 at n = 8192 and 0.6 at n = 1024 for a 100 ms attack at 44.1 kHz
    (``tests/test_gpu_dynamics.py::test_compressor_gap_to_the_frequency_sampling_reference``
    tracks the gap).
    """
    return _dynamics(0, x, sample_rate, threshold_db, ratio, attack_ms, release_ms, knee_db, makeup_gain_db, eps,
                     lookahead_samples)


def expander(
    x: torch.Tensor,
    sample_rate: float,
    threshold_db: torch.Tensor,
    ratio: torch.Tensor,
    attack_ms: torch.Tensor,
    release_ms: torch.Tensor,
    knee_db: torch.Tensor,
    makeup_gain_db: torch.Tensor,
    eps: float = 1e-8,
    lookahead_samples: int = 0,
):
    """Downward expander with the compressor's signature.

    The reference only stubs this op (``functional.py:402-403`` raises
    ``NotImplementedError``), so there is no reference parity to claim: the static curve is the
    soft-knee downward expander of Giannoulis et al. (2012) -- gain ``(R-1)(x_dB-T)`` below the
    knee, quadratic knee of width ``knee_db``, unity above -- followed by the compressor's
    attack smoother and makeup gain.  Pinned to ``oracle.expander``.
    """
    return _dynamics(1, x, sample_rate, threshold_db, ratio, attack_ms, release_ms, knee_db, makeup_gain_db, eps,
                     lookahead_samples)


# --------------------------------------------------------------------------------------
# parametric EQ
# --------------------------------------------------------------------------------------


class _ParametricEqFn(torch.autograd.Function):
    """x (bs, chs, n), params (bs, 18) -> y; six-section biquad cascade."""

    @staticmethod
    def forward(ctx, x, params, sample_rate):
        lib = _abi.lib()
        bs, chs, n = x.shape
        y = torch.empty_like(x)
        need_bwd = any(ctx.needs_input_grad[:2])
        ckpt = None
        with torch.cuda.device(x.device):
            if need_bwd:
                ckpt = torch.empty(max(1, lib.dasp_eq_ckpt_floats(bs, chs, n)), dtype=torch.float32, device=x.device)
            with _timed("eq_fwd", x.device):
                check(lib.dasp_eq_fwd(ptr(x), ptr(params), ptr(y), ptr(ckpt), bs, chs, n, float(sample_rate),
                                      stream_ptr(x.device)), "dasp_eq_fwd")
        if need_bwd:
            ctx.save_for_backward(x, params, ckpt)
        ctx.sample_rate = float(sample_rate)
        return y

    @staticmethod
    def backward(ctx, gy):
        lib = _abi.lib()
        x, params, ckpt = ctx.saved_tensors
        bs, chs, n = x.shape
        gy = gy.contiguous()
        gx = torch.empty_like(x)
        gp = torch.empty_like(params)
        nws = lib.dasp_eq_bwd_workspace_floats(bs, chs)
        ws = _ws(nws, x.device)
        with torch.cuda.device(x.device), _timed("eq_bwd", x.device):
            check(lib.dasp_eq_bwd(ptr(gy), ptr(x), ptr(params), ptr(ckpt), ptr(gx), ptr(gp), ptr(ws), nws, bs, chs, n,
                                  ctx.sample_rate, stream_ptr(x.device)), "dasp_eq_bwd")
        return gx, gp, None


def parametric_eq(
    x: torch.Tensor,
    sample_rate: float,
    low_shelf_gain_db: torch.Tensor,
    low_shelf_cutoff_freq: torch.Tensor,
    low_shelf_q_factor: torch.Tensor,
    band0_gain_db: torch.Tensor,
    band0_cutoff_freq: torch.Tensor,
    band0_q_factor: torch.Tensor,
    band1_gain_db: torch.Tensor,
    band1_cutoff_freq: torch.Tensor,
    band1_q_factor: torch.Tensor,
    band2_gain_db: torch.Tensor,
    band2_cutoff_freq: torch.Tensor,
    band2_q_factor: torch.Tensor,
    band3_gain_db: torch.Tensor,
    band3_cutoff_freq: torch.Tensor,
    band3_q_factor: torch.Tensor,
    high_shelf_gain_db: torch.Tensor,
    high_shelf_cutoff_freq: torch.Tensor,
    high_shelf_q_factor: torch.Tensor,
):
    """Six-band parametric equaliser: low shelf -> four peaking bands -> high shelf
    (reference ``functional.py:118-272``).

    Each parameter holds ``bs`` elements in any shape, or a single element that is broadcast
    over the batch (reference ``examples/virtual_analog.py:204-206``); integer cut-offs are
    accepted (``examples/demo.py:44``).  All channels of an item share the item's filter.

    The cascade is run as the true zero-state recursion (time-parallel scan, fp32 sigma-form
    sections designed in fp64); the reference evaluates the same filter by frequency sampling
    on ``n_fft = 2**ceil(log2(2n-1))`` points, which coincides with it whenever the impulse
    response fits in the ``n_fft - n`` samples of padding: wrap-around < e^-19 for every filter
    of the ``ParametricEQ`` ranges at n = 48000, but up to 3 % for a 20 Hz shelf at n = 4096
    (item 0 of ``tests/golden/parametric_eq.npz`` keeps such a case; DESIGN.md section 2).
    """
    xf, dt = _audio(x)
    bs = xf.shape[0]
    plist = (
        low_shelf_gain_db, low_shelf_cutoff_freq, low_shelf_q_factor,
        band0_gain_db, band0_cutoff_freq, band0_q_factor,
        band1_gain_db, band1_cutoff_freq, band1_q_factor,
        band2_gain_db, band2_cutoff_freq, band2_q_factor,
        band3_gain_db, band3_cutoff_freq, band3_q_factor,
        high_shelf_gain_db, high_shelf_cutoff_freq, high_shelf_q_factor,
    )
    packed = torch.stack([_param(p, bs, xf, f"parametric_eq parameter {i}", allow_broadcast=True)
                          for i, p in enumerate(plist)], dim=1).contiguous()
    y = _ParametricEqFn.apply(xf, packed, sample_rate)
    return y.to(dt)


def _packed(params, bs: int, ncol: int, like: torch.Tensor, name: str) -> torch.Tensor:
    if not torch.is_tensor(params) or params.dim() != 2 or tuple(params.shape) != (bs, ncol):
        raise ValueError(f"{name}: expected a ({bs}, {ncol}) parameter tensor, got {tuple(getattr(params, 'shape', ()))}")
    if params.device != like.device:
        raise DaspError(f"{name} is on {params.device} but x is on {like.device}")
    return params.to(torch.float32).contiguous()


def parametric_eq_packed(x: torch.Tensor, sample_rate: float, params: torch.Tensor):
    """``parametric_eq`` with its 18 parameters already stacked as ``(bs, 18)`` in signature order (physical
    units).  Used by ``modules.ParametricEQ.process_normalized`` so that the whole normalised-parameter path is
    one affine kernel + the EQ kernels (SURVEY.md 8f rank 1); gradients flow to ``params``."""
    xf, dt = _audio(x)
    return _ParametricEqFn.apply(xf, _packed(params, xf.shape[0], 18, xf, "params"), sample_rate).to(dt)


# --------------------------------------------------------------------------------------
# noise-shaped reverberation
# --------------------------------------------------------------------------------------

# Items per pass of the reverb pipeline (bounds the workspace).  Default: one item per SM of the device, so that the
# one-CTA-per-SM FFT kernels run in whole waves (ifft_shape_kernel: R CTAs per item -> exactly R waves; the persistent
# block-transform kernels: the same number of blocks per CTA).  Measured on B200 (148 SMs), chain step at batch 1024:
# 74 -> 14.83 ms, 128 -> 14.61 ms, 148 -> 14.11 ms.  A positive value overrides the default.
REVERB_CHUNK_ITEMS = 0      # 0 = automatic


def reverb_chunk_items(device) -> int:
    """Items per pass of the reverb pipeline on ``device`` (see REVERB_CHUNK_ITEMS)."""
    if REVERB_CHUNK_ITEMS > 0:
        return REVERB_CHUNK_ITEMS
    return int(torch.cuda.get_device_properties(device).multi_processor_count)


def _noise_or_seed(noise, xf, bs, num_samples, num_bandpass_taps):
    """parity mode: validate the caller's noise tensor; default mode: draw the 64-bit Philox key ON THE DEVICE.

    The reference draws its noise with ``torch.randn`` (``functional.py:547-548``), which is reproducible under
    ``torch.manual_seed`` and, on CUDA, graph-safe (fresh values on every replay of a captured graph).  The key of
    the in-kernel generator is therefore one ``random_()`` word of torch's CUDA generator, left in device memory
    and read by the kernels when they run: no host round trip, same reproducibility, and a captured graph
    re-draws it on every replay (torch registers the generator's Philox offset with the graph)."""
    if noise is not None:
        expect = (bs * 2, 12, num_samples + num_bandpass_taps - 1)
        if tuple(noise.shape) != expect:
            raise ValueError(f"noise must have shape {expect}, got {tuple(noise.shape)}")
        return noise.to(device=xf.device, dtype=torch.float32).contiguous(), None
    return None, torch.empty(1, dtype=torch.int64, device=xf.device).random_()


class _ReverbFn(torch.autograd.Function):
    """x (bs, 1|2, n), params (bs, 25) -> y (bs, 2, n)."""

    @staticmethod
    def forward(ctx, x, params, noise, seed, sample_rate, num_samples, taps, chunk):
        lib = _abi.lib()
        bs, in_chs, n = x.shape
        dev = x.device
        y = torch.empty(bs, 2, n, dtype=torch.float32, device=dev)
        need_bwd = any(ctx.needs_input_grad[:2])
        geom = _abi.ReverbGeom()
        with torch.cuda.device(dev):
            check(lib.dasp_reverb_geometry(bs, n, num_samples, taps, chunk, geom), "dasp_reverb_geometry")
            ws = torch.empty(max(geom.fwd_workspace_bytes, 16), dtype=torch.uint8, device=dev)
            wet = fsave = xspec = irspec = None
            if need_bwd:
                wet = torch.empty(geom.wet_floats, dtype=torch.float32, device=dev)
                fsave = torch.empty(geom.f_floats, dtype=torch.float32, device=dev)
                xspec = torch.empty(geom.xspec_c64, dtype=torch.complex64, device=dev)
                irspec = torch.empty(geom.irspec_c64, dtype=torch.complex64, device=dev)
            with _timed("reverb_fwd", dev):
                check(lib.dasp_reverb_fwd(ptr(x), in_chs, ptr(params), ptr(noise), ptr(seed), ptr(y), ptr(wet),
                                          ptr(fsave), ptr(xspec), ptr(irspec), ptr(ws), ws.numel(), bs, n, num_samples,
                                          taps, chunk, float(sample_rate), stream_ptr(dev)), "dasp_reverb_fwd")
        if need_bwd:
            ctx.save_for_backward(x, params, wet, fsave, xspec, irspec)
        ctx.cfg = (num_samples, taps, chunk, geom.bwd_workspace_bytes, 1 if noise is None else 0)
        return y

    @staticmethod
    def backward(ctx, gy):
        lib = _abi.lib()
        x, params, wet, fsave, xspec, irspec = ctx.saved_tensors
        num_samples, taps, chunk, bwd_bytes, device_noise = ctx.cfg
        bs, in_chs, n = x.shape
        dev = x.device
        gy = gy.contiguous()
        gx = torch.empty_like(x)
        gp = torch.empty_like(params)
        ws = torch.empty(max(bwd_bytes, 16), dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev), _timed("reverb_bwd", dev):
            check(lib.dasp_reverb_bwd(ptr(gy), ptr(x), in_chs, ptr(params), ptr(wet), ptr(fsave), ptr(xspec),
                                      ptr(irspec), ptr(gx), ptr(gp), ptr(ws), ws.numel(), bs, n, num_samples, taps,
                                      chunk, device_noise, stream_ptr(dev)), "dasp_reverb_bwd")
        return gx, gp, None, None, None, None, None, None


def noise_shaped_reverberation(
    x: torch.Tensor,
    sample_rate: float,
    band0_gain: torch.Tensor,
    band1_gain: torch.Tensor,
    band2_gain: torch.Tensor,
    band3_gain: torch.Tensor,
    band4_gain: torch.Tensor,
    band5_gain: torch.Tensor,
    band6_gain: torch.Tensor,
    band7_gain: torch.Tensor,
    band8_gain: torch.Tensor,
    band9_gain: torch.Tensor,
    band10_gain: torch.Tensor,
    band11_gain: torch.Tensor,
    band0_decay: torch.Tensor,
    band1_decay: torch.Tensor,
    band2_decay: torch.Tensor,
    band3_decay: torch.Tensor,
    band4_decay: torch.Tensor,
    band5_decay: torch.Tensor,
    band6_decay: torch.Tensor,
    band7_decay: torch.Tensor,
    band8_decay: torch.Tensor,
    band9_decay: torch.Tensor,
    band10_decay: torch.Tensor,
    band11_decay: torch.Tensor,
    mix: torch.Tensor,
    num_samples: int = 65536,
    num_bandpass_taps: int = 1023,
    *,
    noise: Optional[torch.Tensor] = None,
):
    """Filtered-noise artificial reverberation (reference ``functional.py:406-577``).

    Twelve bands (12 Hz low-pass, ten octave band-passes, 18 kHz high-pass; ``signal.py:42-92``),
    each a white-noise signal filtered by a ``num_bandpass_taps`` FIR, shaped by
    ``exp(-(10*decay+1)*t)`` and its gain, averaged into a ``num_samples``-long stereo impulse
    response that is convolved with the input; ``mix`` blends wet and dry.  Mono input is
    duplicated and the output is always stereo, like the reference.

    Keyword-only extension ``noise``: the reference draws
    ``torch.randn(bs*2, 12, num_samples + num_bandpass_taps - 1)`` inside the call
    (``functional.py:547-548``).  Pass that tensor here to reproduce a seeded reference call
    exactly (parity tests); by default fresh N(0,1) noise is generated on the device with
    Philox4x32-10, keyed by one 64-bit word drawn from torch's CUDA generator and kept in device
    memory (``torch.manual_seed`` makes the call reproducible; a captured CUDA graph draws fresh
    noise on every replay, like the reference's ``torch.randn`` would).
    """
    assert num_bandpass_taps % 2 == 1, "num_bandpass_taps must be odd"
    xf, dt = _audio(x)
    bs, chs, n = xf.shape
    assert chs <= 2, "only mono/stereo signals are supported"
    plist = (
        band0_gain, band1_gain, band2_gain, band3_gain, band4_gain, band5_gain,
        band6_gain, band7_gain, band8_gain, band9_gain, band10_gain, band11_gain,
        band0_decay, band1_decay, band2_decay, band3_decay, band4_decay, band5_decay,
        band6_decay, band7_decay, band8_decay, band9_decay, band10_decay, band11_decay,
        mix,
    )
    packed = torch.stack([_param(p, bs, xf, f"noise_shaped_reverberation parameter {i}", allow_broadcast=True)
                          for i, p in enumerate(plist)], dim=1).contiguous()
    noise, seed = _noise_or_seed(noise, xf, bs, num_samples, num_bandpass_taps)
    y = _ReverbFn.apply(xf, packed, noise, seed, sample_rate, int(num_samples), int(num_bandpass_taps),
                        reverb_chunk_items(xf.device))
    return y.to(dt)


def noise_shaped_reverberation_packed(x: torch.Tensor, sample_rate: float, params: torch.Tensor, num_samples: int = 65536,
                                      num_bandpass_taps: int = 1023, *, noise: Optional[torch.Tensor] = None):
    """``noise_shaped_reverberation`` with its 25 parameters stacked as ``(bs, 25)`` (12 gains, 12 decays, mix)."""
    assert num_bandpass_taps % 2 == 1, "num_bandpass_taps must be odd"
    xf, dt = _audio(x)
    bs, chs, _ = xf.shape
    assert chs <= 2, "only mono/stereo signals are supported"
    packed = _packed(params, bs, 25, xf, "params")
    noise, seed = _noise_or_seed(noise, xf, bs, num_samples, num_bandpass_taps)
    y = _ReverbFn.apply(xf, packed, noise, seed, sample_rate, int(num_samples), int(num_bandpass_taps),
                        reverb_chunk_items(xf.device))
    return y.to(dt)
