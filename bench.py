#!/usr/bin/env python
"""Contract benchmark: audio samples/sec (fwd+bwd) of the dasp hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   # this repo's CUDA path
    python bench.py --impl reference [--gpus N] [--steps K] [--warmup W]   # the reference's own CPU path
    python bench.py --impl reference-cuda                                  # the reference's own PyTorch-CUDA path (1 GPU)

Workload (BASELINE.json configs[4], the config the headline metric is quoted on): the chain
parametric_eq -> compressor -> noise_shaped_reverberation (12 bands, 1023 taps, IR 96000) -> distortion
on a GLOBAL batch of 1024 x 2 ch x 48000 samples @ 44.1 kHz, forward + backward of loss = mean(y^2) with
gradients to x and to every parameter.  One "step" = one such pass over one synthetic batch.

Multi-GPU (one process per GPU, NCCL): the path is independent per item, so the batch is sharded by contiguous item
ranges with NO data-path collective.  Default `--scaling strong`: the BASELINE batch of 1024 items is split over the N
ranks (128 items per GPU at N = 8 -- the configuration BASELINE.json names); the same line also carries the
weak-scaling figure (1024 items per GPU) and, separately, the cost of the NCCL scatter/gather EDGES for a caller that
holds the batch on rank 0 (`edges`).  value = samples processed by all ranks / max-over-ranks device time.

The timed region replays ONE CUDA graph of the whole step (captured after the warm-up; the reverb draws fresh device
noise on every replay).  The JSON line carries: value (inputs resident in HBM), e2e (pinned-host inputs copied H2D,
loss + parameter gradients read back, every step), roofline of the dominant stage (algorithmic bytes / CUDA-event time
/ measured HBM peak; per-stage events come from an eager pass of the same step), per-config sub-results (BASELINE
configs 2-4), reference_gpu (the reference's own CUDA path on this GPU), cpu_baseline, clocks.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SR = 44100
N_SAMPLES = 48000
CHS = 2
IR_LEN = 96000
TAPS = 1023
METRIC = "audio samples/sec (fwd+bwd) @ batch=1024x2chx48k"
UNIT = "samples/s"
GLOBAL_BATCH = 1024


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------
# synthetic workload
# ------------------------------------------------------------------------------------------

def eq_ranges(sr=SR):
    g, q = (-20.0, 20.0), (0.1, 6.0)
    hi = (sr // 2) - 1000
    fr = [(20, 2000), (80, 2000), (2000, 8000), (8000, 12000), (12000, hi), (4000, hi)]
    out = []
    for f in fr:
        out += [g, f, q]
    return out


COMP_RANGES = [(-60.0, 0.0), (1.0, 20.0), (5.0, 100.0), (5.0, 100.0), (0.0, 12.0), (0.0, 12.0)]


def make_inputs(bs, seed):
    """seeded synthetic batch: x ~ U(-1,1), parameters ~ U(0,1) mapped through the reference Processor
    ranges (modules.py:136-155, 179-186, 204-230); distortion drive 0..24 dB per (item, channel) row.
    Returns x (bs, 2, N), p (bs, 49) = 18 EQ | 6 compressor | 25 reverb in physical units, drive (bs*2,)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(bs, CHS, N_SAMPLES, generator=g) * 2 - 1
    p01 = torch.rand(bs, 18 + 6 + 25, generator=g)
    p01[:, 22].clamp_(min=0.05)    # knee_db > 0: knee == 0 yields NaN gradients in the reference too
    lo = torch.tensor([r[0] for r in eq_ranges() + COMP_RANGES] + [0.0] * 25)
    hi = torch.tensor([r[1] for r in eq_ranges() + COMP_RANGES] + [1.0] * 25)
    p = p01 * (hi - lo) + lo
    drive = torch.rand(bs * CHS, generator=g) * 24.0
    return x, p, drive


def chain(mod, x, p, drive, **rev_kw):
    """the reference-facing calls: 18 + 6 + 25 per-item parameter tensors (columns of p), reference signatures"""
    cols = p.unbind(1)
    y = mod.parametric_eq(x, SR, *cols[:18])
    y = mod.compressor(y, SR, *cols[18:24])
    y = mod.noise_shaped_reverberation(y, SR, *cols[24:49], num_samples=IR_LEN, num_bandpass_taps=TAPS, **rev_kw)
    return mod.distortion(y, SR, drive)


# ------------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi in the background during the timed region)
# ------------------------------------------------------------------------------------------

class ClockSampler:
    """nvidia-smi polled in the background from before the warm-up; only the samples whose timestamps fall
    inside the timed region [t0, t1] are reported."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self, t0, t1):
        import datetime
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, sm_all, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [c.strip() for c in r.split(",")]
            if len(f) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                clk, cmax = float(f[1]), float(f[2])
            except ValueError:
                continue
            sm_all.append(clk)
            if not (t0 - 0.02 <= ts <= t1 + 0.02):
                continue
            sm.append(clk); mx.append(cmax)
            for nm, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples_in_timed_region": len(sm), "samples_total": len(sm_all), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------
# the reference itself: baseline/_ref holds the UNMODIFIED package (pip install --target, git-ignored, ships to the
# GPU box with the snapshot); when it is absent the oracle port of the same algorithm stands in (kind "port")
# ------------------------------------------------------------------------------------------

def load_reference():
    p = os.path.join(ROOT, "baseline", "_ref")
    if os.path.isdir(os.path.join(p, "dasp_pytorch")):
        if p not in sys.path:
            sys.path.insert(0, p)
        try:
            import dasp_pytorch.functional as ref_f       # noqa: F401
            return ref_f
        except Exception:
            return None
    return None


def reference_chain_seconds(mod, bs, device, rev_kw=None, reps=1, seed=1):
    """seconds per fwd+bwd chain step of `mod` (the reference's functional module, or the oracle port) on `device`.
    On CUDA the call runs under torch.set_default_device("cuda") like examples/demo.py:12-15, because the reference
    draws the reverb noise and builds its filters on the default device (functional.py:537-548)."""
    import torch
    x, p, drive = make_inputs(bs, seed=seed)               # CPU generator, before any default-device switch
    x, p, drive = x.to(device), p.to(device), drive.to(device)
    best = None
    try:
        if device != "cpu":
            torch.set_default_device(device)
        for _ in range(reps):
            leaves = [x.clone().requires_grad_(True), p.clone().requires_grad_(True), drive.clone().requires_grad_(True)]
            if device != "cpu":
                torch.cuda.synchronize()
            t0 = time.perf_counter()
            y = chain(mod, *leaves, **(rev_kw or {}))
            y.pow(2).mean().backward()
            if device != "cpu":
                torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
    finally:
        if device != "cpu":
            torch.set_default_device("cpu")
    return best


def cpu_arm(budget_s, warm=True, calibrate=True):
    """the reference's CPU path on the host cores: bs = 4, 8, 16 (BASELINE.md section 5) as far as the time budget
    allows; returns (samples/s at the largest batch finished, detail dict).

    Thread count: torchrun exports OMP_NUM_THREADS=1 and a 128-core box is NOT fastest with 128 intra-op threads (the
    reference's grouped conv1d collapses there: 93 s per item in round 2's first run, 23 s with 32 threads), so a
    one-item pass is timed at 8, 16, 32, ... threads until more threads stop helping and the fastest setting is kept --
    the reference gets the best configuration found, and `cores` reports it."""
    import torch
    ncpu = os.cpu_count() or 1
    try:
        ncpu = min(ncpu, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    ref = load_reference()
    if ref is not None:
        mod, kind, kw = ref, "reference", {}
    else:
        import oracle
        mod, kind, kw = oracle, "port", {"method": "direct"}
    t_start = time.perf_counter()
    cal = {}
    if calibrate:
        for t in [c for c in (8, 16, 32, 64, 128) if c <= ncpu] or [ncpu]:
            torch.set_num_threads(t)
            cal[t] = reference_chain_seconds(mod, 1, "cpu", kw)   # doubles as the warm-up pass (thread pools, scipy firwin)
            if cal[t] > 1.15 * min(cal.values()) or (time.perf_counter() - t_start) > 0.3 * budget_s:
                break                                             # more threads stopped helping (or the budget is going)
        best_t = min(cal, key=lambda k: cal[k])
        rates, times = {1: CHS * N_SAMPLES / cal[best_t]}, {1: cal[best_t]}
        batches = (4, 8, 16)
    else:
        # inside the GPU arm: no ladder (the reference arm found 16 threads fastest on the 128-core box, and its time
        # per call is dominated by a ~20 s batch-independent part, so a one-item sample would understate it 7x)
        best_t = min(16, ncpu)
        rates, times = {}, {}
        batches = (8, 16)
    torch.set_num_threads(best_t)
    for bs in batches:
        if times:
            est = times[max(times)] * max(1.0, bs / max(times) * 0.6)   # sub-linear in the batch on the boxes measured
            if (time.perf_counter() - t_start) + est > budget_s:
                break
        sec = reference_chain_seconds(mod, bs, "cpu", kw)
        times[bs] = sec
        rates[bs] = bs * CHS * N_SAMPLES / sec
    top = max(rates)
    lin = max(rates.values()) / min(rates.values())
    detail = {"kind": kind, "cores": best_t, "host_cpus": ncpu,
              "threads_tried_s_per_item": {str(k): round(v, 2) for k, v in cal.items()},
              "rates_by_batch": {str(k): round(v, 1) for k, v in rates.items()},
              "seconds_by_batch": {str(k): round(v, 2) for k, v in times.items()},
              "linearity_max_over_min": round(lin, 3),
              "sample": f"{top} item(s) x 2ch x 48000 (of the {GLOBAL_BATCH}-item batch), full chain fwd+bwd, "
                        f"{'the unmodified reference (baseline/_ref)' if kind == 'reference' else 'oracle port of the reference algorithm'}"
                        f": FFT-grid IIRs, time-domain conv1d reverb, CPU noise; {best_t} intra-op threads (best of those "
                        "tried); per-sample rate extrapolates linearly to the full batch"}
    return rates[top], times[top], top, detail


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    t0 = time.perf_counter()
    val, sec, bs, detail = cpu_arm(budget_s=170.0, warm=args.warmup > 0)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(detail["rates_by_batch"]), "steps_requested": args.steps, "warmup": 0, "warmup_requested": args.warmup,
        "note": "a CPU step takes tens of seconds: the run is capped at ~3 minutes whatever --steps / --warmup say; the "
                "timed steps are one fwd+bwd each at batch 1 (thread-count calibration, doubles as warm-up), 4, 8, 16 "
                "(as many as fit), value = rate at the largest batch finished",
        "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": make_config(args.batch, max(world, 1), args.scaling, None, graph=False),
        "cpu_baseline": {"value": val, "unit": UNIT, **detail},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": round(time.perf_counter() - t0, 1),
    }
    print(json.dumps(line), flush=True)


def reference_gpu(budget_s=40.0):
    """the reference's own CUDA path (PyTorch cuFFT / cuDNN dispatch of functional.py:118-577) on this GPU: the
    strongest existing implementation.  Largest batch of (4, 8, 16, 32) that fits the time budget."""
    import torch
    ref = load_reference()
    if ref is None:
        return {"unavailable": "baseline/_ref not present"}
    out = {"kind": "reference", "path": "dasp_pytorch.functional on device='cuda' (torch.set_default_device: the reverb "
                                        "draws its noise on the default device, examples/demo.py:12-15)"}
    try:
        t0 = time.perf_counter()
        reference_chain_seconds(ref, 2, "cuda")            # warm-up (cuDNN/cuFFT plan selection)
        rates = {}
        for bs in (4, 8, 16, 32):
            if time.perf_counter() - t0 > budget_s:
                break
            try:
                sec = reference_chain_seconds(ref, bs, "cuda", reps=2)
            except RuntimeError as e:                      # out of memory / unsupported convolution size
                out["stopped_at"] = f"bs={bs}: {str(e)[:120]}"
                torch.cuda.empty_cache()
                break
            rates[bs] = bs * CHS * N_SAMPLES / sec
        if not rates:
            return {**out, "unavailable": out.get("stopped_at", "no batch finished")}
        top = max(rates, key=lambda k: rates[k])
        out.update({"value": rates[top], "unit": UNIT, "batch": top,
                    "rates_by_batch": {str(k): round(v, 1) for k, v in rates.items()}})
        return out
    except Exception as e:                                 # never let the secondary baseline kill the bench line
        return {**out, "unavailable": f"{type(e).__name__}: {str(e)[:160]}"}
    finally:
        torch.cuda.empty_cache()


def make_config(bs_global, world, scaling, chunk, graph=True):
    per = bs_global // world if scaling == "strong" else bs_global
    cfg = {"workload": "configs[4]: chain eq->comp->reverb(12 bands, IR 96000, 1023 taps, device Philox noise)->dist, "
                        f"global batch {per * world} ({per}/GPU) x 2ch x 48000 @44.1k, fwd+bwd of mean(y^2), grads to x "
                        "and all params",
            "global_batch": per * world, "per_gpu_batch": per,
            "parallelism": f"dp{world} (contiguous item shards, no data-path collective)",
            "l2": "inputs (>= 49 MB/tensor/GPU, 393 MB at N=1) and the reverb's 4.7 MB/item intermediates exceed the "
                  "126 MB L2 within a step: no flush needed", "reverb_chunk_items": chunk,
            "timed_region": "replays of one CUDA graph of the whole step (fwd+bwd)"}
    if not graph:
        cfg["timed_region"] = "one eager fwd+bwd per step on a bounded sample of the batch (see cpu_baseline.sample)"
        cfg.pop("reverb_chunk_items")
        cfg["workload"] = cfg["workload"].replace("device Philox noise", "noise drawn by the reference itself")
    return cfg


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------

class Step:
    """the chain fwd+bwd on static device tensors, captured once into a CUDA graph"""

    def __init__(self, D, dev, bs, seed, pool=None):
        import torch
        self.torch, self.D, self.dev, self.bs = torch, D, dev, bs
        x_h, p_h, d_h = make_inputs(bs, seed)
        self.host = (x_h.pin_memory(), p_h.pin_memory(), d_h.pin_memory())
        self.x = self.host[0].to(dev).requires_grad_(True)
        self.p = self.host[1].to(dev).requires_grad_(True)
        self.d = self.host[2].to(dev).requires_grad_(True)
        self.graph = None
        self.loss = None
        self.y = None
        self.pool = pool

    def eager(self):
        for t in (self.x, self.p, self.d):
            t.grad = None
        self.y = None
        y = chain(self.D, self.x, self.p, self.d)
        loss = y.pow(2).mean()
        loss.backward()
        self.y = y.detach()
        return loss

    def capture(self, warm=3):
        torch = self.torch
        side = torch.cuda.Stream(device=self.dev)
        side.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(side):
            for _ in range(warm):
                self.eager()
        torch.cuda.current_stream(self.dev).wait_stream(side)
        torch.cuda.synchronize(self.dev)
        for t in (self.x, self.p, self.d):
            t.grad = None
        self.y = None
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, pool=self.pool):
            self.loss = self.eager()
        return self

    def replay(self):
        self.graph.replay()


DUMP_ITEMS = 32


def dump_outputs(step, out_dir):
    """Write what the last run of `step` computed as out_dir/<name>.npy (float32): the loss, dL/dp (bs, 49) and
    dL/d(drive) (bs*2,) whole, and y and dL/dx (DUMP_ITEMS, 2, N) for the items picked by a fixed seeded
    permutation of the batch (24.6 MB at N = 48000).  The inputs and the device noise are seeded, so the same
    arguments give the same arrays from one run to the next."""
    import numpy as np
    torch = step.torch
    items = torch.randperm(step.bs, generator=torch.Generator().manual_seed(0))[:DUMP_ITEMS].sort().values.to(step.dev)
    arrays = {"loss": step.loss, "y": step.y[items], "x_grad": step.x.grad[items], "p_grad": step.p.grad,
              "drive_grad": step.d.grad}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


def own_launches_per_step(bs, chunk_items):
    chunks = -(-bs // chunk_items)
    # eq fwd 1, bwd 2; compressor fwd 1, bwd 1; distortion fwd 1, bwd 2; reverb per chunk: fwd 5 (spectral_gen,
    # ifft_shape, x_fft, partition_mac, ifft_mix), bwd 5 (g_fft, partition_mac_bwd, ifft_dx, ifft_irgrad, param_grad)
    # (+ one cuFFT launch per chunk for the IR partitions, not counted: library kernel)
    return 1 + 2 + 1 + 1 + 1 + 2 + chunks * (5 + 5)


def bench_configs(D, F, dev, peak):
    """BASELINE configs 2-4 on one GPU (device-timed, L2 flushed between iterations): sub-results of the line"""
    import torch
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def timeit(fn, iters=5, warmup=2):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(iters):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return statistics.median(ts)

    def fwd_and_fb(fn, x):
        gy = torch.rand(x.shape[0], 2, x.shape[2], device=dev)
        with torch.no_grad():
            f = timeit(lambda: fn(x.detach()))

        def fb():
            fn(x).backward(gy)
            x.grad = None
        return f, timeit(fb)

    out = {}
    g = torch.Generator().manual_seed(7)
    lo = torch.tensor([r[0] for r in eq_ranges()]); hi = torch.tensor([r[1] for r in eq_ranges()])
    # c2: parametric_eq 256 x 2 x 48000
    bs = 256
    x = (torch.rand(bs, 2, N_SAMPLES, generator=g) * 2 - 1).to(dev).requires_grad_(True)
    p = [q.to(dev).requires_grad_(True) for q in (torch.rand(bs, 18, generator=g) * (hi - lo) + lo).unbind(1)]
    f, fb = fwd_and_fb(lambda xx: D.parametric_eq(xx, SR, *p), x)
    e = bs * 2 * N_SAMPLES
    out["c2_parametric_eq_256x2x48000"] = {"fwd_ms": round(f, 4), "fwdbwd_ms": round(fb, 4),
                                          "fwd_frac": round(8 * e / f / 1e6 / peak, 4),
                                          "bwd_frac": round(12 * e / max(fb - f, 1e-6) / 1e6 / peak, 4),
                                          "gsamples_per_s": round(e / fb / 1e6, 2)}
    # c3: compressor + expander 512 x 2 x 48000
    bs = 512
    x = (torch.rand(bs, 2, N_SAMPLES, generator=g) * 2 - 1).to(dev).requires_grad_(True)
    clo = torch.tensor([r[0] for r in COMP_RANGES]); chi = torch.tensor([r[1] for r in COMP_RANGES])
    c01 = torch.rand(bs, 6, generator=g); c01[:, 4].clamp_(min=0.05)
    pc = [q.to(dev).requires_grad_(True) for q in (c01 * (chi - clo) + clo).unbind(1)]
    e = bs * 2 * N_SAMPLES
    for name, fn in (("compressor", D.compressor), ("expander", D.expander)):
        f, fb = fwd_and_fb(lambda xx, fn=fn: fn(xx, SR, *pc), x)
        out[f"c3_{name}_512x2x48000"] = {"fwd_ms": round(f, 4), "fwdbwd_ms": round(fb, 4),
                                         "fwd_frac": round(8 * e / f / 1e6 / peak, 4),
                                         "bwd_frac": round(12 * e / max(fb - f, 1e-6) / 1e6 / peak, 4),
                                         "gsamples_per_s": round(e / fb / 1e6, 2)}
    # c4: noise_shaped_reverberation 256 x 2 x 48000, IR 96000, 12 bands (the reference signature has no 8-band form)
    bs = 256
    x = (torch.rand(bs, 2, N_SAMPLES, generator=g) * 2 - 1).to(dev).requires_grad_(True)
    pr = [torch.rand(bs, generator=g).to(dev).requires_grad_(True) for _ in range(25)]
    f, fb = fwd_and_fb(lambda xx: D.noise_shaped_reverberation(xx, SR, *pr, num_samples=IR_LEN, num_bandpass_taps=TAPS), x)
    e = bs * 2 * N_SAMPLES
    out["c4_reverb_256x2x48000_ir96000"] = {"fwd_ms": round(f, 4), "fwdbwd_ms": round(fb, 4),
                                           "gsamples_per_s": round(e / fb / 1e6, 2)}
    del flush
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference-cuda"])
    ap.add_argument("--batch", type=int, default=GLOBAL_BATCH, help="GLOBAL batch under strong scaling, per-GPU batch "
                                                                   "under weak scaling (BASELINE config: 1024)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--no-extras", action="store_true", help="skip sub-configs / reference_gpu / cpu_baseline / edges")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the outputs of the last one "
                                                          "as DIR/<name>.npy (rank 0's shard when N > 1)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200 only")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if args.impl == "reference-cuda":
        if rank == 0:
            import torch
            torch.cuda.set_device(0)
            r = reference_gpu(budget_s=120.0)
            print(json.dumps({"impl": "reference-cuda", "metric": METRIC, "unit": UNIT, "n_gpus": 1, **r}), flush=True)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist

    import dasp_pytorch_b200 as D
    from dasp_pytorch_b200 import dist as ddist
    from dasp_pytorch_b200 import functional as F

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback exists)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    torch.cuda.manual_seed(1000 + rank)     # torch seeds its CUDA generator at random; the reverb draws its noise from it
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    if args.scaling == "strong":
        lo, hi = ddist.shard_bounds(args.batch, world, rank)
        bs = hi - lo
        total_items = args.batch
    else:
        bs = args.batch
        total_items = args.batch * world
    samples_per_step = total_items * CHS * N_SAMPLES            # whole job

    sampler = ClockSampler(local_rank)
    sampler.start()
    step = Step(D, dev, bs, seed=1000 + rank)
    for _ in range(args.warmup):
        step.eager()
    barrier()

    # ---- per-stage CUDA events: the step run eagerly (events cannot be recorded inside a graph) ----
    n_eager = min(args.steps, 10)
    F.STAGE_TIMING = []
    ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ea.record()
    for _ in range(n_eager):
        step.eager()
    eb.record()
    barrier()
    eager_ms = max_over_ranks(ea.elapsed_time(eb)) / n_eager
    stage_events, F.STAGE_TIMING = F.STAGE_TIMING, None
    stages = {}
    for name, a, b in stage_events:
        stages.setdefault(name, []).append(a.elapsed_time(b))

    step.capture(warm=2)
    for _ in range(args.warmup):
        step.replay()
    barrier()

    # ---- timed region: K replays of the captured step, CUDA events on the launching stream ----
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    wall0 = time.time()
    e0.record()
    for _ in range(args.steps):
        step.replay()
    e1.record()
    barrier()
    wall1 = time.time()
    ms_max = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop(wall0, wall1)
    value = samples_per_step * args.steps / (ms_max * 1e-3)
    loss_val = float(step.loss.item())
    if args.dump_outputs and rank == 0:
        dump_outputs(step, args.dump_outputs)        # before the end-to-end replays below overwrite the outputs

    # ---- end-to-end: pinned host inputs -> H2D -> graph replay -> D2H of loss and parameter gradients ----
    # Every step uploads ITS inputs from pinned host memory into a staging set on a copy stream (overlapping the
    # previous step's compute, like any input pipeline), the step's graph reads its own static tensors after a
    # device-side copy from the staging set, and the loss + all parameter gradients are read back every step.
    copy_stream = torch.cuda.Stream(device=dev)
    stage_bufs = [tuple(torch.empty_like(t, device=dev) for t in step.host) for _ in range(2)]

    def upload(k):
        with torch.cuda.stream(copy_stream):
            for dst, src in zip(stage_bufs[k & 1], step.host):
                dst.copy_(src, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return ev

    def e2e_loop(n_steps):
        ev = upload(0)
        out = None
        done = None
        for k in range(n_steps):
            torch.cuda.current_stream(dev).wait_event(ev)
            with torch.no_grad():
                for dst, src in zip((step.x, step.p, step.d), stage_bufs[k & 1]):
                    dst.copy_(src)
            done = torch.cuda.Event()
            done.record()
            if k + 1 < n_steps:
                copy_stream.wait_event(done)                # staging set (k+1)&1 was last read by step k-1's copy
                ev = upload(k + 1)
            step.replay()
            out = (float(step.loss.item()), step.p.grad.cpu(), step.d.grad.cpu())      # D2H read of this step's results
        return out

    e2e_loop(2)
    barrier()
    t0 = time.perf_counter()
    e2e_loop(args.steps)
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_value = samples_per_step * args.steps / e2e_s
    h2d = sum(t.numel() * 4 for t in step.host)
    d2h = 4 + bs * 49 * 4 + bs * CHS * 4

    extras = {}
    if world > 1:
        # cross-GPU self-check (the driver's pytest box has one GPU, so tests/test_gpu_multi.py is skipped there): every
        # rank runs eq -> compressor -> distortion fwd+bwd on the SAME small seeded batch; outputs and gradients must be
        # bit-identical on all GPUs (items are independent, no atomics, fixed reduction orders)
        gchk = torch.Generator().manual_seed(4242)
        xc = (torch.rand(6, CHS, 6000, generator=gchk) * 2 - 1).to(dev).requires_grad_(True)
        pc01 = torch.rand(6, 24, generator=gchk)
        pc01[:, 22].clamp_(min=0.05)
        lo = torch.tensor([r[0] for r in eq_ranges() + COMP_RANGES]); hi = torch.tensor([r[1] for r in eq_ranges() + COMP_RANGES])
        pc = (pc01 * (hi - lo) + lo).to(dev).requires_grad_(True)
        dc = (torch.rand(12, generator=gchk) * 24).to(dev)
        cols = pc.unbind(1)
        yc = D.distortion(D.compressor(D.parametric_eq(xc, SR, *cols[:18]), SR, *cols[18:24]), SR, dc)
        yc.pow(2).mean().backward()
        sig = torch.cat([yc.detach().reshape(-1), xc.grad.reshape(-1), pc.grad.reshape(-1)]).contiguous()
        allsig = [torch.empty_like(sig) for _ in range(world)]
        dist.all_gather(allsig, sig)
        extras["cross_gpu_bit_identity"] = bool(all(torch.equal(a, allsig[0]) for a in allsig))
        del xc, pc, yc
    if world > 1 and not args.no_extras:
        # ---- (a) the NCCL edges for a caller that holds the whole batch on rank 0: scatter x / params / drive,
        #      gather y (SURVEY 8e(b)); timed separately from the compute, device events, max over ranks ----
        gb = args.batch                                      # the BASELINE batch, split over the ranks
        full = None
        if rank == 0:
            gx_, gp_, gd_ = make_inputs(gb, seed=77)
            full = (gx_.to(dev), gp_.to(dev), gd_.reshape(gb, CHS).to(dev))
        y_local = torch.empty(ddist.shard_sizes(gb, world)[rank], CHS, N_SAMPLES, device=dev)
        sc, ga = [], []
        for it in range(4):
            barrier()
            a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            a.record()
            xs = ddist.scatter_batch(full[0] if rank == 0 else None, gb, (CHS, N_SAMPLES), torch.float32, dev)
            ps = ddist.scatter_batch(full[1] if rank == 0 else None, gb, (49,), torch.float32, dev)
            ds = ddist.scatter_batch(full[2] if rank == 0 else None, gb, (CHS,), torch.float32, dev)
            b.record()
            yg = ddist.gather_batch(y_local, gb)
            c.record()
            barrier()
            if it > 0:
                sc.append(max_over_ranks(a.elapsed_time(b)))
                ga.append(max_over_ranks(b.elapsed_time(c)))
            del xs, ps, ds, yg
        nbytes = gb * CHS * N_SAMPLES * 4
        extras["edges"] = {"what": "NCCL scatter of x/params/drive from rank 0 + gather of y to rank 0 (grouped send/recv, "
                                   "no padding), NOT part of value", "scatter_ms": round(statistics.median(sc), 3),
                           "gather_ms": round(statistics.median(ga), 3), "bytes_each_way": nbytes,
                           "scatter_GBps_root": round(nbytes * (world - 1) / world / statistics.median(sc) / 1e6, 1)}
        del full, y_local
        torch.cuda.empty_cache()
        # ---- (b) the other scaling mode in the same run ----
        other = "weak" if args.scaling == "strong" else "strong"
        obs = args.batch if other == "weak" else ddist.shard_sizes(args.batch, world)[rank]
        del step.graph
        step = None
        torch.cuda.empty_cache()
        st2 = Step(D, dev, obs, seed=2000 + rank).capture(warm=3)
        st2.replay()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n2 = min(args.steps, 10)
        a.record()
        for _ in range(n2):
            st2.replay()
        b.record()
        barrier()
        ms2 = max_over_ranks(a.elapsed_time(b))
        items2 = args.batch * world if other == "weak" else args.batch
        extras[other] = {"scaling": other, "per_gpu_batch": obs, "global_batch": items2, "steps": n2,
                         "ms_per_step": round(ms2 / n2, 4), "value": items2 * CHS * N_SAMPLES * n2 / (ms2 * 1e-3)}
        del st2
        torch.cuda.empty_cache()
        # ---- (c) BASELINE config 4 ("reverb 256 stereo, IR 96000, 1 -> 4 GPU"): the 256 items split over the ranks ----
        b4 = ddist.shard_sizes(256, world)[rank]
        g4 = torch.Generator().manual_seed(7 + rank)
        x4 = (torch.rand(max(b4, 1), CHS, N_SAMPLES, generator=g4) * 2 - 1).to(dev).requires_grad_(True)
        p4 = [torch.rand(max(b4, 1), generator=g4).to(dev).requires_grad_(True) for _ in range(25)]
        gy4 = torch.rand(max(b4, 1), CHS, N_SAMPLES, device=dev)
        flush4 = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

        def c4_step():
            D.noise_shaped_reverberation(x4, SR, *p4, num_samples=IR_LEN, num_bandpass_taps=TAPS).backward(gy4)
            x4.grad = None

        for _ in range(2):
            c4_step()
        ts4 = []
        for _ in range(5):
            flush4.zero_()
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); c4_step(); b.record()
            barrier()
            ts4.append(max_over_ranks(a.elapsed_time(b)))
        ms4 = statistics.median(ts4)
        extras["c4_reverb_256x2x48000_ir96000_sharded"] = {
            "items_per_gpu": ddist.shard_sizes(256, world), "fwdbwd_ms": round(ms4, 4),
            "gsamples_per_s": round(256 * CHS * N_SAMPLES / ms4 / 1e6, 2),
            "note": "eager fwd+bwd of the 256-item batch split over the ranks, device-timed, max over ranks, L2 flushed"}
        del x4, p4, gy4, flush4
        torch.cuda.empty_cache()

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        e = bs * CHS * N_SAMPLES
        leff = min(IR_LEN, N_SAMPLES)       # only the first min(L, N) IR taps can reach the N outputs (DESIGN.md)
        item_rev_fwd = (2 * N_SAMPLES * 4) * 2 + 2 * (2 * leff * 4)                # x in, y out, IR write + read
        item_rev_bwd = 3 * (2 * N_SAMPLES * 4) + 2 * leff * 4 + 2 * (2 * leff * 4) + 2 * 12 * leff * 4
        alg = {  # algorithmic bytes per launch (SURVEY.md 8d): 8 B/sample fwd, 12 B/sample bwd for the streaming ops
            "eq_fwd": 8 * e, "eq_bwd": 12 * e, "comp_fwd": 8 * e, "comp_bwd": 12 * e, "dist_fwd": 8 * e,
            "dist_bwd": 12 * e, "reverb_fwd": item_rev_fwd * bs, "reverb_bwd": item_rev_bwd * bs,
        }
        kern = {"eq_fwd": "eq_fwd_kernel", "eq_bwd": "eq_bwd_kernel (+ eq_param_grad_kernel)", "comp_fwd": "dynamics_fwd_kernel",
                "comp_bwd": "dynamics_bwd_kernel", "dist_fwd": "pointwise_fwd_kernel", "dist_bwd": "pointwise_bwd_kernel",
                "reverb_fwd": "reverb fwd pipeline: spectral_gen_kernel, ifft_shape_kernel, x_fft_kernel, partition_mac_kernel, "
                              "ifft_mix_kernel (own in-shared-memory 8192-point FFT fused with the element-wise stages), "
                              "cuFFT C2C(8192) x1 (IR partitions)",
                "reverb_bwd": "reverb bwd pipeline: g_fft_kernel, partition_mac_kernel x2, ifft_dx_kernel, "
                              "ifft_irgrad_kernel (all on the own in-shared-memory FFT), reverb_param_grad_kernel"}
        # DRAM bytes actually moved by the two reverb pipelines (dram__bytes_read.sum + dram__bytes_write.sum summed
        # over their kernels, one `ncu --set full` capture of a chunk at this geometry): read from the committed
        # summary that tools/summarize_profiles.py writes, never typed in here
        traffic_item = {}
        try:
            with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
                tj = json.load(f)
            if tj.get("geometry") == [N_SAMPLES, IR_LEN, TAPS]:
                traffic_item = {k: float(v) for k, v in tj["dram_bytes_per_item"].items()}
                traffic_src = tj.get("source")
        except Exception:
            traffic_src = None
        breakdown = {}
        for name, v in stages.items():
            m = statistics.mean(v)
            breakdown[name] = {"ms": round(m, 4), "alg_GBps": round(alg[name] / (m * 1e-3) / 1e9, 1),
                               "frac": round(alg[name] / (m * 1e-3) / 1e9 / peak, 4)}
        dom = max(breakdown, key=lambda k: breakdown[k]["ms"]) if breakdown else None
        roofline = None
        if dom:
            roofline = {"bound": "hbm", "kernel": kern[dom], "achieved": breakdown[dom]["alg_GBps"], "peak": peak,
                        "unit": "GB/s", "frac": breakdown[dom]["frac"],
                        "traffic": traffic_item[dom] * bs if dom in traffic_item else None,
                        "traffic_source": traffic_src if dom in traffic_item else None, "peak_source": peak_src,
                        "algorithmic_bytes_per_launch": alg[dom], "ms_per_launch": breakdown[dom]["ms"],
                        "note": "stage = one C-ABI call, timed with CUDA events around it in an eager pass of the same step"}
        if roofline and dom in ("reverb_fwd", "reverb_bwd"):
            # context, not the roofline: the reverb is transform work, not streaming.  Transforms per item (8192-point
            # complex, 5 n log2 n flops): forward 12 bands x R classes (IR synthesis) + J (IR partitions) + 2 I (audio in,
            # wet out); backward I (dL/dy) + I (dL/dx) + J (dL/dIR).  Peak = SMs x 128 lanes x 2 x max SM clock.
            R = -(-(leff + TAPS - 1) // 8192); I = -(-N_SAMPLES // 4096); J = -(-leff // 4096)
            nfft = (12 * R + J + 2 * I) if dom == "reverb_fwd" else (2 * I + J)
            flops = nfft * 5 * 8192 * 13 * bs
            props = torch.cuda.get_device_properties(dev)
            fp32_peak = props.multi_processor_count * 128 * 2 * (clocks.get("sm_max_mhz") or 1965.0) * 1e6 / 1e12
            roofline["fft_context"] = {
                "transforms_per_item": nfft, "fft_TFLOPs": round(flops / (breakdown[dom]["ms"] * 1e-3) / 1e12, 2),
                "fp32_peak_TFLOPs": round(fp32_peak, 1),
                "frac_of_fp32_peak": round(flops / (breakdown[dom]["ms"] * 1e-3) / 1e12 / fp32_peak, 3),
                "note": "5 n log2 n flops of the 8192-point transforms only (generator, MACs, shaping not counted)"}
        chunk_items = F.reverb_chunk_items(dev)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": make_config(args.batch, world, args.scaling, chunk_items),
            "roofline": roofline, "stages": breakdown, "eager_ms_per_step": round(eager_ms, 4),
            "stage_sum_ms": round(sum(v["ms"] for v in breakdown.values()), 4), "loss": loss_val,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": own_launches_per_step(bs, chunk_items) * args.steps, "clocks": clocks, **extras,
        }
        if world == 1 and not args.no_extras:
            del step
            torch.cuda.empty_cache()
            line["configs"] = bench_configs(D, F, dev, peak)
            line["reference_gpu"] = reference_gpu(budget_s=30.0)
            val, sec, cbs, detail = cpu_arm(budget_s=80.0, warm=True, calibrate=False)
            line["cpu_baseline"] = {"value": val, "unit": UNIT, **detail}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
