// compressor / expander forward + backward
// (reference: dasp_pytorch/functional.py:275-399; expander is new, SURVEY.md 8a8).
//
// One CTA per batch item; the CTA walks the item's N samples tile by tile through the TMA
// pipeline in tile_pipe.cuh, all C channels of a tile together (the side chain is the channel
// sum, functional.py:328).  Inside a tile thread t owns E consecutive samples; the attack
// smoother  s[n] = a s[n-1] + (1-a) gc[n]  (functional.py:372-380, there via FFT) is evaluated
// as a time-parallel first-order recurrence:
//     thread-local pass (zero incoming state)  ->  Kogge-Stone scan of the per-thread end
//     states across the warp with shuffles, using the precomputed powers a^(E*2^k)  ->
//     cross-warp carry through shared memory  ->  fix-up  s[j] += a^(j+1) * carry_in,
// with the tile-to-tile carry kept in a register.  Everything else (channel sum, dB, soft-knee
// static curve, makeup, dB->linear, apply) is fused around it, so HBM traffic is the
// algorithmic 8 B/sample forward and 12 B/sample backward.
//
// Backward (SURVEY.md Appendix A.4): the forward stores only the smoother state at every tile
// boundary (one float per tile).  The backward sweeps the tiles in REVERSE time order; per tile
// it recomputes the forward quantities from that checkpoint, then runs the adjoint recurrence
// w[n] = ds[n] + a w[n+1] with the mirrored scan (shfl_down), accumulates the five parameter
// gradients in registers across tiles (deterministic), and writes dL/dx in place.
#include <math.h>

#include "common.cuh"
#include "tile_pipe.cuh"

namespace dasp {
namespace {

constexpr int kE = 7;                 // samples per thread per tile; odd => stride-E smem access is conflict-free
constexpr int kStages = 3;
constexpr int kBwdMinBlocks = 4;      // resident CTAs per SM the backward is compiled for at W = 4 (register budget 65536 / (128 * 4))
constexpr int kMaxChs = 32;
constexpr float kDbPerLog2 = 6.020599913279624f;    // 20*log10(2)
constexpr float kDbGradScale = 8.685889638065035f;  // 20/ln(10)

enum class Curve { Compress, Expand };

struct DynParams {
  const float* x;        // (bs, C, N)
  const float* gy;       // (bs, C, N)   backward only
  float* y;              // (bs, C, N)   forward out / backward gx
  const float* threshold_db;  // [bs]
  const float* ratio;
  const float* attack_ms;
  const float* knee_db;
  const float* makeup_db;
  float* ckpt;           // (bs, ntiles) smoother state entering each tile (fwd: out or null; bwd: in)
  float* gparams;        // (bs, 6) backward out: dT, dR, dAttack, dRelease(=0), dKnee, dMakeup
  float* g_scratch;      // (bs, N) linear gain, only written by the backward when lookahead > 0
  int64_t n;
  int chs;
  int ntiles;
  int lookahead;
  float sample_rate;
  float eps;
  int bulk;
};

struct ChannelRows {      // forward: buffer c <-> channel c of x (in) and y (out)
  const float* x0; float* y0; int64_t n;
  __device__ __forceinline__ const float* src(int b) const { return x0 + (int64_t)b * n; }
  __device__ __forceinline__ float* dst(int b) const { return y0 + (int64_t)b * n; }
};
struct BwdRows {          // backward: buffers [0,C) = x (read only), [C,2C) = gy (in) -> gx (out)
  const float* x0; const float* g0; float* gx0; int64_t n; int chs;
  __device__ __forceinline__ const float* src(int b) const {
    return b < chs ? x0 + (int64_t)b * n : g0 + (int64_t)(b - chs) * n;
  }
  __device__ __forceinline__ float* dst(int b) const { return b < chs ? nullptr : gx0 + (int64_t)(b - chs) * n; }
};

// ---- per-item constants of the smoother ---------------------------------------------------
struct PoleTables {
  float alpha, beta;     // a, 1-a
  float apow[kE + 1];    // a^1 .. a^(E+1)   (apow[j] = a^(j+1))
  float step[5];         // a^(E*2^k), k = 0..4  (warp scan)
  float lane_pow;        // a^(E*lane)
  float warp_pow;        // a^(32E)
};

__device__ __forceinline__ void make_tables(PoleTables& t, float attack_ms, float sample_rate, int lane) {
  // alpha = exp(-ln9 / (sr * attack_ms / 1e3))  (functional.py:339-342), evaluated in fp64; every power is
  // then built from it by fp64 multiplications (one exp2 call instead of fifteen)
  const double l2a = -3.169925001442312 /* log2(9) */ / ((double)sample_rate * ((double)attack_ms * 1e-3));
  const double a = exp2(l2a);
  t.alpha = (float)a;
  t.beta = (float)(1.0 - a);
  double pw = a;
#pragma unroll
  for (int j = 0; j <= kE; ++j) { t.apow[j] = (float)pw; pw *= a; }      // a^1 .. a^(E+1)
  double st = 1.0;
#pragma unroll
  for (int j = 0; j < kE; ++j) st *= a;                                   // a^E
  double lp = 1.0;
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    t.step[k] = (float)st;
    if ((lane >> k) & 1) lp *= st;                                        // a^(E*lane) from the bits of lane
    st *= st;
  }
  t.lane_pow = (float)lp;
  t.warp_pow = (float)st;                                                 // a^(32E)
}

// Forward-in-time scan of first-order states across the CTA.
//   v      : this thread's end state after its zero-state local pass
//   c_tile : state entering the tile (same value in every thread)
// returns the state entering this thread's chunk; c_tile is updated to the state leaving the tile.
template <int W>
__device__ __forceinline__ float scan_forward(float v, float& c_tile, const PoleTables& t, float* agg, int lane,
                                              int warp) {
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    float u = __shfl_up_sync(0xffffffffu, v, 1 << k);
    if (lane >= (1 << k)) v = fmaf(t.step[k], u, v);
  }
  float excl = __shfl_up_sync(0xffffffffu, v, 1);
  if (lane == 0) excl = 0.f;
  float c_warp = c_tile;
  if (W > 1) {
    if (lane == 31) agg[warp] = v;
    __syncthreads();
    float c = c_tile;
#pragma unroll
    for (int w = 0; w < W; ++w) {
      if (w == warp) c_warp = c;
      c = fmaf(t.warp_pow, c, agg[w]);
    }
    c_tile = c;
  } else {
    float tot = __shfl_sync(0xffffffffu, v, 31);
    c_tile = fmaf(t.warp_pow, c_tile, tot);
  }
  return fmaf(t.lane_pow, c_warp, excl);
}

// Mirror image for the adjoint recurrence w[n] = ds[n] + a w[n+1]: information flows from high
// thread index to low.  v = this thread's value at its FIRST sample after the zero-state local
// reverse pass; c_tile = w at the first sample of the NEXT tile (in time).
template <int W>
__device__ __forceinline__ float scan_reverse(float v, float& c_tile, const PoleTables& t, float rlane_pow, float* agg,
                                              int lane, int warp) {
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    float u = __shfl_down_sync(0xffffffffu, v, 1 << k);
    if (lane + (1 << k) < 32) v = fmaf(t.step[k], u, v);
  }
  float excl = __shfl_down_sync(0xffffffffu, v, 1);
  if (lane == 31) excl = 0.f;
  float c_warp = c_tile;
  if (W > 1) {
    if (lane == 0) agg[warp] = v;
    __syncthreads();
    float c = c_tile;
#pragma unroll
    for (int w = W - 1; w >= 0; --w) {
      if (w == warp) c_warp = c;
      c = fmaf(t.warp_pow, c, agg[w]);
    }
    c_tile = c;
  } else {
    float tot = __shfl_sync(0xffffffffu, v, 0);
    c_tile = fmaf(t.warp_pow, c_tile, tot);
  }
  // rlane_pow = a^(E*(31-lane)): distance from the start of thread lane+1 ... to the warp's right edge
  return fmaf(rlane_pow, c_warp, excl);
}

// ---- static gain computer (dB in, dB gain out) + partial derivatives ----------------------
struct CurveOut { float gc, d_xdb, d_t, d_r, d_w; };

// per-item constants of the static curve: every division is done once per item, not once per sample
struct CurveK {
  float T, half, lo, hi;       // threshold, W/2, knee edges T -+ W/2
  float slope;                 // compressor: 1/R - 1          expander: 1 - R
  float inv_w, inv_2w;         // 1/W, 1/(2W)  (W == 0 -> inf, poisoning the knee exactly like the reference's 0/0)
  float inv_r2;                // 1/R^2
  float r_m1;                  // R - 1
};
__device__ __forceinline__ CurveK make_curve(Curve cv, float T, float R, float Wk) {
  CurveK k;
  k.T = T; k.half = 0.5f * Wk; k.lo = T - k.half; k.hi = T + k.half;
  k.slope = (cv == Curve::Compress) ? (1.0f / R - 1.0f) : (1.0f - R);
  k.inv_w = 1.0f / Wk; k.inv_2w = 0.5f * k.inv_w;
  k.inv_r2 = 1.0f / (R * R);
  k.r_m1 = R - 1.0f;
  return k;
}

template <Curve CV, bool GRAD>
__device__ __forceinline__ CurveOut gain_computer(float xdb, const CurveK& k) {
  CurveOut o; o.gc = 0.f; o.d_xdb = 0.f; o.d_t = 0.f; o.d_r = 0.f; o.d_w = 0.f;
  const bool in_knee = (xdb >= k.lo) && (xdb <= k.hi);
  if (CV == Curve::Compress) {
    // functional.py:350-369 expressed as gc = x_sc - x_db
    if (in_knee) {
      const float d = xdb - k.lo;                     // x_db - T + W/2
      const float q = d * d * k.inv_2w;               // d^2 / (2W)
      o.gc = k.slope * q;
      if (GRAD) {
        o.d_xdb = k.slope * d * k.inv_w;
        o.d_t = -o.d_xdb;
        o.d_r = -q * k.inv_r2;
        o.d_w = k.slope * (d * k.inv_2w - q * k.inv_w);
      }
    } else if (xdb > k.hi) {
      o.gc = (xdb - k.T) * k.slope;                   // (T - x)(1 - 1/R)
      if (GRAD) {
        o.d_xdb = k.slope;
        o.d_t = -k.slope;
        o.d_r = (k.T - xdb) * k.inv_r2;
      }
    }
  } else {
    // downward expander (oracle/dasp_oracle.py::_expander_curve)
    if (in_knee) {
      const float d = xdb - k.hi;                     // x_db - T - W/2
      const float q = d * d * k.inv_2w;
      o.gc = k.slope * q;                             // (1 - R) d^2 / (2W)
      if (GRAD) {
        o.d_xdb = k.slope * d * k.inv_w;
        o.d_t = -o.d_xdb;
        o.d_r = -q;
        o.d_w = k.slope * (-d * k.inv_2w - q * k.inv_w);
      }
    } else if (xdb < k.lo) {
      o.gc = k.r_m1 * (xdb - k.T);
      if (GRAD) {
        o.d_xdb = k.r_m1;
        o.d_t = -k.r_m1;
        o.d_r = xdb - k.T;
      }
    }
  }
  return o;
}

// 20 log10(max(|xs|, eps)); __log2f is the single-instruction MUFU.LG2 (|rel err| < 2^-22 for normal inputs,
// i.e. < 1e-5 dB here) -- the accurate log2f costs ~15 instructions in a kernel that is issue bound
__device__ __forceinline__ float level_db(float xs, float eps) { return kDbPerLog2 * __log2f(fmaxf(fabsf(xs), eps)); }

// shared-memory carve-up (dynamic smem): [S mbarriers][pad to 64][agg: 4*W floats][pad to 512][stages]
template <int W>
struct Smem {
  uint64_t* bars; float* agg; float* stages;
  __device__ __forceinline__ Smem(unsigned char* base) {
    bars = reinterpret_cast<uint64_t*>(base);
    agg = reinterpret_cast<float*>(base + 64);        // up to 4 * 16 floats (backward, W = 16)
    stages = reinterpret_cast<float*>(base + 512);
  }
};
constexpr size_t kSmemHeader = 512;

// =============================================================================== forward
// LA: lookahead_samples > 0 (rare; kept out of the common instantiation).  ST: stereo specialisation (C == 2, no
// look-ahead): the two channel values of a sample stay in registers between the side-chain sum and the gain application
// instead of being read from shared memory twice (round 2: the scan kernels are bound by the shared-memory pipe).
template <Curve CV, int W, bool LA, bool ST = false>
__global__ void __launch_bounds__(W * 32) dynamics_fwd_kernel(DynParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  Smem<W> sm(smem_raw);
  const int item = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int C = p.chs;
  const int tile_len = W * 32 * kE;

  const float M = p.makeup_db[item];
  const CurveK ck = make_curve(CV, p.threshold_db[item], p.ratio[item], p.knee_db[item]);
  PoleTables tb;
  make_tables(tb, p.attack_ms[item], p.sample_rate, lane);

  TileGeom g{p.n, tile_len, p.ntiles, false};
  ChannelRows rows{p.x + (int64_t)item * C * p.n, p.y + (int64_t)item * C * p.n, p.n};
  TilePipe<kStages> pipe;
  pipe.init(sm.bars, sm.stages, C, tile_len, p.bulk != 0);
  pipe.prologue(g, rows);

  float c_tile = 0.f;                      // smoother state entering the current tile
  const int off = threadIdx.x * kE;        // this thread's first sample inside a tile
  for (int i = 0; i < p.ntiles; ++i) {
    pipe.acquire(i, g, rows);
    const int st = i % kStages;
    const int64_t n0 = (int64_t)i * tile_len + off;
    if (p.ckpt && threadIdx.x == 0) p.ckpt[(int64_t)item * p.ntiles + i] = c_tile;

    // side chain + static curve + zero-state local pass
    float s[kE];
    float x0[ST ? kE : 1], x1[ST ? kE : 1];
    {
      float xs[kE];
      if (ST) {
        const float* xa = pipe.buf(st, 0) + off;
        const float* xb = pipe.buf(st, 1) + off;
#pragma unroll
        for (int j = 0; j < kE; ++j) { x0[ST ? j : 0] = xa[j]; x1[ST ? j : 0] = xb[j]; xs[j] = xa[j] + xb[j]; }
      } else {
#pragma unroll
        for (int j = 0; j < kE; ++j) xs[j] = 0.f;
        for (int c = 0; c < C; ++c) {
          const float* xb = pipe.buf(st, c) + off;
#pragma unroll
          for (int j = 0; j < kE; ++j) xs[j] += xb[j];
        }
      }
      float run = 0.f;
#pragma unroll
      for (int j = 0; j < kE; ++j) {
        float gc = 0.f;
        if (n0 + j < p.n) gc = gain_computer<CV, false>(level_db(xs[j], p.eps), ck).gc;
        run = fmaf(tb.alpha, run, tb.beta * gc);
        s[j] = run;
      }
    }
    const float c_in = scan_forward<W>(s[kE - 1], c_tile, tb, sm.agg + (i & 1) * W, lane, warp);

    // fix-up, dB -> linear, apply to every channel (in place)
    float G[kE];
#pragma unroll
    for (int j = 0; j < kE; ++j) G[j] = exp2f((fmaf(tb.apow[j], c_in, s[j]) + M) * kLog2Of10Over20);
    if (ST) {
      float* xa = pipe.buf(st, 0) + off;
      float* xb = pipe.buf(st, 1) + off;
#pragma unroll
      for (int j = 0; j < kE; ++j) { xa[j] = x0[ST ? j : 0] * G[j]; xb[j] = x1[ST ? j : 0] * G[j]; }
    } else if (!LA) {
      for (int c = 0; c < C; ++c) {
        float* xb = pipe.buf(st, c) + off;
#pragma unroll
        for (int j = 0; j < kE; ++j) xb[j] *= G[j];
      }
    } else {
      // y[n] = x[n - la] * G[n]  (functional.py:383-385): delayed input straight from global/L2
      for (int c = 0; c < C; ++c) {
        float* xb = pipe.buf(st, c) + off;
        const float* xr = rows.src(c);
#pragma unroll
        for (int j = 0; j < kE; ++j) {
          const int64_t m = n0 + j - p.lookahead;
          xb[j] = (m >= 0 && n0 + j < p.n) ? xr[m] * G[j] : 0.f;
        }
      }
    }
    pipe.release(i, g, rows);
  }
  pipe.drain();
}

// =============================================================================== backward
template <Curve CV, int W, bool LA, bool ST = false>
__global__ void __launch_bounds__(W * 32, (W <= 4) ? (4 * kBwdMinBlocks) / W : (W == 8 ? 2 : 1)) dynamics_bwd_kernel(DynParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  Smem<W> sm(smem_raw);
  __shared__ float red[5][W];
  const int item = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int C = p.chs;
  const int tile_len = W * 32 * kE;
  const int la = p.lookahead;

  const float M = p.makeup_db[item];
  const CurveK ck = make_curve(CV, p.threshold_db[item], p.ratio[item], p.knee_db[item]);
  const float attack = p.attack_ms[item];
  PoleTables tb;
  make_tables(tb, attack, p.sample_rate, lane);
  // a^(E*(31-lane)): the same construction seen from the other end of the warp
  PoleTables tr;
  make_tables(tr, attack, p.sample_rate, 31 - lane);
  const float rlane_pow = tr.lane_pow;

  TileGeom g{p.n, tile_len, p.ntiles, true};
  const int64_t base = (int64_t)item * C * p.n;
  BwdRows rows{p.x + base, p.gy + base, p.y + base, p.n, C};
  TilePipe<kStages> pipe;
  pipe.init(sm.bars, sm.stages, 2 * C, tile_len, p.bulk != 0);
  pipe.prologue(g, rows);

  float w_tile = 0.f;                                 // adjoint state w[first sample of the next tile]
  float acc_m = 0.f, acc_a = 0.f, acc_t = 0.f, acc_r = 0.f, acc_w = 0.f;
  const int off = threadIdx.x * kE;
  for (int i = 0; i < p.ntiles; ++i) {
    pipe.acquire(i, g, rows);
    const int st = i % kStages;
    const int tile = g.tile_of(i);
    const int64_t n0 = (int64_t)tile * tile_len + off;

    // ---- recompute the forward quantities of this tile from its checkpoint ----
    float xs[kE], s[kE], gcv[kE], dxdbv[kE], drv[kE], dwv[kE];   // gain computer value + partials (d/dT = -d/dxdb)
    float x0[ST ? kE : 1], x1[ST ? kE : 1], g0[ST ? kE : 1], g1[ST ? kE : 1];   // stereo: x and dL/dy stay in registers
    if (ST) {
      const float* xa = pipe.buf(st, 0) + off;
      const float* xb = pipe.buf(st, 1) + off;
      const float* ga = pipe.buf(st, 2) + off;
      const float* gb = pipe.buf(st, 3) + off;
#pragma unroll
      for (int j = 0; j < kE; ++j) {
        x0[ST ? j : 0] = xa[j]; x1[ST ? j : 0] = xb[j]; g0[ST ? j : 0] = ga[j]; g1[ST ? j : 0] = gb[j];
        xs[j] = xa[j] + xb[j];
      }
    } else {
#pragma unroll
      for (int j = 0; j < kE; ++j) xs[j] = 0.f;
      for (int c = 0; c < C; ++c) {
        const float* xb = pipe.buf(st, c) + off;
#pragma unroll
        for (int j = 0; j < kE; ++j) xs[j] += xb[j];
      }
    }
    {
      float run = 0.f;
#pragma unroll
      for (int j = 0; j < kE; ++j) {
        CurveOut o; o.gc = 0.f; o.d_xdb = 0.f; o.d_t = 0.f; o.d_r = 0.f; o.d_w = 0.f;
        if (n0 + j < p.n) o = gain_computer<CV, true>(level_db(xs[j], p.eps), ck);
        gcv[j] = o.gc; dxdbv[j] = o.d_xdb; drv[j] = o.d_r; dwv[j] = o.d_w;
        run = fmaf(tb.alpha, run, tb.beta * o.gc);
        s[j] = run;
      }
    }
    float c_tile = p.ckpt[(int64_t)item * p.ntiles + tile];
    const float c_in = scan_forward<W>(s[kE - 1], c_tile, tb, sm.agg + (i & 1) * 2 * W, lane, warp);
#pragma unroll
    for (int j = 0; j < kE; ++j) s[j] = fmaf(tb.apow[j], c_in, s[j]);

    // ---- dL/ds and the zero-state local pass of the adjoint recurrence ----
    float G[kE], wv[kE];
    {
      float dG[kE];
#pragma unroll
      for (int j = 0; j < kE; ++j) dG[j] = ST ? fmaf(g0[ST ? j : 0], x0[ST ? j : 0], g1[ST ? j : 0] * x1[ST ? j : 0]) : 0.f;
      for (int c = 0; c < (ST ? 0 : C); ++c) {
        const float* xb = pipe.buf(st, c) + off;
        const float* gb = pipe.buf(st, C + c) + off;
        if (!LA) {
#pragma unroll
          for (int j = 0; j < kE; ++j) dG[j] = fmaf(gb[j], xb[j], dG[j]);
        } else {
          const float* xr = rows.src(c);
#pragma unroll
          for (int j = 0; j < kE; ++j) {
            const int64_t m = n0 + j - la;
            if (m >= 0 && n0 + j < p.n) dG[j] = fmaf(gb[j], xr[m], dG[j]);
          }
        }
      }
      float run = 0.f;
#pragma unroll
      for (int j = kE - 1; j >= 0; --j) {
        const bool valid = (n0 + j < p.n);
        G[j] = exp2f((s[j] + M) * kLog2Of10Over20);
        const float ds = valid ? dG[j] * G[j] * kLn10Over20 : 0.f;
        acc_m += ds;
        run = fmaf(tb.alpha, run, ds);
        wv[j] = run;
      }
    }
    const float w_in = scan_reverse<W>(wv[0], w_tile, tb, rlane_pow, sm.agg + (i & 1) * 2 * W + W, lane, warp);

    // ---- parameter-gradient integrands and dL/dx ----
    float dxs[kE];
#pragma unroll
    for (int j = 0; j < kE; ++j) {
      // w[j] = local + a^(E-j) * (w at the first sample of the next thread's chunk)
      const float w = fmaf(tb.apow[kE - 1 - j], w_in, wv[j]);
      const bool valid = (n0 + j < p.n);
      const float s_prev = (j == 0) ? c_in : s[j - 1];
      float dx = 0.f;
      if (valid) {
        acc_a = fmaf(w, s_prev - gcv[j], acc_a);
        const float dgc = tb.beta * w;
        acc_t = fmaf(dgc, -dxdbv[j], acc_t);
        acc_r = fmaf(dgc, drv[j], acc_r);
        acc_w = fmaf(dgc, dwv[j], acc_w);
        if (fabsf(xs[j]) >= p.eps) dx = __fdividef(dgc * dxdbv[j] * kDbGradScale, xs[j]);
      }
      dxs[j] = dx;
    }
    if (ST) {
      float* ga = pipe.buf(st, 2) + off;
      float* gb = pipe.buf(st, 3) + off;
#pragma unroll
      for (int j = 0; j < kE; ++j) { ga[j] = fmaf(g0[ST ? j : 0], G[j], dxs[j]); gb[j] = fmaf(g1[ST ? j : 0], G[j], dxs[j]); }
    } else if (!LA) {
      for (int c = 0; c < C; ++c) {
        float* gb = pipe.buf(st, C + c) + off;
#pragma unroll
        for (int j = 0; j < kE; ++j) gb[j] = fmaf(gb[j], G[j], dxs[j]);
      }
    } else {
      // direct term gy[m+la]*G[m+la] is added by dynamics_lookahead_fixup_kernel from g_scratch
      float* gs = p.g_scratch + (int64_t)item * p.n;
#pragma unroll
      for (int j = 0; j < kE; ++j)
        if (n0 + j < p.n) gs[n0 + j] = G[j];
      for (int c = 0; c < C; ++c) {
        float* gb = pipe.buf(st, C + c) + off;
#pragma unroll
        for (int j = 0; j < kE; ++j) gb[j] = dxs[j];
      }
    }
    pipe.release(i, g, rows);
  }
  pipe.drain();

  // ---- block reduction of the five sums, chain rule to the user parameters ----
  acc_m = warp_sum(acc_m); acc_a = warp_sum(acc_a); acc_t = warp_sum(acc_t);
  acc_r = warp_sum(acc_r); acc_w = warp_sum(acc_w);
  if (lane == 0) {
    red[0][warp] = acc_m; red[1][warp] = acc_a; red[2][warp] = acc_t; red[3][warp] = acc_r; red[4][warp] = acc_w;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float sm_[5];
#pragma unroll
    for (int q = 0; q < 5; ++q) {
      float a = 0.f;
#pragma unroll
      for (int w = 0; w < W; ++w) a += red[q][w];
      sm_[q] = a;
    }
    // d alpha / d attack_ms = alpha * ln9 * 1e3 / (sr * attack_ms^2)
    const double dalpha = (double)tb.alpha * 2.1972245773362196 * 1e3 / ((double)p.sample_rate * (double)attack * (double)attack);
    float* gp = p.gparams + (int64_t)item * 6;
    gp[0] = sm_[2];
    gp[1] = sm_[3];
    gp[2] = (float)((double)sm_[1] * dalpha);
    gp[3] = 0.f;                       // release_ms is unused by the reference (functional.py:343-344)
    gp[4] = sm_[4];
    gp[5] = sm_[0];
  }
}

// lookahead > 0 only: gx[b,c,m] += gy[b,c,m+la] * G[b,m+la]
__global__ void dynamics_lookahead_fixup_kernel(const float* __restrict__ gy, const float* __restrict__ G,
                                                float* __restrict__ gx, int64_t n, int chs, int la, int64_t total) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int64_t m = idx % n;
  const int64_t row = idx / n;
  const int64_t item = row / chs;
  if (m + la < n) gx[idx] += gy[idx + la] * G[item * n + m + la];
}

// ---- host side -----------------------------------------------------------------------------
// shared memory a CTA of w warps may ask for: 96 KB (two or more CTAs per SM) up to 8 warps, 200 KB for the one-CTA-per-SM
// geometry W = 16
constexpr size_t kSmemLimit = 96 * 1024, kSmemLimit16 = 200 * 1024;
int pick_warps(int64_t bs, int chs, int nbuf_per_ch) {
  // enough warps to fill the chip, limited by shared memory (S stages * nbuf * tile bytes)
  const int64_t want = 16ll * sm_count();
  int w = 1;
  while (w < 8 && bs * w < want) w *= 2;
  // small batches (at most one item per SM: e.g. 1024 items split over 8 GPUs): one 16-warp CTA per item, so that an SM
  // still runs 16 warps; the item's tiles are walked serially, and a 16-warp tile halves their number
  if (w == 8 && bs <= sm_count()) w = 16;
  { const int f = debug_forced_warps(); if (f == 1 || f == 2 || f == 4 || f == 8 || f == 16) w = f; }
  auto fits = [&](int ww) {
    return (size_t)kStages * nbuf_per_ch * chs * (ww * 32 * kE) * 4 + kSmemHeader <= (ww == 16 ? kSmemLimit16 : kSmemLimit);
  };
  while (w > 1 && !fits(w)) w /= 2;
  return w;
}

// one-off opt-in to the largest dynamic shared memory any launch of `kernel` may ask for (pick_warps caps it at
// 96 KB / 200 KB), cached per (host thread, device, kernel instantiation: a non-type template parameter) instead of a driver call on every launch
template <auto Kernel>
int ensure_smem_optin() {
  static thread_local int done_dev = -1;
  int dev = 0;
  DASP_CUDA_OK(cudaGetDevice(&dev));
  if (done_dev != dev) {
    DASP_CUDA_OK(cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemLimit16));
    done_dev = dev;
  }
  return DASP_OK;
}
size_t smem_bytes(int w, int nbuf) { return kSmemHeader + (size_t)kStages * nbuf * (w * 32 * kE) * 4; }

template <Curve CV, int W, bool LA, bool ST>
int launch_fwd_la(const DynParams& p, int64_t bs, cudaStream_t st) {
  const size_t smem = smem_bytes(W, p.chs);
  { int rc = ensure_smem_optin<dynamics_fwd_kernel<CV, W, LA, ST>>(); if (rc != DASP_OK) return rc; }
  dynamics_fwd_kernel<CV, W, LA, ST><<<(unsigned)bs, W * 32, smem, st>>>(p);
  DASP_LAUNCH_OK("dynamics_fwd_kernel");
  return DASP_OK;
}
template <Curve CV, int W, bool LA, bool ST>
int launch_bwd_la(const DynParams& p, int64_t bs, cudaStream_t st) {
  const size_t smem = smem_bytes(W, 2 * p.chs);
  { int rc = ensure_smem_optin<dynamics_bwd_kernel<CV, W, LA, ST>>(); if (rc != DASP_OK) return rc; }
  dynamics_bwd_kernel<CV, W, LA, ST><<<(unsigned)bs, W * 32, smem, st>>>(p);
  DASP_LAUNCH_OK("dynamics_bwd_kernel");
  return DASP_OK;
}
template <Curve CV, int W>
int launch_fwd_w(const DynParams& p, int64_t bs, cudaStream_t st) {
  if (p.lookahead > 0) return launch_fwd_la<CV, W, true, false>(p, bs, st);
  return p.chs == 2 ? launch_fwd_la<CV, W, false, true>(p, bs, st) : launch_fwd_la<CV, W, false, false>(p, bs, st);
}
template <Curve CV, int W>
int launch_bwd_w(const DynParams& p, int64_t bs, cudaStream_t st) {
  if (p.lookahead > 0) return launch_bwd_la<CV, W, true, false>(p, bs, st);
  return p.chs == 2 ? launch_bwd_la<CV, W, false, true>(p, bs, st) : launch_bwd_la<CV, W, false, false>(p, bs, st);
}

template <Curve CV>
int dispatch(bool bwd, int w, const DynParams& p, int64_t bs, cudaStream_t st) {
  switch (w) {
    case 1: return bwd ? launch_bwd_w<CV, 1>(p, bs, st) : launch_fwd_w<CV, 1>(p, bs, st);
    case 2: return bwd ? launch_bwd_w<CV, 2>(p, bs, st) : launch_fwd_w<CV, 2>(p, bs, st);
    case 4: return bwd ? launch_bwd_w<CV, 4>(p, bs, st) : launch_fwd_w<CV, 4>(p, bs, st);
    case 16: return bwd ? launch_bwd_w<CV, 16>(p, bs, st) : launch_fwd_w<CV, 16>(p, bs, st);
    default: return bwd ? launch_bwd_w<CV, 8>(p, bs, st) : launch_fwd_w<CV, 8>(p, bs, st);
  }
}

int check_common(const float* x, const float* params5[5], int64_t bs, int64_t chs, int64_t n, int64_t lookahead) {
  if (bs > 0 && n > 0) {
    DASP_REQUIRE(x != nullptr, "dynamics: null x");
    for (int i = 0; i < 5; ++i) DASP_REQUIRE(params5[i] != nullptr, "dynamics: null parameter pointer %d", i);
  }
  DASP_REQUIRE(bs >= 0 && n >= 0 && chs >= 1, "dynamics: bad shape bs=%lld chs=%lld n=%lld", (long long)bs,
               (long long)chs, (long long)n);
  DASP_REQUIRE(chs <= kMaxChs, "dynamics: at most %d channels are supported, got %lld", kMaxChs, (long long)chs);
  DASP_REQUIRE(lookahead >= 0 && lookahead < (1ll << 30), "dynamics: bad lookahead_samples %lld", (long long)lookahead);
  DASP_REQUIRE(bs < (1ll << 31), "dynamics: batch too large");
  return DASP_OK;
}

}  // namespace
}  // namespace dasp

using namespace dasp;

extern "C" {

// samples per tile the forward/backward pair will use for this problem shape (checkpoint pitch)
int64_t dasp_dynamics_tile_len(int64_t bs, int64_t chs) {
  if (chs < 1 || chs > kMaxChs) return 0;
  // the backward holds 2 buffers per channel: pick the geometry that fits both directions
  return (int64_t)pick_warps(bs, (int)chs, 2) * 32 * kE;
}

int dasp_dynamics_fwd(int kind, const float* x, const float* threshold_db, const float* ratio,
                      const float* attack_ms, const float* knee_db, const float* makeup_db, float* y,
                      float* ckpt, int64_t bs, int64_t chs, int64_t n, float sample_rate, float eps,
                      int64_t lookahead, void* stream) {
  const float* ps[5] = {threshold_db, ratio, attack_ms, knee_db, makeup_db};
  int rc = check_common(x, ps, bs, chs, n, lookahead);
  if (rc != DASP_OK) return rc;
  DASP_REQUIRE(kind == 0 || kind == 1, "dynamics: kind must be 0 (compressor) or 1 (expander)");
  if (bs == 0 || n == 0) return DASP_OK;
  DASP_REQUIRE(y != nullptr, "dynamics fwd: null y");
  const int w = pick_warps(bs, (int)chs, 2);
  const int tile_len = w * 32 * kE;
  DynParams p{};
  p.x = x; p.y = y; p.threshold_db = threshold_db; p.ratio = ratio; p.attack_ms = attack_ms;
  p.knee_db = knee_db; p.makeup_db = makeup_db; p.ckpt = ckpt; p.n = n; p.chs = (int)chs;
  p.ntiles = (int)((n + tile_len - 1) / tile_len); p.lookahead = (int)lookahead;
  p.sample_rate = sample_rate; p.eps = eps;
  p.bulk = (n % 4 == 0) && aligned16(x) && aligned16(y);
  return kind == 0 ? dispatch<Curve::Compress>(false, w, p, bs, (cudaStream_t)stream)
                   : dispatch<Curve::Expand>(false, w, p, bs, (cudaStream_t)stream);
}

int dasp_dynamics_bwd(int kind, const float* gy, const float* x, const float* threshold_db, const float* ratio,
                      const float* attack_ms, const float* knee_db, const float* makeup_db, const float* ckpt,
                      float* gx, float* gparams, float* g_scratch, int64_t bs, int64_t chs, int64_t n,
                      float sample_rate, float eps, int64_t lookahead, void* stream) {
  const float* ps[5] = {threshold_db, ratio, attack_ms, knee_db, makeup_db};
  int rc = check_common(x, ps, bs, chs, n, lookahead);
  if (rc != DASP_OK) return rc;
  DASP_REQUIRE(kind == 0 || kind == 1, "dynamics: kind must be 0 (compressor) or 1 (expander)");
  if (bs == 0) return DASP_OK;
  cudaStream_t st = (cudaStream_t)stream;
  DASP_REQUIRE(gparams != nullptr, "dynamics bwd: null gparams");
  if (n == 0) { DASP_CUDA_OK(cudaMemsetAsync(gparams, 0, sizeof(float) * 6 * bs, st)); return DASP_OK; }
  DASP_REQUIRE(gy && gx && ckpt, "dynamics bwd: null pointer");
  DASP_REQUIRE(lookahead == 0 || g_scratch != nullptr, "dynamics bwd: lookahead > 0 needs g_scratch (bs*n floats)");
  const int w = pick_warps(bs, (int)chs, 2);
  const int tile_len = w * 32 * kE;
  DynParams p{};
  p.x = x; p.gy = gy; p.y = gx; p.threshold_db = threshold_db; p.ratio = ratio; p.attack_ms = attack_ms;
  p.knee_db = knee_db; p.makeup_db = makeup_db; p.ckpt = const_cast<float*>(ckpt); p.gparams = gparams;
  p.g_scratch = g_scratch; p.n = n; p.chs = (int)chs;
  p.ntiles = (int)((n + tile_len - 1) / tile_len); p.lookahead = (int)lookahead;
  p.sample_rate = sample_rate; p.eps = eps;
  p.bulk = (n % 4 == 0) && aligned16(x) && aligned16(gy) && aligned16(gx);
  rc = kind == 0 ? dispatch<Curve::Compress>(true, w, p, bs, st) : dispatch<Curve::Expand>(true, w, p, bs, st);
  if (rc != DASP_OK) return rc;
  if (lookahead > 0) {
    const int64_t total = bs * chs * n;
    dynamics_lookahead_fixup_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(gy, g_scratch, gx, n, (int)chs,
                                                                                     (int)lookahead, total);
    DASP_LAUNCH_OK("dynamics_lookahead_fixup_kernel");
  }
  return DASP_OK;
}

}  // extern "C"
