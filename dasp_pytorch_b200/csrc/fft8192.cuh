// 8192-point complex FFT of a 512-thread CTA, entirely in shared memory (planar re / im planes).
//
// Why: cuFFT's single-kernel 8192-point C2C is HBM bound (128 KB of traffic per transform); the reverb
// needs the transform BETWEEN two element-wise stages, so running it inside the producing / consuming
// kernel removes whole passes over a 4.7 MB-per-item buffer (DESIGN.md 4.4).
//
// Decomposition 8192 = 8 * 8 * 8 * 16 (four passes, every thread owns 16 points in each pass):
//     n = 1024 n1 + 128 n2 + 16 n3 + n4          k = k1 + 8 k2 + 64 k3 + 512 k4
//     X[k] = sum_n x[n] w^(n k),  w = exp(s 2 pi i / 8192),  s = +1 (INV, unnormalised) or -1
//   P1  DFT8 over n1 (stride 1024)            * w64 ^(n2 k1)                    in place (buffer G, linear)
//   P2  DFT8 over n2 (stride 128)             * w512^(n3 (k1 + 8 k2))           G -> Y, layout A
//   P3  DFT8 over n3 (stride 16)              * w8192^(n4 (k1 + 8 k2 + 64 k3))  Y (A) -> Y (B)
//   P4  DFT16 over n4 (contiguous)                                              Y (B) -> registers
// Thread t of P4 ends with X[t + 512 k4], k4 = 0..15.
//
// Every thread processes TWO adjacent sub-transforms at once in the two lanes of a packed fp32x2 value
// (Blackwell FADD2/FMUL2/FFMA2 take one issue slot for two flops): with planar storage a 64-bit shared load
// of two neighbouring floats IS the packed operand, so there is no pack/unpack traffic.  P4 uses the lanes for
// the even / odd halves of its 16-point transform and finishes with one scalar radix-2 stage.
//
// Layouts (floats, per plane): linear = n;  A(k1,k2,n3,n4) = 1152 k1 + 144 k2 + 16 n3 + n4;
// B(k1,k2,k3,n4) = 18 (k1 + 8 k2 + 64 k3) + n4.  The paddings (144 = 128 + 16, 18 = 16 + 2) make every
// 64-bit access of every pass bank-conflict free.
//
// The arithmetic is written against a small lane-vector interface so that the SAME code runs in a host
// emulation (tests/test_fft8192_host.py drives tools/probe/fft8192_host_check.cpp: threads looped over
// sequentially, packed lanes emulated) and pins the index mathematics without a GPU.
#pragma once

#ifdef __CUDACC__
#define DASP_HD __host__ __device__ __forceinline__
#else
#define DASP_HD inline
#endif

namespace dasp {
namespace fft8k {

constexpr int kN = 8192;
constexpr int kThreads = 512;
constexpr int kPlaneG = 8192;          // floats per plane of the linear buffer
constexpr int kPlaneY = 9216;          // floats per plane of the padded buffer (layouts A and B)
constexpr int kTabFloats = 2 * (2 * 64) + 2 * (2 * 512) + 2 * 1024 + 2 * 128;   // see Tables

// ---- packed lane pair ------------------------------------------------------------------------------
// On the device the lane pair is one packed fp32x2 register pair (FADD2/FMUL2/FFMA2).  A/B on B200
// (profiles/r02_eq_variants.md): although a micro-benchmark shows FFMA2 with three distinct register pairs at half the
// FMA-pipe throughput of two scalar FFMAs (FADD2 is at parity), the packed FFT kernels are 1-6 % FASTER end to end
// than two scalar instructions per pair (reverb forward 6.11 vs 6.47 ms).  The host emulation keeps two scalars.
//
// Twiddles: the seven twiddles a thread needs in a pass are successive powers of one table entry, formed by complex
// multiplication in registers instead of being fetched one by one -- the FFT kernels are bound by the shared-memory
// pipe (data exchange + twiddle fetches), not by the FMA pipe (profiles/r02_reverb_*.md).
#if defined(__CUDA_ARCH__)
struct V2 { float2 v; };
DASP_HD V2 v2(float a, float b) { V2 r; r.v = make_float2(a, b); return r; }
DASP_HD V2 bc(float a) { return v2(a, a); }
DASP_HD V2 operator+(V2 a, V2 b) { V2 r; r.v = __fadd2_rn(a.v, b.v); return r; }
DASP_HD V2 operator-(V2 a, V2 b) { V2 r; r.v = __ffma2_rn(b.v, make_float2(-1.f, -1.f), a.v); return r; }
DASP_HD V2 operator*(V2 a, V2 b) { V2 r; r.v = __fmul2_rn(a.v, b.v); return r; }
DASP_HD V2 fma2(V2 a, V2 b, V2 c) { V2 r; r.v = __ffma2_rn(a.v, b.v, c.v); return r; }            // a b + c
DASP_HD V2 fnma2(V2 a, V2 b, V2 c) { V2 r; r.v = __ffma2_rn(make_float2(-a.v.x, -a.v.y), b.v, c.v); return r; }   // c - a b
DASP_HD V2 neg(V2 a) { return v2(-a.v.x, -a.v.y); }
DASP_HD float lane0(V2 a) { return a.v.x; }
DASP_HD float lane1(V2 a) { return a.v.y; }
DASP_HD V2 ld2(const float* p) { V2 r; r.v = *reinterpret_cast<const float2*>(p); return r; }
DASP_HD void st2(float* p, V2 a) { *reinterpret_cast<float2*>(p) = a.v; }
#else
struct V2 { float x, y; };
DASP_HD V2 v2(float a, float b) { V2 r; r.x = a; r.y = b; return r; }
DASP_HD V2 bc(float a) { return v2(a, a); }
DASP_HD V2 operator+(V2 a, V2 b) { return v2(a.x + b.x, a.y + b.y); }
DASP_HD V2 operator-(V2 a, V2 b) { return v2(a.x - b.x, a.y - b.y); }
DASP_HD V2 operator*(V2 a, V2 b) { return v2(a.x * b.x, a.y * b.y); }
DASP_HD V2 fma2(V2 a, V2 b, V2 c) { return v2(a.x * b.x + c.x, a.y * b.y + c.y); }
DASP_HD V2 fnma2(V2 a, V2 b, V2 c) { return v2(c.x - a.x * b.x, c.y - a.y * b.y); }
DASP_HD V2 neg(V2 a) { return v2(-a.x, -a.y); }
DASP_HD float lane0(V2 a) { return a.x; }
DASP_HD float lane1(V2 a) { return a.y; }
DASP_HD V2 ld2(const float* p) { return v2(p[0], p[1]); }
DASP_HD void st2(float* p, V2 a) { p[0] = a.x; p[1] = a.y; }
#endif

// ---- twiddle tables (shared memory on the device) --------------------------------------------------
// All entries are exp(+2 pi i turns) (the forward transform conjugates).
// w64b / w512b: cos and sin DUPLICATED into both lanes (one 64-bit load = broadcast operand);
// w8k: exp(s 2 pi i m / 8192) for m < 1024, planar; w128: exp(s 2 pi i m / 128), planar.
struct Tables {
  const float* w64b_c;  const float* w64b_s;     // [64][2]
  const float* w512b_c; const float* w512b_s;    // [512][2]
  const float* w8k_c;   const float* w8k_s;      // [1024]
  const float* w128_c;  const float* w128_s;     // [128]
};
DASP_HD Tables carve_tables(float* base) {
  Tables t;
  t.w64b_c = base;            t.w64b_s = base + 128;
  t.w512b_c = base + 256;     t.w512b_s = base + 256 + 1024;
  t.w8k_c = base + 2304;      t.w8k_s = base + 2304 + 1024;
  t.w128_c = base + 4352;     t.w128_s = base + 4352 + 128;
  return t;
}
// entry `e` (0 <= e < 64 + 512 + 1024 + 128) of the table set: where it goes and which angle (in turns) it holds
DASP_HD void table_entry(int e, int& c_off, int& s_off, int& dup, double& turns) {
  if (e < 64)        { c_off = 2 * e;            s_off = 128 + 2 * e;          dup = 1; turns = e / 64.0; }
  else if (e < 576)  { const int m = e - 64;  c_off = 256 + 2 * m;  s_off = 1280 + 2 * m;  dup = 1; turns = m / 512.0; }
  else if (e < 1600) { const int m = e - 576; c_off = 2304 + m;     s_off = 3328 + m;      dup = 0; turns = m / 8192.0; }
  else               { const int m = e - 1600; c_off = 4352 + m;    s_off = 4480 + m;      dup = 0; turns = m / 128.0; }
}
constexpr int kTabEntries = 64 + 512 + 1024 + 128;

// ---- packed 8-point DFT, natural order in and out --------------------------------------------------
// s = +1: X[k] = sum_j x[j] e^{+2 pi i j k / 8};  s = -1: the conjugate kernel
template <bool INV>
DASP_HD void mul_i(V2& r, V2& i) {            // (r + i i) * (s i)
  const V2 t = r;
  if (INV) { r = neg(i); i = t; } else { r = i; i = neg(t); }
}
template <bool INV>
DASP_HD void dft8(V2 (&r)[8], V2 (&i)[8]) {
  const V2 h = bc(0.70710678118654752f);
  V2 ar[4], ai[4], br[4], bi[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    ar[j] = r[j] + r[j + 4]; ai[j] = i[j] + i[j + 4];
    br[j] = r[j] - r[j + 4]; bi[j] = i[j] - i[j + 4];
  }
  // b_j *= W8^j :  W8 = (1 + s i)/sqrt2,  W8^2 = s i,  W8^3 = (-1 + s i)/sqrt2
  {
    const V2 x = br[1], y = bi[1];
    if (INV) { br[1] = (x - y) * h; bi[1] = (x + y) * h; } else { br[1] = (x + y) * h; bi[1] = (y - x) * h; }
  }
  mul_i<INV>(br[2], bi[2]);
  {
    const V2 x = br[3], y = bi[3];
    if (INV) { br[3] = neg(x + y) * h; bi[3] = (x - y) * h; } else { br[3] = (y - x) * h; bi[3] = neg(x + y) * h; }
  }
  // 4-point DFTs: even outputs from a, odd outputs from b
  auto dft4 = [&](V2 (&pr)[4], V2 (&pi)[4], int o) {
    const V2 c0r = pr[0] + pr[2], c0i = pi[0] + pi[2], c1r = pr[1] + pr[3], c1i = pi[1] + pi[3];
    const V2 d0r = pr[0] - pr[2], d0i = pi[0] - pi[2];
    V2 d1r = pr[1] - pr[3], d1i = pi[1] - pi[3];
    mul_i<INV>(d1r, d1i);
    r[o + 0] = c0r + c1r; i[o + 0] = c0i + c1i;
    r[o + 4] = c0r - c1r; i[o + 4] = c0i - c1i;
    r[o + 2] = d0r + d1r; i[o + 2] = d0i + d1i;
    r[o + 6] = d0r - d1r; i[o + 6] = d0i - d1i;
  };
  dft4(ar, ai, 0);
  dft4(br, bi, 1);
}

// (r + i i) *= (wr + s i wi): the tables hold positive angles, the forward transform multiplies by the conjugate
template <bool INV>
DASP_HD void cmul(V2& r, V2& i, V2 wr, V2 wi) {
  if (INV) {
    const V2 t = fnma2(i, wi, r * wr);
    i = fma2(r, wi, i * wr);
    r = t;
  } else {
    const V2 t = fma2(i, wi, r * wr);
    i = fnma2(r, wi, i * wr);
    r = t;
  }
}

// ---- the four passes.  `t` = thread index in [0, 512).  Barriers are the caller's job:
//   p1; SYNC; p2; SYNC; p3_load; SYNC; p3_store; SYNC; p4
template <bool INV>
DASP_HD void p1(float* gr, float* gi, const Tables& tb, int t) {
  const int m = 2 * t, n2 = m >> 7;
  V2 r[8], i[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { r[j] = ld2(gr + 1024 * j + m); i[j] = ld2(gi + 1024 * j + m); }
  dft8<INV>(r, i);
  {  // w64^(n2 k1) = (w64^n2)^k1: one table entry, six complex multiplies instead of six more (pairs of) loads
    const V2 w1r = ld2(tb.w64b_c + 2 * n2), w1i = ld2(tb.w64b_s + 2 * n2);
    V2 wr = w1r, wi = w1i;
#pragma unroll
    for (int k1 = 1; k1 < 8; ++k1) {
      cmul<INV>(r[k1], i[k1], wr, wi);
      if (k1 < 7) cmul<true>(wr, wi, w1r, w1i);
    }
  }
#pragma unroll
  for (int k1 = 0; k1 < 8; ++k1) { st2(gr + 1024 * k1 + m, r[k1]); st2(gi + 1024 * k1 + m, i[k1]); }
}

template <bool INV>
DASP_HD void p2(const float* gr, const float* gi, float* yr, float* yi, const Tables& tb, int t) {
  const int k1 = t >> 6, n3 = (t >> 3) & 7, j = t & 7;
  const int src = 1024 * k1 + 16 * n3 + 2 * j, dst = 1152 * k1 + 16 * n3 + 2 * j;
  V2 r[8], i[8];
#pragma unroll
  for (int n2 = 0; n2 < 8; ++n2) { r[n2] = ld2(gr + src + 128 * n2); i[n2] = ld2(gi + src + 128 * n2); }
  dft8<INV>(r, i);
  // w512^(n3 (k1 + 8 k2)) = w512^(n3 k1) * (w64^n3)^k2: two table entries and seven complex multiplies
  V2 wr = ld2(tb.w512b_c + 2 * (n3 * k1)), wi = ld2(tb.w512b_s + 2 * (n3 * k1));
  const V2 sr = ld2(tb.w64b_c + 2 * n3), si = ld2(tb.w64b_s + 2 * n3);
#pragma unroll
  for (int k2 = 0; k2 < 8; ++k2) {
    cmul<INV>(r[k2], i[k2], wr, wi);
    st2(yr + dst + 144 * k2, r[k2]); st2(yi + dst + 144 * k2, i[k2]);
    if (k2 < 7) cmul<true>(wr, wi, sr, si);
  }
}

struct P3Regs { V2 r[8], i[8]; };

template <bool INV>
DASP_HD void p3_load(const float* yr, const float* yi, int t, P3Regs& q) {
  const int k1 = t >> 6, k2 = (t >> 3) & 7, j = t & 7;
  const int src = 1152 * k1 + 144 * k2 + 2 * j;
#pragma unroll
  for (int n3 = 0; n3 < 8; ++n3) { q.r[n3] = ld2(yr + src + 16 * n3); q.i[n3] = ld2(yi + src + 16 * n3); }
}
template <bool INV>
DASP_HD void p3_store(float* yr, float* yi, const Tables& tb, int t, P3Regs& q) {
  const int k1 = t >> 6, k2 = (t >> 3) & 7, j = t & 7;
  dft8<INV>(q.r, q.i);
  const int qq = k1 + 8 * k2, n4a = 2 * j, n4b = 2 * j + 1;
  const V2 bwr = v2(tb.w8k_c[n4a * qq], tb.w8k_c[n4b * qq]), bwi = v2(tb.w8k_s[n4a * qq], tb.w8k_s[n4b * qq]);
  // w8192^(n4 (qq + 64 k3)) = w8192^(n4 qq) * (w128^n4)^k3: no more multiplies than a per-k3 table lookup needs,
  // 24 fewer scalar loads
  const V2 sr = v2(tb.w128_c[n4a], tb.w128_c[n4b]), si = v2(tb.w128_s[n4a], tb.w128_s[n4b]);
  V2 wr = bwr, wi = bwi;
#pragma unroll
  for (int k3 = 0; k3 < 8; ++k3) {
    cmul<INV>(q.r[k3], q.i[k3], wr, wi);
    const int dst = 18 * (qq + 64 * k3) + 2 * j;
    st2(yr + dst, q.r[k3]); st2(yi + dst, q.i[k3]);
    if (k3 < 7) cmul<true>(wr, wi, sr, si);
  }
}

// out_r[k4], out_i[k4] = X[t + 512 k4]
template <bool INV>
DASP_HD void p4(const float* yr, const float* yi, int t, float (&out_r)[16], float (&out_i)[16]) {
  V2 r[8], i[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { r[j] = ld2(yr + 18 * t + 2 * j); i[j] = ld2(yi + 18 * t + 2 * j); }
  dft8<INV>(r, i);      // lane 0: DFT8 of the even samples (E), lane 1: of the odd samples (O)
  // X[k] = E[k] + W16^k O[k],  X[k + 8] = E[k] - W16^k O[k],  W16 = exp(s 2 pi i / 16)
  constexpr float c16[8] = {1.0f, 0.92387953251128674f, 0.70710678118654752f, 0.38268343236508977f,
                            0.0f, -0.38268343236508977f, -0.70710678118654752f, -0.92387953251128674f};
  constexpr float s16[8] = {0.0f, 0.38268343236508977f, 0.70710678118654752f, 0.92387953251128674f,
                            1.0f, 0.92387953251128674f, 0.70710678118654752f, 0.38268343236508977f};
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float er = lane0(r[k]), ei = lane0(i[k]), orr = lane1(r[k]), oi = lane1(i[k]);
    const float wr = c16[k], wi = INV ? s16[k] : -s16[k];
    const float pr = orr * wr - oi * wi, pi = orr * wi + oi * wr;
    out_r[k] = er + pr; out_i[k] = ei + pi;
    out_r[k + 8] = er - pr; out_i[k + 8] = ei - pi;
  }
}

}  // namespace fft8k
}  // namespace dasp
