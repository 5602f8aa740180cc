// parametric_eq forward + backward: six cascaded biquads as time-parallel linear recurrences
// (reference: dasp_pytorch/functional.py:118-272, signal.py:242-306 design, :136-166 filtering).
//
// The reference never runs a recursion: it samples H = prod B_k/A_k on a 2^17-point FFT grid
// and multiplies spectra (signal.py:7-39).  That equals the zero-state IIR whenever the cascade's
// impulse response has died out inside n_fft - N samples (DESIGN.md "FSM vs recursion"), and it
// is what this file computes directly, in one pass over HBM.
//
// Realisation ("sigma form").  Direct forms are unusable in fp32 for the 20 Hz..2 kHz sections
// (a1 ~ -2, a2 ~ 1: the information sits in 1+a1+a2 ~ 1e-5).  Each section is instead run as
//       s1' = sg*s1 +    s2 + be1*u          sg  = -a1/2          be1 = b1 - a1*b0
//       s2' = q *s1 + sg*s2 + B2 *u          q   = sg^2 - a2      B2  = (b2 - a2*b0) + sg*be1
//       y   = s1 + b0*u
// whose state matrix [[sg,1],[q,sg]] has equal diagonal entries, i.e. is diagonally similar to a
// NORMAL matrix (rotation-scaling for complex poles, symmetric for real poles): round-off is
// amplified by 1/(1-r), not 1/((1-r) w0^2), and the small quantity q = -(r sin w0)^2 is stored
// directly instead of as a difference of O(1) numbers.  6 FMA per sample per section, all fp32;
// measured against the fp64 reference this is 100-1000x more accurate than the reference's own
// fp32 path (DESIGN.md, numerics table).  Coefficients and all matrix powers are designed in fp64.
//
// Parallelisation (round 2: "row pairs on FFMA2, warps decoupled along time").
//   * Two rows (the left/right channel of an item when C = 2; any two consecutive rows otherwise) are the two
//     lanes of Blackwell's packed fp32x2 instructions (FFMA2 / FMUL2 / FADD2): one issue slot, two FMAs.  The
//     kernels are instruction-issue bound (about 100 fp32 instructions per sample in the scalar round-1 form,
//     at the fp32 ridge of the chip), so this halves the cost per sample.  All tables hold (row A, row B) pairs.
//   * One CTA per row pair, W warps.  The row is cut into tiles of 32*E samples; warp w owns tiles w, w+W, ...
//     and runs the WHOLE cascade on a tile with the data in registers: per section a zero-state local pass over
//     the lane's E samples, a Kogge-Stone shuffle scan of the lanes' end states with the precomputed powers
//     A^(E 2^k) (A is constant in time, so the scan operator is a matrix power, not a generic 2x2 product), and a
//     fix-up  y[j] += (A^j c_in)_1  from a per-pair table.
//   * The only coupling between consecutive tiles of a row is the 2-vector carry of each section,
//     c(i+1) = A^(32E) c(i) + total(i).  It travels from the warp of tile i to the warp of tile i+1 through a
//     16-byte shared-memory mailbox guarded by an mbarrier (arrive = release, try_wait = acquire): no block
//     barrier anywhere in the main loop, the W warps drift freely and hide each other's scan/shuffle latency.
//     (The round-1 kernels synchronised the whole CTA once per section per tile and were latency bound.)
//   * Every warp streams its own tiles HBM -> shared memory -> HBM with 1-D TMA bulk copies (UBLKCP) and its own
//     mbarriers/bulk groups, double buffered; the hot loop contains no LDG/STG for audio.
// The forward stores the section states entering every tile (24 floats per tile per pair) as checkpoints.
//
// Backward.  State-space adjoint (SURVEY.md A.3 restated for the sigma form): with lam = adjoint
// state,  lam[n] = A^T lam[n+1] + (g[n],0);  gu[n] = be1*lam1[n+1] + B2*lam2[n+1] + b0*g[n];
//   d sg = sum lam[n+1].s[n],  d q = sum lam2[n+1] s1[n],  d be1 = sum lam1[n+1] u[n],
//   d B2 = sum lam2[n+1] u[n], d b0 = sum g[n] u[n].
// Tiles are swept in reverse time order with the same warp/mailbox structure (the adjoint carry flows from tile
// i+1 to tile i); per tile the six section inputs are recomputed from the checkpoint into per-warp shared memory
// (no cross-tile dependency: every tile's incoming states are checkpointed), then sections are unwound 6 -> 1.
// The 30 sums per row are reduced deterministically; a second tiny kernel adds the channels of an item and applies
// the fp64 Jacobian d(sg,q,be1,B2,b0)/d(gain_dB, fc, Q) (forward-mode dual numbers).
#include <math.h>

#include "common.cuh"

namespace dasp {
namespace {

constexpr int kE = 15;           // samples per lane per tile (odd: conflict-free stride-E shared-memory access)
static_assert(kE % 2 == 1, "E must be odd");
constexpr int kTile = 32 * kE;   // samples per tile (one warp)
constexpr int kSections = 6;
constexpr size_t kSmemPerSm = 227 * 1024;     // usable shared memory of one SM / one CTA

// ------------------------------------------------------------------ coefficient design (fp64)
// forward-mode dual number with 3 directional derivatives (gain_dB, fc, Q)
struct Dual3 {
  double v, d[3];
};
__host__ __device__ inline Dual3 mk(double v) { return {v, {0, 0, 0}}; }
__host__ __device__ inline Dual3 operator+(Dual3 a, Dual3 b) { return {a.v + b.v, {a.d[0] + b.d[0], a.d[1] + b.d[1], a.d[2] + b.d[2]}}; }
__host__ __device__ inline Dual3 operator-(Dual3 a, Dual3 b) { return {a.v - b.v, {a.d[0] - b.d[0], a.d[1] - b.d[1], a.d[2] - b.d[2]}}; }
__host__ __device__ inline Dual3 operator-(Dual3 a) { return {-a.v, {-a.d[0], -a.d[1], -a.d[2]}}; }
__host__ __device__ inline Dual3 operator*(Dual3 a, Dual3 b) {
  return {a.v * b.v, {a.d[0] * b.v + a.v * b.d[0], a.d[1] * b.v + a.v * b.d[1], a.d[2] * b.v + a.v * b.d[2]}};
}
__host__ __device__ inline Dual3 operator/(Dual3 a, Dual3 b) {
  const double inv = 1.0 / b.v, r = a.v * inv;
  return {r, {(a.d[0] - r * b.d[0]) * inv, (a.d[1] - r * b.d[1]) * inv, (a.d[2] - r * b.d[2]) * inv}};
}
__host__ __device__ inline Dual3 operator*(double s, Dual3 a) { return {s * a.v, {s * a.d[0], s * a.d[1], s * a.d[2]}}; }
__host__ __device__ inline Dual3 operator+(double s, Dual3 a) { return {s + a.v, {a.d[0], a.d[1], a.d[2]}}; }
__host__ __device__ inline Dual3 operator-(double s, Dual3 a) { return {s - a.v, {-a.d[0], -a.d[1], -a.d[2]}}; }
__host__ __device__ inline Dual3 chain(Dual3 a, double f, double df) { return {f, {df * a.d[0], df * a.d[1], df * a.d[2]}}; }
__host__ __device__ inline Dual3 dsin(Dual3 a) { return chain(a, sin(a.v), cos(a.v)); }
__host__ __device__ inline Dual3 dcos(Dual3 a) { return chain(a, cos(a.v), -sin(a.v)); }
__host__ __device__ inline Dual3 dexp(Dual3 a) { double e = exp(a.v); return chain(a, e, e); }
__host__ __device__ inline Dual3 dsqrt(Dual3 a) { double s = sqrt(a.v); return chain(a, s, 0.5 / s); }

struct SigmaCoef {   // [sg, q, be1, B2, b0]
  Dual3 c[5];
};

// RBJ cookbook biquad (signal.py:242-306) -> sigma-form coefficients, with derivatives.
// kind: 0 = low shelf (:268-274), 1 = peaking (:275-281), 2 = high shelf (:261-267).
__host__ __device__ inline SigmaCoef design_section(double gain_db, double fc, double qf, double sr, int kind) {
  Dual3 g = {gain_db, {1, 0, 0}}, f = {fc, {0, 1, 0}}, Q = {qf, {0, 0, 1}};
  Dual3 A = dexp((0.05756462732485114 /* ln10/40 */) * g);
  Dual3 w0 = (6.283185307179586 / sr) * f;
  Dual3 alpha = dsin(w0) / (2.0 * Q);
  Dual3 cw = dcos(w0);
  Dual3 b0, b1, b2, a0, a1, a2;
  if (kind == 1) {
    b0 = 1.0 + alpha * A; b1 = -2.0 * cw; b2 = 1.0 - alpha * A;
    a0 = 1.0 + alpha / A; a1 = -2.0 * cw; a2 = 1.0 - alpha / A;
  } else {
    const double sgn = (kind == 0) ? 1.0 : -1.0;     // the shelves differ in the sign of the cos terms
    Dual3 s = 2.0 * dsqrt(A) * alpha;
    Dual3 ap1 = 1.0 + A, am1 = A - mk(1.0);
    Dual3 t = sgn * (am1 * cw);
    b0 = A * (ap1 - t + s);
    b1 = (sgn * 2.0) * (A * (am1 - sgn * (ap1 * cw)));
    b2 = A * (ap1 - t - s);
    a0 = ap1 + t + s;
    a1 = (-sgn * 2.0) * (am1 + sgn * (ap1 * cw));
    a2 = ap1 + t - s;
  }
  b0 = b0 / a0; b1 = b1 / a0; b2 = b2 / a0; a1 = a1 / a0; a2 = a2 / a0;
  SigmaCoef o;
  Dual3 sg = -0.5 * a1;
  Dual3 be1 = b1 - a1 * b0;
  o.c[0] = sg;
  o.c[1] = sg * sg - a2;
  o.c[2] = be1;
  o.c[3] = (b2 - a2 * b0) + sg * be1;
  o.c[4] = b0;
  return o;
}
__host__ __device__ inline int section_kind(int k) { return k == 0 ? 0 : (k == 5 ? 2 : 1); }

// 2x2 fp64 matrix power of [[sg,1],[q,sg]] by binary exponentiation
struct M2d { double a, b, c, d; };
__device__ inline M2d mm(const M2d& x, const M2d& y) {
  return {x.a * y.a + x.b * y.c, x.a * y.b + x.b * y.d, x.c * y.a + x.d * y.c, x.c * y.b + x.d * y.d};
}
__device__ inline M2d mpow(double sg, double q, unsigned n) {
  M2d r = {1, 0, 0, 1}, b = {sg, 1.0, q, sg};
  while (n) {
    if (n & 1u) r = mm(r, b);
    b = mm(b, b);
    n >>= 1;
  }
  return r;
}

// ------------------------------------------------------------------ arithmetic on row pairs (x = row A, y = row B)
// Blackwell's packed FFMA2/FMUL2/FADD2 where both operands are row pairs.  Measured on B200
// (profiles/r02_ffma2_probe.md, profiles/r02_eq_variants.md): in a micro-benchmark an FFMA2 with three distinct
// register-pair operands occupies the FMA pipe ~4.3 cycles per warp (two scalar FFMAs: ~2.4), but inside these kernels
// the packed form still wins over two scalar instructions per pair (forward 0.39 vs 0.45 ms): operand reuse between
// neighbouring instructions is high and the halved issue count matters more.
typedef float2 f2;
__device__ __forceinline__ f2 ffma2(f2 a, f2 b, f2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ f2 fmul2(f2 a, f2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ f2 zero2() { return make_float2(0.f, 0.f); }
__device__ __forceinline__ f2 shfl_up2(f2 v, int d) {
  return make_float2(__shfl_up_sync(0xffffffffu, v.x, d), __shfl_up_sync(0xffffffffu, v.y, d));
}
__device__ __forceinline__ f2 shfl_down2(f2 v, int d) {
  return make_float2(__shfl_down_sync(0xffffffffu, v.x, d), __shfl_down_sync(0xffffffffu, v.y, d));
}
__device__ __forceinline__ f2 shfl2(f2 v, int l) {
  return make_float2(__shfl_sync(0xffffffffu, v.x, l), __shfl_sync(0xffffffffu, v.y, l));
}

// Coefficient type C of the per-pair tables:
//   float : both rows of the pair belong to the SAME item (every pair when the channel count is even -- stereo), so
//           one scalar coefficient serves both rows: half the table bytes, a whole 2x2 matrix per 128-bit load, and
//           the coefficient register is shared by the two scalar FMAs of the pair.  The first packed version of these
//           kernels ran with the shared-memory / shuffle pipe 68 % busy (ncu: l1tex__data_pipe_lsu_wavefronts, 762
//           wavefronts per tile, most of them broadcast 128-bit table loads); this halves that traffic.
//   f2    : the rows belong to different items (odd channel counts): (row A, row B) coefficient pairs, packed FFMA2.
__device__ __forceinline__ f2 cfma(float c, f2 v, f2 a) { return make_float2(fmaf(c, v.x, a.x), fmaf(c, v.y, a.y)); }
__device__ __forceinline__ f2 cfma(f2 c, f2 v, f2 a) { return ffma2(c, v, a); }
__device__ __forceinline__ f2 dup(float c) { return make_float2(c, c); }
__device__ __forceinline__ f2 dup(f2 c) { return c; }

struct St { f2 s1, s2; };                     // the 2-state vector of both rows
template <class C> struct M4 { C a, b, c, d; };   // 2x2 matrix [[a,b],[c,d]]
__device__ __forceinline__ M4<float> ldm(const float* p) {
  const float4 t = *reinterpret_cast<const float4*>(p);
  return {t.x, t.y, t.z, t.w};
}
__device__ __forceinline__ M4<f2> ldm(const f2* p) {
  const float4 lo = *reinterpret_cast<const float4*>(p), hi = *reinterpret_cast<const float4*>(p + 2);
  return {make_float2(lo.x, lo.y), make_float2(lo.z, lo.w), make_float2(hi.x, hi.y), make_float2(hi.z, hi.w)};
}
template <class C>
__device__ __forceinline__ St mv_acc(const M4<C>& m, const St& v, const St& acc) {     // acc + M v
  return {cfma(m.a, v.s1, cfma(m.b, v.s2, acc.s1)), cfma(m.c, v.s1, cfma(m.d, v.s2, acc.s2))};
}
template <class C>
__device__ __forceinline__ St mtv_acc(const M4<C>& m, const St& v, const St& acc) {    // acc + M^T v
  return {cfma(m.a, v.s1, cfma(m.c, v.s2, acc.s1)), cfma(m.b, v.s1, cfma(m.d, v.s2, acc.s2))};
}

// ------------------------------------------------------------------ shared-memory tables of one row pair
constexpr int kStepSlots = 6;     // A^(E 2^s), s = 0..4, and the zero matrix (lanes a scan step does not touch)
template <class C>
struct __align__(16) Tables {
  C cf[kSections][8];                     // sg, q, be1, B2, b0, pad x3
  C fix[kSections][kE][2];                // first row of A^j: (a_j, b_j)
  C step[kSections][kStepSlots][4];       // (a, b, c, d)
  C lane[kSections][32][4];               // A^(E l)
  C warp[kSections][4];                   // A^(32 E)
};
constexpr int kPowPerSection = kE + 5 + 32 + 1;

struct EqParams {
  const float* x;        // (rows, N)
  const float* gy;       // backward
  float* y;              // forward out / backward gx
  const float* params;   // (bs, 18): gain_dB, fc, Q per section, signature order
  float* ckpt;           // (pairs, ntiles, 6) float4: section states (s1A, s1B, s2A, s2B) entering each tile
  float* partial;        // (rows, 30) backward: per-row coefficient-gradient sums
  int64_t n;
  int64_t rows;
  int chs;
  int ntiles;
  float sample_rate;
  int bulk;
};

// component h of coefficient slot `dst` (a scalar table has one component, a pair table two)
__device__ __forceinline__ void put_coef(float& dst, int, float v) { dst = v; }
__device__ __forceinline__ void put_coef(f2& dst, int h, float v) { if (h == 0) dst.x = v; else dst.y = v; }
template <class C> struct Halves { static constexpr int n = 1; };
template <> struct Halves<f2> { static constexpr int n = 2; };

// build the tables of the pair (row A of item ia, row B of item ib; ia == ib for C = float): every thread of the CTA
// participates; ends with __syncthreads()
template <class C>
__device__ void build_tables(Tables<C>& tb, const float* params, int64_t ia, int64_t ib, float sample_rate) {
  __shared__ double cfd[2][kSections][2];   // sg, q in fp64 for the matrix powers
  const int tid = threadIdx.x, nthr = blockDim.x;
  constexpr int halves = Halves<C>::n;
  for (int e = tid; e < halves * kSections; e += nthr) {
    const int h = e / kSections, k = e - h * kSections;
    const float* p18 = params + (h == 0 ? ia : ib) * 18;
    const SigmaCoef sc = design_section((double)p18[3 * k], (double)p18[3 * k + 1], (double)p18[3 * k + 2],
                                        (double)sample_rate, section_kind(k));
#pragma unroll
    for (int j = 0; j < 5; ++j) put_coef(tb.cf[k][j], h, (float)sc.c[j].v);
#pragma unroll
    for (int j = 5; j < 8; ++j) put_coef(tb.cf[k][j], h, 0.f);
    cfd[h][k][0] = sc.c[0].v;
    cfd[h][k][1] = sc.c[1].v;
  }
  __syncthreads();
  for (int idx = tid; idx < halves * kSections * kPowPerSection; idx += nthr) {
    const int h = idx / (kSections * kPowPerSection);
    const int r = idx - h * (kSections * kPowPerSection);
    const int k = r / kPowPerSection, e = r - k * kPowPerSection;
    unsigned n;
    if (e < kE) n = (unsigned)e;
    else if (e < kE + 5) n = (unsigned)kE << (e - kE);
    else if (e < kE + 5 + 32) n = (unsigned)(kE * (e - kE - 5));
    else n = (unsigned)(kE * 32);
    const M2d m = mpow(cfd[h][k][0], cfd[h][k][1], n);
    const float ma = (float)m.a, mb = (float)m.b, mc = (float)m.c, md = (float)m.d;
    if (e < kE) {
      put_coef(tb.fix[k][e][0], h, ma);
      put_coef(tb.fix[k][e][1], h, mb);
    } else {
      C* f;
      if (e < kE + 5) f = &tb.step[k][e - kE][0];
      else if (e < kE + 5 + 32) f = &tb.lane[k][e - kE - 5][0];
      else f = &tb.warp[k][0];
      put_coef(f[0], h, ma); put_coef(f[1], h, mb); put_coef(f[2], h, mc); put_coef(f[3], h, md);
    }
  }
  for (int e = tid; e < halves * kSections * 4; e += nthr) {
    const int h = e / (kSections * 4), r = e - h * (kSections * 4);
    put_coef(tb.step[r / 4][5][r % 4], h, 0.f);
  }
  __syncthreads();
}

// the five section coefficients, expanded to row pairs for the (packed) local passes
struct Cf { f2 sg, q, be1, B2, b0; };
__device__ __forceinline__ Cf load_cf(const Tables<float>& tb, int k) {
  const float4 a = *reinterpret_cast<const float4*>(&tb.cf[k][0]);
  return {dup(a.x), dup(a.y), dup(a.z), dup(a.w), dup(tb.cf[k][4])};
}
__device__ __forceinline__ Cf load_cf(const Tables<f2>& tb, int k) {
  const float4 a = *reinterpret_cast<const float4*>(&tb.cf[k][0]);
  const float4 b = *reinterpret_cast<const float4*>(&tb.cf[k][2]);
  return {make_float2(a.x, a.y), make_float2(a.z, a.w), make_float2(b.x, b.y), make_float2(b.z, b.w), tb.cf[k][4]};
}
// fix-up table entry j of section k: (a_j, b_j)
__device__ __forceinline__ void load_fix(const Tables<float>& tb, int k, int j, float& a, float& b) {
  const float2 t = *reinterpret_cast<const float2*>(&tb.fix[k][j][0]);
  a = t.x; b = t.y;
}
__device__ __forceinline__ void load_fix(const Tables<f2>& tb, int k, int j, f2& a, f2& b) {
  const float4 t = *reinterpret_cast<const float4*>(&tb.fix[k][j][0]);
  a = make_float2(t.x, t.y); b = make_float2(t.z, t.w);
}

// zero-state local pass of section k over the lane's E samples (in place); returns the end state.
// Two dependent packed operations per sample on the (s1, s2) recurrence.
__device__ __forceinline__ St local_pass(f2 (&v)[kE], const Cf& c) {
  f2 s1 = zero2(), s2 = zero2();
#pragma unroll
  for (int j = 0; j < kE; ++j) {
    const f2 u = v[j];
    v[j] = ffma2(c.b0, u, s1);
    const f2 a = ffma2(c.be1, u, s2);
    const f2 b = ffma2(c.q, s1, fmul2(c.B2, u));
    s1 = ffma2(c.sg, s1, a);
    s2 = ffma2(c.sg, s2, b);
  }
  return {s1, s2};
}
// y[j] += (A^j s_in)_1
template <class C>
__device__ __forceinline__ void fix_up(f2 (&v)[kE], const Tables<C>& tb, int k, const St& sin) {
#pragma unroll
  for (int j = 0; j < kE; ++j) {
    C a, b;
    load_fix(tb, k, j, a, b);
    v[j] = cfma(a, sin.s1, cfma(b, sin.s2, v[j]));
  }
}

// ------------------------------------------------------------------ warp scans of the lanes' 2-vectors
// per-lane slot of the step matrices: the real power where the Kogge-Stone step applies to this lane, the zero matrix
// otherwise (so a step is matrix loads + 4 SHFL + 4 FMAs per row without predicates or selects)
struct StepOffsets { int o[5]; };
__device__ __forceinline__ StepOffsets fwd_offsets(int lane) {
  StepOffsets s;
#pragma unroll
  for (int i = 0; i < 5; ++i) s.o[i] = (lane >= (1 << i)) ? i : 5;
  return s;
}
__device__ __forceinline__ StepOffsets rev_offsets(int lane) {
  StepOffsets s;
#pragma unroll
  for (int i = 0; i < 5; ++i) s.o[i] = (lane + (1 << i) < 32) ? i : 5;
  return s;
}

// forward in time.  v: end state of the lane's zero-state local pass.  On return v is the inclusive scan (lane 31
// holds the tile total) and `excl` the contribution of the lower lanes to the state entering this lane's chunk.
template <class C>
__device__ __forceinline__ void scan_fwd(St& v, const Tables<C>& tb, int k, const StepOffsets& so, int lane, St& excl) {
#pragma unroll
  for (int s = 0; s < 5; ++s) {
    const St u = {shfl_up2(v.s1, 1 << s), shfl_up2(v.s2, 1 << s)};
    v = mv_acc(ldm(&tb.step[k][so.o[s]][0]), u, v);
  }
  excl = {shfl_up2(v.s1, 1), shfl_up2(v.s2, 1)};
  if (lane == 0) excl = {zero2(), zero2()};
}
// reverse in time (adjoint): v = adjoint state at the lane's first sample after a zero-terminal local reverse pass;
// on return lane 0 holds the tile total
template <class C>
__device__ __forceinline__ void scan_rev(St& v, const Tables<C>& tb, int k, const StepOffsets& so, int lane, St& excl) {
#pragma unroll
  for (int s = 0; s < 5; ++s) {
    const St u = {shfl_down2(v.s1, 1 << s), shfl_down2(v.s2, 1 << s)};
    v = mtv_acc(ldm(&tb.step[k][so.o[s]][0]), u, v);
  }
  excl = {shfl_down2(v.s1, 1), shfl_down2(v.s2, 1)};
  if (lane == 31) excl = {zero2(), zero2()};
}

// ------------------------------------------------------------------ carry mailboxes between the warps of a CTA
// mailbox (k, w): carry of section k entering the next tile of warp w; written by the warp of the preceding tile.
// Use number u of a mailbox completes phase u of its mbarrier (tile/sequence 0 is pre-arrived with a zero carry).
template <int W>
struct Mail {
  float4* data;     // [kSections][W]
  uint64_t* bar;    // [kSections][W]
  __device__ __forceinline__ void init_all() {       // thread 0, before the CTA-wide barrier
    for (int i = 0; i < kSections * W; ++i) mbar_init(&bar[i], 1);
    fence_barrier_init();
    for (int k = 0; k < kSections; ++k) {
      data[k * W + 0] = make_float4(0.f, 0.f, 0.f, 0.f);
      mbar_arrive(&bar[k * W + 0]);
    }
  }
  __device__ __forceinline__ St take(int k, int w, int use) {
    mbar_wait(&bar[k * W + w], (uint32_t)(use & 1));
    const float4 d = data[k * W + w];
    __syncwarp();                                    // every lane has its copy before the refill may be triggered
    return {make_float2(d.x, d.y), make_float2(d.z, d.w)};
  }
  // called by ONE lane (the one that holds the tile total)
  __device__ __forceinline__ void put(int k, int w, const St& c) {
    data[k * W + w] = make_float4(c.s1.x, c.s1.y, c.s2.x, c.s2.y);
    mbar_arrive(&bar[k * W + w]);
  }
};

// ------------------------------------------------------------------ per-warp tile I/O (TMA bulk copies)
// A "unit" is the pair's two row tiles: [row A: kTile floats][row B: kTile floats].
constexpr int kUnitFloats = 2 * kTile;

struct RowPair {
  int64_t n; int ntiles; bool bulk; bool has_b;
  __device__ __forceinline__ int len_of(int tile) const {
    const int64_t rem = n - (int64_t)tile * kTile;
    return rem < kTile ? (int)rem : kTile;
  }
};

// load tile `tile` of rows (a, b) into `unit`; bulk: lane 0 issues, completion on `bar`; else cooperative + __syncwarp
__device__ __forceinline__ void warp_load(float* unit, const float* a, const float* b, int tile, const RowPair& rp,
                                          uint64_t* bar, int lane) {
  const int64_t pos = (int64_t)tile * kTile;
  const int len = rp.len_of(tile);
  if (rp.bulk) {
    if (lane == 0) {
      mbar_arrive_expect_tx(bar, (uint32_t)len * 8u);
      tma_load_1d(unit, a + pos, (uint32_t)len * 4u, bar);
      tma_load_1d(unit + kTile, b + pos, (uint32_t)len * 4u, bar);
    }
  } else {
    for (int i = lane; i < len; i += 32) { unit[i] = a[pos + i]; unit[kTile + i] = b[pos + i]; }
    __syncwarp();
  }
}
__device__ __forceinline__ void warp_store(const float* unit, float* a, float* b, int tile, const RowPair& rp, int lane) {
  const int64_t pos = (int64_t)tile * kTile;
  const int len = rp.len_of(tile);
  if (rp.bulk) {
    fence_proxy_async_smem();         // my generic-proxy writes -> visible to the TMA engine
    __syncwarp();
    if (lane == 0) {
      tma_store_1d(a + pos, unit, (uint32_t)len * 4u);
      if (rp.has_b) tma_store_1d(b + pos, unit + kTile, (uint32_t)len * 4u);
      tma_store_commit();
    }
  } else {
    __syncwarp();
    for (int i = lane; i < len; i += 32) { a[pos + i] = unit[i]; if (rp.has_b) b[pos + i] = unit[kTile + i]; }
    __syncwarp();
  }
}

// dynamic shared memory carve-up
template <class C, int W, int UNITS_PER_WARP, int BARS_PER_WARP>
struct Smem {
  Tables<C>* tb; float4* mail_data; uint64_t* mail_bar; uint64_t* full; float* units;
  static constexpr size_t kTab = (sizeof(Tables<C>) + 127) / 128 * 128;
  static constexpr size_t kMailData = sizeof(float4) * kSections * W;
  static constexpr size_t kBars = sizeof(uint64_t) * (kSections * W + BARS_PER_WARP * W);
  static constexpr size_t kHdr = (kTab + kMailData + kBars + 127) / 128 * 128;
  static constexpr size_t kBytes = kHdr + sizeof(float) * kUnitFloats * UNITS_PER_WARP * W;
  __device__ __forceinline__ explicit Smem(unsigned char* base) {
    tb = reinterpret_cast<Tables<C>*>(base);
    mail_data = reinterpret_cast<float4*>(base + kTab);
    mail_bar = reinterpret_cast<uint64_t*>(base + kTab + kMailData);
    full = mail_bar + kSections * W;
    units = reinterpret_cast<float*>(base + kHdr);
  }
};

// the two rows of pair `pair`: pairs never straddle items when C = float (pairs per item = ceil(chs / 2), the last
// pair of an item with an odd channel count would repeat its row -- but odd channel counts use C = f2, where pairs
// are simply consecutive rows)
struct PairRows { int64_t row_a, row_b; bool has_b; };
__device__ __forceinline__ PairRows pair_rows(int64_t pair, int64_t rows) {
  PairRows r;
  r.row_a = 2 * pair;
  r.has_b = r.row_a + 1 < rows;
  r.row_b = r.has_b ? r.row_a + 1 : r.row_a;
  return r;
}

// =============================================================================== forward
// per-warp shared memory: two units, double buffered (tile i+W loads while tile i is computed), one barrier each
template <class C, int W>
using FwdSmem = Smem<C, W, 2, 2>;

template <class C, int W>
__global__ void __launch_bounds__(W * 32) eq_fwd_kernel(EqParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  FwdSmem<C, W> sm(smem_raw);
  const Tables<C>& tb = *sm.tb;
  const int lane = threadIdx.x & 31;
  // the warp index, read from lane 0: the compiler then KNOWS it is warp-uniform.  With `threadIdx.x >> 5` the
  // warp-strided tile loop below counts as divergent and every shuffle of the scans is emitted as a five-instruction
  // WARPSYNC.COLLECTIVE / MOV / SHFL / MOV / ENDCOLLECTIVE sequence through two fixed registers (measured on the SASS:
  // 1776 SHFL + 1804 collective brackets + ~2300 extra MOV in eq_bwd_kernel, and no overlap between shuffles).
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const PairRows pr = pair_rows(blockIdx.x, p.rows);

  build_tables(*sm.tb, p.params, pr.row_a / p.chs, pr.row_b / p.chs, p.sample_rate);
  Mail<W> mail{sm.mail_data, sm.mail_bar};
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2 * W; ++i) mbar_init(&sm.full[i], 1);
    mail.init_all();
  }
  __syncthreads();

  const RowPair rp{p.n, p.ntiles, p.bulk != 0, pr.has_b};
  const float* xa = p.x + pr.row_a * p.n;
  const float* xb = p.x + pr.row_b * p.n;
  float* ya = p.y + pr.row_a * p.n;
  float* yb = p.y + pr.row_b * p.n;
  float* my_units = sm.units + (size_t)warp * 2 * kUnitFloats;
  uint64_t* my_full = sm.full + warp * 2;
  const StepOffsets so = fwd_offsets(lane);
  float4* ckpt = p.ckpt ? reinterpret_cast<float4*>(p.ckpt) + (int64_t)blockIdx.x * p.ntiles * kSections : nullptr;

  if (warp < p.ntiles) warp_load(my_units, xa, xb, warp, rp, &my_full[0], lane);
  int jt = 0;
  for (int i = warp; i < p.ntiles; i += W, ++jt) {
    const int st = jt & 1;
    float* unit = my_units + (size_t)st * kUnitFloats;
    if (i + W < p.ntiles) {
      // the other stage was stored from one tile ago: that bulk store must have finished READING it
      if (rp.bulk && lane == 0) tma_store_wait_read<0>();
      warp_load(my_units + (size_t)(st ^ 1) * kUnitFloats, xa, xb, i + W, rp, &my_full[st ^ 1], lane);
    }
    if (rp.bulk) mbar_wait(&my_full[st], (uint32_t)((jt >> 1) & 1));
    const int off = lane * kE;
    const int64_t n0 = (int64_t)i * kTile + off;
    f2 v[kE];
    if ((int64_t)(i + 1) * kTile <= p.n) {           // whole tile inside the row (warp-uniform): no per-sample masks
#pragma unroll
      for (int j = 0; j < kE; ++j) v[j] = make_float2(unit[off + j], unit[kTile + off + j]);
    } else {
#pragma unroll
      for (int j = 0; j < kE; ++j)
        v[j] = (n0 + j < p.n) ? make_float2(unit[off + j], unit[kTile + off + j]) : zero2();
    }

#pragma unroll
    for (int k = 0; k < kSections; ++k) {
      const Cf c = load_cf(tb, k);
      St incl = local_pass(v, c);
      St excl;
      scan_fwd(incl, tb, k, so, lane, excl);
      const St cin = mail.take(k, warp, jt);                      // carry of section k entering this tile
      if (lane == 31 && i + 1 < p.ntiles)                         // lane 31 holds the tile total
        mail.put(k, (warp + 1) % W, mv_acc(ldm(&tb.warp[k][0]), cin, incl));      // A^(32E) c + total
      if (ckpt && lane == 0) ckpt[(int64_t)i * kSections + k] = make_float4(cin.s1.x, cin.s1.y, cin.s2.x, cin.s2.y);
      const St sin = mv_acc(ldm(&tb.lane[k][lane][0]), cin, excl);    // state entering this lane's chunk
      fix_up(v, tb, k, sin);
    }
#pragma unroll
    for (int j = 0; j < kE; ++j) { unit[off + j] = v[j].x; unit[kTile + off + j] = v[j].y; }
    warp_store(unit, ya, yb, i, rp, lane);
  }
  if (rp.bulk && lane == 0) tma_store_wait_all<0>();
}

// =============================================================================== backward
// Warps per row pair.  The backward holds 255 registers per thread, i.e. 8 warps per SM whatever the split: W=8 with
// one load stage (one CTA per SM, least shared memory per warp) measured best on B200 (profiles/r02_eq_variants.md).
constexpr int kBwdWarps = 8;
// per-warp shared memory: the x and dL/dy units (row-pair units, TMA, one barrier) and U1..U4 (interleaved f2, the
// inputs of sections 1..4); the input of section 5 overwrites the dL/dy unit once dL/dy sits in registers, and dL/dx
// leaves through the same unit.
template <class C>
using BwdSmem = Smem<C, kBwdWarps, 6, 1>;

template <class C>
__global__ void __launch_bounds__(kBwdWarps * 32) eq_bwd_kernel(EqParams p) {
  constexpr int W = kBwdWarps;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  BwdSmem<C> sm(smem_raw);
  const Tables<C>& tb = *sm.tb;
  __shared__ double red[W][kSections * 5][2];
  const int lane = threadIdx.x & 31;
  // the warp index, read from lane 0: the compiler then KNOWS it is warp-uniform.  With `threadIdx.x >> 5` the
  // warp-strided tile loop below counts as divergent and every shuffle of the scans is emitted as a five-instruction
  // WARPSYNC.COLLECTIVE / MOV / SHFL / MOV / ENDCOLLECTIVE sequence through two fixed registers (measured on the SASS:
  // 1776 SHFL + 1804 collective brackets + ~2300 extra MOV in eq_bwd_kernel, and no overlap between shuffles).
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const PairRows pr = pair_rows(blockIdx.x, p.rows);
  const int64_t row_a = pr.row_a, row_b = pr.row_b;
  const bool has_b = pr.has_b;

  build_tables(*sm.tb, p.params, row_a / p.chs, row_b / p.chs, p.sample_rate);
  Mail<W> mail{sm.mail_data, sm.mail_bar};
  if (threadIdx.x == 0) {
    for (int i = 0; i < W; ++i) mbar_init(&sm.full[i], 1);
    mail.init_all();
  }
  __syncthreads();

  const RowPair rp{p.n, p.ntiles, p.bulk != 0, has_b};
  const float* xa = p.x + row_a * p.n;
  const float* xb = p.x + row_b * p.n;
  const float* ga = p.gy + row_a * p.n;
  const float* gb = p.gy + row_b * p.n;
  float* oa = p.y + row_a * p.n;
  float* ob = p.y + row_b * p.n;
  float* my = sm.units + (size_t)warp * 6 * kUnitFloats;
  float* xu = my;                                  // x unit
  float* gu = my + kUnitFloats;                    // dL/dy unit, then the input of section 5, then dL/dx
  f2* U = reinterpret_cast<f2*>(my + (size_t)2 * kUnitFloats);     // [4][kTile] f2: inputs of sections 1..4
  uint64_t* full = sm.full + warp;
  const StepOffsets so_f = fwd_offsets(lane), so_r = rev_offsets(lane);
  const float4* ckpt = reinterpret_cast<const float4*>(p.ckpt) + (int64_t)blockIdx.x * p.ntiles * kSections;

  f2 acc[kSections][5];
#pragma unroll
  for (int k = 0; k < kSections; ++k) {
#pragma unroll
    for (int q = 0; q < 5; ++q) acc[k][q] = zero2();
  }

  int jt = 0;
  for (int seq = warp; seq < p.ntiles; seq += W, ++jt) {
    const int tile = p.ntiles - 1 - seq;
    if (rp.bulk && lane == 0) tma_store_wait_read<0>();      // the store of the previous tile has finished reading gu
    __syncwarp();
    {  // x and dL/dy tiles complete on ONE barrier
      const int64_t pos = (int64_t)tile * kTile;
      const int len = rp.len_of(tile);
      if (rp.bulk) {
        if (lane == 0) {
          mbar_arrive_expect_tx(full, (uint32_t)len * 16u);
          tma_load_1d(xu, xa + pos, (uint32_t)len * 4u, full);
          tma_load_1d(xu + kTile, xb + pos, (uint32_t)len * 4u, full);
          tma_load_1d(gu, ga + pos, (uint32_t)len * 4u, full);
          tma_load_1d(gu + kTile, gb + pos, (uint32_t)len * 4u, full);
        }
      } else {
        for (int i = lane; i < len; i += 32) {
          xu[i] = xa[pos + i]; xu[kTile + i] = xb[pos + i];
          gu[i] = ga[pos + i]; gu[kTile + i] = gb[pos + i];
        }
        __syncwarp();
      }
    }
    if (rp.bulk) mbar_wait(full, (uint32_t)(jt & 1));
    f2* U5 = reinterpret_cast<f2*>(gu);            // input of section 5, interleaved, over the consumed dL/dy unit
    const int off = lane * kE;
    const int64_t n0 = (int64_t)tile * kTile + off;
    const bool full_tile = (int64_t)(tile + 1) * kTile <= p.n;       // warp-uniform

    f2 gq[kE];                                     // dL/dy of the lane's samples; becomes dL/du_k section by section
    if (full_tile) {
#pragma unroll
      for (int j = 0; j < kE; ++j) gq[j] = make_float2(gu[off + j], gu[kTile + off + j]);
    } else {
#pragma unroll
      for (int j = 0; j < kE; ++j)
        gq[j] = (n0 + j < p.n) ? make_float2(gu[off + j], gu[kTile + off + j]) : zero2();
    }
    __syncwarp();                                  // all lanes hold their dL/dy before the unit is overwritten

    // ---- phase F: recompute the section inputs u_1..u_5 and every section's state entering the lane's chunk ----
    St sin[kSections];
    {
      f2 v[kE];
      if (full_tile) {
#pragma unroll
        for (int j = 0; j < kE; ++j) v[j] = make_float2(xu[off + j], xu[kTile + off + j]);
      } else {
#pragma unroll
        for (int j = 0; j < kE; ++j)
          v[j] = (n0 + j < p.n) ? make_float2(xu[off + j], xu[kTile + off + j]) : zero2();
      }
#pragma unroll
      for (int k = 0; k < kSections; ++k) {
        const Cf c = load_cf(tb, k);
        St incl = local_pass(v, c);
        St excl;
        scan_fwd(incl, tb, k, so_f, lane, excl);
        const float4 ck = ckpt[(int64_t)tile * kSections + k];
        const St cin = {make_float2(ck.x, ck.y), make_float2(ck.z, ck.w)};
        sin[k] = mv_acc(ldm(&tb.lane[k][lane][0]), cin, excl);
        if (k < kSections - 1) {
          fix_up(v, tb, k, sin[k]);
          f2* uk = (k == kSections - 2) ? U5 + off : U + (size_t)k * kTile + off;
#pragma unroll
          for (int j = 0; j < kE; ++j) uk[j] = v[j];
        }
      }
    }

    // ---- phase B: unwind the sections 6 -> 1 ----
#pragma unroll
    for (int k = kSections - 1; k >= 0; --k) {
      const Cf c = load_cf(tb, k);
      f2 u[kE], s1[kE], s2[kE];
      if (k == 0) {
        if (full_tile) {
#pragma unroll
          for (int j = 0; j < kE; ++j) u[j] = make_float2(xu[off + j], xu[kTile + off + j]);
        } else {
#pragma unroll
          for (int j = 0; j < kE; ++j)
            u[j] = (n0 + j < p.n) ? make_float2(xu[off + j], xu[kTile + off + j]) : zero2();
        }
      } else {
        const f2* uk = (k == kSections - 1) ? U5 + off : U + (size_t)(k - 1) * kTile + off;
#pragma unroll
        for (int j = 0; j < kE; ++j) u[j] = uk[j];
      }
      {  // true-state forward pass: s[j] = state BEFORE sample j
        f2 a1 = sin[k].s1, a2 = sin[k].s2;
#pragma unroll
        for (int j = 0; j < kE; ++j) {
          s1[j] = a1; s2[j] = a2;
          const f2 ta = ffma2(c.be1, u[j], a2);
          const f2 tb2 = ffma2(c.q, a1, fmul2(c.B2, u[j]));
          a1 = ffma2(c.sg, a1, ta);
          a2 = ffma2(c.sg, a2, tb2);
        }
      }
      St incl;
      {  // zero-terminal reverse pass: only the value reaching the chunk's first sample is needed
        f2 l1 = zero2(), l2 = zero2();
#pragma unroll
        for (int j = kE - 1; j >= 0; --j) {
          const f2 t1 = ffma2(c.sg, l1, ffma2(c.q, l2, gq[j]));
          l2 = ffma2(c.sg, l2, l1);
          l1 = t1;
        }
        incl = {l1, l2};
      }
      St excl;
      scan_rev(incl, tb, k, so_r, lane, excl);
      const St ain = mail.take(k, warp, jt);       // adjoint state at the first sample of the NEXT tile (in time)
      if (lane == 0 && seq + 1 < p.ntiles)         // lane 0 holds the tile total of the reverse scan
        mail.put(k, (warp + 1) % W, mtv_acc(ldm(&tb.warp[k][0]), ain, incl));
      // distance from the first sample of lane+1's chunk to the first sample of the next tile: (31-lane) chunks
      const St din = mtv_acc(ldm(&tb.lane[k][31 - lane][0]), ain, excl);
      {  // final reverse pass with the true terminal adjoint state
        f2 l1 = din.s1, l2 = din.s2;               // lambda[n+1] while processing sample n
#pragma unroll
        for (int j = kE - 1; j >= 0; --j) {
          const f2 gj = gq[j];
          acc[k][0] = ffma2(l1, s1[j], ffma2(l2, s2[j], acc[k][0]));
          acc[k][1] = ffma2(l2, s1[j], acc[k][1]);
          acc[k][2] = ffma2(l1, u[j], acc[k][2]);
          acc[k][3] = ffma2(l2, u[j], acc[k][3]);
          acc[k][4] = ffma2(gj, u[j], acc[k][4]);
          gq[j] = ffma2(c.be1, l1, ffma2(c.B2, l2, fmul2(c.b0, gj)));
          const f2 t1 = ffma2(c.sg, l1, ffma2(c.q, l2, gj));
          l2 = ffma2(c.sg, l2, l1);
          l1 = t1;
        }
      }
      if (k == kSections - 1) __syncwarp();        // every lane has read its u_5 before dL/dx may land in the dL/dy unit
    }
#pragma unroll
    for (int j = 0; j < kE; ++j) { gu[off + j] = gq[j].x; gu[kTile + off + j] = gq[j].y; }
    warp_store(gu, oa, ob, tile, rp, lane);
  }
  if (rp.bulk && lane == 0) tma_store_wait_all<0>();

  // ---- deterministic block reduction of the 2 x 30 sums (fp64), one partial row per row of the pair ----
#pragma unroll
  for (int k = 0; k < kSections; ++k) {
#pragma unroll
    for (int q = 0; q < 5; ++q) {
      const double sa = warp_sum((double)acc[k][q].x), sb = warp_sum((double)acc[k][q].y);
      if (lane == 0) { red[warp][k * 5 + q][0] = sa; red[warp][k * 5 + q][1] = sb; }
    }
  }
  __syncthreads();
  for (int o = threadIdx.x; o < kSections * 5 * 2; o += W * 32) {
    const int h = o / (kSections * 5), e = o - h * (kSections * 5);
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < W; ++w) s += red[w][e][h];
    if (h == 0) p.partial[row_a * 30 + e] = (float)s;
    else if (has_b) p.partial[row_b * 30 + e] = (float)s;
  }
}

// one thread per (item, section): add the channel partials, apply the fp64 Jacobian
__global__ void eq_param_grad_kernel(const float* __restrict__ partial, const float* __restrict__ params,
                                     float* __restrict__ gparams, int64_t bs, int chs, float sample_rate) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= bs * kSections) return;
  const int64_t item = idx / kSections;
  const int k = (int)(idx - item * kSections);
  double gc[5] = {0, 0, 0, 0, 0};
  for (int c = 0; c < chs; ++c) {
    const float* pr = partial + ((int64_t)item * chs + c) * 30 + k * 5;
#pragma unroll
    for (int q = 0; q < 5; ++q) gc[q] += (double)pr[q];
  }
  const float* pp = params + item * 18 + 3 * k;
  const SigmaCoef sc = design_section((double)pp[0], (double)pp[1], (double)pp[2], (double)sample_rate, section_kind(k));
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    double s = 0.0;
#pragma unroll
    for (int q = 0; q < 5; ++q) s += gc[q] * sc.c[q].d[d];
    gparams[item * 18 + 3 * k + d] = (float)s;
  }
}

// ---- host side -----------------------------------------------------------------------------
// Warps per row pair of the forward (dasp_debug_force_warps pins 4, 8 or 16).  Measured on B200 at 1024 pairs x 48000
// samples (profiles/r02_eq_variants.md): W=4 with two load stages beats W=2 and the single-wave choices; small batches
// want W=8 to fill the SMs at all.  W = 16 (512 threads, 80 registers): when there is at most one row pair per SM
// (e.g. 1024 stereo items split over 8 GPUs) a pair's CTA is alone on its SM, and sixteen warps walk its tiles twice as
// fast as eight.  The backward cannot follow (255 registers per thread x 512 threads exceed the register file).
int pick_fwd_warps(int64_t pairs) {
  const int f = debug_forced_warps();
  if (f == 4 || f == 8 || f == 16) return f;
  if (pairs <= sm_count()) return 16;
  return (pairs * 4 < 20ll * sm_count()) ? 8 : 4;
}

// one-off opt-in to > 48 KB dynamic shared memory, cached per (host thread, device, kernel INSTANTIATION): the
// kernel is a non-type template parameter, because every instantiation has the same function-pointer type
template <auto Kernel>
int ensure_smem(size_t bytes) {
  static thread_local int done_dev = -1;
  int dev = 0;
  DASP_CUDA_OK(cudaGetDevice(&dev));
  if (done_dev != dev) {
    DASP_CUDA_OK(cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    done_dev = dev;
  }
  return DASP_OK;
}

template <class C, int W>
int launch_fwd(const EqParams& p, int64_t pairs, cudaStream_t st) {
  constexpr size_t smem = FwdSmem<C, W>::kBytes;
  static_assert(smem <= kSmemPerSm, "eq fwd: shared memory of one CTA exceeds the SM");
  int rc = ensure_smem<eq_fwd_kernel<C, W>>(smem);
  if (rc != DASP_OK) return rc;
  eq_fwd_kernel<C, W><<<(unsigned)pairs, W * 32, smem, st>>>(p);
  DASP_LAUNCH_OK("eq_fwd_kernel");
  return DASP_OK;
}
template <class C>
int launch_bwd(const EqParams& p, int64_t pairs, cudaStream_t st) {
  constexpr size_t smem = BwdSmem<C>::kBytes;
  static_assert(smem <= kSmemPerSm, "eq bwd: shared memory of one CTA exceeds the SM");
  int rc = ensure_smem<eq_bwd_kernel<C>>(smem);
  if (rc != DASP_OK) return rc;
  eq_bwd_kernel<C><<<(unsigned)pairs, kBwdWarps * 32, smem, st>>>(p);
  DASP_LAUNCH_OK("eq_bwd_kernel");
  return DASP_OK;
}
template <class C>
int dispatch_fwd(int w, const EqParams& p, int64_t pairs, cudaStream_t st) {
  switch (w) {
    case 4: return launch_fwd<C, 4>(p, pairs, st);
    case 16: return launch_fwd<C, 16>(p, pairs, st);
    default: return launch_fwd<C, 8>(p, pairs, st);
  }
}

}  // namespace
}  // namespace dasp

using namespace dasp;

extern "C" {

int64_t dasp_eq_tile_len(int64_t rows) { (void)rows; return kTile; }
int64_t dasp_eq_ckpt_floats(int64_t bs, int64_t chs, int64_t n) {
  const int64_t pairs = (bs * chs + 1) / 2, ntiles = (n + kTile - 1) / kTile;
  return pairs * (ntiles > 0 ? ntiles : 1) * kSections * 4;
}
int64_t dasp_eq_bwd_workspace_floats(int64_t bs, int64_t chs) { return bs * chs * 30; }

int dasp_eq_fwd(const float* x, const float* params, float* y, float* ckpt, int64_t bs, int64_t chs, int64_t n,
                float sample_rate, void* stream) {
  DASP_REQUIRE(bs >= 0 && chs >= 1 && n >= 0, "eq fwd: bad shape bs=%lld chs=%lld n=%lld", (long long)bs,
               (long long)chs, (long long)n);
  if (bs == 0 || n == 0) return DASP_OK;
  DASP_REQUIRE(x && params && y, "eq fwd: null pointer");
  DASP_REQUIRE(sample_rate > 0.f, "eq fwd: sample_rate must be positive");
  const int64_t rows = bs * chs, pairs = (rows + 1) / 2;
  DASP_REQUIRE(pairs < (1ll << 31), "eq fwd: too many rows");
  const int w = pick_fwd_warps(pairs);
  EqParams p{};
  p.x = x; p.y = y; p.params = params; p.ckpt = ckpt; p.n = n; p.rows = rows; p.chs = (int)chs;
  p.ntiles = (int)((n + kTile - 1) / kTile); p.sample_rate = sample_rate;
  p.bulk = (n % 4 == 0) && aligned16(x) && aligned16(y);
  cudaStream_t st = (cudaStream_t)stream;
  const bool same_item = chs % 2 == 0;      // rows 2p and 2p+1 share their item
  return same_item ? dispatch_fwd<float>(w, p, pairs, st) : dispatch_fwd<f2>(w, p, pairs, st);
}

int dasp_eq_bwd(const float* gy, const float* x, const float* params, const float* ckpt, float* gx,
                float* gparams, float* ws, int64_t ws_floats, int64_t bs, int64_t chs, int64_t n,
                float sample_rate, void* stream) {
  DASP_REQUIRE(bs >= 0 && chs >= 1 && n >= 0, "eq bwd: bad shape bs=%lld chs=%lld n=%lld", (long long)bs,
               (long long)chs, (long long)n);
  if (bs == 0) return DASP_OK;
  cudaStream_t st = (cudaStream_t)stream;
  DASP_REQUIRE(gparams != nullptr, "eq bwd: null gparams");
  if (n == 0) { DASP_CUDA_OK(cudaMemsetAsync(gparams, 0, sizeof(float) * 18 * bs, st)); return DASP_OK; }
  DASP_REQUIRE(gy && x && params && ckpt && gx, "eq bwd: null pointer");
  const int64_t rows = bs * chs, pairs = (rows + 1) / 2;
  DASP_REQUIRE(pairs < (1ll << 31), "eq bwd: too many rows");
  if (ws == nullptr || ws_floats < rows * 30) {
    set_error("eq bwd: workspace needs %lld floats, got %lld", (long long)(rows * 30), (long long)ws_floats);
    return DASP_ERR_WORKSPACE;
  }
  EqParams p{};
  p.x = x; p.gy = gy; p.y = gx; p.params = params; p.ckpt = const_cast<float*>(ckpt); p.partial = ws; p.n = n;
  p.rows = rows; p.chs = (int)chs; p.ntiles = (int)((n + kTile - 1) / kTile); p.sample_rate = sample_rate;
  p.bulk = (n % 4 == 0) && aligned16(x) && aligned16(gy) && aligned16(gx);
  const int rc = chs % 2 == 0 ? launch_bwd<float>(p, pairs, st) : launch_bwd<f2>(p, pairs, st);
  if (rc != DASP_OK) return rc;
  const int64_t tot = bs * kSections;
  eq_param_grad_kernel<<<(unsigned)((tot + 127) / 128), 128, 0, st>>>(ws, params, gparams, bs, (int)chs, sample_rate);
  DASP_LAUNCH_OK("eq_param_grad_kernel");
  return DASP_OK;
}

}  // extern "C"
