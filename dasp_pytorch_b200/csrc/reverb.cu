// noise_shaped_reverberation forward + backward (reference: dasp_pytorch/functional.py:406-577,
// filter bank dasp_pytorch/signal.py:42-92).
//
// The reference builds, per item and channel, an impulse response as the mean of 12 band-filtered
// white-noise signals (1023-tap FIRs, time-domain conv1d, functional.py:551-556), each shaped by an
// exponential envelope and a gain (:561-567), then convolves the audio with it by a second
// time-domain conv1d with an L-tap kernel (:570-572).  >99.9 % of its time is those two direct
// convolutions.  Here both are FFT convolutions (SURVEY.md Appendix A.5) built from ONE transform shape,
// the 8192-point batched C2C that cuFFT runs as a single shared-memory kernel (~4.5 TB/s effective on
// B200; its long transforms reach 0.3-1.5 TB/s), with everything between the transforms fused:
//
//   * Only the first Leff = min(L, N) taps of the impulse response can reach the N output samples
//     (y[n] = sum_{t<=n} IR[t] x[n-t], n < N), so only those are synthesised -- an exact saving.
//   * The LEFT and RIGHT channel of a band / of the audio are packed as real/imag of one complex sequence.
//   * IR synthesis, device noise (default): spectral_gen_kernel draws the FILTERED noise spectrum directly
//     (Philox4x32-10 + Box-Muller; see the comment at the kernel); ifft_shape_kernel = own in-shared-memory inverse
//     FFT (fft8192.cuh) fused with envelope * gain * band mean -> IR written straight into the partition layout of
//     the convolution.  Filter banks of 2047 taps or more (transform length nb > 8192) take batched cuFFT +
//     shape_ir_pp_kernel instead; polyphase factors R > 16 take the overlap-save path of parity mode, fed by
//     time-domain Philox noise.
//   * IR synthesis, parity mode (caller's noise tensor): overlap-save blocks -> C2C -> cmul_filter_pairs ->
//     inverse C2C -> shape_ir_pairs_kernel.
//   * Audio convolution: uniformly partitioned overlap-save in the frequency domain: x_fft_kernel (window gather +
//     FFT), partition_mac_kernel, ifft_mix_kernel (inverse FFT + crop + wet/dry mix), all on the own FFT; rows that
//     are not 16-byte aligned use x_blocks_kernel, cuFFT C2C, mix_blocks_kernel.
//   * Items are processed in chunks (chosen by the caller; the Python host uses one item per SM) to bound the workspace.
//
// Backward (A.5): g_blocks_kernel (+ dL/dmix partials), C2C, two correlation passes of partition_mac_kernel
// against the saved block spectra (dL/dx windows, dL/dIR partitions), two inverse C2C, finish_dx_blocks_kernel,
// ir_grad_*_kernel (dL/dIR * env * f reductions for the 24 band parameters; deterministic two-stage sums).
#include <cufft.h>
#include <curand_kernel.h>
#include <math.h>

#include <map>
#include <mutex>
#include <tuple>
#include <vector>

#include "common.cuh"
#include "fft8192.cuh"

namespace dasp {
namespace {

constexpr int kBands = 12;
constexpr int kB = 4096;          // partition / hop of the audio convolution
constexpr int kNbA = 2 * kB;      // its FFT length (single-kernel cuFFT C2C size)
constexpr double kPi = 3.14159265358979323846;

#define DASP_CUFFT_OK(expr)                                                        \
  do {                                                                             \
    cufftResult r__ = (expr);                                                      \
    if (r__ != CUFFT_SUCCESS) {                                                    \
      ::dasp::set_error("%s failed: cufft error %d (%s:%d)", #expr, (int)r__, __FILE__, __LINE__); \
      return DASP_ERR_CUFFT;                                                       \
    }                                                                              \
  } while (0)

// ------------------------------------------------------------------ filter bank (host, fp64)
// scipy.signal.firwin(numtaps, cutoff, window="hamming", pass_zero, scale=True, fs) restated.
// band = [lo, hi] in Hz; lo == 0 -> low-pass, hi == nyquist -> high-pass.
void firwin_hamming(int numtaps, double lo_hz, double hi_hz, double fs, double* h) {
  const double nyq = 0.5 * fs;
  const double left = lo_hz / nyq, right = hi_hz / nyq;
  const double alpha = 0.5 * (numtaps - 1);
  auto sinc = [](double x) { return x == 0.0 ? 1.0 : sin(kPi * x) / (kPi * x); };
  for (int i = 0; i < numtaps; ++i) {
    const double m = i - alpha;
    double v = right * sinc(right * m) - left * sinc(left * m);
    const double w = (numtaps == 1) ? 1.0 : 0.54 - 0.46 * cos(2.0 * kPi * i / (numtaps - 1));
    h[i] = v * w;
  }
  double scale_frequency;
  if (left == 0.0) scale_frequency = 0.0;
  else if (right == 1.0) scale_frequency = 1.0;
  else scale_frequency = 0.5 * (left + right);
  double s = 0.0;
  for (int i = 0; i < numtaps; ++i) s += h[i] * cos(kPi * (i - alpha) * scale_frequency);
  for (int i = 0; i < numtaps; ++i) h[i] /= s;
}

// the 12 filters of signal.octave_band_filterbank (signal.py:42-92), cast to fp32 like the reference
void octave_filterbank(int taps, double sr, std::vector<float>& out) {
  static const double centres[10] = {31.5, 63, 125, 250, 500, 1000, 2000, 4000, 8000, 16000};
  out.assign((size_t)kBands * taps, 0.f);
  std::vector<double> h(taps);
  auto put = [&](int k) { for (int i = 0; i < taps; ++i) out[(size_t)k * taps + i] = (float)h[i]; };
  firwin_hamming(taps, 0.0, 12.0, sr, h.data());                       // low-pass 12 Hz (signal.py:60-64)
  put(0);
  for (int b = 0; b < 10; ++b) {                                       // octave band-passes (:69-78)
    const double lo = centres[b] / sqrt(2.0);
    double hi = centres[b] * sqrt(2.0);
    const double cap = 0.999 * sr / 2.0;
    if (hi > cap) hi = cap;
    firwin_hamming(taps, lo, hi, sr, h.data());
    put(1 + b);
  }
  firwin_hamming(taps, 18000.0, sr / 2.0, sr, h.data());               // high-pass 18 kHz (:84)
  put(11);
}

// ------------------------------------------------------------------ geometry
struct Geom {
  int64_t bs, n, L, taps, P;
  int64_t leff;                 // min(L, n): the only IR taps that can reach the output
  int64_t nb, hop, nbk, chunk;
  int64_t ib, jb;               // audio convolution: output/input blocks of kB samples, IR partitions of kB taps
  int64_t rpp;                  // polyphase factor of the spectral synthesis: n1 = rpp*nb >= leff + P
  int64_t n1() const { return rpp * nb; }
  int64_t n1c() const { return n1() / 2 + 1; }
  int64_t nparts_pp() const { return (nb + 255) / 256; }
  // complex samples per (item, band) pair in either filtered-noise layout (overlap-save / polyphase)
  int64_t pair_c64() const { return (nbk > rpp ? nbk : rpp) * nb; }
};

int make_geom(int64_t bs, int64_t n, int64_t L, int64_t taps, int64_t chunk, Geom& g) {
  DASP_REQUIRE(bs >= 0 && n >= 1 && L >= 2, "reverb: bad shape bs=%lld n=%lld num_samples=%lld", (long long)bs,
               (long long)n, (long long)L);
  DASP_REQUIRE(taps >= 1 && (taps % 2) == 1, "num_bandpass_taps must be odd");
  g.bs = bs; g.n = n; g.L = L; g.taps = taps; g.P = taps - 1;
  const int64_t discard = ((g.P + 3) / 4) * 4;            // >= P, keeps every block 16-byte aligned
  int64_t nb = 8192;
  while (nb < 4 * (discard + 1)) nb *= 2;
  g.nb = nb;
  g.hop = nb - discard;
  g.leff = L < n ? L : n;
  g.nbk = (g.leff + g.hop - 1) / g.hop;
  g.rpp = (g.leff + g.P + nb - 1) / nb;
  g.ib = (n + kB - 1) / kB;
  g.jb = (g.leff + kB - 1) / kB;
  if (chunk <= 0) chunk = 4;
  g.chunk = chunk < bs ? chunk : (bs > 0 ? bs : 1);
  return DASP_OK;
}

// ------------------------------------------------------------------ plan / filter cache
struct PlanKey {
  int dev; int type; int64_t n, batch, idist, odist;
  bool operator<(const PlanKey& o) const {
    return std::tie(dev, type, n, batch, idist, odist) < std::tie(o.dev, o.type, o.n, o.batch, o.idist, o.odist);
  }
};
struct PlanVal { cufftHandle h; size_t work; };
struct FbKey {
  int dev; int64_t taps, nb; double sr;      // nb < 0: half spectrum at n1 = -nb points (spectral synthesis)
  bool operator<(const FbKey& o) const { return std::tie(dev, taps, nb, sr) < std::tie(o.dev, o.taps, o.nb, o.sr); }
};

std::mutex g_mu;
std::map<PlanKey, PlanVal> g_plans;
std::map<FbKey, cufftComplex*> g_fb;

int get_plan(int type /*0 = R2C, 1 = C2R, 2 = C2C*/, int64_t n, int64_t batch, int64_t idist, int64_t odist, PlanVal& out) {
  int dev = 0;
  DASP_CUDA_OK(cudaGetDevice(&dev));
  PlanKey key{dev, type, n, batch, idist, odist};
  auto it = g_plans.find(key);
  if (it != g_plans.end()) { out = it->second; return DASP_OK; }
  PlanVal pv{};
  DASP_CUFFT_OK(cufftCreate(&pv.h));
  DASP_CUFFT_OK(cufftSetAutoAllocation(pv.h, 0));
  long long nn[1] = {(long long)n};
  long long inembed[1] = {(long long)(type == 1 ? n / 2 + 1 : n)};
  long long onembed[1] = {(long long)(type == 0 ? n / 2 + 1 : n)};
  const cufftType ct = type == 0 ? CUFFT_R2C : (type == 1 ? CUFFT_C2R : CUFFT_C2C);
  DASP_CUFFT_OK(cufftMakePlanMany64(pv.h, 1, nn, inembed, 1, (long long)idist, onembed, 1, (long long)odist, ct,
                                    (long long)batch, &pv.work));
  g_plans[key] = pv;
  out = pv;
  return DASP_OK;
}

// ------------------------------------------------------------------ kernels
// Overlap-save block layout shared by the kernels below.  For item i (chunk-local), band k, block b,
// sample m < nb the complex element  C[((i*12 + k)*nbk + b)*nb + m]  holds (left, right) of the band
// signal at absolute noise position b*hop + m; after the two FFTs it holds the filtered noise f at time
// t = b*hop + m - P (valid for P <= m < P + hop).

// parity mode: gather the user noise (bs*2 rows x 12 bands x (L+P) samples) into the block layout
__global__ void noise_pairs_layout_kernel(const float* __restrict__ noise, float2* __restrict__ C, int64_t item0,
                                          int nbk, int nb, int hop, int64_t lp) {
  // grid = (nbk, 12, items); threads stride over m
  const int b = blockIdx.x, k = blockIdx.y;
  const int64_t il = blockIdx.z;
  const float* nl = noise + (((item0 + il) * 2 + 0) * kBands + k) * lp;
  const float* nr = noise + (((item0 + il) * 2 + 1) * kBands + k) * lp;
  float2* out = C + ((il * kBands + k) * nbk + b) * (int64_t)nb;
  for (int m = threadIdx.x; m < nb; m += blockDim.x) {
    const int64_t pos = (int64_t)b * hop + m;
    float2 v = make_float2(0.f, 0.f);
    if (pos < lp) v = make_float2(nl[pos], nr[pos]);
    out[m] = v;
  }
}

// performance mode: N(0,1) from Philox4x32-10 (cuRAND device API).  The stream of a band signal is
// addressed by its absolute sample position, so the overlapping part of consecutive blocks is simply
// generated twice and nothing depends on the chunking.
__global__ void noise_pairs_philox_kernel(float2* __restrict__ C, int64_t item0, int nbk, int nb, int hop,
                                          const unsigned long long* seed) {
  const int b = blockIdx.x, k = blockIdx.y;
  const int64_t il = blockIdx.z;
  const unsigned long long sig_l = (unsigned long long)(((item0 + il) * 2 + 0) * kBands + k);
  const unsigned long long sig_r = (unsigned long long)(((item0 + il) * 2 + 1) * kBands + k);
  float4* out = reinterpret_cast<float4*>(C + ((il * kBands + k) * nbk + b) * (int64_t)nb);
  for (int q4 = threadIdx.x; q4 < nb / 4; q4 += blockDim.x) {
    const unsigned long long quad = (unsigned long long)(((int64_t)b * hop) / 4 + q4);   // hop % 4 == 0
    curandStatePhilox4_32_10_t sl, sr;
    curand_init(__ldg(seed), (sig_l << 24) + quad, 0ull, &sl);
    curand_init(__ldg(seed), (sig_r << 24) + quad, 0ull, &sr);
    const float4 l = curand_normal4(&sl), r = curand_normal4(&sr);
    out[q4 * 2 + 0] = make_float4(l.x, r.x, l.y, r.y);
    out[q4 * 2 + 1] = make_float4(l.z, r.z, l.w, r.w);
  }
}

// block spectra *= H_band (full nb-point spectrum of the real filter, 1/nb of the inverse FFT folded in)
__global__ void cmul_filter_pairs_kernel(float2* __restrict__ C, const float2* __restrict__ H, int nbk, int nb) {
  const int b = blockIdx.x, k = blockIdx.y;
  const int64_t il = blockIdx.z;
  float2* c = C + ((il * kBands + k) * nbk + b) * (int64_t)nb;
  const float2* h = H + (int64_t)k * nb;
  for (int f = threadIdx.x; f < nb; f += blockDim.x) {
    const float2 a = c[f], w = h[f];
    c[f] = make_float2(a.x * w.x - a.y * w.y, a.x * w.y + a.y * w.x);
  }
}

// packed fp32x2 helpers of the generator's R-point DFT (FFMA2 / FMUL2, see fft8192.cuh)
__device__ __forceinline__ float2 gen_ffma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 gen_fmul2(float2 a, float2 b) { return __fmul2_rn(a, b); }

// ---- spectral synthesis (device-noise mode) ------------------------------------------------------
// The band-filtered noise only has to be a stationary Gaussian process with the FIR's autocovariance on
// the window [0, leff).  A length-n1 PERIODIC white sequence filtered circularly has exactly that
// covariance for every lag inside the window once n1 >= leff + P, and its spectrum has independent bins:
//   G[j] = H_k[j] Z[j],  Z[j] ~ CN(0, n1)  (real N(0, n1) at j = 0 and n1/2),  G[n1-j] = conj(G[j]).
// So the spectrum is drawn directly (no forward FFT, no separate filter pass) and only ONE inverse
// transform remains.  n1 = R*nb is split Cooley-Tukey style so that the inverse is the fast single-kernel
// nb-point batched C2C:   f[R a + b] = sum_{j1<nb} Q_b[j1] e^{2 pi i j1 a / nb},
//   Q_b[j1] = e^{2 pi i j1 b / n1} * sum_{j2<R} G[j1 + nb j2] e^{2 pi i j2 b / R}
// Polyphase layout: C[((item*12 + k)*R + b)*nb + a] = (f_left, f_right)[R a + b].
// Left/right are packed as G_left + i G_right; one Philox call per canonical bin yields both channels.
// Philox4x32-10 (Salmon et al., SC'11), counter = (c0, c1, c2, c3), key = (k0, k1); written out instead of the
// cuRAND state machinery because this kernel needs exactly one block of 4 words per call site
struct PhiloxKeys { uint2 k[10]; };           // the ten round keys (key + r * Weyl constants): one schedule per thread
__device__ __forceinline__ PhiloxKeys philox_keys(unsigned long long sd) {
  PhiloxKeys ks;
  uint2 k = make_uint2((unsigned)sd, (unsigned)(sd >> 32));
#pragma unroll
  for (int r = 0; r < 10; ++r) { ks.k[r] = k; k.x += 0x9E3779B9u; k.y += 0xBB67AE85u; }
  return ks;
}
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, const PhiloxKeys& ks) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const unsigned long long p0 = (unsigned long long)0xD2511F53u * c.x;
    const unsigned long long p1 = (unsigned long long)0xCD9E8D57u * c.z;
    c = make_uint4((unsigned)(p1 >> 32) ^ c.y ^ ks.k[r].x, (unsigned)p1, (unsigned)(p0 >> 32) ^ c.w ^ ks.k[r].y, (unsigned)p0);
  }
  return c;
}
// two independent N(0,1) from two 32-bit words (Box-Muller; u1 in (0,1], angle in turns)
// MUFU-only transcendental path (lg2, rsq, sin, cos: |abs err| ~ 1e-6, irrelevant for a noise source) -- the
// generator kernel is instruction-issue bound and the accurate logf/sqrtf/sincospif were ~55 % of it
__device__ __forceinline__ float2 box_muller(unsigned a, unsigned b) {
  // uniforms from the top 23 bits placed in the mantissa of [1, 2): no I2F (the conversions share the XU pipe with the
  // four MUFU calls below).  u1 = 2 - [1,2) lies in (0, 1]; the angle (v - 1.5) * 2 pi in [-pi, pi)
  const float u1 = 2.0f - __uint_as_float(0x3f800000u | (a >> 9));
  const float ang = fmaf(__uint_as_float(0x3f800000u | (b >> 9)), 6.283185307179586f, -9.42477796076938f);
  const float m = -2.0f * __logf(u1);                                  // >= 0
  const float r = m * rsqrtf(fmaxf(m, 1e-30f));                        // sqrt(m)
  return make_float2(r * __cosf(ang), r * __sinf(ang));
}

// e^{2 pi i m / R} for every polyphase factor R <= 16 (filled once per device on the host side)
__constant__ float2 c_root[17][16];

// One residue class pair (j1, nb - j1) of one band signal: draws the R bins of each class, runs the R-point
// DFT + twiddle ladder and hands  Q_b[j1], Q_b[nb - j1]  (b = 0 .. R-1) to `emit(b, q_j1, q_mirror)`, which
// spectral_gen_kernel stores in the layout its consumer reads.
template <int R, class Emit>
__device__ __forceinline__ void spectral_unit(int j1, int nb, const float2* __restrict__ h, unsigned long long pair,
                                              const PhiloxKeys& keys, Emit&& emit) {
  const int n1 = R * nb, n1h = n1 / 2;
  // the real-valued bins 0 and n1/2 (variance n1 on the real axis instead of n1/2 per component) only occur in the two
  // self-mirrored classes j1 = 0 and j1 = nb/2: everything else takes the branch-free path
  const bool special_unit = (j1 == 0) || (2 * j1 == nb);
  // value of the packed spectrum G_left + i G_right at bin j (0 <= j < n1) and at its mirror n1 - j
  // `canonical` (j <= n1/2) is a compile-time fact of the unrolled call site: for j1 in [0, nb/2] the bin
  // j1 + nb j2 lies in the lower half exactly when 2 j2 < R (the only tie, j = n1/2, is its own mirror)
  auto draw = [&](int j, bool canonical, float2& at_j, float2& at_mirror) {
    const int jc = canonical ? j : n1 - j;
    // counter = (canonical bin, band pair), key = seed: one Philox block -> both channels' complex Gaussian
    const uint4 rnd = philox4x32_10(make_uint4((unsigned)jc, (unsigned)pair, (unsigned)(pair >> 32), 0x5eedu), keys);
    float2 zl = box_muller(rnd.x, rnd.y), zr = box_muller(rnd.z, rnd.w);
    if (special_unit && (jc == 0 || jc == n1h)) {
      zl = make_float2(zl.x * 1.4142135623730951f, 0.f);
      zr = make_float2(zr.x * 1.4142135623730951f, 0.f);
    }
    const float2 w = h[jc];                                          // H_k / n1 * sqrt(n1 / 2), folded on the host
    const float2 sl = make_float2(w.x * zl.x - w.y * zl.y, w.x * zl.y + w.y * zl.x);   // H Z_left
    const float2 sr = make_float2(w.x * zr.x - w.y * zr.y, w.x * zr.y + w.y * zr.x);   // H Z_right
    const float2 canon = make_float2(sl.x - sr.y, sl.y + sr.x);      // S_l + i S_r           (bin jc)
    const float2 mirr = make_float2(sl.x + sr.y, sr.x - sl.y);       // conj(S_l) + i conj(S_r) (bin n1 - jc)
    if (canonical) { at_j = canon; at_mirror = mirr; } else { at_j = mirr; at_mirror = canon; }
  };

  float2 ga[R], gb[R];
#pragma unroll
  for (int j2 = 0; j2 < R; ++j2) {
    float2 a, m;
    draw(j1 + nb * j2, 2 * j2 < R, a, m);
    ga[j2] = a;
    gb[R - 1 - j2] = m;          // mirror of bin j1 + nb j2 is bin (nb - j1) + nb (R-1-j2)
  }
  // The two residue classes (j1 and nb - j1) go through the SAME R-point DFT and twiddle ladder, so they are
  // packed into the two lanes of Blackwell's fp32x2 instructions (FFMA2/FMUL2: one issue slot, two FMAs).
  float2 gx[R], gy[R];                       // (class A, class B) real parts / imaginary parts
#pragma unroll
  for (int j2 = 0; j2 < R; ++j2) { gx[j2] = make_float2(ga[j2].x, gb[j2].x); gy[j2] = make_float2(ga[j2].y, gb[j2].y); }
  float2 rx[R], ry[R], nry[R];               // roots of unity broadcast to both lanes
#pragma unroll
  for (int m = 0; m < R; ++m) {
    const float2 r = c_root[R][m];
    rx[m] = make_float2(r.x, r.x); ry[m] = make_float2(r.y, r.y); nry[m] = make_float2(-r.y, -r.y);
  }
  // per-class twiddle steps e^{2 pi i j1 / n1} and e^{2 pi i (nb - j1) / n1} = e^{2 pi i / R} conj(the former)
  float2 w1a, w1b;
  __sincosf(6.283185307179586f * (float)j1 / (float)n1, &w1a.y, &w1a.x);      // argument <= pi / R
  {
    const float2 r1 = (R == 1) ? make_float2(1.f, 0.f) : c_root[R][1 % R];
    w1b = make_float2(fmaf(r1.x, w1a.x, r1.y * w1a.y), fmaf(r1.y, w1a.x, -r1.x * w1a.y));
  }
  const float2 wx = make_float2(w1a.x, w1b.x), wy = make_float2(w1a.y, w1b.y), nwy = make_float2(-w1a.y, -w1b.y);
  float2 tx = make_float2(1.f, 1.f), ty = make_float2(0.f, 0.f);      // twiddle e^{2 pi i j b / n1}, both classes
  // S[b] = sum_{j2} g[j2] e^{+2 pi i j2 b / R}: generic O(R^2) form, or for R = 6 (IR 96000 on 48000 samples, the
  // BASELINE geometry) radix 2 x 3 with literal constants -- 48 packed operations instead of 144
  float2 Sre[R], Sim[R];
  if constexpr (R == 6) {
    const float2 hlf = make_float2(0.5f, 0.5f), nhlf = make_float2(-0.5f, -0.5f);
    const float2 c3 = make_float2(0.8660254037844386f, 0.8660254037844386f), nc3 = make_float2(-0.8660254037844386f, -0.8660254037844386f);
    const float2 one = make_float2(1.f, 1.f), mone = make_float2(-1.f, -1.f);
    auto add = [&](float2 a, float2 b) { return gen_ffma2(b, one, a); };
    auto sub = [&](float2 a, float2 b) { return gen_ffma2(b, mone, a); };
    // 3-point DFT (positive exponent) of (a0, a1, a2): Y0 = a0 + t, Y1/2 = (a0 - t/2) +- i (sqrt3/2) d
    auto dft3 = [&](float2 a0r, float2 a0i, float2 a1r, float2 a1i, float2 a2r, float2 a2i, float2 (&yr)[3], float2 (&yi)[3]) {
      const float2 tr = add(a1r, a2r), ti = add(a1i, a2i), dr = sub(a1r, a2r), di = sub(a1i, a2i);
      yr[0] = add(a0r, tr); yi[0] = add(a0i, ti);
      const float2 mr = gen_ffma2(tr, nhlf, a0r), mi = gen_ffma2(ti, nhlf, a0i);
      yr[1] = gen_ffma2(di, nc3, mr); yi[1] = gen_ffma2(dr, c3, mi);       // + i c d = (-c d_i, c d_r)
      yr[2] = gen_ffma2(di, c3, mr);  yi[2] = gen_ffma2(dr, nc3, mi);
    };
    float2 er[3], ei[3], orr[3], oi[3];
    dft3(gx[0], gy[0], gx[2], gy[2], gx[4], gy[4], er, ei);
    dft3(gx[1], gy[1], gx[3], gy[3], gx[5], gy[5], orr, oi);
    // X[k] = E[k] + W6^k O[k], X[k+3] = E[k] - W6^k O[k];  W6 = (1/2, sqrt3/2), W6^2 = (-1/2, sqrt3/2)
    float2 pr[3], pi[3];
    pr[0] = orr[0]; pi[0] = oi[0];
    pr[1] = gen_ffma2(orr[1], hlf, gen_fmul2(oi[1], nc3));  pi[1] = gen_ffma2(orr[1], c3, gen_fmul2(oi[1], hlf));
    pr[2] = gen_ffma2(orr[2], nhlf, gen_fmul2(oi[2], nc3)); pi[2] = gen_ffma2(orr[2], c3, gen_fmul2(oi[2], nhlf));
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      Sre[k] = add(er[k], pr[k]); Sim[k] = add(ei[k], pi[k]);
      Sre[k + 3] = sub(er[k], pr[k]); Sim[k + 3] = sub(ei[k], pi[k]);
    }
  } else {
#pragma unroll
    for (int b = 0; b < R; ++b) {
      float2 sre = make_float2(0.f, 0.f), sim = make_float2(0.f, 0.f);
#pragma unroll
      for (int j2 = 0; j2 < R; ++j2) {
        const int m = (j2 * b) % R;
        sre = gen_ffma2(gx[j2], rx[m], gen_ffma2(gy[j2], nry[m], sre));
        sim = gen_ffma2(gx[j2], ry[m], gen_ffma2(gy[j2], rx[m], sim));
      }
      Sre[b] = sre; Sim[b] = sim;
    }
  }
#pragma unroll
  for (int b = 0; b < R; ++b) {
    const float2 sre = Sre[b], sim = Sim[b];
    const float2 ore = gen_ffma2(sre, tx, gen_fmul2(sim, make_float2(-ty.x, -ty.y)));
    const float2 oim = gen_ffma2(sre, ty, gen_fmul2(sim, tx));
    emit(b, make_float2(ore.x, oim.x), make_float2(ore.y, oim.y));
    const float2 ntx = gen_ffma2(tx, wx, gen_fmul2(ty, nwy));
    ty = gen_ffma2(tx, wy, gen_fmul2(ty, wx));
    tx = ntx;
  }
}

// PLANAR == false: C[((item*12 + k)*R + b)*nb + j] = (re, im) pairs, the input layout of the batched cuFFT C2C.
// PLANAR == true : the same 64 KB block per (item, band, class) holds [re plane nb][im plane nb] -- the shared-memory
//                  layout of fft8192.cuh, so ifft_shape_kernel can fetch a class with plain bulk copies.
template <int R, bool PLANAR>
__global__ void spectral_gen_kernel(float2* __restrict__ C, const float2* __restrict__ H1, int64_t item0, int nb,
                                    const unsigned long long* seed) {
  const int j1 = blockIdx.x * blockDim.x + threadIdx.x;       // residue class 0 .. nb/2
  if (j1 > nb / 2) return;
  const int k = blockIdx.y;
  const int64_t il = blockIdx.z;
  const unsigned long long pair = (unsigned long long)((item0 + il) * kBands + k);
  const PhiloxKeys keys = philox_keys(__ldg(seed));
  const bool self_mirror = (j1 == 0) || (2 * j1 == nb);     // class nb - j1 is class j1 itself
  float2* outp = C + ((il * kBands + k) * R) * (int64_t)nb;
  spectral_unit<R>(j1, nb, H1 + (int64_t)k * (R * nb / 2 + 1), pair, keys, [&](int b, float2 q, float2 qm) {
    if (PLANAR) {
      float* pl = reinterpret_cast<float*>(outp + (int64_t)b * nb);
      pl[j1] = q.x; pl[nb + j1] = q.y;
      if (!self_mirror) { pl[nb - j1] = qm.x; pl[2 * nb - j1] = qm.y; }
    } else {
      outp[(int64_t)b * nb + j1] = q;
      if (!self_mirror) outp[(int64_t)b * nb + (nb - j1)] = qm;
    }
  });
}

// torch.linspace(0, 1, L) in fp32 (functional.py:561): symmetric fill around the midpoint
__device__ __forceinline__ float time_axis(int64_t t, int64_t L, float step) {
  return (t < L / 2) ? step * (float)t : 1.0f - step * (float)(L - 1 - t);
}

// same values for L < 2^31 without 64-bit integer conversions
__device__ __forceinline__ float time_axis32(int t, int L, float step) {
  return (t < L / 2) ? step * (float)t : 1.0f - step * (float)(L - 1 - t);
}

// IR[c][t] = (1/12) sum_k gain_k exp(-(10 decay_k + 1) tt(t)) f_c[k][t]  for t < leff, written as (left, right)
// complex pairs into the zero-initialised partition layout of the audio convolution.
// grid = (nbk, items): CTA (b, item) produces samples [b*hop, (b+1)*hop).
__global__ void shape_ir_pairs_kernel(const float2* __restrict__ C, const float* __restrict__ params /* chunk x 25 */,
                                      float2* __restrict__ Hb, int64_t L, int64_t leff, int jb, int nbk, int nb,
                                      int hop, int P) {
  const int b = blockIdx.x;
  const int64_t il = blockIdx.y;
  __shared__ float gk[kBands], rk[kBands];
  if (threadIdx.x < kBands) {
    gk[threadIdx.x] = params[il * 25 + threadIdx.x] * (1.0f / kBands);
    rk[threadIdx.x] = -(params[il * 25 + kBands + threadIdx.x] * 10.0f + 1.0f);
  }
  __syncthreads();
  const float step = 1.0f / (float)(L - 1);
  float2* out = Hb + il * (int64_t)jb * kNbA;      // partition j holds taps [j kB, (j+1) kB) in its first half
  for (int m = threadIdx.x; m < hop; m += blockDim.x) {
    const int64_t t = (int64_t)b * hop + m;
    if (t >= leff) break;
    const float tt = time_axis(t, L, step);
    const float2* c = C + ((il * kBands) * nbk + b) * (int64_t)nb + m + P;
    float al = 0.f, ar = 0.f;
#pragma unroll
    for (int k = 0; k < kBands; ++k) {
      const float2 v = c[(int64_t)k * nbk * nb];
      const float e = gk[k] * expf(rk[k] * tt);
      al = fmaf(e, v.x, al);
      ar = fmaf(e, v.y, ar);
    }
    out[(t / kB) * kNbA + (t % kB)] = make_float2(al, ar);
  }
}

// polyphase layout variant, threads in TIME order (coalesced IR stores; the 12 band loads of a thread are
// issued together).  grid = (ceil(leff / 256), items)
__global__ void shape_ir_pp_kernel(const float2* __restrict__ C, const float* __restrict__ params, float2* __restrict__ Hb,
                                   int64_t L, int64_t leff, int jb, int R, int nb) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t il = blockIdx.y;
  __shared__ float gk[kBands], rk[kBands];
  if (threadIdx.x < kBands) {
    gk[threadIdx.x] = params[il * 25 + threadIdx.x] * (1.0f / kBands);
    rk[threadIdx.x] = -(params[il * 25 + kBands + threadIdx.x] * 10.0f + 1.0f);
  }
  __syncthreads();
  if (t >= leff) return;
  const int a = t / R, ph = t - a * R;
  const float tt = time_axis(t, L, 1.0f / (float)(L - 1));
  const float2* c0 = C + ((il * kBands) * (int64_t)R + ph) * nb + a;
  float2 v[kBands];
#pragma unroll
  for (int k = 0; k < kBands; ++k) v[k] = c0[(int64_t)k * R * nb];
  float al = 0.f, ar = 0.f;
#pragma unroll
  for (int k = 0; k < kBands; ++k) {
    const float e = gk[k] * __expf(rk[k] * tt);
    al = fmaf(e, v[k].x, al);
    ar = fmaf(e, v[k].y, ar);
  }
  Hb[il * (int64_t)jb * kNbA + (t / kB) * kNbA + (t % kB)] = make_float2(al, ar);
}

// ---- inverse FFT + envelope / gain / band mean as one kernel (device-noise mode, nb == 8192) -----------
// Replaces the batched cuFFT C2C + shape_ir_pp_kernel pair: the generator's spectrum is read ONCE (bulk copies
// straight into the planar shared-memory layout of fft8192.cuh, double buffered across the 12 bands), transformed
// in shared memory, and each thread accumulates  gain_k env_k(t) f_k(t) / 12  for its 16 taps in registers.  The
// filtered noise f is written back (over the consumed spectrum block, as (left, right) pairs) only when the
// backward needs it.  grid = (R, items): CTA (c, item) owns polyphase class c, i.e. the IR taps R a + c.
constexpr int kFusedThreads = fft8k::kThreads;
constexpr int kFusedSmemFloats = 2 * 2 * fft8k::kPlaneG + 2 * fft8k::kPlaneY + fft8k::kTabFloats + 32;
constexpr size_t kFftSmemBytes = sizeof(float) * kFusedSmemFloats + 2 * sizeof(uint64_t);   // + the two mbarriers

__global__ void __launch_bounds__(kFusedThreads, 1)
ifft_shape_kernel(float* __restrict__ Cpl, const float* __restrict__ twiddles, const float* __restrict__ params,
                  float2* __restrict__ Hb, int save_f, int L, int leff, int jb, int R) {
  constexpr int nb = fft8k::kN;
  extern __shared__ __align__(128) float sm[];
  float* G = sm;                                   // [buffer][re, im][8192]
  float* Yr = sm + 4 * fft8k::kPlaneG;
  float* Yi = Yr + fft8k::kPlaneY;
  float* tabf = Yi + fft8k::kPlaneY;
  float* gk = tabf + fft8k::kTabFloats;
  float* rk = gk + 16;
  uint64_t* full = reinterpret_cast<uint64_t*>(rk + 16);
  const int t = threadIdx.x, c = blockIdx.x;
  const int64_t il = blockIdx.y;
  float* blk = Cpl + ((il * kBands) * R + c) * (int64_t)(2 * nb);      // band k at blk + k * R * 2 nb
  const int64_t band_stride = (int64_t)R * 2 * nb;

  if (t == 0) {
    mbar_init(&full[0], 1);
    mbar_init(&full[1], 1);
    fence_barrier_init();
  }
  for (int e = t; e < fft8k::kTabFloats; e += kFusedThreads) tabf[e] = twiddles[e];
  if (t < kBands) {
    gk[t] = params[il * 25 + t] * (1.0f / kBands);
    rk[t] = -(params[il * 25 + kBands + t] * 10.0f + 1.0f);
  }
  __syncthreads();
  auto fetch = [&](int k) {                        // thread 0: 64 KB spectrum block of band k -> G[k & 1]
    uint64_t* bar = &full[k & 1];
    float* dst = G + (k & 1) * 2 * fft8k::kPlaneG;
    const float* src = blk + k * band_stride;
    mbar_arrive_expect_tx(bar, 2u * nb * 4u);
#pragma unroll
    for (int i = 0; i < 4; ++i) tma_load_1d(dst + i * 4096, src + i * 4096, 16384u, bar);
  };
  if (t == 0) { fetch(0); fetch(1); }
  const fft8k::Tables tb = fft8k::carve_tables(tabf);
  const float step = 1.0f / (float)(L - 1);
  float accr[16], acci[16];
#pragma unroll
  for (int q = 0; q < 16; ++q) { accr[q] = 0.f; acci[q] = 0.f; }

  for (int k = 0; k < kBands; ++k) {
    mbar_wait(&full[k & 1], (uint32_t)((k >> 1) & 1));
    float* gr = G + (k & 1) * 2 * fft8k::kPlaneG;
    float* gi = gr + fft8k::kPlaneG;
    fft8k::p1<true>(gr, gi, tb, t);
    __syncthreads();
    fft8k::p2<true>(gr, gi, Yr, Yi, tb, t);
    fence_proxy_async_smem();                      // pass-1 stores to G (generic proxy) before the bulk refill
    __syncthreads();
    if (t == 0 && k + 2 < kBands) fetch(k + 2);
    fft8k::P3Regs q3;
    fft8k::p3_load<true>(Yr, Yi, t, q3);
    __syncthreads();
    fft8k::p3_store<true>(Yr, Yi, tb, t, q3);
    __syncthreads();
    float xr[16], xi[16];
    fft8k::p4<true>(Yr, Yi, t, xr, xi);
    float e_prev = 0.f;
    const float g = gk[k], rr = rk[k];
    float2* fout = reinterpret_cast<float2*>(blk + k * band_stride);
    // envelope gain_k exp(rr tt(tau)) at the thread's taps tau_q = R (t + 512 q) + c: evaluated at every 4th tap,
    // the three taps in between follow by the constant ratio exp(rr step 512 R) (tt is linear in tau up to fp32
    // rounding of the linspace, so this stays within ~1e-6 of the per-tap evaluation)
    const float rho = __expf(rr * step * (float)(512 * R));
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      const int a = t + 512 * q;
      float e;
      if ((q & 3) == 0) e = g * __expf(rr * time_axis32(R * a + c, L, step));
      else e = e_prev * rho;
      e_prev = e;
      accr[q] = fmaf(e, xr[q], accr[q]);
      acci[q] = fmaf(e, xi[q], acci[q]);
      if (save_f) fout[a] = make_float2(xr[q], xi[q]);
    }
    // (Y is next written by pass 2 of the following band, behind the barrier after its pass 1)
  }
  float2* out = Hb + il * (int64_t)jb * kNbA;
#pragma unroll
  for (int q = 0; q < 16; ++q) {
    const int tau = R * (t + 512 * q) + c;
    if (tau < leff) out[(tau / kB) * kNbA + (tau % kB)] = make_float2(accr[q], acci[q]);
  }
}

// ---- block transforms of the audio convolution on the same in-shared-memory FFT ---------------------------
// Persistent CTAs (one per SM) walk the (item, block) list; the input of block m + 2 is bulk-copied into the free
// half of the double buffer while block m is transformed, so the copy engine, the FFT and the epilogue stores overlap.
struct FftSmem {
  float* G; float* Yr; float* Yi; float* tabf; uint64_t* full;
  __device__ __forceinline__ explicit FftSmem(float* sm) {
    G = sm;
    Yr = sm + 4 * fft8k::kPlaneG;
    Yi = Yr + fft8k::kPlaneY;
    tabf = Yi + fft8k::kPlaneY;
    full = reinterpret_cast<uint64_t*>(tabf + fft8k::kTabFloats + 32);
  }
  __device__ __forceinline__ void init(const float* twiddles, int t) {
    if (t == 0) {
      mbar_init(&full[0], 1);
      mbar_init(&full[1], 1);
      fence_barrier_init();
    }
    for (int e = t; e < fft8k::kTabFloats; e += kFusedThreads) tabf[e] = twiddles[e];
    __syncthreads();
  }
};
// the four passes on buffer (gr, gi); `refill()` runs as soon as nobody reads the buffer any more, `early()` two
// passes before the results exist (the place to issue global loads the epilogue needs, so that their latency is
// covered by passes 3 and 4 -- with one lock-stepped CTA per SM nothing else would hide it)
template <bool INV, class Refill, class Early>
__device__ __forceinline__ void fft8192_in_smem(float* gr, float* gi, const FftSmem& s, const fft8k::Tables& tb, int t,
                                                Refill&& refill, Early&& early, float (&xr)[16], float (&xi)[16]) {
  fft8k::p1<INV>(gr, gi, tb, t);
  __syncthreads();
  fft8k::p2<INV>(gr, gi, s.Yr, s.Yi, tb, t);
  fence_proxy_async_smem();                        // pass-1 stores to G (generic proxy) before the bulk refill
  __syncthreads();
  refill();
  fft8k::P3Regs q3;
  fft8k::p3_load<INV>(s.Yr, s.Yi, t, q3);
  __syncthreads();
  early();
  fft8k::p3_store<INV>(s.Yr, s.Yi, tb, t, q3);
  __syncthreads();
  fft8k::p4<INV>(s.Yr, s.Yi, t, xr, xi);
}

// Xb[(il*I + i)*kNbA + f] = FFT of the window (x_left + i x_right)[(i-1) kB + m], m < kNbA  (zero outside [0, n)):
// x_blocks_kernel + forward C2C in one kernel.  Requires n % 4 == 0 and 16-byte aligned rows (bulk copies).
__global__ void __launch_bounds__(kFusedThreads, 1)
x_fft_kernel(const float* __restrict__ x, float2* __restrict__ Xb, const float* __restrict__ twiddles, int64_t item0,
             int I, int64_t n, int in_chs, int nblocks) {
  extern __shared__ __align__(128) float sm[];
  FftSmem s(sm);
  const int t = threadIdx.x;
  s.init(twiddles, t);
  const fft8k::Tables tb = fft8k::carve_tables(s.tabf);
  auto fetch = [&](int it, int m) {                // all threads: zero padding; thread 0: the bulk copies
    if (m >= nblocks) return;
    const int64_t il = m / I;
    const int i = m - (int)il * I;
    float* re = s.G + (it & 1) * 2 * fft8k::kPlaneG;
    float* im = re + fft8k::kPlaneG;
    const int64_t s0 = (int64_t)(i - 1) * kB;      // first sample of the window
    const int lo = (i == 0) ? kB : 0;
    const int64_t rem = n - s0;
    const int hi = rem < kNbA ? (int)rem : kNbA;   // valid window samples are [lo, hi)
    for (int e = t; e < lo; e += kFusedThreads) { re[e] = 0.f; im[e] = 0.f; }
    for (int e = hi + t; e < kNbA; e += kFusedThreads) { re[e] = 0.f; im[e] = 0.f; }
    if (t == 0) {
      const float* xl = x + ((item0 + il) * in_chs) * n + s0;
      const float* xr = in_chs == 1 ? xl : xl + n;
      uint64_t* bar = &s.full[it & 1];
      mbar_arrive_expect_tx(bar, 2u * (uint32_t)(hi - lo) * 4u);
      for (int o = lo; o < hi; o += 4096) {
        const uint32_t bytes = (uint32_t)((hi - o < 4096 ? hi - o : 4096) * 4);
        tma_load_1d(re + o, xl + o, bytes, bar);
        tma_load_1d(im + o, xr + o, bytes, bar);
      }
    }
  };
  fetch(0, blockIdx.x);
  fetch(1, blockIdx.x + gridDim.x);
  __syncthreads();                                 // the zero padding of the first two buffers is in place
  int it = 0;
  for (int m = blockIdx.x; m < nblocks; m += gridDim.x, ++it) {
    mbar_wait(&s.full[it & 1], (uint32_t)((it >> 1) & 1));
    float* gr = s.G + (it & 1) * 2 * fft8k::kPlaneG;
    float xr[16], xi[16];
    fft8192_in_smem<false>(gr, gr + fft8k::kPlaneG, s, tb, t, [&] { fetch(it + 2, m + 2 * gridDim.x); }, [] {}, xr, xi);
    float2* out = Xb + (int64_t)m * kNbA;
#pragma unroll
    for (int q = 0; q < 16; ++q) out[t + 512 * q] = make_float2(xr[q], xi[q]);
  }
}

// inverse C2C of the (planar) product spectra + mix_blocks_kernel in one kernel: block i of item il yields the wet
// samples [i kB, (i+1) kB) as the second half of the transform; y = x + mix (wet - x).
__global__ void __launch_bounds__(kFusedThreads, 1)
ifft_mix_kernel(const float* __restrict__ Ypl, const float* __restrict__ twiddles, const float* __restrict__ x,
                const float* __restrict__ params, float* __restrict__ y, float* __restrict__ wet_save, int64_t item0,
                int I, int64_t n, int in_chs, int nblocks) {
  extern __shared__ __align__(128) float sm[];
  FftSmem s(sm);
  const int t = threadIdx.x;
  s.init(twiddles, t);
  const fft8k::Tables tb = fft8k::carve_tables(s.tabf);
  auto fetch = [&](int it, int m) {
    if (t != 0 || m >= nblocks) return;
    uint64_t* bar = &s.full[it & 1];
    float* dst = s.G + (it & 1) * 2 * fft8k::kPlaneG;
    const float* src = Ypl + (int64_t)m * 2 * kNbA;
    mbar_arrive_expect_tx(bar, 2u * kNbA * 4u);
#pragma unroll
    for (int q = 0; q < 4; ++q) tma_load_1d(dst + q * 4096, src + q * 4096, 16384u, bar);
  };
  fetch(0, blockIdx.x);
  fetch(1, blockIdx.x + gridDim.x);
  int it = 0;
  for (int m = blockIdx.x; m < nblocks; m += gridDim.x, ++it) {
    mbar_wait(&s.full[it & 1], (uint32_t)((it >> 1) & 1));
    float* gr = s.G + (it & 1) * 2 * fft8k::kPlaneG;
    float xr[16], xi[16];
    const int64_t il = m / I, b = item0 + il;
    const int i = m - (int)il * I;
    const float mix = params[b * 25 + 24];
    const float* xl = x + (b * in_chs) * n;
    const float* xrr = in_chs == 1 ? xl : xl + n;
    float a0[8], a1[8];                            // the dry samples of this thread's 8 outputs
    fft8192_in_smem<true>(gr, gr + fft8k::kPlaneG, s, tb, t, [&] { fetch(it + 2, m + 2 * gridDim.x); },
                          [&] {
#pragma unroll
                            for (int q = 0; q < 8; ++q) {
                              const int64_t tg = (int64_t)i * kB + (t + 512 * q);
                              a0[q] = tg < n ? xl[tg] : 0.f;
                              a1[q] = tg < n ? xrr[tg] : 0.f;
                            }
                          },
                          xr, xi);
#pragma unroll
    for (int q = 8; q < 16; ++q) {                 // outputs kB .. 2 kB - 1 of the transform
      const int64_t tg = (int64_t)i * kB + (t + 512 * q - kB);
      if (tg < n) {
        y[(b * 2 + 0) * n + tg] = fmaf(mix, xr[q] - a0[q - 8], a0[q - 8]);
        y[(b * 2 + 1) * n + tg] = fmaf(mix, xi[q] - a1[q - 8], a1[q - 8]);
        if (wet_save) { wet_save[(b * 2 + 0) * n + tg] = xr[q]; wet_save[(b * 2 + 1) * n + tg] = xi[q]; }
      }
    }
  }
}

// ---- the backward's block transforms on the same in-shared-memory FFT --------------------------------------
// g_fft_kernel     = g_blocks_kernel + forward C2C:  Gs[i] = FFT([0 .. 0 | mix g block i]),  + dL/dmix partials
// ifft_dx_kernel   = inverse C2C + finish_dx_blocks_kernel: one CTA walks the windows of an item in order and keeps
//                    the second half of window i in registers until the first half of window i + 1 arrives, so the
//                    overlap-add of the two windows that cover a sample needs no second pass and no atomics
// ifft_irgrad_kernel = inverse C2C of the dL/dIR partitions + ir_grad_pp_kernel: the 4096 taps of a partition go to
//                    shared memory and are correlated with the filtered noise f read class by class (coalesced)

// Gb[(il*I + i)*kNbA + f] = FFT of [zeros(kB) | mix (g_left + i g_right)[i kB + m], m < kB];
// mix_part[il*I + i] = sum over the block and both channels of g (wet - x)
__global__ void __launch_bounds__(kFusedThreads, 1)
g_fft_kernel(const float* __restrict__ gy, const float* __restrict__ x, const float* __restrict__ wet,
             const float* __restrict__ params, float2* __restrict__ Gb, float* __restrict__ mix_part,
             const float* __restrict__ twiddles, int64_t item0, int I, int64_t n, int in_chs, int nblocks) {
  extern __shared__ __align__(128) float sm[];
  FftSmem s(sm);
  __shared__ float wp[kFusedThreads / 32];
  const int t = threadIdx.x;
  s.init(twiddles, t);
  const fft8k::Tables tb = fft8k::carve_tables(s.tabf);
  auto fetch = [&](int it, int m) {                // all threads: zero padding; thread 0: the bulk copies
    if (m >= nblocks) return;
    const int64_t il = m / I;
    const int i = m - (int)il * I;
    float* re = s.G + (it & 1) * 2 * fft8k::kPlaneG;
    float* im = re + fft8k::kPlaneG;
    const int64_t s0 = (int64_t)i * kB;            // first sample of the block (lands at offset kB of the window)
    const int64_t rem = n - s0;
    const int len = rem < kB ? (int)rem : kB;
    for (int e = t; e < kB; e += kFusedThreads) { re[e] = 0.f; im[e] = 0.f; }
    for (int e = kB + len + t; e < kNbA; e += kFusedThreads) { re[e] = 0.f; im[e] = 0.f; }
    if (t == 0) {
      const float* gl = gy + ((item0 + il) * 2) * n + s0;
      uint64_t* bar = &s.full[it & 1];
      mbar_arrive_expect_tx(bar, 2u * (uint32_t)len * 4u);
      tma_load_1d(re + kB, gl, (uint32_t)len * 4u, bar);
      tma_load_1d(im + kB, gl + n, (uint32_t)len * 4u, bar);
    }
  };
  fetch(0, blockIdx.x);
  fetch(1, blockIdx.x + gridDim.x);
  __syncthreads();
  int it = 0;
  for (int m = blockIdx.x; m < nblocks; m += gridDim.x, ++it) {
    mbar_wait(&s.full[it & 1], (uint32_t)((it >> 1) & 1));
    float* gr = s.G + (it & 1) * 2 * fft8k::kPlaneG;
    const int64_t il = m / I, b = item0 + il;
    const int i = m - (int)il * I;
    const float mix = params[b * 25 + 24];
    // dL/dmix partial: the block's g sits in shared memory (second half of the planes), wet and x come from HBM
    float acc = 0.f;
    {
      const float* xl = x + (b * in_chs) * n;
      const float* xr = in_chs == 1 ? xl : xl + n;
      const float* wl = wet + (b * 2) * n;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const int mm = t + 512 * q;
        const int64_t tg = (int64_t)i * kB + mm;
        if (tg < n) {
          const float g0 = gr[kB + mm], g1 = gr[fft8k::kPlaneG + kB + mm];
          acc = fmaf(g0, wl[tg] - xl[tg], fmaf(g1, wl[n + tg] - xr[tg], acc));
        }
      }
    }
    __syncthreads();                                 // pass 1 transforms the planes in place
    float xr_[16], xi_[16];
    fft8192_in_smem<false>(gr, gr + fft8k::kPlaneG, s, tb, t, [&] { fetch(it + 2, m + 2 * gridDim.x); }, [] {}, xr_, xi_);
    float2* out = Gb + (int64_t)m * kNbA;
#pragma unroll
    for (int q = 0; q < 16; ++q) out[t + 512 * q] = make_float2(mix * xr_[q], mix * xi_[q]);
    acc = warp_sum(acc);
    if ((t & 31) == 0) wp[t >> 5] = acc;
    __syncthreads();
    if (t == 0) {
      float sum = 0.f;
#pragma unroll
      for (int w = 0; w < kFusedThreads / 32; ++w) sum += wp[w];
      mix_part[m] = sum;
    }
    // (wp is next written after the barriers inside the following transform)
  }
}

// gx[t] = (1-mix) g[t] + D[q][kB + t - q kB] + D[q+1][t - q kB], q = t / kB, from the planar product spectra Dpl
// (one CTA per item at a time; mono input receives the sum of both channel gradients)
__global__ void __launch_bounds__(kFusedThreads, 1)
ifft_dx_kernel(const float* __restrict__ Dpl, const float* __restrict__ twiddles, const float* __restrict__ gy,
               const float* __restrict__ params, float* __restrict__ gx, int64_t item0, int items, int I, int64_t n,
               int in_chs) {
  extern __shared__ __align__(128) float sm[];
  FftSmem s(sm);
  const int t = threadIdx.x;
  s.init(twiddles, t);
  const fft8k::Tables tb = fft8k::carve_tables(s.tabf);
  // work list of this CTA: windows (il, i), il = blockIdx.x, blockIdx.x + gridDim.x, ..., i = 0 .. I-1
  const int my_items = (items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int total = my_items * I;
  auto fetch = [&](int it) {
    if (t != 0 || it >= total) return;
    const int64_t il = blockIdx.x + (int64_t)(it / I) * gridDim.x;
    const int i = it % I;
    uint64_t* bar = &s.full[it & 1];
    float* dst = s.G + (it & 1) * 2 * fft8k::kPlaneG;
    const float* src = Dpl + (il * I + i) * (int64_t)(2 * kNbA);
    mbar_arrive_expect_tx(bar, 2u * kNbA * 4u);
#pragma unroll
    for (int q = 0; q < 4; ++q) tma_load_1d(dst + q * 4096, src + q * 4096, 16384u, bar);
  };
  fetch(0);
  fetch(1);
  float pr[8], pi[8];                                // second half of the previous window of this item
  for (int it = 0; it < total; ++it) {
    mbar_wait(&s.full[it & 1], (uint32_t)((it >> 1) & 1));
    float* gr = s.G + (it & 1) * 2 * fft8k::kPlaneG;
    const int64_t il = blockIdx.x + (int64_t)(it / I) * gridDim.x, b = item0 + il;
    const int i = it % I;
    const float mix = params[b * 25 + 24];
    const float* g0p = gy + (b * 2) * n;
    // the block finished by this window is i - 1 (its first half); after the last window also block I - 1
    float ga[8], gb[8];
    float xr[16], xi[16];
    fft8192_in_smem<true>(gr, gr + fft8k::kPlaneG, s, tb, t, [&] { fetch(it + 2); },
                          [&] {
#pragma unroll
                            for (int q = 0; q < 8; ++q) {
                              const int64_t t0 = (int64_t)(i - 1) * kB + (t + 512 * q);
                              ga[q] = (i > 0 && t0 < n) ? g0p[t0] : 0.f;
                              gb[q] = (i > 0 && t0 < n) ? g0p[n + t0] : 0.f;
                            }
                          },
                          xr, xi);
    const float om = 1.0f - mix;
    if (i > 0) {
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const int64_t tg = (int64_t)(i - 1) * kB + (t + 512 * q);
        if (tg < n) {
          const float o0 = fmaf(om, ga[q], pr[q] + xr[q]), o1 = fmaf(om, gb[q], pi[q] + xi[q]);
          if (in_chs == 1) gx[b * n + tg] = o0 + o1;
          else { gx[(b * 2) * n + tg] = o0; gx[(b * 2 + 1) * n + tg] = o1; }
        }
      }
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) { pr[q] = xr[q + 8]; pi[q] = xi[q + 8]; }
    if (i == I - 1) {
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const int64_t tg = (int64_t)i * kB + (t + 512 * q);
        if (tg < n) {
          const float o0 = fmaf(om, g0p[tg], pr[q]), o1 = fmaf(om, g0p[n + tg], pi[q]);
          if (in_chs == 1) gx[b * n + tg] = o0 + o1;
          else { gx[(b * 2) * n + tg] = o0; gx[(b * 2 + 1) * n + tg] = o1; }
        }
      }
    }
  }
}

// unit (il, j): dIR taps [j kB, (j+1) kB) = first half of IFFT(Epl[il][j]) (left, right);
// part[((il*J + j)*12 + k)*2 + {0,1}] = sum_t (dIR_l f_l + dIR_r f_r) env_k(t) {1, tt(t)}  over the partition's taps,
// f in the polyphase layout C[((il*12 + k)*R + c)*nb + a] = f[R a + c].
__global__ void __launch_bounds__(kFusedThreads, 1)
ifft_irgrad_kernel(const float* __restrict__ Epl, const float* __restrict__ twiddles, const float2* __restrict__ C,
                   const float* __restrict__ params /* chunk x 25 */, float* __restrict__ part, int L, int leff, int J,
                   int R, int nunits) {
  constexpr int nb = fft8k::kN;
  extern __shared__ __align__(128) float sm[];
  FftSmem s(sm);
  __shared__ float red[kFusedThreads / 32][2 * kBands];
  __shared__ float rk[kBands];
  __shared__ int cls_lo[17], cls_off[17];            // per class: first a of the partition, prefix count of taps
  const int t = threadIdx.x;
  s.init(twiddles, t);
  const fft8k::Tables tb = fft8k::carve_tables(s.tabf);
  auto fetch = [&](int it, int m) {
    if (t != 0 || m >= nunits) return;
    uint64_t* bar = &s.full[it & 1];
    float* dst = s.G + (it & 1) * 2 * fft8k::kPlaneG;
    const float* src = Epl + (int64_t)m * 2 * kNbA;
    mbar_arrive_expect_tx(bar, 2u * kNbA * 4u);
#pragma unroll
    for (int q = 0; q < 4; ++q) tma_load_1d(dst + q * 4096, src + q * 4096, 16384u, bar);
  };
  fetch(0, blockIdx.x);
  fetch(1, blockIdx.x + gridDim.x);
  const float step = 1.0f / (float)(L - 1);
  float2* D = reinterpret_cast<float2*>(s.Yr);        // the partition's taps, after pass 4 has consumed Y
  int it = 0;
  for (int m = blockIdx.x; m < nunits; m += gridDim.x, ++it) {
    mbar_wait(&s.full[it & 1], (uint32_t)((it >> 1) & 1));
    float* gr = s.G + (it & 1) * 2 * fft8k::kPlaneG;
    const int64_t il = m / J;
    const int j = m - (int)il * J;
    const int lo = j * kB, hi = (lo + kB < leff) ? lo + kB : leff;      // taps [lo, hi)
    float xr[16], xi[16];
    fft8192_in_smem<true>(gr, gr + fft8k::kPlaneG, s, tb, t, [&] { fetch(it + 2, m + 2 * gridDim.x); }, [] {}, xr, xi);
    __syncthreads();                                  // every thread is done reading Y (pass 4) and the previous unit's D
    if (t < kBands) rk[t] = -(params[il * 25 + kBands + t] * 10.0f + 1.0f);
    if (t == 0) {
      int off = 0;
      for (int c = 0; c < R; ++c) {
        const int a_lo = (lo - c + R - 1) / R, a_hi = (hi - c + R - 1) / R;      // taps R a + c in [lo, hi)
        cls_lo[c] = a_lo;
        cls_off[c] = off;
        off += (a_hi > a_lo) ? a_hi - a_lo : 0;
      }
      cls_off[R] = off;
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) D[t + 512 * q] = make_float2(xr[q], xi[q]);
    __syncthreads();
    float s0[kBands], s1[kBands];
#pragma unroll
    for (int k = 0; k < kBands; ++k) { s0[k] = 0.f; s1[k] = 0.f; }
    const float2* cb = C + (il * kBands) * (int64_t)R * nb;
    const int ntaps = cls_off[R];
    for (int idx = t; idx < ntaps; idx += kFusedThreads) {
      int c = 0;
      while (c + 1 < R && idx >= cls_off[c + 1]) ++c;
      const int a = cls_lo[c] + (idx - cls_off[c]);
      const int tau = R * a + c;
      const float2 gd = D[tau - lo];
      const float tt = time_axis32(tau, L, step);
      const float2* c0 = cb + (int64_t)c * nb + a;
      float2 v[kBands];
#pragma unroll
      for (int k = 0; k < kBands; ++k) v[k] = c0[(int64_t)k * R * nb];
#pragma unroll
      for (int k = 0; k < kBands; ++k) {
        const float w = fmaf(gd.x, v[k].x, gd.y * v[k].y) * __expf(rk[k] * tt);
        s0[k] += w;
        s1[k] = fmaf(w, tt, s1[k]);
      }
    }
    const int lane = t & 31, warp = t >> 5;
#pragma unroll
    for (int k = 0; k < kBands; ++k) {
      const float x0 = warp_sum(s0[k]), x1 = warp_sum(s1[k]);
      if (lane == 0) { red[warp][2 * k] = x0; red[warp][2 * k + 1] = x1; }
    }
    __syncthreads();
    if (t < 2 * kBands) {
      float acc = 0.f;
#pragma unroll
      for (int w = 0; w < kFusedThreads / 32; ++w) acc += red[w][t];
      part[((int64_t)m * kBands) * 2 + t] = acc;
    }
    // red / rk / cls_* / D are rewritten only after the __syncthreads that follows the next transform
  }
}

// part[((item*nparts + blockIdx.x)*12 + k)*2 + {0,1}], nparts = gridDim.x; threads stride over time
__global__ void ir_grad_pp_kernel(const float2* __restrict__ Et, const float2* __restrict__ C,
                                  const float* __restrict__ params, float* __restrict__ part, int64_t L, int64_t leff,
                                  int jb, int R, int nb) {
  const int64_t il = blockIdx.y;
  __shared__ float rk[kBands];
  __shared__ float red[8][2 * kBands];
  if (threadIdx.x < kBands) rk[threadIdx.x] = -(params[il * 25 + kBands + threadIdx.x] * 10.0f + 1.0f);
  __syncthreads();
  const float step = 1.0f / (float)(L - 1);
  const float2* de = Et + il * (int64_t)jb * kNbA;       // dL/dIR (left, right) in the first half of partition t/kB
  const float2* cb = C + (il * kBands) * (int64_t)R * nb;
  float s0[kBands], s1[kBands];
#pragma unroll
  for (int k = 0; k < kBands; ++k) { s0[k] = 0.f; s1[k] = 0.f; }
  // two time points per iteration: 24 independent 8-byte loads in flight per thread
  const int stride = gridDim.x * blockDim.x;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < leff; t += 2 * stride) {
    const int t2 = t + stride;
    const bool has2 = t2 < leff;
    const int a = t / R, ph = t - a * R;
    const int a2 = has2 ? t2 / R : a, ph2 = has2 ? t2 - a2 * R : ph;
    const float2 gd = de[(t / kB) * kNbA + (t % kB)];
    const float2 gd2 = has2 ? de[(t2 / kB) * kNbA + (t2 % kB)] : make_float2(0.f, 0.f);
    const float2* c0 = cb + (int64_t)ph * nb + a;
    const float2* c1 = cb + (int64_t)ph2 * nb + a2;
    float2 v[kBands], v2[kBands];
#pragma unroll
    for (int k = 0; k < kBands; ++k) { v[k] = c0[(int64_t)k * R * nb]; v2[k] = c1[(int64_t)k * R * nb]; }
    const float tt = time_axis(t, L, step), tt2 = time_axis(has2 ? t2 : t, L, step);
#pragma unroll
    for (int k = 0; k < kBands; ++k) {
      const float w = fmaf(gd.x, v[k].x, gd.y * v[k].y) * __expf(rk[k] * tt);
      const float w2 = fmaf(gd2.x, v2[k].x, gd2.y * v2[k].y) * __expf(rk[k] * tt2);
      s0[k] += w + w2;
      s1[k] = fmaf(w, tt, fmaf(w2, tt2, s1[k]));
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < kBands; ++k) {
    const float x0 = warp_sum(s0[k]), x1 = warp_sum(s1[k]);
    if (lane == 0) { red[warp][2 * k] = x0; red[warp][2 * k + 1] = x1; }
  }
  __syncthreads();
  if (threadIdx.x < 2 * kBands) {
    float acc = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) acc += red[w][threadIdx.x];
    part[((il * gridDim.x + blockIdx.x) * kBands) * 2 + threadIdx.x] = acc;
  }
}

// ---- audio convolution: uniformly partitioned overlap-save in the frequency domain -----------------
// y[n] = sum_{t<=n} IR[t] x[n-t] (n < N) with the IR split into J partitions of kB taps and the audio into
// I blocks of kB samples; every transform is the fast single-kernel kNbA-point batched C2C, with the LEFT
// and RIGHT channel packed as real/imag (the channels have different IRs, so the multiply kernels untangle
// the packed spectra through their Hermitian symmetry and re-pack the products).
//   Xs[i] = FFT(x window [(i-1) kB, (i+1) kB)),  Hs[j] = FFT(IR[j kB, (j+1) kB) zero padded)
//   y block i = last kB samples of IFFT(sum_{j<=i} Xs[i-j] Hs[j]) / kNbA
// Backward: Gs[i] = FFT(mix g block i, in the second half), dx windows = IFFT(sum_j conj(Hs[j]) Gs[q+j]),
//   dIR partition j = first kB samples of IFFT(sum_i conj(Xs[i-j]) Gs[i]).

// Xb[(il*I + i)*kNbA + m] = (x_left, x_right)[(i-1) kB + m]
__global__ void x_blocks_kernel(const float* __restrict__ x, float2* __restrict__ Xb, int64_t item0, int I, int64_t n,
                                int in_chs) {
  const int i = blockIdx.x;
  const int64_t il = blockIdx.y;
  const float* xl = x + ((item0 + il) * in_chs) * n;
  const float* xr = in_chs == 1 ? xl : xl + n;
  float2* out = Xb + (il * I + i) * (int64_t)kNbA;
  for (int m = threadIdx.x; m < kNbA; m += blockDim.x) {
    const int64_t idx = (int64_t)(i - 1) * kB + m;
    float2 v = make_float2(0.f, 0.f);
    if (idx >= 0 && idx < n) v = make_float2(xl[idx], xr[idx]);
    out[m] = v;
  }
}

// packed spectrum of (a + i b), a and b real: A[f] = (Z[f] + conj(Z[-f]))/2, B[f] = (Z[f] - conj(Z[-f]))/(2i)
__device__ __forceinline__ void untangle(float2 z, float2 zm, float2& a, float2& b) {
  a = make_float2(0.5f * (z.x + zm.x), 0.5f * (z.y - zm.y));
  b = make_float2(0.5f * (z.y + zm.y), -0.5f * (z.x - zm.x));
}
__device__ __forceinline__ void cfma(float2& acc, float2 p, float2 q) {          // acc += p q
  acc.x = fmaf(p.x, q.x, fmaf(-p.y, q.y, acc.x));
  acc.y = fmaf(p.x, q.y, fmaf(p.y, q.x, acc.y));
}
__device__ __forceinline__ void cfma_conj(float2& acc, float2 p, float2 q) {     // acc += p conj(q)
  acc.x = fmaf(p.x, q.x, fmaf(p.y, q.y, acc.x));
  acc.y = fmaf(p.y, q.x, fmaf(-p.x, q.y, acc.y));
}

// CORR == false: out[o] = sum_{j<nbm, j<=o} A[o-j] B[j]           (o < nout)      forward
// CORR == true : out[o] = sum_{j<nbm, o+j<na} A[o+j] conj(B[j])   (o < nout)      both backward products
// A: [items][na][kNbA], Bm: [items][nbm][kNbA], Out: [items][nout][kNbA]; per channel, packed spectra.
// grid = (ceil((kNbA/2+1)/128), items); thread = frequency pair (f, kNbA - f).  MAXB > 0: operands cached
// in registers (na, nbm <= MAXB); MAXB == 0: generic loop straight from L2.
// PLANAR: every output block is stored as [re plane kNbA][im plane kNbA] (what ifft_mix_kernel bulk-copies into the
// shared-memory layout of fft8192.cuh) instead of (re, im) pairs (what cuFFT reads).
template <int MAXB, bool CORR, bool PLANAR = false>
__global__ void __launch_bounds__(128) partition_mac_kernel(const float2* __restrict__ A, const float2* __restrict__ Bm,
                                                            float2* __restrict__ Out, int na, int nbm, int nout,
                                                            float scale) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f > kNbA / 2) return;
  const int fm = (kNbA - f) & (kNbA - 1);
  const int64_t il = blockIdx.y;
  const float2* a = A + il * (int64_t)na * kNbA;
  const float2* bq = Bm + il * (int64_t)nbm * kNbA;
  float2* out = Out + il * (int64_t)nout * kNbA;
  auto emit = [&](int o, float2 sl, float2 sr) {
    sl.x *= scale; sl.y *= scale; sr.x *= scale; sr.y *= scale;
    if (PLANAR) {
      float* pl = reinterpret_cast<float*>(out + (int64_t)o * kNbA);
      pl[f] = sl.x - sr.y; pl[kNbA + f] = sl.y + sr.x;
      if (fm != f) { pl[fm] = sl.x + sr.y; pl[kNbA + fm] = sr.x - sl.y; }
    } else {
      out[(int64_t)o * kNbA + f] = make_float2(sl.x - sr.y, sl.y + sr.x);                 // L + i R
      if (fm != f) out[(int64_t)o * kNbA + fm] = make_float2(sl.x + sr.y, sr.x - sl.y);   // conj(L) + i conj(R)
    }
  };
  if constexpr (MAXB > 0) {
    float2 al[MAXB], ar[MAXB], bl[MAXB], br[MAXB];
#pragma unroll
    for (int i = 0; i < MAXB; ++i) {
      al[i] = ar[i] = bl[i] = br[i] = make_float2(0.f, 0.f);      // operands beyond na / nbm are zero
      if (i < na) untangle(a[(int64_t)i * kNbA + f], a[(int64_t)i * kNbA + fm], al[i], ar[i]);
      if (i < nbm) untangle(bq[(int64_t)i * kNbA + f], bq[(int64_t)i * kNbA + fm], bl[i], br[i]);
    }
#pragma unroll
    for (int o = 0; o < MAXB; ++o) {
      if (o < nout) {
        float2 sl = make_float2(0.f, 0.f), sr = make_float2(0.f, 0.f);
#pragma unroll
        for (int j = 0; j < MAXB; ++j) {
          const int ia = CORR ? o + j : o - j;                       // compile-time after unrolling
          if (ia >= 0 && ia < MAXB) {
            if (CORR) { cfma_conj(sl, al[ia], bl[j]); cfma_conj(sr, ar[ia], br[j]); }
            else      { cfma(sl, al[ia], bl[j]); cfma(sr, ar[ia], br[j]); }
          }
        }
        emit(o, sl, sr);
      }
    }
  } else {
    for (int o = 0; o < nout; ++o) {
      float2 sl = make_float2(0.f, 0.f), sr = make_float2(0.f, 0.f);
      for (int j = 0; j < nbm; ++j) {
        const int ia = CORR ? o + j : o - j;
        if (ia < 0 || ia >= na) continue;
        float2 pl, pr, ql, qr;
        untangle(a[(int64_t)ia * kNbA + f], a[(int64_t)ia * kNbA + fm], pl, pr);
        untangle(bq[(int64_t)j * kNbA + f], bq[(int64_t)j * kNbA + fm], ql, qr);
        if (CORR) { cfma_conj(sl, pl, ql); cfma_conj(sr, pr, qr); }
        else      { cfma(sl, pl, ql); cfma(sr, pr, qr); }
      }
      emit(o, sl, sr);
    }
  }
}

// Both correlation products of the backward in ONE pass over the gradient spectra (each was HBM bound on its own):
//   D[q] = sum_{j<J, q+j<I} G[q+j] conj(H[j])  (q < I)   dL/dx windows
//   E[j] = sum_{p<I, j+p<I} G[j+p] conj(X[p])  (j < J)   dL/dIR partitions
// G is read and untangled once; H and X take turns in the same registers.  Planar outputs (own inverse FFT kernels).
template <int MAXB>
__global__ void __launch_bounds__(128) partition_mac_bwd_kernel(const float2* __restrict__ G, const float2* __restrict__ H,
                                                                const float2* __restrict__ X, float2* __restrict__ D,
                                                                float2* __restrict__ E, int I, int J, float scale) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f > kNbA / 2) return;
  const int fm = (kNbA - f) & (kNbA - 1);
  const int64_t il = blockIdx.y;
  const float2* g = G + il * (int64_t)I * kNbA;
  float2 al[MAXB], ar[MAXB], bl[MAXB], br[MAXB];
#pragma unroll
  for (int i = 0; i < MAXB; ++i) {
    al[i] = ar[i] = make_float2(0.f, 0.f);
    if (i < I) untangle(g[(int64_t)i * kNbA + f], g[(int64_t)i * kNbA + fm], al[i], ar[i]);
  }
#pragma unroll
  for (int pass = 0; pass < 2; ++pass) {
    const float2* bq = (pass == 0 ? H + il * (int64_t)J * kNbA : X + il * (int64_t)I * kNbA);
    const int nbm = pass == 0 ? J : I, nout = pass == 0 ? I : J;
    float2* out = (pass == 0 ? D + il * (int64_t)I * kNbA : E + il * (int64_t)J * kNbA);
#pragma unroll
    for (int i = 0; i < MAXB; ++i) {
      bl[i] = br[i] = make_float2(0.f, 0.f);
      if (i < nbm) untangle(bq[(int64_t)i * kNbA + f], bq[(int64_t)i * kNbA + fm], bl[i], br[i]);
    }
#pragma unroll
    for (int o = 0; o < MAXB; ++o) {
      if (o < nout) {
        float2 sl = make_float2(0.f, 0.f), sr = make_float2(0.f, 0.f);
#pragma unroll
        for (int j = 0; j < MAXB; ++j) {
          if (o + j < MAXB) { cfma_conj(sl, al[o + j], bl[j]); cfma_conj(sr, ar[o + j], br[j]); }   // operands beyond I / nbm are zero
        }
        sl.x *= scale; sl.y *= scale; sr.x *= scale; sr.y *= scale;
        float* pl = reinterpret_cast<float*>(out + (int64_t)o * kNbA);
        pl[f] = sl.x - sr.y; pl[kNbA + f] = sl.y + sr.x;
        if (fm != f) { pl[fm] = sl.x + sr.y; pl[kNbA + fm] = sr.x - sl.y; }
      }
    }
  }
}

// y = (1-mix) x + mix wet; wet[n] = Yt[(il*I + n/kB)*kNbA + kB + n%kB]; also saves wet for the backward
__global__ void mix_blocks_kernel(const float* __restrict__ x, const float2* __restrict__ Yt,
                                  const float* __restrict__ params, float* __restrict__ y, float* __restrict__ wet_save,
                                  int64_t item0, int I, int64_t n, int in_chs) {
  const int i = blockIdx.x;
  const int64_t il = blockIdx.y, b = item0 + il;
  const float mix = params[b * 25 + 24];
  const float* xl = x + (b * in_chs) * n;
  const float* xr = in_chs == 1 ? xl : xl + n;
  const float2* yt = Yt + (il * I + i) * (int64_t)kNbA + kB;
  for (int m = threadIdx.x; m < kB; m += blockDim.x) {
    const int64_t t = (int64_t)i * kB + m;
    if (t >= n) break;
    const float2 w = yt[m];
    const float a0 = xl[t], a1 = xr[t];
    y[(b * 2 + 0) * n + t] = fmaf(mix, w.x - a0, a0);
    y[(b * 2 + 1) * n + t] = fmaf(mix, w.y - a1, a1);
    if (wet_save) { wet_save[(b * 2 + 0) * n + t] = w.x; wet_save[(b * 2 + 1) * n + t] = w.y; }
  }
}

// backward: Gb[(il*I + i)*kNbA + kB + m] = mix (g_left, g_right)[i kB + m], first half zero;
// mix_part[il*I + i] = sum over the block and both channels of g (wet - x)
__global__ void g_blocks_kernel(const float* __restrict__ gy, const float* __restrict__ x, const float* __restrict__ wet,
                                const float* __restrict__ params, float2* __restrict__ Gb, float* __restrict__ mix_part,
                                int64_t item0, int I, int64_t n, int in_chs) {
  const int i = blockIdx.x;
  const int64_t il = blockIdx.y, b = item0 + il;
  const float mix = params[b * 25 + 24];
  const float* xl = x + (b * in_chs) * n;
  const float* xr = in_chs == 1 ? xl : xl + n;
  const float* gl = gy + (b * 2 + 0) * n;
  const float* gr = gy + (b * 2 + 1) * n;
  const float* wl = wet + (b * 2 + 0) * n;
  const float* wr = wet + (b * 2 + 1) * n;
  float2* out = Gb + (il * I + i) * (int64_t)kNbA;
  float acc = 0.f;
  for (int m = threadIdx.x; m < kB; m += blockDim.x) {
    const int64_t t = (int64_t)i * kB + m;
    float2 v = make_float2(0.f, 0.f);
    if (t < n) {
      const float g0 = gl[t], g1 = gr[t];
      v = make_float2(mix * g0, mix * g1);
      acc = fmaf(g0, wl[t] - xl[t], fmaf(g1, wr[t] - xr[t], acc));
    }
    out[m] = make_float2(0.f, 0.f);
    out[kB + m] = v;
  }
  __shared__ float wp[32];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) wp[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float sum = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) sum += wp[w];
    mix_part[il * I + i] = sum;
  }
}

// gx[t] = (1-mix) g[t] + Dt[q][t - (q-1) kB] + Dt[q+1][t - q kB], q = t / kB (every sample sits in two windows);
// mono input receives the sum of both channel gradients
__global__ void finish_dx_blocks_kernel(const float* __restrict__ gy, const float2* __restrict__ Dt,
                                        const float* __restrict__ params, float* __restrict__ gx, int64_t item0, int I,
                                        int64_t n, int in_chs) {
  const int i = blockIdx.x;
  const int64_t il = blockIdx.y, b = item0 + il;
  const float mix = params[b * 25 + 24];
  const float2* d0 = Dt + (il * I + i) * (int64_t)kNbA + kB;
  const float2* d1 = (i + 1 < I) ? Dt + (il * I + i + 1) * (int64_t)kNbA : nullptr;
  for (int m = threadIdx.x; m < kB; m += blockDim.x) {
    const int64_t t = (int64_t)i * kB + m;
    if (t >= n) break;
    float2 v = d0[m];
    if (d1) { const float2 u = d1[m]; v.x += u.x; v.y += u.y; }
    const float g0 = gy[(b * 2 + 0) * n + t], g1 = gy[(b * 2 + 1) * n + t];
    const float o0 = fmaf(1.0f - mix, g0, v.x), o1 = fmaf(1.0f - mix, g1, v.y);
    if (in_chs == 1) gx[b * n + t] = o0 + o1;
    else { gx[(b * 2 + 0) * n + t] = o0; gx[(b * 2 + 1) * n + t] = o1; }
  }
}

// per (item, block): S0[k] = sum_t (dIR_l f_l + dIR_r f_r) env_k ;  S1[k] = sum_t (...) env_k tt
// part[((item*nbk + b)*12 + k)*2 + {0,1}]
__global__ void ir_grad_pairs_kernel(const float2* __restrict__ Et, const float2* __restrict__ C,
                                     const float* __restrict__ params, float* __restrict__ part, int64_t L,
                                     int64_t leff, int jb, int nbk, int nb, int hop, int P) {
  const int b = blockIdx.x;
  const int64_t il = blockIdx.y;
  __shared__ float rk[kBands];
  __shared__ float red[8][2 * kBands];
  if (threadIdx.x < kBands) rk[threadIdx.x] = -(params[il * 25 + kBands + threadIdx.x] * 10.0f + 1.0f);
  __syncthreads();
  const float step = 1.0f / (float)(L - 1);
  const float2* de = Et + il * (int64_t)jb * kNbA;
  float s0[kBands], s1[kBands];
#pragma unroll
  for (int k = 0; k < kBands; ++k) { s0[k] = 0.f; s1[k] = 0.f; }
  for (int m = threadIdx.x; m < hop; m += blockDim.x) {
    const int64_t t = (int64_t)b * hop + m;
    if (t >= leff) break;
    const float tt = time_axis(t, L, step);
    const float2 gd = de[(t / kB) * kNbA + (t % kB)];
    const float gl = gd.x, gr = gd.y;
    const float2* c = C + ((il * kBands) * nbk + b) * (int64_t)nb + m + P;
#pragma unroll
    for (int k = 0; k < kBands; ++k) {
      const float2 v = c[(int64_t)k * nbk * nb];
      const float w = fmaf(gl, v.x, gr * v.y) * expf(rk[k] * tt);
      s0[k] += w;
      s1[k] = fmaf(w, tt, s1[k]);
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < kBands; ++k) {
    const float a = warp_sum(s0[k]), c1 = warp_sum(s1[k]);
    if (lane == 0) { red[warp][2 * k] = a; red[warp][2 * k + 1] = c1; }
  }
  __syncthreads();
  if (threadIdx.x < 2 * kBands) {
    float a = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) a += red[w][threadIdx.x];
    part[((il * nbk + b) * kBands) * 2 + threadIdx.x] = a;
  }
}

// one thread per (item, param): gains (0..11), decays (12..23), mix (24)
__global__ void reverb_param_grad_kernel(const float* __restrict__ ir_part, const float* __restrict__ mix_part,
                                         const float* __restrict__ params, float* __restrict__ gparams, int64_t item0,
                                         int64_t items, int nbk, int mix_blocks) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= items * 25) return;
  const int64_t bl = idx / 25;
  const int q = (int)(idx - bl * 25);
  const float* pp = params + (item0 + bl) * 25;
  double s = 0.0;
  if (q < 24) {
    const int k = q % kBands;
    const float* pr = ir_part + (bl * nbk * kBands + k) * 2 + (q < kBands ? 0 : 1);
    for (int i = 0; i < nbk; ++i) s += (double)pr[(int64_t)i * kBands * 2];
    if (q < kBands) s *= (1.0 / kBands);
    else s *= (double)pp[k] * (-10.0 / kBands);
  } else {
    for (int i = 0; i < mix_blocks; ++i) s += (double)mix_part[bl * mix_blocks + i];
  }
  gparams[(item0 + bl) * 25 + q] = (float)s;
}

// device-resident band spectra H_k: 12 x nb complex (full spectrum of the real taps), scaled by 1/nb;
// built once per (device, taps, sr, nb)
int get_filterbank(const Geom& g, double sr, cudaStream_t st, const float2** out) {
  int dev = 0;
  DASP_CUDA_OK(cudaGetDevice(&dev));
  FbKey key{dev, g.taps, g.nb, sr};
  auto it = g_fb.find(key);
  if (it != g_fb.end()) { *out = reinterpret_cast<const float2*>(it->second); return DASP_OK; }
  DASP_REQUIRE(sr / 2.0 > 18000.0, "sample_rate %.1f too low: the filter bank needs 18 kHz < sr/2 (signal.py:84)", sr);
  std::vector<float> taps;
  octave_filterbank((int)g.taps, sr, taps);
  std::vector<float2> padded((size_t)kBands * g.nb, make_float2(0.f, 0.f));
  const float inv = 1.0f / (float)g.nb;
  for (int k = 0; k < kBands; ++k)
    for (int64_t i = 0; i < g.taps; ++i) padded[(size_t)k * g.nb + i].x = taps[(size_t)k * g.taps + i] * inv;
  cufftComplex* d_buf = nullptr;
  void* d_work = nullptr;
  DASP_CUDA_OK(cudaMalloc(&d_buf, sizeof(cufftComplex) * padded.size()));
  DASP_CUDA_OK(cudaMemcpyAsync(d_buf, padded.data(), sizeof(float2) * padded.size(), cudaMemcpyHostToDevice, st));
  PlanVal pv;
  int rc = get_plan(2, g.nb, kBands, g.nb, g.nb, pv);
  if (rc != DASP_OK) return rc;
  DASP_CUDA_OK(cudaMalloc(&d_work, pv.work > 0 ? pv.work : 16));
  DASP_CUFFT_OK(cufftSetStream(pv.h, st));
  DASP_CUFFT_OK(cufftSetWorkArea(pv.h, d_work));
  DASP_CUFFT_OK(cufftExecC2C(pv.h, d_buf, d_buf, CUFFT_FORWARD));
  DASP_CUDA_OK(cudaStreamSynchronize(st));   // one-off (cache fill): host vector and temp buffers die here
  cudaFree(d_work);
  g_fb[key] = d_buf;
  *out = reinterpret_cast<const float2*>(d_buf);
  return DASP_OK;
}

// half spectrum of the taps on the n1-point grid of the spectral synthesis: 12 x (n1/2+1) complex, scaled sqrt(n1/2)/n1
int get_filterbank_n1(const Geom& g, double sr, cudaStream_t st, const float2** out) {
  int dev = 0;
  DASP_CUDA_OK(cudaGetDevice(&dev));
  const int64_t n1 = g.n1(), n1c = g.n1c();
  const bool flat = debug_flat_filterbank();        // test hook: H_k = 1 -> f_k is the white periodic sequence itself
  FbKey key{dev, flat ? -g.taps : g.taps, -n1, sr};
  auto it = g_fb.find(key);
  if (it != g_fb.end()) { *out = reinterpret_cast<const float2*>(it->second); return DASP_OK; }
  DASP_REQUIRE(sr / 2.0 > 18000.0, "sample_rate %.1f too low: the filter bank needs 18 kHz < sr/2 (signal.py:84)", sr);
  {
    float2 roots[17][16];
    for (int r = 0; r <= 16; ++r)
      for (int m = 0; m < 16; ++m) {
        const double a = (r > 0) ? 2.0 * kPi * (double)(m % r) / (double)r : 0.0;
        roots[r][m] = make_float2((float)cos(a), (float)sin(a));
      }
    DASP_CUDA_OK(cudaMemcpyToSymbolAsync(c_root, roots, sizeof(roots), 0, cudaMemcpyHostToDevice, st));
    DASP_CUDA_OK(cudaStreamSynchronize(st));
  }
  std::vector<float> taps;
  octave_filterbank((int)g.taps, sr, taps);
  if (flat) {
    taps.assign(taps.size(), 0.f);
    for (int k = 0; k < kBands; ++k) taps[(size_t)k * g.taps] = 1.0f;      // unit impulse at lag 0
  }
  std::vector<float> padded((size_t)kBands * n1, 0.f);
  // 1/n1 of the inverse transform and the sqrt(n1/2) of the bins' complex Gaussians (Z ~ CN(0, n1)) are folded in
  const float inv = (float)(sqrt(0.5 * (double)n1) / (double)n1);
  for (int k = 0; k < kBands; ++k)
    for (int64_t i = 0; i < g.taps; ++i) padded[(size_t)k * n1 + i] = taps[(size_t)k * g.taps + i] * inv;
  float* d_in = nullptr;
  cufftComplex* d_out = nullptr;
  void* d_work = nullptr;
  DASP_CUDA_OK(cudaMalloc(&d_in, sizeof(float) * padded.size()));
  DASP_CUDA_OK(cudaMalloc(&d_out, sizeof(cufftComplex) * kBands * n1c));
  DASP_CUDA_OK(cudaMemcpyAsync(d_in, padded.data(), sizeof(float) * padded.size(), cudaMemcpyHostToDevice, st));
  PlanVal pv;
  int rc = get_plan(0, n1, kBands, n1, n1c, pv);
  if (rc != DASP_OK) return rc;
  DASP_CUDA_OK(cudaMalloc(&d_work, pv.work > 0 ? pv.work : 16));
  DASP_CUFFT_OK(cufftSetStream(pv.h, st));
  DASP_CUFFT_OK(cufftSetWorkArea(pv.h, d_work));
  DASP_CUFFT_OK(cufftExecR2C(pv.h, d_in, d_out));
  DASP_CUDA_OK(cudaStreamSynchronize(st));   // one-off cache fill
  cudaFree(d_in);
  cudaFree(d_work);
  g_fb[key] = d_out;
  *out = reinterpret_cast<const float2*>(d_out);
  return DASP_OK;
}

template <int R>
void launch_spectral(float2* C, const float2* H1, int64_t item0, int64_t items, int nb, const unsigned long long* seed,
                     bool planar, cudaStream_t st) {
  const int threads = 128;
  dim3 grid((unsigned)((nb / 2 + 1 + threads - 1) / threads), kBands, (unsigned)items);
  if (planar) spectral_gen_kernel<R, true><<<grid, threads, 0, st>>>(C, H1, item0, nb, seed);
  else        spectral_gen_kernel<R, false><<<grid, threads, 0, st>>>(C, H1, item0, nb, seed);
}
bool dispatch_spectral(int R, float2* C, const float2* H1, int64_t item0, int64_t items, int nb,
                       const unsigned long long* seed, bool planar, cudaStream_t st) {
  switch (R) {
#define DASP_R(r) case r: launch_spectral<r>(C, H1, item0, items, nb, seed, planar, st); return true;
    DASP_R(1) DASP_R(2) DASP_R(3) DASP_R(4) DASP_R(5) DASP_R(6) DASP_R(7) DASP_R(8) DASP_R(9) DASP_R(10)
    DASP_R(11) DASP_R(12) DASP_R(13) DASP_R(14) DASP_R(15) DASP_R(16)
#undef DASP_R
    default: return false;       // very long IRs fall back to the time-domain Philox + overlap-save path
  }
}
constexpr int kMaxSpectralR = 16;

// twiddle tables of fft8192.cuh (fp64 on the host, once per device)
std::map<int, float*> g_fft_tab;
int get_fft_tables(cudaStream_t st, const float** out) {
  int dev = 0;
  DASP_CUDA_OK(cudaGetDevice(&dev));
  auto it = g_fft_tab.find(dev);
  if (it == g_fft_tab.end()) {
    std::vector<float> h(fft8k::kTabFloats, 0.f);
    for (int e = 0; e < fft8k::kTabEntries; ++e) {
      int co, so, dup;
      double turns;
      fft8k::table_entry(e, co, so, dup, turns);
      const float c = (float)cos(2.0 * kPi * turns), sn = (float)sin(2.0 * kPi * turns);
      h[co] = c; h[so] = sn;
      if (dup) { h[co + 1] = c; h[so + 1] = sn; }
    }
    float* d = nullptr;
    DASP_CUDA_OK(cudaMalloc(&d, sizeof(float) * h.size()));
    DASP_CUDA_OK(cudaMemcpyAsync(d, h.data(), sizeof(float) * h.size(), cudaMemcpyHostToDevice, st));
    DASP_CUDA_OK(cudaStreamSynchronize(st));   // one-off cache fill (h goes out of scope)
    it = g_fft_tab.emplace(dev, d).first;
  }
  *out = it->second;
  return DASP_OK;
}
int configure_fft_kernels();
int launch_ifft_shape(float2* C, const float* tw, const float* params, float2* hs, bool save_f, int64_t items,
                      const Geom& g, int jb, cudaStream_t st) {
  int rc = configure_fft_kernels();
  if (rc != DASP_OK) return rc;
  const size_t smem = kFftSmemBytes;
  ifft_shape_kernel<<<dim3((unsigned)g.rpp, (unsigned)items), kFusedThreads, smem, st>>>(
      reinterpret_cast<float*>(C), tw, params, hs, save_f ? 1 : 0, (int)g.L, (int)g.leff, jb, (int)g.rpp);
  DASP_LAUNCH_OK("ifft_shape_kernel");
  return DASP_OK;
}
int g_last_path = 0;                                 // test hook: IR-synthesis path of the last forward chunk

struct Plans { PlanVal blk_c2c, pp_c2c, xi_c2c, hj_c2c; size_t work; };
int get_plans(const Geom& g, int64_t items, Plans& p) {
  int rc;
  if ((rc = get_plan(2, g.nb, items * kBands * g.nbk, g.nb, g.nb, p.blk_c2c)) != DASP_OK) return rc;
  if ((rc = get_plan(2, g.nb, items * kBands * g.rpp, g.nb, g.nb, p.pp_c2c)) != DASP_OK) return rc;
  if ((rc = get_plan(2, kNbA, items * g.ib, kNbA, kNbA, p.xi_c2c)) != DASP_OK) return rc;
  if ((rc = get_plan(2, kNbA, items * g.jb, kNbA, kNbA, p.hj_c2c)) != DASP_OK) return rc;
  p.work = p.blk_c2c.work;
  if (p.pp_c2c.work > p.work) p.work = p.pp_c2c.work;
  if (p.xi_c2c.work > p.work) p.work = p.xi_c2c.work;
  if (p.hj_c2c.work > p.work) p.work = p.hj_c2c.work;
  return DASP_OK;
}

inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// workspace carve-up shared by the geometry query and the two entry points
struct FwdWs { size_t ys, xsp, hsp, fchunk, cufft, total; };
struct BwdWs { size_t gs, ds, es, irpart, mixpart, cufft, total; };

void fwd_layout(const Geom& g, size_t cufft_work, FwdWs& w) {
  size_t o = 0;
  w.ys = o;  o += align256(sizeof(float2) * (size_t)(g.chunk * g.ib * kNbA));
  // transient homes for what a forward WITHOUT a backward does not keep (null *_save pointers)
  w.xsp = o; o += align256(sizeof(float2) * (size_t)(g.chunk * g.ib * kNbA));
  w.hsp = o; o += align256(sizeof(float2) * (size_t)(g.chunk * g.jb * kNbA));
  w.fchunk = o; o += align256(sizeof(float2) * (size_t)(g.chunk * kBands * g.pair_c64()));
  w.cufft = o; o += align256(cufft_work);
  w.total = o;
}
void bwd_layout(const Geom& g, size_t cufft_work, BwdWs& w) {
  size_t o = 0;
  w.gs = o; o += align256(sizeof(float2) * (size_t)(g.chunk * g.ib * kNbA));
  w.ds = o; o += align256(sizeof(float2) * (size_t)(g.chunk * g.ib * kNbA));
  w.es = o; o += align256(sizeof(float2) * (size_t)(g.chunk * g.jb * kNbA));
  int64_t nparts = g.nbk > g.nparts_pp() ? g.nbk : g.nparts_pp();
  if (g.jb > nparts) nparts = g.jb;
  w.irpart = o; o += align256(sizeof(float) * (size_t)(g.chunk * nparts * kBands * 2));
  w.mixpart = o; o += align256(sizeof(float) * (size_t)(g.chunk * g.ib));
  w.cufft = o; o += align256(cufft_work);
  w.total = o;
}

// out = conv / corr of packed block spectra, register-cached when both operands have <= 16 blocks
template <bool CORR, bool PLANAR = false>
void launch_mac(const float2* A, const float2* Bm, float2* Out, int na, int nbm, int nout, int64_t items, float scale,
                cudaStream_t st) {
  dim3 grid((kNbA / 2 + 1 + 127) / 128, (unsigned)items);
  const int m = na > nbm ? na : nbm;
  if (m <= 12)      partition_mac_kernel<12, CORR, PLANAR><<<grid, 128, 0, st>>>(A, Bm, Out, na, nbm, nout, scale);
  else if (m <= 16) partition_mac_kernel<16, CORR, PLANAR><<<grid, 128, 0, st>>>(A, Bm, Out, na, nbm, nout, scale);
  else              partition_mac_kernel<0, CORR, PLANAR><<<grid, 128, 0, st>>>(A, Bm, Out, na, nbm, nout, scale);
}

// one-off opt-in to the large dynamic shared memory of the FFT kernels (per device, guarded by g_mu)
int configure_fft_kernels() {
  static std::map<int, bool> configured;
  int dev = 0;
  DASP_CUDA_OK(cudaGetDevice(&dev));
  if (!configured[dev]) {
    DASP_CUDA_OK(cudaFuncSetAttribute(ifft_shape_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFftSmemBytes));
    DASP_CUDA_OK(cudaFuncSetAttribute(x_fft_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFftSmemBytes));
    DASP_CUDA_OK(cudaFuncSetAttribute(ifft_mix_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFftSmemBytes));
    DASP_CUDA_OK(cudaFuncSetAttribute(g_fft_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFftSmemBytes));
    DASP_CUDA_OK(cudaFuncSetAttribute(ifft_dx_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFftSmemBytes));
    DASP_CUDA_OK(cudaFuncSetAttribute(ifft_irgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFftSmemBytes));
    configured[dev] = true;
  }
  return DASP_OK;
}

}  // namespace

void reverb_shutdown() {
  std::lock_guard<std::mutex> lk(g_mu);
  for (auto& kv : g_plans) cufftDestroy(kv.second.h);
  g_plans.clear();
  for (auto& kv : g_fb) cudaFree(kv.second);
  g_fb.clear();
  for (auto& kv : g_fft_tab) cudaFree(kv.second);
  g_fft_tab.clear();
}

}  // namespace dasp

using namespace dasp;

extern "C" {

int dasp_debug_reverb_last_path(void) { return g_last_path; }

// host-side restatement of signal.octave_band_filterbank: writes 12*taps floats (no GPU needed)
int dasp_reverb_filterbank(int64_t taps, double sample_rate, float* out) {
  DASP_REQUIRE(out != nullptr && taps >= 1 && (taps % 2) == 1, "filterbank: taps must be odd and out non-null");
  DASP_REQUIRE(sample_rate / 2.0 > 18000.0, "filterbank: needs 18 kHz < sample_rate/2");
  std::vector<float> v;
  octave_filterbank((int)taps, sample_rate, v);
  for (size_t i = 0; i < v.size(); ++i) out[i] = v[i];
  return DASP_OK;
}

namespace {
int plans_for(const Geom& g, Plans& pfull, Plans& prem, size_t& work) {
  int rc;
  if ((rc = get_plans(g, g.chunk, pfull)) != DASP_OK) return rc;
  work = pfull.work;
  const int64_t rem = g.bs % g.chunk;
  if (rem) {
    if ((rc = get_plans(g, rem, prem)) != DASP_OK) return rc;
    if (prem.work > work) work = prem.work;
  }
  return DASP_OK;
}
}  // namespace

int dasp_reverb_geometry(int64_t bs, int64_t n, int64_t num_samples, int64_t taps, int64_t chunk_items,
                         dasp_reverb_geom* out) {
  DASP_REQUIRE(out != nullptr, "reverb geometry: null out");
  Geom g;
  int rc = make_geom(bs, n, num_samples, taps, chunk_items, g);
  if (rc != DASP_OK) return rc;
  std::lock_guard<std::mutex> lk(g_mu);
  size_t work = 0;
  if (bs > 0) {
    Plans p{}, q{};
    if ((rc = plans_for(g, p, q, work)) != DASP_OK) return rc;
  }
  FwdWs fw; BwdWs bw;
  fwd_layout(g, work, fw);
  bwd_layout(g, work, bw);
  out->nb = g.nb; out->hop = g.hop; out->nbk = g.nbk; out->leff = g.leff; out->rpp = g.rpp;
  out->conv_block = kB; out->x_blocks = g.ib; out->ir_partitions = g.jb; out->chunk_items = g.chunk;
  out->f_floats = bs * kBands * g.pair_c64() * 2;
  out->xspec_c64 = bs * g.ib * kNbA;
  out->irspec_c64 = bs * g.jb * kNbA;
  out->wet_floats = bs * 2 * n;
  out->fwd_workspace_bytes = (int64_t)fw.total;
  out->bwd_workspace_bytes = (int64_t)bw.total;
  return DASP_OK;
}

int dasp_reverb_fwd(const float* x, int64_t in_chs, const float* params, const float* noise, const uint64_t* seed_dev, float* y,
                    float* wet_save, float* f_save, void* xspec_save, void* irspec_save, void* workspace,
                    int64_t workspace_bytes, int64_t bs, int64_t n, int64_t num_samples, int64_t taps,
                    int64_t chunk_items, float sample_rate, void* stream) {
  Geom g;
  int rc = make_geom(bs, n, num_samples, taps, chunk_items, g);
  if (rc != DASP_OK) return rc;
  DASP_REQUIRE(in_chs == 1 || in_chs == 2, "only mono/stereo signals are supported");
  if (bs == 0) return DASP_OK;
  DASP_REQUIRE(x && params && y && workspace, "reverb fwd: null pointer");
  DASP_REQUIRE(noise != nullptr || seed_dev != nullptr, "reverb fwd: device-noise mode needs seed_dev (a device pointer)");
  const unsigned long long* seed = reinterpret_cast<const unsigned long long*>(seed_dev);
  cudaStream_t st = (cudaStream_t)stream;
  std::lock_guard<std::mutex> lk(g_mu);
  const float2 *H = nullptr, *H1 = nullptr;
  const bool spectral = (noise == nullptr) && g.rpp <= kMaxSpectralR;
  if (spectral) { if ((rc = get_filterbank_n1(g, (double)sample_rate, st, &H1)) != DASP_OK) return rc; }
  else          { if ((rc = get_filterbank(g, (double)sample_rate, st, &H)) != DASP_OK) return rc; }
  Plans pfull{}, prem{};
  size_t work = 0;
  if ((rc = plans_for(g, pfull, prem, work)) != DASP_OK) return rc;
  FwdWs w;
  fwd_layout(g, work, w);
  if ((int64_t)w.total > workspace_bytes) {
    set_error("reverb fwd: workspace needs %lld bytes, got %lld", (long long)w.total, (long long)workspace_bytes);
    return DASP_ERR_WORKSPACE;
  }
  unsigned char* base = (unsigned char*)workspace;
  float2* ws_ys = (float2*)(base + w.ys);
  void* ws_cufft = base + w.cufft;
  const int64_t lp = g.L + g.P;
  const int nbk = (int)g.nbk, nb = (int)g.nb, hop = (int)g.hop, P = (int)g.P, I = (int)g.ib, J = (int)g.jb;

  for (int64_t item0 = 0; item0 < bs; item0 += g.chunk) {
    const int64_t items = (bs - item0 < g.chunk) ? bs - item0 : g.chunk;
    const Plans& pl = (items == g.chunk) ? pfull : prem;
    // kept for the backward when the caller passes *_save buffers, transient workspace otherwise
    float2* C = f_save ? reinterpret_cast<float2*>(f_save) + item0 * kBands * g.pair_c64()
                       : reinterpret_cast<float2*>(base + w.fchunk);
    float2* xs = xspec_save ? (float2*)xspec_save + item0 * I * (int64_t)kNbA : (float2*)(base + w.xsp);
    float2* hs = irspec_save ? (float2*)irspec_save + item0 * J * (int64_t)kNbA : (float2*)(base + w.hsp);
    const dim3 gblk((unsigned)nbk, kBands, (unsigned)items);

    // ---- IR synthesis: (left, right) taps land in the zero-initialised partition layout hs ----
    DASP_CUDA_OK(cudaMemsetAsync(hs, 0, sizeof(float2) * items * J * kNbA, st));
    // device-noise IR synthesis (the same Philox stream on both paths):
    //   nb == 8192: generator -> ifft_shape_kernel (own in-shared-memory FFT fused with the shaping)
    //   other nb  : generator -> batched cuFFT -> shape_ir_pp_kernel
    const bool own_fft = spectral && nb == fft8k::kN && g.L < (int64_t)1 << 31;
    // audio convolution: block transforms on the own FFT (fused with their pre/post kernels) when the rows allow bulk copies
    const bool own_conv = (n % 4 == 0) && aligned16(x);
    const float* tw = nullptr;
    if ((own_fft || own_conv) && (rc = get_fft_tables(st, &tw)) != DASP_OK) return rc;
    g_last_path = own_fft ? 2 : 0;
    if (own_fft) {
      dispatch_spectral((int)g.rpp, C, H1, item0, items, nb, seed, /*planar=*/true, st);
      DASP_LAUNCH_OK("spectral_gen_kernel");
      if ((rc = launch_ifft_shape(C, tw, params + item0 * 25, hs, f_save != nullptr, items, g, J, st)) != DASP_OK) return rc;
    } else if (spectral) {
      // device noise: draw the filtered spectrum directly, one inverse transform (polyphase layout)
      dispatch_spectral((int)g.rpp, C, H1, item0, items, nb, seed, /*planar=*/false, st);
      DASP_LAUNCH_OK("spectral_gen_kernel");
      DASP_CUFFT_OK(cufftSetStream(pl.pp_c2c.h, st));
      DASP_CUFFT_OK(cufftSetWorkArea(pl.pp_c2c.h, ws_cufft));
      DASP_CUFFT_OK(cufftExecC2C(pl.pp_c2c.h, (cufftComplex*)C, (cufftComplex*)C, CUFFT_INVERSE));
      shape_ir_pp_kernel<<<dim3((unsigned)((g.leff + 255) / 256), (unsigned)items), 256, 0, st>>>(
          C, params + item0 * 25, hs, g.L, g.leff, J, (int)g.rpp, nb);
      DASP_LAUNCH_OK("shape_ir_pp_kernel");
    } else {
      // parity mode (caller's noise tensor) or very long IR: time-domain noise, overlap-save blocks
      if (noise) noise_pairs_layout_kernel<<<gblk, 256, 0, st>>>(noise, C, item0, nbk, nb, hop, lp);
      else       noise_pairs_philox_kernel<<<gblk, 256, 0, st>>>(C, item0, nbk, nb, hop, seed);
      DASP_LAUNCH_OK("reverb noise kernel");
      DASP_CUFFT_OK(cufftSetStream(pl.blk_c2c.h, st));
      DASP_CUFFT_OK(cufftSetWorkArea(pl.blk_c2c.h, ws_cufft));
      DASP_CUFFT_OK(cufftExecC2C(pl.blk_c2c.h, (cufftComplex*)C, (cufftComplex*)C, CUFFT_FORWARD));
      cmul_filter_pairs_kernel<<<gblk, 256, 0, st>>>(C, H, nbk, nb);
      DASP_LAUNCH_OK("cmul_filter_pairs_kernel");
      DASP_CUFFT_OK(cufftExecC2C(pl.blk_c2c.h, (cufftComplex*)C, (cufftComplex*)C, CUFFT_INVERSE));
      shape_ir_pairs_kernel<<<dim3((unsigned)nbk, (unsigned)items), 256, 0, st>>>(C, params + item0 * 25, hs, g.L, g.leff,
                                                                               J, nbk, nb, hop, P);
      DASP_LAUNCH_OK("shape_ir_pairs_kernel");
    }

    // ---- audio convolution (partitioned, frequency domain) ----
    const int nblk = (int)(items * I);
    const unsigned fft_grid = (unsigned)(nblk < sm_count() ? nblk : sm_count());
    DASP_CUFFT_OK(cufftSetStream(pl.hj_c2c.h, st));
    DASP_CUFFT_OK(cufftSetWorkArea(pl.hj_c2c.h, ws_cufft));
    DASP_CUFFT_OK(cufftExecC2C(pl.hj_c2c.h, (cufftComplex*)hs, (cufftComplex*)hs, CUFFT_FORWARD));
    if (own_conv) {
      if ((rc = configure_fft_kernels()) != DASP_OK) return rc;
      x_fft_kernel<<<fft_grid, kFusedThreads, kFftSmemBytes, st>>>(x, xs, tw, item0, I, n, (int)in_chs, nblk);
      DASP_LAUNCH_OK("x_fft_kernel");
      launch_mac<false, true>(xs, hs, ws_ys, I, J, I, items, 1.0f / (float)kNbA, st);
      DASP_LAUNCH_OK("partition_mac_kernel");
      ifft_mix_kernel<<<fft_grid, kFusedThreads, kFftSmemBytes, st>>>(reinterpret_cast<const float*>(ws_ys), tw, x, params, y,
                                                                     wet_save, item0, I, n, (int)in_chs, nblk);
      DASP_LAUNCH_OK("ifft_mix_kernel");
      continue;
    }
    x_blocks_kernel<<<dim3((unsigned)I, (unsigned)items), 256, 0, st>>>(x, xs, item0, I, n, (int)in_chs);
    DASP_LAUNCH_OK("x_blocks_kernel");
    DASP_CUFFT_OK(cufftSetStream(pl.xi_c2c.h, st));
    DASP_CUFFT_OK(cufftSetWorkArea(pl.xi_c2c.h, ws_cufft));
    DASP_CUFFT_OK(cufftExecC2C(pl.xi_c2c.h, (cufftComplex*)xs, (cufftComplex*)xs, CUFFT_FORWARD));
    launch_mac<false>(xs, hs, ws_ys, I, J, I, items, 1.0f / (float)kNbA, st);
    DASP_LAUNCH_OK("partition_mac_kernel");
    DASP_CUFFT_OK(cufftExecC2C(pl.xi_c2c.h, (cufftComplex*)ws_ys, (cufftComplex*)ws_ys, CUFFT_INVERSE));
    mix_blocks_kernel<<<dim3((unsigned)I, (unsigned)items), 256, 0, st>>>(x, ws_ys, params, y, wet_save, item0, I, n,
                                                                        (int)in_chs);
    DASP_LAUNCH_OK("mix_blocks_kernel");
  }
  return DASP_OK;
}

int dasp_reverb_bwd(const float* gy, const float* x, int64_t in_chs, const float* params, const float* wet_save,
                    const float* f_save, const void* xspec_save, const void* irspec_save, float* gx, float* gparams,
                    void* workspace, int64_t workspace_bytes, int64_t bs, int64_t n, int64_t num_samples, int64_t taps,
                    int64_t chunk_items, int64_t device_noise, void* stream) {
  Geom g;
  int rc = make_geom(bs, n, num_samples, taps, chunk_items, g);
  if (rc != DASP_OK) return rc;
  DASP_REQUIRE(in_chs == 1 || in_chs == 2, "only mono/stereo signals are supported");
  if (bs == 0) return DASP_OK;
  const bool polyphase = device_noise != 0 && g.rpp <= kMaxSpectralR;   // layout the forward left in f_save
  DASP_REQUIRE(gy && x && params && wet_save && f_save && xspec_save && irspec_save && gx && gparams && workspace,
               "reverb bwd: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  std::lock_guard<std::mutex> lk(g_mu);
  Plans pfull{}, prem{};
  size_t work = 0;
  if ((rc = plans_for(g, pfull, prem, work)) != DASP_OK) return rc;
  BwdWs w;
  bwd_layout(g, work, w);
  if ((int64_t)w.total > workspace_bytes) {
    set_error("reverb bwd: workspace needs %lld bytes, got %lld", (long long)w.total, (long long)workspace_bytes);
    return DASP_ERR_WORKSPACE;
  }
  unsigned char* base = (unsigned char*)workspace;
  float2* ws_gs = (float2*)(base + w.gs);
  float2* ws_ds = (float2*)(base + w.ds);
  float2* ws_es = (float2*)(base + w.es);
  float* ws_irpart = (float*)(base + w.irpart);
  float* ws_mixpart = (float*)(base + w.mixpart);
  void* ws_cufft = base + w.cufft;
  const float inv = 1.0f / (float)kNbA;
  const int nbk = (int)g.nbk, nb = (int)g.nb, hop = (int)g.hop, P = (int)g.P, I = (int)g.ib, J = (int)g.jb;

  for (int64_t item0 = 0; item0 < bs; item0 += g.chunk) {
    const int64_t items = (bs - item0 < g.chunk) ? bs - item0 : g.chunk;
    const Plans& pl = (items == g.chunk) ? pfull : prem;
    const float2* C = reinterpret_cast<const float2*>(f_save) + item0 * kBands * g.pair_c64();
    const float2* xs = (const float2*)xspec_save + item0 * I * (int64_t)kNbA;
    const float2* hs = (const float2*)irspec_save + item0 * J * (int64_t)kNbA;

    // block transforms on the own in-shared-memory FFT (fused with their neighbours) when the rows allow bulk copies
    const bool own_conv = (n % 4 == 0) && aligned16(gy);
    const bool own_irgrad = own_conv && polyphase && nb == fft8k::kN && g.L < (int64_t)1 << 31;
    const float* tw = nullptr;
    if (own_conv) {
      if ((rc = get_fft_tables(st, &tw)) != DASP_OK) return rc;
      if ((rc = configure_fft_kernels()) != DASP_OK) return rc;
    }
    const int nblk = (int)(items * I);
    const unsigned fft_grid = (unsigned)(nblk < sm_count() ? nblk : sm_count());
    const int mb = I > J ? I : J;
    const bool fused_mac = own_irgrad && mb <= 16;
    if (own_conv) {
      g_fft_kernel<<<fft_grid, kFusedThreads, kFftSmemBytes, st>>>(gy, x, wet_save, params, ws_gs, ws_mixpart, tw, item0, I, n,
                                                                   (int)in_chs, nblk);
      DASP_LAUNCH_OK("g_fft_kernel");
      if (fused_mac) {
        dim3 mgrid((kNbA / 2 + 1 + 127) / 128, (unsigned)items);
        if (mb <= 12) partition_mac_bwd_kernel<12><<<mgrid, 128, 0, st>>>(ws_gs, hs, xs, ws_ds, ws_es, I, J, inv);
        else          partition_mac_bwd_kernel<16><<<mgrid, 128, 0, st>>>(ws_gs, hs, xs, ws_ds, ws_es, I, J, inv);
        DASP_LAUNCH_OK("partition_mac_bwd_kernel");
      } else {
        launch_mac<true, true>(ws_gs, hs, ws_ds, I, J, I, items, inv, st);      // dx windows: sum_j conj(H[j]) G[q+j]
        DASP_LAUNCH_OK("partition_mac_kernel<corr>");
      }
      const unsigned dx_grid = (unsigned)(items < sm_count() ? items : sm_count());
      ifft_dx_kernel<<<dx_grid, kFusedThreads, kFftSmemBytes, st>>>(reinterpret_cast<const float*>(ws_ds), tw, gy, params, gx,
                                                                    item0, (int)items, I, n, (int)in_chs);
      DASP_LAUNCH_OK("ifft_dx_kernel");
    } else {
      g_blocks_kernel<<<dim3((unsigned)I, (unsigned)items), 256, 0, st>>>(gy, x, wet_save, params, ws_gs, ws_mixpart, item0,
                                                                        I, n, (int)in_chs);
      DASP_LAUNCH_OK("g_blocks_kernel");
      DASP_CUFFT_OK(cufftSetStream(pl.xi_c2c.h, st));
      DASP_CUFFT_OK(cufftSetWorkArea(pl.xi_c2c.h, ws_cufft));
      DASP_CUFFT_OK(cufftExecC2C(pl.xi_c2c.h, (cufftComplex*)ws_gs, (cufftComplex*)ws_gs, CUFFT_FORWARD));
      launch_mac<true>(ws_gs, hs, ws_ds, I, J, I, items, inv, st);
      DASP_LAUNCH_OK("partition_mac_kernel<corr>");
      DASP_CUFFT_OK(cufftExecC2C(pl.xi_c2c.h, (cufftComplex*)ws_ds, (cufftComplex*)ws_ds, CUFFT_INVERSE));
      finish_dx_blocks_kernel<<<dim3((unsigned)I, (unsigned)items), 256, 0, st>>>(gy, ws_ds, params, gx, item0, I, n,
                                                                                (int)in_chs);
      DASP_LAUNCH_OK("finish_dx_blocks_kernel");
    }
    int nparts;
    if (own_irgrad) {
      if (!fused_mac) {
        launch_mac<true, true>(ws_gs, xs, ws_es, I, I, J, items, inv, st);      // dIR partitions: sum_p conj(X[p]) G[j+p]
        DASP_LAUNCH_OK("partition_mac_kernel<corr>");
      }
      nparts = J;
      const int nunits = (int)(items * J);
      const unsigned ig_grid = (unsigned)(nunits < sm_count() ? nunits : sm_count());
      ifft_irgrad_kernel<<<ig_grid, kFusedThreads, kFftSmemBytes, st>>>(reinterpret_cast<const float*>(ws_es), tw, C,
                                                                        params + item0 * 25, ws_irpart, (int)g.L,
                                                                        (int)g.leff, J, (int)g.rpp, nunits);
      DASP_LAUNCH_OK("ifft_irgrad_kernel");
    } else {
      launch_mac<true>(ws_gs, xs, ws_es, I, I, J, items, inv, st);
      DASP_LAUNCH_OK("partition_mac_kernel<corr>");
      DASP_CUFFT_OK(cufftSetStream(pl.hj_c2c.h, st));
      DASP_CUFFT_OK(cufftSetWorkArea(pl.hj_c2c.h, ws_cufft));
      DASP_CUFFT_OK(cufftExecC2C(pl.hj_c2c.h, (cufftComplex*)ws_es, (cufftComplex*)ws_es, CUFFT_INVERSE));
      if (polyphase) {
        nparts = (int)g.nparts_pp();
        ir_grad_pp_kernel<<<dim3((unsigned)nparts, (unsigned)items), 256, 0, st>>>(ws_es, C, params + item0 * 25, ws_irpart,
                                                                                  g.L, g.leff, J, (int)g.rpp, nb);
      } else {
        nparts = nbk;
        ir_grad_pairs_kernel<<<dim3((unsigned)nbk, (unsigned)items), 256, 0, st>>>(ws_es, C, params + item0 * 25, ws_irpart,
                                                                                    g.L, g.leff, J, nbk, nb, hop, P);
      }
      DASP_LAUNCH_OK("ir_grad kernel");
    }
    reverb_param_grad_kernel<<<(unsigned)((items * 25 + 127) / 128), 128, 0, st>>>(ws_irpart, ws_mixpart, params, gparams,
                                                                                   item0, items, nparts, I);
    DASP_LAUNCH_OK("reverb_param_grad_kernel");
  }
  return DASP_OK;
}

}  // extern "C"
