/* dasp_b200.h -- C ABI of libdasp_b200.so: the B200 (sm_100a) kernels behind
 * dasp_pytorch.functional's batched audio-processor hot path.
 *
 * The reference (csteinmetz1/dasp-pytorch @ c9ae0126) is pure Python and has no FFI of its
 * own; each entry point below replaces the arithmetic of one reference function and is what
 * a ctypes/cffi binding inside that function would call (INTEGRATION.md shows the binding).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to contiguous fp32 (unless stated), owned by the
 *     caller; the library never allocates tensors -- scratch comes in through `ws`
 *     arguments sized by the matching *_workspace_* query;
 *   - audio tensors are (batch, channels, samples) row-major, exactly the reference's
 *     tensor contract (README.md:38);
 *   - `stream` is a cudaStream_t; all work is enqueued on it, nothing synchronises -- with ONE documented
 *     exception: the first call on a device for a new (taps, sample_rate, geometry) builds library-owned caches
 *     (cuFFT plans, filter-bank spectra, FFT twiddle tables: cudaMalloc + one cudaStreamSynchronize).  Warm the
 *     shapes up once before capturing a CUDA graph; later calls are pure enqueues;
 *   - return value 0 = ok, negative = error (see DASP_ERR_*); the message is available
 *     from dasp_last_error() (thread-local).  No exception crosses this boundary;
 *   - reentrant from several host threads as long as they use distinct streams.
 */
#ifndef DASP_B200_H_
#define DASP_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DASP_ABI_VERSION 2

#define DASP_OK 0
#define DASP_ERR_INVALID (-1)   /* bad shape / null pointer / misalignment        */
#define DASP_ERR_CUDA (-2)      /* CUDA runtime call or kernel launch failed      */
#define DASP_ERR_CUFFT (-3)     /* cuFFT call failed                              */
#define DASP_ERR_WORKSPACE (-4) /* caller workspace smaller than *_workspace_*()  */

/* ---- library ---------------------------------------------------------------------- */
int dasp_abi_version(void);
const char* dasp_last_error(void);
/* compiled-for architecture as an integer (1000 for sm_100a) */
int dasp_compiled_arch(void);
/* frees cached cuFFT plans and device-side filter-bank spectra */
void dasp_shutdown(void);
/* The dasp_debug_* entry points are TEST HOOKS: process-global switches, not thread-safe, not for production
 * callers (they exist so that every kernel variant can be pinned against the oracle at small sizes). */
/* test hook: pin the warps-per-row variant of the scan kernels (1, 2, 4, 8, 16; 0 = automatic choice).  The EQ
 * forward has 4, 8 and 16, the EQ backward a single variant, the compressor all five; a kernel family without the
 * requested variant keeps its automatic choice */
void dasp_debug_force_warps(int warps);
/* test hook: IR synthesis used by the last chunk of the most recent dasp_reverb_fwd: 0 = cuFFT pipeline (or the
   caller's noise tensor), 2 = generator + own in-shared-memory FFT/shaping kernel (device noise, 8192-point blocks) */
int dasp_debug_reverb_last_path(void);

/* test hook: 1 = the spectral IR synthesis uses unit-impulse filters, so the f_save buffer of dasp_reverb_fwd
   returns the periodic white sequences w_k themselves (used to rebuild a reference-style noise tensor) */
void dasp_debug_reverb_flat_filterbank(int on);

/* ---- Processor.denormalize_param_dict on the device      (reference modules.py:13-14, 70-91) ------
 * out[r][c] = lo[c] + p01[r][c] * span[c].  The reference's range check (ValueError when a value leaves [0, 1])
 * cannot raise from the device: an offending element becomes NaN and bit 0 of *flag (device int, may be NULL)
 * is set; the host reads the flag whenever it can afford to (modules.Processor does so outside graph capture). */
int dasp_denormalize(const float* p01, const float* lo /* [cols] */, const float* span /* [cols] */, float* out,
                     int* flag, int64_t rows, int64_t cols, void* stream);

/* ---- gain: y = x * 10^(gain_db/20)            (reference functional.py:10-29) ------ */
int dasp_gain_fwd(const float* x, const float* gain_db /* [bs] */, float* y, int64_t bs, int64_t chs,
                  int64_t n, void* stream);
int dasp_gain_bwd(const float* gy, const float* x, const float* gain_db, float* gx,
                  float* g_gain_db /* [bs] */, float* ws, int64_t ws_floats, int64_t bs, int64_t chs,
                  int64_t n, void* stream);

/* ---- distortion: y = tanh(x * 10^(drive_db/20))   (reference functional.py:65-78) --
 * rows = bs*chs; one drive value per row (the reference's drive_db.view(bs, chs, -1)). */
int dasp_distortion_fwd(const float* x, const float* drive_db /* [rows] */, float* y, int64_t rows,
                        int64_t n, void* stream);
int dasp_distortion_bwd(const float* gy, const float* x, const float* drive_db, float* gx,
                        float* g_drive_db /* [rows] */, float* ws, int64_t ws_floats, int64_t rows,
                        int64_t n, void* stream);
/* floats of scratch the two *_bwd calls above need (rows = bs for gain with n = chs*N) */
int64_t dasp_pointwise_bwd_workspace_floats(int64_t rows, int64_t n);

/* ---- stereo_widener / stereo_panner / stereo_bus      (reference functional.py:580-604, 607-636, 32-62) --
 * widener: x, y (bs, 2, n), width [bs].   panner: x (bs, tracks, n), pan [bs*tracks], y (bs, 2, tracks, n).
 * bus: x (bs, 2, tracks, n), send_db [bs*tracks], y (bs, 2, n).
 * ws: dasp_stereo_bwd_workspace_floats(rows, n) floats with rows = bs (widener), bs*tracks (panner),
 * bs*2*tracks (bus). */
int64_t dasp_stereo_bwd_workspace_floats(int64_t rows, int64_t n);
int dasp_widener_fwd(const float* x, const float* width, float* y, int64_t bs, int64_t n, void* stream);
int dasp_widener_bwd(const float* gy, const float* x, const float* width, float* gx, float* g_width, float* ws,
                     int64_t ws_floats, int64_t bs, int64_t n, void* stream);
int dasp_panner_fwd(const float* x, const float* pan, float* y, int64_t bs, int64_t tracks, int64_t n, void* stream);
int dasp_panner_bwd(const float* gy, const float* x, const float* pan, float* gx, float* g_pan, float* ws,
                    int64_t ws_floats, int64_t bs, int64_t tracks, int64_t n, void* stream);
int dasp_bus_fwd(const float* x, const float* send_db, float* y, int64_t bs, int64_t tracks, int64_t n, void* stream);
int dasp_bus_bwd(const float* gy, const float* x, const float* send_db, float* gx, float* g_send_db, float* ws,
                 int64_t ws_floats, int64_t bs, int64_t tracks, int64_t n, void* stream);

/* ---- compressor / expander            (reference functional.py:275-399; :402-403 stub) --
 * kind: 0 = compressor (reference semantics: attack-only smoothing, release_ms unused),
 *       1 = downward expander (new op, same signature; the reference only stubs it).
 * Parameters are [bs] arrays.  `ckpt` (fwd: optional out, bwd: in) holds the smoother state at
 * every tile boundary: bs * ceil(n / dasp_dynamics_tile_len(bs, chs)) floats; pass NULL in the
 * forward when no backward will follow.  gparams is [bs][6] in signature order
 * (threshold, ratio, attack, release(=0), knee, makeup).  g_scratch (bs*n floats) is only
 * needed when lookahead > 0. */
int64_t dasp_dynamics_tile_len(int64_t bs, int64_t chs);
int dasp_dynamics_fwd(int kind, const float* x, const float* threshold_db, const float* ratio,
                      const float* attack_ms, const float* knee_db, const float* makeup_db, float* y,
                      float* ckpt, int64_t bs, int64_t chs, int64_t n, float sample_rate, float eps,
                      int64_t lookahead, void* stream);
int dasp_dynamics_bwd(int kind, const float* gy, const float* x, const float* threshold_db,
                      const float* ratio, const float* attack_ms, const float* knee_db,
                      const float* makeup_db, const float* ckpt, float* gx, float* gparams,
                      float* g_scratch, int64_t bs, int64_t chs, int64_t n, float sample_rate, float eps,
                      int64_t lookahead, void* stream);

/* ---- parametric_eq: six cascaded biquads   (reference functional.py:118-272 with
 *      signal.biquad signal.py:242-306 and signal.sosfilt_via_fsm signal.py:136-166) ------
 * params is [bs][18] = (gain_dB, cutoff_Hz, Q) for low shelf, band0..band3, high shelf, i.e. the
 * 18 tensors of the reference signature stacked in order; the same filter is applied to every
 * channel of an item (signal.py:157-158).  Rows (item, channel) are processed in pairs; ckpt (fwd: optional out,
 * bwd: in) holds the section states of a pair at every tile boundary: dasp_eq_ckpt_floats(bs, chs, n) floats
 * (tiles of dasp_eq_tile_len() samples).  gparams is [bs][18]; ws needs dasp_eq_bwd_workspace_floats(bs, chs)
 * floats. */
int64_t dasp_eq_tile_len(int64_t rows);
int64_t dasp_eq_ckpt_floats(int64_t bs, int64_t chs, int64_t n);
int64_t dasp_eq_bwd_workspace_floats(int64_t bs, int64_t chs);
int dasp_eq_fwd(const float* x, const float* params, float* y, float* ckpt, int64_t bs, int64_t chs,
                int64_t n, float sample_rate, void* stream);
int dasp_eq_bwd(const float* gy, const float* x, const float* params, const float* ckpt, float* gx,
                float* gparams, float* ws, int64_t ws_floats, int64_t bs, int64_t chs, int64_t n,
                float sample_rate, void* stream);

/* ---- noise_shaped_reverberation          (reference functional.py:406-577, filter bank
 *      signal.octave_band_filterbank signal.py:42-92) --------------------------------------
 * params is [bs][25] = 12 band gains, 12 band decays, mix (signature order).  x is (bs, in_chs, n)
 * with in_chs 1 or 2; y is always (bs, 2, n) (mono is duplicated, functional.py:493-495).
 * noise: NULL -> white noise is generated on the device (Philox4x32-10, keyed by the 64-bit value the kernels read
 *        from the DEVICE pointer `seed_dev` when they run -- so a captured CUDA graph draws fresh noise on every
 *        replay as long as the caller's graph also refreshes that word, as torch's graph-safe generator does);
 *        else the (bs*2, 12, num_samples + taps - 1) tensor the reference would have drawn
 *        (functional.py:547-548) -- the parity-test entry.
 * Buffers kept for the backward (pass NULL for all four when no backward follows):
 *   wet_save  bs*2*n floats, f_save  geom.f_floats floats (band-filtered noise blocks, left/right
 *   channel interleaved as complex pairs),
 *   xspec_save  geom.xspec_c64 complex64, irspec_save  geom.irspec_c64 complex64 (block spectra).
 * workspace: geom.fwd_workspace_bytes / geom.bwd_workspace_bytes bytes of device memory. */
typedef struct dasp_reverb_geom {
  int64_t nb, hop, nbk;       /* IR synthesis, overlap-save path: block length, hop, blocks per band signal */
  int64_t leff;               /* min(num_samples, n): IR taps that can reach the n output samples */
  int64_t rpp;                /* IR synthesis, spectral path: polyphase factor (n1 = rpp * nb >= leff + taps - 1) */
  int64_t conv_block;         /* audio convolution: partition / hop length (its FFT length is twice that) */
  int64_t x_blocks;           /* ceil(n / conv_block) */
  int64_t ir_partitions;      /* ceil(leff / conv_block) */
  int64_t chunk_items;        /* items processed per pass */
  int64_t f_floats, xspec_c64, irspec_c64, wet_floats;      /* sizes of the buffers kept for the backward */
  int64_t fwd_workspace_bytes, bwd_workspace_bytes;
} dasp_reverb_geom;
int dasp_reverb_geometry(int64_t bs, int64_t n, int64_t num_samples, int64_t taps, int64_t chunk_items,
                         dasp_reverb_geom* out);
int dasp_reverb_fwd(const float* x, int64_t in_chs, const float* params, const float* noise, const uint64_t* seed_dev,
                    float* y, float* wet_save, float* f_save, void* xspec_save, void* irspec_save,
                    void* workspace, int64_t workspace_bytes, int64_t bs, int64_t n, int64_t num_samples,
                    int64_t taps, int64_t chunk_items, float sample_rate, void* stream);
int dasp_reverb_bwd(const float* gy, const float* x, int64_t in_chs, const float* params,
                    const float* wet_save, const float* f_save, const void* xspec_save,
                    const void* irspec_save, float* gx, float* gparams, void* workspace,
                    int64_t workspace_bytes, int64_t bs, int64_t n, int64_t num_samples, int64_t taps,
                    int64_t chunk_items, int64_t device_noise /* 1 iff the forward ran with noise == NULL */,
                    void* stream);
/* host-only: the 12 x taps fp32 filter bank (scipy.signal.firwin restated; no GPU needed) */
int dasp_reverb_filterbank(int64_t taps, double sample_rate, float* out);

#ifdef __cplusplus
}
#endif
#endif /* DASP_B200_H_ */
