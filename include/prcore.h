/*
 * prcore.h -- C ABI of libprcore.so, the B200 (sm_100a) passive-radar DSP core.
 *
 * This is the drop-in boundary for the hot path of Max-Manning/passiveRadar.
 * The reference has no FFI of its own (it is pure Python), so each entry point
 * below names the *Python function* whose arithmetic it replaces; the Python
 * wrappers in passiveradar_b200/ keep those functions' signatures and bind these
 * symbols through ctypes (see INTEGRATION.md for the stub a maintainer of the
 * reference would add).
 *
 * Conventions
 *   - complex64 data are interleaved (re, im) float pairs: `prc_c64`.
 *   - every function returns PRC_OK (0) or a negative PRC_E_* code; the message
 *     for the calling thread is available from prc_last_error().
 *   - `mem_kind` says where the data pointers live:
 *         PRC_MEM_HOST   (0)  host memory; the library copies H2D / D2H itself
 *         PRC_MEM_DEVICE (1)  device memory on `device`; no copies are made
 *   - `stream` is a cudaStream_t (as void*).  NULL: the library uses a private
 *     stream owned by the calling thread and the call is synchronous.  Non-NULL:
 *     all work is enqueued on that stream; unless PRC_FLAG_ASYNC is set the call
 *     waits for it to finish before returning.
 *   - the library is re-entrant: dask's threaded scheduler calls the Python
 *     wrappers concurrently (main.py:169-194); ctypes drops the GIL, every
 *     (thread | stream) owns its workspace, errors are thread-local.
 *   - inputs are never modified; outputs are caller-allocated.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point
 *     fails with PRC_E_CUDA.
 */
#ifndef PRCORE_H
#define PRCORE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct prc_c64 { float re, im; } prc_c64;

#define PRC_VERSION 200          /* 0.2.0 */

/* status codes */
#define PRC_OK            0
#define PRC_E_INVALID    -1      /* bad argument (message says which) */
#define PRC_E_CUDA       -2      /* CUDA runtime error / no device */
#define PRC_E_SINGULAR   -3      /* LS normal equations not positive definite */
#define PRC_E_NOMEM      -4

/* mem_kind */
#define PRC_MEM_HOST      0
#define PRC_MEM_DEVICE    1

/* flags */
#define PRC_FLAG_ASYNC        1u   /* do not synchronise `stream` before returning */
#define PRC_FLAG_WINDOW_F32   2u   /* `window` points at float, not double */
#define PRC_FLAG_ABS_C64      4u   /* prc_cfar2d_f32: `x` is a complex64 map, |x| is used */

/* ---- lifecycle / diagnostics ------------------------------------------------ */
int         prc_version(void);
const char* prc_last_error(void);                /* thread-local, never NULL */
int         prc_device_count(int* count);
int         prc_init(int device);                /* optional: create the context early */
void        prc_shutdown(void);                  /* free every workspace and private stream */
int         prc_sync(int device, void* stream);  /* cudaStreamSynchronize on `stream` (or the thread's) */
uint64_t    prc_launch_count(void);              /* kernels launched by this library so far */

/* per-kernel device timing (CUDA events on the launching stream around every launch).
 * enable -> run -> collect (synchronises) -> read(idx) for idx < prc_profile_kernels() */
int prc_profile_enable(int on);
int prc_profile_collect(void);
int prc_profile_kernels(void);
int prc_profile_read(int idx, const char** name, double* total_ms, uint64_t* launches);
int prc_profile_reset(void);

/* pinned host memory helpers (so numpy buffers can take the async copy path) */
int prc_host_alloc(void** ptr, uint64_t bytes);
int prc_host_free(void* ptr);
int prc_host_register(void* ptr, uint64_t bytes);
int prc_host_unregister(void* ptr);

/* ---- cross-ambiguity function ---------------------------------------------------
 * Replaces fast_xambg(), reference passiveRadar/range_doppler_processing.py:12-90,
 * for inputs already padded to their final length `n` (the zero-padding of :52-55,
 * named windows of :57-58 and the (F, R+1, 1) reshape stay in the Python wrapper).
 *
 *   out[f*(range_bins+1) + k],  f = 0..freq_bins-1 (fftshift-ed Doppler),
 *                               k = 0..range_bins   (delay range_bins - k)
 *
 * window : n doubles (or floats with PRC_FLAG_WINDOW_F32) or NULL      (:83-84)
 * dtaps  : decimator taps (doubles) or NULL for the reference's default boxcar of
 *          int(n/freq_bins)+1 ones (:69-72); ndtaps = their count         (:73-78)
 */
int prc_xambg_c64(const prc_c64* ref, const prc_c64* srv, int64_t n,
                  int range_bins, int freq_bins,
                  const void* window, const double* dtaps, int64_t ndtaps,
                  prc_c64* out, int mem_kind, int device, void* stream, unsigned flags);

/* ---- block least-squares clutter filter ---------------------------------------------
 * Replaces LS_Filter(), reference passiveRadar/clutter_removal.py:6-56.
 *   out  : n cleaned surveillance samples
 *   taps : filter_len + peek taps, or NULL                                    (:53-56)
 * The Gram matrix of :39 is Hermitian Toeplitz (circular autocorrelation of ref);
 * the library computes its first column and the right-hand side of :45 as lag
 * correlations, solves (T + reg I) w = rhs in float64 and applies the circular FIR
 * of :51.
 */
int prc_ls_filter_c64(const prc_c64* ref, const prc_c64* srv, int64_t n,
                      int filter_len, int peek, float reg,
                      prc_c64* out, prc_c64* taps,
                      int mem_kind, int device, void* stream, unsigned flags);

/* ---- Toeplitz least-squares clutter filter (what main.py actually calls) ---------------------------
 * prc_ls_toeplitz_c64 replaces LS_Filter_Toeplitz(), reference passiveRadar/clutter_removal.py:109-160:
 * reference rolled by -peek (:139), LINEAR (zero-padded) auto/cross correlations (:142-147), Levinson
 * solve without regularisation (:150, float64 here as in SciPy), linear convolution + subtraction
 * (:153-155).  prc_ls_multiple_c64 replaces LS_Filter_Multiple() (:162-187): the filter is applied once
 * per Doppler bin on the running residual, the reference being frequency-shifted by bin Hz first
 * (signal_utils.py:24-27, float32 phase ramp as in the reference).  doppler_bins == NULL means [0].
 * Results are complex64; the Python wrappers widen them to complex128 like the reference returns.
 */
int prc_ls_toeplitz_c64(const prc_c64* ref, const prc_c64* srv, int64_t n, int filter_len, int peek,
                        prc_c64* out, prc_c64* taps, int mem_kind, int device, void* stream, unsigned flags);
int prc_ls_multiple_c64(const prc_c64* ref, const prc_c64* srv, int64_t n, int filter_len, int peek,
                        double sample_rate, const double* doppler_bins, int nbins,
                        prc_c64* out, prc_c64* taps_last,
                        int mem_kind, int device, void* stream, unsigned flags);

/* prc_ls_multiple_frames_c64: LS_Filter_Multiple on nframes independent chunks per call (device pointers; frame i at
 * ref/srv/out + i*frame_stride): what main.py:169-176 does per dask chunk, several chunks at a time.  One launch of each
 * kernel per Doppler bin covers the batch.
 */
int prc_ls_multiple_frames_c64(const prc_c64* ref, const prc_c64* srv, int64_t n, int nframes, int64_t frame_stride,
                               int filter_len, int peek, double sample_rate, const double* doppler_bins, int nbins,
                               prc_c64* out, int mem_kind, int device, void* stream, unsigned flags);

/* ---- NLMS / block-NLMS clutter filter ---------------------------------------------------
 * Replaces NLMS_filter(), reference passiveRadar/clutter_removal.py:189-249
 * (block_len == 1) and provides block_NLMS (block_len > 1; not in the reference,
 * defined in DESIGN.md).
 *   init_taps : filter_len + peek initial taps or NULL (zeros)              (:218-225)
 *   out       : n samples; out[0:filter_len] and out[n-peek:] are zero        (:231,:244)
 *   taps_out  : final taps or NULL                                            (:246-249)
 */
int prc_nlms_c64(const prc_c64* ref, const prc_c64* srv, int64_t n,
                 int filter_len, int peek, float mu, int block_len,
                 const prc_c64* init_taps, prc_c64* out, prc_c64* taps_out,
                 int mem_kind, int device, void* stream, unsigned flags);

/* ---- one CPI frame: LS_Filter -> fast_xambg with filterLen = range_bins-like chaining ----
 * The composition main.py performs per chunk (main.py:169-194 with LS_Filter in place
 * of LS_Filter_Multiple): cleaned = LS_Filter(ref, srv, filter_len, reg, peek);
 * map = fast_xambg(ref, cleaned, range_bins, freq_bins, n, window).
 * The cleaned surveillance channel stays in device memory.
 *   taps_out, cleaned_out : optional (NULL to skip)
 */
int prc_frame_c64(const prc_c64* ref, const prc_c64* srv, int64_t n,
                  int filter_len, int peek, float reg,
                  int range_bins, int freq_bins, const void* window,
                  prc_c64* out_map, prc_c64* taps_out, prc_c64* cleaned_out,
                  int mem_kind, int device, void* stream, unsigned flags);

/* prc_frames_c64: the same composition for `nframes` frames in one call -- frame i reads ref + i*frame_stride and
 * srv + i*frame_stride (strides in samples; device or host pointers as mem_kind says) and writes
 * out_maps + i*freq_bins*(range_bins+1), taps_out + i*(filter_len+peek), cleaned_out + i*frame_stride.  This is the unit
 * of work of the dask graph (one chunk = one frame, main.py:169-194) handed over several chunks at a time, so that one
 * launch of each kernel covers the whole batch (gridDim.y = frame).  prc_frame_c64 is nframes = 1.
 * With PRC_FLAG_ASYNC the Toeplitz-solve status of every frame stays on the device: prc_ls_status() reads it back
 * (0 = ok, 1 = normal equations not positive definite) after synchronising `stream`.
 */
int prc_frames_c64(const prc_c64* ref, const prc_c64* srv, int64_t n, int nframes, int64_t frame_stride,
                   int filter_len, int peek, float reg, int range_bins, int freq_bins, const void* window,
                   prc_c64* out_maps, prc_c64* taps_out, prc_c64* cleaned_out,
                   int mem_kind, int device, void* stream, unsigned flags);
int prc_ls_status(int device, void* stream, int* status, int nframes);

/* The other two operators of the path on nframes independent frames per call (same layout rules as prc_frames_c64):
 * prc_nlms_frames_c64 -- NLMS_filter / block_NLMS (clutter_removal.py:189-249): the recurrence of one frame is serial,
 *   so every frame gets its own CTA (one SM) and the batch fills the GPU; init_taps (filter_len + peek taps or NULL)
 *   is shared by all frames, taps_out receives nframes * (filter_len + peek) taps.
 * prc_xambg_frames_c64 -- fast_xambg (range_doppler_processing.py:12-90, default boxcar decimator) with one window for
 *   all frames; out receives nframes maps of freq_bins x (range_bins + 1).
 */
int prc_nlms_frames_c64(const prc_c64* ref, const prc_c64* srv, int64_t n, int nframes, int64_t frame_stride,
                        int filter_len, int peek, float mu, int block_len, const prc_c64* init_taps,
                        prc_c64* out, prc_c64* taps_out, int mem_kind, int device, void* stream, unsigned flags);
int prc_xambg_frames_c64(const prc_c64* ref, const prc_c64* srv, int64_t n, int nframes, int64_t frame_stride,
                         int range_bins, int freq_bins, const void* window, prc_c64* out,
                         int mem_kind, int device, void* stream, unsigned flags);

/* ---- run-time switches (also read once from the environment: PRC_FFT, PRC_FFT_MIN_N) ----------------
 *   "fft"        1 (default): LS correlations, clutter FIR and CAF block sums as FFT-domain block correlations
 *                (csrc/fftcorr.cuh);  0: direct form on tcgen05 / FP32 (csrc/toepcorr.cuh, firtc.cuh, lagstream.cuh)
 *   "fft_min_n"  smallest channel length the FFT-domain path takes (default 8192)
 */
int prc_set_option(const char* name, int value);
int prc_get_option(const char* name, int* value);

/* ---- direct (time-domain) cross-ambiguity function ------------------------------------------------
 * Replaces direct_xambg(), reference passiveRadar/range_doppler_processing.py:93-124: for Doppler bin f
 * the reference channel is frequency-shifted by (f - freq_bins/2) / CPI Hz (signal_utils.py:24-27,
 * float32 phase ramp and complex64 exponential as in the reference) and LINEARLY cross-correlated
 * with srv (xcorr(ref_shifted, srv, range_bins, 0), signal_utils.py:29-32).  out: freq_bins x
 * (range_bins + 1) complex64, column k <-> delay range_bins - k (same orientation as prc_xambg_c64).
 */
int prc_direct_xambg_c64(const prc_c64* ref, const prc_c64* srv, int64_t n, int range_bins, int freq_bins,
                         double sample_rate, prc_c64* out, int mem_kind, int device, void* stream, unsigned flags);

/* ---- front end: the chain main.py:105-166 runs on every input chunk before the clutter filter -------
 * in_kind : PRC_IQ_C64 (n complex64 samples), PRC_IQ_I8 / PRC_IQ_I16 (2n interleaved I,Q integers:
 *           deinterleave_IQ(), reference passiveRadar/signal_utils.py:19-22)
 * mode    : PRC_MIX_NONE, or frequency_shift(x, fc, fs, phase_offset) (signal_utils.py:24-27) with the
 *           reference's float32 phase ramp; PRC_MIX_C64 = phase_offset is a Python scalar (complex64
 *           arithmetic throughout), PRC_MIX_C128 = phase_offset is a NumPy float64 (main.py:127-130;
 *           the exponential is then evaluated in float64).  Results are complex64 either way.
 * prc_frontend_c64 additionally applies resample() = scipy.signal.resample_poly(x, up, down,
 * padtype='line') (signal_utils.py:15-17) in the same pass: h = the nh = 2*half_len+1 low-pass taps
 * ALREADY multiplied by up (what resample_poly hands to upfirdn; host doubles, designed by the caller
 * with scipy.signal.firwin exactly as resample_poly does).  out receives prc_resample_out_len() samples.
 */
#define PRC_IQ_C64   0
#define PRC_IQ_I8    1
#define PRC_IQ_I16   2
#define PRC_MIX_NONE 0
#define PRC_MIX_C64  1
#define PRC_MIX_C128 2
#define PRC_MIX_F64  3   /* fc was a NumPy float64 scalar: the phase ramp is evaluated in float64 */
#define PRC_MIX_FS64 4   /* only fs was a NumPy float64 scalar: float32 product, float64 division */
int prc_iq_mix_c64(const void* in, int in_kind, int64_t n, int mode, double fc, double fs, double phase_offset,
                   prc_c64* out, int mem_kind, int device, void* stream, unsigned flags);
int prc_resample_out_len(int64_t n_in, int up, int down, int nh, int64_t* n_out);
int prc_frontend_c64(const void* in, int in_kind, int64_t n, int mode, double fc, double fs, double phase_offset,
                     int up, int down, const double* h, int nh, prc_c64* out, int64_t out_capacity,
                     int mem_kind, int device, void* stream, unsigned flags);

/* ---- CFAR detector ---------------------------------------------------------------------------------
 * Replaces CFAR_2D(X, fw, gw, thresh), reference passiveRadar/target_detection.py:683-703: X / mean|X|
 * divided by the wrapped 2-D box average (fw x fw window minus the guard hole) + 1e-10.
 * x: rows x cols float32 (or complex64 with PRC_FLAG_ABS_C64: the magnitude is taken on the device, so
 * a map can go from prc_xambg_c64 to the detector without leaving HBM).  cr_out (float32) and/or
 * det_out (uint8, cr > *thresh) are written; thresh may be NULL when det_out is NULL.
 */
int prc_cfar2d_f32(const void* x, int rows, int cols, int fw, int gw, const float* thresh, float* cr_out,
                   uint8_t* det_out, int mem_kind, int device, void* stream, unsigned flags);

/* ---- long-lag correlation and channel alignment (csrc/xcorr.cuh) -----------------------------------
 * Replace xcorr() and find_channel_offset(), reference passiveRadar/signal_utils.py:29-78; main.py:54 and
 * :83 call find_channel_offset(refc1, srvc1, 1, 5000000) once per run to align the two receiver channels.
 * The correlation is a circular FP32 transform of P = 2^20 .. 2^24 points (four-step, float64-built
 * twiddles); lag windows and inputs too long for one transform are tiled / segmented by the library.
 *
 * prc_xcorr_c64: xcorr(s1, s2, nlead, nlag) = scipy.signal.correlate(s1, np.pad(s2, (nlag, nlead)), 'valid')
 *   is this lag window with, for L2 = ny + nlag + nlead, lag0 = ny - nx + nlead and nlags = L2 - nx + 1 when
 *   L2 >= nx, else lag0 = -nlag and nlags = nx - L2 + 1.  nlags < 2^31.
 *
 * prc_channel_offset: B1, B2 = scipy.signal.decimate(s, nd) (zero-phase: sosfiltfilt with the caller's
 *   sections, odd extension of 3 (2 nsections + 1) samples, sosfilt_zi initial states, float64 state), then
 *   xc = |xcorr(B1, B2, nl, nl)| (|Re| for real inputs) and *offset = (argmax xc - nl) * nd, the first index
 *   winning ties.  sos: nsections x 6 host doubles with sos[s][3] == 1 (scipy.signal.cheby1(8, 0.05, 0.8 / nd,
 *   output='sos') for decimate's default filter).  in_kind: one PRC_SIG_* (real integers are upcast to
 *   float64 as decimate does).  xc_abs: optional, receives the nlags floats of |xc| (2 nl + 1 when both
 *   decimated channels have the same length).  offset is one int64 in memory of mem_kind.
 */
#define PRC_SIG_C64   0   /* complex64 samples */
#define PRC_SIG_I8    1   /* real int8 samples (the raw arrays main.py:81-83 reads) */
#define PRC_SIG_I16   2   /* real int16 samples */
#define PRC_SIG_F64   3   /* real float64 samples */
#define PRC_SIG_C128  4   /* complex128 samples */
int prc_xcorr_c64(const prc_c64* x, int64_t nx, const prc_c64* y, int64_t ny, int64_t lag0, int64_t nlags,
                  prc_c64* out, int mem_kind, int device, void* stream, unsigned flags);
int prc_channel_offset(const void* s1, int64_t n1, const void* s2, int64_t n2, int in_kind, int nd, int64_t nl,
                       const double* sos, int nsections, int64_t* offset, float* xc_abs,
                       int mem_kind, int device, void* stream, unsigned flags);

#ifdef __cplusplus
}
#endif
#endif /* PRCORE_H */
