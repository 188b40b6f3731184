/*
 * impdar_b200.h - C ABI of libimpdar_b200.so: the B200 (sm_100a) backend for ImpDAR's radargram
 * migration + filtering hot path.
 *
 * Reference interfaces replaced (paths relative to the reference's src/impdar/lib/):
 *   - migrationlib/mig_cython.h:11            void mig_kirch_loop(...)     the one C-ABI precedent
 *   - migrationlib/mig_python.py:35-123       migrationKirchhoff[Loop]
 *   - migrationlib/mig_python.py:126-208      migrationStolt
 *   - migrationlib/mig_python.py:211-287,361-540  migrationPhaseShift / phaseShift (const, layered, v(x,z) FFD)
 *   - migrationlib/mig_python.py:290-355      migrationTimeWavenumber (taper-only stub)
 *   - RadarData/_RadarDataFiltering.py:469-549  vertical_band_pass  (filtfilt / FIR lfilter)
 *   - RadarData/_RadarDataFiltering.py:93-135   horizontalfilt
 *   - RadarData/_RadarDataFiltering.py:19-90    adaptivehfilt
 *   - RadarData/_RadarDataFiltering.py:138-440  highpass / lowpass / horizontal_band_pass / winavg_hfilt
 *   - RadarData/_RadarDataProcessing.py:456-496 rangegain / agc
 *   - RadarData/_RadarDataFiltering.py:552-587  denoise (Wiener)
 *   - RadarData/_RadarDataProcessing.py:20-637  reverse / crop / hcrop / restack / nmo / constant_space / elev_correct
 *
 * Conventions
 *   - A radargram is a C-order (snum, tnum) array: row = time sample, column = trace, traces contiguous
 *     (RadarData/__init__.py:136-137).  `batch` profiles are stacked (batch, snum, tnum).
 *   - Unless a parameter is documented as HOST, pointers are DEVICE pointers on the current CUDA device.
 *     Small coefficient vectors (filter taps, states) are HOST pointers and are copied at launch.
 *   - `stream` is a cudaStream_t passed as void*.  Calls enqueue work and return; they never synchronise
 *     (except the *_host entry points, which own their transfers and return finished results).
 *   - Return value: 0 ok; 1 bad argument; 2 CUDA error; 3 cuFFT error.  impdar_b200_last_error() gives
 *     the message of the last failure on the calling thread.
 *   - No torch types, no C++ types: plain pointers and sizes.
 */
#ifndef IMPDAR_B200_H
#define IMPDAR_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IMPDAR_B200_OK 0
#define IMPDAR_B200_EINVAL 1
#define IMPDAR_B200_ECUDA 2
#define IMPDAR_B200_ECUFFT 3

int impdar_b200_version(void);
const char *impdar_b200_last_error(void);
/* Number of kernels launched by this library on the calling process since load (bench `gpu_launches`). */
unsigned long long impdar_b200_launch_count(void);
/* Measurement hook (bench.py roofline): while on, the dominant kernel of every path is bracketed by CUDA events
 * on the stream it is launched on.  impdar_b200_kernel_timer(1) clears earlier records; returns the previous
 * state.  _read sums the recorded launches of `kernel` (a __global__ function name such as "kirch_table_kernel";
 * NULL = all timed kernels) and synchronises on their events.                                           */
int impdar_b200_kernel_timer(int on);
int impdar_b200_kernel_timer_read(const char *kernel, double *total_ms, int *launches);

/* ---------------------------------------------------------------- taper (mig_python.py:152-157) --- */
/* y = x * h[t] * v[s],  h = min(min(t, T-1-t)/htaper, 1), v likewise.  trunc_int != 0 reproduces the
 * reference's cast back to an integer input dtype (truncation toward zero).  x == y allowed.          */
int impdar_taper_f32(const float *x, float *y, int snum, int tnum, int batch, double htaper,
                     double vtaper, int trunc_int, void *stream);
/* float64 radargrams: y = x * (h[t] * v[s]), one rounding per product in the reference's order (the time-wavenumber
 * stub's in-place `data *= H * V`, mig_python.py:330-335) - bit-exact against numpy.                   */
int impdar_taper_f64(const double *x, double *y, int snum, int tnum, int batch, double htaper, double vtaper,
                     void *stream);

/* ----------------------------------------------- horizontalfilt (_RadarDataFiltering.py:93-135) --- */
/* y[s,t] = x[s,t] - (T)(mean(x[s, htr1:htrn]) * taper[s]);  taper: device, snum doubles.
 * trunc_avg != 0 truncates the scaled mean toward zero first (integer input dtype).                   */
int impdar_hfilt_f32(const float *x, float *y, int snum, int tnum, int batch, int htr1, int htrn,
                     const double *taper, int trunc_avg, void *stream);
int impdar_hfilt_f64(const double *x, double *y, int snum, int tnum, int batch, int htr1, int htrn,
                     const double *taper, int trunc_avg, void *stream);

/* ------------------------------------------------ adaptivehfilt (_RadarDataFiltering.py:19-90) --- */
/* Per trace i the mean over the reference's column window, the 7-tap triangular time filter that
 * filtfilt([.25]*4, 1, .) amounts to on the odd-extended mean trace, the exp taper, the subtraction.
 * Requires snum > 12 (scipy's padlen).  workspace: impdar_ahfilt_workspace_bytes() bytes (may be 0). */
size_t impdar_ahfilt_workspace_bytes(int snum, int tnum, int batch);
/* Testing hook: 0 = auto (register-scan strip kernel for float radargrams with tnum % 4 == 0, first strip kernel
 * otherwise; warp-sliding kernel for windows wider than their buffers), 1 = the one-row-per-CTA kernel, 2 = the first
 * strip kernel, 3 = the warp-sliding kernel.                                                                        */
int impdar_ahfilt_force_rowwise(int on);
int impdar_ahfilt_f32(const float *x, float *y, int snum, int tnum, int batch, int window_size,
                      const double *taper, void *workspace, size_t workspace_bytes, void *stream);
int impdar_ahfilt_f64(const double *x, double *y, int snum, int tnum, int batch, int window_size,
                      const double *taper, void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------- vertical_band_pass (_RadarDataFiltering.py:469-549): filtfilt --- */
/* scipy.signal.filtfilt(b, a, x, axis=0), padtype 'odd': transposed direct-form-II in fp64 state, one
 * trace per thread.  b, a, zi: HOST pointers; b and a have ncoef entries (normalised so a[0] == 1,
 * zero-padded to a common length), zi has ncoef-1 entries (scipy.signal.lfilter_zi).
 * 2 <= ncoef <= 33, snum > padlen.  workspace holds the forward pass over the padded trace.           */
size_t impdar_filtfilt_workspace_bytes(int snum, int tnum, int batch, int padlen, int elem_bytes);
int impdar_filtfilt_f32(const float *x, float *y, int snum, int tnum, int batch, const double *b,
                        const double *a, int ncoef, const double *zi, int padlen, void *workspace,
                        size_t workspace_bytes, void *stream);
int impdar_filtfilt_f64(const double *x, double *y, int snum, int tnum, int batch, const double *b,
                        const double *a, int ncoef, const double *zi, int padlen, void *workspace,
                        size_t workspace_bytes, void *stream);
/* y = scipy.signal.lfilter(taps, 1, x, axis=0) (the 'fir' branch, :536-540).  taps: HOST, ntaps<=1024 */
int impdar_fir_f32(const float *x, float *y, int snum, int tnum, int batch, const double *taps,
                   int ntaps, void *stream);
int impdar_fir_f64(const double *x, double *y, int snum, int tnum, int batch, const double *taps,
                   int ntaps, void *stream);

/* ------------------------------------------------- sibling filters (SURVEY.md 8f rank 2) --- */
/* winavg_hfilt (_RadarDataFiltering.py:353-440): y[s,i] = x[s,i] - (T)(mean(x[s, max(0,i-half) : min(T,i+half)])
 * * taper[s]), half = (avg_win - 1) / 2 after the reference's odd/size corrections (:392-398); taper: device, snum
 * doubles (the 'full' or 'pexp' taper, :399-409).  workspace: impdar_winavg_workspace_bytes() bytes (may be 0).  */
size_t impdar_winavg_workspace_bytes(int snum, int tnum, int batch);
int impdar_winavg_f32(const float *x, float *y, int snum, int tnum, int batch, int half, const double *taper,
                      void *workspace, size_t workspace_bytes, void *stream);
int impdar_winavg_f64(const double *x, double *y, int snum, int tnum, int batch, int half, const double *taper,
                      void *workspace, size_t workspace_bytes, void *stream);
/* highpass / lowpass / horizontal_band_pass (_RadarDataFiltering.py:138-350): scipy.signal.filtfilt(b, a, x, axis=-1),
 * i.e. along the TRACE axis, one recurrence per sample row.  Arguments as impdar_filtfilt_*; tnum > padlen.        */
size_t impdar_filtfilt_rows_workspace_bytes(int snum, int tnum, int batch, int padlen, int elem_bytes);
int impdar_filtfilt_rows_f32(const float *x, float *y, int snum, int tnum, int batch, const double *b,
                             const double *a, int ncoef, const double *zi, int padlen, void *workspace,
                             size_t workspace_bytes, void *stream);
int impdar_filtfilt_rows_f64(const double *x, double *y, int snum, int tnum, int batch, const double *b,
                             const double *a, int ncoef, const double *zi, int padlen, void *workspace,
                             size_t workspace_bytes, void *stream);
/* agc / rangegain (_RadarDataProcessing.py:456-496).  rowabsmax: out[b*snum + s] = max_t |x[b,s,t]| (device doubles;
 * NaN propagates).  rowgain: y[s,t] = x[s,t] * gain[s] where s > trig[t] (trig: device tnum ints, NULL = every
 * row); gain: device snum doubles; in_double != 0 forms the product in float64 and casts back (numpy's in-place
 * multiply by a float64 gain), 0 casts the gain to the data type first (agc's .astype(dtype)).  x == y allowed.   */
int impdar_rowabsmax_f32(const float *x, double *out, int snum, int tnum, int batch, void *stream);
int impdar_rowabsmax_f64(const double *x, double *out, int snum, int tnum, int batch, void *stream);
int impdar_rowgain_f32(const float *x, float *y, int snum, int tnum, int batch, const double *gain, const int *trig,
                       int in_double, void *stream);
int impdar_rowgain_f64(const double *x, double *y, int snum, int tnum, int batch, const double *gain, const int *trig,
                       int in_double, void *stream);

/* ------------------------------------------------------ Kirchhoff (mig_python.py:35-123) --- */
/* out[:, x - x_begin] for output traces x in [x_begin, x_end) of the (snum, tnum) radargram `data`
 * (the whole input is needed: the aperture is only limited by 2r/v <= max(tt)).
 *   dist_m : HOST, tnum doubles, trace positions in metres (dat.dist * 1e3, mig_python.py:108)
 *   tt_s   : HOST, snum doubles, two-way travel time in seconds (strictly ascending)
 *   grad_coef : HOST, 3*snum doubles: rows a, b, c of np.gradient's stencil g[s] = a f[s-1] + b f[s] + c f[s+1]
 *            (b == 0 everywhere selects numpy's uniform-spacing branch; see impdar_b200/migrationlib.py)
 *   out    : (snum, x_end - x_begin) floats
 * The nearest-sample pick and the 2r/v > max(tt) cut are evaluated with the reference's float64
 * operation sequence wherever float32 could decide differently, so the chosen samples are identical. */
size_t impdar_kirchhoff_workspace_bytes(int snum, int tnum, int nearfield);
int impdar_kirchhoff_f32(const float *data, float *out, int snum, int tnum, const double *dist_m,
                         const double *tt_s, const double *grad_coef, double vel, int nearfield,
                         int x_begin, int x_end, void *workspace, size_t workspace_bytes, void *stream);
/* Row-range form of impdar_kirchhoff_f32 for overlapping the diffraction sum with a collective (the multi-GPU path
 * broadcasts the input bottom-up in row chunks and gathers finished output rows while the next chunk runs): computes
 * output rows [s_begin, s_end) of the range [x_begin, x_end) into the full (snum, x_end - x_begin) buffer `out`.  An
 * output row only reads input rows >= s_begin - 1, so only those need to be valid in `data`.  Calls of one image go
 * bottom-up on the same workspace and stream: the first passes g_hi = snum (full preparation), every later one passes
 * the previous call's s_begin (its d/dt rows and the tables are reused).  Uniform trace spacing only (status 1
 * otherwise: use impdar_kirchhoff_f32).                                                                          */
int impdar_kirchhoff_rows_f32(const float *data, float *out, int snum, int tnum, const double *dist_m,
                              const double *tt_s, const double *grad_coef, double vel, int nearfield, int x_begin,
                              int x_end, int s_begin, int s_end, int g_hi, void *workspace, size_t workspace_bytes,
                              void *stream);
/* Column-window form (the multi-GPU halo exchange): `data` holds only the radargram columns [col0, col0 + ncols)
 * (row stride ld floats) and `out` has row stride ldo (>= x_end - x_begin; pass the full image + x_begin with ldo = tnum
 * to write a rank's block straight into its final place - also through a peer-mapped pointer).  Geometry vectors stay
 * those of the WHOLE radargram, so tables, picks and summation order - and therefore the result - are bit for bit what
 * impdar_kirchhoff_f32 gives on the whole input.  The window must cover every column the range can read:
 * impdar_kirchhoff_input_window() returns that interval (range + one aperture each side, by distance and by trace
 * count).  s_begin / s_end / g_hi as in impdar_kirchhoff_rows_f32; (0, snum, snum) = whole image, any geometry.   */
int impdar_kirchhoff_input_window(int snum, int tnum, const double *dist_m, const double *tt_s, double vel,
                                  int x_begin, int x_end, int *col0, int *col1);
int impdar_kirchhoff_window_f32(const float *data, int col0, int ncols, int ld, float *out, int ldo, int snum,
                                int tnum, const double *dist_m, const double *tt_s, const double *grad_coef,
                                double vel, int nearfield, int x_begin, int x_end, int s_begin, int s_end, int g_hi,
                                void *workspace, size_t workspace_bytes, void *stream);
/* Host-to-host Kirchhoff with the transfers overlapped (the RadarData.migrate(mtype='kirch') call on a host array):
 * h_data HOST (snum, tnum) floats, h_out HOST (snum, tnum) doubles - page-locked memory makes the copies truly
 * asynchronous.  An output row only reads input rows at or below it (the hyperbola runs downwards in time), so the
 * image is processed bottom-up in `nchunks` row chunks: upload | d/dt + diffraction sum | widen to float64 + download
 * on three streams.  Uniform trace spacing only; irregular geometry runs the three phases back to back.  The call
 * returns after enqueueing; synchronise `stream` before reading h_out.                                           */
size_t impdar_kirchhoff_host_workspace_bytes(int snum, int tnum, int nearfield);
int impdar_kirchhoff_host_pipelined_f64(const float *h_data, double *h_out, int snum, int tnum, const double *dist_m,
                                        const double *tt_s, const double *grad_coef, double vel, int nearfield,
                                        int nchunks, void *workspace, size_t workspace_bytes, void *stream);
/* Depth-varying velocity: the _vz forms take vel_s, HOST, snum doubles - the RMS velocity of each output row (straight
 * rays; row ti migrates with v[ti] wherever the scalar forms use vel).  Each must be finite and > 0 (status 1
 * otherwise).  A constant vector gives bit for bit the scalar form's result.  impdar_kirchhoff_window_vz_f32 with
 * (col0, ncols) = (0, tnum) and rows (0, snum, snum) is the whole-image call, for any trace order, like
 * impdar_kirchhoff_f32; otherwise it is the column-window / row-chunk form above.                                  */
int impdar_kirchhoff_window_vz_f32(const float *data, int col0, int ncols, int ld, float *out, int ldo, int snum,
                                   int tnum, const double *dist_m, const double *tt_s, const double *grad_coef,
                                   const double *vel_s, int nearfield, int x_begin, int x_end, int s_begin, int s_end,
                                   int g_hi, void *workspace, size_t workspace_bytes, void *stream);
int impdar_kirchhoff_input_window_vz(int snum, int tnum, const double *dist_m, const double *tt_s, const double *vel_s,
                                     int x_begin, int x_end, int *col0, int *col1);
int impdar_kirchhoff_host_pipelined_vz_f64(const float *h_data, double *h_out, int snum, int tnum,
                                           const double *dist_m, const double *tt_s, const double *grad_coef,
                                           const double *vel_s, int nearfield, int nchunks, void *workspace,
                                           size_t workspace_bytes, void *stream);
/* Laterally varying velocity: output trace xi migrates with profile col_profile[xi] of `profiles` (HOST, nprof x snum
 * doubles, RMS velocities, each finite and > 0; col_profile: HOST, tnum ints in [0, nprof); status 1 otherwise).
 * Column xi equals column xi of impdar_kirchhoff_window_vz_f32 run with that profile.  Window arguments as there (the
 * window must cover impdar_kirchhoff_input_window_vz's interval for the row-wise largest velocity); whole image only
 * (no row chunks); (col0, ncols) = (0, tnum) accepts any trace order.  Path: with uniform trace spacing and runs of one
 * profile at least 192 traces wide on average over all tnum traces, one single-profile table-path call per run of
 * [x_begin, x_end) on its own input sub-window
 * (bit for bit the whole-image single-profile call for finite input); otherwise the lateral general kernel
 * (impdar_kirchhoff_last_path() == 4).  The workspace has impdar_kirchhoff_lateral_workspace_bytes() bytes.      */
size_t impdar_kirchhoff_lateral_workspace_bytes(int snum, int tnum, int nprof, int nearfield);
int impdar_kirchhoff_window_vxz_f32(const float *data, int col0, int ncols, int ld, float *out, int ldo, int snum,
                                    int tnum, const double *dist_m, const double *tt_s, const double *grad_coef,
                                    const double *profiles, int nprof, const int *col_profile, int nearfield,
                                    int x_begin, int x_end, void *workspace, size_t workspace_bytes, void *stream);
/* Counters of the last impdar_kirchhoff_f32 call (for the roofline): (output sample, input trace) pairs
 * inside the aperture and pairs that took the float64 exact path.  Counting pairs costs an instruction
 * per pair, so it is off unless enabled.  last_stats synchronises the stream of that call.            */
int impdar_kirchhoff_enable_stats(int on);
/* Kernel selection (per host thread): 0 = automatic (uniform-geometry table path when the trace spacing is uniform,
 * the general-geometry kernel otherwise), 1 = always the general kernel, 2 = require the table path (shared-memory
 * tile kernel for the far-field sum, global-gather table kernel for near field / non-finite input), 3 = table path
 * with the global-gather kernel only.  impdar_kirchhoff_last_path(): 1 general, 2 table (gather), 3 table (tile),
 * 4 lateral general kernel.                                                                                        */
int impdar_kirchhoff_set_mode(int mode);
int impdar_kirchhoff_last_path(void);
/* After a table-path call whose last_path is 3 (shared-memory tile kernel launched): *stood_down = 1 when the tile
 * kernel left the work to the gather kernel (non-finite input, or hyperbola intervals wider than its staging
 * segments), 0 when it did the work; -1 when the last call did not launch it.  Synchronises that call's stream. */
int impdar_kirchhoff_last_tile_standdown(int *stood_down);
int impdar_kirchhoff_last_stats(unsigned long long *pairs, unsigned long long *exact_pairs);

/* Peer-mapped image (multi-GPU Kirchhoff, the serial trace loop of mig_python.py:35-60 split into output-trace ranges
 * over one process per GPU): the rank that holds the radargram allocates the (snum, tnum) image with impdar_peer_alloc
 * (cudaMalloc on the current device; `handle64` HOST, 64 bytes: the CUDA IPC handle to hand to the other processes of
 * the node), every other rank maps it with impdar_peer_open (current device = its own GPU; peer access over NVLink /
 * NVSwitch) and passes `mapped + x_begin` with ldo = tnum as `out` of impdar_kirchhoff_window_f32: the diffraction-sum
 * kernels store their block straight into the holder's memory while they run.  Close every mapping before the holder
 * frees.  impdar_copy2d_f32 is a strided device-to-device block copy (rows x cols floats) on `stream`.            */
int impdar_peer_alloc(size_t bytes, void **ptr, void *handle64);
int impdar_peer_free(void *ptr);
int impdar_peer_open(const void *handle64, void **ptr);
int impdar_peer_close(void *ptr);
int impdar_copy2d_f32(const float *src, size_t lds, float *dst, size_t ldd, int rows, int cols, void *stream);

/* Reference prototype, migrationlib/mig_cython.h:11 - HOST pointers, float64, synchronous.  Linking
 * the reference's own Cython shim (_mig_cython.pyx) against libimpdar_b200.so resolves this symbol.
 * nearfield != 0 needs the un-differentiated data, which this prototype does not carry: the call then
 * fills migdata with NaN and records an error (use impdar_kirchhoff_host_f64 instead).                */
void mig_kirch_loop(double *migdata, int tnum, int snum, double *dist, double *zs, double *zs2,
                    double *tt_sec, double vel, double *gradD, double max_travel_time, int nearfield);
/* Same, with the data pointer and a status: HOST float64 in/out (the drop-in for migrationKirchhoff). */
int impdar_kirchhoff_host_f64(const double *data, double *migdata, int snum, int tnum,
                              const double *dist_m, const double *tt_s, double vel, int nearfield);

/* ---------------------------------------------------------- Stolt (mig_python.py:126-208) --- */
/* data (batch, snum, tnum) -> out (batch, 2*(snum/2), tnum).  dx = mean trace spacing [m] (:163-168). */
size_t impdar_stolt_workspace_bytes(int snum, int tnum, int batch);
int impdar_stolt_f32(const float *data, float *out, int snum, int tnum, int batch, double dt, double dx,
                     double vel, double htaper, double vtaper, int trunc_int, void *workspace,
                     size_t workspace_bytes, void *stream);

/* Testing hook: 1 forces the generic R2C/C2R pipeline even where the paired-trace C2C pipeline (even snum and
 * tnum) applies; 0 restores automatic selection.                                                      */
int impdar_stolt_force_r2c(int on);
/* Pipeline selection: 0 automatic (the five-pass hand-written transform kernels for snum in {512..8192} and tnum in
 * {8192..131072}, powers of two; otherwise cuFFT paired-trace C2C for even shapes; otherwise cuFFT R2C/C2R),
 * 1 cuFFT R2C/C2R, 2 cuFFT paired C2C, 3 five-pass kernels (EINVAL at call time for shapes they do not cover). */
int impdar_stolt_set_pipeline(int mode);
/* 1, 2 or 3 as above: what the last impdar_stolt_f32 call ran. */
int impdar_stolt_last_pipeline(void);
/* Testing hook for the five-pass pipeline: stop after pass 1..5 (0 = run everything).  After pass 1 or 4 `out`
 * holds W1 (snum x tnum/2 complex); after pass 2 or 3 the workspace (256-byte aligned) holds the transposed half
 * spectrum (tnum/2 x snum complex).  tests/stolt_stage_model.py restates each stage.                    */
int impdar_stolt_debug_stop_after(int stage);

/* -------------------------------------- phase shift (mig_python.py:211-287, 361-493) --- */
/* data (snum, tnum) -> out (snum, tnum).  vmig == NULL: constant velocity `vel` (:396-420);
 * otherwise vmig: device, snum doubles, the layered profile from getVelocityProfile (:439-487) and
 * thr2: device, snum doubles, the per-tau evanescent threshold (tau/travel_time[-1]/1e6)^2 (:484).
 * tt0 is unused by the reference arithmetic and therefore absent.                                      */
size_t impdar_phsh_workspace_bytes(int snum, int tnum);
int impdar_phsh_f32(const float *data, float *out, int snum, int tnum, double dt, double dx, double vel,
                    const double *vmig, const double *thr2, double htaper, double vtaper,
                    void *workspace, size_t workspace_bytes, void *stream);

/* Laterally varying velocity v(x, z): split-step Fourier + explicit finite-difference branch of phaseShift
 * (mig_python.py:428-432, 439-487; fourierFiniteDiff :496-525; Sp_Matr :528-540).  float64 end to end (the thin-lens
 * phase reaches 1e9 rad and the update is one serial chain over snum * nt steps).
 *   data, out : device (snum, tnum) doubles;  vmig : device (snum, tnum) doubles from getVelocityProfile (:606-640)
 *   thr2 : device snum doubles (as above);  dx : mean trace spacing used for kx (:260-265);
 *   dx_fd : np.mean(dat.trace_int), the spacing fourierFiniteDiff uses (:517)                            */
size_t impdar_phsh_ffd_workspace_bytes(int snum, int tnum);
int impdar_phsh_ffd_f64(const double *data, double *out, int snum, int tnum, double dt, double dx, double dx_fd,
                        const double *vmig, const double *thr2, double htaper, double vtaper, void *workspace,
                        size_t workspace_bytes, void *stream);

/* Kernel selection of impdar_phsh_f32 (testing / A-B hook): 0 = automatic - constant velocity runs as a per-kx complex
 * matrix product on the tensor cores (tcgen05.mma kind::tf32 with the 3xTF32 split, accumulators in TMEM, drained every
 * stage; csrc/phaseshift_tc.cu), layered velocity on the (+w, -w) pair kernel; 1 = the first-generation
 * one-bin-per-state SIMT kernels; 2 = same as 0; 3 = the SIMT pair kernels for both velocity models.              */
int impdar_phsh_set_legacy(int mode);

/* ------------------------------------ index / resampling operations (_RadarDataProcessing.py:20-637) --- */
/* All bit-exact against the reference's numpy 2.3 / scipy 1.18 arithmetic (operation order, no FMA contraction).
 * Suffix _f32 / _f64: input and output in that type (the device-resident lane); _f32_f64: float32 input,
 * float64 output (what the reference produces on the host for a float32 radargram).
 *
 * crop (:238-313 crop, :352-421 hcrop, :20-29 reverse): y (r1-r0, c1-c0) = x[r0:r1, c0:c1], flip_lr != 0 = np.fliplr. */
int impdar_crop_f32(const float *x, float *y, int snum, int tnum, int batch, int r0, int r1, int c0, int c1,
                    int flip_lr, void *stream);
int impdar_crop_f64(const double *x, double *y, int snum, int tnum, int batch, int r0, int r1, int c0, int c1,
                    int flip_lr, void *stream);
/* the same block copy for any element size in {1, 2, 4, 8, 16} bytes (integer and complex radargrams). */
int impdar_crop_bytes(const void *x, void *y, int snum, int tnum, int batch, int r0, int r1, int c0, int c1,
                      int flip_lr, int elem_bytes, void *stream);
/* per-trace vertical shift with NaN fill (:314-330 crop(dimension='pretrig') with a trigger vector, shift = trig;
 * :587-637 elev_correct, shift = -top_ind):  y[i, t] = x[i + shift[t], t] if 0 <= i + shift[t] < snum_in else NaN.
 * shift: device, tnum ints.  y is (snum_out, tnum).                                                         */
int impdar_shift_traces_f32(const float *x, float *y, int snum_in, int tnum, int snum_out, const int *shift,
                            void *stream);
int impdar_shift_traces_f32_f64(const float *x, double *y, int snum_in, int tnum, int snum_out, const int *shift,
                                void *stream);
int impdar_shift_traces_f64(const double *x, double *y, int snum_in, int tnum, int snum_out, const int *shift,
                            void *stream);
/* restack (:424-477): y (snum, tnum / traces) = np.mean over consecutive groups of `traces` columns, summed in
 * numpy's pairwise order in the input precision.                                                            */
int impdar_restack_f32(const float *x, float *y, int snum, int tnum, int traces, void *stream);
int impdar_restack_f32_f64(const float *x, double *y, int snum, int tnum, int traces, void *stream);
int impdar_restack_f64(const double *x, double *y, int snum, int tnum, int traces, void *stream);
/* linear interpolation between two source rows (:66-188 nmo, :50-63 constant_sample_depth_spacing) or two source
 * columns (:499-584 constant_space) per output row / column.  nodes: device array of snum_out (tnum_out) records
 * of impdar_interp_node_bytes() bytes { int lo, hi; double a, b, den; int exact, pad; }, built on the host in
 * float64 (O(n)).  mode 0 = scipy interp1d._call_linear: y = a*x[hi] + b*x[lo];  mode 1 = numpy.interp:
 * slope = (x[hi]-x[lo])/den, y = slope*a + x[lo] (exact != 0: y = x[lo]; NaN: retried as slope*b + x[hi]).   */
size_t impdar_interp_node_bytes(void);
int impdar_interp_rows_f32(const float *x, float *y, int snum_in, int tnum, int snum_out, const void *nodes,
                           int mode, void *stream);
int impdar_interp_rows_f32_f64(const float *x, double *y, int snum_in, int tnum, int snum_out, const void *nodes,
                               int mode, void *stream);
int impdar_interp_rows_f64(const double *x, double *y, int snum_in, int tnum, int snum_out, const void *nodes,
                           int mode, void *stream);
int impdar_interp_cols_f32(const float *x, float *y, int snum, int tnum_in, int tnum_out, const void *nodes,
                           int mode, void *stream);
int impdar_interp_cols_f32_f64(const float *x, double *y, int snum, int tnum_in, int tnum_out, const void *nodes,
                               int mode, void *stream);
int impdar_interp_cols_f64(const double *x, double *y, int snum, int tnum_in, int tnum_out, const void *nodes,
                           int mode, void *stream);

/* ------------------------------------------------------- denoise (_RadarDataFiltering.py:552-587) --- */
/* scipy.signal.wiener(x, mysize=(vert_win, hor_win), noise): float64 box statistics, float64 output y (snum, tnum).
 * estimate_noise != 0: noise = mean of the local variance (scipy's noise=None), `noise` is ignored.
 * scratch: device, 16 bytes; after the call scratch[0] (double) holds the sum of the local variance and the int at
 * byte 8 is 1 if some local variance is exactly zero (scipy divides by it; the reference raises ValueError).    */
int impdar_wiener_f32(const float *x, double *y, int snum, int tnum, int vert_win, int hor_win, int estimate_noise,
                      double noise, double *scratch, void *stream);
int impdar_wiener_f64(const double *x, double *y, int snum, int tnum, int vert_win, int hor_win, int estimate_noise,
                      double noise, double *scratch, void *stream);
/* denoise(ftype='median') = scipy.ndimage.median_filter(x, size=(vert_win, hor_win)) (mode 'reflect'): rank
 * (vert_win*hor_win)/2 of the window rows [s - V/2, s - V/2 + V), columns likewise; bit-exact selection.  Windows of up
 * to 256 samples; y != x.  NaN ordering is unspecified (as in scipy).                                              */
int impdar_median_f32(const float *x, float *y, int snum, int tnum, int vert_win, int hor_win, void *stream);
int impdar_median_f64(const double *x, double *y, int snum, int tnum, int vert_win, int hor_win, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* IMPDAR_B200_H */
