/*
 * wavelets_b200.h -- C ABI of the B200 (sm_100a) à trous / WOW hot path.
 *
 * The reference (frederic-auchere/wavelets, "watroo" 0.0.4) is pure Python: it has no FFI of its own, its hot path
 * bottoms out in cv2.filter2D / numexpr / NumPy calls.  Each entry point below replaces one of those call sites;
 * the reference-side binding a maintainer would add is a ctypes stub (see INTEGRATION.md).  The host layer that
 * mirrors the reference's Python API on top of this ABI is wavelets_b200/{wavelets,utils}.py.
 *
 * Conventions (all entry points):
 *   - every pointer is a DEVICE pointer on the current CUDA device; the caller allocates every output and every
 *     workspace (the library never allocates or frees device memory);
 *   - images are row-major, innermost stride 1; `*_pitch` is the row stride and `*_bstride` the frame (batch)
 *     stride, both in ELEMENTS; `batch` frames are processed by one launch;
 *   - dtype: WB_F32 or WB_F64 (the arithmetic type of the path: the reference computes in the image dtype);
 *   - taps: WB_TRIANGLE (3 taps, [1/4,1/2,1/4]) or WB_B3SPLINE (5 taps, [1/16,1/4,3/8,1/4,1/16])
 *     (watroo/wavelets.py:239, :268);
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous and never synchronise the device;
 *   - return value: 0 on success, a negative WB_E* code for a rejected argument, or a positive cudaError_t;
 *     wb_error_string() renders both.  Nothing is written when a negative code is returned.
 *   - border rule everywhere: half-sample symmetric reflection (cv2.BORDER_REFLECT == np.pad 'symmetric'),
 *     any number of reflections.
 */
#ifndef WAVELETS_B200_H
#define WAVELETS_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WB_ABI_VERSION 2
#define WB_MAX_PEERS 16 /* ranks of one NVLink domain whose band buffers wb_atrous_scale_band_p2p can address */

enum { WB_F32 = 0, WB_F64 = 1 };
enum { WB_TRIANGLE = 3, WB_B3SPLINE = 5 };
/* border rule of wb_atrous_axis: half-sample symmetric (cv2.BORDER_REFLECT, every 2-D / 3-D pass of the reference) or
 * whole-sample mirror (scipy.ndimage mode='mirror', the reference's 1-D signals) */
enum { WB_BORDER_SYMMETRIC = 0, WB_BORDER_MIRROR = 1 };

enum {
    WB_OK = 0,
    WB_EINVAL_DTYPE = -1,
    WB_EINVAL_TAPS = -2,
    WB_EINVAL_SHAPE = -3,
    WB_EINVAL_SCALE = -4,
    WB_EINVAL_POINTER = -5,
    WB_EINVAL_ARG = -6,
    WB_ENOT_FUSABLE = -7 /* wb_wow_scale only: shape/alignment outside the fused kernel; use the two-pass route */
};

/* ABI version of the loaded library (== WB_ABI_VERSION of the header it was built from). */
int wb_abi_version(void);

/* Human-readable text for a status returned by any entry point. */
const char *wb_error_string(int status);

/* Which kernel variant wb_atrous_scale would launch for this problem: 1 = TMA row-pipeline kernel,
 * 0 = generic gather kernel (unaligned / tiny images).  For tests and the benchmark report. */
int wb_atrous_scale_path(int H, int W, long long in_pitch, long long out_pitch, int scale, int taps, int dtype,
                         const void *in, const void *out_c, const void *out_w);

/*
 * One scale of the plain cascade.  Replaces watroo/wavelets.py:35-45 (`convolution`, 2-D branch: cv2.filter2D with
 * the dilated dense kernel of :191-197 and BORDER_REFLECT) fused with the subtraction of :442:
 *     out_c(y,x) = sum_i sum_j h_i h_j in(R(y+(i-c)2^scale), R(x+(j-c)2^scale))          (c_{s+1})
 *     out_w      = in - out_c                                                            (w_s)
 * `in` is never written.  `out_w` may be NULL (smooth only); `out_c` may be NULL (detail plane only).
 * `out_c`/`out_w` must not alias `in` (rows of `in` are re-read as halo by neighbouring thread blocks).
 */
int wb_atrous_scale(const void *in, void *out_c, void *out_w, int batch, int H, int W,
                    long long in_pitch, long long in_bstride,
                    long long out_c_pitch, long long out_c_bstride,
                    long long out_w_pitch, long long out_w_bstride,
                    int scale, int taps, int dtype, void *stream);

/*
 * The whole plain cascade.  Replaces AtrousTransform.atrous_standard with bilateral=None
 * (watroo/wavelets.py:408-432,442-444).  `planes` is the (batch, levels+1, H, W) C-contiguous coefficient array
 * ([w_0 .. w_{L-1}, c_L] per frame); `scratch` is a caller-provided workspace of 2*batch*H*W elements that holds
 * the running smooth planes (c_s ping-pong).  `in` (pitch in_pitch, frame stride in_bstride) is not modified.
 * levels == 0 copies the image into plane 0.
 */
int wb_atrous_transform(const void *in, void *planes, void *scratch, int batch, int H, int W,
                        long long in_pitch, long long in_bstride, int levels, int taps, int dtype, void *stream);

/*
 * One scale of the plain cascade on ONE ROW BAND of a taller image (multi-GPU row-band sharding, no reference
 * equivalent: the reference is single-process).  The band owns global rows [band_y0, band_y0 + band_rows) of an image
 * of height global_H.  `in` is a buffer whose row `in_row_offset + i` holds global row band_y0 + i, for every i in
 * [-c*2^scale, band_rows + c*2^scale) that falls inside the image (c = taps/2): the halo rows just outside the band
 * must have been filled by the caller (neighbour exchange); rows beyond the global top/bottom are taken by symmetric
 * reflection about global_H and must then lie inside the same window.  Output row i goes to row
 * out_*_row_offset + i of out_c / out_w.  The arithmetic is the same as wb_atrous_scale's, so a banded cascade is
 * bit-identical to the single-device one.
 */
int wb_atrous_scale_band(const void *in, void *out_c, void *out_w, int band_rows, int W, int global_H,
                         long long band_y0, long long in_row_offset, long long in_pitch,
                         long long out_c_row_offset, long long out_c_pitch,
                         long long out_w_row_offset, long long out_w_pitch,
                         int scale, int taps, int dtype, void *stream);

/*
 * One scale of the plain cascade with the border rule of the reference's RECURSIVE algorithm
 * (AtrousTransform.atrous_recursive, watroo/wavelets.py:330-406, parity mode of `recursive=True`): the image is seen as
 * its 2^scale x 2^scale decimated sub-arrays and every tap reflects (half-sample symmetric) at the edges of ITS
 * sub-array, not of the full image.  Always the generic gather kernel (a parity mode, not a fast path).  The caller
 * pads the image symmetrically by (taps/2) * 2^(levels-1) first and crops the planes afterwards, as the reference does.
 */
int wb_atrous_scale_lattice(const void *in, void *out_c, void *out_w, int H, int W, long long in_pitch,
                            long long out_c_pitch, long long out_w_pitch, int scale, int taps, int dtype, void *stream);

/*
 * wb_atrous_scale_bilateral on ONE ROW BAND of a taller image (multi-GPU row bands, no reference equivalent): same
 * window conventions as wb_atrous_scale_band -- `in` holds the band's rows of c_s plus the halo rows of the neighbours
 * ((taps/2) * 2^scale above and below, filled by the caller), taps reflect about global_H.  Same arithmetic as the
 * unsharded kernel: bit-identical planes.
 */
int wb_atrous_scale_bilateral_band(const void *in, void *out_c, void *out_w, int band_rows, int W, int global_H,
                                   long long band_y0, long long in_row_offset, long long in_pitch,
                                   long long out_c_row_offset, long long out_c_pitch, long long out_w_row_offset,
                                   long long out_w_pitch, int scale, int taps, int dtype, double var_factor,
                                   void *stream);

/*
 * The bilateral counterpart of wb_atrous_scale_lattice: one scale of the reference's RECURSIVE algorithm with
 * AtrousTransform(bilateral=...) (watroo/wavelets.py:371-378: sdev_loc and atrous_convolution on every decimated
 * sub-array, each with the symmetric border at ITS OWN edges).  Generic gather kernel (a parity mode).
 */
int wb_atrous_scale_bilateral_lattice(const void *in, void *out_c, void *out_w, int H, int W, long long in_pitch,
                                      long long out_c_pitch, long long out_w_pitch, int scale, int taps, int dtype,
                                      double var_factor, void *stream);

/*
 * wb_wow_whiten_scale on ONE ROW BAND of a taller image (row-band sharded WOW, no reference equivalent): same window
 * conventions as wb_atrous_scale_band -- `w_raw` holds the band's raw detail rows plus the halo rows of the
 * neighbours (c * 2^scale above and below, filled by the caller), reflections about global_H.  `noise_dev`, when
 * given, points to ONE device scalar (frame 0).
 */
int wb_wow_whiten_scale_band(const void *w_raw, void *out, int band_rows, int W, int global_H, long long band_y0,
                             long long in_row_offset, long long in_pitch, long long out_row_offset, long long out_pitch,
                             int scale, int taps, int dtype, int sig_mode, double sigma, double sigma_e,
                             double noise_host, const double *noise_dev, double weight, void *stream);

/*
 * wb_atrous_scale_band that also PUSHES the next scale's halo rows to the neighbouring bands (no reference equivalent;
 * multi-GPU row bands, SURVEY.md 8(e)): output rows [0, push_up_rows) of c_{s+1} are stored a second time at
 * push_up + i * out_c_pitch and output rows [band_rows - push_dn_rows, band_rows) at push_dn + i * out_c_pitch, where
 * push_up / push_dn are the addresses -- valid ON THIS DEVICE: peer-mapped memory over NVLink (CUDA IPC / symmetric
 * memory) -- of the place this band's output row 0 has in the upper / lower neighbour's padded c buffer (its halo
 * zone).  Pass NULL / 0 rows at the global top / bottom.  The remote stores are posted writes that overlap with this
 * launch's own streaming; the next scale then reads local memory only (plain wb_atrous_scale_band semantics for
 * everything else).  The caller orders the ranks with one device-side barrier per scale: a neighbour's buffer may be
 * written only after that neighbour has finished the scale that read it, and read only after this launch has completed.
 */
int wb_atrous_scale_band_push(const void *in, void *out_c, void *out_w, int band_rows, int W, int global_H,
                              long long band_y0, long long in_row_offset, long long in_pitch, long long out_c_row_offset,
                              long long out_c_pitch, long long out_w_row_offset, long long out_w_pitch, void *push_up,
                              int push_up_rows, void *push_dn, int push_dn_rows, int scale, int taps, int dtype,
                              void *stream);

/*
 * Row-band scale with the halo rows read IN PLACE from the neighbours' band buffers over NVLink (no halo copy, no
 * padded buffer, no reference equivalent).  The running smooth plane c_s of a global_H-row image is distributed over
 * n_peers ranks: rank k owns global rows [peer_y0[k], peer_y0[k+1]) (peer_y0 has n_peers + 1 entries, peer_y0[0] = 0,
 * peer_y0[n_peers] = global_H) in a buffer that starts at peer_in[k] -- an address valid ON THIS DEVICE (the local
 * buffer for k == rank, peer-mapped memory otherwise: CUDA IPC / symmetric memory).  All buffers share `in_pitch`.
 * The kernel resolves every chain row (after the symmetric reflection about global_H) to its owner and fetches it
 * with the same TMA bulk copy as a local row.  Output row i (global row peer_y0[rank] + i) goes to row i of
 * out_c / out_w (local memory).  `peer_in` and `peer_y0` are HOST arrays, copied into the launch parameters.
 * The caller orders the ranks: every rank must have finished writing its c_s (and reading the buffer that out_c
 * overwrites) before any rank launches this scale -- one device-side barrier per scale.  Same arithmetic as
 * wb_atrous_scale, hence bit-identical to the unsharded cascade.
 */
int wb_atrous_scale_band_p2p(const void *const *peer_in, const long long *peer_y0, int n_peers, int rank,
                             void *out_c, void *out_w, int W, int global_H, long long in_pitch,
                             long long out_c_pitch, long long out_w_pitch, int scale, int taps, int dtype,
                             void *stream);

/*
 * One scale of the BILATERAL cascade.  Replaces, per scale, watroo/wavelets.py:433-442: sdev_loc (:24-32), the
 * variance scaling (:434-436), atrous_convolution(..., bilateral_variance) (:74-105) and the subtraction (:442):
 *     var = S[in^2] - S[in]^2 (<= 0 -> 1e-20),  V = var * var_factor,  var_factor = sigma_b[s]^2 * (s+1 | 1)
 *     out_c = (k_c x + sum_t k_t exp(-(x - x_t)^2 / V / 2) x_t) / (k_c + sum_t k_t exp(...)),   out_w = in - out_c
 * Same pointer rules as wb_atrous_scale.
 */
int wb_atrous_scale_bilateral(const void *in, void *out_c, void *out_w, int batch, int H, int W,
                              long long in_pitch, long long in_bstride,
                              long long out_c_pitch, long long out_c_bstride,
                              long long out_w_pitch, long long out_w_bstride,
                              int scale, int taps, int dtype, double var_factor, void *stream);

/*
 * WOW whitening of one detail plane.  Replaces the body of the per-scale loop of watroo/utils.py:177,193-203:
 *     P   = S_scale[w_raw^2] (plain smooth, never bilateral; <= 0 -> 1e-15),  lp = sqrt(P)
 *     out = w_raw * significance(w_raw) * (weight / lp)
 * significance (watroo/wavelets.py:129-143): sig_mode 0 -> 1; 1 -> erf(|w / thr|); 2 -> (|w| > thr), with
 * thr = (sigma * noise) * sigma_e and noise read from `noise_dev[frame]` (device, e.g. written by wb_abs_median)
 * when non-NULL, else `noise_host`; noise == 0 -> 1.  `out` must not alias `w_raw`.
 */
int wb_wow_whiten_scale(const void *w_raw, void *out, int batch, int H, int W,
                        long long in_pitch, long long in_bstride, long long out_pitch, long long out_bstride,
                        int scale, int taps, int dtype, int sig_mode, double sigma, double sigma_e,
                        double noise_host, const double *noise_dev, double weight, void *stream);

/*
 * wb_wow_whiten_scale with a PER-PIXEL noise map (watroo/wavelets.py:133-141 with an array `noise`), per pixel:
 *     tmp = the sig_mode 0 whitening of w_raw                      (rounded to the plane dtype)
 *     thr = (double)((T)sigma * map) * sigma_e
 *     s   = soft ? erf(|(double)w_raw / thr|) : (|(double)w_raw| > thr ? 1 : 0)      (float64)
 *     out = (T)((double)tmp * s)
 * Bit-identical to wb_wow_whiten_scale (sig_mode 0) -> wb_significance (same map) -> the float64 product.  `noise_map`
 * has the plane dtype; its element (frame, y, x) is at frame * map_bstride + y * map_pitch + x (map_bstride 0: one map
 * for every frame).  sigma == 0 is rejected (WB_EINVAL_ARG): such scales take wb_wow_whiten_scale with sig_mode 0.
 * `out` must alias neither `w_raw` nor `noise_map`.
 */
int wb_wow_whiten_scale_map(const void *w_raw, void *out, const void *noise_map, int batch, int H, int W,
                            long long in_pitch, long long in_bstride, long long out_pitch, long long out_bstride,
                            long long map_pitch, long long map_bstride, int scale, int taps, int dtype, int soft,
                            double sigma, double sigma_e, double weight, void *stream);

/*
 * One WOW scale fused in a single pass: the smooth + subtraction of wb_atrous_scale (watroo/wavelets.py:35-45, :442)
 * AND the whitening of wb_wow_whiten_scale (watroo/utils.py:177,193-203) without ever writing the raw detail plane:
 *     out_c = S_scale[in]                                 (c_{s+1}, needed by the next scale)
 *     w     = in - out_c;  P = S_scale[w^2] (<= 0 -> 1e-15)
 *     out_w = w * significance(w) * (weight / sqrt(P))    (the final, whitened plane s)
 * 3 elements of HBM traffic per pixel instead of 5; results are bit-identical to wb_atrous_scale followed by
 * wb_wow_whiten_scale.  The fused kernel stages whole rows on chip: it takes 16-byte aligned, vector-multiple widths
 * up to 4096 (float32) / 2048 (float64) columns; anything else returns WB_ENOT_FUSABLE before launching anything
 * (wb_wow_scale_path() == 0 tells beforehand) and the caller takes the two-pass route.  Significance arguments as in
 * wb_wow_whiten_scale.  `out_c`, `out_w` and `in` must be three distinct buffers.
 */
int wb_wow_scale_path(int batch, int H, int W, long long in_pitch, long long out_c_pitch, long long out_w_pitch,
                      int scale, int taps, int dtype, const void *in, const void *out_c, const void *out_w);
int wb_wow_scale(const void *in, void *out_c, void *out_w, int batch, int H, int W,
                 long long in_pitch, long long in_bstride,
                 long long out_c_pitch, long long out_c_bstride,
                 long long out_w_pitch, long long out_w_bstride,
                 int scale, int taps, int dtype, int sig_mode, double sigma, double sigma_e,
                 double noise_host, const double *noise_dev, double weight, void *stream);

/*
 * Exact median of |x| over n contiguous elements per frame, on the device and without host synchronisation.
 * Replaces np.median(np.abs(data[0])) of Coefficients.get_noise (watroo/wavelets.py:126-127); bit-identical to
 * np.median (mean of the two middle values, in the plane dtype).  `out_median` (dtype of x, one per frame) and/or
 * `out_noise` (float64, one per frame: (median / 0.6745 in the plane dtype) / sigma_e0 in float64, i.e. get_noise
 * under NumPy >= 2) are written.  `workspace`: `workspace_bytes` bytes of device memory, at least
 * wb_abs_median_workspace_bytes(dtype, batch, 0) (selection state only: every counting pass then streams the plane);
 * with wb_abs_median_workspace_bytes(dtype, batch, n) bytes (state + a quarter of the plane per frame) the first pass
 * copies the values inside the sampled bracket of the median into the workspace and the later passes read only those
 * (one streaming read of the plane instead of two or more).  The result does not depend on the workspace size.
 */
size_t wb_abs_median_workspace_bytes(int dtype, int batch, long long n);
int wb_abs_median(const void *x, long long n, int batch, long long bstride, int dtype, void *out_median,
                  double *out_noise, double sigma_e0, void *workspace, size_t workspace_bytes, void *stream);

/*
 * Population moments of n contiguous elements per frame: out[frame] = {mean, variance, std} (float64).
 * Replaces np.std(c) (watroo/utils.py:187) and data[:-1].std(axis=(1,2)) (watroo/wavelets.py:227).
 * `workspace`: wb_plane_moments_workspace_bytes(batch) bytes.
 */
size_t wb_plane_moments_workspace_bytes(int batch);
int wb_plane_moments(const void *x, long long n, int batch, long long bstride, int dtype, double *out,
                     void *workspace, void *stream);

/*
 * Significance map of one plane (Coefficients.significance, watroo/wavelets.py:129-143).
 * soft != 0: out is float64[n] = erf(|w / thr|); soft == 0: out is uint8[n] = (|w| > thr).
 * thr = (sigma * noise) * sigma_e; noise = *noise_dev if non-NULL else noise_host, or a per-pixel `noise_map`
 * (dtype of w) if non-NULL.  Scalar noise == 0 -> all ones.
 */
int wb_significance(const void *w, long long n, int dtype, double sigma, double sigma_e, double noise_host,
                    const double *noise_dev, const void *noise_map, int soft, void *out, void *stream);

/*
 * In-place denoise of one plane per frame: w <- dtype(float64(w) * (weight * significance(w))), the statement
 * `c *= wgt * self.significance(sig, scl)` of Coefficients.denoise (watroo/wavelets.py:145-149).
 * sig_mode as in wb_wow_whiten_scale (0 multiplies by `weight` only).
 */
int wb_denoise_plane(void *w, long long n, int batch, long long bstride, int dtype, int sig_mode, double sigma,
                     double sigma_e, double noise_host, const double *noise_dev, const void *noise_map,
                     double weight, void *stream);

/*
 * Residual plane of WOW: c <- c * dtype(weight / std), std = moments[frame][2] rounded to the plane dtype,
 * non-positive -> 1e-15 (watroo/utils.py:185-189, :203).
 */
int wb_residual_rescale(void *c, long long n, int batch, long long bstride, int dtype, const double *moments,
                        double weight, void *stream);

/*
 * One dilated filter pass along ONE axis of a C-contiguous (n_outer, n_axis, n_inner) array: what the 1-D and 3-D
 * branches of `convolution` need beyond the 2-D kernels (watroo/wavelets.py:46-69):
 *   - 1-D signal of n samples: n_outer = 1, n_axis = n, n_inner = 1, border = WB_BORDER_MIRROR
 *     (scipy.ndimage.convolve(arr, atrous_kernel(s), mode='mirror'), :64-69);
 *   - depth pass of a (D, H, W) volume after wb_atrous_scale has smoothed every slice: n_outer = 1, n_axis = D,
 *     n_inner = H*W, border = WB_BORDER_SYMMETRIC (cv2.filter2D with the (K,1) kernel on every [:, :, i] slice, :55-63).
 *     out_c[i] = sum_k h_k in[.., R(a + (k-c) 2^scale), ..]        out_w = sub_from - out_c
 * `sub_from` is the plane the detail coefficients refer to (c_s, watroo/wavelets.py:442); it may equal `in` (1-D) or
 * be the unsmoothed volume (3-D).  `out_w` may be NULL (then `sub_from` is ignored), `out_c` may be NULL.
 */
int wb_atrous_axis(const void *in, const void *sub_from, void *out_c, void *out_w, long long n_outer, long long n_axis,
                   long long n_inner, int scale, int taps, int dtype, int border, void *stream);

/*
 * One scale of the BILATERAL cascade of a 1-D signal (ndim = 1, shape (1, 1, n2)) or a 3-D volume (ndim = 3, shape
 * (n0, n1, n2), C-contiguous): replaces watroo/wavelets.py:433-442 for those inputs -- sdev_loc (:24-32) through the
 * n-D branches of convolution (:46-69: 1-D whole-sample 'mirror' border, 3-D half-sample symmetric) and the
 * dimension-generic atrous_convolution (:74-105: K^ndim - 1 range-weighted taps through np.pad 'symmetric').
 * out_c = c_{s+1}, out_w = c_s - c_{s+1} (either may be NULL).  A parity path: one thread per sample.
 */
int wb_atrous_scale_bilateral_nd(const void *in, void *out_c, void *out_w, int ndim, long long n0, long long n1,
                                 long long n2, int scale, int taps, int dtype, double var_factor, void *stream);

/*
 * Dense 2-D correlation with a small arbitrary kernel and the symmetric border: the PSF filters of richardson_lucy
 * (watroo/utils.py:252-255 with the flipped PSF = convolution, :283-286 with the PSF as is = correlation; both
 * cv2.filter2D(..., (-1,-1), 0, cv2.BORDER_REFLECT)).  `kernel` is a DEVICE array of kh*kw coefficients of the image
 * dtype, row-major; the anchor is the kernel centre (kh/2, kw/2); flip != 0 applies the kernel rotated by 180 degrees.
 */
int wb_filter2d(const void *in, void *out, int H, int W, long long in_pitch, long long out_pitch, const void *kernel,
                int kh, int kw, int flip, int dtype, void *stream);

/*
 * Synthesis: out = ((p_0 + p_1) + p_2) + ... over `nplanes` planes `plane_stride` elements apart, in the plane
 * dtype and in plane order -- np.sum(coefficients, axis=0) (watroo/utils.py:98, :205).
 */
int wb_synthesis(const void *planes, int nplanes, long long plane_stride, long long n, int batch,
                 long long in_bstride, void *out, long long out_bstride, int dtype, void *stream);

/*
 * The whole WOW pipeline of a stack of frames in one call -- the loop of `wow` (plain or bilateral cascade) with whitening
 * (watroo/utils.py:172-205: per scale the smooth + detail of watroo/wavelets.py:35-45,:442, the local power, the
 * significance and the weighting; np.std and the rescale of the residual plane, :185-189,:203; np.sum, :205): per scale
 * wb_wow_scale, or wb_atrous_scale [+ wb_abs_median] + wb_wow_whiten_scale where the fused kernel declines the shape or
 * the MAD noise must first be estimated from the raw w_0; then wb_plane_moments + wb_residual_rescale + wb_synthesis.
 * Bit-identical to issuing those calls one by one; it exists for frames small enough that a host-language loop is
 * slower than the device (interpreter + FFI time per launch).
 *   planes  (batch, n_scales+1, H, W) contiguous: the whitened coefficients (out)
 *   scratch (3, batch, H, W): two ping-pong smooth planes and one raw detail plane
 *   recon   (batch, H, W): the sum of the planes (out)
 *   weights[n_scales+1], sigmas[n_scales] (denoise coefficient per scale, 0 = no threshold), sigma_e[n_scales]: HOST arrays
 *   var_factors: NULL = plain cascade; else HOST array [n_scales] of the bilateral variance factors of
 *   wb_atrous_scale_bilateral (watroo/wavelets.py:433-440): every scale then runs K2 + the whitening pass
 *   soft != 0: erf significance, else hard masks.  Noise: estimate_noise == 0 -> noise_dev[frame] when non-NULL, else
 *   noise_host; estimate_noise != 0 -> the MAD estimate is written to noise_dev[batch] at the first scale that
 *   thresholds (from the raw w_0 at scale 0, from the already whitened plane 0 later: watroo/wavelets.py:131-132).
 *   workspace: wb_wow_cascade_workspace_bytes(dtype, batch, H*W) bytes of device memory.
 */
size_t wb_wow_cascade_workspace_bytes(int dtype, int batch, long long n);
int wb_wow_cascade(const void *in, long long in_pitch, long long in_bstride, void *planes, void *scratch, void *recon,
                   int batch, int H, int W, int n_scales, int taps, int dtype, const double *weights, const double *sigmas,
                   const double *sigma_e, const double *var_factors, int soft, double noise_host, double *noise_dev,
                   int estimate_noise, void *workspace, size_t workspace_bytes, void *stream);

/*
 * wb_wow_cascade with the noise taken from a per-pixel map (no MAD estimate).  Every scale takes two passes: K1
 * (wb_atrous_scale) or K2 (wb_atrous_scale_bilateral) writes the raw detail plane into scratch, then
 * wb_wow_whiten_scale_map whitens it where sigmas[s] != 0 and wb_wow_whiten_scale (sig_mode 0) elsewhere; moments,
 * rescale and synthesis as in wb_wow_cascade.  Bit-identical to issuing those calls one by one.  Map layout as in
 * wb_wow_whiten_scale_map; the other arguments and the workspace as in wb_wow_cascade.
 */
int wb_wow_cascade_map(const void *in, long long in_pitch, long long in_bstride, void *planes, void *scratch, void *recon,
                       int batch, int H, int W, int n_scales, int taps, int dtype, const double *weights,
                       const double *sigmas, const double *sigma_e, const double *var_factors, int soft,
                       const void *noise_map, long long map_pitch, long long map_bstride, void *workspace,
                       size_t workspace_bytes, void *stream);

/*
 * wb_wow_cascade with the gamma blend (h > 0, watroo/utils.py:157-158, :207-217) and / or preserve_variance
 * (:178-184): the whole image branch of `wow` for those options in one call.  Every scale takes two passes: K1 / K2
 * write the raw detail plane into scratch, [wb_plane_moments of it when preserve_variance,] K3 whitens it into the
 * plane when `whitening` (map mode where sigmas[s] != 0 and a map is used), and a K5 epilogue then
 *   - forms dn = dtype(double(w) * significance) (w itself for unthresholded scales and a zero host-scalar noise),
 *   - adds dn to the gamma plane (h > 0),
 *   - scales the whitened plane by pn = dtype(sqrt(mean(w^2))) (whitening and preserve_variance), or writes
 *     dtype(dn * factor), factor = dtype(pn * dtype(weight)) or dtype(weight) (no whitening).
 * The residual plane is added to the gamma plane, then c_L <- c_L * dtype(weight_L [* std] [/ max(std, 1e-15)]) in
 * float64 with std rounded to the dtype; recon = the sum of the planes, or with h > 0
 *   dtype(dtype(1 - h) * sum + dtype(h) * clamp((gamma - lo) / (hi - lo), 0, 1) ** (1 / gamma))
 * with lo / hi the per-frame min / max of the gamma plane or the given gamma_min / gamma_max, every operation rounded
 * to the dtype as the element-wise route of `wow` rounds it.
 *   whitening: the caller passes `whitening and h < 1` (utils.py:186, :193).
 *   gamma_plane: (batch, H, W) scratch, required when h > 0 (then gamma != 0); not read otherwise.
 *   n_scales may be 0 (h >= 1 without denoise coefficients): plane 0 is then the image.  scratch may be NULL then.
 *   Noise: host scalar / noise_dev / estimate as in wb_wow_cascade; use_map != 0 takes the per-pixel noise_map instead
 *   (layout of wb_wow_whiten_scale_map; estimate_noise must then be 0).
 *   workspace: wb_wow_cascade_blend_workspace_bytes(dtype, batch, H*W) bytes of device memory.
 * The other arguments as in wb_wow_cascade.
 */
size_t wb_wow_cascade_blend_workspace_bytes(int dtype, int batch, long long n);
int wb_wow_cascade_blend(const void *in, long long in_pitch, long long in_bstride, void *planes, void *scratch,
                         void *recon, void *gamma_plane, int batch, int H, int W, int n_scales, int taps, int dtype,
                         const double *weights, const double *sigmas, const double *sigma_e, const double *var_factors,
                         int soft, double noise_host, double *noise_dev, int estimate_noise, int use_map,
                         const void *noise_map, long long map_pitch, long long map_bstride, int whitening,
                         int preserve_variance, double h, double gamma, double gamma_min, int gamma_min_given,
                         double gamma_max, int gamma_max_given, void *workspace, size_t workspace_bytes, void *stream);

/*
 * Volumes: a C-contiguous (D, H, W) array is a volume (watroo/wavelets.py:322), not a stack of frames.  A scale is the 2-D
 * smooth of every [i] slice (wb_atrous_scale with the D slices as frames) followed by the depth pass with the
 * half-sample symmetric border (cv2.filter2D with the (K, 1) kernel on every [:, :, i] slice, :55-63, any number of
 * reflections when D is smaller than the halo).  Bit-identical to wb_atrous_scale + wb_atrous_axis(WB_BORDER_SYMMETRIC).
 *
 * wb_atrous_scale_volume: out_c = S_scale[in], out_w = in - out_c (either may be NULL).  tmp: (D, H, W) scratch of the
 * dtype for the slice smooth.
 */
int wb_atrous_scale_volume(const void *in, void *out_c, void *out_w, void *tmp, int D, int H, int W, int scale, int taps,
                           int dtype, void *stream);

/*
 * Scratch of wb_atrous_transform_volume / wb_wow_cascade_volume for `levels` scales: one volume for the slice smooth
 * and, from two scales on, two ping-pong smooth volumes (0 bytes for levels == 0).
 */
size_t wb_volume_scratch_bytes(int dtype, int D, int H, int W, int levels);

/*
 * The plain cascade of a volume over `levels` scales: planes (levels + 1, D, H, W) = [w_0 .. w_{L-1}, c_L]
 * (AtrousTransform on a 3-D array, watroo/wavelets.py:408-444).  scratch: wb_volume_scratch_bytes bytes.
 */
int wb_atrous_transform_volume(const void *in, void *planes, void *scratch, int D, int H, int W, int levels, int taps,
                               int dtype, void *stream);

/*
 * wow() of a volume (watroo/utils.py:172-205, h == 0, no preserve_variance) in one call, bit-identical to the element-wise
 * route (the reference's order and dtypes, every operation rounded once).  Per scale: the transform scale above; then
 *   whitening != 0: the local power S_s[dtype(w * w)] (slice smooth of the squares + depth pass) and, in the depth pass,
 *       w <- dtype(double(w) * significance) * dtype(weight / sqrt(P <= 0 ? 1e-15 : P))  (sqrt, divide, multiply);
 *   whitening == 0: w <- dtype(double(w) * significance) * dtype(weight).
 * Then the residual plane: c_L * dtype(weight_L / max(std(c_L), 1e-15)) (whitening) or c_L * dtype(weight_L), and
 * recon (D, H, W) = the sum of the planes.
 *   planes (n_scales + 1, D, H, W) out; scratch: wb_volume_scratch_bytes(dtype, D, H, W, n_scales) bytes;
 *   weights[n_scales + 1], sigmas[n_scales], sigma_e[n_scales]: HOST arrays as in wb_wow_cascade; soft: erf or hard mask.
 *   Noise: estimate_noise != 0 -> the MAD estimate of plane 0 as it stands when a threshold first needs it
 *   (watroo/wavelets.py:131-132), written to noise_dev[0]; else noise_dev[0] when non-NULL, else noise_host; or a
 *   per-voxel map of the plane dtype (noise_map != NULL, estimate_noise == 0): element (z, y, x) at
 *   z * map_zstride + y * W + x, map_zstride 0 (one (H, W) map for every slice) or >= H * W.
 *   workspace: wb_wow_cascade_volume_workspace_bytes(dtype, D, H, W) bytes of device memory.
 */
size_t wb_wow_cascade_volume_workspace_bytes(int dtype, int D, int H, int W);
int wb_wow_cascade_volume(const void *in, void *planes, void *scratch, void *recon, int D, int H, int W, int n_scales,
                          int taps, int dtype, const double *weights, const double *sigmas, const double *sigma_e,
                          int soft, int whitening, double noise_host, double *noise_dev, int estimate_noise,
                          const void *noise_map, long long map_zstride, void *workspace, size_t workspace_bytes,
                          void *stream);

/*
 * n standard-normal float32 samples (Philox4x32-10 + Box-Muller), the device stand-in for
 * np.random.normal(...).astype(np.float32) of compute_noise_weights (watroo/wavelets.py:225).
 * `offset` advances the counter so that successive calls with one seed give independent fields.
 */
int wb_randn_f32(float *out, long long n, unsigned long long seed, unsigned long long offset, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* WAVELETS_B200_H */
