// The WOW pipeline of a stack of frames in ONE library call: the loop of watroo/utils.py:172-205 (whitening on) on the
// plain or the bilateral cascade, as a sequence of the per-scale entry points -- per scale wb_wow_scale (or, for
// bilateral scales, where the fused kernel declines, or when the MAD noise has to be estimated from the raw w_0 first:
// wb_atrous_scale / wb_atrous_scale_bilateral [+ wb_abs_median] + wb_wow_whiten_scale), then wb_plane_moments +
// wb_residual_rescale of the residual plane and wb_synthesis.  wb_wow_cascade_map runs the same loop with a per-pixel
// noise map: two passes at every scale, the thresholded ones whitened by wb_wow_whiten_scale_map.
// wb_wow_cascade_blend adds the gamma blend (h > 0) and preserve_variance (utils.py:157-158, :174-217): two passes at
// every scale, [wb_plane_moments of the raw plane +] K3 where it whitens, then the K5 blend epilogue; the residual and
// the synthesis take the blend kernels.  This is the only place that decides, per scale, between the fused and the
// two-pass route and when the noise is estimated; wow(), wow_batch() and wow_stream() with whitening or the blend call
// it.  Host code only: it exists because a 512^2 .. 2048^2 frame is finished on the device long before a Python loop
// has issued its fifteen launches (0.27 - 0.30 ms of interpreter and ctypes time per wow() call, measured;
// profiles/r2_sizes.json).
#include "common.cuh"

namespace wb {

static size_t align256(size_t n) { return (n + 255) & ~(size_t)255; }

// Where the thresholds of a cascade come from: a host scalar, device scalars per frame (noise_dev, given or estimated
// here when `estimate`), or a per-pixel noise map (map != nullptr; every scale then takes the two-pass route).
struct CascadeNoise {
    double host;
    double *dev;
    int estimate;
    const void *map;
    long long map_pitch, map_bstride;
};

// The gamma blend and preserve_variance of wb_wow_cascade_blend.  `gamma` is NULL when h <= 0 (no blend); `minmax` is
// the per-frame [min, max, NaN] slot of the workspace.
struct CascadeBlend {
    void *gamma;
    int whitening, preserve_variance;
    double h, gamma_exp_base, gamma_min, gamma_max;
    int min_given, max_given;
    unsigned long long *minmax;
};

static int wow_cascade_impl(const void *in, long long in_pitch, long long in_bstride, void *planes, void *scratch,
                            void *recon, int batch, int H, int W, int n_scales, int taps, int dtype,
                            const double *weights, const double *sigmas, const double *sigma_e,
                            const double *var_factors, int soft, const CascadeNoise &nz, const CascadeBlend *blend,
                            void *workspace, size_t workspace_bytes, void *stream) {
    int rc = check_common(batch, H, W, taps, dtype);
    if (rc) return rc;
    if (n_scales < (blend ? 0 : 1) || n_scales > 30) return WB_EINVAL_SCALE;
    if (!in || !planes || (!scratch && n_scales > 0) || !recon || !weights || !sigmas || !sigma_e || !workspace)
        return WB_EINVAL_POINTER;
    if (nz.estimate && !nz.dev) return WB_EINVAL_POINTER;
    const long long n = (long long)H * W;
    if (workspace_bytes < (blend ? wb_wow_cascade_blend_workspace_bytes : wb_wow_cascade_workspace_bytes)(dtype, batch, n))
        return WB_EINVAL_ARG;
    const double noise_host = nz.host;
    double *noise_dev = nz.dev;
    const int estimate_noise = nz.estimate;
    const size_t es = (size_t)dtype_size(dtype);
    const int L = n_scales;
    char *pl = reinterpret_cast<char *>(planes);    // (batch, L + 1, H, W)
    char *sc = reinterpret_cast<char *>(scratch);   // (3, batch, H, W): two ping-pong smooth planes, one raw detail plane
    const long long plane_bs = (long long)(L + 1) * n;  // elements between the same plane of consecutive frames
    auto plane = [&](int s) { return pl + (size_t)s * (size_t)n * es; };
    auto scr = [&](int i) { return sc + (size_t)i * (size_t)batch * (size_t)n * es; };
    char *ws = reinterpret_cast<char *>(workspace);
    const size_t med_bytes = align256(wb_abs_median_workspace_bytes(dtype, batch, n));
    void *med_ws = ws;
    void *mom_ws = ws + med_bytes;
    double *mom = reinterpret_cast<double *>(ws + med_bytes + align256(wb_plane_moments_workspace_bytes(batch)));

    bool have_noise = !estimate_noise;  // a given noise: host scalar, or device scalars when noise_dev != NULL
    const double *nz_dev = estimate_noise ? nullptr : noise_dev;
    const bool white = !blend || blend->whitening;
    const bool pv = blend && blend->preserve_variance;
    if (blend && blend->gamma) {
        cudaError_t e = cudaMemsetAsync(blend->minmax, 0, (size_t)batch * 3 * sizeof(unsigned long long),
                                        (cudaStream_t)stream);
        if (e != cudaSuccess) return (int)e;
    }
    if (L == 0) {  // blend route only: h >= 1 without denoise coefficients plans no scale (utils.py:123-124)
        rc = wb_atrous_transform(in, planes, nullptr, batch, H, W, in_pitch, in_bstride, 0, taps, dtype, stream);
        if (rc) return rc;
    }
    const void *src = in;
    long long src_pitch = in_pitch, src_bs = in_bstride;
    for (int s = 0; s < L; ++s) {
        void *dst_c = (s == L - 1) ? (void *)plane(L) : (void *)scr(s & 1);
        const long long c_bs = (s == L - 1) ? plane_bs : n;
        const bool need_sig = sigmas[s] != 0.0;
        const int mode = need_sig ? (soft ? 1 : 2) : 0;
        const double sg = need_sig ? sigmas[s] : 0.0, se = need_sig ? sigma_e[s] : 1.0;
        // bilateral scale (var_factors[s] = sigma_bilateral[s]^2 (s + 1 if bilateral_scaling else 1)): the range-weighted
        // gather K2 writes the raw detail plane, K3 whitens it
        // a noise map: two passes at every scale (the fused kernel has no map mode), K3 with the map where sigmas[s] != 0
        // the blend needs the raw plane after K3: two passes at every scale
        const bool bilateral = var_factors != nullptr;
        bool two_pass = bilateral || nz.map || blend, median_of_raw = false;
        if (need_sig && !have_noise) {
            if (s == 0) {
                two_pass = median_of_raw = true;  // from the raw w_0: a grid-wide dependency inside the scale
            } else {
                // lazily, from the current state of plane 0 (already whitened here) -- watroo/wavelets.py:131-132
                rc = wb_abs_median(plane(0), n, batch, plane_bs, dtype, nullptr, noise_dev, sigma_e[0], med_ws, med_bytes, stream);
                if (rc) return rc;
                have_noise = true;
                nz_dev = noise_dev;
            }
        }
        if (!two_pass) {
            rc = wb_wow_scale(src, dst_c, plane(s), batch, H, W, src_pitch, src_bs, W, c_bs, W, plane_bs, s, taps, dtype, mode,
                              sg, se, need_sig ? noise_host : 0.0, need_sig ? nz_dev : nullptr, weights[s], stream);
            if (rc == WB_ENOT_FUSABLE) two_pass = true;
            else if (rc) return rc;
        }
        if (two_pass) {
            void *raw = scr(2);
            rc = bilateral ? wb_atrous_scale_bilateral(src, dst_c, raw, batch, H, W, src_pitch, src_bs, W, c_bs, W, n, s, taps,
                                                       dtype, var_factors[s], stream)
                           : wb_atrous_scale(src, dst_c, raw, batch, H, W, src_pitch, src_bs, W, c_bs, W, n, s, taps, dtype, stream);
            if (rc) return rc;
            if (median_of_raw) {
                rc = wb_abs_median(raw, n, batch, n, dtype, nullptr, noise_dev, sigma_e[0], med_ws, med_bytes, stream);
                if (rc) return rc;
                have_noise = true;
                nz_dev = noise_dev;
            }
            if (pv) {
                rc = wb_plane_moments(raw, n, batch, n, dtype, mom, mom_ws, stream);
                if (rc) return rc;
            }
            if (!white)
                rc = WB_OK;
            else if (nz.map && need_sig)
                rc = wb_wow_whiten_scale_map(raw, plane(s), nz.map, batch, H, W, W, n, W, plane_bs, nz.map_pitch,
                                             nz.map_bstride, s, taps, dtype, soft, sg, se, weights[s], stream);
            else
                rc = wb_wow_whiten_scale(raw, plane(s), batch, H, W, W, n, W, plane_bs, s, taps, dtype, mode, sg,
                                         se, need_sig ? noise_host : 0.0, need_sig ? nz_dev : nullptr, weights[s],
                                         stream);
            if (rc) return rc;
            // blend epilogue: significance where Coefficients._denoise_plane would launch (a threshold and a noise
            // that is not a host zero), the gamma sum, and the plane K3 does not finish
            const int write_mode = white ? (pv ? 1 : 0) : 2;
            if (blend && (blend->gamma || write_mode)) {
                const int sig_mode = (need_sig && (nz.map || nz_dev || noise_host != 0.0)) ? mode : 0;
                rc = blend_scale(raw, plane(s), plane_bs, blend->gamma, n, W, batch, dtype, s == 0, write_mode, sig_mode,
                                 sg, se, noise_host, nz_dev, nz.map, nz.map_pitch, nz.map_bstride, pv ? mom : nullptr,
                                 weights[s], (cudaStream_t)stream);
                if (rc) return rc;
            }
        }
        src = dst_c;
        src_pitch = W;
        src_bs = c_bs;
    }
    if (blend) {
        // residual plane (as _wow_general, the plane-by-plane route, treats it), then the plane sum and the blend
        if (pv || white) {
            rc = wb_plane_moments(plane(L), n, batch, plane_bs, dtype, mom, mom_ws, stream);
            if (rc) return rc;
        }
        rc = blend_residual(plane(L), n, batch, plane_bs, blend->gamma, L == 0, dtype, mom, weights[L], pv, white,
                            blend->minmax, (cudaStream_t)stream);
        if (rc) return rc;
        if (!blend->gamma) return wb_synthesis(planes, L + 1, n, n, batch, plane_bs, recon, n, dtype, stream);
        return synthesis_blend(planes, L + 1, n, n, batch, plane_bs, blend->gamma, recon, dtype, blend->minmax, blend->h,
                               blend->gamma_exp_base, blend->gamma_min, blend->min_given, blend->gamma_max,
                               blend->max_given, (cudaStream_t)stream);
    }
    // residual plane: c_L *= weight_L / std(c_L)  (watroo/utils.py:185-189, :203), then the sum of the planes (:205)
    rc = wb_plane_moments(plane(L), n, batch, plane_bs, dtype, mom, mom_ws, stream);
    if (rc) return rc;
    rc = wb_residual_rescale(plane(L), n, batch, plane_bs, dtype, mom, weights[L], stream);
    if (rc) return rc;
    return wb_synthesis(planes, L + 1, n, n, batch, plane_bs, recon, n, dtype, stream);
}

}  // namespace wb

extern "C" {

size_t wb_wow_cascade_workspace_bytes(int dtype, int batch, long long n) {
    if (batch < 1) batch = 1;
    return wb::align256(wb_abs_median_workspace_bytes(dtype, batch, n)) + wb::align256(wb_plane_moments_workspace_bytes(batch)) +
           wb::align256((size_t)batch * 3 * sizeof(double));
}

int wb_wow_cascade(const void *in, long long in_pitch, long long in_bstride, void *planes, void *scratch, void *recon,
                   int batch, int H, int W, int n_scales, int taps, int dtype, const double *weights, const double *sigmas,
                   const double *sigma_e, const double *var_factors, int soft, double noise_host, double *noise_dev,
                   int estimate_noise, void *workspace, size_t workspace_bytes, void *stream) {
    const wb::CascadeNoise nz{noise_host, noise_dev, estimate_noise, nullptr, 0, 0};
    return wb::wow_cascade_impl(in, in_pitch, in_bstride, planes, scratch, recon, batch, H, W, n_scales, taps, dtype,
                                weights, sigmas, sigma_e, var_factors, soft, nz, nullptr, workspace, workspace_bytes,
                                stream);
}

int wb_wow_cascade_map(const void *in, long long in_pitch, long long in_bstride, void *planes, void *scratch, void *recon,
                       int batch, int H, int W, int n_scales, int taps, int dtype, const double *weights,
                       const double *sigmas, const double *sigma_e, const double *var_factors, int soft,
                       const void *noise_map, long long map_pitch, long long map_bstride, void *workspace,
                       size_t workspace_bytes, void *stream) {
    if (!noise_map) return WB_EINVAL_POINTER;
    if (map_pitch < W || map_bstride < 0) return WB_EINVAL_ARG;
    const wb::CascadeNoise nz{0.0, nullptr, 0, noise_map, map_pitch, map_bstride};
    return wb::wow_cascade_impl(in, in_pitch, in_bstride, planes, scratch, recon, batch, H, W, n_scales, taps, dtype,
                                weights, sigmas, sigma_e, var_factors, soft, nz, nullptr, workspace, workspace_bytes,
                                stream);
}

size_t wb_wow_cascade_blend_workspace_bytes(int dtype, int batch, long long n) {
    if (batch < 1) batch = 1;
    return wb_wow_cascade_workspace_bytes(dtype, batch, n) + wb::align256((size_t)batch * 3 * sizeof(unsigned long long));
}

int wb_wow_cascade_blend(const void *in, long long in_pitch, long long in_bstride, void *planes, void *scratch,
                         void *recon, void *gamma_plane, int batch, int H, int W, int n_scales, int taps, int dtype,
                         const double *weights, const double *sigmas, const double *sigma_e, const double *var_factors,
                         int soft, double noise_host, double *noise_dev, int estimate_noise, int use_map,
                         const void *noise_map, long long map_pitch, long long map_bstride, int whitening,
                         int preserve_variance, double h, double gamma, double gamma_min, int gamma_min_given,
                         double gamma_max, int gamma_max_given, void *workspace, size_t workspace_bytes, void *stream) {
    if (use_map) {
        if (!noise_map) return WB_EINVAL_POINTER;
        if (map_pitch < W || map_bstride < 0 || estimate_noise) return WB_EINVAL_ARG;
    }
    if (h > 0.0) {
        if (!gamma_plane) return WB_EINVAL_POINTER;
        if (gamma == 0.0) return WB_EINVAL_ARG;
    }
    const wb::CascadeNoise nz{noise_host, use_map ? nullptr : noise_dev, use_map ? 0 : estimate_noise,
                              use_map ? noise_map : nullptr, map_pitch, map_bstride};
    char *ws = reinterpret_cast<char *>(workspace);
    const wb::CascadeBlend blend{h > 0.0 ? gamma_plane : nullptr, whitening ? 1 : 0, preserve_variance ? 1 : 0, h, gamma,
                                 gamma_min, gamma_max, gamma_min_given ? 1 : 0, gamma_max_given ? 1 : 0,
                                 reinterpret_cast<unsigned long long *>(
                                     ws ? ws + wb_wow_cascade_workspace_bytes(dtype, batch, (long long)H * W) : nullptr)};
    return wb::wow_cascade_impl(in, in_pitch, in_bstride, planes, scratch, recon, batch, H, W, n_scales, taps, dtype,
                                weights, sigmas, sigma_e, var_factors, soft, nz, &blend, workspace, workspace_bytes,
                                stream);
}

}  // extern "C"
