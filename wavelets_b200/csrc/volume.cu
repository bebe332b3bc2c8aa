// Volumes (D, H, W): the plain 3-D cascade (watroo/wavelets.py:46-63 on a 3-D array) and wow() of a volume
// (watroo/utils.py:172-205 with whitening or the plain weighting), bit-identical to the element-wise route of
// wavelets_b200/utils.py::_wow_nd.
//
// A scale of a volume is the 2-D smooth of every [i] slice (K1 with the D slices as frames) followed by the depth pass:
// the column pass of a D x (H*W) image with pitch H*W and no row pass.  The depth pass has no horizontal taps, so there
// is nothing to share through shared memory: every thread owns one 16-byte vector of columns, walks one dilation chain
// z = r, r + d, r + 2d, ... (a segment of it) and keeps the running column sums of K1 (col_feed) in registers.  Every
// voxel of the input is read once per chain segment (plus 2 * (taps / 2) halo rows per segment), every output written
// once, with the tap order and FMAs of wb_atrous_axis (acc = h_0 v_0, then fma(h_k, v_k, acc)).  The border is the
// half-sample symmetric reflection with any number of reflections (D smaller than the halo).
//
// Epilogues of the depth pass:
//   EPI_TRANSFORM  out_c = acc, out_w = sub_from - acc (the detail plane refers to c_s, not to the slice-smoothed volume)
//   EPI_WHITEN     acc is the local power S[T(w * w)]; the plane w_s (read and rewritten in place) becomes, per voxel,
//                  the chain of _wow_nd with every operation rounded once (nothing contracted):
//                      lp = sqrt_rn(acc <= 0 ? T(1e-15) : acc)
//                      w  = T(double(w) * significance)   (erf / hard mask in float64, as wb_significance)
//                      w  = w * div_rn(T(weight), lp)
//                  This is NOT the rsqrt epilogue of the 2-D whitening kernels, whose results differ by design.
// Without whitening, volume_scale_kernel applies the same chain without the local power (w * T(weight)).
#include "pipeline.cuh"

namespace wb {

int atrous_power_slices(const void *w, void *out, int batch, int H, int W, int scale, int taps, int dtype,
                        cudaStream_t st);

enum { EPI_TRANSFORM = 0, EPI_WHITEN = 1 };

struct DepthParams {
    const void *in;        // the slice-smoothed volume
    const void *sub_from;  // EPI_TRANSFORM: c_s
    void *out_c, *out_w;   // EPI_TRANSFORM: c_{s+1}, w_s (either may be NULL); EPI_WHITEN: out_w = w_s, in place
    long long n;           // H * W: elements per slice (the pitch of the depth axis)
    long long col_blocks;  // thread blocks across the H * W columns
    int D, d, chains, seg;
    // EPI_WHITEN and volume_scale_kernel
    int sig_mode;  // 0: none, 1: soft (erf), 2: hard
    double sigma, sigma_e, noise_host;
    const double *noise_dev;  // device scalar, or NULL
    const void *noise_map;    // per-voxel map of the plane dtype (element z * map_zstride + yx), or NULL
    long long map_zstride;    // 0: one (H, W) map for every slice
    double weight;
};

template <typename T> __device__ __forceinline__ T sqrt_rn(T x);
template <> __device__ __forceinline__ float sqrt_rn<float>(float x) { return __fsqrt_rn(x); }
template <> __device__ __forceinline__ double sqrt_rn<double>(double x) { return __dsqrt_rn(x); }
template <typename T> __device__ __forceinline__ T div_rn(T a, T b);
template <> __device__ __forceinline__ float div_rn<float>(float a, float b) { return __fdiv_rn(a, b); }
template <> __device__ __forceinline__ double div_rn<double>(double a, double b) { return __ddiv_rn(a, b); }
template <typename T> __device__ __forceinline__ T mul_rn(T a, T b);
template <> __device__ __forceinline__ float mul_rn<float>(float a, float b) { return __fmul_rn(a, b); }
template <> __device__ __forceinline__ double mul_rn<double>(double a, double b) { return __dmul_rn(a, b); }

// The significance and weighting of one coefficient; `thr` is the scalar threshold (sigma * noise) * sigma_e when there
// is no map.  WHITE: `power` is the local power S[T(w * w)] at that voxel.
template <typename T, bool WHITE, bool MAP>
__device__ __forceinline__ T volume_epilogue(T w, T power, int mode, double thr, T noise, const DepthParams &p, T weight) {
    T factor = weight;
    if constexpr (WHITE) factor = div_rn<T>(weight, sqrt_rn<T>(power <= T(0) ? T(1e-15) : power));
    if (mode) {
        if constexpr (MAP) thr = map_threshold<T>(noise, p.sigma, p.sigma_e);
        const double v = (double)w;
        const double s = mode == 1 ? erf(fabs(v / thr)) : (fabs(v) > thr ? 1.0 : 0.0);
        w = (T)__dmul_rn(v, s);
    }
    return mul_rn<T>(w, factor);
}

// Threshold mode and scalar threshold of a launch (a scalar noise of 0 means significance 1, watroo/wavelets.py:134).
template <bool MAP>
__device__ __forceinline__ int volume_mode(const DepthParams &p, double &thr) {
    int mode = p.sig_mode;
    thr = 0.0;
    if (!MAP && mode) {
        const double nz = p.noise_dev ? *p.noise_dev : p.noise_host;
        if (nz == 0.0) mode = 0;
        thr = (p.sigma * nz) * p.sigma_e;
    }
    return mode;
}

template <typename T, int V> __device__ __forceinline__ Pack<T, V> ld_pack(const T *p) {
    if constexpr (V == 1) {
        Pack<T, 1> r;
        r.v[0] = *p;
        return r;
    } else {
        return ld_vec(p);
    }
}
template <typename T, int V> __device__ __forceinline__ void st_pack(T *p, const Pack<T, V> &r) {
    if constexpr (V == 1) *p = r.v[0];
    else st_vec(p, r);
}

// One thread: V columns (one 16-byte vector, or one element when H * W or an address breaks the vectors) of one
// segment of one dilation chain.
template <typename T, int TAPS, int V, int EPI, bool MAP>
__global__ void __launch_bounds__(256) depth_pass_kernel(const DepthParams p) {
    constexpr int C = TAPS / 2;
    long long b = blockIdx.x;
    const long long cb = b % p.col_blocks;
    b /= p.col_blocks;
    const int r = (int)(b % p.chains);
    const int g = (int)(b / p.chains);
    const long long col = (cb * blockDim.x + threadIdx.x) * V;
    if (col >= p.n) return;
    const int n_chain = (p.D - r + p.d - 1) / p.d;
    const int i0 = g * p.seg;
    const int n_out = min(p.seg, n_chain - i0);
    if (n_out <= 0) return;

    const T *__restrict__ in = reinterpret_cast<const T *>(p.in) + col;
    const T *__restrict__ sub = reinterpret_cast<const T *>(p.sub_from);
    T *__restrict__ oc = reinterpret_cast<T *>(p.out_c);
    T *__restrict__ ow = reinterpret_cast<T *>(p.out_w);
    const T *__restrict__ map = reinterpret_cast<const T *>(p.noise_map);
    double thr = 0.0;
    int mode = 0;
    if constexpr (EPI == EPI_WHITEN) mode = volume_mode<MAP>(p, thr);
    const T weight = (T)p.weight;

    T S[V][TAPS - 1];
#pragma unroll
    for (int e = 0; e < V; ++e)
#pragma unroll
        for (int t = 0; t < TAPS - 1; ++t) S[e][t] = T(0);

    // input rows r + (i0 - C + j) d of the chain, reflected: a position q on the period 2D advanced by d mod 2D per row
    const int P = 2 * p.D;
    const int dm = (int)(p.d % P);
    int q = (int)(((long long)r + (long long)(i0 - C) * p.d) % P);
    if (q < 0) q += P;
    auto next_row = [&]() {
        const int z = q < p.D ? q : P - 1 - q;
        q += dm;
        if (q >= P) q -= P;
        return (long long)z * p.n;
    };
    // the first 2 * C rows of the segment only fill the running sums
#pragma unroll
    for (int j = 0; j < 2 * C; ++j) {
        const Pack<T, V> v = ld_pack<T, V>(in + next_row());
#pragma unroll
        for (int e = 0; e < V; ++e) (void)col_feed<T, TAPS>(S[e], v.v[e]);
    }
    const long long ostep = (long long)p.d * p.n;
    long long zo = (long long)r + (long long)i0 * p.d;
    long long o = zo * p.n + col;
    for (int i = 0; i < n_out; ++i, zo += p.d, o += ostep) {
        const Pack<T, V> v = ld_pack<T, V>(in + next_row());
        Pack<T, V> acc;
#pragma unroll
        for (int e = 0; e < V; ++e) acc.v[e] = col_feed<T, TAPS>(S[e], v.v[e]);
        if constexpr (EPI == EPI_TRANSFORM) {
            if (oc) st_pack<T, V>(oc + o, acc);
            if (ow) {
                Pack<T, V> w = ld_pack<T, V>(sub + o);
#pragma unroll
                for (int e = 0; e < V; ++e) w.v[e] -= acc.v[e];
                st_pack<T, V>(ow + o, w);
            }
        } else {
            Pack<T, V> w = ld_pack<T, V>(ow + o);
            Pack<T, V> nz;
            if constexpr (MAP) {
                if (mode) nz = ld_pack<T, V>(map + zo * p.map_zstride + col);
            }
#pragma unroll
            for (int e = 0; e < V; ++e)
                w.v[e] = volume_epilogue<T, true, MAP>(w.v[e], acc.v[e], mode, thr, MAP ? nz.v[e] : T(0), p, weight);
            st_pack<T, V>(ow + o, w);
        }
    }
}

// The epilogue without whitening on a whole plane of D * H * W voxels: w = T(double(w) * significance) * T(weight).
template <typename T, bool MAP>
__global__ void __launch_bounds__(256) volume_scale_kernel(const DepthParams p, long long total) {
    T *w = reinterpret_cast<T *>(p.out_w);
    const T *map = reinterpret_cast<const T *>(p.noise_map);
    double thr;
    const int mode = volume_mode<MAP>(p, thr);
    const T weight = (T)p.weight;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        T nz = T(0);
        if (MAP && mode) nz = map[(i / p.n) * p.map_zstride + i % p.n];
        w[i] = volume_epilogue<T, false, MAP>(w[i], T(0), mode, thr, nz, p, weight);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Host
// ---------------------------------------------------------------------------------------------------------------
static bool vectors_ok(const DepthParams &p, int V) {
    if (p.n % V) return false;
    for (const void *q : {p.in, p.sub_from, (const void *)p.out_c, (const void *)p.out_w, p.noise_map})
        if (q && !aligned16(q)) return false;
    return !p.noise_map || p.map_zstride % V == 0;
}

// Chain segments: enough (column vector, chain, segment) items for a few waves of resident threads, but never segments
// so short that the 2 * (taps / 2) halo rows per segment dominate.
static void plan_depth(DepthParams &p, int taps, int V) {
    const long long vec_cols = (p.n + V - 1) / V;
    p.chains = p.d < p.D ? p.d : p.D;
    const int n_max = (p.D + p.d - 1) / p.d;
    const long long target = 2LL * 2048 * device_sm_count();
    const long long per = vec_cols * p.chains;
    long long n_seg = (target + per - 1) / per;
    if (n_seg > n_max) n_seg = n_max;
    if (n_seg < 1) n_seg = 1;
    int seg = (int)((n_max + n_seg - 1) / n_seg);
    const int min_seg = 8 * (taps / 2);
    if (seg < min_seg) seg = min_seg;
    if (seg > n_max) seg = n_max;
    p.seg = seg;
    p.col_blocks = (vec_cols + 255) / 256;
}

template <typename T, int TAPS, int EPI>
static int launch_depth(DepthParams &p, cudaStream_t st) {
    constexpr int VV = VecOf<T>::V;
    const bool vec = vectors_ok(p, VV);
    plan_depth(p, TAPS, vec ? VV : 1);
    const long long n_seg = ((p.D + p.d - 1) / p.d + p.seg - 1) / p.seg;
    const dim3 grid((unsigned)(p.col_blocks * p.chains * n_seg));
    const bool map = EPI == EPI_WHITEN && p.noise_map;
    if (vec) {
        if (map) depth_pass_kernel<T, TAPS, VV, EPI, EPI == EPI_WHITEN><<<grid, 256, 0, st>>>(p);
        else depth_pass_kernel<T, TAPS, VV, EPI, false><<<grid, 256, 0, st>>>(p);
    } else {
        if (map) depth_pass_kernel<T, TAPS, 1, EPI, EPI == EPI_WHITEN><<<grid, 256, 0, st>>>(p);
        else depth_pass_kernel<T, TAPS, 1, EPI, false><<<grid, 256, 0, st>>>(p);
    }
    return launch_status();
}

template <int EPI>
static int depth_pass(DepthParams &p, int taps, int dtype, cudaStream_t st) {
    if (dtype == WB_F32) return taps == WB_TRIANGLE ? launch_depth<float, 3, EPI>(p, st) : launch_depth<float, 5, EPI>(p, st);
    return taps == WB_TRIANGLE ? launch_depth<double, 3, EPI>(p, st) : launch_depth<double, 5, EPI>(p, st);
}

static int volume_scale(DepthParams &p, int dtype, cudaStream_t st) {
    const long long total = (long long)p.D * p.n;
    long long blocks = (total + 255) / 256;
    if (blocks > 32LL * device_sm_count()) blocks = 32LL * device_sm_count();
    const dim3 grid((unsigned)blocks);
    const bool map = p.noise_map && p.sig_mode;
    if (dtype == WB_F32) {
        if (map) volume_scale_kernel<float, true><<<grid, 256, 0, st>>>(p, total);
        else volume_scale_kernel<float, false><<<grid, 256, 0, st>>>(p, total);
    } else {
        if (map) volume_scale_kernel<double, true><<<grid, 256, 0, st>>>(p, total);
        else volume_scale_kernel<double, false><<<grid, 256, 0, st>>>(p, total);
    }
    return launch_status();
}

static DepthParams depth_params(int D, int H, int W, int scale) {
    DepthParams p;
    memset(&p, 0, sizeof(p));
    p.D = D;
    p.n = (long long)H * W;
    p.d = 1 << scale;
    return p;
}

// One scale of the plain cascade of a volume: tmp = the 2-D smooth of every slice of `in`, then the depth pass.
static int scale_volume(const void *in, void *out_c, void *out_w, void *tmp, int D, int H, int W, int scale, int taps,
                        int dtype, cudaStream_t st) {
    const long long n = (long long)H * W;
    int rc = wb_atrous_scale(in, tmp, nullptr, D, H, W, W, n, W, n, W, n, scale, taps, dtype, st);
    if (rc) return rc;
    DepthParams p = depth_params(D, H, W, scale);
    p.in = tmp; p.sub_from = in; p.out_c = out_c; p.out_w = out_w;
    return depth_pass<EPI_TRANSFORM>(p, taps, dtype, st);
}

static int check_volume(int D, int H, int W, int taps, int dtype) {
    int rc = check_common(D, H, W, taps, dtype);
    if (rc) return rc;
    if ((long long)D * H * W > (1LL << 46)) return WB_EINVAL_SHAPE;
    return WB_OK;
}

static size_t align256(size_t n) { return (n + 255) & ~(size_t)255; }

}  // namespace wb

extern "C" {

int wb_atrous_scale_volume(const void *in, void *out_c, void *out_w, void *tmp, int D, int H, int W, int scale, int taps,
                           int dtype, void *stream) {
    int rc = wb::check_volume(D, H, W, taps, dtype);
    if (rc) return rc;
    if (scale < 0 || scale > 30) return WB_EINVAL_SCALE;
    if (!in || !tmp || (!out_c && !out_w)) return WB_EINVAL_POINTER;
    if (in == out_c || in == out_w || tmp == in || tmp == out_c || tmp == out_w || (out_c && out_c == out_w))
        return WB_EINVAL_POINTER;
    return wb::scale_volume(in, out_c, out_w, tmp, D, H, W, scale, taps, dtype, (cudaStream_t)stream);
}

size_t wb_volume_scratch_bytes(int dtype, int D, int H, int W, int levels) {
    if (levels < 1 || D < 1 || H < 1 || W < 1) return 0;
    const size_t vol = (size_t)D * (size_t)H * (size_t)W * (size_t)wb::dtype_size(dtype);
    return (levels > 1 ? 3 : 1) * vol;
}

int wb_atrous_transform_volume(const void *in, void *planes, void *scratch, int D, int H, int W, int levels, int taps,
                               int dtype, void *stream) {
    int rc = wb::check_volume(D, H, W, taps, dtype);
    if (rc) return rc;
    if (levels < 0 || levels > 30) return WB_EINVAL_SCALE;
    if (!in || !planes || (levels > 0 && !scratch)) return WB_EINVAL_POINTER;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t vol = (size_t)D * (size_t)H * (size_t)W * (size_t)wb::dtype_size(dtype);
    char *pl = reinterpret_cast<char *>(planes);
    char *sc = reinterpret_cast<char *>(scratch);
    if (levels == 0) return (int)cudaMemcpyAsync(planes, in, vol, cudaMemcpyDeviceToDevice, st);
    void *tmp = sc;  // scratch: [tmp, c ping, c pong]
    for (int s = 0; s < levels; ++s) {
        const void *src = s == 0 ? in : (const void *)(sc + (size_t)(1 + ((s - 1) & 1)) * vol);
        void *dst_c = s == levels - 1 ? (void *)(pl + (size_t)levels * vol) : (void *)(sc + (size_t)(1 + (s & 1)) * vol);
        rc = wb::scale_volume(src, dst_c, pl + (size_t)s * vol, tmp, D, H, W, s, taps, dtype, st);
        if (rc) return rc;
    }
    return WB_OK;
}

size_t wb_wow_cascade_volume_workspace_bytes(int dtype, int D, int H, int W) {
    return wb_wow_cascade_workspace_bytes(dtype, 1, (long long)D * H * W);
}

int wb_wow_cascade_volume(const void *in, void *planes, void *scratch, void *recon, int D, int H, int W, int n_scales,
                          int taps, int dtype, const double *weights, const double *sigmas, const double *sigma_e,
                          int soft, int whitening, double noise_host, double *noise_dev, int estimate_noise,
                          const void *noise_map, long long map_zstride, void *workspace, size_t workspace_bytes,
                          void *stream) {
    int rc = wb::check_volume(D, H, W, taps, dtype);
    if (rc) return rc;
    if (n_scales < 0 || n_scales > 30) return WB_EINVAL_SCALE;
    if (!in || !planes || (n_scales > 0 && !scratch) || !recon || !weights || (n_scales > 0 && (!sigmas || !sigma_e)) ||
        !workspace)
        return WB_EINVAL_POINTER;
    if (estimate_noise && !noise_dev) return WB_EINVAL_POINTER;
    const long long n = (long long)H * W, nv = (long long)D * n;
    if (noise_map && (estimate_noise || map_zstride < 0 || (map_zstride > 0 && map_zstride < n))) return WB_EINVAL_ARG;
    if (workspace_bytes < wb_wow_cascade_volume_workspace_bytes(dtype, D, H, W)) return WB_EINVAL_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t vol = (size_t)nv * (size_t)wb::dtype_size(dtype);
    char *pl = reinterpret_cast<char *>(planes);
    char *sc = reinterpret_cast<char *>(scratch);
    auto plane = [&](int s) { return (void *)(pl + (size_t)s * vol); };
    char *ws = reinterpret_cast<char *>(workspace);
    const size_t med_bytes = wb::align256(wb_abs_median_workspace_bytes(dtype, 1, nv));
    void *mom_ws = ws + med_bytes;
    double *mom = reinterpret_cast<double *>(ws + med_bytes + wb::align256(wb_plane_moments_workspace_bytes(1)));
    const int L = n_scales;
    bool have_noise = !estimate_noise;
    const double *nz_dev = estimate_noise ? nullptr : noise_dev;

    if (L == 0) {
        cudaError_t e = cudaMemcpyAsync(planes, in, vol, cudaMemcpyDeviceToDevice, st);
        if (e != cudaSuccess) return (int)e;
    }
    void *tmp = sc;
    for (int s = 0; s < L; ++s) {
        const void *src = s == 0 ? in : (const void *)(sc + (size_t)(1 + ((s - 1) & 1)) * vol);
        void *dst_c = s == L - 1 ? plane(L) : (void *)(sc + (size_t)(1 + (s & 1)) * vol);
        rc = wb::scale_volume(src, dst_c, plane(s), tmp, D, H, W, s, taps, dtype, st);
        if (rc) return rc;
        const bool need_sig = sigmas[s] != 0.0;
        if (need_sig && !have_noise) {
            // lazily, from plane 0 as it stands (raw at scale 0, already whitened later: watroo/wavelets.py:131-132)
            rc = wb_abs_median(plane(0), nv, 1, 0, dtype, nullptr, noise_dev, sigma_e[0], ws, med_bytes, stream);
            if (rc) return rc;
            have_noise = true;
            nz_dev = noise_dev;
        }
        wb::DepthParams p = wb::depth_params(D, H, W, s);
        p.out_w = plane(s);
        p.sig_mode = need_sig ? (soft ? 1 : 2) : 0;
        p.sigma = sigmas[s];
        p.sigma_e = need_sig ? sigma_e[s] : 1.0;
        p.noise_host = noise_host;
        p.noise_dev = noise_map ? nullptr : nz_dev;
        p.noise_map = need_sig ? noise_map : nullptr;
        p.map_zstride = map_zstride;
        p.weight = weights[s];
        if (whitening) {
            rc = wb::atrous_power_slices(plane(s), tmp, D, H, W, s, taps, dtype, st);
            if (rc) return rc;
            p.in = tmp;
            rc = wb::depth_pass<wb::EPI_WHITEN>(p, taps, dtype, st);
        } else if (p.sig_mode || weights[s] != 1.0) {
            rc = wb::volume_scale(p, dtype, st);
        }
        if (rc) return rc;
    }
    // residual plane: c_L * T(weight_L) / max(std, 1e-15) with whitening (watroo/utils.py:185-189, :203), else c_L * T(w)
    if (whitening) {
        rc = wb_plane_moments(plane(L), nv, 1, 0, dtype, mom, mom_ws, stream);
        if (rc) return rc;
        rc = wb_residual_rescale(plane(L), nv, 1, 0, dtype, mom, weights[L], stream);
    } else if (weights[L] != 1.0) {
        wb::DepthParams p = wb::depth_params(D, H, W, 0);
        p.out_w = plane(L);
        p.weight = weights[L];
        rc = wb::volume_scale(p, dtype, st);
    }
    if (rc) return rc;
    return wb_synthesis(planes, L + 1, nv, nv, 1, 0, recon, nv, dtype, stream);
}

}  // extern "C"
