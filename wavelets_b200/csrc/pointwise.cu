// K5 -- element-wise pieces of the hot path (all HBM-streaming, 128-bit accesses where alignment allows):
//   * significance map            Coefficients.significance      watroo/wavelets.py:129-143
//   * in-place denoise of a plane Coefficients.denoise           watroo/wavelets.py:145-149
//   * residual-plane rescale      wow(), last plane              watroo/utils.py:185-189,203
//   * synthesis sum               np.sum(coefficients, axis=0)   watroo/utils.py:98,205
//   * gamma blend / preserve_variance epilogues of wow()         watroo/utils.py:157-158,174-217
//   * N(0,1) fp32 noise fields    np.random.normal               watroo/wavelets.py:225 (device Philox4x32-10)
#include "common.cuh"

namespace wb {

// out: soft -> float64 erf(|w / thr|); hard -> uint8 (|w| > thr).  thr = (sigma * noise) * sigma_e, in float64
// exactly as NumPy >= 2 evaluates it; noise is a host scalar, a device scalar or a per-pixel map.
template <typename T>
__global__ void __launch_bounds__(256) significance_kernel(const T *w, long long n, double sigma, double sigma_e,
                                                           double noise_host, const double *noise_dev,
                                                           const T *noise_map, int soft, double *out_soft,
                                                           unsigned char *out_hard) {
    const double nz = noise_dev ? *noise_dev : noise_host;
    const bool ones = (!noise_map && nz == 0.0);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        if (ones) {
            if (soft) out_soft[i] = 1.0; else out_hard[i] = 1;
            continue;
        }
        const double thr = threshold_at<T>(noise_map, i, sigma, nz, sigma_e);
        const double v = (double)w[i];
        if (soft) out_soft[i] = erf(fabs(v / thr));
        else out_hard[i] = fabs(v) > thr ? 1 : 0;
    }
}

// w <- T( double(w) * (weight * significance) ): the product is formed in float64 and rounded once, like
// `c *= wgt * self.significance(...)` (wavelets.py:149).  sig_mode 0 multiplies by `weight` only.
template <typename T>
__global__ void __launch_bounds__(256) denoise_plane_kernel(T *w, long long n, int batch, long long bstride,
                                                            int sig_mode, double sigma, double sigma_e,
                                                            double noise_host, const double *noise_dev,
                                                            const T *noise_map, double weight) {
    pdl_launch_dependents();
    pdl_wait();  // may be launched with programmatic stream serialisation (WOW tail)
    const int frame = blockIdx.y;
    T *wf = w + (long long)frame * bstride;
    int mode = sig_mode;
    const double nz = noise_dev ? noise_dev[frame] : noise_host;
    if (mode && !noise_map && nz == 0.0) mode = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const double v = (double)wf[i];
        double f = weight;
        if (mode) {
            const double thr = threshold_at<T>(noise_map, i, sigma, nz, sigma_e);
            if (mode == 1) f = weight * erf(fabs(v / thr));
            else f = weight * (fabs(v) > thr ? 1.0 : 0.0);
        }
        wf[i] = (T)(v * f);
    }
}

// c_L <- c_L * T(weight / std_T), std_T = population std rounded to the plane dtype, non-positive -> 1e-15
// (utils.py:185-189, :203).  `moments` = [mean, var, std] per frame from wb_plane_moments.
template <typename T>
__global__ void __launch_bounds__(256) residual_rescale_kernel(T *c, long long n, int batch, long long bstride,
                                                               const double *moments, double weight) {
    pdl_launch_dependents();
    pdl_wait();  // may be launched with programmatic stream serialisation (WOW tail)
    const int frame = blockIdx.y;
    T *cf = c + (long long)frame * bstride;
    T sd = (T)moments[frame * 3 + 2];
    if (sd <= T(0)) sd = T(1e-15);
    const T ratio = (T)weight / sd;
    constexpr int V = VecOf<T>::V;
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long nth = (long long)gridDim.x * blockDim.x;
    if ((reinterpret_cast<uintptr_t>(cf) & 15u) == 0) {
        const long long nvec = n / V;
        for (long long i = tid; i < nvec; i += nth) {
            Pack<T, V> p = ld_vec(cf + i * V);
#pragma unroll
            for (int e = 0; e < V; ++e) p.v[e] *= ratio;
            st_vec(cf + i * V, p);
        }
        for (long long i = nvec * V + tid; i < n; i += nth) cf[i] *= ratio;
    } else {
        for (long long i = tid; i < n; i += nth) cf[i] *= ratio;
    }
}

// out = ((p_0 + p_1) + p_2) + ... in plane order and in the plane dtype, as np.sum(axis=0) does.
template <typename T>
__global__ void __launch_bounds__(256) synthesis_kernel(const T *planes, int nplanes, long long plane_stride,
                                                        long long n, int batch, long long in_bstride, T *out,
                                                        long long out_bstride) {
    pdl_launch_dependents();
    pdl_wait();  // may be launched with programmatic stream serialisation (WOW tail)
    const int frame = blockIdx.y;
    const T *pf = planes + (long long)frame * in_bstride;
    T *of = out + (long long)frame * out_bstride;
    constexpr int V = VecOf<T>::V;
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long nth = (long long)gridDim.x * blockDim.x;
    const bool vec_ok = ((reinterpret_cast<uintptr_t>(pf) & 15u) == 0) && ((reinterpret_cast<uintptr_t>(of) & 15u) == 0) &&
                        (plane_stride % V == 0);
    if (vec_ok) {
        const long long nvec = n / V;
        for (long long i = tid; i < nvec; i += nth) {
            Pack<T, V> acc = ld_vec(pf + i * V);
            for (int k = 1; k < nplanes; ++k) {
                Pack<T, V> p = ld_vec(pf + (long long)k * plane_stride + i * V);
#pragma unroll
                for (int e = 0; e < V; ++e) acc.v[e] += p.v[e];
            }
            st_vec(of + i * V, acc);
        }
        for (long long i = nvec * V + tid; i < n; i += nth) {
            T acc = pf[i];
            for (int k = 1; k < nplanes; ++k) acc += pf[(long long)k * plane_stride + i];
            of[i] = acc;
        }
    } else {
        for (long long i = tid; i < n; i += nth) {
            T acc = pf[i];
            for (int k = 1; k < nplanes; ++k) acc += pf[(long long)k * plane_stride + i];
            of[i] = acc;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Gamma blend (h > 0) and preserve_variance of wow() (watroo/utils.py:157-158, :174-217) as three passes of the
// cascade call: a per-scale epilogue, the residual plane, and the synthesis with the blend.  Each reproduces the
// torch element-wise ops of the plane-by-plane route one by one: every op rounds to the plane dtype on its own, so the
// explicit _rn intrinsics keep nvcc from contracting a multiply and an add into an FMA.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float sub_rn(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ double sub_rn(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ float div_rn(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ double div_rn(double a, double b) { return __ddiv_rn(a, b); }
__device__ __forceinline__ float sqrt_rn(float a) { return __fsqrt_rn(a); }
__device__ __forceinline__ double sqrt_rn(double a) { return __dsqrt_rn(a); }

__device__ __forceinline__ float rsqrt_t(float a) { return rsqrtf(a); }
__device__ __forceinline__ double rsqrt_t(double a) { return rsqrt(a); }
__device__ __forceinline__ float pow_t(float a, float e) { return powf(a, e); }
__device__ __forceinline__ double pow_t(double a, double e) { return pow(a, e); }

// Total order of the bit patterns (-0 < +0), as unsigned keys for atomicMin / atomicMax.
__device__ __forceinline__ unsigned long long order_key(float x) {
    const uint32_t u = __float_as_uint(x);
    return (u & 0x80000000u) ? (unsigned long long)(~u) : (unsigned long long)(u | 0x80000000u);
}
__device__ __forceinline__ unsigned long long order_key(double x) {
    const unsigned long long u = (unsigned long long)__double_as_longlong(x);
    return (u & 0x8000000000000000ull) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ unsigned long long bits_of(float x) { return (unsigned long long)__float_as_uint(x); }
__device__ __forceinline__ unsigned long long bits_of(double x) { return (unsigned long long)__double_as_longlong(x); }
template <typename T> __device__ __forceinline__ T from_bits(unsigned long long b);
template <> __device__ __forceinline__ float from_bits<float>(unsigned long long b) { return __uint_as_float((uint32_t)b); }
template <> __device__ __forceinline__ double from_bits<double>(unsigned long long b) { return __longlong_as_double((long long)b); }
template <typename T> __device__ __forceinline__ T from_order_key(unsigned long long k);
template <> __device__ __forceinline__ float from_order_key<float>(unsigned long long k) {
    const uint32_t u = (uint32_t)k;
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}
template <> __device__ __forceinline__ double from_order_key<double>(unsigned long long k) {
    return __longlong_as_double((long long)((k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k));
}

// Per-scale epilogue, reading the raw w_s (frame stride n) that K1 / K2 left in scratch:
//   dn     = T(double(w) * significance)  where the plane-by-plane route launched wb_denoise_plane (sig_mode != 0;
//            the same expression as denoise_plane_kernel with weight 1), else w itself
//   gamma <- T(gamma + dn)                 (accumulate; `first`: T(+0 + dn), since zeros_like + (-0.0) is +0.0)
//   write_mode 1: plane <- T(plane * pn)   (whitening and preserve_variance: K3's output times the power norm)
//   write_mode 2: plane <- T(dn * factor)  (no whitening: factor = T(pn * T(weight)) or T(weight); dn itself when
//                                           neither preserve_variance nor a weight != 1 asks for the product)
// pn = T(sqrt(var + mean * mean)) of the raw plane from wb_plane_moments (`moments`, NULL without preserve_variance).
template <typename T>
__global__ void __launch_bounds__(256) blend_scale_kernel(const T *raw, T *plane, long long plane_bs, T *gamma,
                                                          long long n, int W, int first, int accumulate, int write_mode,
                                                          int sig_mode, double sigma, double sigma_e, double noise_host,
                                                          const double *noise_dev, const T *noise_map,
                                                          long long map_pitch, long long map_bstride,
                                                          const double *moments, double weight, double unit) {
    pdl_launch_dependents();
    pdl_wait();
    const int frame = blockIdx.y;
    const T *rf = raw + (long long)frame * n;
    T *pf = plane + (long long)frame * plane_bs;
    T *gf = accumulate ? gamma + (long long)frame * n : nullptr;
    const T *mf = noise_map ? noise_map + (long long)frame * map_bstride : nullptr;
    int mode = sig_mode;
    const double nz = noise_dev ? noise_dev[frame] : noise_host;
    if (mode && !noise_map && nz == 0.0) mode = 0;
    T pn = T(0);
    if (moments) {
        const double mean = moments[frame * 3 + 0], var = moments[frame * 3 + 1];
        pn = (T)__dsqrt_rn(__dadd_rn(var, __dmul_rn(mean, mean)));
    }
    const bool scale_dn = moments != nullptr || weight != 1.0;
    const T factor = moments ? mul_rn(pn, (T)weight) : (T)weight;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const T w = rf[i];
        T dn = w;
        if (sig_mode) {
            const double v = (double)w;
            double f = unit;
            if (mode) {
                const T *m = mf ? mf + (map_pitch == W ? i : (i / W) * map_pitch + i % W) : nullptr;
                const double thr = threshold_at<T>(m, 0, sigma, nz, sigma_e);
                if (mode == 1) f = unit * erf(fabs(v / thr));
                else f = unit * (fabs(v) > thr ? 1.0 : 0.0);
            }
            dn = (T)(v * f);
        }
        if (gf) gf[i] = add_rn(first ? T(0) : gf[i], dn);
        if (write_mode == 1) pf[i] = mul_rn(pf[i], pn);
        else if (write_mode == 2) pf[i] = scale_dn ? mul_rn(dn, factor) : dn;
    }
}

// Residual plane (as _wow_general treats it): gamma <- T(gamma + c_L) with the raw c_L (T(+0 + c_L) when `first`:
// no scale), then c_L <- T(c_L * T(factor)), factor = double(weight) [* double(T(std)) with preserve_variance]
// [/ max(double(T(std)), 1e-15) with whitening] in float64.  With `gamma`, also the exact per-frame min and max of the
// final gamma plane: minmax[frame] = {max of the inverted keys (the min), max of the keys, the largest NaN bit pattern
// seen}, zeroed by the caller.  A NaN anywhere makes both bounds that NaN, as torch.min / torch.max return a NaN
// element.
template <typename T>
__global__ void __launch_bounds__(256) blend_residual_kernel(T *c, long long n, long long bstride, T *gamma,
                                                             int first, const double *moments, double weight,
                                                             int preserve_variance, int whitening,
                                                             unsigned long long *minmax) {
    pdl_launch_dependents();
    pdl_wait();
    const int frame = blockIdx.y;
    T *cf = c + (long long)frame * bstride;
    T *gf = gamma ? gamma + (long long)frame * n : nullptr;
    double f = weight;
    if (preserve_variance || whitening) {
        double sd = (double)(T)moments[frame * 3 + 2];
        if (preserve_variance) f = __dmul_rn(f, sd);
        if (whitening) f = __ddiv_rn(f, sd <= 0.0 ? 1e-15 : sd);
    }
    const T tf = (T)f;
    unsigned long long kmin_inv = 0, kmax = 0, nan = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const T v = cf[i];
        if (gf) {
            const T g = add_rn(first ? T(0) : gf[i], v);
            gf[i] = g;
            if (g != g) {
                nan = max(nan, bits_of(g));
            } else {
                const unsigned long long k = order_key(g);
                kmin_inv = max(kmin_inv, ~k);
                kmax = max(kmax, k);
            }
        }
        cf[i] = mul_rn(v, tf);
    }
    if (!gf) return;
    for (int o = 16; o > 0; o >>= 1) {
        kmin_inv = max(kmin_inv, __shfl_down_sync(0xffffffffu, kmin_inv, o));
        kmax = max(kmax, __shfl_down_sync(0xffffffffu, kmax, o));
        nan = max(nan, __shfl_down_sync(0xffffffffu, nan, o));
    }
    __shared__ unsigned long long r[3][8];
    if ((threadIdx.x & 31) == 0) {
        r[0][threadIdx.x >> 5] = kmin_inv;
        r[1][threadIdx.x >> 5] = kmax;
        r[2][threadIdx.x >> 5] = nan;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < (int)(blockDim.x >> 5); ++k) {
            kmin_inv = max(kmin_inv, r[0][k]);
            kmax = max(kmax, r[1][k]);
            nan = max(nan, r[2][k]);
        }
        unsigned long long *mm = minmax + frame * 3;
        atomicMax(mm + 0, kmin_inv);
        atomicMax(mm + 1, kmax);
        if (nan) atomicMax(mm + 2, nan);
    }
}

// gamma_scaled.pow_(1 / gamma) as torch dispatches it: exponent 0 fills ones, 1 copies, 0.5 / -0.5 / -1 take sqrt /
// rsqrt / reciprocal; with the exponent rounded to the dtype, 2 / 3 / -2 take products, anything else pow().
enum { POW_FILL = 0, POW_COPY, POW_SQRT, POW_RSQRT, POW_RECIP, POW_SQUARE, POW_CUBE, POW_INV_SQUARE, POW_GENERAL };
template <typename T>
__device__ __forceinline__ T pow_like_torch(T b, int mode, T e) {
    switch (mode) {
        case POW_FILL: return T(1);
        case POW_COPY: return b;
        case POW_SQRT: return sqrt_rn(b);
        case POW_RSQRT: return rsqrt_t(b);
        case POW_RECIP: return div_rn(T(1), b);
        case POW_SQUARE: return mul_rn(b, b);
        case POW_CUBE: return mul_rn(mul_rn(b, b), b);
        case POW_INV_SQUARE: return (T)__ddiv_rn(1.0, (double)mul_rn(b, b));
        default: return pow_t(b, e);
    }
}

// Scalars of the blend, in the plane dtype as torch forms them: lo / hi are the given bounds (rounded to T) or the
// per-frame min / max; with both given the division is a multiplication by inv = T(1) / T(hi - lo) (a host-scalar
// divisor), otherwise a true division by T(hi - lo); c1 = T(1 - h), c2 = T(h).
template <typename T> struct BlendScalars {
    T lo, hi, inv, c1, c2, e;
    int lo_given, hi_given, pow_mode;
};

// recon = T(T(c1 * sum) + T(c2 * g'')) with sum the plane-order sum of synthesis_kernel and
// g'' = pow(clamp(T(T(gamma - lo) / T(hi - lo)), 0, 1), 1 / gamma); the clamp keeps NaN.
template <typename T>
__global__ void __launch_bounds__(256) synthesis_blend_kernel(const T *planes, int nplanes, long long plane_stride,
                                                              long long n, long long in_bstride, const T *gamma, T *out,
                                                              const unsigned long long *minmax, BlendScalars<T> p) {
    pdl_launch_dependents();
    pdl_wait();
    const int frame = blockIdx.y;
    const T *pf = planes + (long long)frame * in_bstride;
    const T *gf = gamma + (long long)frame * n;
    T *of = out + (long long)frame * n;
    const unsigned long long *mm = minmax + frame * 3;
    const bool nan = mm[2] != 0;
    const T lo = p.lo_given ? p.lo : nan ? from_bits<T>(mm[2]) : from_order_key<T>(~mm[0]);
    const T hi = p.hi_given ? p.hi : nan ? from_bits<T>(mm[2]) : from_order_key<T>(mm[1]);
    const bool by_inverse = p.lo_given && p.hi_given;
    const T range = sub_rn(hi, lo);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        T acc = pf[i];
        for (int k = 1; k < nplanes; ++k) acc = add_rn(acc, pf[(long long)k * plane_stride + i]);
        T g = sub_rn(gf[i], lo);
        g = by_inverse ? mul_rn(g, p.inv) : div_rn(g, range);
        if (!(g != g)) g = g < T(0) ? T(0) : (g > T(1) ? T(1) : g);
        g = pow_like_torch<T>(g, p.pow_mode, p.e);
        of[i] = add_rn(mul_rn(p.c1, acc), mul_rn(p.c2, g));
    }
}

// Philox4x32-10 counter-based generator + Box-Muller: 4 standard normals per counter.
__device__ __forceinline__ void philox_round(uint32_t &c0, uint32_t &c1, uint32_t &c2, uint32_t &c3, uint32_t k0,
                                             uint32_t k1) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
}

__global__ void __launch_bounds__(256) randn_kernel(float *out, long long n, unsigned long long seed,
                                                    unsigned long long offset) {
    const long long nquad = (n + 3) / 4;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nquad;
         i += (long long)gridDim.x * blockDim.x) {
        const unsigned long long ctr = (unsigned long long)i + offset;
        uint32_t c0 = (uint32_t)ctr, c1 = (uint32_t)(ctr >> 32), c2 = 0x5EEDu, c3 = 0;
        uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            philox_round(c0, c1, c2, c3, k0, k1);
            k0 += 0x9E3779B9u;
            k1 += 0xBB67AE85u;
        }
        // uniforms in (0, 1]: (x + 1) * 2^-32
        const float u0 = ((float)c0 + 1.0f) * 2.3283064365386963e-10f;
        const float u1 = ((float)c1) * 2.3283064365386963e-10f;
        const float u2 = ((float)c2 + 1.0f) * 2.3283064365386963e-10f;
        const float u3 = ((float)c3) * 2.3283064365386963e-10f;
        const float r0 = sqrtf(-2.0f * logf(fminf(u0, 1.0f))), r1 = sqrtf(-2.0f * logf(fminf(u2, 1.0f)));
        float s0, co0, s1, co1;
        sincospif(2.0f * u1, &s0, &co0);
        sincospif(2.0f * u3, &s1, &co1);
        const float v[4] = {r0 * co0, r0 * s0, r1 * co1, r1 * s1};
        const long long base = i * 4;
        if (base + 3 < n && ((reinterpret_cast<uintptr_t>(out) & 15u) == 0)) {
            *reinterpret_cast<float4 *>(out + base) = make_float4(v[0], v[1], v[2], v[3]);
        } else {
            for (int e = 0; e < 4; ++e)
                if (base + e < n) out[base + e] = v[e];
        }
    }
}

static unsigned grid_for(long long work_items) {
    long long blocks = (work_items + 255) / 256;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0) sms = v;
    const long long cap = 16LL * sms;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (unsigned)blocks;
}


// One dilated filter pass along ONE axis of an (outer, axis, inner) row-major array -- the pieces of the 1-D and 3-D
// transforms that the 2-D row-pipeline kernels do not cover:
//   * 1-D signals (watroo/wavelets.py:64-69): scipy.ndimage.convolve(..., mode='mirror'), whole-sample reflection;
//   * the depth pass of a volume (watroo/wavelets.py:55-63): cv2.filter2D with the (K, 1) column kernel on every
//     [:, :, i] slice, BORDER_REFLECT (half-sample reflection), after the 2-D smooth of every [i] slice.
// out_c = filtered(in); out_w = sub_from - out_c (the detail plane refers to the plane BEFORE any pass of this scale).
// One thread per element, taps gathered straight from global memory (adjacent threads read adjacent addresses).
template <typename T, int TAPS>
__global__ void __launch_bounds__(256) axis_filter_kernel(const T *in, const T *sub_from, T *out_c, T *out_w,
                                                          long long n_axis, long long n_inner, long long total,
                                                          long long d, int border) {
    constexpr int C = TAPS / 2;
    const long long period = border == WB_BORDER_MIRROR ? 2 * (n_axis - 1) : 2 * n_axis;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long a = (idx / n_inner) % n_axis;
        const long long base = idx - a * n_inner;
        T acc = T(0);
#pragma unroll
        for (int k = 0; k < TAPS; ++k) {
            long long m = a + (long long)(k - C) * d;
            if (period > 0) {
                m %= period;
                if (m < 0) m += period;
                if (m >= n_axis) m = (border == WB_BORDER_MIRROR) ? period - m : period - 1 - m;
            } else {
                m = 0;  // a single sample mirrors onto itself
            }
            const T v = in[base + m * n_inner];
            acc = (k == 0) ? Taps<T, TAPS>::h(0) * v : fma_t<T>(Taps<T, TAPS>::h(k), v, acc);
        }
        if (out_c) out_c[idx] = acc;
        if (out_w) out_w[idx] = sub_from[idx] - acc;
    }
}


// One scale of the BILATERAL cascade of a 1-D signal or a 3-D volume (watroo/wavelets.py:433-442 with the n-D branches
// of convolution, :46-69, and the dimension-generic atrous_convolution, :74-105).  One thread per sample:
//   var = S[x^2] - S[x]^2 with the border of `convolution` for that dimensionality (1-D: whole-sample 'mirror', 3-D:
//         half-sample symmetric on every axis), in the centred form sum k_t D_t^2 - (sum k_t D_t)^2;
//   c'  = x - sum_t g_t D_t / (k_c + sum_t g_t),  g_t = k_t exp(-D_t^2 / (2 V)),  V = max(var, 1e-20) * var_factor,
//         over the K^n - 1 off-centre taps read through np.pad(..., 'symmetric') -- ALWAYS symmetric, also in 1-D.
// A parity path (124 exponentials per voxel for B3spline volumes), not a fast path.
__device__ __forceinline__ long long reflect_border(long long i, long long n, bool mirror) {
    const long long period = mirror ? 2 * (n - 1) : 2 * n;
    if (period <= 0) return 0;
    long long m = i % period;
    if (m < 0) m += period;
    if (m >= n) m = mirror ? period - m : period - 1 - m;
    return m;
}

template <typename T, int TAPS>
__global__ void __launch_bounds__(256) bilateral_nd_kernel(const T *in, T *out_c, T *out_w, long long n0, long long n1,
                                                           long long n2, int ndim, long long d, T var_factor) {
    constexpr int C = TAPS / 2;
    const long long total = n0 * n1 * n2;
    const int t0 = ndim == 3 ? TAPS : 1, t1 = ndim == 3 ? TAPS : 1;  // a 1-D signal is (1, 1, n)
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long x = idx % n2, y = (idx / n2) % n1, z = idx / (n1 * n2);
        const T xc = in[idx];
        // local variance, with the border rule of convolution() for this dimensionality
        T s1 = T(0), s2 = T(0);
        for (int a = 0; a < t0; ++a) {
            const long long zz = ndim == 3 ? reflect_border(z + (long long)(a - C) * d, n0, false) : 0;
            for (int b = 0; b < t1; ++b) {
                const long long yy = ndim == 3 ? reflect_border(y + (long long)(b - C) * d, n1, false) : 0;
                const T kab = (ndim == 3 ? Taps<T, TAPS>::h(a) * Taps<T, TAPS>::h(b) : T(1));
                const T *row = in + (zz * n1 + yy) * n2;
#pragma unroll
                for (int c = 0; c < TAPS; ++c) {
                    const long long xx = reflect_border(x + (long long)(c - C) * d, n2, ndim == 1);
                    const T dd = xc - row[xx];
                    const T kd = kab * Taps<T, TAPS>::h(c) * dd;
                    s1 += kd;
                    s2 = fma_t<T>(kd, dd, s2);
                }
            }
        }
        T var = s2 - s1 * s1;
        if (var <= T(0)) var = T(1e-20);
        const T nhi = T(-1) / (T(2) * var * var_factor);
        // range-weighted gather through the symmetric border
        T num = T(0), den = T(0);
        for (int a = 0; a < t0; ++a) {
            const long long zz = ndim == 3 ? reflect_border(z + (long long)(a - C) * d, n0, false) : 0;
            for (int b = 0; b < t1; ++b) {
                const long long yy = ndim == 3 ? reflect_border(y + (long long)(b - C) * d, n1, false) : 0;
                const T kab = (ndim == 3 ? Taps<T, TAPS>::h(a) * Taps<T, TAPS>::h(b) : T(1));
                const T *row = in + (zz * n1 + yy) * n2;
#pragma unroll
                for (int c = 0; c < TAPS; ++c) {
                    const T k = kab * Taps<T, TAPS>::h(c);
                    const bool centre = (ndim == 1 || (a == C && b == C)) && c == C;
                    const long long xx = reflect_border(x + (long long)(c - C) * d, n2, false);
                    const T dd = xc - row[xx];
                    const T gw = centre ? k : k * exp(dd * dd * nhi);
                    den += gw;
                    num = fma_t<T>(gw, dd, num);
                }
            }
        }
        const T cn = xc - num / den;
        if (out_c) out_c[idx] = cn;
        if (out_w) out_w[idx] = xc - cn;
    }
}


// Dense 2-D correlation with a small arbitrary kernel (the PSF of richardson_lucy, watroo/utils.py:252-255,283-286:
// cv2.filter2D(img, -1, psf, out, (-1,-1), 0, cv2.BORDER_REFLECT)): anchor at the kernel centre (kh/2, kw/2), half-sample
// symmetric border.  One thread per pixel; coefficients are warp-uniform loads, pixels coalesced and L1-resident.
// Products are accumulated in float64 and rounded once (cv2 uses a double DFT for kernels of this size).
template <typename T>
__global__ void __launch_bounds__(256) filter2d_kernel(const T *in, T *out, int H, int W, long long in_pitch,
                                                       long long out_pitch, const T *kern, int kh, int kw, int flip) {
    const long long n = (long long)H * W;
    const int ay = kh / 2, ax = kw / 2;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n;
         idx += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(idx / W), x = (int)(idx % W);
        double acc = 0.0;
        for (int i = 0; i < kh; ++i) {
            const T *row = in + (long long)reflect_any((long long)y + i - ay, H) * in_pitch;
            const T *krow = kern + (long long)(flip ? kh - 1 - i : i) * kw;
            for (int j = 0; j < kw; ++j) {
                const T kv = __ldg(krow + (flip ? kw - 1 - j : j));
                acc = fma((double)kv, (double)row[reflect_any((long long)x + j - ax, W)], acc);
            }
        }
        out[(long long)y * out_pitch + x] = (T)acc;
    }
}

// Launchers of the blend kernels for wb_wow_cascade_blend (csrc/cascade.cu), which has validated the arguments.
int blend_scale(const void *raw, void *plane, long long plane_bs, void *gamma, long long n, int W, int batch, int dtype,
                int first, int write_mode, int sig_mode, double sigma, double sigma_e, double noise_host,
                const double *noise_dev, const void *noise_map, long long map_pitch, long long map_bstride,
                const double *moments, double weight, cudaStream_t st) {
    dim3 grid(grid_for(n), (unsigned)batch);
    const int acc = gamma != nullptr;
    if (dtype == WB_F32)
        return launch_pdl_v(blend_scale_kernel<float>, grid, dim3(256), 0, st, reinterpret_cast<const float *>(raw),
                            reinterpret_cast<float *>(plane), plane_bs, reinterpret_cast<float *>(gamma), n, W, first, acc,
                            write_mode, sig_mode, sigma, sigma_e, noise_host, noise_dev,
                            reinterpret_cast<const float *>(noise_map), map_pitch, map_bstride, moments, weight, 1.0);
    return launch_pdl_v(blend_scale_kernel<double>, grid, dim3(256), 0, st, reinterpret_cast<const double *>(raw),
                        reinterpret_cast<double *>(plane), plane_bs, reinterpret_cast<double *>(gamma), n, W, first, acc,
                        write_mode, sig_mode, sigma, sigma_e, noise_host, noise_dev,
                        reinterpret_cast<const double *>(noise_map), map_pitch, map_bstride, moments, weight, 1.0);
}

int blend_residual(void *c, long long n, int batch, long long bstride, void *gamma, int first, int dtype,
                   const double *moments, double weight, int preserve_variance, int whitening, unsigned long long *minmax,
                   cudaStream_t st) {
    dim3 grid(grid_for(n), (unsigned)batch);
    if (dtype == WB_F32)
        return launch_pdl_v(blend_residual_kernel<float>, grid, dim3(256), 0, st, reinterpret_cast<float *>(c), n, bstride,
                            reinterpret_cast<float *>(gamma), first, moments, weight, preserve_variance, whitening,
                            minmax);
    return launch_pdl_v(blend_residual_kernel<double>, grid, dim3(256), 0, st, reinterpret_cast<double *>(c), n, bstride,
                        reinterpret_cast<double *>(gamma), first, moments, weight, preserve_variance, whitening,
                        minmax);
}

template <typename T>
static BlendScalars<T> blend_scalars(double h, double gamma, double gamma_min, int min_given, double gamma_max,
                                     int max_given) {
    BlendScalars<T> p;
    p.lo = (T)gamma_min;
    p.hi = (T)gamma_max;
    p.lo_given = min_given;
    p.hi_given = max_given;
    p.inv = (min_given && max_given) ? T(1) / (T)(gamma_max - gamma_min) : T(0);
    p.c1 = (T)(1.0 - h);
    p.c2 = (T)h;
    const double e = 1.0 / gamma;
    p.e = (T)e;
    p.pow_mode = e == 0.0 ? POW_FILL : e == 1.0 ? POW_COPY : e == 0.5 ? POW_SQRT : e == -0.5 ? POW_RSQRT
               : e == -1.0 ? POW_RECIP : p.e == T(2) ? POW_SQUARE : p.e == T(3) ? POW_CUBE
               : p.e == T(-2) ? POW_INV_SQUARE : POW_GENERAL;
    return p;
}

int synthesis_blend(const void *planes, int nplanes, long long plane_stride, long long n, int batch,
                    long long in_bstride, const void *gamma, void *out, int dtype, const unsigned long long *minmax,
                    double h, double gamma_exp_base, double gamma_min, int min_given, double gamma_max, int max_given,
                    cudaStream_t st) {
    dim3 grid(grid_for(n), (unsigned)batch);
    if (dtype == WB_F32)
        return launch_pdl_v(synthesis_blend_kernel<float>, grid, dim3(256), 0, st, reinterpret_cast<const float *>(planes),
                            nplanes, plane_stride, n, in_bstride, reinterpret_cast<const float *>(gamma),
                            reinterpret_cast<float *>(out), minmax,
                            blend_scalars<float>(h, gamma_exp_base, gamma_min, min_given, gamma_max, max_given));
    return launch_pdl_v(synthesis_blend_kernel<double>, grid, dim3(256), 0, st, reinterpret_cast<const double *>(planes),
                        nplanes, plane_stride, n, in_bstride, reinterpret_cast<const double *>(gamma),
                        reinterpret_cast<double *>(out), minmax,
                        blend_scalars<double>(h, gamma_exp_base, gamma_min, min_given, gamma_max, max_given));
}

}  // namespace wb

extern "C" {

int wb_significance(const void *w, long long n, int dtype, double sigma, double sigma_e, double noise_host,
                    const double *noise_dev, const void *noise_map, int soft, void *out, void *stream) {
    if (dtype != WB_F32 && dtype != WB_F64) return WB_EINVAL_DTYPE;
    if (n < 1) return WB_EINVAL_SHAPE;
    if (!w || !out) return WB_EINVAL_POINTER;
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = wb::grid_for(n);
    double *os = soft ? reinterpret_cast<double *>(out) : nullptr;
    unsigned char *oh = soft ? nullptr : reinterpret_cast<unsigned char *>(out);
    if (dtype == WB_F32)
        wb::significance_kernel<float><<<grid, 256, 0, st>>>(reinterpret_cast<const float *>(w), n, sigma, sigma_e,
                                                             noise_host, noise_dev,
                                                             reinterpret_cast<const float *>(noise_map), soft, os, oh);
    else
        wb::significance_kernel<double><<<grid, 256, 0, st>>>(reinterpret_cast<const double *>(w), n, sigma, sigma_e,
                                                              noise_host, noise_dev,
                                                              reinterpret_cast<const double *>(noise_map), soft, os, oh);
    return wb::launch_status();
}

int wb_denoise_plane(void *w, long long n, int batch, long long bstride, int dtype, int sig_mode, double sigma,
                     double sigma_e, double noise_host, const double *noise_dev, const void *noise_map, double weight,
                     void *stream) {
    if (dtype != WB_F32 && dtype != WB_F64) return WB_EINVAL_DTYPE;
    if (n < 1 || batch < 1 || batch > 65535) return WB_EINVAL_SHAPE;
    if (!w) return WB_EINVAL_POINTER;
    if (sig_mode < 0 || sig_mode > 2) return WB_EINVAL_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid(wb::grid_for(n), (unsigned)batch);
    if (dtype == WB_F32)
        wb::denoise_plane_kernel<float><<<grid, 256, 0, st>>>(reinterpret_cast<float *>(w), n, batch, bstride, sig_mode,
                                                              sigma, sigma_e, noise_host, noise_dev,
                                                              reinterpret_cast<const float *>(noise_map), weight);
    else
        wb::denoise_plane_kernel<double><<<grid, 256, 0, st>>>(reinterpret_cast<double *>(w), n, batch, bstride,
                                                               sig_mode, sigma, sigma_e, noise_host, noise_dev,
                                                               reinterpret_cast<const double *>(noise_map), weight);
    return wb::launch_status();
}

int wb_residual_rescale(void *c, long long n, int batch, long long bstride, int dtype, const double *moments,
                        double weight, void *stream) {
    if (dtype != WB_F32 && dtype != WB_F64) return WB_EINVAL_DTYPE;
    if (n < 1 || batch < 1 || batch > 65535) return WB_EINVAL_SHAPE;
    if (!c || !moments) return WB_EINVAL_POINTER;
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid(wb::grid_for(n / 4 + 1), (unsigned)batch);
    if (dtype == WB_F32)
        return wb::launch_pdl_v(wb::residual_rescale_kernel<float>, grid, dim3(256), 0, st, reinterpret_cast<float *>(c), n, batch, bstride, moments, weight);
    return wb::launch_pdl_v(wb::residual_rescale_kernel<double>, grid, dim3(256), 0, st, reinterpret_cast<double *>(c), n, batch, bstride, moments, weight);
}

int wb_synthesis(const void *planes, int nplanes, long long plane_stride, long long n, int batch,
                 long long in_bstride, void *out, long long out_bstride, int dtype, void *stream) {
    if (dtype != WB_F32 && dtype != WB_F64) return WB_EINVAL_DTYPE;
    if (n < 1 || nplanes < 1 || batch < 1 || batch > 65535) return WB_EINVAL_SHAPE;
    if (!planes || !out) return WB_EINVAL_POINTER;
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid(wb::grid_for(n / 4 + 1), (unsigned)batch);
    if (dtype == WB_F32)
        return wb::launch_pdl_v(wb::synthesis_kernel<float>, grid, dim3(256), 0, st, reinterpret_cast<const float *>(planes), nplanes,
                                plane_stride, n, batch, in_bstride, reinterpret_cast<float *>(out), out_bstride);
    return wb::launch_pdl_v(wb::synthesis_kernel<double>, grid, dim3(256), 0, st, reinterpret_cast<const double *>(planes), nplanes,
                            plane_stride, n, batch, in_bstride, reinterpret_cast<double *>(out), out_bstride);
}

int wb_randn_f32(float *out, long long n, unsigned long long seed, unsigned long long offset, void *stream) {
    if (n < 1) return WB_EINVAL_SHAPE;
    if (!out) return WB_EINVAL_POINTER;
    wb::randn_kernel<<<wb::grid_for(n / 4 + 1), 256, 0, (cudaStream_t)stream>>>(out, n, seed, offset);
    return wb::launch_status();
}

int wb_atrous_axis(const void *in, const void *sub_from, void *out_c, void *out_w, long long n_outer, long long n_axis,
                   long long n_inner, int scale, int taps, int dtype, int border, void *stream) {
    if (dtype != WB_F32 && dtype != WB_F64) return WB_EINVAL_DTYPE;
    if (taps != WB_TRIANGLE && taps != WB_B3SPLINE) return WB_EINVAL_TAPS;
    if (n_outer < 1 || n_axis < 1 || n_inner < 1) return WB_EINVAL_SHAPE;
    if (scale < 0 || scale > 30) return WB_EINVAL_SCALE;
    if (border != WB_BORDER_SYMMETRIC && border != WB_BORDER_MIRROR) return WB_EINVAL_ARG;
    if (!in || (!out_c && !out_w) || (out_w && !sub_from) || in == out_c || in == out_w) return WB_EINVAL_POINTER;
    const long long total = n_outer * n_axis * n_inner;
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = wb::grid_for(total);
    const long long d = 1LL << scale;
#define WB_AXIS(T, TAPS)                                                                                          \
    wb::axis_filter_kernel<T, TAPS><<<grid, 256, 0, st>>>(reinterpret_cast<const T *>(in),                         \
                                                         reinterpret_cast<const T *>(sub_from),                   \
                                                         reinterpret_cast<T *>(out_c), reinterpret_cast<T *>(out_w), \
                                                         n_axis, n_inner, total, d, border)
    if (dtype == WB_F32) {
        if (taps == WB_TRIANGLE) WB_AXIS(float, 3); else WB_AXIS(float, 5);
    } else {
        if (taps == WB_TRIANGLE) WB_AXIS(double, 3); else WB_AXIS(double, 5);
    }
#undef WB_AXIS
    return wb::launch_status();
}

int wb_atrous_scale_bilateral_nd(const void *in, void *out_c, void *out_w, int ndim, long long n0, long long n1,
                                 long long n2, int scale, int taps, int dtype, double var_factor, void *stream) {
    if (dtype != WB_F32 && dtype != WB_F64) return WB_EINVAL_DTYPE;
    if (taps != WB_TRIANGLE && taps != WB_B3SPLINE) return WB_EINVAL_TAPS;
    if ((ndim != 1 && ndim != 3) || n0 < 1 || n1 < 1 || n2 < 1 || (ndim == 1 && (n0 != 1 || n1 != 1))) return WB_EINVAL_SHAPE;
    if (scale < 0 || scale > 30) return WB_EINVAL_SCALE;
    if (!in || (!out_c && !out_w) || in == out_c || in == out_w) return WB_EINVAL_POINTER;
    if (!(var_factor > 0)) return WB_EINVAL_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = wb::grid_for(n0 * n1 * n2);
    const long long d = 1LL << scale;
#define WB_BNd(T, TAPS)                                                                                          \
    wb::bilateral_nd_kernel<T, TAPS><<<grid, 256, 0, st>>>(reinterpret_cast<const T *>(in), reinterpret_cast<T *>(out_c), \
                                                          reinterpret_cast<T *>(out_w), n0, n1, n2, ndim, d, (T)var_factor)
    if (dtype == WB_F32) {
        if (taps == WB_TRIANGLE) WB_BNd(float, 3); else WB_BNd(float, 5);
    } else {
        if (taps == WB_TRIANGLE) WB_BNd(double, 3); else WB_BNd(double, 5);
    }
#undef WB_BNd
    return wb::launch_status();
}

int wb_filter2d(const void *in, void *out, int H, int W, long long in_pitch, long long out_pitch, const void *kernel,
                int kh, int kw, int flip, int dtype, void *stream) {
    if (dtype != WB_F32 && dtype != WB_F64) return WB_EINVAL_DTYPE;
    if (H < 1 || W < 1 || kh < 1 || kw < 1) return WB_EINVAL_SHAPE;
    if (!in || !out || !kernel || in == out) return WB_EINVAL_POINTER;
    if (in_pitch < W || out_pitch < W) return WB_EINVAL_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = wb::grid_for((long long)H * W);
    if (dtype == WB_F32)
        wb::filter2d_kernel<float><<<grid, 256, 0, st>>>(reinterpret_cast<const float *>(in), reinterpret_cast<float *>(out),
                                                        H, W, in_pitch, out_pitch,
                                                        reinterpret_cast<const float *>(kernel), kh, kw, flip);
    else
        wb::filter2d_kernel<double><<<grid, 256, 0, st>>>(reinterpret_cast<const double *>(in),
                                                         reinterpret_cast<double *>(out), H, W, in_pitch, out_pitch,
                                                         reinterpret_cast<const double *>(kernel), kh, kw, flip);
    return wb::launch_status();
}

}  // extern "C"
