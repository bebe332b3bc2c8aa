// Whitening epilogue shared by K3 (wb_wow_whiten_scale) and the fused K1+K3 kernel (wb_wow_scale).
#pragma once

#include "pipeline.cuh"

namespace wb {

__device__ __forceinline__ float rsqrt_fast(float x) {
    float y;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// Whitening of one coefficient (watroo/utils.py:195-203 + watroo/wavelets.py:129-143), P = S_s[w^2] at that pixel:
//     w' = w * significance(w) * (weight / sqrt(P > 0 ? P : 1e-15))
// fp32: weight / sqrt(P) is evaluated as weight * rsqrt.approx(P) (MUFU.RSQ, <= 2 ulp) instead of the reference's
// sqrt -> divide -> multiply chain (three roundings): a few 1e-7 relative, far inside the 1e-5 parity budget, and
// 5 instructions per pixel instead of ~30 (the fused kernel is issue-bound, not HBM-bound, otherwise).
// fp64: weight * rsqrt(P) (CUDA's double-precision rsqrt, <= 1 ulp; the sqrt -> divide chain cost ~40 FP64 instructions per
// pixel and made the fp64 whitening pass FP64-pipe-bound at twice its HBM time); the difference to the reference's
// two roundings is <= 3 ulp, four orders of magnitude inside the 1e-12 budget.  Soft threshold: erf(|w / thr|) with the reciprocal of thr hoisted (fp32);
// hard threshold: NumPy >= 2 compares |w| (fp32) with the float64 threshold; |w| > thr in float64 is equivalent to
// |w| > RD(thr) in fp32 (RD = round towards -inf), so the mask stays bit-exact without float64 instructions.
//
// Map mode (sig_mode == SIG_MAP, a per-pixel noise map): the composition of the mode-0 whitening with the significance
// of wb_significance and the float64 product of Coefficients.significance, per pixel, so that the result is bit-identical
// to running those three steps one after the other:
//     tmp = T(w * g)                                       (mode 0, the same instructions as apply / apply_lane)
//     thr = double(T(sigma) * map) * sigma_e               (map_threshold, common.cuh)
//     s   = soft ? erf(|double(w) / thr|) : (|double(w)| > thr ? 1.0 : 0.0)
//     out = T(double(tmp) * s)
// The last step is a multiply, not a select: masked negative coefficients stay -0.0, and a zero or negative map entry
// gives the inf / NaN / sign of the unfused composition.
template <typename T> struct WhitenEpilogue {
    int mode;
    T thr_cmp;  // hard threshold in the plane dtype, rounded down
    T thr;      // fp64: the threshold itself (soft); fp32: unused
    T inv_thr;  // soft: 1 / thr
    T weight;
    double sigma, sigma_e;  // map mode
    int map_soft;           // map mode: erf (1) or the hard mask (0); uniform over the launch
    // MAP: the kernel was compiled for the map mode (sig_mode == SIG_MAP; the thresholds are per pixel, see map_sig)
    template <bool MAP = false>
    __device__ __forceinline__ void init(const ScaleParams &p, int frame) {
        mode = p.sig_mode;
        if constexpr (MAP) {
            sigma = p.sigma;
            sigma_e = p.sigma_e;
            map_soft = p.map_soft;
            weight = (T)p.weight;
            return;
        }
        double t = 0.0;
        if (mode) {
            const double noise = p.noise_dev ? p.noise_dev[frame] : p.noise_host;
            if (noise == 0.0) mode = 0;  // scalar noise == 0 -> significance is all ones (wavelets.py:134-135)
            t = (p.sigma * noise) * p.sigma_e;  // (sigma * noise) * sigma_e, float64 as in the reference
        }
        if constexpr (sizeof(T) == 4) {
            thr_cmp = __double2float_rd(t);
            thr = (T)t;
            // a denormal threshold must not turn 1 / thr into inf (0 * inf would poison pixels where w == 0, for which the
            // reference's erf(|w / thr|) is 0): clamp to the largest finite float
            inv_thr = (T)fmin(1.0 / t, 3.4028234663852886e38);
        } else {
            thr_cmp = t;
            thr = t;
            inv_thr = fmin(1.0 / t, 1.7976931348623157e308);  // hoisted reciprocal (one rounding more than w / thr)
        }
        weight = (T)p.weight;
    }
    __device__ __forceinline__ T apply(T w, T power) const {
        power = (power <= T(0)) ? T(1e-15) : power;
        T g;
        if constexpr (sizeof(T) == 4) g = weight * rsqrt_fast(power);
        else g = weight * rsqrt(power);  // MUFU.RSQ64H seed + Newton steps, <= 1 ulp: ~10 FP64 instructions instead of the ~40 of sqrt + divide
        if (mode == 1) {
            // the reference multiplies by erf() evaluated in float64 and rounds the product to the plane dtype
            if constexpr (sizeof(T) == 4) w = w * erff(fabsf(w * inv_thr));
            else w = w * erf(fabs(w * inv_thr));
        } else if (mode == 2) {
            w = (fabs(w) > thr_cmp) ? w : T(0);
        }
        return w * g;
    }
    // Two pixels at once (fp32 only): the same operations as apply() with the multiplies packed.  MODE is the
    // significance mode the kernel was compiled for; `mode` can still be 0 at run time (noise == 0).
    template <int MODE>
    __device__ __forceinline__ u64 apply2(u64 w2, u64 power2) const {
        float p0, p1, w0, w1;
        up2(power2, p0, p1);
        p0 = (p0 <= 0.f) ? 1e-15f : p0;
        p1 = (p1 <= 0.f) ? 1e-15f : p1;
        const u64 g2 = mul2(pk2((float)weight, (float)weight), pk2(rsqrt_fast(p0), rsqrt_fast(p1)));
        if (MODE == 1 && mode == 1) {
            up2(w2, w0, w1);
            w2 = mul2(w2, pk2(erff(fabsf(w0 * (float)inv_thr)), erff(fabsf(w1 * (float)inv_thr))));
        } else if (MODE == 2 && mode == 2) {
            up2(w2, w0, w1);
            w2 = pk2((fabsf(w0) > (float)thr_cmp) ? w0 : 0.f, (fabsf(w1) > (float)thr_cmp) ? w1 : 0.f);
        }
        return mul2(w2, g2);
    }
    // One 64-bit lane of a lean kernel: two packed fp32 pixels (apply2) or one double (apply with the compiled-in mode).
    template <int MODE>
    __device__ __forceinline__ u64 apply_lane(u64 w, u64 power) const {
        if constexpr (sizeof(T) == 4) {
            return apply2<MODE>(w, power);
        } else {
            double x = Lane<double>::d(w), pw = Lane<double>::d(power);
            pw = (pw <= 0.0) ? 1e-15 : pw;
            const double g = weight * rsqrt(pw);
            if (MODE == 1 && mode == 1) x = x * erf(fabs(x * inv_thr));
            else if (MODE == 2 && mode == 2) x = (fabs(x) > thr_cmp) ? x : 0.0;
            return Lane<double>::u(x * g);
        }
    }
    // Map mode, one pixel: raw w, its mode-0 whitening tmp (apply / apply_lane) and its noise-map entry.
    __device__ __forceinline__ T map_sig(T w, T tmp, T noise) const {
        const double thr = map_threshold<T>(noise, sigma, sigma_e);
        const double v = (double)w;
        const double s = map_soft ? erf(fabs(v / thr)) : (fabs(v) > thr ? 1.0 : 0.0);
        return (T)((double)tmp * s);
    }
    // Map mode, one 64-bit lane of a lean kernel: raw w, its whitening tmp (apply_lane) and the map, as stored.
    __device__ __forceinline__ u64 map_lane(u64 w, u64 tmp, u64 noise) const {
        if constexpr (sizeof(T) == 4) {
            float w0, w1, t0, t1, n0, n1;
            up2(w, w0, w1);
            up2(tmp, t0, t1);
            up2(noise, n0, n1);
            return pk2(map_sig(w0, t0, n0), map_sig(w1, t1, n1));
        } else {
            return Lane<double>::u(map_sig(Lane<double>::d(w), Lane<double>::d(tmp), Lane<double>::d(noise)));
        }
    }
};

// Read-only streaming load of one 16-byte noise-map vector (read once per thresholded scale; not kept in L1).
__device__ __forceinline__ P4 ldg_p4_stream(const void *p) {
    P4 r;
    asm("ld.global.nc.L1::no_allocate.v2.b64 {%0, %1}, [%2];" : "=l"(r.lo), "=l"(r.hi) : "l"(p));
    return r;
}
__device__ __forceinline__ Pack<float, 4> ld_vec_stream(const float *p) {
    const P4 r = ldg_p4_stream(p);
    Pack<float, 4> v;
    up2(r.lo, v.v[0], v.v[1]);
    up2(r.hi, v.v[2], v.v[3]);
    return v;
}
__device__ __forceinline__ Pack<double, 2> ld_vec_stream(const double *p) {
    const P4 r = ldg_p4_stream(p);
    Pack<double, 2> v;
    v.v[0] = Lane<double>::d(r.lo);
    v.v[1] = Lane<double>::d(r.hi);
    return v;
}

}  // namespace wb
