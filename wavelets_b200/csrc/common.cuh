// Shared device/host helpers for the sm_100a à trous kernels.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/wavelets_b200.h"

namespace wb {

// ---------------------------------------------------------------------------------------------------------------
// 16-byte vectors: 4 x fp32 or 2 x fp64.  Every thread of the row-pipeline kernels owns whole vectors of columns so
// that shared-memory reads are LDS.128 and global stores are STG.128.
// ---------------------------------------------------------------------------------------------------------------
template <typename T> struct VecOf;
template <> struct VecOf<float> { using type = float4; static constexpr int V = 4; };
template <> struct VecOf<double> { using type = double2; static constexpr int V = 2; };

template <typename T, int V> struct Pack { T v[V]; };

__device__ __forceinline__ Pack<float, 4> ld_vec(const float *p) {
    float4 t = *reinterpret_cast<const float4 *>(p);
    Pack<float, 4> r; r.v[0] = t.x; r.v[1] = t.y; r.v[2] = t.z; r.v[3] = t.w; return r;
}
__device__ __forceinline__ Pack<double, 2> ld_vec(const double *p) {
    double2 t = *reinterpret_cast<const double2 *>(p);
    Pack<double, 2> r; r.v[0] = t.x; r.v[1] = t.y; return r;
}
__device__ __forceinline__ void st_vec(float *p, const Pack<float, 4> &r) {
    *reinterpret_cast<float4 *>(p) = make_float4(r.v[0], r.v[1], r.v[2], r.v[3]);
}
__device__ __forceinline__ void st_vec(double *p, const Pack<double, 2> &r) {
    *reinterpret_cast<double2 *>(p) = make_double2(r.v[0], r.v[1]);
}
// Streaming (evict-first) 128-bit global store: planes that nobody re-reads soon (w_s) should not displace the
// running smooth plane c_{s+1} from L2.
__device__ __forceinline__ void st_vec_cs(float *p, const Pack<float, 4> &r) {
    __stcs(reinterpret_cast<float4 *>(p), make_float4(r.v[0], r.v[1], r.v[2], r.v[3]));
}
__device__ __forceinline__ void st_vec_cs(double *p, const Pack<double, 2> &r) {
    __stcs(reinterpret_cast<double2 *>(p), make_double2(r.v[0], r.v[1]));
}

// Half-sample symmetric reflection into [0, n), any number of reflections (cv2.BORDER_REFLECT, np.pad 'symmetric').
__host__ __device__ __forceinline__ int reflect_any(long long i, int n) {
    long long period = 2LL * n;
    long long m = i % period;
    if (m < 0) m += period;
    return (int)(m < n ? m : period - 1 - m);
}

// Border rule of the reference's RECURSIVE algorithm (watroo/wavelets.py:330-406): at scale s the image is split into
// the 2^s x 2^s decimated sub-arrays and each one is filtered with the undilated kernel and BORDER_REFLECT at ITS OWN
// edges -- i.e. tap `off` of pixel i reflects inside the sub-lattice {o, o + d, o + 2d, ...} (o = i mod d) instead of
// inside the full axis.  Differs from the standard algorithm within (taps/2) * 2^s samples of the borders.
__host__ __device__ __forceinline__ int reflect_lattice(long long i, int off, int d, int n) {
    const int o = (int)(i % d);
    const int t = (int)(i / d);
    const int n_sub = (n - o + d - 1) / d;
    return o + reflect_any((long long)t + off, n_sub) * d;
}

template <typename T> __device__ __forceinline__ T fma_t(T a, T b, T c);
template <> __device__ __forceinline__ float fma_t<float>(float a, float b, float c) { return fmaf(a, b, c); }
template <> __device__ __forceinline__ double fma_t<double>(double a, double b, double c) { return fma(a, b, c); }

// Filter taps (watroo/wavelets.py:239 Triangle, :268 B3spline); dyadic rationals, exact in fp32.
template <typename T, int TAPS> struct Taps;
template <typename T> struct Taps<T, 3> {
    __host__ __device__ static constexpr T h(int k) { return k == 1 ? T(0.5) : T(0.25); }
};
template <typename T> struct Taps<T, 5> {
    __host__ __device__ static constexpr T h(int k) {
        return k == 2 ? T(0.375) : ((k == 1 || k == 3) ? T(0.25) : T(0.0625));
    }
};

// threshold = (sigma * noise) * sigma_e evaluated like NumPy >= 2: with a scalar noise everything is float64; with a
// per-pixel noise map of the plane dtype, `sigma * noise` stays in that dtype and only the product with the
// float64 sigma_e is promoted (watroo/wavelets.py:137,141).  The one definition used by wb_significance,
// wb_denoise_plane and the map mode of the whitening kernels (whiten.cuh).
template <typename T>
__device__ __forceinline__ double map_threshold(T noise, double sigma, double sigma_e) {
    return (double)((T)sigma * noise) * sigma_e;
}
template <typename T>
__device__ __forceinline__ double threshold_at(const T *noise_map, long long i, double sigma, double scalar,
                                               double sigma_e) {
    if (noise_map) return map_threshold<T>(noise_map[i], sigma, sigma_e);
    return (sigma * scalar) * sigma_e;
}

// ---------------------------------------------------------------------------------------------------------------
// mbarrier + TMA bulk-copy PTX (sm_90+; on sm_100a the copy shows up in SASS as UBLKCP)
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
// The suspend-time hint lets the hardware park a waiting warp instead of having it spin through try_wait / branch
// pairs that steal issue slots from the warps doing arithmetic.
static constexpr uint32_t kMbarSuspendHintNs = 2000;
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WB_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
        "@p bra WB_DONE_%=;\n"
        "bra WB_WAIT_%=;\n"
        "WB_DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity), "r"(kMbarSuspendHintNs)
        : "memory");
}
// 1-D bulk asynchronous copy global -> shared, completion signalled on an mbarrier (bytes % 16 == 0, both 16B aligned).
__device__ __forceinline__ void tma_load_1d(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// L2 eviction-priority policies (createpolicy) for the per-access cache hints below.  The running smooth plane c_{s+1}
// written by one scale is the ONLY data the next launch re-reads: it is stored evict-last while everything that is
// dead after this launch (the c_s rows being read, the detail plane w_s) goes evict-first, so that the 64 MiB plane
// survives in the 126 MB L2 until the next scale consumes it.
__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void tma_load_1d_hint(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar,
                                                 uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
            smem_u32(smem_dst)),
        "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}
__device__ __forceinline__ void st_vec_hint(float *p, const Pack<float, 4> &r, uint64_t policy) {
    asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(p), "f"(r.v[0]), "f"(r.v[1]),
                 "f"(r.v[2]), "f"(r.v[3]), "l"(policy)
                 : "memory");
}
__device__ __forceinline__ void st_vec_hint(double *p, const Pack<double, 2> &r, uint64_t policy) {
    asm volatile("st.global.L2::cache_hint.v2.f64 [%0], {%1, %2}, %3;" ::"l"(p), "d"(r.v[0]), "d"(r.v[1]), "l"(policy)
                 : "memory");
}

// ---------------------------------------------------------------------------------------------------------------
// Packed fp32x2 arithmetic (sm_100a FADD2 / FMUL2 / FFMA2): two IEEE fp32 operations per lane per issue slot on a
// 64-bit register pair.  Same roundings as the scalar instructions, half the issue slots (tools/fma2bench.cu).
// ---------------------------------------------------------------------------------------------------------------
typedef unsigned long long u64;
__device__ __forceinline__ u64 pk2(float lo, float hi) {
    u64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void up2(u64 v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ u64 add2(u64 a, u64 b) { u64 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 sub2(u64 a, u64 b) { u64 d; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 mul2(u64 a, u64 b) { u64 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) {
    u64 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ u64 lds64(uint32_t a) {
    u64 r;
    asm volatile("ld.shared.b64 %0, [%1];" : "=l"(r) : "r"(a));
    return r;
}
__device__ __forceinline__ u64 swap2(u64 v) { float lo, hi; up2(v, lo, hi); return pk2(hi, lo); }
// four consecutive fp32 (one 16-byte vector) as two packed pairs
struct P4 { u64 lo, hi; };
__device__ __forceinline__ P4 lds_p4(uint32_t a) {
    P4 r;
    asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(r.lo), "=l"(r.hi) : "r"(a));
    return r;
}
__device__ __forceinline__ void sts_p4(uint32_t a, const P4 &v) {
    asm volatile("st.shared.v2.b64 [%0], {%1, %2};" ::"r"(a), "l"(v.lo), "l"(v.hi) : "memory");
}
__device__ __forceinline__ void stg_p4(void *p, const P4 &v) {
    asm volatile("st.global.v2.b64 [%0], {%1, %2};" ::"l"(p), "l"(v.lo), "l"(v.hi) : "memory");
}
__device__ __forceinline__ void stg_p4_cs(void *p, const P4 &v) {
    asm volatile("st.global.cs.v2.b64 [%0], {%1, %2};" ::"l"(p), "l"(v.lo), "l"(v.hi) : "memory");
}
__device__ __forceinline__ void stg_p4_hint(void *p, const P4 &v, uint64_t policy) {
    asm volatile("st.global.L2::cache_hint.v2.b64 [%0], {%1, %2}, %3;" ::"l"(p), "l"(v.lo), "l"(v.hi), "l"(policy)
                 : "memory");
}
// the mirrored vector read backwards
__device__ __forceinline__ P4 reverse_p4(const P4 &t) { return P4{swap2(t.hi), swap2(t.lo)}; }

// Lane arithmetic of the lean kernels: a 16-byte vector travels as two 64-bit registers -- two packed fp32 pixels each
// (float: FFMA2 / FMUL2 / FADD2) or one double each (DFMA / DMUL / DADD).  Same operations, same order, per dtype.
template <typename T> struct Lane;
template <> struct Lane<float> {
    static __device__ __forceinline__ u64 mul(u64 a, u64 b) { return mul2(a, b); }
    static __device__ __forceinline__ u64 fma(u64 a, u64 b, u64 c) { return fma2(a, b, c); }
    static __device__ __forceinline__ u64 sub(u64 a, u64 b) { return sub2(a, b); }
    static __device__ __forceinline__ u64 bcast(float h) { return pk2(h, h); }
    static __device__ __forceinline__ P4 reverse(const P4 &t) { return reverse_p4(t); }
};
template <> struct Lane<double> {
    static __device__ __forceinline__ double d(u64 a) { return __longlong_as_double((long long)a); }
    static __device__ __forceinline__ u64 u(double a) { return (u64)__double_as_longlong(a); }
    static __device__ __forceinline__ u64 mul(u64 a, u64 b) { return u(__dmul_rn(d(a), d(b))); }
    static __device__ __forceinline__ u64 fma(u64 a, u64 b, u64 c) { return u(__fma_rn(d(a), d(b), d(c))); }
    static __device__ __forceinline__ u64 sub(u64 a, u64 b) { return u(__dsub_rn(d(a), d(b))); }
    static __device__ __forceinline__ u64 bcast(double h) { return u(h); }
    static __device__ __forceinline__ P4 reverse(const P4 &t) { return P4{t.hi, t.lo}; }
};

// ---------------------------------------------------------------------------------------------------------------
// Programmatic dependent launch: the scale kernels of a cascade are launched back to back on one stream, each one
// consuming what the previous one wrote.  With the stream-serialisation attribute (launch_pdl below) the blocks of
// scale s+1 are scheduled as the blocks of scale s retire and run their prologue (barrier init, tap plans) while the
// tail of scale s is still in flight; griddepcontrol.wait then blocks until the previous grid has completed and its
// writes are visible.  Every global access of the kernel (reads AND writes: the ping-pong scratch is rewritten) comes
// after the wait.  Without the launch attribute both instructions are no-ops.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------------------------
// Host side
// ---------------------------------------------------------------------------------------------------------------
inline int dtype_size(int dtype) { return dtype == WB_F32 ? 4 : (dtype == WB_F64 ? 8 : 0); }

inline int check_common(int batch, int H, int W, int taps, int dtype) {
    if (dtype != WB_F32 && dtype != WB_F64) return WB_EINVAL_DTYPE;
    if (taps != WB_TRIANGLE && taps != WB_B3SPLINE) return WB_EINVAL_TAPS;
    if (batch < 1 || H < 1 || W < 1 || batch > 65535) return WB_EINVAL_SHAPE;
    return WB_OK;
}

inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Measured and NOT kept (profiles/r2_l2_persist.log): raising cudaLimitPersistingL2CacheSize so that the evict-last
// stores of c_{s+1} land in the L2 set-aside.  ncu inside a running cascade shows c_{s+1} read back from DRAM in full
// either way (L2 sector hit rate 9 %), and the carve-out only shrinks the cache for everything else: the 10-scale
// transform went from 0.341 ms to 0.436 ms (32 MiB) and 0.603 ms (device maximum).  The library leaves the limit alone.

// WB_L2_HINTS=0 in the environment disables the L2 eviction-priority hints (A/B measurements).
inline int l2_hints_enabled() {
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("WB_L2_HINTS");
        v = (e && e[0] == '0') ? 0 : 1;
    }
    return v;
}

// Launch-time error check that does not synchronise.
inline int launch_status() {
    cudaError_t e = cudaGetLastError();
    return (int)e;
}

// WB_PDL=0 in the environment launches the cascade kernels without programmatic dependent launch (A/B measurements).
inline bool pdl_enabled() {
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("WB_PDL");
        v = (e && e[0] == '0') ? 0 : 1;
    }
    return v != 0;
}

// Launch `kern(param)` with the programmatic-stream-serialisation attribute (the kernel must call pdl_wait() before
// its first global access).
template <typename P>
inline int launch_pdl(void (*kern)(const P), dim3 grid, dim3 block, size_t smem, cudaStream_t st, const P &param) {
    if (!pdl_enabled()) {
        kern<<<grid, block, smem, st>>>(param);
        return launch_status();
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, param);
    return (int)e;
}

// The same for kernels with any parameter list (the small reduction / point-wise kernels of the WOW tail and of the exact
// median: a dozen dependent launches of a few microseconds each, where the launch-to-launch gap is a large share).
template <typename... KArgs, typename... Args>
inline int launch_pdl_v(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    if (!pdl_enabled()) {
        kern<<<grid, block, smem, st>>>(KArgs(args)...);
        return launch_status();
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return (int)cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

// Gamma-blend / preserve_variance passes of wb_wow_cascade_blend (kernels in csrc/pointwise.cu).
int blend_scale(const void *raw, void *plane, long long plane_bs, void *gamma, long long n, int W, int batch, int dtype,
                int first, int write_mode, int sig_mode, double sigma, double sigma_e, double noise_host,
                const double *noise_dev, const void *noise_map, long long map_pitch, long long map_bstride,
                const double *moments, double weight, cudaStream_t st);
int blend_residual(void *c, long long n, int batch, long long bstride, void *gamma, int first, int dtype,
                   const double *moments, double weight, int preserve_variance, int whitening, unsigned long long *minmax,
                   cudaStream_t st);
int synthesis_blend(const void *planes, int nplanes, long long plane_stride, long long n, int batch,
                    long long in_bstride, const void *gamma_plane, void *out, int dtype, const unsigned long long *minmax,
                    double h, double gamma, double gamma_min, int min_given, double gamma_max, int max_given,
                    cudaStream_t st);

}  // namespace wb
