// K2 -- one scale of the BILATERAL à trous cascade, fused: local variance + range-weighted 25-tap gather + w_s.
//
// Replaces, per scale, watroo/wavelets.py:433-442:  sdev_loc (two dense filter2D, :24-32), the scaling by sigma_b^2
// (:434-436), atrous_convolution with bilateral_variance (np.pad + 24 full-image numexpr passes, :74-105) and the
// subtraction (:442).  One read of c_s, one write of c_{s+1}, one write of w_s.
//
// Maths (x = c_s at the output pixel, x_t the K^2-1 off-centre dilated taps through the symmetric border, k_t = h_i h_j):
//     var = S[x^2] - S[x]^2  ==  sum_t k_t D_t^2 - (sum_t k_t D_t)^2,   D_t = x - x_t      (shift invariance)
//     V   = max(var, 1e-20) * sigma_b^2 * (s+1 if bilateral_scaling)
//     g_t = k_t exp(-D_t^2 / V / 2),  N = k_c + sum_t g_t
//     c_{s+1} = (k_c x + sum_t g_t x_t) / N  ==  x - (sum_t g_t D_t) / N
// The centred form has no catastrophic cancellation, so the fp32 kernel follows the reference's float64 result
// more closely than the reference's own fp32 path does (SURVEY Appendix C).  Not HBM-bound: 24 exponentials
// per pixel put it on the MUFU/FMA pipes; it shares the TMA row pipeline of K1 (taps rows resident in the ring).
#include <utility>

#include "pipeline.cuh"

namespace wb {

struct BilateralParams {
    ScaleParams sp;
    double var_factor;    // sigma_b[s]^2 * (s + 1 if bilateral_scaling else 1)
    float var_factor_f;   // the same, rounded once on the host (no F2F in the fp32 step loop)
};

__device__ __forceinline__ float exp2_fast(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// g = k * exp(-D^2 / V / 2) with nhalf_inv = -log2(e) / (2 V) (fp32) or -1 / (2 V) (fp64)
__device__ __forceinline__ float range_weight(float k, float d2, float nhalf_inv) { return k * exp2_fast(d2 * nhalf_inv); }
__device__ __forceinline__ double range_weight(double k, double d2, double nhalf_inv) { return k * exp(d2 * nhalf_inv); }
template <typename T> __device__ __forceinline__ T nhalf_inverse(T v);
template <> __device__ __forceinline__ float nhalf_inverse<float>(float v) { return -1.4426950408889634f / (2.0f * v); }
template <> __device__ __forceinline__ double nhalf_inverse<double>(double v) { return -0.5 * __drcp_rn(v); }

// ---------------------------------------------------------------------------------------------------------------
// fp64 range weights: 2^a with a <= 0 from a 256-entry table of 2^(i/256) and a degree-4 polynomial -- 8 double-precision
// operations and one shared-memory load instead of the ~28 of exp() (the fp64 kernel is bound by the FP64 pipe: 24
// exponentials per pixel were 70 % of its work).  a = n / 256 + r with n = round(256 a) read off the mantissa after
// adding 1.5 * 2^44 (ulp 2^-8), |r| <= 2^-9: 2^a = 2^(n >> 8) * tab[n & 255] * exp(r ln 2); the truncated series is
// good to (2^-9 ln 2)^5 / 120 = 4e-17 and the table is the host's exp2, so the weights are accurate to ~2 ulp.
// ---------------------------------------------------------------------------------------------------------------
static constexpr int kExp2TabBits = 8;
static constexpr int kExp2TabSize = 1 << kExp2TabBits;
__device__ double g_exp2_tab[kExp2TabSize];

static int ensure_exp2_table() {
    static bool done[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && done[dev]) return 0;
    double host[kExp2TabSize];
    for (int i = 0; i < kExp2TabSize; ++i) host[i] = exp2((double)i / kExp2TabSize);
    cudaError_t e = cudaMemcpyToSymbol(g_exp2_tab, host, sizeof(host));
    if (e != cudaSuccess) return (int)e;
    if (dev >= 0 && dev < 64) done[dev] = true;
    return 0;
}

__device__ __forceinline__ double exp2_tab(double a, const double *tab) {
    a = fmax(a, -1000.0);  // 2^-1000 == 0 for every purpose here; keeps the exponent arithmetic below in range
    const double magic = 26388279066624.0;  // 1.5 * 2^44
    const double t = a + magic;
    const int n = __double2loint(t);  // round(256 a), two's complement (the low mantissa word of 1.5 * 2^44 is zero)
    const double r = (a - (t - magic)) * 0.6931471805599453;  // (a - n / 256) ln 2
    double p = fma(r, 1.0 / 24.0, 1.0 / 6.0);
    p = fma(r, p, 0.5);
    p = fma(r, p, 1.0);
    p = fma(r, p, 1.0);
    const double v = tab[n & (kExp2TabSize - 1)] * p;
    return __hiloint2double(__double2hiint(v) + ((n >> kExp2TabBits) << 20), __double2loint(v));
}
template <int TAPS> struct TapLog2d;
template <> struct TapLog2d<3> { __host__ __device__ static constexpr double l(int k) { return k == 1 ? -1.0 : -2.0; } };
template <> struct TapLog2d<5> {
    __host__ __device__ static constexpr double l(int k) { return k == 2 ? -1.4150374992788437 : ((k == 1 || k == 3) ? -2.0 : -4.0); }
};

// Values of the TAPS horizontal taps of one staged row for the V columns of a vector.
template <typename T, int TAPS, int DMODE>
__device__ __forceinline__ void row_taps(const T *srow, const TapPlan<PlanSize<TAPS, DMODE>::NV> &tp,
                                         T (&out)[TAPS][VecOf<T>::V]) {
    constexpr int V = VecOf<T>::V;
    constexpr int C = TAPS / 2;
    if constexpr (DMODE == 0) {
#pragma unroll
        for (int k = 0; k < TAPS; ++k) {
            Pack<T, V> t = ld_vec(srow + tp.off[k]);
            if ((tp.rev >> k) & 1u) reverse_vec<T, V>(t);
#pragma unroll
            for (int e = 0; e < V; ++e) out[k][e] = t.v[e];
        }
    } else {
        T win[3 * V];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            Pack<T, V> t = ld_vec(srow + tp.off[k]);
            if ((tp.rev >> k) & 1u) reverse_vec<T, V>(t);
#pragma unroll
            for (int e = 0; e < V; ++e) win[k * V + e] = t.v[e];
        }
#pragma unroll
        for (int k = 0; k < TAPS; ++k)
#pragma unroll
            for (int e = 0; e < V; ++e) out[k][e] = win[V + e + (k - C) * DMODE];
    }
}

// Row pipeline for float64 (and the fp32 shapes the pair kernels decline): one 16-byte vector of columns per thread.
// Round 2: nothing is held in registers across output rows except the accumulators (the 25 x V differences of round 1
// cost 166 registers, ONE block per SM, and left the FP64 pipe half idle): the taps are re-read from the staged rows
// where they are used, the variance comes from per-row statistics kept in a per-thread shared-memory ring (the same
// law-of-total-variance form as the fp32 kernels, see row_stats), and the fp64 weights come from exp2_tab -- two blocks
// per SM.  Per pixel ~330 double-precision operations instead of ~800.
template <typename T, int TAPS, int DMODE>
__global__ void __launch_bounds__(288, 2) bilateral_rows_kernel(const BilateralParams bp) {
    const ScaleParams &p = bp.sp;
    pdl_launch_dependents();
    constexpr int V = VecOf<T>::V;
    constexpr int C = TAPS / 2;
    constexpr int NV = PlanSize<TAPS, DMODE>::NV;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    T *rows = reinterpret_cast<T *>(smem_raw);
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw + (size_t)p.slots * p.row_stride * sizeof(T));
    uint64_t *empty = full + p.slots;
    double *tab = reinterpret_cast<double *>(empty + p.slots);  // fp64: 2^(i/256), see exp2_tab
    // row statistics (a, b) of the last TAPS chain rows: [TAPS][256 threads][2][V], row j lives in slot j % TAPS
    T *stats = reinterpret_cast<T *>(tab + kExp2TabSize);

    const int nt = blockDim.x - 32;
    const int nwc = nt >> 5;
    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int lane = tid & 31;

    int bx = blockIdx.x;
    const int strip = bx % p.n_strips;
    bx /= p.n_strips;
    const int r = bx % p.d;
    const int g = bx / p.d;
    const int frame = blockIdx.y;

    const int n_chain = (r < p.H) ? (p.H - r + p.d - 1) / p.d : 0;
    const int i0 = g * p.seg;
    const int n_out = min(p.seg, n_chain - i0);
    if (n_out <= 0) return;
    const int n_load = n_out + 2 * C;

    const int x0 = strip * p.wt;
    const int lo = max(0, x0 - p.halo_al);
    const int hi = min(p.W, x0 + p.wt + p.halo_al);
    const uint32_t row_bytes = (uint32_t)(hi - lo) * (uint32_t)sizeof(T);

    if (tid == 0) {
        for (int s = 0; s < p.slots; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], nwc);
        }
        fence_mbar_init();
    }
    if constexpr (sizeof(T) == 8) {
        for (int i = tid; i < kExp2TabSize; i += blockDim.x) tab[i] = g_exp2_tab[i];
    }
    __syncthreads();
    pdl_wait();  // everything below touches global memory written or read by the previous launch

    if (warp == nwc) {
        if (lane == 0) {
            const T *src = reinterpret_cast<const T *>(p.in) + (long long)frame * p.in_bstride + lo;
            int slot = 0;
            uint32_t round = 0;
            for (int j = 0; j < n_load; ++j) {
                if (round > 0) {
                    while (!mbar_test(&empty[slot], (round - 1) & 1)) __nanosleep(500);
                }
                const long long y = reflect_any(p.gwy0 + r + (long long)(i0 - C + j) * p.d, p.Hg) - p.gwy0 + p.row_off_in;
                mbar_arrive_expect_tx(&full[slot], row_bytes);
                tma_load_1d(rows + (size_t)slot * p.row_stride, src + y * p.in_pitch, row_bytes,
                            &full[slot]);
                if (++slot == p.slots) { slot = 0; ++round; }
            }
        }
        return;
    }

    T *out_c = reinterpret_cast<T *>(p.out_c);
    T *out_w = reinterpret_cast<T *>(p.out_w);
    if (out_c) out_c += (long long)frame * p.c_bstride;
    if (out_w) out_w += (long long)frame * p.w_bstride;

    const int xg = x0 + tid * V;
    const bool act = xg < p.W;
    const TapPlan<NV> plan = make_tap_plan<V, NV>(act ? xg : x0, DMODE == 0 ? p.d : V, p.W, lo);
    const int own = (act ? xg : x0) - lo;  // this thread's own vector inside a staged row
    const T var_factor = (T)bp.var_factor;
    T *my_stats = stats + (size_t)tid * 2 * V;
    constexpr int kStatSlot = 256 * 2 * V;  // elements per stats slot

    long long orow = (long long)r + (long long)i0 * p.d;
    int slot = 0, fslot = 0;  // slot of row j, slot of row j - 2C (first row of the window, next to be released)
    int sslot = 0;            // j % TAPS
    uint32_t parity = 0;
    for (int j = 0; j < n_load; ++j) {
        mbar_wait(&full[slot], parity);
        {
            // statistics of the newest row relative to its own centre column:
            // a = sum_k h_k (x_k - x_c), b = sum_k h_k (x_k - x_c)^2
            T tv[TAPS][V];
            row_taps<T, TAPS, DMODE>(rows + (size_t)slot * p.row_stride, plan, tv);
            Pack<T, V> sa, sb;
#pragma unroll
            for (int e = 0; e < V; ++e) {
                T a = T(0), b = T(0);
#pragma unroll
                for (int k = 0; k < C; ++k) {
                    const T dl = tv[k][e] - tv[C][e], dr = tv[TAPS - 1 - k][e] - tv[C][e];
                    a = fma_t<T>(Taps<T, TAPS>::h(k), dl + dr, a);
                    b = fma_t<T>(Taps<T, TAPS>::h(k), fma_t<T>(dr, dr, dl * dl), b);
                }
                sa.v[e] = a;
                sb.v[e] = b;
            }
            st_vec(my_stats + (size_t)sslot * kStatSlot, sa);
            st_vec(my_stats + (size_t)sslot * kStatSlot + V, sb);
        }
        if (j >= 2 * C) {
            if (act) {
                int cs = fslot + C;
                if (cs >= p.slots) cs -= p.slots;
                const Pack<T, V> xc = ld_vec(rows + (size_t)cs * p.row_stride + own);
                // window moments from the row statistics, rows top to bottom (window row i is chain row j - 2C + i)
                T s1[V], s2[V];
#pragma unroll
                for (int e = 0; e < V; ++e) { s1[e] = T(0); s2[e] = T(0); }
                int ws = fslot, ss = sslot + 1;  // (j - 2C) % TAPS == (j + 1) % TAPS
                if (ss == TAPS) ss = 0;
#pragma unroll
                for (int i = 0; i < TAPS; ++i) {
                    const T hi_ = Taps<T, TAPS>::h(i);
                    const Pack<T, V> sa = ld_vec(my_stats + (size_t)ss * kStatSlot);
                    const Pack<T, V> sb = ld_vec(my_stats + (size_t)ss * kStatSlot + V);
                    if (i == C) {
#pragma unroll
                        for (int e = 0; e < V; ++e) {
                            s1[e] = fma_t<T>(-hi_, sa.v[e], s1[e]);
                            s2[e] = fma_t<T>(hi_, sb.v[e], s2[e]);
                        }
                    } else {
                        const Pack<T, V> xi = ld_vec(rows + (size_t)ws * p.row_stride + own);
#pragma unroll
                        for (int e = 0; e < V; ++e) {
                            const T dc = xc.v[e] - xi.v[e];
                            const T t = fma_t<T>(T(-2), sa.v[e], dc);
                            const T u = fma_t<T>(dc, t, sb.v[e]);
                            s1[e] = fma_t<T>(hi_, dc - sa.v[e], s1[e]);
                            s2[e] = fma_t<T>(hi_, u, s2[e]);
                        }
                    }
                    if (++ws == p.slots) ws = 0;
                    if (++ss == TAPS) ss = 0;
                }
                T nhi[V], num[V], den[V];
#pragma unroll
                for (int e = 0; e < V; ++e) {
                    T var = s2[e] - s1[e] * s1[e];
                    if (var <= T(0)) var = T(1e-20);
                    nhi[e] = nhalf_inverse<T>(var * var_factor);
                    if constexpr (sizeof(T) == 8) nhi[e] *= 1.4426950408889634;  // exponent in base 2 for exp2_tab
                    num[e] = T(0);
                    den[e] = Taps<T, TAPS>::h(C) * Taps<T, TAPS>::h(C);
                }
                ws = fslot;
#pragma unroll
                for (int i = 0; i < TAPS; ++i) {
                    T tv[TAPS][V];
                    row_taps<T, TAPS, DMODE>(rows + (size_t)ws * p.row_stride, plan, tv);
#pragma unroll
                    for (int k = 0; k < TAPS; ++k) {
                        if (i == C && k == C) continue;
#pragma unroll
                        for (int e = 0; e < V; ++e) {
                            const T dd = xc.v[e] - tv[k][e];
                            T gw;
                            if constexpr (sizeof(T) == 8)
                                gw = exp2_tab(fma(dd * dd, nhi[e], TapLog2d<TAPS>::l(i) + TapLog2d<TAPS>::l(k)), tab);
                            else
                                gw = range_weight(Taps<T, TAPS>::h(i) * Taps<T, TAPS>::h(k), dd * dd, nhi[e]);
                            den[e] += gw;
                            num[e] = fma_t<T>(gw, dd, num[e]);
                        }
                    }
                    if (++ws == p.slots) ws = 0;
                }
                Pack<T, V> cn, wv;
#pragma unroll
                for (int e = 0; e < V; ++e) {
                    if constexpr (sizeof(T) == 8) cn.v[e] = xc.v[e] - num[e] * __drcp_rn(den[e]);
                    else cn.v[e] = xc.v[e] - num[e] / den[e];
                    wv.v[e] = xc.v[e] - cn.v[e];
                }
                if (out_c) st_vec(out_c + (orow + p.row_off_c) * p.c_pitch + xg, cn);
                if (out_w) st_vec_cs(out_w + (orow + p.row_off_w) * p.w_pitch + xg, wv);
            }
            orow += p.d;
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[fslot]);
            if (++fslot == p.slots) fslot = 0;
        }
        if (++slot == p.slots) { slot = 0; parity ^= 1; }
        if (++sslot == TAPS) sslot = 0;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// fp32 fast path: packed fp32x2 arithmetic (FADD2 / FMUL2 / FFMA2), one PAIR of adjacent pixels per thread.
//
// The kernel is bound by the FMA and MUFU pipes, not by HBM (24 exponentials and ~190 fp32 operations per pixel), and
// with scalar code it is bound by instruction ISSUE before either pipe saturates (ncu: 350 instructions per pixel, 64 %
// issue-active, FMA pipe 44 %, XU pipe 41 %).  sm_100a's packed fp32 instructions do two fp32 operations per lane per
// issue slot (tools/fma2bench.cu: 8 FFMA2 + 2 MUFU sustain 117 fma/clk/SM with the MUFU pipe at 92 %, 16 FFMA + 2 MUFU
// only 98), so the pixel pair is carried as one 64-bit register pair end to end: LDS.64 delivers it, every D, k*D,
// D^2, exponent argument and accumulation is one packed instruction, only the two ex2.approx are scalar.
// Reflected taps are the mirrored pair read backwards (halves swapped), a path only border threads take.
// Differences to the scalar formulation (all far below the fp32 parity budget): the tap weight enters through the
// exponent (2^(a + log2 k) instead of k 2^a), 1/(2V) and the final num/den use rcp.approx.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float rcp_fast(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// log2 of the taps (dyadic rationals except 3/8): log2(h_i h_k) = l_i + l_k
template <int TAPS> struct TapLog2;
template <> struct TapLog2<3> { __host__ __device__ static constexpr float l(int k) { return k == 1 ? -1.0f : -2.0f; } };
template <> struct TapLog2<5> {
    __host__ __device__ static constexpr float l(int k) { return k == 2 ? -1.4150374992788437f : ((k == 1 || k == 3) ? -2.0f : -4.0f); }
};

// DMODE 0: dilation even (>= 2): tap pair k is one aligned LDS.64 at column x + (k - C) d.
// DMODE 1: dilation 1: three aligned LDS.64 at x-2, x, x+2 form a 6-pixel window the taps are picked from.
template <int TAPS, int DMODE> struct PairPlan { static constexpr int NL = (DMODE == 0) ? TAPS : 3; };

template <int TAPS, int DMODE, bool MIRROR>
__device__ __forceinline__ void pair_taps(uint32_t rowb, const uint32_t (&colb)[PairPlan<TAPS, DMODE>::NL], unsigned rev,
                                          u64 (&out)[TAPS]) {
    constexpr int C = TAPS / 2;
    if constexpr (DMODE == 0) {
#pragma unroll
        for (int k = 0; k < TAPS; ++k) {
            u64 t = lds64(rowb + colb[k]);
            if (MIRROR) {
                const u64 u = swap2(t);
                t = ((rev >> k) & 1u) ? u : t;
            }
            out[k] = t;
        }
    } else {
        float win[6];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            u64 t = lds64(rowb + colb[k]);
            if (MIRROR) {
                const u64 u = swap2(t);
                t = ((rev >> k) & 1u) ? u : t;
            }
            up2(t, win[2 * k], win[2 * k + 1]);
        }
#pragma unroll
        for (int k = 0; k < TAPS; ++k) out[k] = pk2(win[2 + (k - C)], win[3 + (k - C)]);
    }
}

// Row statistics for the variance (law of total variance over the window rows).  For one staged row and this thread's
// pixel pair, relative to the row's own centre-column pixel x_c:   a = sum_k h_k (x_k - x_c),  b = sum_k h_k (x_k - x_c)^2.
// They depend on (row, column) only, so they are computed ONCE per input row (when it becomes the newest window row)
// and kept in registers for the 2C later windows that contain the row.  With e_i = x_ic - x_cc
// (row centre minus window centre) the window moments are
//     s1 = sum_i h_i (a_i + e_i),      s2 = sum_i h_i (b_i + e_i (2 a_i + e_i)),      var = s2 - s1^2
// -- still differences only (no cancellation), 60 packed operations per pixel pair instead of 96.
template <int TAPS>
__device__ __forceinline__ P4 row_stats(const u64 (&tv)[TAPS]) {
    constexpr int C = TAPS / 2;
    u64 a = 0ull, b = 0ull;
#pragma unroll
    for (int k = 0; k < C; ++k) {
        const float hk = Taps<float, TAPS>::h(k);
        const u64 dl = sub2(tv[k], tv[C]), dr = sub2(tv[TAPS - 1 - k], tv[C]);
        const u64 sum = add2(dl, dr);
        const u64 sq = fma2(dr, dr, mul2(dl, dl));
        a = (k == 0) ? mul2(pk2(hk, hk), sum) : fma2(pk2(hk, hk), sum, a);
        b = (k == 0) ? mul2(pk2(hk, hk), sq) : fma2(pk2(hk, hk), sq, b);
    }
    return P4{a, b};
}

// ---------------------------------------------------------------------------------------------------------------
// fp32 fast path, round 2: the 5x5 tap VALUES of the pixel pair held in a REGISTER sliding window
// (bilateral_window_kernel).  The round-1 kernel re-loaded all 25 tap pairs for every output row: ncu counted 457 warp
// instructions per warp-row of which 255 were FP / MUFU, the rest being 30 LDS.64 with one address add each, a
// row-statistics ring in shared memory and its indexing.  Here a staged row is read ONCE per thread, when it arrives
// (TAPS LDS.64), into the window X[row slot][tap]; its row statistics (a, b) stay in registers too.  The step loop is
// unrolled by TAPS so that the rotating row slot is a compile-time index: no register moves, no shared-memory ring
// beyond the TMA staging slots (released right after the loads), ~250 warp instructions per warp-row of which 48 are
// the MUFU ex2 that bound the kernel (2 per packed tap: 24 * 4096^2 exponentials per plane = 87 us of MUFU pipe).
// The lean kernel below runs the same operations in the same order, faster; this one serves what it declines (one
// output, L2 hints off, staged rows over 16 KiB, d * pitch over 2^31 bytes) with bit-identical planes.
// ---------------------------------------------------------------------------------------------------------------
// 8 consumer warps + a ninth warp whose lane 0 streams the rows.  Two blocks per SM at the 96 registers ptxas budgets
// for this block size (a few spilled values; __maxnreg__(104) or (112) removes them but the register file then
// holds ONE block per SM: 204 - 222 instead of 150 us).  At 96 registers ptxas emits sub -> mul -> fma -> 2 MUFU ->
// accumulate serially per tap; larger register budgets (setmaxnreg producer warp groups, 160-thread blocks at 128
// registers, a row prefetched one step ahead) interleave the taps but measured within 3 % of this geometry
// (DESIGN §4 K2; those variants were deleted).
template <int TAPS, int DMODE>
__global__ void __launch_bounds__(288, 2) bilateral_window_kernel(const BilateralParams bp) {
    const ScaleParams &p = bp.sp;
    pdl_launch_dependents();
    constexpr int C = TAPS / 2;
    constexpr int NL = PairPlan<TAPS, DMODE>::NL;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float *rows = reinterpret_cast<float *>(smem_raw);
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw + (size_t)p.slots * p.row_stride * sizeof(float));
    uint64_t *empty = full + p.slots;

    constexpr int nt = 256, nwc = 8;  // consumer threads / warps; warp 8 is the TMA producer
    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int lane = tid & 31;

    int bx = blockIdx.x;
    const int strip = bx % p.n_strips;
    bx /= p.n_strips;
    const int r = bx % p.d;
    const int g = bx / p.d;
    const int frame = blockIdx.y;

    const int n_chain = (r < p.H) ? (p.H - r + p.d - 1) / p.d : 0;
    const int i0 = g * p.seg;
    const int n_out = min(p.seg, n_chain - i0);
    if (n_out <= 0) return;
    const int n_load = n_out + 2 * C;

    const int x0 = strip * p.wt;
    const int lo = max(0, x0 - p.halo_al);
    const int hi = min(p.W, x0 + p.wt + p.halo_al);
    const uint32_t row_bytes = (uint32_t)(hi - lo) * (uint32_t)sizeof(float);
    const uint32_t RB = (uint32_t)p.row_stride * (uint32_t)sizeof(float);

    if (tid == 0) {
        for (int s = 0; s < p.slots; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], nwc);
        }
        fence_mbar_init();
    }
    __syncthreads();
    pdl_wait();  // everything below touches global memory written or read by the previous launch

    // loader state (one thread): the next chain row to request, its ring slot and its position in the 2 Hg-periodic
    // symmetric extension of the (global) image, walked incrementally
    const float *src = reinterpret_cast<const float *>(p.in) + (long long)frame * p.in_bstride + lo;
    const uint64_t pol_in = policy_evict_first();  // c_s is dead once this launch has read it
    int next_load = 0, lslot = 0;
    uint32_t lround = 0;
    const long long period = 2LL * p.Hg;
    const long long d_mod = (long long)p.d % period;
    long long m_pos = 0;
    if (tid == nt) {
        m_pos = (p.gwy0 + r + (long long)(i0 - C) * p.d) % period;
        if (m_pos < 0) m_pos += period;
    }
    auto issue_load = [&]() {
        const long long y = (m_pos < p.Hg ? m_pos : period - 1 - m_pos) - p.gwy0 + p.row_off_in;
        mbar_arrive_expect_tx(&full[lslot], row_bytes);
        if (p.l2_hints) tma_load_1d_hint(rows + (size_t)lslot * p.row_stride, src + y * p.in_pitch, row_bytes, &full[lslot], pol_in);
        else tma_load_1d(rows + (size_t)lslot * p.row_stride, src + y * p.in_pitch, row_bytes, &full[lslot]);
        ++next_load;
        if (++lslot == p.slots) { lslot = 0; ++lround; }
        m_pos += d_mod;
        if (m_pos >= period) m_pos -= period;
    };
    if (warp >= nwc) {
        if (warp == nwc && lane == 0) {
            // one row per iteration: unrolled, this loop would only add instruction-cache footprint
#pragma unroll 1
            while (next_load < n_load) {
                // blocking try_wait: a test + nanosleep poll measured identical (154 us, 91.8 M warp instructions per
                // plane for 1000 / 5000 ns sleeps), so the waiting lane takes no issue slots from the arithmetic either way
                if (lround > 0) mbar_wait(&empty[lslot], (lround - 1) & 1);
                issue_load();
            }
        }
        return;
    }

    float *out_c = reinterpret_cast<float *>(p.out_c);
    float *out_w = reinterpret_cast<float *>(p.out_w);

    int xg = x0 + tid * 2;
    const bool act = xg < p.W && xg < x0 + p.wt;
    if (!act) xg = x0;  // idle threads shadow the first pair of the strip; their stores are masked
    uint32_t colb[NL];
    unsigned rev = 0;
#pragma unroll
    for (int k = 0; k < NL; ++k) {
        const int pcol = xg + (k - NL / 2) * (DMODE == 0 ? p.d : 2);  // even; one reflection at most
        const bool left = pcol < 0, right = pcol >= p.W;
        const int q = left ? (-2 - pcol) : (right ? (2 * p.W - 2 - pcol) : pcol);
        colb[k] = smem_u32(rows) + (uint32_t)(q - lo) * 4u;  // absolute address of the tap in ring slot 0
        if (left || right) rev |= 1u << k;
    }
    const float var_factor = bp.var_factor_f;
    const uint64_t pol_keep = p.l2_hints ? policy_evict_last() : 0ull;  // c_{s+1}: the next scale reads it back
    const float kc = Taps<float, TAPS>::h(C) * Taps<float, TAPS>::h(C);

    // per-thread output pointers of the first output row; one add per row afterwards
    const long long orow0 = (long long)r + (long long)i0 * p.d;
    float *c_dst = out_c ? out_c + (long long)frame * p.c_bstride + (orow0 + p.row_off_c) * p.c_pitch + xg : nullptr;
    float *w_dst = out_w ? out_w + (long long)frame * p.w_bstride + (orow0 + p.row_off_w) * p.w_pitch + xg : nullptr;
    const long long c_step = (long long)p.d * p.c_pitch, w_step = (long long)p.d * p.w_pitch;

    auto run = [&](auto mirror) {
        constexpr bool MIRROR = decltype(mirror)::value != 0;
        u64 X[TAPS][TAPS];       // X[row slot][tap]: tap pairs of the last TAPS chain rows (row j lives in slot j % TAPS)
        u64 SA[TAPS], SB[TAPS];  // row statistics (a, b) of those rows, see row_stats
        int slot = 0;
        uint32_t parity = 0;
        // Step j = TAPS u + I: chain row j lands -> its tap pairs and statistics enter slot I; from j = 2C on, the
        // output row j - C (centre slot (I - C) mod TAPS) is produced from the window.
        auto step = [&](auto ic, const int j) {
            constexpr int I = decltype(ic)::value;
            if (j >= n_load) return;
            mbar_wait(&full[slot], parity);
            pair_taps<TAPS, DMODE, MIRROR>((uint32_t)slot * RB, colb, rev, X[I]);
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[slot]);  // the staged row is read exactly once per thread
            if (++slot == p.slots) { slot = 0; parity ^= 1; }
            {
                const P4 st = row_stats<TAPS>(X[I]);
                SA[I] = st.lo;
                SB[I] = st.hi;
            }
            if (j < 2 * C) return;
            constexpr int RC = (I + TAPS - C) % TAPS;  // slot of the centre row
            const u64 xc = X[RC][C];
            // window moments from the row statistics (law of total variance, differences only), rows top to bottom
            u64 s1 = 0ull, s2 = 0ull;
#pragma unroll
            for (int i = 0; i < TAPS; ++i) {
                const int rs = (I + 1 + i) % TAPS;  // compile-time after unrolling
                const float hi_ = Taps<float, TAPS>::h(i);
                if (i == C) {
                    s1 = fma2(pk2(-hi_, -hi_), SA[rs], s1);
                    s2 = fma2(pk2(hi_, hi_), SB[rs], s2);
                } else {
                    const u64 dc = sub2(xc, X[rs][C]);
                    const u64 t = fma2(pk2(-2.0f, -2.0f), SA[rs], dc);
                    const u64 u = fma2(dc, t, SB[rs]);
                    s1 = fma2(pk2(hi_, hi_), sub2(dc, SA[rs]), s1);
                    s2 = fma2(pk2(hi_, hi_), u, s2);
                }
            }
            // var = S[x^2] - S[x]^2 in centred form; V = max(var, 1e-20) * var_factor (kept a normal number: a tiny
            // var_factor must not turn 1 / V into inf and the weight of an equal neighbour into 0 * inf);
            // exponent scale -log2(e) / (2 V)
            float v0, v1;
            up2(sub2(s2, mul2(s1, s1)), v0, v1);
            v0 = (v0 <= 0.0f) ? 1e-20f : v0;
            v1 = (v1 <= 0.0f) ? 1e-20f : v1;
            const u64 nhi = pk2(-0.72134752044448170f * rcp_fast(fmaxf(v0 * var_factor, 1e-37f)),
                                -0.72134752044448170f * rcp_fast(fmaxf(v1 * var_factor, 1e-37f)));
            u64 num = 0ull, den = pk2(kc, kc);
#pragma unroll
            for (int i = 0; i < TAPS; ++i) {
                const int rs = (I + 1 + i) % TAPS;
#pragma unroll
                for (int k = 0; k < TAPS; ++k) {
                    if (i == C && k == C) continue;
                    const float lk = TapLog2<TAPS>::l(i) + TapLog2<TAPS>::l(k);
                    const u64 dd = sub2(xc, X[rs][k]);
                    float a0, a1;
                    up2(fma2(mul2(dd, dd), nhi, pk2(lk, lk)), a0, a1);
                    const u64 gw = pk2(exp2_fast(a0), exp2_fast(a1));
                    den = add2(den, gw);
                    num = fma2(gw, dd, num);
                }
            }
            float n0, n1, d0, d1, x0v, x1v;
            up2(num, n0, n1);
            up2(den, d0, d1);
            up2(xc, x0v, x1v);
            const float c0 = fmaf(-n0, rcp_fast(d0), x0v), c1 = fmaf(-n1, rcp_fast(d1), x1v);  // one FFMA each, spelled out: left to
            // the compiler's contraction, one kernel fused both halves of the pair and another only one (1-ulp differences)
            if (act) {
                if (c_dst) {
                    if (pol_keep)
                        asm volatile("st.global.L2::cache_hint.v2.f32 [%0], {%1, %2}, %3;" ::"l"(c_dst), "f"(c0), "f"(c1), "l"(pol_keep) : "memory");
                    else
                        *reinterpret_cast<float2 *>(c_dst) = make_float2(c0, c1);
                }
                if (w_dst) __stcs(reinterpret_cast<float2 *>(w_dst), make_float2(x0v - c0, x1v - c1));
            }
            if (c_dst) c_dst += c_step;
            if (w_dst) w_dst += w_step;
        };
#pragma unroll 1
        for (int jb = 0; jb < n_load; jb += TAPS) {
            step(IC<0>{}, jb + 0);
            step(IC<1>{}, jb + 1);
            step(IC<2>{}, jb + 2);
            if constexpr (TAPS == 5) {
                step(IC<3>{}, jb + 3);
                step(IC<4>{}, jb + 4);
            }
        }
    };
    // warps that own no reflected column (all but the first / last strip's edge warps) run the variant without the
    // mirror selects; the choice is warp-uniform, so no thread diverges inside the step
    if (__any_sync(0xffffffffu, rev != 0)) run(IC<1>{});
    else run(IC<0>{});
}

// ---------------------------------------------------------------------------------------------------------------
// fp32, round 2 (second half): the register-window kernel made LEAN (bilateral_lean_kernel).  tools/k2mimic.cu replays
// the arithmetic of one window step (162 packed operations, 52 MUFU, ~15 others) on the same SM: 506 cycles per
// warp-row whatever the warp count, i.e. 114 us per 4096^2 plane, and every further instruction costs about one more
// cycle (a packed fp32x2 instruction holds the issue port for two cycles, nothing hides under it).  The window kernel
// executes 350 - 374 instructions per warp-row: ~130 of them are not arithmetic -- dynamic ring-slot arithmetic (slot *
// stride, wrap, parity), one address add per LDS.64, null-pointer / activity / hint selects, parameters re-read from the
// constant bank, spills.  Here the staging ring has as many slots as the unrolled step loop has steps (5 for B3spline,
// 6 for Triangle: a staged row is read once, on arrival, so a few rows of prefetch suffice) and a fixed 16 KiB
// stride: ring slot, barrier and parity are compile-time / one bit per loop iteration and every LDS.64 is
// [register + immediate]; both outputs and the L2 hints are unconditional (the dispatcher sends everything else to the
// window kernel).  Same operations in the same order: bit-identical planes.
// ---------------------------------------------------------------------------------------------------------------
static constexpr int kK2LeanRB = 16384;  // ring slot stride in bytes (a 512-column strip + 2 x 2 C d halo columns, d <= 448)
template <int TAPS> struct K2LeanRing { static constexpr int R = (TAPS == 5) ? 5 : 6; };  // ring slots == unrolled steps

template <int OFF> __device__ __forceinline__ u64 lds64_imm(uint32_t a) {
    u64 r;
    asm volatile("ld.shared.b64 %0, [%1+%2];" : "=l"(r) : "r"(a), "n"(OFF));
    return r;
}
// taps k = 0 .. TAPS-1 of an interior pair at dilation 2^LD: [own + slot offset + (k - C) * 4 * 2^LD], all immediates
template <int TAPS, int SLOT_OFF, int LD, int... K>
__device__ __forceinline__ void lean_load_taps(uint32_t own, u64 (&x)[TAPS], std::integer_sequence<int, K...>) {
    ((x[K] = lds64_imm<SLOT_OFF + (K - TAPS / 2) * (4 << LD)>(own)), ...);
}

// LD >= 0: the dilation is 2^LD, known at compile time -- the taps of an interior pair are then [own + immediate] and cost
// neither registers nor address arithmetic (held as five addresses they were spilled: four LDL per step); LD < 0: any
// dilation, tap addresses formed from own and the stride.
template <int TAPS, int DMODE, int LD>
__global__ void __launch_bounds__(288, 2) bilateral_lean_kernel(const BilateralParams bp) {
    const ScaleParams &p = bp.sp;
    pdl_launch_dependents();
    constexpr int C = TAPS / 2;
    constexpr int NL = PairPlan<TAPS, DMODE>::NL;
    constexpr int R = K2LeanRing<TAPS>::R;
    constexpr int RB = kK2LeanRB;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw + (size_t)R * RB);
    uint64_t *empty = full + R;
    const uint32_t rows0 = smem_u32(smem_raw);
    constexpr int FULL_OFF = R * RB, EMPTY_OFF = R * RB + 8 * R;  // barriers behind the ring: [ring base + immediate]

    constexpr int nt = 256, nwc = 8;  // consumer threads / warps; warp 8 is the TMA producer
    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int lane = tid & 31;

    int bx = blockIdx.x;
    const int strip = bx % p.n_strips;
    bx /= p.n_strips;
    const int r = bx % p.d;
    const int g = bx / p.d;
    const int frame = blockIdx.y;

    const int n_chain = (r < p.H) ? (p.H - r + p.d - 1) / p.d : 0;
    const int i0 = g * p.seg;
    const int n_out = min(p.seg, n_chain - i0);
    if (n_out <= 0) return;
    const int n_load = n_out + 2 * C;

    const int x0 = strip * p.wt;
    const int lo = max(0, x0 - p.halo_al);
    const int hi = min(p.W, x0 + p.wt + p.halo_al);
    const uint32_t row_bytes = (uint32_t)(hi - lo) * (uint32_t)sizeof(float);

    if (tid == 0) {
        for (int s = 0; s < R; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], nwc);
        }
        fence_mbar_init();
    }
    __syncthreads();
    pdl_wait();  // everything below touches global memory written or read by the previous launch

    if (warp == nwc) {
        if (lane == 0) {
            // loader: the next chain row's position in the 2 Hg-periodic symmetric extension, walked incrementally
            const float *src = reinterpret_cast<const float *>(p.in) + (long long)frame * p.in_bstride + lo;
            const uint64_t pol_in = policy_evict_first();  // c_s is dead once this launch has read it
            const long long period = 2LL * p.Hg;
            const long long d_mod = (long long)p.d % period;
            long long m_pos = (p.gwy0 + r + (long long)(i0 - C) * p.d) % period;
            if (m_pos < 0) m_pos += period;
            int lslot = 0;
            uint32_t lround = 0;
            for (int j = 0; j < n_load; ++j) {
                if (lround > 0) mbar_wait(&empty[lslot], (lround - 1) & 1);
                const long long y = (m_pos < p.Hg ? m_pos : period - 1 - m_pos) - p.gwy0 + p.row_off_in;
                mbar_arrive_expect_tx(&full[lslot], row_bytes);
                tma_load_1d_hint(smem_raw + (size_t)lslot * RB, src + y * p.in_pitch, row_bytes, &full[lslot], pol_in);
                if (++lslot == R) { lslot = 0; ++lround; }
                m_pos += d_mod;
                if (m_pos >= period) m_pos -= period;
            }
        }
        return;
    }

    int xg = x0 + tid * 2;
    const bool act = xg < p.W && xg < x0 + p.wt;
    if (!act) xg = x0;  // idle threads shadow the first pair of the strip; their stores are masked
    uint32_t colb[NL];
    unsigned rev = 0;
#pragma unroll
    for (int k = 0; k < NL; ++k) {
        const int pcol = xg + (k - NL / 2) * (DMODE == 0 ? p.d : 2);  // even; one reflection at most
        const bool left = pcol < 0, right = pcol >= p.W;
        const int q = left ? (-2 - pcol) : (right ? (2 * p.W - 2 - pcol) : pcol);
        colb[k] = rows0 + (uint32_t)(q - lo) * 4u;  // absolute address of the tap in ring slot 0
        if (left || right) rev |= 1u << k;
    }
    const float var_factor = bp.var_factor_f;
    const uint64_t pol_keep = policy_evict_last();  // c_{s+1}: the next scale reads it back
    const float kc = Taps<float, TAPS>::h(C) * Taps<float, TAPS>::h(C);
    // values ptxas must HOLD (under register pressure it otherwise recomputes the shared-memory base from special
    // registers and the 64-bit row steps from the constant bank in every step): ring base, own tap address and tap
    // stride (interior warps address tap k as own + (k - C) stride), byte steps of the two output pointers
    const uint32_t sbase = opaque_u32(rows0);
    const uint32_t own = opaque_u32(colb[NL / 2]);
    const uint32_t tstep = opaque_u32((uint32_t)(DMODE == 0 ? p.d : 2) * 4u);
    const bool mirror_warp = __any_sync(0xffffffffu, rev != 0);
    if (mirror_warp) {
#pragma unroll
        for (int k = 0; k < NL; ++k) colb[k] = opaque_u32(colb[k]);
        rev = opaque_u32(rev);
    }

    // per-thread output pointers of the first output row; one 32-bit byte step per row afterwards (the host checks that
    // d * pitch * 4 fits)
    const long long orow0 = (long long)r + (long long)i0 * p.d;
    char *c_dst = reinterpret_cast<char *>(reinterpret_cast<float *>(p.out_c) + (long long)frame * p.c_bstride + (orow0 + p.row_off_c) * p.c_pitch + xg);
    char *w_dst = reinterpret_cast<char *>(reinterpret_cast<float *>(p.out_w) + (long long)frame * p.w_bstride + (orow0 + p.row_off_w) * p.w_pitch + xg);
    const uint32_t c_step = opaque_u32((uint32_t)((long long)p.d * p.c_pitch * 4)), w_step = opaque_u32((uint32_t)((long long)p.d * p.w_pitch * 4));

    auto run = [&](auto mirror) {
        constexpr bool MIRROR = decltype(mirror)::value != 0;
        u64 X[TAPS][TAPS];       // X[window slot][tap]: tap pairs of the last TAPS chain rows (row j lives in slot j % TAPS)
        u64 SA[TAPS], SB[TAPS];  // row statistics (a, b) of those rows, see row_stats
        // Step j = R u + I: chain row j lands in ring slot I -> its tap pairs and statistics enter window slot I % TAPS;
        // from j = 2C on, the output row j - C (centre slot (I - C) mod TAPS) is produced from the window.
        // interior warps: tap k of the pair is own + (k - C) * stride, formed where it is used -- held as five addresses
        // they were spilled (four LDL per step, long-scoreboard stalls); the volatile asm keeps ptxas from hoisting them
        auto tap_addr = [&](int m) -> uint32_t {
            if (m == 0) return own;
            uint32_t a;
            if (m == 1) asm volatile("add.u32 %0, %1, %2;" : "=r"(a) : "r"(own), "r"(tstep));
            else if (m == -1) asm volatile("sub.u32 %0, %1, %2;" : "=r"(a) : "r"(own), "r"(tstep));
            else if (m == 2) asm volatile("mad.lo.u32 %0, %2, 2, %1;" : "=r"(a) : "r"(own), "r"(tstep));
            else asm volatile("{.reg .u32 t; shl.b32 t, %2, 1; sub.u32 %0, %1, t;}" : "=r"(a) : "r"(own), "r"(tstep));
            return a;
        };
        auto step = [&](auto ic, const int j, const uint32_t parity) {
            constexpr int I = decltype(ic)::value;
            constexpr int WS = I % TAPS;
            if (j >= n_load) return;
            mbar_wait_imm<FULL_OFF + 8 * I>(sbase, parity);
            if constexpr (DMODE == 0 && !MIRROR && LD >= 0) {
                lean_load_taps<TAPS, I * RB, (LD >= 0 ? LD : 0)>(own, X[WS], std::make_integer_sequence<int, TAPS>{});
            } else if constexpr (DMODE == 0) {
#pragma unroll
                for (int k = 0; k < TAPS; ++k) {
                    u64 t = lds64_imm<I * RB>(MIRROR ? colb[k] : tap_addr(k - C));
                    if (MIRROR) {
                        const u64 u = swap2(t);
                        t = ((rev >> k) & 1u) ? u : t;
                    }
                    X[WS][k] = t;
                }
            } else {
                float win[6];
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    u64 t = lds64_imm<I * RB>(MIRROR ? colb[k] : tap_addr(k - 1));
                    if (MIRROR) {
                        const u64 u = swap2(t);
                        t = ((rev >> k) & 1u) ? u : t;
                    }
                    up2(t, win[2 * k], win[2 * k + 1]);
                }
#pragma unroll
                for (int k = 0; k < TAPS; ++k) X[WS][k] = pk2(win[2 + (k - C)], win[3 + (k - C)]);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive_imm<EMPTY_OFF + 8 * I>(sbase);  // the staged row is read exactly once per thread
            {
                const P4 st = row_stats<TAPS>(X[WS]);
                SA[WS] = st.lo;
                SB[WS] = st.hi;
            }
            if (j < 2 * C) return;
            constexpr int RC = (WS + TAPS - C) % TAPS;  // window slot of the centre row
            const u64 xc = X[RC][C];
            // window moments from the row statistics (law of total variance, differences only), rows top to bottom
            u64 s1 = 0ull, s2 = 0ull;
#pragma unroll
            for (int i = 0; i < TAPS; ++i) {
                const int rs = (WS + 1 + i) % TAPS;  // compile-time after unrolling
                const float hi_ = Taps<float, TAPS>::h(i);
                if (i == C) {
                    s1 = fma2(pk2(-hi_, -hi_), SA[rs], s1);
                    s2 = fma2(pk2(hi_, hi_), SB[rs], s2);
                } else {
                    const u64 dc = sub2(xc, X[rs][C]);
                    const u64 t = fma2(pk2(-2.0f, -2.0f), SA[rs], dc);
                    const u64 u = fma2(dc, t, SB[rs]);
                    s1 = fma2(pk2(hi_, hi_), sub2(dc, SA[rs]), s1);
                    s2 = fma2(pk2(hi_, hi_), u, s2);
                }
            }
            float v0, v1;
            up2(sub2(s2, mul2(s1, s1)), v0, v1);
            v0 = (v0 <= 0.0f) ? 1e-20f : v0;
            v1 = (v1 <= 0.0f) ? 1e-20f : v1;
            const u64 nhi = pk2(-0.72134752044448170f * rcp_fast(fmaxf(v0 * var_factor, 1e-37f)),
                                -0.72134752044448170f * rcp_fast(fmaxf(v1 * var_factor, 1e-37f)));
            u64 num = 0ull, den = pk2(kc, kc);
#pragma unroll
            for (int i = 0; i < TAPS; ++i) {
                const int rs = (WS + 1 + i) % TAPS;
#pragma unroll
                for (int k = 0; k < TAPS; ++k) {
                    if (i == C && k == C) continue;
                    const float lk = TapLog2<TAPS>::l(i) + TapLog2<TAPS>::l(k);
                    const u64 dd = sub2(xc, X[rs][k]);
                    float a0, a1;
                    up2(fma2(mul2(dd, dd), nhi, pk2(lk, lk)), a0, a1);
                    const u64 gw = pk2(exp2_fast(a0), exp2_fast(a1));
                    den = add2(den, gw);
                    num = fma2(gw, dd, num);
                }
            }
            float n0, n1, d0, d1, x0v, x1v;
            up2(num, n0, n1);
            up2(den, d0, d1);
            up2(xc, x0v, x1v);
            const float c0 = fmaf(-n0, rcp_fast(d0), x0v), c1 = fmaf(-n1, rcp_fast(d1), x1v);  // one FFMA each, spelled out: left to
            // the compiler's contraction, one kernel fused both halves of the pair and another only one (1-ulp differences)
            if (act) {
                asm volatile("st.global.L2::cache_hint.v2.f32 [%0], {%1, %2}, %3;" ::"l"(c_dst), "f"(c0), "f"(c1), "l"(pol_keep) : "memory");
                __stcs(reinterpret_cast<float2 *>(w_dst), make_float2(x0v - c0, x1v - c1));
            }
            c_dst += c_step;
            w_dst += w_step;
        };
        uint32_t parity = 0;
#pragma unroll 1
        for (int jb = 0; jb < n_load; jb += R) {
            step(IC<0>{}, jb + 0, parity);
            step(IC<1>{}, jb + 1, parity);
            step(IC<2>{}, jb + 2, parity);
            step(IC<3>{}, jb + 3, parity);
            step(IC<4>{}, jb + 4, parity);
            if constexpr (R == 6) step(IC<5>{}, jb + 5, parity);
            parity ^= 1u;
        }
    };
    // warps that own no reflected column (all but the first / last strip's edge warps) run the variant without the
    // mirror selects; the choice is warp-uniform, so no thread diverges inside the step
    if (mirror_warp) run(IC<1>{});
    else run(IC<0>{});
}

template <typename T, int TAPS>
__global__ void __launch_bounds__(256) bilateral_generic_kernel(const BilateralParams bp) {
    const ScaleParams &p = bp.sp;
    constexpr int C = TAPS / 2;
    const long long n = (long long)p.H * p.W;
    const int frame = blockIdx.y;
    const T *in = reinterpret_cast<const T *>(p.in) + (long long)frame * p.in_bstride;
    T *out_c = reinterpret_cast<T *>(p.out_c);
    T *out_w = reinterpret_cast<T *>(p.out_w);
    const T var_factor = (T)bp.var_factor;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n;
         idx += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(idx / p.W), x = (int)(idx % p.W);
        // band mode: output row y is global row gwy0 + y, found at buffer row y + row_off_in (see ScaleParams)
        const T xc = in[((long long)y + p.row_off_in) * p.in_pitch + x];
        T dlt[TAPS][TAPS];
        T s1 = T(0), s2 = T(0);
#pragma unroll
        for (int i = 0; i < TAPS; ++i) {
            // lattice: the recursive algorithm's border rule (every decimated sub-array reflects at its own edges)
            const T *row = in + (p.lattice ? (long long)reflect_lattice(y, i - C, p.d, p.H)
                                           : (long long)reflect_any(p.gwy0 + y + (long long)(i - C) * p.d, p.Hg) - p.gwy0 +
                                                 p.row_off_in) * p.in_pitch;
#pragma unroll
            for (int k = 0; k < TAPS; ++k) {
                const T dd = xc - row[p.lattice ? reflect_lattice(x, k - C, p.d, p.W)
                                                : reflect_any((long long)x + (long long)(k - C) * p.d, p.W)];
                dlt[i][k] = dd;
                const T kd = Taps<T, TAPS>::h(i) * Taps<T, TAPS>::h(k) * dd;
                s1 += kd;
                s2 = fma_t<T>(kd, dd, s2);
            }
        }
        T var = s2 - s1 * s1;
        if (var <= T(0)) var = T(1e-20);
        const T nhi = nhalf_inverse<T>(var * var_factor);
        T num = T(0), den = Taps<T, TAPS>::h(C) * Taps<T, TAPS>::h(C);
#pragma unroll
        for (int i = 0; i < TAPS; ++i)
#pragma unroll
            for (int k = 0; k < TAPS; ++k) {
                if (i == C && k == C) continue;
                const T gw = range_weight(Taps<T, TAPS>::h(i) * Taps<T, TAPS>::h(k), dlt[i][k] * dlt[i][k], nhi);
                den += gw;
                num = fma_t<T>(gw, dlt[i][k], num);
            }
        const T cn = xc - num / den;
        if (out_c) out_c[(long long)frame * p.c_bstride + ((long long)y + p.row_off_c) * p.c_pitch + x] = cn;
        if (out_w) out_w[(long long)frame * p.w_bstride + ((long long)y + p.row_off_w) * p.w_pitch + x] = xc - cn;
    }
}

template <typename T, int TAPS, int DMODE>
static int launch_bilateral(const BilateralParams &bp, int batch, int nt, cudaStream_t st) {
    auto kern = bilateral_rows_kernel<T, TAPS, DMODE>;
    const ScaleParams &p = bp.sp;
    if (sizeof(T) == 8) {
        const int rc = ensure_exp2_table();
        if (rc) return rc;
    }
    const size_t smem = (size_t)p.slots * p.row_stride * sizeof(T) + 16 * (size_t)p.slots + kExp2TabSize * sizeof(double) +
                        (size_t)TAPS * 256 * 32;  // + row-statistics ring: TAPS slots x 256 threads x 2 vectors
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem);
        if (e != cudaSuccess) return (int)e;
        if (dev >= 0 && dev < 64) configured[dev] = true;
    }
    dim3 grid((unsigned)((long long)p.n_strips * p.d * p.n_seg), (unsigned)batch);
    return launch_pdl<BilateralParams>(kern, grid, dim3((unsigned)(nt + 32)), smem, st, bp);
}

// Geometry for K2: one vector per thread, 256 consumer threads, the ring holds the `taps` window rows plus prefetch.
static bool plan_bilateral(ScaleParams &p, int taps, int esize, int batch) {
    const int V = 16 / esize;
    const int c = taps / 2;
    const int nt = 256;
    p.wt = nt * V;
    p.n_strips = (p.W + p.wt - 1) / p.wt;
    p.halo_al = round_up(c * p.d, V);
    long long rs = (long long)p.wt + 2LL * p.halo_al;
    if (rs > p.W) rs = p.W;
    p.row_stride = (int)rs;
    int slots = taps + 3;
    const int min_slots = taps + 1;
    const long long extra = kExp2TabSize * (long long)sizeof(double) + (long long)taps * 256 * 32;
    // two resident blocks per SM when the rows allow it
    while (slots > min_slots && (long long)slots * p.row_stride * esize + 16LL * slots + extra > kMaxSmem / 2 - 1024) --slots;
    if ((long long)slots * p.row_stride * esize + 16LL * slots + extra > kMaxSmem) return false;
    p.slots = slots;
    const int n_max = (p.H + p.d - 1) / p.d;
    // compute-bound kernel: many short segments balance better than few long ones; halo rows only cost L2 reads
    const long long chains = (long long)p.n_strips * (p.d < p.H ? p.d : p.H) * batch;
    const long long target = 8LL * device_sm_count();
    long long per_chain = (target + chains - 1) / chains;
    if (per_chain < 1) per_chain = 1;
    int seg = (int)((n_max + per_chain - 1) / per_chain);
    if (seg < 8 * c) seg = 8 * c;
    if (seg > n_max) seg = n_max;
    p.seg = seg;
    p.n_seg = (n_max + seg - 1) / seg;
    return true;
}

template <int TAPS, int DMODE>
static int launch_bilateral_window(const BilateralParams &bp, int batch, cudaStream_t st) {
    auto kern = bilateral_window_kernel<TAPS, DMODE>;
    const ScaleParams &p = bp.sp;
    const size_t smem = (size_t)p.slots * p.row_stride * sizeof(float) + 16 * (size_t)p.slots;
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem);
        if (e != cudaSuccess) return (int)e;
        if (dev >= 0 && dev < 64) configured[dev] = true;
    }
    dim3 grid((unsigned)((long long)p.n_strips * p.d * p.n_seg), (unsigned)batch);
    return launch_pdl<BilateralParams>(kern, grid, dim3(256 + 32), smem, st, bp);
}

template <int TAPS, int DMODE, int LD = -1>
static int launch_bilateral_lean(const BilateralParams &bp, int batch, cudaStream_t st) {
    auto kern = bilateral_lean_kernel<TAPS, DMODE, LD>;
    const ScaleParams &p = bp.sp;
    const size_t smem = (size_t)K2LeanRing<TAPS>::R * kK2LeanRB + 16 * (size_t)K2LeanRing<TAPS>::R;
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem);
        if (e != cudaSuccess) return (int)e;
        if (dev >= 0 && dev < 64) configured[dev] = true;
    }
    dim3 grid((unsigned)((long long)p.n_strips * p.d * p.n_seg), (unsigned)batch);
    return launch_pdl<BilateralParams>(kern, grid, dim3(256 + 32), smem, st, bp);
}

// The lean kernel takes the common case only: both outputs, L2 hints on, staged rows within its 16 KiB ring slots.
static bool k2_lean_ok(const ScaleParams &p) {
    return p.out_c && p.out_w && p.l2_hints && (long long)p.row_stride * 4 <= kK2LeanRB &&
           (long long)p.d * p.c_pitch * 4 < (1LL << 31) && (long long)p.d * p.w_pitch * 4 < (1LL << 31);
}

// The fp32 pair path: the lean kernel, 8 - 15 % faster than the register-window kernel at every scale
// (profiles/r2_bench_k2_lean.json), and the window kernel for the calls it declines.
template <int TAPS, int DMODE>
static int launch_bilateral_pair_path(const BilateralParams &bp, int batch, cudaStream_t st) {
    if (!k2_lean_ok(bp.sp)) return launch_bilateral_window<TAPS, DMODE>(bp, batch, st);
    if constexpr (TAPS == 5 && DMODE == 0) {
        // the B3spline scales of a dyadic cascade: dilation as a template parameter (immediate tap offsets)
        switch (bp.sp.d) {
            case 2: return launch_bilateral_lean<TAPS, DMODE, 1>(bp, batch, st);
            case 4: return launch_bilateral_lean<TAPS, DMODE, 2>(bp, batch, st);
            case 8: return launch_bilateral_lean<TAPS, DMODE, 3>(bp, batch, st);
            case 16: return launch_bilateral_lean<TAPS, DMODE, 4>(bp, batch, st);
            case 32: return launch_bilateral_lean<TAPS, DMODE, 5>(bp, batch, st);
            case 64: return launch_bilateral_lean<TAPS, DMODE, 6>(bp, batch, st);
            case 128: return launch_bilateral_lean<TAPS, DMODE, 7>(bp, batch, st);
            case 256: return launch_bilateral_lean<TAPS, DMODE, 8>(bp, batch, st);
            case 512: return launch_bilateral_lean<TAPS, DMODE, 9>(bp, batch, st);
            default: break;
        }
    }
    return launch_bilateral_lean<TAPS, DMODE>(bp, batch, st);
}

// Geometry for the fp32 pair kernels: 256 consumer threads x 2 pixels = 512-column strips, two resident blocks per SM.
static bool plan_bilateral_pair_path(ScaleParams &p, int taps, int batch) {
    const int c = taps / 2;
    p.wt = 512;
    p.n_strips = (p.W + p.wt - 1) / p.wt;
    p.halo_al = round_up(c * p.d, 4);
    long long rs = (long long)p.wt + 2LL * p.halo_al;
    if (rs > p.W) rs = p.W;
    p.row_stride = (int)rs;
    int slots = taps + 3;
    const int min_slots = taps + 1;
    // keep a block under half of the shared memory if possible
    while (slots > min_slots && (long long)slots * (p.row_stride * 4 + 16LL) > kMaxSmem / 2 - 1024) --slots;
    if ((long long)slots * (p.row_stride * 4 + 16LL) > kMaxSmem) return false;
    p.slots = slots;
    const int n_max = (p.H + p.d - 1) / p.d;
    // Compute-bound kernel: about 4 waves of 2 resident blocks per SM; halo rows only cost L2 reads.
    const long long chains = (long long)p.n_strips * (p.d < p.H ? p.d : p.H) * batch;
    const long long target = 4LL * 2 * device_sm_count();
    long long per_chain = (target + chains - 1) / chains;
    if (per_chain < 1) per_chain = 1;
    int seg = (int)((n_max + per_chain - 1) / per_chain);
    if (seg < 8 * c) seg = 8 * c;
    if (seg > n_max) seg = n_max;
    p.seg = seg;
    p.n_seg = (n_max + seg - 1) / seg;
    return true;
}

template <typename T, int TAPS>
static int dispatch_bilateral(BilateralParams &bp, int batch, cudaStream_t st) {
    constexpr int V = VecOf<T>::V;
    ScaleParams &p = bp.sp;
    if constexpr (sizeof(T) == 4) {
        // packed fp32x2 pair kernel: dilation 1 or even (every scale of a dyadic cascade)
        if (fast_path_ok(p, TAPS, 4) && (p.d == 1 || p.d % 2 == 0) && plan_bilateral_pair_path(p, TAPS, batch))
            return p.d == 1 ? launch_bilateral_pair_path<TAPS, 1>(bp, batch, st) : launch_bilateral_pair_path<TAPS, 0>(bp, batch, st);
    }
    if (fast_path_ok(p, TAPS, (int)sizeof(T)) && plan_bilateral(p, TAPS, (int)sizeof(T), batch)) {
        const int dmode = (p.d % V == 0) ? 0 : p.d;
        if (dmode == 0) return launch_bilateral<T, TAPS, 0>(bp, batch, 256, st);
        if (dmode == 1) return launch_bilateral<T, TAPS, 1>(bp, batch, 256, st);
        if constexpr (V == 4) {
            if (dmode == 2) return launch_bilateral<T, TAPS, 2>(bp, batch, 256, st);
        }
    }
    const long long n = (long long)p.H * p.W;
    long long blocks = (n + 255) / 256;
    const long long cap = 32LL * device_sm_count();
    if (blocks > cap) blocks = cap;
    bilateral_generic_kernel<T, TAPS><<<dim3((unsigned)blocks, (unsigned)batch), 256, 0, st>>>(bp);
    return launch_status();
}

}  // namespace wb

extern "C" {

int wb_atrous_scale_bilateral_band(const void *in, void *out_c, void *out_w, int band_rows, int W, int global_H,
                                   long long band_y0, long long in_row_offset, long long in_pitch,
                                   long long out_c_row_offset, long long out_c_pitch, long long out_w_row_offset,
                                   long long out_w_pitch, int scale, int taps, int dtype, double var_factor,
                                   void *stream) {
    int rc = wb::check_common(1, band_rows, W, taps, dtype);
    if (rc) return rc;
    if (scale < 0 || scale > 30) return WB_EINVAL_SCALE;
    if (!in || (!out_c && !out_w) || in == out_c || in == out_w) return WB_EINVAL_POINTER;
    if (global_H < band_rows || band_y0 < 0 || band_y0 + band_rows > global_H || in_pitch < W ||
        (out_c && out_c_pitch < W) || (out_w && out_w_pitch < W) || !(var_factor > 0))
        return WB_EINVAL_ARG;
    wb::BilateralParams bp;
    memset(&bp, 0, sizeof(bp));
    wb::ScaleParams &p = bp.sp;
    p.in = in; p.out_c = out_c; p.out_w = out_w;
    p.H = band_rows; p.W = W; p.d = 1 << scale; p.Hg = global_H;
    p.gwy0 = band_y0; p.row_off_in = in_row_offset; p.row_off_c = out_c_row_offset; p.row_off_w = out_w_row_offset;
    p.in_pitch = in_pitch; p.c_pitch = out_c_pitch; p.w_pitch = out_w_pitch;
    bp.var_factor = var_factor;
    bp.var_factor_f = (float)var_factor;
    p.l2_hints = wb::l2_hints_enabled();
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == WB_F32)
        return taps == 3 ? wb::dispatch_bilateral<float, 3>(bp, 1, st) : wb::dispatch_bilateral<float, 5>(bp, 1, st);
    return taps == 3 ? wb::dispatch_bilateral<double, 3>(bp, 1, st) : wb::dispatch_bilateral<double, 5>(bp, 1, st);
}

int wb_atrous_scale_bilateral_lattice(const void *in, void *out_c, void *out_w, int H, int W, long long in_pitch,
                                      long long out_c_pitch, long long out_w_pitch, int scale, int taps, int dtype,
                                      double var_factor, void *stream) {
    int rc = wb::check_common(1, H, W, taps, dtype);
    if (rc) return rc;
    if (scale < 0 || scale > 30) return WB_EINVAL_SCALE;
    if (!in || (!out_c && !out_w) || in == out_c || in == out_w) return WB_EINVAL_POINTER;
    if (in_pitch < W || (out_c && out_c_pitch < W) || (out_w && out_w_pitch < W) || !(var_factor > 0)) return WB_EINVAL_ARG;
    wb::BilateralParams bp;
    memset(&bp, 0, sizeof(bp));
    wb::ScaleParams &p = bp.sp;
    p.in = in; p.out_c = out_c; p.out_w = out_w;
    p.H = H; p.W = W; p.d = 1 << scale; p.Hg = H;
    p.in_pitch = in_pitch; p.c_pitch = out_c_pitch; p.w_pitch = out_w_pitch;
    p.lattice = 1;
    bp.var_factor = var_factor;
    bp.var_factor_f = (float)var_factor;
    const long long n = (long long)H * W;
    long long blocks = (n + 255) / 256;
    const long long cap = 32LL * wb::device_sm_count();
    if (blocks > cap) blocks = cap;
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid((unsigned)blocks, 1);
    if (dtype == WB_F32) {
        if (taps == 3) wb::bilateral_generic_kernel<float, 3><<<grid, 256, 0, st>>>(bp);
        else wb::bilateral_generic_kernel<float, 5><<<grid, 256, 0, st>>>(bp);
    } else {
        if (taps == 3) wb::bilateral_generic_kernel<double, 3><<<grid, 256, 0, st>>>(bp);
        else wb::bilateral_generic_kernel<double, 5><<<grid, 256, 0, st>>>(bp);
    }
    return wb::launch_status();
}

int wb_atrous_scale_bilateral(const void *in, void *out_c, void *out_w, int batch, int H, int W, long long in_pitch,
                              long long in_bstride, long long out_c_pitch, long long out_c_bstride,
                              long long out_w_pitch, long long out_w_bstride, int scale, int taps, int dtype,
                              double var_factor, void *stream) {
    int rc = wb::check_common(batch, H, W, taps, dtype);
    if (rc) return rc;
    if (scale < 0 || scale > 30) return WB_EINVAL_SCALE;
    if (!in || (!out_c && !out_w)) return WB_EINVAL_POINTER;
    if (in == out_c || in == out_w) return WB_EINVAL_POINTER;
    if (in_pitch < W || (out_c && out_c_pitch < W) || (out_w && out_w_pitch < W) || !(var_factor > 0)) return WB_EINVAL_ARG;
    wb::BilateralParams bp;
    memset(&bp, 0, sizeof(bp));
    wb::ScaleParams &p = bp.sp;
    p.in = in; p.out_c = out_c; p.out_w = out_w;
    p.H = H; p.W = W; p.d = 1 << scale; p.Hg = H;
    p.in_pitch = in_pitch; p.in_bstride = in_bstride;
    p.c_pitch = out_c_pitch; p.c_bstride = out_c_bstride;
    p.w_pitch = out_w_pitch; p.w_bstride = out_w_bstride;
    bp.var_factor = var_factor;
    bp.var_factor_f = (float)var_factor;
    p.l2_hints = wb::l2_hints_enabled();
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == WB_F32)
        return taps == 3 ? wb::dispatch_bilateral<float, 3>(bp, batch, st) : wb::dispatch_bilateral<float, 5>(bp, batch, st);
    return taps == 3 ? wb::dispatch_bilateral<double, 3>(bp, batch, st) : wb::dispatch_bilateral<double, 5>(bp, batch, st);
}

}  // extern "C"
