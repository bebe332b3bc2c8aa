// Pieces shared by the row-pipeline kernels (K1 transform, K3 whitening, K2 bilateral): launch parameters, the
// reflecting vector tap loader, the separable row pass and the host-side geometry planner.
#pragma once

#include "common.cuh"

namespace wb {

static constexpr int kMaxPeers = WB_MAX_PEERS;

struct ScaleParams {
    const void *in;
    void *out_c;
    void *out_w;
    int H, W, d;     // H = number of OUTPUT rows (the whole image, or one row band of it)
    // Row-band mode (multi-GPU, wb_atrous_scale_band): the buffers hold a window of a taller global image.
    // Output row i of this launch is global row gwy0 + i; taps reflect about the GLOBAL height Hg; a global row g is
    // found at buffer row g - gwy0 + row_off_in of `in` (halo rows materialised by the caller), and output row i is
    // written to buffer row i + row_off_c / row_off_w of out_c / out_w.  Single image: Hg = H, everything else 0.
    int Hg;
    long long gwy0;
    long long row_off_in, row_off_c, row_off_w;
    long long in_pitch, in_bstride, c_pitch, c_bstride, w_pitch, w_bstride;
    int wt;          // strip width in elements (= consumer threads * V * NG)
    int n_strips;    // column strips per row
    int seg;         // chain rows produced per thread block
    int n_seg;       // segments per chain
    int slots;       // depth of the shared-memory row ring
    int row_stride;  // elements per ring slot
    int halo_al;     // x halo kept in shared memory on each side of a strip (multiple of V)
    // --- whitening epilogue (OP_WHITEN): out_w = significance(raw) * raw * (weight / sqrt(max(S[raw^2], 1e-15)))
    int sig_mode;              // 0: no thresholding, 1: soft (erf), 2: hard, SIG_MAP: per-pixel noise map
    double sigma, sigma_e;     // threshold = (sigma * noise) * sigma_e   (watroo/wavelets.py:137,141)
    double noise_host;         // used when noise_dev == nullptr
    const double *noise_dev;   // device scalar per frame (from wb_abs_median), or nullptr
    double weight;             // recomposition weight of this plane
    int l2_hints;              // 1: L2 eviction-priority hints on loads / stores (see common.cuh)
    int lattice;               // generic kernel only: reflect inside the 2^s sub-lattice (recursive algorithm's border rule)
    // --- peer-window mode (wb_atrous_scale_band_p2p): the rows of c_s live in the band buffers of ALL ranks, every
    // one mapped into this process (NVLink peer memory).  Rank k's buffer starts at peer_in[k] and its row 0 is global
    // row peer_y0[k]; peer_y0[n_peers] = Hg.  n_peers == 0: a single window `in` (everything above).
    int n_peers;
    long long peer_y0[kMaxPeers + 1];
    const void *peer_in[kMaxPeers];
    // --- halo push (wb_atrous_scale_band_push): the rows of c_{s+1} that fall into a neighbour's halo of the NEXT scale
    // are stored a second time, straight into that neighbour's padded band buffer (posted writes over NVLink that overlap
    // with this launch's own streaming) -- the next scale then reads local memory only.  push_up / push_dn: address, in
    // the upper / lower neighbour's buffer, of this band's output row 0 (same pitch as out_c); output rows
    // [0, push_up_rows) go up, rows [push_dn_from, H) go down.  nullptr: no neighbour on that side.
    void *push_up, *push_dn;
    int push_up_rows, push_dn_from;
    // --- whitening with a noise map (sig_mode == SIG_MAP, wb_wow_whiten_scale_map): map of the plane dtype, element
    // (frame, y, x) at frame * map_bstride + y * map_pitch + x (map_bstride 0: one map for every frame); map_soft
    // selects erf (1) or the hard mask (0).  Last, so that the parameter offsets of the other kernels stay put.
    const void *noise_map;
    long long map_pitch, map_bstride;
    int map_soft;
};

// Second store of a c_{s+1} vector into the neighbours' halo zones (see ScaleParams::push_up).  `c_ptr` points at the
// vector inside out_c (row `row` of the band), `base` at row 0 of out_c incl. its row offset.
template <typename T, typename V>
__device__ __forceinline__ void push_store(const ScaleParams &p, const T *c_ptr, const T *base, int row, const V &val) {
    if (p.push_up && row < p.push_up_rows)
        *reinterpret_cast<V *>(reinterpret_cast<T *>(p.push_up) + (c_ptr - base)) = val;
    if (p.push_dn && row >= p.push_dn_from)
        *reinterpret_cast<V *>(reinterpret_cast<T *>(p.push_dn) + (c_ptr - base)) = val;
}

// Address of global input row gy (already reflected into [0, Hg)) of this launch's frame-0 window.
template <typename T>
__device__ __forceinline__ const T *input_row(const ScaleParams &p, long long gy) {
    if (p.n_peers == 0) return reinterpret_cast<const T *>(p.in) + (gy - p.gwy0 + p.row_off_in) * p.in_pitch;
    int k = 0;
    while (k + 1 < p.n_peers && gy >= p.peer_y0[k + 1]) ++k;
    return reinterpret_cast<const T *>(p.peer_in[k]) + (gy - p.peer_y0[k]) * p.in_pitch;
}

// OP_POWER: the row pipeline filters the squares of the staged rows (rounded, as T(w * w)) and writes only out_c.
enum { OP_TRANSFORM = 0, OP_WHITEN = 1, OP_POWER = 2 };
enum { SIG_MAP = 3 };  // ScaleParams::sig_mode of the noise-map whitening (wb_wow_whiten_scale_map)

// Per-thread, per-column-group tap plan, computed ONCE per thread block: the shared-memory element offset of the
// aligned vector that holds each tap (relative to the start of a staged row) and whether that vector has to be read
// backwards (symmetric border).  Nothing here depends on the row, so the inner loop is LDS.128 + FMA only.
//   DMODE == 0 (d % V == 0): NV = TAPS vectors at columns x + (k - C) d.
//   DMODE == d in {1, 2} (d < V): NV = 3 vectors (previous, current, next); the taps are picked from that window.
template <int NV> struct TapPlan {
    int off[NV];
    unsigned rev;  // bit k: vector k is mirrored
};

template <int V, int NV>
__device__ __forceinline__ TapPlan<NV> make_tap_plan(int x, int step, int W, int lo) {
    TapPlan<NV> tp;
    tp.rev = 0;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        const int p = x + (k - NV / 2) * step;  // p % V == 0, -W <= p < 2W (single reflection)
        const bool left = p < 0, right = p >= W;
        const int q = left ? (-V - p) : (right ? (2 * W - V - p) : p);
        tp.off[k] = q - lo;
        if (left || right) tp.rev |= 1u << k;
    }
    return tp;
}

template <typename T, int V> __device__ __forceinline__ void reverse_vec(Pack<T, V> &t) {
#pragma unroll
    for (int e = 0; e < V / 2; ++e) {
        T a = t.v[e];
        t.v[e] = t.v[V - 1 - e];
        t.v[V - 1 - e] = a;
    }
}

template <int TAPS, int DMODE> struct PlanSize { static constexpr int NV = (DMODE == 0) ? TAPS : 3; };

// Row pass for one vector of columns.  SQUARE: filter the squares of the staged values (local power of WOW).
template <typename T, int TAPS, int DMODE, bool SQUARE, bool MIRROR>
__device__ __forceinline__ Pack<T, VecOf<T>::V> row_pass_impl(const T *srow, const TapPlan<PlanSize<TAPS, DMODE>::NV> &tp) {
    constexpr int V = VecOf<T>::V;
    constexpr int C = TAPS / 2;
    Pack<T, V> acc;
    if constexpr (DMODE == 0) {
#pragma unroll
        for (int k = 0; k < TAPS; ++k) {
            Pack<T, V> t = ld_vec(srow + tp.off[k]);
            if (MIRROR && ((tp.rev >> k) & 1u)) reverse_vec<T, V>(t);
#pragma unroll
            for (int e = 0; e < V; ++e) {
                const T v = SQUARE ? t.v[e] * t.v[e] : t.v[e];
                acc.v[e] = (k == 0) ? Taps<T, TAPS>::h(0) * v : fma_t<T>(Taps<T, TAPS>::h(k), v, acc.v[e]);
            }
        }
    } else {
        T win[3 * V];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            Pack<T, V> t = ld_vec(srow + tp.off[k]);
            if (MIRROR && ((tp.rev >> k) & 1u)) reverse_vec<T, V>(t);
#pragma unroll
            for (int e = 0; e < V; ++e) win[k * V + e] = SQUARE ? t.v[e] * t.v[e] : t.v[e];
        }
#pragma unroll
        for (int e = 0; e < V; ++e) {
#pragma unroll
            for (int k = 0; k < TAPS; ++k) {
                const T v = win[V + e + (k - C) * DMODE];
                acc.v[e] = (k == 0) ? Taps<T, TAPS>::h(0) * v : fma_t<T>(Taps<T, TAPS>::h(k), v, acc.v[e]);
            }
        }
    }
    return acc;
}

template <typename T, int TAPS, int DMODE, bool SQUARE>
__device__ __forceinline__ Pack<T, VecOf<T>::V> row_pass(const T *srow, const TapPlan<PlanSize<TAPS, DMODE>::NV> &tp) {
    // interior threads (the vast majority) never mirror: keep their path free of the select chains
    if (tp.rev == 0) return row_pass_impl<T, TAPS, DMODE, SQUARE, false>(srow, tp);
    return row_pass_impl<T, TAPS, DMODE, SQUARE, true>(srow, tp);
}

// Column pass over the register ring of the last TAPS row-filtered rows, oldest row first:
// ((((h_0 r_0) + h_1 r_1) + h_2 r_2) + ...).  The fused WOW kernel (wow_scale.cu, col_feed) accumulates in the same
// order, so that its planes equal K1 followed by K3 bit for bit wherever no virtual (reflected) row is involved.
template <typename T, int TAPS, int NG>
__device__ __forceinline__ T col_pass(const Pack<T, VecOf<T>::V> (&ring)[TAPS][NG], int q, int e) {
    T a = Taps<T, TAPS>::h(0) * ring[0][q].v[e];
#pragma unroll
    for (int k = 1; k < TAPS; ++k) a = fma_t<T>(Taps<T, TAPS>::h(k), ring[k][q].v[e], a);
    return a;
}

// 16-byte shared-memory accesses on 32-bit shared-window addresses (address = per-thread offset + block-uniform base,
// which ptxas folds into the [R + UR] addressing mode: no per-load address arithmetic).
__device__ __forceinline__ Pack<float, 4> lds_vec_f(uint32_t a) {
    Pack<float, 4> r;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]) : "r"(a));
    return r;
}
__device__ __forceinline__ Pack<double, 2> lds_vec_d(uint32_t a) {
    Pack<double, 2> r;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(r.v[0]), "=d"(r.v[1]) : "r"(a));
    return r;
}
template <typename T> __device__ __forceinline__ Pack<T, VecOf<T>::V> lds_vec(uint32_t a);
template <> __device__ __forceinline__ Pack<float, 4> lds_vec<float>(uint32_t a) { return lds_vec_f(a); }
template <> __device__ __forceinline__ Pack<double, 2> lds_vec<double>(uint32_t a) { return lds_vec_d(a); }
__device__ __forceinline__ void sts_vec(uint32_t a, const Pack<float, 4> &r) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(r.v[0]), "f"(r.v[1]), "f"(r.v[2]), "f"(r.v[3])
                 : "memory");
}
__device__ __forceinline__ void sts_vec(uint32_t a, const Pack<double, 2> &r) {
    asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(a), "d"(r.v[0]), "d"(r.v[1]) : "memory");
}
// non-blocking probe of an mbarrier phase
__device__ __forceinline__ bool mbar_test(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}

// Per-thread tap plan in BYTES for one column vector (see TapPlan in pipeline.cuh).
template <int NV> struct BytePlan {
    uint32_t off[NV];
    unsigned rev;
};

// Row pass of one vector from the staged row at shared address `base` (block-uniform).  SQUARE filters the squares.
template <typename T, int TAPS, int DMODE, bool SQUARE, bool MIRROR>
__device__ __forceinline__ Pack<T, VecOf<T>::V> row_pass_b_impl(uint32_t base, const BytePlan<PlanSize<TAPS, DMODE>::NV> &tp) {
    constexpr int V = VecOf<T>::V;
    constexpr int C = TAPS / 2;
    Pack<T, V> acc;
    if constexpr (DMODE == 0) {
#pragma unroll
        for (int k = 0; k < TAPS; ++k) {
            Pack<T, V> t = lds_vec<T>(base + tp.off[k]);
            if (MIRROR && ((tp.rev >> k) & 1u)) reverse_vec<T, V>(t);
#pragma unroll
            for (int e = 0; e < V; ++e) {
                const T v = SQUARE ? t.v[e] * t.v[e] : t.v[e];
                acc.v[e] = (k == 0) ? Taps<T, TAPS>::h(0) * v : fma_t<T>(Taps<T, TAPS>::h(k), v, acc.v[e]);
            }
        }
    } else {
        T win[3 * V];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            Pack<T, V> t = lds_vec<T>(base + tp.off[k]);
            if (MIRROR && ((tp.rev >> k) & 1u)) reverse_vec<T, V>(t);
#pragma unroll
            for (int e = 0; e < V; ++e) win[k * V + e] = SQUARE ? t.v[e] * t.v[e] : t.v[e];
        }
#pragma unroll
        for (int e = 0; e < V; ++e) {
#pragma unroll
            for (int k = 0; k < TAPS; ++k) {
                const T v = win[V + e + (k - C) * DMODE];
                acc.v[e] = (k == 0) ? Taps<T, TAPS>::h(0) * v : fma_t<T>(Taps<T, TAPS>::h(k), v, acc.v[e]);
            }
        }
    }
    return acc;
}
template <typename T, int TAPS, int DMODE, bool SQUARE>
__device__ __forceinline__ Pack<T, VecOf<T>::V> row_pass_b(uint32_t base, const BytePlan<PlanSize<TAPS, DMODE>::NV> &tp) {
    if (tp.rev == 0) return row_pass_b_impl<T, TAPS, DMODE, SQUARE, false>(base, tp);
    return row_pass_b_impl<T, TAPS, DMODE, SQUARE, true>(base, tp);
}

// Column pass as running partial sums: S[t] is the partial sum of the output row that completes t+1 rows from now.
// Feeding the row-filtered vector v of the newest row returns the completed output (centre = C rows ago):
//     out = S[0] + h_{T-1} v;  S[t] = S[t+1] + h_{T-2-t} v;  S[T-2] = h_0 v
// i.e. ((((h_0 r_0) + h_1 r_1) + h_2 r_2) + ...) oldest row first -- the same order as K1's col_pass -- with every FMA
// writing the register the next step reads: no ring rotation, no moves, TAPS-1 live values per element.
template <typename T, int TAPS>
__device__ __forceinline__ T col_feed(T (&S)[TAPS - 1], T v) {
    const T out = fma_t<T>(Taps<T, TAPS>::h(TAPS - 1), v, S[0]);
#pragma unroll
    for (int t = 0; t + 2 < TAPS; ++t) S[t] = fma_t<T>(Taps<T, TAPS>::h(TAPS - 2 - t), v, S[t + 1]);
    S[TAPS - 2] = Taps<T, TAPS>::h(0) * v;
    return out;
}

// ---------------------------------------------------------------------------------------------------------------
// Packed fp32x2 forms of the row pass and of the running column sums (fp32, DMODE 0 or 2: every tap of a pixel pair
// is again an aligned pair).  Same operations in the same order as row_pass_b / col_feed, two pixels per issue slot.
// ---------------------------------------------------------------------------------------------------------------
template <int TAPS, typename T = float> struct PackedTaps {
    u64 h[TAPS];
    __device__ __forceinline__ PackedTaps() {
#pragma unroll
        for (int k = 0; k < TAPS; ++k) h[k] = Lane<T>::bcast(Taps<T, TAPS>::h(k));
    }
};

template <int TAPS, int DMODE, bool MIRROR>
__device__ __forceinline__ P4 row_pass_p_impl(uint32_t base, const BytePlan<PlanSize<TAPS, DMODE>::NV> &tp,
                                              const PackedTaps<TAPS> &H) {
    static_assert(DMODE == 0 || DMODE == 2, "packed row pass: d % 4 == 0 or d == 2");
    constexpr int C = TAPS / 2;
    P4 acc;
    if constexpr (DMODE == 0) {
#pragma unroll
        for (int k = 0; k < TAPS; ++k) {
            P4 t = lds_p4(base + tp.off[k]);
            if (MIRROR && ((tp.rev >> k) & 1u)) t = reverse_p4(t);
            acc.lo = (k == 0) ? mul2(H.h[0], t.lo) : fma2(H.h[k], t.lo, acc.lo);
            acc.hi = (k == 0) ? mul2(H.h[0], t.hi) : fma2(H.h[k], t.hi, acc.hi);
        }
    } else {
        u64 win[6];  // previous, current, next vector as six pixel pairs
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            P4 t = lds_p4(base + tp.off[k]);
            if (MIRROR && ((tp.rev >> k) & 1u)) t = reverse_p4(t);
            win[2 * k] = t.lo;
            win[2 * k + 1] = t.hi;
        }
#pragma unroll
        for (int k = 0; k < TAPS; ++k) {
            const int i = 2 + (k - C);  // pair that holds tap k of pixels (0, 1); pixels (2, 3) use the next pair
            acc.lo = (k == 0) ? mul2(H.h[0], win[i]) : fma2(H.h[k], win[i], acc.lo);
            acc.hi = (k == 0) ? mul2(H.h[0], win[i + 1]) : fma2(H.h[k], win[i + 1], acc.hi);
        }
    }
    return acc;
}
template <int TAPS, int DMODE>
__device__ __forceinline__ P4 row_pass_p(uint32_t base, const BytePlan<PlanSize<TAPS, DMODE>::NV> &tp,
                                         const PackedTaps<TAPS> &H) {
    if (tp.rev == 0) return row_pass_p_impl<TAPS, DMODE, false>(base, tp, H);
    return row_pass_p_impl<TAPS, DMODE, true>(base, tp, H);
}

template <int TAPS, typename T>
__device__ __forceinline__ u64 col_feed_p(u64 (&S)[TAPS - 1], u64 v, const PackedTaps<TAPS, T> &H) {
    const u64 out = Lane<T>::fma(H.h[TAPS - 1], v, S[0]);
#pragma unroll
    for (int t = 0; t + 2 < TAPS; ++t) S[t] = Lane<T>::fma(H.h[TAPS - 2 - t], v, S[t + 1]);
    S[TAPS - 2] = Lane<T>::mul(H.h[0], v);
    return out;
}

// ---------------------------------------------------------------------------------------------------------------
// Pieces of the LEAN fp32 kernels (wow_rows_lean_kernel, atrous_rows_lean_kernel): fixed 16 KiB ring slots so that
// every shared-memory access is [per-thread register + immediate], step loops unrolled by the ring.
// ---------------------------------------------------------------------------------------------------------------
template <int OFF> __device__ __forceinline__ P4 lds_p4_imm(uint32_t a) {
    P4 r;
    asm volatile("ld.shared.v2.b64 {%0, %1}, [%2+%3];" : "=l"(r.lo), "=l"(r.hi) : "r"(a), "n"(OFF));
    return r;
}
template <int OFF> __device__ __forceinline__ void sts_p4_imm(uint32_t a, const P4 &v) {
    asm volatile("st.shared.v2.b64 [%0+%1], {%2, %3};" ::"r"(a), "n"(OFF), "l"(v.lo), "l"(v.hi) : "memory");
}
template <int OFF> __device__ __forceinline__ void mbar_wait_imm(uint32_t bar0, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WB_LWAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0+%1], %2, %3;\n"
        "@p bra WB_LDONE_%=;\n"
        "bra WB_LWAIT_%=;\n"
        "WB_LDONE_%=:\n"
        "}\n" ::"r"(bar0), "n"(OFF), "r"(parity), "r"(kMbarSuspendHintNs)
        : "memory");
}
template <int OFF> __device__ __forceinline__ void mbar_arrive_imm(uint32_t bar0) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0+%1];" ::"r"(bar0), "n"(OFF) : "memory");
}

// Row pass of one 16-byte vector from ring slot offset OFF; a[k] are the per-thread tap addresses in slot 0.
// SQUARE filters the squares of the staged values (the local power reads the raw w_s rows).  MIRROR (warp-uniform
// variant for warps that own border columns): a reflected tap is the mirrored vector read backwards -- a per-thread
// select, no branch.
template <int TAPS, int DMODE, int OFF, bool SQUARE, bool MIRROR, typename T>
__device__ __forceinline__ P4 lean_row_pass(const uint32_t (&a)[PlanSize<TAPS, DMODE>::NV], unsigned rev,
                                            const PackedTaps<TAPS, T> &H) {
    using L = Lane<T>;
    constexpr int C = TAPS / 2;
    constexpr int NV = PlanSize<TAPS, DMODE>::NV;
    P4 t[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        t[k] = lds_p4_imm<OFF>(a[k]);
        if constexpr (MIRROR) {
            const bool m = (rev >> k) & 1u;
            const P4 u = L::reverse(t[k]);
            t[k].lo = m ? u.lo : t[k].lo;
            t[k].hi = m ? u.hi : t[k].hi;
        }
        if constexpr (SQUARE) {
            t[k].lo = L::mul(t[k].lo, t[k].lo);
            t[k].hi = L::mul(t[k].hi, t[k].hi);
        }
    }
    P4 acc;
    if constexpr (DMODE == 0) {
#pragma unroll
        for (int k = 0; k < TAPS; ++k) {
            acc.lo = (k == 0) ? L::mul(H.h[0], t[k].lo) : L::fma(H.h[k], t[k].lo, acc.lo);
            acc.hi = (k == 0) ? L::mul(H.h[0], t[k].hi) : L::fma(H.h[k], t[k].hi, acc.hi);
        }
    } else if constexpr (sizeof(T) == 8) {
        // float64, d == 1: previous, current, next vector as six doubles; tap k of element e is win[2 + e + (k - C)]
        static_assert(DMODE == 1, "float64 vectors hold two elements: d == 1 is the only dilation below the vector width");
        const u64 win[6] = {t[0].lo, t[0].hi, t[1].lo, t[1].hi, t[2].lo, t[2].hi};
#pragma unroll
        for (int k = 0; k < TAPS; ++k) {
            const int i = 2 + (k - C);
            acc.lo = (k == 0) ? L::mul(H.h[0], win[i]) : L::fma(H.h[k], win[i], acc.lo);
            acc.hi = (k == 0) ? L::mul(H.h[0], win[i + 1]) : L::fma(H.h[k], win[i + 1], acc.hi);
        }
    } else if constexpr (DMODE == 2) {
        // d == 2: previous, current, next vector as six pixel pairs; every tap of a pair is again an aligned pair
        const u64 win[6] = {t[0].lo, t[0].hi, t[1].lo, t[1].hi, t[2].lo, t[2].hi};
#pragma unroll
        for (int k = 0; k < TAPS; ++k) {
            const int i = 2 + (k - C);
            acc.lo = (k == 0) ? mul2(H.h[0], win[i]) : fma2(H.h[k], win[i], acc.lo);
            acc.hi = (k == 0) ? mul2(H.h[0], win[i + 1]) : fma2(H.h[k], win[i + 1], acc.hi);
        }
    } else {
        // d == 1: taps of a pixel pair straddle register pairs -> scalar FMAs on the 12-element window
        float win[12];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            up2(t[k].lo, win[4 * k], win[4 * k + 1]);
            up2(t[k].hi, win[4 * k + 2], win[4 * k + 3]);
        }
        float o[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
#pragma unroll
            for (int k = 0; k < TAPS; ++k) {
                const float v = win[4 + e + (k - C)];
                o[e] = (k == 0) ? Taps<float, TAPS>::h(0) * v : fmaf(Taps<float, TAPS>::h(k), v, o[e]);
            }
        }
        acc.lo = pk2(o[0], o[1]);
        acc.hi = pk2(o[2], o[3]);
    }
    return acc;
}

// Row pass of a PAIR of vectors M dilation steps apart (columns x and x + M d, d % 4 == 0): their taps x + (k - C) d
// overlap in TAPS - M vectors, so TAPS + M LDS.128 (and squarings) serve two outputs instead of 2 TAPS -- the lean
// kernels are limited by shared-memory wavefronts and LDS latency before arithmetic.  Every output sums the same
// values in the same order as lean_row_pass: bit-identical planes.
template <int TAPS, int M, int OFF, bool SQUARE, bool MIRROR, typename T>
__device__ __forceinline__ void lean_row_pass_pair(const uint32_t (&a)[TAPS + M], unsigned rev, const PackedTaps<TAPS, T> &H,
                                                   P4 &o0, P4 &o1) {
    using L = Lane<T>;
    P4 t[TAPS + M];
#pragma unroll
    for (int k = 0; k < TAPS + M; ++k) {
        t[k] = lds_p4_imm<OFF>(a[k]);
        if constexpr (MIRROR) {
            const bool m = (rev >> k) & 1u;
            const P4 u = L::reverse(t[k]);
            t[k].lo = m ? u.lo : t[k].lo;
            t[k].hi = m ? u.hi : t[k].hi;
        }
        if constexpr (SQUARE) {
            t[k].lo = L::mul(t[k].lo, t[k].lo);
            t[k].hi = L::mul(t[k].hi, t[k].hi);
        }
    }
#pragma unroll
    for (int k = 0; k < TAPS; ++k) {
        o0.lo = (k == 0) ? L::mul(H.h[0], t[k].lo) : L::fma(H.h[k], t[k].lo, o0.lo);
        o0.hi = (k == 0) ? L::mul(H.h[0], t[k].hi) : L::fma(H.h[k], t[k].hi, o0.hi);
        o1.lo = (k == 0) ? L::mul(H.h[0], t[k + M].lo) : L::fma(H.h[k], t[k + M].lo, o1.lo);
        o1.hi = (k == 0) ? L::mul(H.h[0], t[k + M].hi) : L::fma(H.h[k], t[k + M].hi, o1.hi);
    }
}

// Thread -> first vector of its pair: runs of M dv consecutive vectors (dv = d / 4 vectors per dilation step) alternate
// between first and second halves of the pairs.  M dv >= 8, so eight consecutive lanes read eight consecutive vectors
// (conflict-free LDS.128) and a warp stores runs of >= 128 contiguous bytes.
__device__ __forceinline__ int pair_first_vector(int tid, int run) { return (tid / run) * 2 * run + (tid % run); }

// The TAPS + M tap addresses (slot 0; the staged row starts at column lo) of a pair whose first vector starts at
// column x0, with the symmetric border: returns the mirror bits.  V = elements per 16-byte vector.  Taps that belong
// only to a masked second vector may fall outside one reflection: clamped.
template <int TAPS, int M, int V = 4>
__device__ __forceinline__ unsigned make_pair_plan(int x0, int d, int W, int lo, uint32_t base, uint32_t (&a)[TAPS + M]) {
    constexpr int C = TAPS / 2;
    unsigned rv = 0;
#pragma unroll
    for (int k = 0; k < TAPS + M; ++k) {
        const int pc = x0 + (k - C) * d;
        const bool left = pc < 0, right = pc >= W;
        int q = left ? (-V - pc) : (right ? (2 * W - V - pc) : pc);
        if (q < lo || q > W - V) q = lo;
        a[k] = base + (uint32_t)(q - lo) * (uint32_t)(16 / V);
        if (left || right) rv |= 1u << k;
    }
    return rv;
}

template <int I> struct IC { static constexpr int value = I; };

// A value ptxas may not rematerialise: under register pressure it otherwise recomputes the reflected tap offsets
// from threadIdx inside the step loop (60 integer instructions per step) instead of holding them.
__device__ __forceinline__ uint32_t opaque_u32(uint32_t v) {
    uint32_t r;
    asm volatile("mov.u32 %0, %1;" : "=r"(r) : "r"(v));
    return r;
}

// ---------------------------------------------------------------------------------------------------------------
// Host: geometry planning
// ---------------------------------------------------------------------------------------------------------------
struct K1Config { int nt, ng, slots, seg; };

extern K1Config g_override[32];
extern bool g_override_set[32];

static constexpr int kMaxSmem = 227 * 1024;
static constexpr int kRegsPerThread = 64;  // budget assumed by the occupancy estimate of the planner

inline int device_sm_count() {
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
    }
    return sms;
}

inline int round_up(int a, int b) { return (a + b - 1) / b * b; }

inline bool fast_path_ok(const ScaleParams &p, int taps, int esize) {
    const int V = 16 / esize;
    const int c = taps / 2;
    if (p.W % V || p.W < 8 * V) return false;
    if ((long long)c * p.d > p.W) return false;  // more than one reflection in x
    if (p.in_pitch % V || p.in_bstride % V || !aligned16(p.in)) return false;
    if (p.out_c && (p.c_pitch % V || p.c_bstride % V || !aligned16(p.out_c))) return false;
    if (p.out_w && (p.w_pitch % V || p.w_bstride % V || !aligned16(p.out_w))) return false;
    // the map is read in the vectors of the output
    if (p.noise_map && (p.map_pitch % V || p.map_bstride % V || !aligned16(p.noise_map))) return false;
    // the vector path stores 16-byte vectors into the neighbours' buffers too (halo push)
    if ((p.push_up && !aligned16(p.push_up)) || (p.push_dn && !aligned16(p.push_dn))) return false;
    return true;
}

// Fill in the strip/segment/ring geometry.  Returns false if no geometry fits in shared memory.
inline bool plan_fast(ScaleParams &p, int taps, int esize, int batch, int scale, K1Config *cfg_out,
                      bool transform_op = true) {
    const int V = 16 / esize;
    const int c = taps / 2;
    K1Config cfg;
    if (scale < 32 && g_override_set[scale]) {
        cfg = g_override[scale];
    } else {
        cfg.ng = 2;
        const int vecs = (p.W + V - 1) / V;
        cfg.nt = round_up((vecs + cfg.ng - 1) / cfg.ng, 32);
        // a strip is at most 16 KiB of row data (4096 fp32 / 2048 fp64 columns)
        const int nt_cap = 16384 / (16 * cfg.ng);
        if (cfg.nt > nt_cap) cfg.nt = nt_cap;
        if (cfg.nt > 512) cfg.nt = 512;
        cfg.slots = 8;
        cfg.seg = 0;  // decided below
    }
    if (cfg.nt % 32 || cfg.nt < 32 || cfg.nt > 512 || (cfg.ng != 1 && cfg.ng != 2)) return false;
    p.wt = cfg.nt * V * cfg.ng;
    p.n_strips = (p.W + p.wt - 1) / p.wt;
    p.halo_al = round_up(c * p.d, V);
    long long rs = (long long)p.wt + 2LL * p.halo_al;
    if (rs > p.W) rs = p.W;
    p.row_stride = (int)rs;
    const int min_slots = c + 2;
    int slots = cfg.slots;
    while (slots > min_slots && (long long)slots * p.row_stride * esize + 16LL * slots > kMaxSmem) --slots;
    if ((long long)slots * p.row_stride * esize + 16LL * slots > kMaxSmem || slots < min_slots) return false;
    p.slots = slots;
    const int n_max = (p.H + p.d - 1) / p.d;  // longest chain
    int seg = cfg.seg;
    if (seg <= 0) {
        // One full wave: as many equal segments as there are block slots (SMs x resident blocks), so that no SM
        // idles in a partial last wave, but never shorter than the taps.
        const long long chains = (long long)p.n_strips * (p.d < p.H ? p.d : p.H) * batch;
        const size_t smem = (size_t)slots * p.row_stride * esize + 16 * (size_t)slots;
        int occ = (int)(kMaxSmem / (smem + 1024));
        const int occ_regs = 65536 / ((cfg.nt + 32) * kRegsPerThread);
        if (occ > occ_regs) occ = occ_regs;
        // the lean fp32 kernels (whole rows wider than 1024 columns, see dispatch in atrous_scale.cu) always stage 16 KiB
        // ring slots: one block per SM whatever the row width
        // -- except the cascade kernel on rows of <= 2048 columns, which has an 8 KiB-slot form (two blocks per SM)
        if (esize == 4 && p.n_strips == 1 && p.W > 1024 && cfg.ng == 2 && slots == 8)
            occ = (transform_op && p.W <= 2048 && p.l2_hints) ? 2 : 1;
        if (occ < 1) occ = 1;
        const long long slots_total = (long long)device_sm_count() * occ;
        long long per_chain = slots_total / chains;  // segments per chain that still fit in one wave
        if (per_chain < 1) per_chain = 1;
        seg = (int)((n_max + per_chain - 1) / per_chain);
        // (never shorter than the taps; small frames are bound by the number of steps per block, not by the halo bytes)
        if (seg < 2 * c) seg = 2 * c;
    }
    if (seg > n_max) seg = n_max;
    p.seg = seg;
    p.n_seg = (n_max + seg - 1) / seg;
    cfg.slots = slots;
    cfg.seg = seg;
    if (cfg_out) *cfg_out = cfg;
    return true;
}


}  // namespace wb
