// K1+K3 fused -- one WOW scale in ONE pass over HBM: c_{s+1} = S_s[c_s], w_s = c_s - c_{s+1},
// P = S_s[w_s^2], w'_s = w_s * significance(w_s) * (weight / sqrt(max(P, 1e-15))).
//
// Replaces, per scale, watroo/wavelets.py:35-45 + :442 (smooth + subtraction) AND the loop body of
// watroo/utils.py:177,193-203 (power = c**2, convolution(power), clamp, sqrt, significance, weighting).  The raw detail
// plane w_s never reaches HBM: 3*sizeof(T) bytes per pixel per scale (read c_s, write c_{s+1}, write w'_s) instead of
// the 5*sizeof(T) of K1 followed by K3.
//
// Same chain walk as K1 (see atrous_scale.cu): the local power uses the SAME dilation as the smooth, so it only couples
// rows of the same chain.  A thread block (512 threads, every one a consumer, NG = 2 column vectors per thread; thread
// 0 also issues the TMA row loads) walks a chain segment once; per step j
//   A  input row j lands (TMA, mbarrier) -> row pass -> running column sums in registers -> c_{s+1} of row j-C:
//      128-bit store (rows of the segment only); w_s = raw - c_{s+1} goes to a shared-memory ring (other threads need
//      it for the x taps of the power filter); one mbarrier arrival per warp;
//   B  (one step later) wait on that mbarrier -- a SPLIT-PHASE barrier: warps drift by a step instead of marching in
//      lock-step -> row pass over the squares of the w row -> second set of running sums -> P; epilogue with the raw
//      w_s of the centre row (same ring) -> streaming 128-bit store of w'_s.  The same barrier completion tells thread
//      0 which input slot is free for the next TMA load.
// Two kernels implement it: wow_rows_kernel (any dtype / width up to one 16 KiB row; keeps a separate w^2 ring and a
// third phase C) and wow_rows_lean_kernel (fp32 rows of 513 .. 4096 columns: unrolled ring, immediate addressing,
// packed fp32x2, squares on the fly -- see the comment above it).
// Rows outside the image are symmetric reflections: the loader fetches the reflected rows; because the symmetric
// extension commutes with the symmetric smooth, c_{s+1} / w_s evaluated at such a virtual row equal their reflected
// values (up to the rounding of a reversed summation order), which is what the power filter needs at the border.
// The strip is normally the whole row, so the x border is an index reflection inside the staged row for both row
// passes (same tap plan); wow_rows_kernel can also walk column strips (see plan_wow).  Away from the top/bottom border the arithmetic is exactly K1 followed by K3.
#include "pipeline.cuh"
#include "whiten.cuh"

namespace wb {

static constexpr int kInRing = 8;  // input rows staged by TMA (C+1 live, the rest prefetch)
static constexpr int kWRing = 4;   // raw w_s rows (read back by the writing thread C+1 steps later)
static constexpr int kW2Ring = 2;  // w_s^2 rows (cross-thread, guarded by the split-phase barriers)

template <typename T, int TAPS, int DMODE, int NG, bool HINTS>
__global__ void __launch_bounds__(512, 1) wow_rows_kernel(const ScaleParams p) {
    constexpr int V = VecOf<T>::V;
    constexpr int C = TAPS / 2;
    constexpr int NV = PlanSize<TAPS, DMODE>::NV;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const uint32_t RB = (uint32_t)p.row_stride * (uint32_t)sizeof(T);  // bytes per staged row
    const uint32_t in_base = smem_u32(smem_raw);                       // kInRing rows of c_s (TMA)
    const uint32_t w_base = in_base + (uint32_t)kInRing * RB;           // kWRing rows of raw w_s
    const uint32_t w2_base = w_base + (uint32_t)kWRing * RB;            // kW2Ring rows of w_s^2
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw + (size_t)(kInRing + kWRing + kW2Ring) * RB);
    uint64_t *wbar = full + kInRing;  // split-phase "w / w^2 row complete" barriers, one arrival per warp

    pdl_launch_dependents();
    const int tid = threadIdx.x;
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
    const int n_load = n_out + 4 * C;  // input rows i0-2C .. i0+n_out+2C-1 of the chain (virtual rows are reflected)
    // Column strip [x0, x1) of the outputs (whole row: one strip, halo_al = 0).  The power filter needs w_s on
    // [e_lo, e_hi) = strip +- C d, which needs c_s on [lo, hi) = strip +- 2 C d: the block stages [lo, hi), every thread
    // owns columns of [e_lo, e_hi) for BOTH passes, and only the columns inside the strip are stored (the halo
    // columns' power sums read ring positions nobody wrote; they are never stored).
    const int x0 = strip * p.wt;
    const int x1 = min(p.W, x0 + p.wt);
    const int e_lo = max(0, x0 - p.halo_al), e_hi = min(p.W, x1 + p.halo_al);
    const int lo = max(0, x0 - 2 * p.halo_al), hi = min(p.W, x1 + 2 * p.halo_al);
    const uint32_t row_bytes = (uint32_t)(hi - lo) * (uint32_t)sizeof(T);
    const T *src = reinterpret_cast<const T *>(p.in) + (long long)frame * p.in_bstride + lo;
    const long long y_first = (long long)r + (long long)(i0 - 2 * C) * p.d;  // image row of input row 0

    const uint64_t pol_in = policy_evict_first();   // c_s is dead once this launch has read it
    const uint64_t pol_keep = policy_evict_last();  // c_{s+1}: the next scale reads it back
    constexpr bool hints = HINTS, hints_c = HINTS;
    int next_load = 0;  // thread 0: next chain row to request
    pdl_wait();  // everything below touches global memory written or read by the previous launch
    if (tid == 0) {
        for (int s = 0; s < kInRing; ++s) mbar_init(&full[s], 1);
        for (int s = 0; s < kW2Ring; ++s) mbar_init(&wbar[s], blockDim.x >> 5);
        fence_mbar_init();
        const int n0 = min(kInRing, n_load);
        for (; next_load < n0; ++next_load) {
            const long long y = reflect_any(y_first + (long long)next_load * p.d, p.H);
            mbar_arrive_expect_tx(&full[next_load], row_bytes);
            if (hints) tma_load_1d_hint(smem_raw + (size_t)next_load * RB, src + y * p.in_pitch, row_bytes, &full[next_load], pol_in);
            else tma_load_1d(smem_raw + (size_t)next_load * RB, src + y * p.in_pitch, row_bytes, &full[next_load]);
        }
    }
    __syncthreads();

    WhitenEpilogue<T> epi;
    epi.init(p, frame);

    uint32_t xb[NG];  // byte offset of this thread's own vector inside a staged row
    int xg[NG];
    bool act[NG], outm[NG];  // act: the vector exists (shared-memory stores); outm: it lies inside the strip (global stores)
    BytePlan<NV> plan[NG];
#pragma unroll
    for (int q = 0; q < NG; ++q) {
        xg[q] = e_lo + (q * (int)blockDim.x + tid) * V;
        act[q] = xg[q] < e_hi;
        if (!act[q]) xg[q] = e_lo;  // idle threads shadow the first vector; only their stores are masked
        outm[q] = act[q] && xg[q] >= x0 && xg[q] < x1;
        xb[q] = (uint32_t)(xg[q] - lo) * (uint32_t)sizeof(T);
        const TapPlan<NV> tp = make_tap_plan<V, NV>(xg[q], DMODE == 0 ? p.d : V, p.W, lo);
#pragma unroll
        for (int k = 0; k < NV; ++k) plan[q].off[k] = (uint32_t)tp.off[k] * (uint32_t)sizeof(T);
        plan[q].rev = tp.rev;
    }

    T SA[NG][V][TAPS - 1], SB[NG][V][TAPS - 1];  // running column sums of the smooth and of the power filter
#pragma unroll
    for (int q = 0; q < NG; ++q)
#pragma unroll
        for (int e = 0; e < V; ++e)
#pragma unroll
            for (int t = 0; t < TAPS - 1; ++t) { SA[q][e][t] = T(0); SB[q][e][t] = T(0); }

    T *c_ptr = reinterpret_cast<T *>(p.out_c) + (long long)frame * p.c_bstride +
               ((long long)r + (long long)(i0 - C) * p.d) * p.c_pitch;  // row of the first c produced (part C)
    T *o_ptr = reinterpret_cast<T *>(p.out_w) + (long long)frame * p.w_bstride +
               ((long long)r + (long long)i0 * p.d) * p.w_pitch;        // row of the first output
    const long long c_step = (long long)p.d * p.c_pitch, o_step = (long long)p.d * p.w_pitch;

    // Step j: A  input row j lands -> row pass -> column feed (c of the row C steps back)
    //         B  [for the w^2 row written during step j-1] row pass -> column feed -> P, epilogue, store w'
    //         C  c row m = j-2C: store, w = raw - c and w^2 -> shared rings, arrive on wbar
    // One extra drain step (j == n_load) runs part B only.  All ring slots are j-derived with power-of-two rings.
    for (int j = 0; j <= n_load; ++j) {
        Pack<T, V> cv[NG];
        if (j < n_load) {
            mbar_wait(&full[j & (kInRing - 1)], (uint32_t)(j / kInRing) & 1u);
            const uint32_t row = in_base + (uint32_t)(j & (kInRing - 1)) * RB;
#pragma unroll
            for (int q = 0; q < NG; ++q) {
                const Pack<T, V> v = row_pass_b<T, TAPS, DMODE, false>(row, plan[q]);
#pragma unroll
                for (int e = 0; e < V; ++e) cv[q].v[e] = col_feed<T, TAPS>(SA[q][e], v.v[e]);
            }
        }
        if (j > 2 * C) {
            const int mb = j - 1 - 2 * C;  // count index of the w row handled here (written during step j-1)
            mbar_wait(&wbar[mb & (kW2Ring - 1)], (uint32_t)(mb / kW2Ring) & 1u);
            if (tid == 0) {
                // every warp is past part C of step j-1: input rows <= j-1-C are free
                while (next_load < n_load && next_load - kInRing <= j - 1 - C) {
                    const int sl = next_load & (kInRing - 1);
                    const long long y = reflect_any(y_first + (long long)next_load * p.d, p.H);
                    mbar_arrive_expect_tx(&full[sl], row_bytes);
                    if (hints) tma_load_1d_hint(smem_raw + (size_t)sl * RB, src + y * p.in_pitch, row_bytes, &full[sl], pol_in);
                    else tma_load_1d(smem_raw + (size_t)sl * RB, src + y * p.in_pitch, row_bytes, &full[sl]);
                    ++next_load;
                }
            }
            const uint32_t row = w2_base + (uint32_t)(mb & (kW2Ring - 1)) * RB;
            Pack<T, V> pw[NG];
#pragma unroll
            for (int q = 0; q < NG; ++q) {
                const Pack<T, V> v = row_pass_b<T, TAPS, DMODE, false>(row, plan[q]);
#pragma unroll
                for (int e = 0; e < V; ++e) pw[q].v[e] = col_feed<T, TAPS>(SB[q][e], v.v[e]);
            }
            if (j > 4 * C) {
                // P row i = j-1-4C (relative to i0); its raw w row has count index i + C
                const uint32_t wrow = w_base + (uint32_t)((j - 1 - 3 * C) & (kWRing - 1)) * RB;
#pragma unroll
                for (int q = 0; q < NG; ++q) {
                    Pack<T, V> raw = lds_vec<T>(wrow + xb[q]);
#pragma unroll
                    for (int e = 0; e < V; ++e) raw.v[e] = epi.apply(raw.v[e], pw[q].v[e]);
                    if (outm[q]) st_vec_cs(o_ptr + xg[q], raw);
                }
                o_ptr += o_step;
            }
        }
        if (j >= 2 * C && j < n_load) {
            const int mc = j - 2 * C;                       // count index of this c / w row
            const bool store_c = (mc >= C) && (mc - C < n_out);  // chain index relative to i0 is mc - C
            const uint32_t crow = in_base + (uint32_t)((j - C) & (kInRing - 1)) * RB;
            const uint32_t wrow = w_base + (uint32_t)(mc & (kWRing - 1)) * RB;
            const uint32_t w2row = w2_base + (uint32_t)(mc & (kW2Ring - 1)) * RB;
#pragma unroll
            for (int q = 0; q < NG; ++q) {
                if (store_c && outm[q]) {
                    if (hints_c) st_vec_hint(c_ptr + xg[q], cv[q], pol_keep);
                    else st_vec(c_ptr + xg[q], cv[q]);
                }
                Pack<T, V> raw = lds_vec<T>(crow + xb[q]);
                Pack<T, V> sq;
#pragma unroll
                for (int e = 0; e < V; ++e) {
                    raw.v[e] -= cv[q].v[e];
                    sq.v[e] = raw.v[e] * raw.v[e];
                }
                if (act[q]) {
                    sts_vec(wrow + xb[q], raw);
                    sts_vec(w2row + xb[q], sq);
                }
            }
            c_ptr += c_step;
            __syncwarp();
            if (lane == 0) mbar_arrive(&wbar[mc & (kW2Ring - 1)]);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// fp32 fast path: the same pipeline, LEAN.  ncu on the kernel above (4096^2, scale 3): 37-47 M warp instructions per
// plane of which only ~110 of 580 per warp-step are floating point -- the rest is ring-index arithmetic, tap offsets
// rematerialised under register pressure, loop conditionals, a 64-bit modulo in the loader (warp 0 becomes the
// straggler every step, 32 polls of the row barrier per step in every other warp) and barrier polling; TMA never
// waits.  This version removes the overhead instead of the arithmetic:
//   * the step loop is unrolled by 8 (= the input ring; the w / w^2 rings divide it) and ring slots have a fixed
//     16 KiB stride, so every shared-memory access is [per-thread register + immediate] -- no index arithmetic;
//   * pixel pairs are carried as 64-bit register pairs (FFMA2 / FMUL2 / FADD2: two IEEE fp32 operations per issue
//     slot, same roundings as the scalar instructions) from LDS.128 to STG.128;
//   * the loader walks the reflected row index incrementally (no division);
//   * output pointers are per-thread and advance by one add per row; the second column vector is +8 KiB.
// Operation order and roundings are those of wow_rows_kernel: the planes are bit-identical.
// ---------------------------------------------------------------------------------------------------------------
// MODE: significance compiled into the epilogue (0 none, 1 soft, 2 hard); the step loop is small enough to stay in
// the instruction cache only without the inlined erff of the modes that are not used.
// PAIR = M > 0 (DMODE 0, d >= 8): a thread's two column vectors are M dilation steps apart (x and x + M d) instead of
// half a row apart, so both row passes load TAPS + M tap vectors for the two of them instead of 2 TAPS
// (lean_row_pass_pair): with M = 1 (d >= 32) 18 instead of 26 LDS/STS.128 per thread and step; M = 2 for d = 16 (20), M = 4
// for d = 8 (24) keep eight consecutive lanes on eight consecutive vectors (see pair_first_vector).
// DYN: the step loop is NOT unrolled -- ring slots and barrier parities are computed from the step index (warp-uniform
// values: one more address term per shared-memory access) and the kernel is a quarter of the code.  The unrolled
// kernel (60 - 90 KB) does not fit the instruction cache levels below L2, and every change of kernel inside a cascade
// starts cold (see atrous_rows_lean_kernel).
// NTK: threads per block = half the vectors of the widest row the instantiation takes -- 512 (rows of 2049 .. 4096
// columns, 16 KiB ring slots, one block per SM) or 256 (513 .. 2048 columns, 8 KiB slots, two blocks per SM).
template <int TAPS, int DMODE, bool HINTS, int MODE, int PAIR = 0, bool DYN = false, int NTK = 512>
__global__ void __launch_bounds__(NTK, NTK == 512 ? 1 : 2) wow_rows_lean_kernel(const ScaleParams p) {
    static_assert(PAIR == 0 || (DMODE == 0 && PAIR < TAPS), "paired columns need d % 4 == 0 and overlapping taps");
    static_assert(NTK == 512 || NTK == 256, "block sizes the ring geometry was laid out for");
    using T = float;
    constexpr int V = 4, NG = 2, NT = NTK;
    constexpr int C = TAPS / 2;
    constexpr int NV = PlanSize<TAPS, DMODE>::NV;
    constexpr int RB = NT * NG * V * (int)sizeof(T);  // bytes per ring slot: one row of the widest frame the block takes
    constexpr int W_OFF = kInRing * RB;  // the w ring follows the input ring
    constexpr int BSH = (RB == 16384) ? 11 : 10;  // slot byte offset >> BSH = byte offset of the slot's 8-byte barrier
    static_assert(kInRing == 8 && kWRing == 4, "the step loop is unrolled by the w ring; the input ring is twice that");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const uint32_t in_base = smem_u32(smem_raw);
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw + (size_t)(kInRing + kWRing) * RB);
    uint64_t *wbar = full + kInRing;  // "raw w row complete" barriers (one per w slot), one arrival per warp
    const uint32_t full0 = smem_u32(full), wbar0 = smem_u32(wbar);

    pdl_launch_dependents();
    const int tid = threadIdx.x;
    const int lane = tid & 31;

    int bx = blockIdx.x;
    const int r = bx % p.d;
    const int g = bx / p.d;
    const int frame = blockIdx.y;

    const int n_chain = (r < p.H) ? (p.H - r + p.d - 1) / p.d : 0;
    const int i0 = g * p.seg;
    const int n_out = min(p.seg, n_chain - i0);
    if (n_out <= 0) return;
    const int n_load = n_out + 4 * C;  // input rows i0-2C .. i0+n_out+2C-1 of the chain (virtual rows are reflected)
    const uint32_t row_bytes = (uint32_t)p.W * (uint32_t)sizeof(T);
    const T *src = reinterpret_cast<const T *>(p.in) + (long long)frame * p.in_bstride;

    // loader state (thread 0): position of the next row in the 2H-periodic symmetric extension, walked incrementally
    const uint64_t pol_in = policy_evict_first();
    const uint64_t pol_keep = policy_evict_last();
    int next_load = 0;
    const int period = 2 * p.H;
    const int d_mod = p.d % period;
    int m_pos = 0;
    auto issue_load = [&]() {
        const int y = m_pos < p.H ? m_pos : period - 1 - m_pos;
        const int sl = next_load & (kInRing - 1);
        mbar_arrive_expect_tx(&full[sl], row_bytes);
        if (HINTS) tma_load_1d_hint(smem_raw + (size_t)sl * RB, src + (long long)y * p.in_pitch, row_bytes, &full[sl], pol_in);
        else tma_load_1d(smem_raw + (size_t)sl * RB, src + (long long)y * p.in_pitch, row_bytes, &full[sl]);
        ++next_load;
        m_pos += d_mod;
        if (m_pos >= period) m_pos -= period;
    };
    pdl_wait();  // everything below touches global memory written or read by the previous launch
    if (tid == 0) {
        for (int s = 0; s < kInRing; ++s) mbar_init(&full[s], 1);
        for (int s = 0; s < kWRing; ++s) mbar_init(&wbar[s], NT >> 5);
        fence_mbar_init();
        long long m0 = ((long long)r + (long long)(i0 - 2 * C) * p.d) % period;
        if (m0 < 0) m0 += period;
        m_pos = (int)m0;
        const int n0 = min(kInRing, n_load);
        while (next_load < n0) issue_load();
    }
    __syncthreads();

    WhitenEpilogue<T> epi;
    epi.init(p, frame);
    const PackedTaps<TAPS> H;

    // per-thread addresses inside ring slot 0: own vector and taps, for both column groups
    constexpr int NTAP = PAIR ? 1 : NG, NPT = TAPS + PAIR;
    uint32_t own[NG], tap[NTAP][NV], ptap[NPT];
    unsigned rev[NG] = {0u, 0u};
    bool act[NG];
    int xg0 = 0;
    // interior warps: tap k of a vector is its own address + (k - NV/2) * step bytes (nothing to hold per tap)
    const uint32_t tap_step = (uint32_t)(DMODE == 0 ? p.d : V) * (uint32_t)sizeof(T);
    bool mirror_warp;
    if constexpr (PAIR) {
        const int run = PAIR * (p.d >> 2), nvec = p.W >> 2;  // vectors between the two of a pair (>= 8), vectors per row
        const int v0 = pair_first_vector(tid, run);
        act[0] = v0 < nvec;
        act[1] = v0 + run < nvec;
        xg0 = act[0] ? v0 * V : 0;  // idle threads shadow the first pair of the row; only their stores are masked
        own[0] = opaque_u32(in_base + (uint32_t)xg0 * (uint32_t)sizeof(T));
        own[1] = opaque_u32(act[1] ? own[0] + PAIR * tap_step : own[0]);
        const unsigned rv = make_pair_plan<TAPS, PAIR>(xg0, p.d, p.W, 0, in_base, ptap);
        rev[0] = rv;
        mirror_warp = __any_sync(0xffffffffu, rv != 0 || !act[0]);
        if (mirror_warp) {
#pragma unroll
            for (int k = 0; k < TAPS + PAIR; ++k) ptap[k] = opaque_u32(ptap[k]);
            rev[0] = opaque_u32(rev[0]);
        }
    } else {
#pragma unroll
        for (int q = 0; q < NG; ++q) {
            int xg = (q * NT + tid) * V;
            act[q] = xg < p.W;
            // idle threads shadow a vector in the middle of the row (interior unless the dilation is huge); only their
            // stores are masked
            if (!act[q]) xg = (p.W / 2) & ~(V - 1);
            if (q == 0) xg0 = xg;
            own[q] = opaque_u32(in_base + (uint32_t)xg * (uint32_t)sizeof(T));
            const TapPlan<NV> tp = make_tap_plan<V, NV>(xg, DMODE == 0 ? p.d : V, p.W, 0);
#pragma unroll
            for (int k = 0; k < NV; ++k) tap[q][k] = in_base + (uint32_t)tp.off[k] * (uint32_t)sizeof(T);
            rev[q] = tp.rev;
        }
        mirror_warp = __any_sync(0xffffffffu, (rev[0] | rev[1]) != 0);
        if (mirror_warp) {
#pragma unroll
            for (int q = 0; q < NG; ++q) {
#pragma unroll
                for (int k = 0; k < NV; ++k) tap[q][k] = opaque_u32(tap[q][k]);
                rev[q] = opaque_u32(rev[q]);
            }
        }
    }
    // the second column vector of a thread: one dilation step (PAIR) or half a ring slot (NT vectors) further
    auto q_off = [&](int q) -> long long {
        if constexpr (PAIR) return q ? (long long)PAIR * p.d : 0LL;
        else return (long long)q * (NT * V);
    };

    u64 SA[NG][2][TAPS - 1], SB[NG][2][TAPS - 1];  // running column sums, one pixel pair per entry
#pragma unroll
    for (int q = 0; q < NG; ++q)
#pragma unroll
        for (int e = 0; e < 2; ++e)
#pragma unroll
            for (int t = 0; t < TAPS - 1; ++t) { SA[q][e][t] = 0ull; SB[q][e][t] = 0ull; }

    // per-thread output pointers (column group 0; group 1 is NT * V elements further when active)
    T *c_ptr = reinterpret_cast<T *>(p.out_c) + (long long)frame * p.c_bstride +
               ((long long)r + (long long)(i0 - C) * p.d) * p.c_pitch + xg0;
    T *o_ptr = reinterpret_cast<T *>(p.out_w) + (long long)frame * p.w_bstride +
               ((long long)r + (long long)i0 * p.d) * p.w_pitch + xg0;
    const long long c_step = (long long)p.d * p.c_pitch, o_step = (long long)p.d * p.w_pitch;
    const int j_store_end = 3 * C + n_out;

    // Step j = 4 u + I (input slot = I + 4 (u & 1): `half` is that slot's byte offset, 0 or 4 RB):
    //   A  input row j lands -> row pass -> column feed -> c row j-C: store (rows of the segment), w = raw - c into the
    //      w ring, arrive on that row's barrier;
    //   B  wait until every warp has written w row j-1-2C -> row pass over its squares -> column feed -> P of row
    //      j-1-3C, epilogue with this thread's own raw w of that row -> streaming store.
    // One drain step (j == n_load) runs part B only.  A slot of the w ring is rewritten 4 steps after it was filled;
    // its cross-thread readers finished 3 steps earlier (no warp is more than one step behind a passed barrier).
    auto step = [&](auto ic, auto mirror, const int j, const uint32_t half, const uint32_t half_c, const uint32_t par_in) {
        constexpr int I = decltype(ic)::value;
        constexpr bool MIRROR = decltype(mirror)::value != 0;
        if (j > n_load) return;
        // ring slots touched by this step, as [dynamic byte offset] + immediate: unrolled loop -> the immediates carry the
        // slot and only the input ring has a dynamic part (its half); DYN -> everything from j, immediates 0
        constexpr int SCs = (I - C + 4) & 3;                             // raw centre row j-C (input ring)
        constexpr bool other_half = I < C;
        constexpr int SWs = (I - 2 * C + 8) & (kWRing - 1);              // w row j-2C, written by part A
        constexpr int SPs = (I - 1 - 2 * C + 16) & (kWRing - 1);         // w row j-1-2C (all threads' columns), part B
        constexpr int SEs = (I - 1 - 3 * C + 16) & (kWRing - 1);         // own raw w of the P row completed in this step
        constexpr int IMM_IN = DYN ? 0 : I * RB, IMM_C = DYN ? 0 : SCs * RB, IMM_SW = DYN ? 0 : SWs * RB;
        constexpr int IMM_SP = DYN ? 0 : SPs * RB, IMM_SE = DYN ? 0 : SEs * RB;
        const uint32_t o_in = DYN ? ((uint32_t)j & (kInRing - 1)) * RB : half;
        const uint32_t o_c = DYN ? ((uint32_t)(j - C) & (kInRing - 1)) * RB : (other_half ? half_c : half);
        const uint32_t o_sw = DYN ? ((uint32_t)(j - 2 * C) & (kWRing - 1)) * RB : 0u;
        const uint32_t o_sp = DYN ? ((uint32_t)(j - 1 - 2 * C) & (kWRing - 1)) * RB : 0u;
        const uint32_t o_se = DYN ? ((uint32_t)(j - 1 - 3 * C) & (kWRing - 1)) * RB : 0u;
        if (j < n_load) {
            // barrier of the input slot: 8 bytes per 16 KiB slot
            mbar_wait_imm<IMM_IN / RB * 8>(full0 + (o_in >> BSH), DYN ? ((uint32_t)j >> 3) & 1u : par_in);
            // raw centre row j-C, requested first so that its latency hides behind the row pass
            P4 rawc[NG];
#pragma unroll
            for (int q = 0; q < NG; ++q) rawc[q] = lds_p4_imm<IMM_C>(own[q] + o_c);
            P4 cv[NG];
            if constexpr (PAIR) {
                uint32_t a[TAPS + PAIR];
#pragma unroll
                for (int k = 0; k < TAPS + PAIR; ++k) a[k] = (MIRROR ? ptap[k] : own[0] + (uint32_t)(k - C) * tap_step) + o_in;
                P4 v[NG];
                lean_row_pass_pair<TAPS, PAIR, IMM_IN, false, MIRROR>(a, rev[0], H, v[0], v[1]);
#pragma unroll
                for (int q = 0; q < NG; ++q) {
                    cv[q].lo = col_feed_p<TAPS>(SA[q][0], v[q].lo, H);
                    cv[q].hi = col_feed_p<TAPS>(SA[q][1], v[q].hi, H);
                }
            } else {
#pragma unroll
                for (int q = 0; q < NG; ++q) {
                    uint32_t a[NV];
#pragma unroll
                    for (int k = 0; k < NV; ++k)
                        a[k] = (MIRROR ? tap[q][k] : own[q] + (uint32_t)(k - NV / 2) * tap_step) + o_in;
                    const P4 v = lean_row_pass<TAPS, DMODE, IMM_IN, false, MIRROR>(a, rev[q], H);
                    cv[q].lo = col_feed_p<TAPS>(SA[q][0], v.lo, H);
                    cv[q].hi = col_feed_p<TAPS>(SA[q][1], v.hi, H);
                }
            }
            if (j >= 2 * C) {
                const bool store_c = (j >= 3 * C) && (j < j_store_end);
#pragma unroll
                for (int q = 0; q < NG; ++q) {
                    if (store_c && act[q]) {
                        if (HINTS) stg_p4_hint(c_ptr + q_off(q), cv[q], pol_keep);
                        else stg_p4(c_ptr + q_off(q), cv[q]);
                    }
                    P4 raw = rawc[q];
                    raw.lo = sub2(raw.lo, cv[q].lo);
                    raw.hi = sub2(raw.hi, cv[q].hi);
                    if (act[q]) sts_p4_imm<W_OFF + IMM_SW>(own[q] + o_sw, raw);
                }
                c_ptr += c_step;
                __syncwarp();
                if (lane == 0) mbar_arrive_imm<IMM_SW / RB * 8>(wbar0 + (o_sw >> BSH));
            }
        }
        if (j > 2 * C) {
            mbar_wait_imm<IMM_SP / RB * 8>(wbar0 + (o_sp >> BSH), ((uint32_t)(j - 1 - 2 * C) >> 2) & 1u);
            if (tid == 0) {
                // every warp is past part A of step j-1: input rows <= j-1-C are free
                while (next_load < n_load && next_load - kInRing <= j - 1 - C) issue_load();
            }
            P4 roww[NG];
#pragma unroll
            for (int q = 0; q < NG; ++q) roww[q] = lds_p4_imm<W_OFF + IMM_SE>(own[q] + o_se);
            P4 pw[NG];
            if constexpr (PAIR) {
                uint32_t a[TAPS + PAIR];
#pragma unroll
                for (int k = 0; k < TAPS + PAIR; ++k) a[k] = (MIRROR ? ptap[k] : own[0] + (uint32_t)(k - C) * tap_step) + o_sp;
                P4 v[NG];
                lean_row_pass_pair<TAPS, PAIR, W_OFF + IMM_SP, true, MIRROR>(a, rev[0], H, v[0], v[1]);
#pragma unroll
                for (int q = 0; q < NG; ++q) {
                    pw[q].lo = col_feed_p<TAPS>(SB[q][0], v[q].lo, H);
                    pw[q].hi = col_feed_p<TAPS>(SB[q][1], v[q].hi, H);
                }
            } else {
#pragma unroll
                for (int q = 0; q < NG; ++q) {
                    uint32_t a[NV];
#pragma unroll
                    for (int k = 0; k < NV; ++k)
                        a[k] = (MIRROR ? tap[q][k] : own[q] + (uint32_t)(k - NV / 2) * tap_step) + o_sp;
                    const P4 v = lean_row_pass<TAPS, DMODE, W_OFF + IMM_SP, true, MIRROR>(a, rev[q], H);
                    pw[q].lo = col_feed_p<TAPS>(SB[q][0], v.lo, H);
                    pw[q].hi = col_feed_p<TAPS>(SB[q][1], v.hi, H);
                }
            }
            if (j > 4 * C) {
#pragma unroll
                for (int q = 0; q < NG; ++q) {
                    P4 raw = roww[q];
                    raw.lo = epi.template apply2<MODE>(raw.lo, pw[q].lo);
                    raw.hi = epi.template apply2<MODE>(raw.hi, pw[q].hi);
                    if (act[q]) stg_p4_cs(o_ptr + q_off(q), raw);
                }
                o_ptr += o_step;
            }
        }
    };
    auto run = [&](auto mirror) {
        if constexpr (DYN) {
#pragma unroll 1
            for (int j = 0; j <= n_load; ++j) step(IC<0>{}, mirror, j, 0u, 0u, 0u);
            return;
        }
#pragma unroll 1
        for (int jb = 0; jb <= n_load; jb += 4) {
            const uint32_t half = (jb & 4) ? 4u * RB : 0u;   // input slots 4..7 on odd iterations
            const uint32_t half_c = half ^ (4u * RB);        // the half loaded one iteration earlier
            const uint32_t par_in = (uint32_t)(jb >> 3) & 1u;
            step(IC<0>{}, mirror, jb + 0, half, half_c, par_in);
            step(IC<1>{}, mirror, jb + 1, half, half_c, par_in);
            step(IC<2>{}, mirror, jb + 2, half, half_c, par_in);
            step(IC<3>{}, mirror, jb + 3, half, half_c, par_in);
        }
    };
    // warps that own no border column (the vast majority at shallow scales) run the variant without the selects
    if (mirror_warp) run(IC<1>{});
    else run(IC<0>{});
}

// ---------------------------------------------------------------------------------------------------------------
// Host
// ---------------------------------------------------------------------------------------------------------------
struct WowGeom { int nt, ng; size_t smem; };

// narrowest rows the 256-thread lean kernel takes (below that most of its threads would idle; the generic kernel sizes its
// blocks to the row)
static constexpr int kLean256MinW = 512;

// WB_WOW_STRIPS=k in the environment forces k column strips (>= 2) where the whole row would fit (A/B measurements).
static int wow_forced_strips() {
    const char *e = getenv("WB_WOW_STRIPS");
    return e ? atoi(e) : 0;
}

static bool plan_wow(ScaleParams &p, int taps, int esize, int batch, WowGeom *geo) {
    const int V = 16 / esize;
    const int c = taps / 2;
    if (!fast_path_ok(p, taps, esize)) return false;
    if (!p.out_c || !p.out_w) return false;
    const int ng = 2;
    const int rows = kInRing + kWRing + kW2Ring;
    const int forced = wow_forced_strips();
    int nt = 0;
    size_t smem = 0;
    // Whole-row strips when the row fits 512 threads x 2 vectors (W <= 4096 fp32 / 2048 fp64).  The kernel also runs
    // COLUMN strips (WB_WOW_STRIPS=k: the fewest >= k strips whose staged range, strip + 4 C d columns, fits the 14-row
    // ring and whose extended range, strip + 2 C d, fits the block), built for float64 rows of 4096 columns -- and
    // measured SLOWER than the two-pass route there (4096^2 float64: 142 - 229 us per scale against 75 + 60 us for K1 +
    // K3, profiles/r2_bench_wow_f64_v2.json: this generic kernel is bound by instruction issue, not by the bytes the
    // fusion saves), so wider rows are declined (WB_ENOT_FUSABLE -> two passes) unless the variable forces strips.
    const int halo = round_up(c * p.d, V);
    int k_strips = 0;
    for (int k = (forced >= 2 ? forced : 1); k <= 64; ++k) {
        const int wt = (k == 1) ? p.W : round_up((p.W + k - 1) / k, V);
        const int h = (k == 1) ? 0 : halo;
        long long stage = (long long)wt + 4LL * h, ext = (long long)wt + 2LL * h;
        if (stage > p.W) stage = p.W;
        if (ext > p.W) ext = p.W;
        const int need = round_up((int)((ext / V + ng - 1) / ng), 32);
        const size_t sm = (size_t)rows * (size_t)stage * esize + 8 * (size_t)(kInRing + kW2Ring);
        if (k > 1 && forced < 2) break;  // see the note above: strips are not chosen automatically
        if (k > 1 && (2 * h > wt || 5 * ext > 8 * (long long)wt)) break;  // halo too wide: more than 1.6 x the columns
        if (need <= 512 && sm <= (size_t)kMaxSmem) {
            k_strips = k;
            p.wt = wt;
            p.halo_al = h;
            p.row_stride = (int)stage;
            nt = need;
            smem = sm;
            break;
        }
    }
    if (!k_strips) return false;
    p.n_strips = (p.W + p.wt - 1) / p.wt;
    p.slots = kInRing;
    const int n_max = (p.H + p.d - 1) / p.d;
    const long long chains = (long long)p.n_strips * (p.d < p.H ? p.d : p.H) * batch;
    int occ = (int)(kMaxSmem / (smem + 1024));
    const int occ_regs = 65536 / (nt * 128);
    if (occ > occ_regs) occ = occ_regs;
    // the 256-thread lean kernel (fp32 rows of 513 .. 2048 columns, see launch_wow_h) runs two blocks per SM
    if (esize == 4 && p.n_strips == 1 && p.W > kLean256MinW && p.W <= 2048 && occ > 2) occ = 2;
    if (occ < 1) occ = 1;
    const long long slots_total = (long long)device_sm_count() * occ;
    long long per_chain = slots_total / chains;
    if (per_chain < 1) per_chain = 1;
    int seg = (int)((n_max + per_chain - 1) / per_chain);
    // never shorter than the taps: a step costs ~1 us of latency whatever the row width, so small frames want MANY short
    // segments (512^2: 12 steps per block instead of 32) and pay the 4c warm-up rows in bytes they do not miss; large
    // frames never get here (4096^2: 28-row segments fill one wave)
    if (seg < 2 * c) seg = 2 * c;
    if (seg > n_max) seg = n_max;
    p.seg = seg;
    p.n_seg = (n_max + seg - 1) / seg;
    geo->nt = nt;
    geo->ng = ng;
    geo->smem = smem;
    return true;
}

// WB_WOW_LEAN=0 in the environment selects the generic kernel for fp32 too (A/B measurements, bit-identity tests).
static bool wow_packed_enabled() {
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("WB_WOW_LEAN");
        v = (e && e[0] == '0') ? 0 : 1;
    }
    return v != 0;
}

// WB_WOW_PAIR=0 in the environment keeps the half-row column groups at every dilation (A/B measurements).
static int wow_pair_level() {
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("WB_WOW_PAIR");
        v = e ? atoi(e) : 1;
    }
    return v;
}

// Which lean kernels run with the step loop NOT unrolled (DYN).  Measured at 4096^2 (profiles/r2_fused_dyn.json): not
// unrolled, a kernel is 22 - 33 KB instead of 54 - 92 KB and a change of kernel inside a cascade no longer costs ~5 us of
// cold instruction cache, but the plain d % 4 == 0 kernels lose 2 us per launch in the steady state (47.1 -> 49.7,
// 41.5 -> 43.4 us: no scheduling across steps); the d = 1 / d = 2 kernels lose nothing (39.8 us) and the kernels with
// an inlined erff / hard threshold are faster (scales 0 / 1: 55.8 -> 52.3 us, paired: 65.5 -> 62.8 us).  Default: not
// unrolled unless the kernel is the plain d % 4 == 0 one; WB_WOW_DYN=0 / 1 in the environment: never / always.
static bool wow_dyn_for(int dmode, int sig_mode) {
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("WB_WOW_DYN");
        v = e ? (e[0] == '0' ? 0 : 1) : 2;
    }
    if (v < 2) return v != 0;
    return dmode != 0 || sig_mode != 0;
}

template <int TAPS, int DMODE, bool HINTS, int M, bool DYN>
static auto wow_lean_kernel_mode(int sig_mode) -> void (*)(const ScaleParams) {
    return sig_mode == 0 ? wow_rows_lean_kernel<TAPS, DMODE, HINTS, 0, M, DYN>
                         : (sig_mode == 1 ? wow_rows_lean_kernel<TAPS, DMODE, HINTS, 1, M, DYN>
                                          : wow_rows_lean_kernel<TAPS, DMODE, HINTS, 2, M, DYN>);
}

template <typename T, int TAPS, int DMODE, bool HINTS>
static auto wow_kernel_for(bool packed, int pair, bool dyn, int sig_mode) -> void (*)(const ScaleParams) {
    if constexpr (sizeof(T) == 4) {
        if constexpr (HINTS) {
            if constexpr (DMODE == 0) {
                if (packed && pair == 1)
                    return dyn ? wow_lean_kernel_mode<TAPS, 0, true, 1, true>(sig_mode)
                               : wow_lean_kernel_mode<TAPS, 0, true, 1, false>(sig_mode);
            }
            if (packed && dyn) return wow_lean_kernel_mode<TAPS, DMODE, true, 0, true>(sig_mode);
        }
        if (packed) return wow_lean_kernel_mode<TAPS, DMODE, HINTS, 0, false>(sig_mode);
    }
    return wow_rows_kernel<T, TAPS, DMODE, 2, HINTS>;
}

// Paired columns (x, x + M d): M = 1 from d = 32 on (runs of d / 4 >= 8 consecutive vectors keep the LDS.128 of eight
// consecutive lanes conflict-free).  M = 2 at d = 16 and M = 4 at d = 8 were built and measured (the kernel template
// takes them): alone the d = 16 launch gains 7 us (48 -> 41), inside wow() the two additional kernels per cascade cost
// more than that (0.611 -> 0.619 ms, profiles/r2_pair_levels.json) -- not instantiated.
// Thread t owns vectors (t / run) 2 run + t % run and + run of the row (pair_first_vector, run = d / 4): the block's nt
// threads must cover every first vector of the W / 4 vectors.  They do not at d = W (Triangle on a power-of-two row:
// the second vectors all fall beyond the row and half of it would never be written), so that case, like the K1 kernels
// (k1_pair_step), keeps the half-row column groups.
static int wow_pair_step(int taps, int d, int W, int nt) {
    (void)taps;
    if (d < 32 || (d & (d - 1)) != 0 || wow_pair_level() <= 0) return 0;
    const int run = d / 4, nvec = W / 4;
    const int need = ((nvec + 2 * run - 1) / (2 * run)) * run;
    return need <= nt ? 1 : 0;
}

// Rows of 513 .. 2048 columns: 256-thread blocks on 8 KiB slots, two per SM, with the default choice of not-unrolled /
// unrolled kernels only (hints on).
template <int TAPS, int DMODE>
static auto wow_lean256_kernel(int pair, int sig_mode) -> void (*)(const ScaleParams) {
    if constexpr (DMODE == 0) {
        if (pair == 1)
            return sig_mode == 0 ? wow_rows_lean_kernel<TAPS, 0, true, 0, 1, false, 256>
                                 : (sig_mode == 1 ? wow_rows_lean_kernel<TAPS, 0, true, 1, 1, true, 256>
                                                  : wow_rows_lean_kernel<TAPS, 0, true, 2, 1, true, 256>);
        return sig_mode == 0 ? wow_rows_lean_kernel<TAPS, 0, true, 0, 0, false, 256>
                             : (sig_mode == 1 ? wow_rows_lean_kernel<TAPS, 0, true, 1, 0, true, 256>
                                              : wow_rows_lean_kernel<TAPS, 0, true, 2, 0, true, 256>);
    } else {
        return sig_mode == 0 ? wow_rows_lean_kernel<TAPS, DMODE, true, 0, 0, true, 256>
                             : (sig_mode == 1 ? wow_rows_lean_kernel<TAPS, DMODE, true, 1, 0, true, 256>
                                              : wow_rows_lean_kernel<TAPS, DMODE, true, 2, 0, true, 256>);
    }
}

template <typename T, int TAPS, int DMODE, bool HINTS>
static int launch_wow_h(const ScaleParams &p, int batch, const WowGeom &geo, cudaStream_t st) {
    // the lean kernel runs 512 threads x 2 vectors on 16 KiB ring slots (rows of 2049 .. 4096 columns) or 256 threads on
    // 8 KiB slots (513 .. 2048 columns; hints on); narrower rows and float64 keep the generic kernel
    const bool lean_ok = sizeof(T) == 4 && p.n_strips == 1 && wow_packed_enabled();
    const bool packed = lean_ok && p.W > 2048;
    const bool packed256 = lean_ok && HINTS && p.W > kLean256MinW && p.W <= 2048 && geo.ng == 2;
    const int pair = ((packed || packed256) && DMODE == 0 && HINTS) ? wow_pair_step(TAPS, p.d, p.W, packed ? 512 : 256) : 0;
    const bool dyn = packed && HINTS && wow_dyn_for(DMODE, p.sig_mode);
    void (*kern)(const ScaleParams) = nullptr;
    if constexpr (sizeof(T) == 4 && HINTS) {
        if (packed256) kern = wow_lean256_kernel<TAPS, DMODE>(pair, p.sig_mode);
    }
    if (!kern) kern = wow_kernel_for<T, TAPS, DMODE, HINTS>(packed, pair, dyn, p.sig_mode);
    const int nt = packed ? 512 : (packed256 ? 256 : geo.nt);
    const size_t smem = (packed || packed256) ? (size_t)(kInRing + kWRing) * (size_t)nt * 32 + 8 * (size_t)(kInRing + kWRing) : geo.smem;
    // generic, lean x 3 significance modes x {plain, paired} x {unrolled, not}, lean-256 x 3 x {plain, paired}; per device
    static bool configured[19][64] = {};
    const int kidx = packed ? 1 + p.sig_mode + 3 * pair + 6 * (dyn ? 1 : 0) : (packed256 ? 13 + p.sig_mode + 3 * pair : 0);
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !configured[kidx][dev]) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem);
        if (e != cudaSuccess) return (int)e;
        if (dev >= 0 && dev < 64) configured[kidx][dev] = true;
    }
    dim3 grid((unsigned)((long long)p.n_strips * p.d * p.n_seg), (unsigned)batch);
    return launch_pdl<ScaleParams>(kern, grid, dim3((unsigned)nt), smem, st, p);
}

template <typename T, int TAPS, int DMODE>
static int launch_wow(const ScaleParams &p, int batch, const WowGeom &geo, cudaStream_t st) {
    return p.l2_hints ? launch_wow_h<T, TAPS, DMODE, true>(p, batch, geo, st)
                      : launch_wow_h<T, TAPS, DMODE, false>(p, batch, geo, st);
}

template <typename T, int TAPS>
static int dispatch_wow(const ScaleParams &p, int batch, const WowGeom &geo, cudaStream_t st) {
    constexpr int V = VecOf<T>::V;
    const int dmode = (p.d % V == 0) ? 0 : p.d;
    if (dmode == 0) return launch_wow<T, TAPS, 0>(p, batch, geo, st);
    if (dmode == 1) return launch_wow<T, TAPS, 1>(p, batch, geo, st);
    if constexpr (V == 4) {
        if (dmode == 2) return launch_wow<T, TAPS, 2>(p, batch, geo, st);
    }
    return WB_ENOT_FUSABLE;
}

static int fill_wow_params(ScaleParams &p, const void *in, void *out_c, void *out_w, int batch, int H, int W,
                           long long in_pitch, long long in_bstride, long long c_pitch, long long c_bstride,
                           long long w_pitch, long long w_bstride, int scale, int taps, int dtype) {
    int rc = check_common(batch, H, W, taps, dtype);
    if (rc) return rc;
    if (scale < 0 || scale > 30) return WB_EINVAL_SCALE;
    if (!in || !out_c || !out_w || in == out_c || in == out_w || out_c == out_w) return WB_EINVAL_POINTER;
    if (in_pitch < W || c_pitch < W || w_pitch < W) return WB_EINVAL_ARG;
    memset(&p, 0, sizeof(p));
    p.in = in; p.out_c = out_c; p.out_w = out_w;
    p.H = H; p.W = W; p.d = 1 << scale; p.Hg = H;
    p.in_pitch = in_pitch; p.in_bstride = in_bstride;
    p.c_pitch = c_pitch; p.c_bstride = c_bstride;
    p.w_pitch = w_pitch; p.w_bstride = w_bstride;
    {
        static int v = -1;  // WB_L2_HINTS_WOW=0/1/2/3 (bit 0: input evict-first, bit 1: c_{s+1} evict-last); A/B measurements
        if (v < 0) {
            const char *e = getenv("WB_L2_HINTS_WOW");
            v = e ? atoi(e) : 3;
        }
        p.l2_hints = l2_hints_enabled() ? v : 0;
    }

    return WB_OK;
}

}  // namespace wb

extern "C" {

int wb_wow_scale_path(int batch, int H, int W, long long in_pitch, long long out_c_pitch, long long out_w_pitch,
                      int scale, int taps, int dtype, const void *in, const void *out_c, const void *out_w) {
    wb::ScaleParams p;
    if (wb::fill_wow_params(p, in, const_cast<void *>(out_c), const_cast<void *>(out_w), batch, H, W, in_pitch, 0,
                            out_c_pitch, 0, out_w_pitch, 0, scale, taps, dtype))
        return 0;
    wb::WowGeom geo;
    return wb::plan_wow(p, taps, wb::dtype_size(dtype), batch, &geo) ? 1 : 0;
}

int wb_wow_scale(const void *in, void *out_c, void *out_w, int batch, int H, int W, long long in_pitch,
                 long long in_bstride, long long out_c_pitch, long long out_c_bstride, long long out_w_pitch,
                 long long out_w_bstride, int scale, int taps, int dtype, int sig_mode, double sigma, double sigma_e,
                 double noise_host, const double *noise_dev, double weight, void *stream) {
    wb::ScaleParams p;
    int rc = wb::fill_wow_params(p, in, out_c, out_w, batch, H, W, in_pitch, in_bstride, out_c_pitch, out_c_bstride,
                                 out_w_pitch, out_w_bstride, scale, taps, dtype);
    if (rc) return rc;
    if (sig_mode < 0 || sig_mode > 2) return WB_EINVAL_ARG;
    p.sig_mode = sig_mode; p.sigma = sigma; p.sigma_e = sigma_e;
    p.noise_host = noise_host; p.noise_dev = noise_dev; p.weight = weight;
    wb::WowGeom geo;
    if (!wb::plan_wow(p, taps, wb::dtype_size(dtype), batch, &geo)) return WB_ENOT_FUSABLE;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == WB_F32)
        return taps == 3 ? wb::dispatch_wow<float, 3>(p, batch, geo, st) : wb::dispatch_wow<float, 5>(p, batch, geo, st);
    return taps == 3 ? wb::dispatch_wow<double, 3>(p, batch, geo, st) : wb::dispatch_wow<double, 5>(p, batch, geo, st);
}

}  // extern "C"
