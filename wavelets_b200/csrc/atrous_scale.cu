// K1 -- one scale of the plain à trous cascade, fused: c_{s+1} = S_s[c_s] and w_s = c_s - c_{s+1} in one pass.
//
// Replaces watroo/wavelets.py:35-45 (cv2.filter2D with the dense dilated kernel of :191-197, BORDER_REFLECT) and the
// in-place subtraction of :442.  HBM-bound: 3*sizeof(T) algorithmic bytes per pixel (read c_s, write c_{s+1}, w_s).
//
// Design (see DESIGN.md, "K1"):
//   * The dilated separable filter only couples pixels that are 2^s apart, so the image splits into 2^s row
//     "chains" (rows r, r+d, r+2d, ... with d = 2^s).  A thread block owns a segment of one chain over one column
//     strip and walks down it with a sliding window: every input row is fetched ONCE per block, as one contiguous
//     TMA bulk copy (cp.async.bulk -> UBLKCP) into a shared-memory ring guarded by full/empty mbarriers, issued by a
//     dedicated producer warp.  The column halo costs (taps-1) extra row loads per segment whatever the dilation,
//     so deep scales are as cheap as shallow ones (no 2^s-wide halo, no dense kernel).
//   * Row pass: each consumer thread owns NG 16-byte vectors of columns and reads its taps x + k*d straight from
//     the staged row with LDS.128 (conflict-free: consecutive threads read consecutive vectors).  When the strip is
//     the whole row the x halo is free -- the symmetric border is an index reflection inside the same staged row
//     (a reflected aligned vector is the mirrored vector read backwards).
//   * Column pass: the last `taps` row-filtered vectors live in a register ring; c_{s+1} comes out of registers,
//     w_s = raw - c_{s+1} uses the raw centre row still resident in the ring, and both are written with 128-bit
//     coalesced stores (w_s with an evict-first hint so it does not push c_{s+1} out of L2 before scale s+1 reads it).
//   * Anything the vector path cannot take (W % V != 0, unaligned pointers, 2^s*c > W so more than one reflection)
//     goes to a generic gather kernel with the full modular reflection.
#include "pipeline.cuh"
#include "whiten.cuh"

namespace wb {

// MAP (OP_WHITEN only): the noise-map mode of the epilogue (sig_mode == SIG_MAP, see whiten.cuh).
template <typename T, int TAPS, int DMODE, int NG, int OP, bool MAP = false>
__global__ void __launch_bounds__(544) atrous_rows_kernel(const ScaleParams p) {
    constexpr int V = VecOf<T>::V;
    constexpr int C = TAPS / 2;
    constexpr int NV = PlanSize<TAPS, DMODE>::NV;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    T *rows = reinterpret_cast<T *>(smem_raw);
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw + (size_t)p.slots * p.row_stride * sizeof(T));
    uint64_t *empty = full + p.slots;

    pdl_launch_dependents();
    const int nt = blockDim.x - 32;  // consumer threads; the last warp is the TMA producer
    const int nwc = nt >> 5;
    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int lane = tid & 31;

    // block -> (strip, chain residue r, segment g); r varies fastest so concurrent blocks touch adjacent rows
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
    __syncthreads();
    pdl_wait();  // everything below touches global memory written or read by the previous launch

    if (warp == nwc) {
        // ---------------- producer warp: one lane streams the chain rows into the ring ----------------
        if (lane == 0) {
            const long long foff = (long long)frame * p.in_bstride + lo;
            const uint64_t pol_in = policy_evict_first();  // c_s is dead once this launch has read it
            int slot = 0;
            uint32_t round = 0;
            for (int j = 0; j < n_load; ++j) {
                if (round > 0) mbar_wait(&empty[slot], (round - 1) & 1);
                // the row may live in a neighbour's band buffer (peer-window mode): same bulk copy, over NVLink
                const T *src = input_row<T>(p, reflect_any(p.gwy0 + r + (long long)(i0 - C + j) * p.d, p.Hg)) + foff;
                mbar_arrive_expect_tx(&full[slot], row_bytes);
                if (p.l2_hints)
                    tma_load_1d_hint(rows + (size_t)slot * p.row_stride, src, row_bytes, &full[slot], pol_in);
                else
                    tma_load_1d(rows + (size_t)slot * p.row_stride, src, row_bytes, &full[slot]);
                if (++slot == p.slots) { slot = 0; ++round; }
            }
        }
        return;
    }

    // ---------------- consumer warps ----------------
    T *c_ptr = reinterpret_cast<T *>(p.out_c);
    T *w_ptr = reinterpret_cast<T *>(p.out_w);
    // first output row of this block; the pointers advance by one chain step (d rows) per output row
    const long long orow = (long long)r + (long long)i0 * p.d;
    const T *c_base = c_ptr ? c_ptr + (long long)frame * p.c_bstride + p.row_off_c * p.c_pitch : nullptr;  // output row 0
    if (c_ptr) c_ptr += (long long)frame * p.c_bstride + (orow + p.row_off_c) * p.c_pitch;
    if (w_ptr) w_ptr += (long long)frame * p.w_bstride + (orow + p.row_off_w) * p.w_pitch;
    const long long c_step = (long long)p.d * p.c_pitch, w_step = (long long)p.d * p.w_pitch;
    const bool pushing = (p.push_up != nullptr) | (p.push_dn != nullptr);
    int out_row = (int)orow;  // band row of the next output

    WhitenEpilogue<T> epi;
    if constexpr (OP == OP_WHITEN) epi.template init<MAP>(p, frame);
    // map mode: row pointer into the noise map (whole-frame launches: no row offset)
    const T *m_ptr = nullptr;
    long long m_step = 0;
    if constexpr (MAP) {
        m_ptr = reinterpret_cast<const T *>(p.noise_map) + (long long)frame * p.map_bstride + orow * p.map_pitch;
        m_step = (long long)p.d * p.map_pitch;
    }
    const uint64_t pol_keep = policy_evict_last();  // c_{s+1}: the next scale reads it back
    const bool hints = p.l2_hints != 0;

    int xg[NG];
    uint32_t xb[NG];  // byte offset of this thread's own vector inside a staged row
    bool act[NG];
    BytePlan<NV> plan[NG];
#pragma unroll
    for (int q = 0; q < NG; ++q) {
        xg[q] = x0 + (q * nt + tid) * V;
        act[q] = xg[q] < p.W && xg[q] < x0 + p.wt;
        if (!act[q]) xg[q] = x0;  // idle threads shadow the first vector of the strip; only their stores are masked
        xb[q] = (uint32_t)(xg[q] - lo) * (uint32_t)sizeof(T);
        const TapPlan<NV> tp = make_tap_plan<V, NV>(xg[q], DMODE == 0 ? p.d : V, p.W, lo);
#pragma unroll
        for (int k = 0; k < NV; ++k) plan[q].off[k] = (uint32_t)tp.off[k] * (uint32_t)sizeof(T);
        plan[q].rev = tp.rev;
    }

    // running column sums (col_feed): TAPS-1 live values per element, no register-ring rotation
    T S[NG][V][TAPS - 1];
#pragma unroll
    for (int q = 0; q < NG; ++q)
#pragma unroll
        for (int e = 0; e < V; ++e)
#pragma unroll
            for (int t = 0; t < TAPS - 1; ++t) S[q][e][t] = T(0);

    const uint32_t RB = (uint32_t)p.row_stride * (uint32_t)sizeof(T);
    const uint32_t ring_base = smem_u32(rows), ring_end = ring_base + (uint32_t)p.slots * RB;
    uint32_t row_addr = ring_base, crow_addr = ring_base;  // staged row j and centre row j - C
    int slot = 0, cslot = 0;
    uint32_t parity = 0;
    for (int j = 0; j < n_load; ++j) {
        mbar_wait(&full[slot], parity);
        Pack<T, V> cv[NG];
#pragma unroll
        for (int q = 0; q < NG; ++q) {
            const Pack<T, V> v = row_pass_b<T, TAPS, DMODE, OP != OP_TRANSFORM>(row_addr, plan[q]);
#pragma unroll
            for (int e = 0; e < V; ++e) cv[q].v[e] = col_feed<T, TAPS>(S[q][e], v.v[e]);
        }
        if (j >= 2 * C) {
#pragma unroll
            for (int q = 0; q < NG; ++q) {
                if constexpr (OP == OP_TRANSFORM) {
                    if (c_ptr && act[q]) {
                        if (hints) st_vec_hint(c_ptr + xg[q], cv[q], pol_keep);
                        else st_vec(c_ptr + xg[q], cv[q]);
                        if (pushing) push_store(p, c_ptr + xg[q], c_base, out_row, cv[q]);
                    }
                    if (w_ptr) {
                        Pack<T, V> raw = lds_vec<T>(crow_addr + xb[q]);
#pragma unroll
                        for (int e = 0; e < V; ++e) raw.v[e] -= cv[q].v[e];
                        if (act[q]) st_vec_cs(w_ptr + xg[q], raw);
                    }
                } else if constexpr (OP == OP_POWER) {
                    if (act[q]) st_vec(c_ptr + xg[q], cv[q]);
                } else {
                    const Pack<T, V> raw = lds_vec<T>(crow_addr + xb[q]);
                    Pack<T, V> out;
#pragma unroll
                    for (int e = 0; e < V; ++e) out.v[e] = epi.apply(raw.v[e], cv[q].v[e]);
                    if (MAP && act[q]) {
                        const Pack<T, V> nz = ld_vec_stream(m_ptr + xg[q]);
#pragma unroll
                        for (int e = 0; e < V; ++e) out.v[e] = epi.map_sig(raw.v[e], out.v[e], nz.v[e]);
                    }
                    if (act[q]) st_vec_cs(w_ptr + xg[q], out);
                }
            }
            if (c_ptr) c_ptr += c_step;
            if (w_ptr) w_ptr += w_step;
            if constexpr (MAP) m_ptr += m_step;
            out_row += p.d;
        }
        if (j >= C) {
            // the raw row j-C is not needed any more: hand its slot back to the producer
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[cslot]);
            crow_addr += RB;
            if (++cslot == p.slots) { cslot = 0; crow_addr = ring_base; }
        }
        row_addr += RB;
        if (++slot == p.slots) { slot = 0; row_addr = ring_base; parity ^= 1; }
    }
    (void)ring_end;
}

// ---------------------------------------------------------------------------------------------------------------
// K1, fp32 whole-row strips: the same pipeline, LEAN (see wow_scale.cu for the measurements behind the recipe).  The
// kernel above spends ~330 warp instructions per warp-step of which ~100 are floating point (ncu: 22.5 M warp
// instructions per 4096^2 plane, 67 % issue-active).  Here the consumer loop is unrolled by half the 8-slot ring, ring
// slots have a fixed 16 KiB stride (every LDS is [register + immediate]), pixel pairs are carried as 64-bit
// register pairs (FFMA2 / FMUL2 / FADD2, same roundings as the scalar instructions) and the output pointers are
// per-thread and advance by one add per row.  Same operation order as atrous_rows_kernel: bit-identical planes.
// ---------------------------------------------------------------------------------------------------------------
static constexpr int kLeanSlots = 8;

// OP_WHITEN (K3 of the two-pass WOW routes, MODE = significance compiled into the epilogue): the row pass filters the
// SQUARES of the staged raw w_s rows and the epilogue whitens the raw centre value -- same pipeline, 2*T bytes per pixel.
// PAIR = M > 0 (DMODE 0, d >= 8): a thread's two column vectors are M dilation steps apart (x, x + M d) and share
// TAPS - M of their tap vectors (lean_row_pass_pair, see wow_rows_lean_kernel): 8 instead of 12 LDS.128 per step at M = 1.
// The step loop is unrolled by half the ring and the ring's two halves alternate: one more address term per access than
// a loop unrolled by the whole ring, but HALF the code -- a 60 KB kernel does not fit the 32 KB instruction cache level,
// and every change of kernel inside a cascade starts cold.
// T / RBK (round 2): float64 rows (one double per 64-bit lane: DFMA instead of FFMA2, see Lane<T>) and COLUMN STRIPS -- a
// block stages columns [x0 - halo, x0 + wt + halo) of its strip in ring slots of RBK KiB (16: whole rows of <= 4096 fp32
// columns, the geometry the kernel was written for; 24: strips of 4096 fp32 / 2048 fp64 columns with up to 1024 / 512
// halo columns per side, i.e. rows wider than one slot at every dilation up to 512 / 256).
template <typename T, int TAPS, int DMODE, bool HINTS, int OP, int MODE, int PAIR, int RBK>
__global__ void __launch_bounds__(544) atrous_rows_lean_kernel(const ScaleParams p) {
    static_assert(PAIR == 0 || (DMODE == 0 && PAIR < TAPS), "paired columns need d % V == 0 and overlapping taps");
    constexpr int V = VecOf<T>::V, NG = 2;
    constexpr int C = TAPS / 2;
    constexpr int NV = PlanSize<TAPS, DMODE>::NV;
    constexpr int RB = RBK * 1024;
    using L = Lane<T>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const uint32_t in_base = smem_u32(smem_raw);
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw + (size_t)kLeanSlots * RB);
    uint64_t *empty = full + kLeanSlots;
    const uint32_t full0 = smem_u32(full), empty0 = smem_u32(empty);

    pdl_launch_dependents();
    const int nt = blockDim.x - 32;  // consumer threads; the last warp is the TMA producer
    const int nwc = nt >> 5;
    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int lane = tid & 31;

    // block -> (strip, chain residue r, segment g); whole-row launches have one strip
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
        for (int s = 0; s < kLeanSlots; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], nwc);
        }
        fence_mbar_init();
    }
    __syncthreads();
    pdl_wait();  // everything below touches global memory written or read by the previous launch

    if (warp == nwc) {
        // ---------------- producer warp: one lane streams the chain rows into the ring ----------------
        if (lane == 0) {
            const long long foff = (long long)frame * p.in_bstride + lo;
            const uint64_t pol_in = policy_evict_first();  // c_s is dead once this launch has read it
            for (int j = 0; j < n_load; ++j) {
                const int slot = j & (kLeanSlots - 1);
                if (j >= kLeanSlots) mbar_wait(&empty[slot], (uint32_t)((j >> 3) - 1) & 1u);
                // the row may live in a neighbour's band buffer (peer-window mode): same bulk copy, over NVLink
                const T *src = input_row<T>(p, reflect_any(p.gwy0 + r + (long long)(i0 - C + j) * p.d, p.Hg)) + foff;
                mbar_arrive_expect_tx(&full[slot], row_bytes);
                if (HINTS) tma_load_1d_hint(smem_raw + (size_t)slot * RB, src, row_bytes, &full[slot], pol_in);
                else tma_load_1d(smem_raw + (size_t)slot * RB, src, row_bytes, &full[slot]);
            }
        }
        return;
    }

    // ---------------- consumer warps ----------------
    const PackedTaps<TAPS, T> H;
    const uint64_t pol_keep = policy_evict_last();  // c_{s+1}: the next scale reads it back
    WhitenEpilogue<T> epi;
    if constexpr (OP == OP_WHITEN) epi.template init<MODE == SIG_MAP>(p, frame);

    constexpr int NTAP = PAIR ? 1 : NG, NPT = TAPS + PAIR;
    uint32_t own[NG], tap[NTAP][NV], ptap[NPT];
    unsigned rev[NG] = {0u, 0u};
    bool act[NG];
    int xg0 = 0;
    bool mirror_warp;
    const int x_end = min(p.W, x0 + p.wt);  // columns [x0, x_end) are this block's
    if constexpr (PAIR) {
        const int run = PAIR * (p.d / V);  // vectors between the two of a pair (>= 8)
        const int xa = x0 + pair_first_vector(tid, run) * V, xb = xa + PAIR * p.d;
        act[0] = xa < x_end;
        act[1] = xb < x_end;
        xg0 = act[0] ? xa : x0;  // idle threads shadow the first pair of the strip; only their stores are masked
        own[0] = opaque_u32(in_base + (uint32_t)(xg0 - lo) * (uint32_t)sizeof(T));
        own[1] = opaque_u32(act[1] ? own[0] + (uint32_t)(PAIR * p.d) * (uint32_t)sizeof(T) : own[0]);
        rev[0] = opaque_u32(make_pair_plan<TAPS, PAIR, V>(xg0, p.d, p.W, lo, in_base, ptap));
#pragma unroll
        for (int k = 0; k < TAPS + PAIR; ++k) ptap[k] = opaque_u32(ptap[k]);
        mirror_warp = __any_sync(0xffffffffu, rev[0] != 0 || !act[0]);
    } else {
#pragma unroll
        for (int q = 0; q < NG; ++q) {
            int xg = x0 + (q * nt + tid) * V;
            act[q] = xg < x_end;
            // idle threads shadow an interior vector of the strip (its middle for whole rows, where the dilation can be
            // half the width; its first vector otherwise); only their stores are masked
            if (!act[q]) xg = (p.n_strips == 1) ? ((p.W / 2) & ~(V - 1)) : x0;
            if (q == 0) xg0 = xg;
            own[q] = opaque_u32(in_base + (uint32_t)(xg - lo) * (uint32_t)sizeof(T));
            const TapPlan<NV> tp = make_tap_plan<V, NV>(xg, DMODE == 0 ? p.d : V, p.W, lo);
#pragma unroll
            for (int k = 0; k < NV; ++k) tap[q][k] = opaque_u32(in_base + (uint32_t)tp.off[k] * (uint32_t)sizeof(T));
            rev[q] = opaque_u32(tp.rev);
        }
        mirror_warp = __any_sync(0xffffffffu, (rev[0] | rev[1]) != 0);
    }
    // the second column vector of a thread: M dilation steps (PAIR) or nt vectors further (when active)
    const long long q_off = PAIR ? (long long)PAIR * p.d : (long long)nt * V;

    u64 S[NG][2][TAPS - 1];  // running column sums, one pixel pair per entry
#pragma unroll
    for (int q = 0; q < NG; ++q)
#pragma unroll
        for (int e = 0; e < 2; ++e)
#pragma unroll
            for (int t = 0; t < TAPS - 1; ++t) S[q][e][t] = 0ull;

    T *c_ptr = reinterpret_cast<T *>(p.out_c);
    T *w_ptr = reinterpret_cast<T *>(p.out_w);
    const long long orow = (long long)r + (long long)i0 * p.d;  // first output row of this block
    const T *c_base = c_ptr ? c_ptr + (long long)frame * p.c_bstride + p.row_off_c * p.c_pitch : nullptr;  // output row 0
    if (c_ptr) c_ptr += (long long)frame * p.c_bstride + (orow + p.row_off_c) * p.c_pitch + xg0;
    if (w_ptr) w_ptr += (long long)frame * p.w_bstride + (orow + p.row_off_w) * p.w_pitch + xg0;
    const long long c_step = (long long)p.d * p.c_pitch, w_step = (long long)p.d * p.w_pitch;
    // map mode: the noise-map vectors of the output vectors (whole-frame launches: no row offset)
    const T *m_ptr = nullptr;
    long long m_step = 0;
    if constexpr (MODE == SIG_MAP) {
        m_ptr = reinterpret_cast<const T *>(p.noise_map) + (long long)frame * p.map_bstride + orow * p.map_pitch + xg0;
        m_step = (long long)p.d * p.map_pitch;
    }
    const bool has_c = c_ptr != nullptr, has_w = w_ptr != nullptr;
    const bool pushing = (p.push_up != nullptr) | (p.push_dn != nullptr);
    int out_row = (int)orow;  // band row of the next output

    // Step j = 4 u + I: input row j lands (ring slot j % 8 = I + (half ? 4 : 0)) -> row pass -> column feed -> c row
    // j-C; w = raw centre row - c; release the centre row's slot.  `half` / `half_c`: byte offset (0 or 4 RB) of the ring
    // half this iteration's rows land in / of the other half.
    auto step = [&](auto ic, auto mirror, const int j, const uint32_t par, const uint32_t half, const uint32_t half_c) {
        constexpr int I = decltype(ic)::value;
        constexpr bool MIRROR = decltype(mirror)::value != 0;
        if (j >= n_load) return;
        mbar_wait_imm<8 * I>(full0 + (half ? 32u : 0u), par);  // 8 bytes of barrier per slot: the second half starts at 32
        P4 cv[NG];
        if constexpr (PAIR) {
            uint32_t a[TAPS + PAIR];
#pragma unroll
            for (int k = 0; k < TAPS + PAIR; ++k) a[k] = ptap[k] + half;
            P4 v[NG];
            lean_row_pass_pair<TAPS, PAIR, I * RB, OP == OP_WHITEN, MIRROR>(a, rev[0], H, v[0], v[1]);
#pragma unroll
            for (int q = 0; q < NG; ++q) {
                cv[q].lo = col_feed_p<TAPS>(S[q][0], v[q].lo, H);
                cv[q].hi = col_feed_p<TAPS>(S[q][1], v[q].hi, H);
            }
        } else {
#pragma unroll
            for (int q = 0; q < NG; ++q) {
                uint32_t a[NV];
#pragma unroll
                for (int k = 0; k < NV; ++k) a[k] = tap[q][k] + half;
                const P4 v = lean_row_pass<TAPS, DMODE, I * RB, OP == OP_WHITEN, MIRROR>(a, rev[q], H);
                cv[q].lo = col_feed_p<TAPS>(S[q][0], v.lo, H);
                cv[q].hi = col_feed_p<TAPS>(S[q][1], v.hi, H);
            }
        }
        // raw centre row j-C: slot (I - C) mod 4 of this half, or of the other half when the index wraps
        constexpr int SC = (I - C + 4) & 3;
        const uint32_t hc = (I < C) ? half_c : half;
        if (j >= 2 * C) {
            if constexpr (OP == OP_WHITEN) {
#pragma unroll
                for (int q = 0; q < NG; ++q) {
                    P4 raw = lds_p4_imm<SC * RB>(own[q] + hc);
                    P4 out;
                    out.lo = epi.template apply_lane<MODE>(raw.lo, cv[q].lo);
                    out.hi = epi.template apply_lane<MODE>(raw.hi, cv[q].hi);
                    if constexpr (MODE == SIG_MAP) {
                        if (act[q]) {
                            const P4 nz = ldg_p4_stream(m_ptr + q * q_off);
                            out.lo = epi.map_lane(raw.lo, out.lo, nz.lo);
                            out.hi = epi.map_lane(raw.hi, out.hi, nz.hi);
                        }
                    }
                    if (act[q]) stg_p4_cs(w_ptr + q * q_off, out);
                }
                w_ptr += w_step;
                if constexpr (MODE == SIG_MAP) m_ptr += m_step;
            } else {
#pragma unroll
            for (int q = 0; q < NG; ++q) {
                if (has_c && act[q]) {
                    if (HINTS) stg_p4_hint(c_ptr + q * q_off, cv[q], pol_keep);
                    else stg_p4(c_ptr + q * q_off, cv[q]);
                    if (pushing) push_store(p, c_ptr + q * q_off, c_base, out_row, cv[q]);
                }
                if (has_w) {
                    P4 raw = lds_p4_imm<SC * RB>(own[q] + hc);
                    raw.lo = L::sub(raw.lo, cv[q].lo);
                    raw.hi = L::sub(raw.hi, cv[q].hi);
                    if (act[q]) stg_p4_cs(w_ptr + q * q_off, raw);
                }
            }
            if (has_c) c_ptr += c_step;
            if (has_w) w_ptr += w_step;
            out_row += p.d;
            }
        }
        if (j >= C) {
            // the raw row j-C is not needed any more: hand its slot back to the producer
            __syncwarp();
            if (lane == 0) mbar_arrive_imm<8 * SC>(empty0 + (hc ? 32u : 0u));
        }
    };
    auto run = [&](auto mirror) {
#pragma unroll 1
        for (int jb = 0; jb < n_load; jb += 4) {
            const uint32_t par = (uint32_t)(jb >> 3) & 1u;
            const uint32_t half = (jb & 4) ? 4u * RB : 0u;
            const uint32_t half_c = half ^ (4u * RB);
            step(IC<0>{}, mirror, jb + 0, par, half, half_c);
            step(IC<1>{}, mirror, jb + 1, par, half, half_c);
            step(IC<2>{}, mirror, jb + 2, par, half, half_c);
            step(IC<3>{}, mirror, jb + 3, par, half, half_c);
        }
    };
    if (mirror_warp) run(IC<1>{});
    else run(IC<0>{});
}

// Generic path: one thread per output pixel, full modular reflection, any shape / alignment.
template <typename T, int TAPS, int OP, bool MAP = false>
__global__ void __launch_bounds__(256) atrous_generic_kernel(const ScaleParams p) {
    constexpr int C = TAPS / 2;
    const long long n = (long long)p.H * p.W;
    const int frame = blockIdx.y;
    const long long foff = (long long)frame * p.in_bstride;
    T *out_c = reinterpret_cast<T *>(p.out_c);
    T *out_w = reinterpret_cast<T *>(p.out_w);
    WhitenEpilogue<T> epi;
    if constexpr (OP == OP_WHITEN) epi.template init<MAP>(p, frame);
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n;
         idx += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(idx / p.W), x = (int)(idx % p.W);
        int xs[TAPS];
#pragma unroll
        for (int k = 0; k < TAPS; ++k)
            xs[k] = p.lattice ? reflect_lattice(x, k - C, p.d, p.W) : reflect_any((long long)x + (long long)(k - C) * p.d, p.W);
        T acc = T(0);
#pragma unroll
        for (int i = 0; i < TAPS; ++i) {
            const T *row = input_row<T>(p, p.lattice ? reflect_lattice(y, i - C, p.d, p.H)
                                                     : reflect_any(p.gwy0 + y + (long long)(i - C) * p.d, p.Hg)) + foff;
            T ra = T(0);
#pragma unroll
            for (int k = 0; k < TAPS; ++k) {
                T v = row[xs[k]];
                if (OP != OP_TRANSFORM) v = v * v;
                ra = (k == 0) ? Taps<T, TAPS>::h(0) * v : fma_t<T>(Taps<T, TAPS>::h(k), v, ra);
            }
            acc = (i == 0) ? Taps<T, TAPS>::h(0) * ra : fma_t<T>(Taps<T, TAPS>::h(i), ra, acc);
        }
        const T raw = (input_row<T>(p, p.gwy0 + y) + foff)[x];
        if constexpr (OP == OP_TRANSFORM) {
            if (out_c) {
                T *dst = out_c + (long long)frame * p.c_bstride + ((long long)y + p.row_off_c) * p.c_pitch + x;
                *dst = acc;
                push_store(p, dst, out_c + (long long)frame * p.c_bstride + p.row_off_c * p.c_pitch, y, acc);
            }
            if (out_w) out_w[(long long)frame * p.w_bstride + ((long long)y + p.row_off_w) * p.w_pitch + x] = raw - acc;
        } else if constexpr (OP == OP_POWER) {
            out_c[(long long)frame * p.c_bstride + (long long)y * p.c_pitch + x] = acc;
        } else {
            T v = epi.apply(raw, acc);
            if constexpr (MAP)
                v = epi.map_sig(raw, v, reinterpret_cast<const T *>(p.noise_map)[(long long)frame * p.map_bstride +
                                                                                  (long long)y * p.map_pitch + x]);
            out_w[(long long)frame * p.w_bstride + ((long long)y + p.row_off_w) * p.w_pitch + x] = v;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Host: dispatch
// ---------------------------------------------------------------------------------------------------------------
K1Config g_override[32];
bool g_override_set[32];

template <typename T, int TAPS, int DMODE, int NG, int OP, bool MAP>
static int launch_rows(const ScaleParams &p, int batch, int nt, cudaStream_t st) {
    auto kern = atrous_rows_kernel<T, TAPS, DMODE, NG, OP, MAP>;
    const size_t smem = (size_t)p.slots * p.row_stride * sizeof(T) + 16 * (size_t)p.slots;
    static bool configured[64] = {};  // per instantiation, per device
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem);
        if (e != cudaSuccess) return (int)e;
        if (dev >= 0 && dev < 64) configured[dev] = true;
    }
    dim3 grid((unsigned)((long long)p.n_strips * p.d * p.n_seg), (unsigned)batch);
    return launch_pdl<ScaleParams>(kern, grid, dim3((unsigned)(nt + 32)), smem, st, p);
}

// Paired columns (x, x + M d) with M = 1 from d = 32 on.  M = 2 at d = 16 and M = 4 at d = 8 were built and measured (the
// kernel template takes them): no gain per launch and two more distinct kernels per cascade (0.336 -> 0.358 ms per
// transform with the step loop unrolled by 8, profiles/r2_pair_levels.json) -- not instantiated.
static bool k1_pair_step(int d, int cols, int nt, int V = 4) {
    // runs of d / V >= 8 consecutive vectors: eight consecutive lanes read eight consecutive vectors
    if (d < 8 * V || (d & (d - 1)) != 0) return false;
    // thread t owns vectors (t / run) 2 run + t % run and + run of its strip: the consumer threads must cover every first
    // vector of the `cols` columns a block owns
    const int run = d / V, nvec = cols / V;
    const int need = ((nvec + 2 * run - 1) / (2 * run)) * run;
    return need <= nt;
}

// The lean kernel on ring slots of RBK KiB: 16 (whole fp32 rows of 2049 .. 4096 columns), 8 (whole fp32 rows of
// 1025 .. 2048 columns: two blocks per SM, so a 2048^2 frame runs 296 segments of 7 rows instead of 148 of 14 -- the
// launch is bound by the number of steps per block) or kLeanStripKiB (column strips and float64 rows).
template <typename T, int TAPS, int DMODE, bool HINTS, int OP, int MODE, int PAIR, int RBK>
static int launch_rows_lean(const ScaleParams &p, int batch, int nt, cudaStream_t st) {
    auto kern = atrous_rows_lean_kernel<T, TAPS, DMODE, HINTS, OP, MODE, PAIR, RBK>;
    const size_t smem = (size_t)kLeanSlots * RBK * 1024 + 16 * (size_t)kLeanSlots;
    static bool configured[64] = {};  // per instantiation, per device
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem);
        if (e != cudaSuccess) return (int)e;
        if (dev >= 0 && dev < 64) configured[dev] = true;
    }
    dim3 grid((unsigned)((long long)p.n_strips * p.d * p.n_seg), (unsigned)batch);
    return launch_pdl<ScaleParams>(kern, grid, dim3((unsigned)(nt + 32)), smem, st, p);
}

// The lean kernel on column strips / float64 rows: ring slots of 24 KiB (a strip of 16 KiB plus the halo columns of
// both sides), L2 hints on.
static constexpr int kLeanStripKiB = 24;

template <typename T, int TAPS, int DMODE, int OP, int PAIR>
static int launch_rows_lean_strip(const ScaleParams &p, int batch, int nt, cudaStream_t st) {
#define WB_STRIP(MODE) launch_rows_lean<T, TAPS, DMODE, true, OP, MODE, PAIR, kLeanStripKiB>(p, batch, nt, st)
    if constexpr (OP == OP_WHITEN) {
        if (p.sig_mode == SIG_MAP) return WB_STRIP(SIG_MAP);
        if constexpr (sizeof(T) == 4) {
            if (p.sig_mode == 1) return WB_STRIP(1);
        }
        if (p.sig_mode == 2) return WB_STRIP(2);
    }
    return WB_STRIP(0);
#undef WB_STRIP
}

template <typename T, int TAPS, int OP>
static int dispatch(ScaleParams &p, int batch, int scale, cudaStream_t st) {
    constexpr int V = VecOf<T>::V;
    const bool map = OP == OP_WHITEN && p.sig_mode == SIG_MAP;
    K1Config cfg;
    if (fast_path_ok(p, TAPS, (int)sizeof(T)) && plan_fast(p, TAPS, (int)sizeof(T), batch, scale, &cfg, OP == OP_TRANSFORM)) {
        const int dmode = (p.d % V == 0) ? 0 : p.d;
        // a geometry override (wb_tune_k1) runs the row kernel
        const bool lean_ok = cfg.ng == 2 && cfg.slots == kLeanSlots && !(scale < 32 && g_override_set[scale]);
        if constexpr (sizeof(T) == 4 && OP == OP_TRANSFORM) {
            // whole-row strips with two vectors per thread and the default ring: the lean kernel
            if (p.n_strips == 1 && p.W > 1024 && lean_ok) {
                const bool pair = dmode == 0 && k1_pair_step(p.d, p.W, cfg.nt);
#define WB_LEAN(DM, H, PR, RBK) launch_rows_lean<T, TAPS, DM, H, OP, 0, PR, RBK>(p, batch, cfg.nt, st)
                if (p.W <= 2048 && p.l2_hints) {  // 8 KiB slots (the planner counted on two blocks per SM: plan_fast)
                    if (pair) return WB_LEAN(0, true, 1, 8);
                    if (dmode == 0) return WB_LEAN(0, true, 0, 8);
                    if (dmode == 1) return WB_LEAN(1, true, 0, 8);
                    if (dmode == 2) return WB_LEAN(2, true, 0, 8);
                }
                if (pair && p.l2_hints) return WB_LEAN(0, true, 1, 16);
                if (dmode == 0) return p.l2_hints ? WB_LEAN(0, true, 0, 16) : WB_LEAN(0, false, 0, 16);
                if (dmode == 1) return p.l2_hints ? WB_LEAN(1, true, 0, 16) : WB_LEAN(1, false, 0, 16);
                if (dmode == 2) return p.l2_hints ? WB_LEAN(2, true, 0, 16) : WB_LEAN(2, false, 0, 16);
#undef WB_LEAN
            }
        }
        if constexpr (sizeof(T) == 4 && OP == OP_WHITEN) {
            // the whitening pass of the two-pass WOW routes on whole-row strips: lean kernel, hints on
            if (p.n_strips == 1 && p.W > 1024 && lean_ok) {
#define WB_LEANW(DM, PR, M) launch_rows_lean<T, TAPS, DM, true, OP, M, PR, 16>(p, batch, cfg.nt, st)
#define WB_LEANW_M(DM, PR)                                                                                            \
    (p.sig_mode == 0 ? WB_LEANW(DM, PR, 0) : p.sig_mode == 1 ? WB_LEANW(DM, PR, 1)                                    \
                     : p.sig_mode == 2 ? WB_LEANW(DM, PR, 2) : WB_LEANW(DM, PR, SIG_MAP))
                if (dmode == 0 && k1_pair_step(p.d, p.W, cfg.nt)) return WB_LEANW_M(0, 1);
                if (dmode == 0) return WB_LEANW_M(0, 0);
                if (dmode == 1) return WB_LEANW_M(1, 0);
                if (dmode == 2) return WB_LEANW_M(2, 0);
#undef WB_LEANW_M
#undef WB_LEANW
            }
        }
        // float64 rows, and fp32 rows wider than one 16 KiB ring slot (column strips): the lean kernel on 24 KiB slots when a
        // staged row (strip + halo columns) fits one.  These launches stream footprints far beyond L2 and sit at what a
        // 1-read : 2-write stream reaches there (5.4 - 5.5 TB/s) with either kernel; measured (profiles/r2_wide_rows.json):
        // fp32 strips 2 - 11 % faster at d >= 4 (kept; d < 4 keeps the generic kernel), float64 K1 equal within 2 % except
        // with paired columns (d >= 16: 1 - 5 us faster, kept), float64 K3 12 - 22 us faster per 4096^2 plane except with
        // the soft threshold (the inlined double-precision erf: 10 us slower, generic kept).
        if (OP != OP_POWER && (sizeof(T) == 8 || p.n_strips > 1) && lean_ok && p.l2_hints &&
            (long long)p.row_stride * (long long)sizeof(T) <= (long long)kLeanStripKiB * 1024 &&
            // (only where the planner laid the segments out for ONE block per SM, which is what 24 KiB slots give)
            2 * ((long long)kLeanSlots * p.row_stride * (long long)sizeof(T) + 16 * kLeanSlots + 1024) > (long long)kMaxSmem) {
            const int cols = p.n_strips == 1 ? p.W : p.wt;
            const bool pair = dmode == 0 && k1_pair_step(p.d, cols, cfg.nt, V);
            if constexpr (OP == OP_POWER) {
            } else if constexpr (sizeof(T) == 4) {
                if (pair) return launch_rows_lean_strip<T, TAPS, 0, OP, 1>(p, batch, cfg.nt, st);
                if (dmode == 0) return launch_rows_lean_strip<T, TAPS, 0, OP, 0>(p, batch, cfg.nt, st);
            } else if constexpr (OP == OP_TRANSFORM) {
                if (pair) return launch_rows_lean_strip<T, TAPS, 0, OP, 1>(p, batch, cfg.nt, st);
            } else {
                if (p.sig_mode != 1) {
                    if (pair) return launch_rows_lean_strip<T, TAPS, 0, OP, 1>(p, batch, cfg.nt, st);
                    if (dmode == 0) return launch_rows_lean_strip<T, TAPS, 0, OP, 0>(p, batch, cfg.nt, st);
                    if (dmode == 1) return launch_rows_lean_strip<T, TAPS, 1, OP, 0>(p, batch, cfg.nt, st);
                }
            }
        }
#define WB_LAUNCH_M(DM, M)                                                              \
    (cfg.ng == 1 ? launch_rows<T, TAPS, DM, 1, OP, M>(p, batch, cfg.nt, st)             \
                 : launch_rows<T, TAPS, DM, 2, OP, M>(p, batch, cfg.nt, st))
#define WB_LAUNCH(DM) (map ? WB_LAUNCH_M(DM, OP == OP_WHITEN) : WB_LAUNCH_M(DM, false))
        if (dmode == 0) return WB_LAUNCH(0);
        if (dmode == 1) return WB_LAUNCH(1);
        if constexpr (V == 4) {
            if (dmode == 2) return WB_LAUNCH(2);
        }
#undef WB_LAUNCH
#undef WB_LAUNCH_M
    }
    const long long n = (long long)p.H * p.W;
    long long blocks = (n + 255) / 256;
    const long long cap = 32LL * device_sm_count();
    if (blocks > cap) blocks = cap;
    if (map) atrous_generic_kernel<T, TAPS, OP, OP == OP_WHITEN><<<dim3((unsigned)blocks, (unsigned)batch), 256, 0, st>>>(p);
    else atrous_generic_kernel<T, TAPS, OP><<<dim3((unsigned)blocks, (unsigned)batch), 256, 0, st>>>(p);
    return launch_status();
}

template <int OP>
static int dispatch_typed(ScaleParams &p, int batch, int scale, int taps, int dtype, cudaStream_t st) {
    if (dtype == WB_F32)
        return taps == 3 ? dispatch<float, 3, OP>(p, batch, scale, st) : dispatch<float, 5, OP>(p, batch, scale, st);
    return taps == 3 ? dispatch<double, 3, OP>(p, batch, scale, st) : dispatch<double, 5, OP>(p, batch, scale, st);
}

static int scale_impl(const void *in, void *out_c, void *out_w, int batch, int H, int W, long long in_pitch,
                      long long in_bstride, long long c_pitch, long long c_bstride, long long w_pitch,
                      long long w_bstride, int scale, int taps, int dtype, cudaStream_t st) {
    int rc = check_common(batch, H, W, taps, dtype);
    if (rc) return rc;
    if (scale < 0 || scale > 30) return WB_EINVAL_SCALE;
    if (!in || (!out_c && !out_w)) return WB_EINVAL_POINTER;
    if (in == out_c || in == out_w) return WB_EINVAL_POINTER;
    if (in_pitch < W || (out_c && c_pitch < W) || (out_w && w_pitch < W)) return WB_EINVAL_ARG;
    ScaleParams p;
    memset(&p, 0, sizeof(p));
    p.in = in; p.out_c = out_c; p.out_w = out_w;
    p.H = H; p.W = W; p.d = 1 << scale; p.Hg = H;
    p.in_pitch = in_pitch; p.in_bstride = in_bstride;
    p.c_pitch = c_pitch; p.c_bstride = c_bstride;
    p.w_pitch = w_pitch; p.w_bstride = w_bstride;
    p.l2_hints = l2_hints_enabled();
    return dispatch_typed<OP_TRANSFORM>(p, batch, scale, taps, dtype, st);
}

// OP_POWER: out = S_s[T(w * w)] of every frame (the local power of a volume's wow(), smoothed within each slice).
int atrous_power_slices(const void *w, void *out, int batch, int H, int W, int scale, int taps, int dtype, cudaStream_t st) {
    int rc = check_common(batch, H, W, taps, dtype);
    if (rc) return rc;
    if (scale < 0 || scale > 30) return WB_EINVAL_SCALE;
    if (!w || !out || w == out) return WB_EINVAL_POINTER;
    ScaleParams p;
    memset(&p, 0, sizeof(p));
    p.in = w; p.out_c = out;
    p.H = H; p.W = W; p.d = 1 << scale; p.Hg = H;
    p.in_pitch = W; p.in_bstride = (long long)H * W;
    p.c_pitch = W; p.c_bstride = (long long)H * W;
    p.l2_hints = l2_hints_enabled();
    return dispatch_typed<OP_POWER>(p, batch, scale, taps, dtype, st);
}

}  // namespace wb

extern "C" {

int wb_atrous_scale_path(int H, int W, long long in_pitch, long long out_pitch, int scale, int taps, int dtype,
                         const void *in, const void *out_c, const void *out_w) {
    if (wb::check_common(1, H, W, taps, dtype) || scale < 0 || scale > 30) return -1;
    wb::ScaleParams p;
    memset(&p, 0, sizeof(p));
    p.in = in; p.out_c = const_cast<void *>(out_c); p.out_w = const_cast<void *>(out_w);
    p.H = H; p.W = W; p.d = 1 << scale; p.Hg = H;
    p.in_pitch = in_pitch; p.c_pitch = out_pitch; p.w_pitch = out_pitch;
    const int esize = wb::dtype_size(dtype);
    return (wb::fast_path_ok(p, taps, esize) && wb::plan_fast(p, taps, esize, 1, scale, nullptr)) ? 1 : 0;
}

// Tuning hook (benchmark sweeps only): override the K1 geometry of one scale; nt == 0 clears the override.
int wb_tune_k1(int scale, int nt, int ng, int slots, int seg) {
    if (scale < 0 || scale >= 32) return WB_EINVAL_SCALE;
    if (nt == 0) { wb::g_override_set[scale] = false; return WB_OK; }
    wb::g_override[scale] = wb::K1Config{nt, ng, slots, seg};
    wb::g_override_set[scale] = true;
    return WB_OK;
}

int wb_atrous_scale(const void *in, void *out_c, void *out_w, int batch, int H, int W, long long in_pitch,
                    long long in_bstride, long long out_c_pitch, long long out_c_bstride, long long out_w_pitch,
                    long long out_w_bstride, int scale, int taps, int dtype, void *stream) {
    return wb::scale_impl(in, out_c, out_w, batch, H, W, in_pitch, in_bstride, out_c_pitch, out_c_bstride,
                          out_w_pitch, out_w_bstride, scale, taps, dtype, (cudaStream_t)stream);
}

int wb_atrous_scale_lattice(const void *in, void *out_c, void *out_w, int H, int W, long long in_pitch,
                            long long out_c_pitch, long long out_w_pitch, int scale, int taps, int dtype, void *stream) {
    int rc = wb::check_common(1, H, W, taps, dtype);
    if (rc) return rc;
    if (scale < 0 || scale > 30) return WB_EINVAL_SCALE;
    if (!in || (!out_c && !out_w) || in == out_c || in == out_w) return WB_EINVAL_POINTER;
    if (in_pitch < W || (out_c && out_c_pitch < W) || (out_w && out_w_pitch < W)) return WB_EINVAL_ARG;
    wb::ScaleParams p;
    memset(&p, 0, sizeof(p));
    p.in = in; p.out_c = out_c; p.out_w = out_w;
    p.H = H; p.W = W; p.d = 1 << scale; p.Hg = H;
    p.in_pitch = in_pitch; p.c_pitch = out_c_pitch; p.w_pitch = out_w_pitch;
    p.lattice = 1;
    const long long n = (long long)H * W;
    long long blocks = (n + 255) / 256;
    const long long cap = 32LL * wb::device_sm_count();
    if (blocks > cap) blocks = cap;
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid((unsigned)blocks, 1);
    if (dtype == WB_F32) {
        if (taps == 3) wb::atrous_generic_kernel<float, 3, wb::OP_TRANSFORM><<<grid, 256, 0, st>>>(p);
        else wb::atrous_generic_kernel<float, 5, wb::OP_TRANSFORM><<<grid, 256, 0, st>>>(p);
    } else {
        if (taps == 3) wb::atrous_generic_kernel<double, 3, wb::OP_TRANSFORM><<<grid, 256, 0, st>>>(p);
        else wb::atrous_generic_kernel<double, 5, wb::OP_TRANSFORM><<<grid, 256, 0, st>>>(p);
    }
    return wb::launch_status();
}

int wb_atrous_scale_band(const void *in, void *out_c, void *out_w, int band_rows, int W, int global_H,
                         long long band_y0, long long in_row_offset, long long in_pitch, long long out_c_row_offset,
                         long long out_c_pitch, long long out_w_row_offset, long long out_w_pitch, int scale, int taps,
                         int dtype, void *stream) {
    int rc = wb::check_common(1, band_rows, W, taps, dtype);
    if (rc) return rc;
    if (scale < 0 || scale > 30) return WB_EINVAL_SCALE;
    if (!in || (!out_c && !out_w) || in == out_c || in == out_w) return WB_EINVAL_POINTER;
    if (global_H < band_rows || band_y0 < 0 || band_y0 + band_rows > global_H || in_pitch < W ||
        (out_c && out_c_pitch < W) || (out_w && out_w_pitch < W))
        return WB_EINVAL_ARG;
    wb::ScaleParams p;
    memset(&p, 0, sizeof(p));
    p.in = in; p.out_c = out_c; p.out_w = out_w;
    p.H = band_rows; p.W = W; p.d = 1 << scale; p.Hg = global_H;
    p.gwy0 = band_y0; p.row_off_in = in_row_offset; p.row_off_c = out_c_row_offset; p.row_off_w = out_w_row_offset;
    p.in_pitch = in_pitch; p.c_pitch = out_c_pitch; p.w_pitch = out_w_pitch;
    return wb::dispatch_typed<wb::OP_TRANSFORM>(p, 1, scale, taps, dtype, (cudaStream_t)stream);
}

int wb_atrous_scale_band_push(const void *in, void *out_c, void *out_w, int band_rows, int W, int global_H,
                              long long band_y0, long long in_row_offset, long long in_pitch, long long out_c_row_offset,
                              long long out_c_pitch, long long out_w_row_offset, long long out_w_pitch, void *push_up,
                              int push_up_rows, void *push_dn, int push_dn_rows, int scale, int taps, int dtype,
                              void *stream) {
    int rc = wb::check_common(1, band_rows, W, taps, dtype);
    if (rc) return rc;
    if (scale < 0 || scale > 30) return WB_EINVAL_SCALE;
    if (!in || !out_c || in == out_c || in == out_w) return WB_EINVAL_POINTER;
    if (global_H < band_rows || band_y0 < 0 || band_y0 + band_rows > global_H || in_pitch < W || out_c_pitch < W ||
        (out_w && out_w_pitch < W) || push_up_rows < 0 || push_dn_rows < 0)
        return WB_EINVAL_ARG;
    if ((push_up && (push_up == out_c || push_up == in)) || (push_dn && (push_dn == out_c || push_dn == in)))
        return WB_EINVAL_POINTER;
    wb::ScaleParams p;
    memset(&p, 0, sizeof(p));
    p.in = in; p.out_c = out_c; p.out_w = out_w;
    p.H = band_rows; p.W = W; p.d = 1 << scale; p.Hg = global_H;
    p.gwy0 = band_y0; p.row_off_in = in_row_offset; p.row_off_c = out_c_row_offset; p.row_off_w = out_w_row_offset;
    p.in_pitch = in_pitch; p.c_pitch = out_c_pitch; p.w_pitch = out_w_pitch;
    p.push_up = push_up_rows > 0 ? push_up : nullptr;
    p.push_dn = push_dn_rows > 0 ? push_dn : nullptr;
    p.push_up_rows = push_up_rows < band_rows ? push_up_rows : band_rows;
    p.push_dn_from = push_dn_rows < band_rows ? band_rows - push_dn_rows : 0;
    p.l2_hints = wb::l2_hints_enabled();
    return wb::dispatch_typed<wb::OP_TRANSFORM>(p, 1, scale, taps, dtype, (cudaStream_t)stream);
}

int wb_atrous_scale_band_p2p(const void *const *peer_in, const long long *peer_y0, int n_peers, int rank,
                             void *out_c, void *out_w, int W, int global_H, long long in_pitch,
                             long long out_c_pitch, long long out_w_pitch, int scale, int taps, int dtype,
                             void *stream) {
    if (!peer_in || !peer_y0) return WB_EINVAL_POINTER;
    if (n_peers < 1 || n_peers > WB_MAX_PEERS || rank < 0 || rank >= n_peers) return WB_EINVAL_ARG;
    if (peer_y0[0] != 0 || peer_y0[n_peers] != global_H) return WB_EINVAL_ARG;
    for (int k = 0; k < n_peers; ++k) {
        if (peer_y0[k + 1] <= peer_y0[k]) return WB_EINVAL_ARG;  // every rank owns at least one row
        if (!peer_in[k] || peer_in[k] == out_c || peer_in[k] == out_w) return WB_EINVAL_POINTER;
    }
    const long long band_rows = peer_y0[rank + 1] - peer_y0[rank];
    if (band_rows > 0x7fffffffLL) return WB_EINVAL_SHAPE;
    int rc = wb::check_common(1, (int)band_rows, W, taps, dtype);
    if (rc) return rc;
    if (scale < 0 || scale > 30) return WB_EINVAL_SCALE;
    if (!out_c && !out_w) return WB_EINVAL_POINTER;
    if (in_pitch < W || (out_c && out_c_pitch < W) || (out_w && out_w_pitch < W)) return WB_EINVAL_ARG;
    wb::ScaleParams p;
    memset(&p, 0, sizeof(p));
    p.in = peer_in[rank]; p.out_c = out_c; p.out_w = out_w;
    p.H = (int)band_rows; p.W = W; p.d = 1 << scale; p.Hg = global_H;
    p.gwy0 = peer_y0[rank];
    p.in_pitch = in_pitch; p.c_pitch = out_c_pitch; p.w_pitch = out_w_pitch;
    p.n_peers = n_peers;
    for (int k = 0; k < n_peers; ++k) {
        p.peer_in[k] = peer_in[k];
        p.peer_y0[k] = peer_y0[k];
        // the vector path needs every window 16-byte aligned; otherwise the generic kernel takes the launch
        if (!wb::aligned16(peer_in[k])) p.in = peer_in[k];
    }
    p.peer_y0[n_peers] = peer_y0[n_peers];
    p.l2_hints = wb::l2_hints_enabled();
    return wb::dispatch_typed<wb::OP_TRANSFORM>(p, 1, scale, taps, dtype, (cudaStream_t)stream);
}

int wb_wow_whiten_scale(const void *w_raw, void *out, int batch, int H, int W, long long in_pitch,
                        long long in_bstride, long long out_pitch, long long out_bstride, int scale, int taps,
                        int dtype, int sig_mode, double sigma, double sigma_e, double noise_host,
                        const double *noise_dev, double weight, void *stream) {
    int rc = wb::check_common(batch, H, W, taps, dtype);
    if (rc) return rc;
    if (scale < 0 || scale > 30) return WB_EINVAL_SCALE;
    if (!w_raw || !out || w_raw == out) return WB_EINVAL_POINTER;
    if (in_pitch < W || out_pitch < W || sig_mode < 0 || sig_mode > 2) return WB_EINVAL_ARG;
    wb::ScaleParams p;
    memset(&p, 0, sizeof(p));
    p.in = w_raw; p.out_c = nullptr; p.out_w = out;
    p.H = H; p.W = W; p.d = 1 << scale; p.Hg = H;
    p.in_pitch = in_pitch; p.in_bstride = in_bstride;
    p.w_pitch = out_pitch; p.w_bstride = out_bstride;
    p.sig_mode = sig_mode; p.sigma = sigma; p.sigma_e = sigma_e;
    p.noise_host = noise_host; p.noise_dev = noise_dev; p.weight = weight;
    p.l2_hints = wb::l2_hints_enabled();
    return wb::dispatch_typed<wb::OP_WHITEN>(p, batch, scale, taps, dtype, (cudaStream_t)stream);
}

int wb_wow_whiten_scale_map(const void *w_raw, void *out, const void *noise_map, int batch, int H, int W,
                            long long in_pitch, long long in_bstride, long long out_pitch, long long out_bstride,
                            long long map_pitch, long long map_bstride, int scale, int taps, int dtype, int soft,
                            double sigma, double sigma_e, double weight, void *stream) {
    int rc = wb::check_common(batch, H, W, taps, dtype);
    if (rc) return rc;
    if (scale < 0 || scale > 30) return WB_EINVAL_SCALE;
    if (!w_raw || !out || !noise_map || w_raw == out || noise_map == out) return WB_EINVAL_POINTER;
    if (in_pitch < W || out_pitch < W || map_pitch < W || map_bstride < 0 || sigma == 0.0) return WB_EINVAL_ARG;
    wb::ScaleParams p;
    memset(&p, 0, sizeof(p));
    p.in = w_raw; p.out_c = nullptr; p.out_w = out;
    p.H = H; p.W = W; p.d = 1 << scale; p.Hg = H;
    p.in_pitch = in_pitch; p.in_bstride = in_bstride;
    p.w_pitch = out_pitch; p.w_bstride = out_bstride;
    p.sig_mode = wb::SIG_MAP; p.sigma = sigma; p.sigma_e = sigma_e; p.weight = weight;
    p.noise_map = noise_map; p.map_pitch = map_pitch; p.map_bstride = map_bstride; p.map_soft = soft ? 1 : 0;
    p.l2_hints = wb::l2_hints_enabled();
    return wb::dispatch_typed<wb::OP_WHITEN>(p, batch, scale, taps, dtype, (cudaStream_t)stream);
}

int wb_wow_whiten_scale_band(const void *w_raw, void *out, int band_rows, int W, int global_H, long long band_y0,
                             long long in_row_offset, long long in_pitch, long long out_row_offset, long long out_pitch,
                             int scale, int taps, int dtype, int sig_mode, double sigma, double sigma_e,
                             double noise_host, const double *noise_dev, double weight, void *stream) {
    int rc = wb::check_common(1, band_rows, W, taps, dtype);
    if (rc) return rc;
    if (scale < 0 || scale > 30) return WB_EINVAL_SCALE;
    if (!w_raw || !out || w_raw == out) return WB_EINVAL_POINTER;
    if (global_H < band_rows || band_y0 < 0 || band_y0 + band_rows > global_H || in_pitch < W || out_pitch < W ||
        sig_mode < 0 || sig_mode > 2)
        return WB_EINVAL_ARG;
    wb::ScaleParams p;
    memset(&p, 0, sizeof(p));
    p.in = w_raw; p.out_c = nullptr; p.out_w = out;
    p.H = band_rows; p.W = W; p.d = 1 << scale; p.Hg = global_H;
    p.gwy0 = band_y0; p.row_off_in = in_row_offset; p.row_off_w = out_row_offset;
    p.in_pitch = in_pitch; p.w_pitch = out_pitch;
    p.sig_mode = sig_mode; p.sigma = sigma; p.sigma_e = sigma_e;
    p.noise_host = noise_host; p.noise_dev = noise_dev; p.weight = weight;
    return wb::dispatch_typed<wb::OP_WHITEN>(p, 1, scale, taps, dtype, (cudaStream_t)stream);
}

int wb_atrous_transform(const void *in, void *planes, void *scratch, int batch, int H, int W, long long in_pitch,
                        long long in_bstride, int levels, int taps, int dtype, void *stream) {
    int rc = wb::check_common(batch, H, W, taps, dtype);
    if (rc) return rc;
    if (levels < 0 || levels > 30) return WB_EINVAL_SCALE;
    if (!in || !planes || (levels > 1 && !scratch)) return WB_EINVAL_POINTER;
    if (in_pitch < W) return WB_EINVAL_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t es = (size_t)wb::dtype_size(dtype);
    const long long plane = (long long)H * W;
    const long long fstride = (long long)(levels + 1) * plane;  // frame stride inside `planes`
    char *pl = reinterpret_cast<char *>(planes);
    char *sc = reinterpret_cast<char *>(scratch);
    if (levels == 0) {
        cudaError_t e = cudaMemcpy2DAsync(pl, (size_t)W * es, in, (size_t)in_pitch * es, (size_t)W * es, (size_t)H,
                                          cudaMemcpyDeviceToDevice, st);
        for (int b = 1; b < batch && e == cudaSuccess; ++b)
            e = cudaMemcpy2DAsync(pl + (size_t)b * fstride * es, (size_t)W * es,
                                  reinterpret_cast<const char *>(in) + (size_t)b * in_bstride * es,
                                  (size_t)in_pitch * es, (size_t)W * es, (size_t)H, cudaMemcpyDeviceToDevice, st);
        return (int)e;
    }
    for (int s = 0; s < levels; ++s) {
        // c_s: the image itself for s == 0, else the scratch half written by the previous scale
        const void *src = (s == 0) ? in : (const void *)(sc + (size_t)((s - 1) & 1) * batch * plane * es);
        const long long src_pitch = (s == 0) ? in_pitch : W;
        const long long src_bstride = (s == 0) ? in_bstride : plane;
        // c_{s+1}: the other scratch half, or plane L of the output for the last scale
        const bool last = (s == levels - 1);
        void *dst_c = last ? (void *)(pl + (size_t)levels * plane * es) : (void *)(sc + (size_t)(s & 1) * batch * plane * es);
        const long long c_bstride = last ? fstride : plane;
        void *dst_w = pl + (size_t)s * plane * es;
        rc = wb::scale_impl(src, dst_c, dst_w, batch, H, W, src_pitch, src_bstride, W, c_bstride, W, fstride, s, taps,
                            dtype, st);
        if (rc) return rc;
    }
    return WB_OK;
}

}  // extern "C"
