// drs_pair2d.cuh -- TWO single-step 2D sweeps in one launch, bit for bit (drs_run on 2D plans after drs_plan_set_pairs).
//
// drs_run's ping-pong schedule on a step-1 plan reads and writes the whole grid once per timestep.  This kernel
// advances the grid by two timesteps per HBM round trip and leaves in the interior of its output exactly what two
// launches of the single-step kernel would leave there.  It is the scatter machine of drs_sweep2d.cuh at DRS_TS == 2 --
// one warp per (x strip, row chunk), the per-warp TMA row ring with one mbarrier per stage, partial sums w[2][2RJ+1][C]
// in registers with the levels evaluated top-down, level 1's column halo exchanged by shuffle, strips overlapping by
// 2 * HW -- with what the single-step semantics needs instead of the composed operator's:
//   * the frozen ring is that of ONE step (H = Halo of the plan, not 2 * Halo): level 2 is stored on rows [H, M-H) and
//     columns [H, N-H);
//   * DRS_SCATTER is the exact scatter (generate.hpp: emit_scatter2_exact): every point of both levels is evaluated
//     with the single-step chain DRS_CHAIN, same literals, same order; no row factorisation, no deferred scale;
//   * the ring cells of each level are the ring of the buffer that level lives in.  drs_run's level l is the interior
//     written by sweep l-1 together with the ring of bufs[l % 2]: a pair starts from an even level (ring of A) and
//     passes through an odd one (ring of B).  So
//       - level 0: when the input is B, the ring rows (y < H, y >= M-H) and ring columns (x < H, x >= N-H) of every
//         staged row are overwritten with A's cells as soon as the stage has arrived;
//       - level 1: every ring cell of the row a thread has just completed is replaced by B's cell before anything
//         reads it (the level-2 scatter, an operand parked in a partial-sum slot, the shuffles).
//     Only warps whose box reaches into the ring do any of this (warp-uniform branches).
//
// Stage lifecycle: a stage that holds generic writes of the level-0 patch is fenced (fence.proxy.async by every lane
// that wrote, then __syncwarp) before anything else happens to it; it is handed back to the TMA unit after the warp's
// last read of it, exactly as in s2d::iteration.  Every wait is the time-bounded mbar_wait.
//
// The kernel reuses drs_sweep2d.cuh's constants (at DRS_TS == 2), Stream, Tile, load_row and store_row; the row loop
// below carries a copy of s2d::iteration's stage handling and of s2d::row_step's shuffles (test_exact_pairs2d.py keeps
// the copies identical).  drs_sweep2d.cuh also instantiates its own kernel under DRS_NAME; that one is never launched.
//
// Generated translation unit must define: DRS_T DRS_PAIR_NAME DRS_NAME DRS_RJ DRS_E DRS_TS (= 2) DRS_NW DRS_ST DRS_RB
// DRS_VT DRS_MINB DRS_SCATTER(P,U).
#pragma once
#include "drs_sweep2d.cuh"

#if DRS_FLAT
#error "the exact 2D pair kernel needs a 16-byte row pitch (tensor-map row boxes)"
#endif

namespace drs {
namespace s2p {

using s2d::C;
using s2d::DEPTH;
using s2d::E;
using s2d::E0;
using s2d::HW;
using s2d::NW;
using s2d::R2;
using s2d::RB;
using s2d::RJ;
using s2d::RP;
using s2d::ST;
using s2d::STAGE_STRIDE;
using s2d::VW;
using s2d::WARP_SMEM;
using s2d::WB;
using s2d::WT;
using s2d::WU;
using s2d::mod_r2;
using s2d::Stream;
using s2d::Tile;
static_assert(s2d::TS == 2 && s2d::NLV == 2 && s2d::SW == C, "two levels of partial sums");

// Where the ring cells of the two levels come from
struct Ring {
    const real* a;      // level 0's ring (when the input is B)
    const real* b;      // level 1's ring
    int M, N, H;        // (extents below 2^31: capi.cpp check_sizes)
    int yrow0;          // input row of iteration 0
    int n1_lo, n1_hi;   // iterations that complete a level-1 row outside the ring rows: n1_lo <= n < n1_hi
    bool patch0;        // the input is B: level 0's ring cells are patched in from A
    bool edge0_x;       // the warp's TMA box reaches into the ring columns
    bool edge1_x;       // the warp's level-1 columns [X0, X0 + WT) reach into the ring columns
    // whether iteration n completes a level-1 row with ring cells in this warp's columns (warp-uniform)
    __device__ __forceinline__ bool ring1(int n) const { return edge1_x || n < n1_lo || n >= n1_hi; }
};

// B's cells of the level-1 row completed by iteration n, in this thread's columns: ring cells in `v`, the rest untouched.
// Loaded one iteration ahead (row_step), so that the load's latency hides behind a whole row of arithmetic.  Ring cells
// are never written by a sweep, so both rings are read-only for the kernel's lifetime (ld.global.nc).
__device__ __forceinline__ void load_ring1(const Ring& g, const Tile& t, int n, real (&v)[C]) {
    const int y1 = g.yrow0 + n - RJ;
    if (y1 < 0 || y1 >= g.M) return;
    const bool ring_row = y1 < g.H || y1 >= g.M - g.H;
    const real* pb = g.b + (drs_i64)y1 * g.N;
#pragma unroll
    for (int k = 0; k < C; ++k) {
        const int gx = t.x_first + k;
        if (gx >= 0 && gx < g.N && (ring_row || gx < g.H || gx >= g.N - g.H)) v[k] = __ldg(pb + gx);
    }
}

// Level 0, input B: A's ring rows and ring columns of the staged rows y0 .. y0 + RB - 1.  Every lane takes part.
__device__ __forceinline__ void patch_level0(const Ring& g, const Stream& st, real* stage, int y0) {
    // (rows unrolled: the loads of a stage are in flight together)
#pragma unroll
    for (int r = 0; r < RB; ++r) {
        const int gy = y0 + r;
        if (gy < 0 || gy >= g.M) continue;
        const real* pa = g.a + (drs_i64)gy * g.N;
        real* row = stage + r * RP;
        if (gy < g.H || gy >= g.M - g.H) {
            for (int bx = st.lane; bx < WB; bx += 32) {
                const int gx = st.x_box + bx;
                if (gx >= 0 && gx < g.N) row[bx] = __ldg(pa + gx);
            }
        } else if (g.edge0_x) {
            for (int q = st.lane; q < 2 * g.H; q += 32) {
                const int gx = q < g.H ? q : g.N - 2 * g.H + q;
                const int bx = gx - st.x_box;
                if (bx >= 0 && bx < WB && gx >= 0 && gx < g.N) row[bx] = __ldg(pa + gx);
            }
        }
    }
    fence_proxy_async();     // generic writes to a stage the TMA unit refills later
    __syncwarp();
}

// One iteration of the row pipeline; PH = iteration mod R2 (compile-time: static rotation).  Input row yrow0 + n
// enters level 1; level-1 row yrow0 + n - RJ completes and takes its ring cells from B; level-2 row y_out0 + n
// completes and is stored.
template <int PH>
__device__ __forceinline__ void row_step(real (&w)[2][R2][C], real (&rb)[C], const real* __restrict__ srow, const Tile& t,
                                         const Ring& g, int n) {
#pragma unroll
    for (int s = 2; s >= 1; --s) {
        real u[VW];
        if (s == 1) {
            s2d::load_row(u, srow, t.lane);
        } else {
            // the level s-1 row completed by the previous iteration; neighbours by shuffle
            const real (&src)[C] = w[0][mod_r2(PH - 1 - RJ)];
#pragma unroll
            for (int v = 0; v < C; ++v) u[E + v] = src[v];
#pragma unroll
            for (int e = 0; e < E; ++e) {
                u[e] = __shfl_up_sync(0xffffffffu, src[C - E + e], 1);
                u[E + C + e] = __shfl_down_sync(0xffffffffu, src[e], 1);
            }
        }
#pragma unroll
        for (int v = 0; v < C; ++v) {
#define DRS_U_(di) u[E + v + (di)]
#define DRS_P_(dj) w[s - 1][mod_r2(PH - (dj))][v]
            DRS_SCATTER(DRS_P_, DRS_U_)
#undef DRS_U_
#undef DRS_P_
        }
        if (s == 1) {
            // ---- the row of level 1 completed by this iteration: its ring cells are B's (rb, loaded by the previous
            //      iteration), then the next iteration's cells are requested ----
            if (g.ring1(n)) {                         // warp-uniform
                const int y1 = g.yrow0 + n - RJ;
                if (y1 >= 0 && y1 < g.M) {
                    const bool ring_row = y1 < g.H || y1 >= g.M - g.H;
#pragma unroll
                    for (int v = 0; v < C; ++v) {
                        const int gx = t.x_first + v;
                        if (gx >= 0 && gx < g.N && (ring_row || gx < g.H || gx >= g.N - g.H)) w[0][mod_r2(PH - RJ)][v] = rb[v];
                    }
                }
            }
            if (g.ring1(n + 1)) load_ring1(g, t, n + 1, rb);
        } else if (n >= t.n_first && n < t.n_end) {
            // ---- level 2: the output row ----
            real o[C];
#pragma unroll
            for (int v = 0; v < C; ++v) o[v] = w[1][mod_r2(PH - RJ)][v];
            s2d::store_row(t, n, o);
        }
    }
}

// One input row: wait for its stage (and patch it) if it is the stage's first row, run the row through both levels,
// hand the stage back to the TMA unit if it was the stage's last row.
template <int PH>
__device__ __forceinline__ bool iteration(real (&w)[2][R2][C], real (&rb)[C], const Stream& st, const Tile& t, const Ring& g,
                                          int n) {
    const int rr = n & (RB - 1);
    const int c = n / RB;
    const int s = c & (ST - 1);
    if (rr == 0) {
        if (!mbar_wait(&st.bars[s], (drs_u32)((c / ST) & 1), st.fault)) return false;
        const int y0 = st.yrow0 + c * RB;
        if (g.patch0 && (g.edge0_x || y0 < g.H || y0 + RB > g.M - g.H))     // warp-uniform
            patch_level0(g, st, reinterpret_cast<real*>(st.wbase + s * STAGE_STRIDE), y0);
    }
    const real* srow = reinterpret_cast<const real*>(st.wbase + s * STAGE_STRIDE) + rr * RP;
    row_step<PH>(w, rb, srow, t, g, n);
    if (rr == RB - 1) {
        __syncwarp();
        if (st.lane == 0 && c + ST < st.NCH) {
            fence_proxy_async();
            st.issue(c + ST);
        }
    }
    return true;
}

// R2 consecutive rows with the phase known at compile time (static register rotation)
template <int PH>
__device__ __forceinline__ bool phases(real (&w)[2][R2][C], real (&rb)[C], const Stream& st, const Tile& t, const Ring& g,
                                       int n0) {
    if constexpr (PH < R2) {
        if (!iteration<PH>(w, rb, st, t, g, n0 + PH)) return false;
        return phases<PH + 1>(w, rb, st, t, g, n0);
    } else {
        return true;
    }
}

__device__ __forceinline__ void sweep(const TensorMap& tmap, const Params& p, const real* ring_a, const real* ring_b) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const drs_i64 tile = (drs_i64)blockIdx.x * NW + warp;
    if (tile >= (drs_i64)p.nxs * p.nys) return;
    const int xs = (int)(tile % p.nxs);
    const int yc = (int)(tile / p.nxs);

    Stream st;
    st.wbase = smem_raw + warp * WARP_SMEM;
    st.bars = reinterpret_cast<drs_u64*>(smem_raw + NW * WARP_SMEM) + warp * ST;
    st.tmap = &tmap;
    st.fault = p.fault;
    st.lane = lane;
    st.in = p.in;
    st.M = p.M;
    st.N = p.N;
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < ST; ++s) mbar_init(&st.bars[s], 1);
        fence_mbar_init();
        fence_proxy_async();
    }
    __syncwarp();

    const int H = p.halo;
    const int X0 = (H / kVec) * kVec + xs * WU - HW;   // column of lane 0, element 0
    const drs_i64 ya = p.slow_lo + (drs_i64)yc * p.chunk;
    const drs_i64 yb = (ya + p.chunk < p.slow_hi) ? ya + p.chunk : p.slow_hi;
    // iterations: chunk rows + pipeline depth, rounded up to whole rotations so that the unrolled phases need no guard;
    // the surplus iterations stream rows past the chunk (or zero fill) and store nothing
    const int n_end = (int)(yb - ya) + DEPTH;
    st.NIT = (n_end + R2 - 1) / R2 * R2;
    st.NCH = (st.NIT + RB - 1) / RB;
    st.yrow0 = (int)(ya - 2 * RJ);                      // first input row the chunk depends on
    st.x_box = X0 - E0;

    Tile t;
    t.lane = lane;
    t.x_first = X0 + lane * C;
    {
        const drs_i64 lo = (H > X0 + HW) ? H : X0 + HW;
        const drs_i64 hi = (p.N - H < X0 + HW + WU) ? p.N - H : X0 + HW + WU;
        t.v_lo = (int)(lo - t.x_first);
        t.v_hi = (int)(hi - t.x_first);
    }
    t.n_first = DEPTH;
    t.n_end = n_end;
    t.y_out0 = ya - DEPTH;
    t.N = p.N;
    t.out = p.out;

    Ring g;
    g.a = ring_a;
    g.b = ring_b;
    g.M = (int)p.M;
    g.N = (int)p.N;
    g.H = H;
    g.yrow0 = st.yrow0;
    g.n1_lo = H - st.yrow0 + RJ;            // y1 = yrow0 + n - RJ >= H
    g.n1_hi = g.M - H - st.yrow0 + RJ;      // y1 < M - H
    g.patch0 = p.in != ring_a;
    g.edge0_x = st.x_box < H || st.x_box + WB > g.N - H;
    g.edge1_x = X0 < H || X0 + WT > g.N - H;

    if (lane == 0) {
        for (int c = 0; c < ST && c < st.NCH; ++c) st.issue(c);
    }

    real w[2][R2][C];
#pragma unroll
    for (int s = 0; s < 2; ++s)
#pragma unroll
        for (int r = 0; r < R2; ++r)
#pragma unroll
            for (int x = 0; x < C; ++x) w[s][r][x] = (real)0;
    real rb[C];             // B's ring cells of the level-1 row the next iteration completes
#pragma unroll
    for (int x = 0; x < C; ++x) rb[x] = (real)0;
    if (g.ring1(0)) load_ring1(g, t, 0, rb);

#pragma unroll 1
    for (int n0 = 0; n0 < st.NIT; n0 += R2) {
        if (!phases<0>(w, rb, st, t, g, n0)) return;
    }
}

}  // namespace s2p
}  // namespace drs

// Same parameter list as the 3D drpair_ (one launch path): tmap_a is not read here, A's ring cells are patched in by
// generic loads from ring_a.
extern "C" __global__ void __launch_bounds__(DRS_NW * 32, DRS_MINB)
DRS_PAIR_NAME(const __grid_constant__ drs::TensorMap tmap, const __grid_constant__ drs::TensorMap tmap_a,
              const __grid_constant__ drs::Params p, const DRS_T* ring_a, const DRS_T* ring_b) {
    drs::s2p::sweep(tmap, p, ring_a, ring_b);
}
