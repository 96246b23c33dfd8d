// drs_slabpair3d.cuh -- the slab entry of the exact pair kernel: TWO single-step 3D sweeps of a slab with DEEP ghost
// regions (drs_plan_set_slab_pairs: 2 * Halo planes per side) in one launch, bit for bit, with the halo push and the
// in-kernel step flags of drs_run_slab.
//
// The arithmetic is that of kernels/pair/drs_pair3d.cuh, whose plane loop this header carries a copy of (the scatter,
// the shuffles, the publication of level 1 and the stage lifecycle are the same text; tests/test_exact_slabpair.py
// keeps them so).  What differs:
//   * the input is the whole local array, deep ghost planes included: they hold the neighbours' planes of the input
//     level.  Level 1 is computed wherever its inputs are in the array, so on the ghost planes [Halo, 2 * Halo) next
//     to an interior face as well (redundantly, from the neighbour's data); it stays in registers as in drpair_;
//   * the frozen ring along the slow axis is the GLOBAL one: ring planes are those outside [ring_lo, ring_hi) in local
//     coordinates (the global planes [0, Halo) and [G - Halo, G), and the out-of-grid ghost planes of the first and
//     last rank).  Level 0 of such planes comes through A's tensor map, level 1 is B's cell, as drpair_ does with the
//     array's own edge planes.  At an interior face nothing is ring; the lateral ring (rows, columns) is unchanged;
//   * the output planes [push_lo0, push_lo1) / [push_hi0, push_hi1) (the 2 * Halo owned planes next to a neighbour) are
//     stored a second time into that neighbour's deep ghost planes (Params::peer_lo / peer_hi);
//   * with the step flags of drs_run_slab (Params::my_flags), chunks run face first (slab_chunk_order); thread 0 of a
//     face CTA waits for the neighbours before the first TMA request and the CTA shares its verdict, and after the
//     CTA's last store thread 0 arrives on the face counter.  The unit of the protocol is the CTA.
// DESIGN.md section 5 has the correctness argument (face rule, surplus planes, flag hazards).
//
// Generated translation unit must define: DRS_T DRS_SLABPAIR_NAME DRS_RK DRS_RJ DRS_E DRS_NW DRS_RY DRS_ST DRS_MINB
// DRS_SCATTER3(P,U).
#pragma once
#include "drs_common.cuh"

#if DRS_FLAT
#error "the exact pair kernel needs a 16-byte row pitch (tensor-map plane boxes)"
#endif

namespace drs {
namespace s3sp {

constexpr int RK = DRS_RK, RJ = DRS_RJ, E = DRS_E;
constexpr int K2 = 2 * RK + 1;
constexpr int RY = DRS_RY, NW = DRS_NW, ST = DRS_ST, NT = NW * 32;
constexpr int E0 = ((E + kVec - 1) / kVec) * kVec;
constexpr int HW = E0;                        // columns lost per side (one intermediate level)
constexpr int HY = RJ;                        // rows lost per side
constexpr int WT = 32 * kVec, WU = WT - 2 * HW, WB = WT + 2 * E0;
constexpr int TY = NW * RY, TYU = TY - 2 * HY, YB = TY + 2 * RJ;
constexpr int RP = WB;                        // row pitch of every plane in shared memory
constexpr int PLANE_BYTES = WB * YB * (int)sizeof(real);
constexpr int PLANE_STRIDE = (RP * YB * (int)sizeof(real) + 127) / 128 * 128;
constexpr int DEPTH = 4 * RK + 1;             // iterations from a chunk's first input plane to its first output plane
static_assert(ST >= 2, "at least two stages");
static_assert(WU > 0 && TYU > 0, "tile too small");
__device__ __forceinline__ int ring_slot(int n) { return (ST & (ST - 1)) == 0 ? (n & (ST - 1)) : n % ST; }
__device__ __forceinline__ drs_u32 ring_phase(int n) { return (drs_u32)((n / ST) & 1); }
__device__ __forceinline__ constexpr int mod_k2(int v) { return ((v % K2) + K2) % K2; }
__device__ __forceinline__ constexpr int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

struct Ctx {
    unsigned char* ring;     // ST input planes
    unsigned char* lv;       // 2 published planes of level 1 (by iteration parity)
    drs_u64* bars;
    const TensorMap* tmap;   // the input buffer
    const TensorMap* tmap_a; // A: level-0 ring planes
    int* fault;
    int x_box, y_box, z0;    // TMA coordinates of iteration 0
    int NIT;
    int warp, lane;
    int x_first, v_lo, v_hi;
    int y_first;             // global row of this warp's tile row 0
    int y_lo, y_hi;          // storable tile rows of this warp: y_lo <= y < y_hi
    drs_i64 z_out0;
    int n_first, n_end;
    int H, L, M, N;
    int ring_lo, ring_hi;    // local planes outside [ring_lo, ring_hi) are global ring (or out-of-grid) planes; 0 <= ring_lo <= ring_hi <= L
    bool edge;               // the CTA's box reaches into the ring rows / columns (CTA-uniform)
    bool patch0;             // edge, and the input is B: level-0 ring rows / columns come from A
    real* out;
    const real* ring_a;
    const real* ring_b;
    // peer stores: output planes [lo0, lo1) also go to plane z + lo_shift of peer_lo, likewise for peer_hi
    real* peer_lo; real* peer_hi;
    drs_i64 lo0, lo1, lo_shift, hi0, hi1, hi_shift;
    __device__ __forceinline__ void issue(int n) const {
        const int s = ring_slot(n);
        const int z = z0 + n;
        mbar_expect_tx(&bars[s], PLANE_BYTES);
        tma_load_3d(ring + s * PLANE_STRIDE, (z < ring_lo || z >= ring_hi) ? tmap_a : tmap, x_box, y_box, z, &bars[s]);
    }
};

// Level 0, input B: A's ring rows [0, H) / [M-H, M) and ring columns [0, H) / [N-H, N) of staged plane z.  Every thread
// of the CTA takes part; the plane is read by all warps after the barrier.
__device__ __forceinline__ void patch_level0(const Ctx& c, real* stage, int z) {
    const real* pa = c.ring_a + (drs_i64)z * c.M * c.N;
    const int H = c.H, rows = 2 * H * WB, total = rows + 2 * H * YB;
    for (int q = (int)threadIdx.x; q < total; q += NT) {
        int by, bx;
        if (q < rows) {
            const int r = q / WB;
            by = (r < H ? r : c.M - 2 * H + r) - c.y_box;
            bx = q % WB;
        } else {
            const int q2 = q - rows, cc = q2 / YB;
            bx = (cc < H ? cc : c.N - 2 * H + cc) - c.x_box;
            by = q2 % YB;
        }
        const int gy = c.y_box + by, gx = c.x_box + bx;
        if (by >= 0 && by < YB && bx >= 0 && bx < WB && gy >= 0 && gy < c.M && gx >= 0 && gx < c.N)
            stage[by * RP + bx] = pa[(drs_i64)gy * c.N + gx];
    }
    fence_proxy_async();     // generic writes to a stage the TMA unit refills later
    __syncthreads();
}

template <int PH>
__device__ __forceinline__ bool iteration(real (&pw)[2][K2][RY][kVec], const Ctx& c, int n) {
#pragma unroll
    for (int s = 2; s >= 1; --s) {
        // ---- source plane of level s-1 as this thread sees it: own rows/columns + neighbours ----
        const real* src;
        if (s == 1) {
            if (!mbar_wait(&c.bars[ring_slot(n)], ring_phase(n), c.fault)) return false;
            real* stage = reinterpret_cast<real*>(c.ring + ring_slot(n) * PLANE_STRIDE);
            const int z = c.z0 + n;
            if (c.patch0 && z >= c.ring_lo && z < c.ring_hi) patch_level0(c, stage, z);     // CTA-uniform
            src = stage;
        } else {
            src = reinterpret_cast<const real*>(c.lv + ((n + 1) & 1) * PLANE_STRIDE);
        }
        const real* mine = src + (c.warp * RY + RJ) * RP + E0 + c.lane * kVec;   // tile row 0, element 0
        // ---- scatter into the partial sums of level s (operands as in drs_sweep3d_t.cuh, DRS_T3_OWNREG 4) ----
        // level 2: the thread's own part of level 1 is still in its registers, the column halo comes from the
        // adjacent lanes; level 1: the input plane's own vectors are loaded once and the column halo is shuffled
        real xl[RY][E > 0 ? E : 1], xr[RY][E > 0 ? E : 1];
        if (s == 2) {
#pragma unroll
            for (int y = 0; y < RY; ++y)
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    xl[y][e] = __shfl_up_sync(0xffffffffu, pw[0][mod_k2(PH - 1 - RK)][y][kVec - E + e], 1);
                    xr[y][e] = __shfl_down_sync(0xffffffffu, pw[0][mod_k2(PH - 1 - RK)][y][e], 1);
                }
        }
        real u0[RY][kVec];
        if (s == 1) {
#pragma unroll
            for (int y = 0; y < RY; ++y) lds_vec(u0[y], mine + y * RP);
#pragma unroll
            for (int y = 0; y < RY; ++y)
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    xl[y][e] = __shfl_up_sync(0xffffffffu, u0[y][kVec - E + e], 1);
                    xr[y][e] = __shfl_down_sync(0xffffffffu, u0[y][e], 1);
                    if constexpr (HW < 2 * E) {
                        if (c.lane == 0) xl[y][e] = mine[y * RP - E + e];
                        if (c.lane == 31) xr[y][e] = mine[y * RP + kVec + e];
                    }
                }
        }
#define DRS_XNBR_(yy, xx) ((xx) < 0 ? xl[yy][E + (xx)] : xr[yy][(xx) - kVec])
#define DRS_OWN_(yy, xx) (((xx) >= 0 && (xx) < kVec) ? pw[0][mod_k2(PH - 1 - RK)][clampi(yy, 0, RY - 1)][clampi(xx, 0, kVec - 1)] \
                                                     : DRS_XNBR_(clampi(yy, 0, RY - 1), xx))
#define DRS_OWN0_(yy, xx) (((xx) >= 0 && (xx) < kVec) ? u0[clampi(yy, 0, RY - 1)][clampi(xx, 0, kVec - 1)] \
                                                      : DRS_XNBR_(clampi(yy, 0, RY - 1), xx))
#define DRS_U_(dj, di) (((y + (dj)) >= 0 && (y + (dj)) < RY) ? (s == 2 ? DRS_OWN_(y + (dj), v + (di)) : DRS_OWN0_(y + (dj), v + (di))) \
                                                             : mine[(y + (dj)) * RP + v + (di)])
#pragma unroll
        for (int y = 0; y < RY; ++y) {
#pragma unroll
            for (int v = 0; v < kVec; ++v) {
#define DRS_P_(dk) pw[s - 1][mod_k2(PH - (dk))][y][v]
                DRS_SCATTER3(DRS_P_, DRS_U_)
#undef DRS_P_
            }
        }
#undef DRS_U_
#undef DRS_OWN0_
#undef DRS_OWN_
#undef DRS_XNBR_
        if (s == 1) {
            // ---- the plane of level 1 completed by this iteration: its ring cells are B's ----
            const int z1 = c.z0 + n - RK;
            if (z1 >= 0 && z1 < c.L) {
                const bool ring_plane = z1 < c.ring_lo || z1 >= c.ring_hi;
                if (ring_plane || c.edge) {       // CTA-uniform
                    const real* pb = c.ring_b + (drs_i64)z1 * c.M * c.N;
#pragma unroll
                    for (int y = 0; y < RY; ++y) {
                        const int gy = c.y_first + y;
                        if (gy < 0 || gy >= c.M) continue;
                        const bool ring_row = ring_plane || gy < c.H || gy >= c.M - c.H;
#pragma unroll
                        for (int v = 0; v < kVec; ++v) {
                            const int gx = c.x_first + v;
                            if (gx >= 0 && gx < c.N && (ring_row || gx < c.H || gx >= c.N - c.H))
                                pw[0][mod_k2(PH - RK)][y][v] = pb[(drs_i64)gy * c.N + gx];
                        }
                    }
                }
            }
            // ---- its edge rows are published for the warps above / below (nobody else reads the rest) ----
            real* dst = reinterpret_cast<real*>(c.lv + (n & 1) * PLANE_STRIDE) + (c.warp * RY + RJ) * RP + E0 + c.lane * kVec;
#pragma unroll
            for (int y = 0; y < RY; ++y) {
                if (y >= RJ && y < RY - RJ) continue;
                real o[kVec];
#pragma unroll
                for (int v = 0; v < kVec; ++v) o[v] = pw[0][mod_k2(PH - RK)][y][v];
                if constexpr (sizeof(real) == 8) *reinterpret_cast<double2*>(dst + y * RP) = make_double2(o[0], o[1]);
                else *reinterpret_cast<float4*>(dst + y * RP) = make_float4(o[0], o[1], o[2], o[3]);
            }
        } else if (n >= c.n_first && n < c.n_end) {
            // ---- level 2: the output plane, and a second time into a neighbour's deep ghost planes ----
            const drs_i64 z = c.z_out0 + n;
            const drs_i64 row0 = (drs_i64)c.y_first * c.N + c.x_first;
            // one pass per destination: a single base pointer is live at a time (as in drs_sweep3d_t.cuh)
            auto store_plane = [&](real* base) {
#pragma unroll
                for (int y = 0; y < RY; ++y) {
                    if (y >= c.y_lo && y < c.y_hi) {
                        real o[kVec];
#pragma unroll
                        for (int v = 0; v < kVec; ++v) o[v] = pw[1][mod_k2(PH - RK)][y][v];
                        real* dst = base + (drs_i64)y * c.N;
                        if (c.v_lo <= 0 && c.v_hi >= kVec) {
                            stg_vec(dst, o);
                        } else {
#pragma unroll
                            for (int v = 0; v < kVec; ++v)
                                if (v >= c.v_lo && v < c.v_hi) dst[v] = o[v];
                        }
                    }
                }
            };
            const drs_i64 MN = (drs_i64)c.M * c.N;
            store_plane(c.out + z * MN + row0);
            if (c.peer_lo != nullptr && z >= c.lo0 && z < c.lo1) store_plane(c.peer_lo + (z + c.lo_shift) * MN + row0);
            if (c.peer_hi != nullptr && z >= c.hi0 && z < c.hi1) store_plane(c.peer_hi + (z + c.hi_shift) * MN + row0);
        }
    }
    // published planes visible to every warp; the input stage is consumed by all of them
    __syncthreads();
    if (threadIdx.x == 0 && n + ST < c.NIT) {
        fence_proxy_async();
        c.issue(n + ST);
    }
    return true;
}

template <int PH>
__device__ __forceinline__ bool phases(real (&pw)[2][K2][RY][kVec], const Ctx& c, int n0) {
    if constexpr (PH < K2) {
        if (!iteration<PH>(pw, c, n0 + PH)) return false;
        return phases<PH + 1>(pw, c, n0);
    } else {
        return true;
    }
}

__device__ __forceinline__ void sweep(const TensorMap& tmap, const TensorMap& tmap_a, const Params& p, const real* ring_a,
                                      const real* ring_b, int ring_lo, int ring_hi) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Ctx c;
    c.warp = threadIdx.x >> 5;
    c.lane = threadIdx.x & 31;
    c.ring = smem_raw;
    c.lv = smem_raw + ST * PLANE_STRIDE;
    c.bars = reinterpret_cast<drs_u64*>(smem_raw + (ST + 2) * PLANE_STRIDE);
    c.tmap = &tmap;
    c.tmap_a = &tmap_a;
    c.fault = p.fault;

    // one tile per CTA and at most 2^31 - 1 CTAs per launch (capi.cpp): 32-bit index arithmetic
    const unsigned int tile = blockIdx.x;
    const unsigned int per_chunk = (unsigned int)p.nxs * (unsigned int)p.nys;
    const int zc = slab_chunk_order(p, (int)(tile / per_chunk));      // face chunks first (flagged launches)
    const int rem = (int)(tile % per_chunk);
    const int cy = rem / p.nxs, cx = rem % p.nxs;

    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < ST; ++s) mbar_init(&c.bars[s], 1);
        fence_mbar_init();
        fence_proxy_async();
    }
    // the published-plane buffers start out zeroed so that never-written halo cells are finite
    for (int x = threadIdx.x; x < 2 * PLANE_STRIDE / 16; x += blockDim.x)
        reinterpret_cast<uint4*>(c.lv)[x] = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();

    const int H = p.halo;
    c.H = H;
    c.L = (int)p.L; c.M = (int)p.M; c.N = (int)p.N;
    const int X0 = (H / kVec) * kVec + cx * WU - HW;
    const int Y0 = H + cy * TYU - HY;
    const drs_i64 za = p.slow_lo + (drs_i64)zc * p.chunk;
    const drs_i64 zb = (za + p.chunk < p.slow_hi) ? za + p.chunk : p.slow_hi;
    const int n_end = (int)(zb - za) + DEPTH;
    c.NIT = (n_end + K2 - 1) / K2 * K2;
    c.z0 = (int)(za - 2 * RK);
    c.x_box = X0 - E0;
    c.y_box = Y0 - RJ;
    c.x_first = X0 + c.lane * kVec;
    {
        const drs_i64 lo = (H > X0 + HW) ? H : X0 + HW;
        const drs_i64 hi = (p.N - H < X0 + HW + WU) ? p.N - H : X0 + HW + WU;
        c.v_lo = (int)(lo - c.x_first);
        c.v_hi = (int)(hi - c.x_first);
    }
    c.y_first = Y0 + c.warp * RY;
    {
        const drs_i64 lo = (H > Y0 + HY) ? H : Y0 + HY;
        const drs_i64 hi = (p.M - H < Y0 + HY + TYU) ? p.M - H : Y0 + HY + TYU;
        c.y_lo = (int)(lo - c.y_first);
        c.y_hi = (int)(hi - c.y_first);
    }
    c.n_first = DEPTH;
    c.n_end = n_end;
    c.z_out0 = za - DEPTH;
    c.out = p.out;
    c.ring_a = ring_a;
    c.ring_b = ring_b;
    c.edge = c.x_box < H || c.x_box + WB > c.N - H || c.y_box < H || c.y_box + YB > c.M - H;
    c.patch0 = c.edge && p.in != ring_a;
    c.ring_lo = ring_lo;
    c.ring_hi = ring_hi;
    c.peer_lo = p.peer_lo;
    c.peer_hi = p.peer_hi;
    c.lo0 = p.push_lo0; c.lo1 = p.push_lo1; c.lo_shift = p.peer_lo_shift;
    c.hi0 = p.push_hi0; c.hi1 = p.push_hi1; c.hi_shift = p.peer_hi_shift;

    // flagged launches (drs_run_slab): thread 0 of a face CTA waits for the neighbours' previous launch before the
    // first TMA request, and the whole CTA leaves on a failed wait (fault code 2 is set; nothing was requested)
    {
        int go = 1;
        if (threadIdx.x == 0) {
            const int face = slab_face(p, zc);
            go = (!face || slab_wait(p, face & 1, face & 2)) ? 1 : 0;
        }
        if (!__syncthreads_and(go)) return;
    }
    if (threadIdx.x == 0)
        for (int n = 0; n < ST && n < c.NIT; ++n) c.issue(n);

    real pw[2][K2][RY][kVec];
#pragma unroll
    for (int s = 0; s < 2; ++s)
#pragma unroll
        for (int d = 0; d < K2; ++d)
#pragma unroll
            for (int y = 0; y < RY; ++y)
#pragma unroll
                for (int v = 0; v < kVec; ++v) pw[s][d][y][v] = (real)0;

#pragma unroll 1
    for (int n0 = 0; n0 < c.NIT; n0 += K2) {
        if (!phases<0>(pw, c, n0)) return;       // watchdog: every warp of the CTA fails the same wait
    }
    // the unit of the slab protocol is the CTA: its stores (own planes and pushes) are ordered before the arrival
    const int face = slab_face(p, slab_chunk_order(p, (int)(blockIdx.x / ((unsigned int)p.nxs * (unsigned int)p.nys))));
    if (face) {                                  // CTA-uniform
        __syncthreads();
        if (threadIdx.x == 0) slab_arrive(p, face & 1, face & 2);
    }
}

}  // namespace s3sp
}  // namespace drs

// ring_lo / ring_hi: the local planes outside [ring_lo, ring_hi) are the global frozen ring (and out-of-grid planes),
// clamped to [0, L) (capi.cpp: launch_slabpair)
extern "C" __global__ void __launch_bounds__(DRS_NW * 32, DRS_MINB)
DRS_SLABPAIR_NAME(const __grid_constant__ drs::TensorMap tmap, const __grid_constant__ drs::TensorMap tmap_a,
                  const __grid_constant__ drs::Params p, const DRS_T* ring_a, const DRS_T* ring_b, int ring_lo, int ring_hi) {
    drs::s3sp::sweep(tmap, tmap_a, p, ring_a, ring_b, ring_lo, ring_hi);
}
