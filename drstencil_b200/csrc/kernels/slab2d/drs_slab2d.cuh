// drs_slab2d.cuh -- slab entry of the 2D sweep (drslab_<name>): one rank of a grid cut into row slabs across GPUs.
//
// The row loop is the one of drs_sweep2d.cuh -- same tile geometry, same TMA ring (s2d::Stream, s2d::iteration's stage
// handling), same gather chain and scatter levels, byte for byte -- with two additions (DESIGN.md section 5):
//   * peer stores: an output row y in [push_lo0, push_lo1) is stored a second time at row y + peer_lo_shift of
//     peer_lo (the lower neighbour's array, mapped over NVLink); likewise push_hi* / peer_hi.  The second store is the
//     same register values as the first, so the neighbour's ghost row equals this rank's owned row bit for bit;
//   * step flags (drs_run_slab, Params::my_flags != nullptr): the warp is the unit of the protocol, as in
//     drs_sweep3d.cuh.  A warp whose row chunk touches a face waits for that neighbour's flag before its first stage
//     request and arrives on the face counter after its last store; face chunks are scheduled first.
// With my_flags == nullptr (drs_sweep / drs_run on a slab plan, the sub-range launches of drs_run_host_slab) the kernel
// pushes and does nothing else.
//
// Memory ordering of the peer stores: they are plain generic-proxy stores of this warp.  In a flagged launch the warp
// executes __syncwarp() after its last row, so every lane's stores -- own rows and pushed rows -- are ordered before
// lane 0's slab_arrive (release at GPU scope on the face counter; the last arriver acquires it, fences at system scope
// and release-stores the flag at system scope).  The neighbour acquires the flag in slab_wait and issues
// fence.proxy.async.global before its TMA reads the ghost rows.  In an unflagged launch the caller orders the kernel
// against the neighbour's next one (stream order on one device, a barrier of the caller's across devices, or the
// wait_/signal_ kernels of drs_run_host_slab, which come after the kernel's completion in stream order).
//
// The generated translation unit defines what drs_sweep2d.cuh needs, plus DRS_SLAB_NAME (this entry).  Its DRS_NAME
// names the plain kernel drs_sweep2d.cuh instantiates along with the shared code; that one is never launched.
#pragma once
#include "drs_sweep2d.cuh"

namespace drs {
namespace slab2d {

using s2d::C;
using s2d::DEPTH;
using s2d::E;
using s2d::NLV;
using s2d::NW;
using s2d::R2;
using s2d::RB;
using s2d::RJ;
using s2d::ST;
using s2d::SW;
using s2d::TS;
using s2d::VT;
using s2d::VW;
using s2d::mod_r2;

// Chunk order of a flagged launch over the p.nys row chunks (drs_common.cuh: slab_chunk_order counts plane chunks):
// the chunks of the lower face, then those of the upper face, then the interior.
__device__ __forceinline__ int row_chunk_order(const Params& p, int i) {
    if (p.my_flags == nullptr) return i;
    if (i < p.face_lo_chunks) return i;
    if (i < p.face_lo_chunks + p.face_hi_chunks) return p.nys - p.face_hi_chunks + (i - p.face_lo_chunks);
    return i - p.face_hi_chunks;
}

// s2d::Tile plus the peer stores of the rows this tile outputs
struct Tile : s2d::Tile {
    real* peer_lo;
    real* peer_hi;
    drs_i64 lo0, lo1, lo_shift, hi0, hi1, hi_shift;
};

__device__ __forceinline__ void store_row(const Tile& t, int n, const real (&o)[C]) {
    const drs_i64 y = t.y_out0 + n;
    real* dst = t.out + y * t.N + t.x_first;
    const bool push_lo = t.peer_lo != nullptr && y >= t.lo0 && y < t.lo1;
    const bool push_hi = t.peer_hi != nullptr && y >= t.hi0 && y < t.hi1;
    real* plo = push_lo ? t.peer_lo + (y + t.lo_shift) * t.N + t.x_first : nullptr;
    real* phi = push_hi ? t.peer_hi + (y + t.hi_shift) * t.N + t.x_first : nullptr;
    if (t.v_lo <= 0 && t.v_hi >= C) {
#pragma unroll
        for (int j = 0; j < VT; ++j) {
            real ov[kVec];
#pragma unroll
            for (int v = 0; v < kVec; ++v) ov[v] = o[j * kVec + v];
            stg_vec(dst + j * kVec, ov);
            if (push_lo) stg_vec(plo + j * kVec, ov);
            if (push_hi) stg_vec(phi + j * kVec, ov);
        }
    } else {
#pragma unroll
        for (int v = 0; v < C; ++v)
            if (v >= t.v_lo && v < t.v_hi) {
                dst[v] = o[v];
                if (push_lo) plo[v] = o[v];
                if (push_hi) phi[v] = o[v];
            }
    }
}

// s2d::row_step with this header's store_row (the arithmetic is the same text)
template <int PH>
__device__ __forceinline__ void row_step(real (&w)[NLV][R2][SW], const real* __restrict__ srow, const Tile& t, int n) {
#if DRS_TS == 1
    {
        constexpr int PP = mod_r2(PH - 1);
        real o[C];
#pragma unroll
        for (int v = 0; v < C; ++v) {
            real acc;
#define DRS_W_(dj) w[0][mod_r2(PP + (dj) - RJ)]
#define DRS_MUL_(dk, dj, di, c) acc = rmul(DRS_W_(dj)[E + v + (di)], (real)(c));
#define DRS_FMA_(dk, dj, di, c) acc = rfma(DRS_W_(dj)[E + v + (di)], (real)(c), acc);
            DRS_CHAIN(DRS_MUL_, DRS_FMA_)
#undef DRS_MUL_
#undef DRS_FMA_
#undef DRS_W_
            o[v] = acc;
        }
        if (n >= t.n_first && n < t.n_end) store_row(t, n, o);
        s2d::load_row(w[0][PH], srow, t.lane);
    }
#else
    {
#pragma unroll
        for (int s = TS; s >= 1; --s) {
            real u[VW];
            if (s == 1) {
                s2d::load_row(u, srow, t.lane);
            } else {
                const real (&src)[SW] = w[s >= 2 ? s - 2 : 0][mod_r2(PH - 1 - RJ)];
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
#if DRS_FACTORED
                real hacc;
                DRS_HROW(DRS_U_)
#endif
                DRS_SCATTER(DRS_P_, DRS_U_)
#undef DRS_U_
#undef DRS_P_
            }
            if (s == TS && n >= t.n_first && n < t.n_end) {
                real o[C];
#pragma unroll
                for (int v = 0; v < C; ++v) {
#ifdef DRS_OUT_SCALE
                    o[v] = rmul(w[TS - 1][mod_r2(PH - RJ)][v], (real)DRS_OUT_SCALE);
#else
                    o[v] = w[TS - 1][mod_r2(PH - RJ)][v];
#endif
                }
                store_row(t, n, o);
            }
        }
    }
#endif
}

// s2d::iteration with this header's row_step
template <int PH>
__device__ __forceinline__ bool iteration(real (&w)[NLV][R2][SW], const s2d::Stream& st, const Tile& t, int n) {
    const int rr = n & (RB - 1);
    const int c = n / RB;
    const int s = c & (ST - 1);
    if (rr == 0) {
        if (!mbar_wait(&st.bars[s], (drs_u32)((c / ST) & 1), st.fault)) return false;
    }
#if DRS_FLAT == 1
    const real* srow = reinterpret_cast<const real*>(st.wbase + s * s2d::STAGE_STRIDE) + rr * s2d::RP +
                       flat_shift((drs_i64)(st.yrow0 + n) * st.N + st.x_box);
#else
    const real* srow = reinterpret_cast<const real*>(st.wbase + s * s2d::STAGE_STRIDE) + rr * s2d::RP;
#endif
    row_step<PH>(w, srow, t, n);
    if (rr == RB - 1) {
        __syncwarp();
#if DRS_FLAT == 2
        if (c + ST < st.NCH) st.issue(c + ST);
#else
        if (st.lane == 0 && c + ST < st.NCH) {
            fence_proxy_async();
            st.issue(c + ST);
        }
#endif
    }
    return true;
}

template <int PH>
__device__ __forceinline__ bool phases(real (&w)[NLV][R2][SW], const s2d::Stream& st, const Tile& t, int n0) {
    if constexpr (PH < R2) {
        if (!iteration<PH>(w, st, t, n0 + PH)) return false;
        return phases<PH + 1>(w, st, t, n0);
    } else {
        return true;
    }
}

// The chunk of this warp after row_chunk_order (recomputed where needed instead of being kept live over the row loop)
__device__ __forceinline__ int row_chunk(const Params& p) {
    const drs_i64 tile = (drs_i64)blockIdx.x * NW + (threadIdx.x >> 5);
    return row_chunk_order(p, (int)(tile / p.nxs));
}

__device__ __forceinline__ void sweep(const TensorMap& tmap, const Params& p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const drs_i64 tile = (drs_i64)blockIdx.x * NW + warp;
    if (tile >= (drs_i64)p.nxs * p.nys) return;
    const int xs = (int)(tile % p.nxs);
    const int yc = row_chunk(p);

    s2d::Stream st;
    st.wbase = smem_raw + warp * s2d::WARP_SMEM;
    st.bars = reinterpret_cast<drs_u64*>(smem_raw + NW * s2d::WARP_SMEM) + warp * ST;
    st.tmap = &tmap;
    st.fault = p.fault;
    st.lane = lane;
    st.in = p.in;
    st.M = p.M;
    st.N = p.N;
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < ST; ++s) mbar_init(&st.bars[s], DRS_FLAT == 2 ? 32 : 1);
        fence_mbar_init();
        fence_proxy_async();
    }
    __syncwarp();

    const int H = p.halo;
    const int X0 = (H / kVec) * kVec + xs * s2d::WU - s2d::HW;
    const drs_i64 ya = p.slow_lo + (drs_i64)yc * p.chunk;
    const drs_i64 yb = (ya + p.chunk < p.slow_hi) ? ya + p.chunk : p.slow_hi;
    // as in s2d::sweep: the surplus iterations of the last rotation stream rows past the chunk and store nothing.  Those
    // rows may be ghost rows a neighbour is rewriting for its next sweep (this warp did not wait for it if its chunk
    // is not a face chunk); they only feed partial sums of rows past yb - 1, which are discarded (DESIGN.md 5)
    const int n_end = (int)(yb - ya) + DEPTH;
    st.NIT = (n_end + R2 - 1) / R2 * R2;
    st.NCH = (st.NIT + RB - 1) / RB;
    st.yrow0 = (int)(ya - TS * RJ);
    st.x_box = X0 - s2d::E0;

    Tile t;
    t.lane = lane;
    t.x_first = X0 + lane * C;
    {
        const drs_i64 lo = (H > X0 + s2d::HW) ? H : X0 + s2d::HW;
        const drs_i64 hi = (p.N - H < X0 + s2d::HW + s2d::WU) ? p.N - H : X0 + s2d::HW + s2d::WU;
        t.v_lo = (int)(lo - t.x_first);
        t.v_hi = (int)(hi - t.x_first);
    }
    t.n_first = DEPTH;
    t.n_end = n_end;
    t.y_out0 = ya - DEPTH;
    t.N = p.N;
    t.out = p.out;
    t.peer_lo = p.peer_lo;
    t.peer_hi = p.peer_hi;
    t.lo0 = p.push_lo0; t.lo1 = p.push_lo1; t.lo_shift = p.peer_lo_shift;
    t.hi0 = p.push_hi0; t.hi1 = p.push_hi1; t.hi_shift = p.peer_hi_shift;

    {
        const int face = slab_face(p, yc);       // warp-uniform; 0 without flags
        if (face) {
            int ok = 1;
            if (lane == 0) ok = slab_wait(p, face & 1, face & 2) ? 1 : 0;
            if (!__shfl_sync(0xffffffffu, ok, 0)) return;
        }
    }

    if (DRS_FLAT == 2 || lane == 0) {
        for (int c = 0; c < ST && c < st.NCH; ++c) st.issue(c);
    }

    real w[NLV][R2][SW];
#pragma unroll
    for (int s = 0; s < NLV; ++s)
#pragma unroll
        for (int r = 0; r < R2; ++r)
#pragma unroll
            for (int x = 0; x < SW; ++x) w[s][r][x] = (real)0;

#pragma unroll 1
    for (int n0 = 0; n0 < st.NIT; n0 += R2) {
        if (!phases<0>(w, st, t, n0)) return;
    }
    const int face = slab_face(p, row_chunk(p));
    if (face) {
        __syncwarp();
        if (lane == 0) slab_arrive(p, face & 1, face & 2);
    }
}

}  // namespace slab2d
}  // namespace drs

extern "C" __global__ void __launch_bounds__(DRS_NW * 32, DRS_MINB)
DRS_SLAB_NAME(const __grid_constant__ drs::TensorMap tmap, const __grid_constant__ drs::Params p) {
    drs::slab2d::sweep(tmap, p);
}
