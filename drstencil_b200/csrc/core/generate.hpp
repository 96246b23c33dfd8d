// Kernel specialisation: (stencil, knobs) -> launch geometry + the CUDA C++ translation unit
// that instantiates the hand-written sm_100a templates in ../kernels/ for exactly this stencil.
//
// This is the engine's replacement for the reference's emitters
//   /root/reference/codegen_2d.hpp  (codeGen_2d::header_gen / gpu_code_gen* / gold_gpu_code_gen)
//   /root/reference/codegen.hpp     (codeGen::...)
// The reference prints a whole kernel per configuration; here the kernel bodies are fixed
// templates and the generator only prints the stencil-specific part: the ordered mul/fma chain
// with literal coefficients, the operator extents and the tile/pipeline constants.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <sstream>
#include <string>
#include <vector>

#include "../../../include/drstencil.h"
#include "stencil.hpp"

namespace drs {

struct KernelSpec {
    // problem
    int dim = 2, dtype = DRS_F64, step = 1, fuse = DRS_FUSE_TEMPORAL;
    int ts = 1;                 // sub-steps evaluated per sweep inside the kernel
    int halo = 0;               // frozen ring (reference macro Halo) = step * order(base)
    int rk = 0, rj = 0, e = 0;  // extents of the operator one sub-step evaluates
    std::vector<Term> chain;    // that operator, gold (std::map) order
    std::vector<Term> gold;     // the composed operator, gold order
    // geometry (see drs_sweep2d.cuh / drs_sweep3d.cuh)
    int nw = 2, st = 4, rb = 4, ry = 8, vt = 1, minb = 1, chunk = 128;
    bool tma_ok = true;         // false -> the naive kernel does the sweep (operator too deep, flat array too long)
    // row pitch not a multiple of 16 bytes (drs_common.cuh: DRS_FLAT): 1 = one TMA request per row of a tile from a
    // {total, 1} tensor map, consumers add the row's shift; 2 = the warp fills the stages itself with cp.async
    // (arrays of 2^31 elements or more, the fused 3D temporal kernel).  Scalar stores in both.
    int flat = 0;
    // 3D arrays far beyond the L2: plane loads carry an L2 evict_last policy, so that the tile halos the neighbouring CTAs
    // re-read outlive the output lines streaming through the cache (drs_common.cuh: DRS_LD_HINT; DESIGN.md 3.5)
    bool keep_planes = false;
    // 3D `--step n` in temporal mode: n launches of the single-step kernel with frozen rings of
    // r, 2r, ... n*r through plan-owned scratch buffers (sub-steps exactly as a fused kernel would
    // evaluate them; not yet fused in one kernel -- no HBM saving, but no 25/35-point operator either)
    int sub_launches = 1;
    int base_order = 0;         // Halo of one sub-step
    // 3D `--step n` fused in one kernel (drs_sweep3d_t.cuh): a CTA of nw warps stacked along y
    bool fused3d = false;
    // engine override share_x / share_y (the c4 / c5 presets): single-step 3D sweep whose sx * sy warps share one
    // input ring per CTA (drs_sweep3d_cta.cuh) instead of one private ring per warp
    bool share3d = false;
    int sx = 1, sy = 1;
    // row-factorised evaluation (temporal mode only): out = sum_dj w[dj] * H(row j+dj) + residual terms,
    // H(row)(x) = sum_di h[di] * u[row][x+di] computed once per row and reused by every output row
    bool factored = false;
    std::vector<double> fh;                 // h[di + e]
    std::vector<double> fw;                 // w[dj + rj]
    std::vector<Term> fres;                 // residual terms (coefficient = K - w*h where that is not zero)
    int fops = 0;                           // arithmetic operations per output in factored form
    // deferred scale of the factorised form: every sub-step evaluates K / fscale (h is divided by one of its own
    // entries, which turns that entry's multiply into nothing), the values of level s carry a factor fscale^-s and
    // the store multiplies by fscale^ts once.  1.0 = not used.
    double fscale = 1.0;
    // `--fuse reuse`: the reference's forward/backward evaluation (drs_reuse.cuh); block shape rbx x rby
    bool reuse = false;
    int dist = 0, rbx = 128, rby = 1;
    std::vector<Term> fwd_slow, fwd_mid, fwd_fast, bwd;
    std::string name = "stencil";
    std::string note;           // why a requested mode was changed, for logs

    int vec() const { return dtype == DRS_F64 ? 2 : 4; }
    int esize() const { return dtype == DRS_F64 ? 8 : 4; }
    int e0() const { return (e + vec() - 1) / vec() * vec(); }
    int hw() const { return ((ts - 1) * e + vec() - 1) / vec() * vec(); }
    int cols() const { return (dim == 2 ? vt : 1) * vec(); }   // consecutive columns per thread
    int wt() const { return 32 * cols(); }
    int wu() const { return (dim == 2 || fused3d) ? wt() - 2 * hw() : wt(); }
    int wb() const { return (share3d ? sx * wt() : wt()) + 2 * e0(); }
    // 3D: rows of one tile (a warp's, or the whole CTA's when fused3d), rows it stores, rows of its TMA box
    int tile_rows() const { return fused3d ? nw * ry : ry; }
    int tile_rows_useful() const { return fused3d ? nw * ry - 2 * (ts - 1) * rj : ry; }
    int box_rows() const { return (share3d ? sy * ry : tile_rows()) + 2 * rj; }
    int rp() const { return flat == 1 ? ((wb() + vec()) * esize() + 127) / 128 * 128 / esize() : wb(); }   // smem row pitch, elements
    int stage_bytes() const { return dim == 2 ? rb * rp() * esize() : rp() * box_rows() * esize(); }
    int stage_stride() const { return (stage_bytes() + 127) / 128 * 128; }
    int smem_bytes() const {
        if (fused3d) return (st + 2 * (ts - 1)) * stage_stride() + st * 8;
        if (share3d) return st * stage_stride() + 2 * st * 8;      // one ring, full + empty barriers
        return nw * st * stage_stride() + nw * st * 8;
    }
    // tiles handled by one CTA
    int tiles_per_cta() const { return fused3d ? 1 : nw; }
    // CTAs of one launch over nxs x nys x nzs warp tiles
    long long ctas(long long nxs, long long nys, long long nzs) const {
        if (share3d) return ((nxs + sx - 1) / sx) * ((nys + sy - 1) / sy) * nzs;
        return (nxs * nys * nzs + tiles_per_cta() - 1) / tiles_per_cta();
    }
};

inline int pow2_floor(int v) { int p = 1; while (p * 2 <= v) p *= 2; return p; }
inline int pow2_ceil(int v) { int p = 1; while (p < v) p *= 2; return p; }

inline bool knob_given(const drs_knobs& k, int bit) { return (k.explicit_mask >> bit) & 1; }
enum KnobBit { KB_STEP = 0, KB_DIST, KB_STREAMING, KB_BX, KB_BY, KB_SN, KB_UNROLL, KB_BMX, KB_BMY, KB_CMX, KB_CMY,
               KB_PREFETCH, KB_MERGE_FWD, KB_CHECK, KB_DTYPE, KB_FUSE };

inline bool factorise_rows(KernelSpec& s);

// A deferred scale eta makes the values of level s carry eta^-s and the store multiply by eta^ts.  Both have to stay
// far inside the dtype's range: a leading coefficient of 1e-10 at depth 4 in fp32 would give levels of ~1e40 (Inf)
// and a scale of 1e-40 (subnormal).  2^60 leaves fp32 a factor 2^68 for the values themselves, 2^500 leaves fp64
// 2^524.  (The shipped stencils need at most 13.3 bits: 2d9pt_cross at depth 4.)
inline bool scale_in_range(double eta, int ts, int dtype) {
    return ts * std::fabs(std::log2(std::fabs(eta))) <= (dtype == DRS_F64 ? 500.0 : 60.0);
}

// Chooses the specialisation.  Returns "" or an error text (-> DRS_E_ARG).
//
// How the reference's knobs (main.cpp:12-56) map onto this engine when given explicitly:
//   --step n          temporal depth (sub-steps per sweep), or composed operator with --fuse algebraic
//   --sn n            slow-axis outputs per warp tile (rows in 2D, planes in 3D)
//   --bx x --by y     CTA size: x*y/32 warps (2D --streaming: x/32, as the reference ignores by there)
//   --stream-unroll u rows per TMA stage in 2D (rounded down to a power of two)
//   --prefetch        ring depth: 8 stages instead of 4 (the TMA ring *is* the prefetch)
//   --block-merge-x m  2D: 128-bit vectors of adjacent columns per thread (1 or 2)
//   --block-merge-y / --cyclic-merge-y m   3D: rows per thread = 4*m
//   --streaming, --dist, --merge-forward, merge-x: accepted; the first is always on, the
//                     others only matter to the reference's forward/backward partition
// Knobs not given explicitly fall back to B200 heuristics, not to the reference's defaults
// (bx = by = sn = 16 describe an sm_80 thread block, not a warp pipeline).
inline std::string choose_spec(const Stencil& base_in, const drs_knobs& k, KernelSpec& s) {
    if (k.step < 1) return "step must be >= 1";
    if (base_in.step != 1) return "plan needs the un-composed stencil (step is a plan knob)";
    Stencil st = base_in;
    s.dim = st.dim;
    s.dtype = k.dtype;
    s.step = k.step;
    s.fuse = k.fuse;
    const int order = st.order_of(st.base);
    const int radius = Stencil::radius_of(st.base);
    if (st.base.empty()) return "stencil has no points";
    if (radius > order)
        return "an offset exceeds Halo (the largest positive slow-axis offset): the reference would read across "
               "rows there (drstencil_2d.hpp:82-92); unsupported";
    s.halo = order * k.step;
    Stencil comp = st;
    comp.compose(k.step);
    s.gold = comp.terms();
    const int vec = s.vec();
    if (k.fuse == DRS_FUSE_REUSE) {
        // the reference's own scheme on the composed operator, with its own knobs and its own refusals
        Analysis a;
        if (!comp.analyze(k.dist, k.merge_forward, a)) return "NOREUSE:No data to reuse. You can try another dist.";
        s.reuse = true;
        s.dist = a.dist;
        s.ts = 1;
        s.chain = s.gold;
        s.base_order = order;
        for (const Term& t : s.chain) {
            s.rk = std::max(s.rk, std::abs(t.dk)); s.rj = std::max(s.rj, std::abs(t.dj)); s.e = std::max(s.e, std::abs(t.di));
        }
        s.fwd_slow = comp.partial_sum(a, 0); s.fwd_mid = comp.partial_sum(a, 1);
        s.fwd_fast = comp.partial_sum(a, 2); s.bwd = comp.partial_sum(a, 3);
        s.rbx = knob_given(k, KB_BX) ? k.bx : (s.dim == 2 ? 128 : 32);
        s.rby = s.dim == 3 ? (knob_given(k, KB_BY) ? k.by : 8) : 1;
        s.chunk = knob_given(k, KB_SN) && k.sn > 0 ? k.sn : 32;
        // codegen_2d.hpp:52-56, codegen.hpp:50-55: tiles that do not cover the halo while a cross-thread forward exists
        if ((2 * s.halo >= s.rbx && !s.fwd_fast.empty()) || (s.dim == 3 && 2 * s.halo >= s.rby && !s.fwd_mid.empty()))
            return "CONFIG:Invalid configuration!";
        if (s.rbx <= 2 * s.halo || (s.dim == 3 && s.rby <= 2 * s.halo) || s.rbx * s.rby > 1024 || s.rbx < 1 || s.rby < 1)
            return "CONFIG:Invalid configuration!";
        if (s.dist > s.halo) return "CONFIG:Invalid configuration!";
        s.tma_ok = false;
        s.flat = false;
        return "";
    }
    if ((st.N % vec) != 0) {      // row pitch not a multiple of 16 bytes (drs_common.cuh: DRS_FLAT)
        // per-row TMA needs flat element indices in a signed 32-bit coordinate; the surplus iterations of a tile run
        // a few rows / planes past the end of the array
        const long double total = (long double)(s.dim == 3 ? st.L + 64 : 1) * (long double)(st.M + 256) * (long double)st.N;
        s.flat = total < 2147483647.0L ? 1 : 2;
        // development aid / tests: DRS_FLAT_MODE=2 forces the cp.async form on small grids too
        if (const char* e = std::getenv("DRS_FLAT_MODE")) if (std::atoi(e) == 2) s.flat = 2;
    }
    // (measured on B200, c5: 388.5 -> 393.0 GStencil/s, depth 2 644.5 -> 649.6; evict_first instead: 321 / 463;
    // DRS_NO_LD_HINT is the A/B switch)
    s.keep_planes = s.dim == 3 && !s.flat && !std::getenv("DRS_NO_LD_HINT") &&
                    (long double)st.L * (long double)st.M * (long double)st.N * (s.dtype == DRS_F64 ? 8 : 4) >= 1073741824.0L;
    bool temporal = (k.fuse == DRS_FUSE_TEMPORAL) && k.step > 1;
    if (temporal) {
        // The reference multiplies the operator out and prints the result with 6 significant digits
        // (drstencil_2d.hpp:174).  Sub-steps of the base operator reproduce that only if no composed
        // coefficient loses digits on the way; otherwise parity comes first: the composed operator is
        // evaluated literally unless temporal mode was asked for explicitly.
        double worst = 0;
        for (const auto& [p, c] : comp.points)
            if (c != 0.0) worst = std::max(worst, std::fabs(coef_literal_value(c) - c) / std::fabs(c));
        if (worst > 1e-13) {
            char b[160];
            if (knob_given(k, KB_FUSE)) {
                std::snprintf(b, sizeof b, "composed coefficients change by up to %.1e when printed with 6 digits: temporal "
                              "sub-steps follow the exact operator, not the reference's literals", worst);
                s.note = b;
            } else {
                std::snprintf(b, sizeof b, "composed coefficients change by up to %.1e when printed with 6 digits: composed "
                              "operator used for parity (--fuse temporal overrides)", worst);
                s.note = b;
                temporal = false;
            }
        }
    }
    bool multi3d = false, fused3d = false;
    if (temporal && s.dim == 3) {
        temporal = false;
        int emax = 0;
        for (const auto& [p, c] : st.base) emax = std::max(emax, std::abs(std::get<2>(p)));
        const bool fits = 32 * vec - 2 * (((k.step - 1) * emax + vec - 1) / vec * vec) >= vec && k.step <= 4;
        if (fits && !(k.reserved[6] & 2)) fused3d = true;
        else {
            multi3d = true;
            s.note = "3D temporal depth runs as one single-step launch per sub-step (not fused in-kernel)";
        }
    }
    int need_vt = 1;      // a level's x neighbours come from the adjacent lane: E <= columns per thread
    if (temporal) {
        int emax = 0;
        for (const auto& [p, c] : st.base) emax = std::max(emax, std::abs(std::get<2>(p)));
        if (emax > vec) need_vt = 2;
        const int cols = need_vt * vec;
        if (emax > cols || 32 * cols + 2 * ((emax + vec - 1) / vec * vec) > 256) {
            temporal = false; s.note = "x extent exceeds what one lane can hand its neighbour: composed operator used";
        } else if (32 * vec - 2 * (((k.step - 1) * emax + vec - 1) / vec * vec) < vec) {   // (vt = 1 worst case)
            temporal = false; s.note = "depth leaves no useful columns per warp: composed operator used";
        }
    }
    s.base_order = order;
    if (temporal) { s.ts = k.step; s.chain = st.base_terms(); }
    else if (fused3d) { s.ts = k.step; s.chain = st.base_terms(); s.fused3d = true; if (s.flat) s.flat = 2; }
    else if (multi3d) { s.ts = 1; s.chain = st.base_terms(); s.sub_launches = k.step; }
    else { s.ts = 1; s.chain = s.gold; s.fuse = k.step > 1 ? DRS_FUSE_ALGEBRAIC : k.fuse; }
    s.rk = s.rj = s.e = 0;
    for (const Term& t : s.chain) {
        s.rk = std::max(s.rk, std::abs(t.dk));
        s.rj = std::max(s.rj, std::abs(t.dj));
        s.e = std::max(s.e, std::abs(t.di));
    }
    if (s.ts > 1 && !(k.reserved[6] & 1)) factorise_rows(s);
    if (s.ts > 1 && !s.factored && !std::getenv("DRS_NO_DEFERRED_SCALE")) {
        // Deferred scale for the plain scatter forms (2D temporal, fused 3D temporal): every sub-step evaluates
        // K / eta with eta = the coefficient of the first term an output receives, so that its partial sum starts
        // as a copy instead of a product (3d7pt_star: 7 -> 6 operations per point and level); the store multiplies
        // by eta^ts.  Tolerance-checked modes only (the bit-exact chain is never scaled).
        for (const Term& t : s.chain) {
            const int lead = s.dim == 3 ? t.dk : t.dj;
            if (lead == -(s.dim == 3 ? s.rk : s.rj)) {
                if (t.coef != 0.0 && t.coef != 1.0 && scale_in_range(t.coef, s.ts, s.dtype)) s.fscale = t.coef;
                break;
            }
        }
    }
    // --- geometry ---
    const long long slow = s.dim == 3 ? st.L : st.M;
    const long long slow_out = std::max<long long>(1, slow - 2 * s.halo);
    // defaults distilled from the tuner runs on B200 (profiles/r01_tune_*.json): two warps per CTA,
    // a shallow ring (the many resident warps provide the bytes in flight), fp64 threads own two
    // 128-bit vectors, chunks sized so that a large grid yields several thousand tiles
    if (s.dim == 2) {
        s.nw = 2; s.st = 2;
        s.rb = s.dtype == DRS_F64 ? 4 : 8;
        s.vt = s.dtype == DRS_F64 ? 2 : 1;
        // enough tiles for ~60 (fp64) / ~240 (fp32) warps' worth of work per SM, but chunks long
        // enough to amortise the pipeline depth
        const int depth = s.ts == 1 ? 2 * s.rj + 1 : 2 * s.ts * s.rj + s.ts - 1;
        const int cols_per_warp = 32 * s.vt * vec - 2 * ((((s.ts - 1) * s.e) + vec - 1) / vec * vec);
        const long long nxs = std::max<long long>(1, (st.N + cols_per_warp - 1) / std::max(1, cols_per_warp));
        const long long want = 148LL * 60 * (s.dtype == DRS_F64 ? 1 : 4);
        const long long nys = std::max<long long>(1, (want + nxs - 1) / nxs);
        long long c = (slow_out + nys - 1) / nys;
        c = std::max<long long>(c, std::max(s.dtype == DRS_F64 ? 128 : 64, 16 * depth));   // per-tile start-up cost
        c = std::min<long long>(c, 512);
        s.chunk = (int)((c + 7) / 8 * 8);
    } else if (s.fused3d) {
        // probe on B200 (profiles/): 8 warps x 4 rows, two CTAs per SM, long chunks
        if (s.ts == 2) { s.nw = 8; s.ry = 4; } else { s.nw = 16; s.ry = 2; }
        s.st = 2; s.chunk = 128;
    } else {
        // rows per thread: 4 for k radius <= 1 (tuned), 8 for deeper windows.  NOTE for the next tuning pass
        // (ptxas -v, sm_100a; not yet timed, so not changed): the deep windows of composed operators are register
        // bound -- 3d7pt composed twice: 171 registers at 4 rows, 244 at 8; 3d9pt_cross composed twice: 255 + 12 B of
        // spills at 4 rows, 620 B at 8; 3d7pt composed three times: 241 at 2 rows, 980 B of spills at 8.
        s.nw = 2; s.ry = s.rk <= 1 ? 4 : 8; s.chunk = 16;
        s.st = pow2_ceil(2 * s.rk + 2);
        if (s.st < 4) s.st = 4;
    }
    if (knob_given(k, KB_SN) && k.sn > 0) s.chunk = k.sn;
    if (knob_given(k, KB_BX) || knob_given(k, KB_BY)) {
        int threads = (s.dim == 2 && k.streaming) ? k.bx : k.bx * k.by;
        s.nw = std::max(1, std::min(16, threads / 32));
    }
    if (s.dim == 2 && knob_given(k, KB_UNROLL) && k.stream_unroll > 0) s.rb = std::min(64, pow2_floor(k.stream_unroll));
    if (knob_given(k, KB_PREFETCH) && k.prefetch) s.st = std::max(s.st, 8);
    if (s.dim == 2 && knob_given(k, KB_BMX) && k.block_merge_x >= 1) s.vt = std::min(2, k.block_merge_x);
    if (k.reserved[5] > 0 && s.dim == 2) s.vt = std::min(2, k.reserved[5]);
    if (s.dim == 2 && s.vt < need_vt && s.ts > 1) s.vt = need_vt;
    if (s.dim == 2 && s.wb() > 256) s.vt = 1;   // a TMA box is at most 256 elements wide
    if (s.dim == 3) {
        const int my = std::max(k.block_merge_y, k.cyclic_merge_y);
        if ((knob_given(k, KB_BMY) || knob_given(k, KB_CMY)) && my >= 1) s.ry = std::min(32, 4 * my);
    }
    // reserved[] carries engine-only tuning overrides (the tuner's extra axes); 0 = keep
    if (k.reserved[0] > 0) s.st = s.fused3d ? std::max(2, k.reserved[0]) : pow2_ceil(k.reserved[0]);   // (the fused 3D temporal ring takes any depth)
    if (k.reserved[2] > 0) s.nw = k.reserved[2];
    if (k.reserved[3] > 0 && s.dim == 3) s.ry = k.reserved[3];
    if (k.reserved[4] > 0 && s.dim == 2) s.rb = pow2_floor(k.reserved[4]);
    {
        // reserved[6] bits 2-3 / 4-5: warps of a CTA along x / y that share one ring (value - 1); 0 = private rings
        const int shx = ((k.reserved[6] >> 2) & 3) + 1, shy = ((k.reserved[6] >> 4) & 3) + 1;
        if (s.dim == 3 && !s.fused3d && s.ts == 1 && shx * shy > 1 && !s.flat) {   // (the shared ring has no flat form)
            s.share3d = true; s.sx = shx; s.sy = shy; s.nw = shx * shy;
            if (s.wb() > 256 || s.box_rows() > 256) return "shared tile exceeds the 256-element TMA box";
        }
    }
    if (s.fused3d) {
        // knobs are hints: a band that does not fit the shared memory (e.g. --block-merge-y 2 at depth 4, where
        // the reference happily emits a program) is thinned until it does -- rows per thread first, then warps
        if (s.st < 2) s.st = 2;
        while (s.smem_bytes() > 227 * 1024 && s.ry > 1) s.ry = std::max(1, s.ry / 2);
        while (s.smem_bytes() > 227 * 1024 && s.st > 2) s.st = std::max(2, s.st / 2);
        while (s.smem_bytes() > 227 * 1024 && s.nw > 2 && (s.nw / 2) * s.ry - 2 * (s.ts - 1) * s.rj >= 1) s.nw /= 2;
    }
    {
        // register budget: the window / queue plus working set; __launch_bounds__ minimum blocks
        // per SM is the most that budget allows (never forces spills)
        const int live = s.fused3d ? (s.ts * (2 * s.rk + 1) * s.ry * vec + 16) * (s.esize() / 4)
                         : s.dim == 3 ? (2 * s.rk + 1) * s.ry * vec * (s.esize() / 4)
                         : s.ts == 1 ? (2 * s.rj + 1) * (s.cols() + 2 * s.e) * (s.esize() / 4)
                                     : (s.ts * (2 * s.rj + 1) * s.cols() + 2 * (s.cols() + 2 * s.e)) * (s.esize() / 4);
        const int est = std::min(255, live + (s.dim == 2 ? 56 : 72));
        s.minb = std::max(1, std::min(32 / s.nw, 65536 / (est * s.nw * 32)));
        if (s.fused3d && s.nw * 32 <= 256) s.minb = std::max(s.minb, 2);   // 128 registers: no spills measured
    }
    if (k.reserved[1] > 0) s.minb = k.reserved[1];
    if (s.dim == 3 && !s.fused3d && s.st < pow2_ceil(2 * s.rk + 2)) s.st = pow2_ceil(2 * s.rk + 2);
    if (s.fused3d) {
        while (s.tile_rows_useful() < 1 && s.nw < 16) s.nw *= 2;
        if (s.tile_rows_useful() < 1) return "temporal depth too large for a 3D tile";
    }
    if (s.chunk > slow_out) s.chunk = (int)slow_out;
    if (s.chunk < 1) s.chunk = 1;

    while (s.smem_bytes() > 227 * 1024 && s.nw > 1 && !s.fused3d && !s.share3d) s.nw /= 2;
    while (s.smem_bytes() > 227 * 1024 && s.st > (s.dim == 3 ? pow2_ceil(2 * s.rk + 2) : 2)) s.st /= 2;
    s.tma_ok = true;
    if (s.smem_bytes() > 227 * 1024) {
        // e.g. a radius-3 3D operator composed three times (radius 9: a ring of 32 planes): the reference still
        // emits a program for it, so the plan falls back to the naive one-thread-per-point kernel instead of failing
        s.tma_ok = false;
        s.note = "operator too deep for the shared-memory plane ring: naive kernel used";
    }
    return "";
}

// Row factorisation of a 2D operator K[dj][di] (SURVEY.md hard part "fp64 compute ceiling"):
// if the rows of K are multiples of one row vector h up to a few entries, then
//     out(j, x) = sum_dj w[dj] * H(j + dj, x)  +  sum_residual r * u[j+dj][x+di],   H(row, x) = sum_di h[di] * u[row][x+di]
// and H(row, .) is shared by all the output rows that touch `row`.  2d9pt_box (0.3 / 0.2 / 0.1):
// h = (0.1, 0.2, 0.1), w = (1, 2, 1), one residual -0.1 at the centre -> 6 operations per output
// instead of 9.  Exact in real arithmetic (w*h reproduces K bit for bit or leaves an explicit
// residual), but it re-associates the sum, so it is used only where the result is held to a
// tolerance (temporal depth > 1), never for the bit-exact single-step chain.
inline bool factorise_rows(KernelSpec& s) {
    if (s.dim != 2 || s.chain.size() < 6) return false;
    const int RJ = s.rj, E = s.e, NR = 2 * RJ + 1, NC = 2 * E + 1;
    std::vector<double> K(NR * NC, 0.0);
    double kmax = 0;
    for (const Term& t : s.chain) { K[(t.dj + RJ) * NC + t.di + E] = t.coef; kmax = std::max(kmax, std::fabs(t.coef)); }
    const double tol = 4e-16 * kmax;
    int best_ops = (int)s.chain.size();
    bool found = false;
    for (int r0 = 0; r0 < NR; ++r0) {                       // candidate base row
        std::vector<double> h(K.begin() + r0 * NC, K.begin() + (r0 + 1) * NC);
        int hn = 0;
        for (double v : h) hn += v != 0.0;
        if (hn < 2) continue;
        std::vector<double> w(NR, 0.0);
        std::vector<Term> res;
        int nterms = 0;
        for (int r = 0; r < NR; ++r) {
            const double* kr = &K[r * NC];
            int rn = 0;
            for (int c = 0; c < NC; ++c) rn += kr[c] != 0.0;
            if (rn == 0) continue;
            double bw = 0; int bres = rn;                   // w = 0: the row stays as plain terms
            for (int c0 = 0; c0 < NC; ++c0) {
                if (h[c0] == 0.0 || kr[c0] == 0.0) continue;
                const double cand = kr[c0] / h[c0];
                int nres = 0;
                for (int c = 0; c < NC; ++c) nres += std::fabs(kr[c] - cand * h[c]) > tol;
                if (nres + 1 < bres + (bw != 0.0)) { bres = nres; bw = cand; }
            }
            w[r] = bw;
            nterms += (bw != 0.0);
            for (int c = 0; c < NC; ++c) {
                const double rv = kr[c] - bw * h[c];
                if (std::fabs(rv) > tol) { res.push_back({0, r - RJ, c - E, rv}); ++nterms; }
            }
        }
        bool unit = false;
        for (double v : w) unit = unit || v == 1.0;
        const int ops = hn + (nterms - 1) + (unit ? 0 : 1);
        if (ops < best_ops) { best_ops = ops; s.fh = h; s.fw = w; s.fres = res; found = true; }
    }
    if (!found || best_ops * 5 > (int)s.chain.size() * 4) return false;   // want >= 20 % fewer operations
    s.factored = true;
    s.fops = best_ops;
    // Deferred scale: dividing h by one of its entries gives the row pass a unit coefficient (one multiply less per
    // point and level: 2d9pt_box 6 -> 5 operations); the residual terms are divided too, the row weights w are not
    // affected (K / eta = w (x) (h / eta) + res / eta), and the store multiplies by eta^ts.  Chosen only when it
    // removes an operation from the row pass.
    auto hrow_ops = [&](const std::vector<double>& h) {
        int terms = 0, adds = 0; bool unit = false;
        if (h[E] != 0.0) { ++terms; unit = unit || h[E] == 1.0; }
        for (int d = 1; d <= E; ++d) {
            const double a = h[E - d], b = h[E + d];
            if (a != 0.0 && a == b) { ++terms; ++adds; unit = unit || a == 1.0; }
            else { if (a != 0.0) { ++terms; unit = unit || a == 1.0; } if (b != 0.0) { ++terms; unit = unit || b == 1.0; } }
        }
        return adds + (terms - 1) + (unit ? 0 : 1);
    };
    const int base = hrow_ops(s.fh);
    double best_eta = 1.0; int best = base;
    for (double eta : s.fh) {
        if (eta == 0.0 || eta == 1.0 || !scale_in_range(eta, s.ts, s.dtype)) continue;
        std::vector<double> h2 = s.fh;
        for (double& v : h2) v /= eta;
        const int ops = hrow_ops(h2);
        if (ops < best) { best = ops; best_eta = eta; }
    }
    if (best_eta != 1.0 && s.ts >= 2 && !std::getenv("DRS_NO_DEFERRED_SCALE")) {   // (the switch is a development aid: A/B timing)
        for (double& v : s.fh) v /= best_eta;
        for (Term& t : s.fres) t.coef /= best_eta;
        s.fscale = best_eta;
        s.fops -= base - best;
    }
    return true;
}

inline std::string lit17(double v) {
    char b[64];
    std::snprintf(b, sizeof b, "%.17g", v);
    std::string t = b;
    if (t.find_first_of(".eEn") == std::string::npos) t += ".0";
    return t;
}

// Scatter form for temporal kernels (drs_sweep2d.cuh): the statements that push one source row
// into the partial sums of the output rows it touches.  P(dj) is the partial sum of the output
// row that sees the source row at offset dj (dj = -RJ is that output's first contribution and
// therefore an assignment, dj = +RJ its last); U(di) is the source row at column offset di.
// With a row factorisation, DRS_HROW(U) first computes `hacc` = h . u.
inline void emit_scatter(std::ostringstream& o, const KernelSpec& s) {
    const int E = s.e, RJ = s.rj;
    if (s.factored) {
        o << "#define DRS_FACTORED 1\n#define DRS_HROW(U)";
        // terms of h . u: the centre, then the symmetric pairs (one add, one coefficient) or single entries; a term
        // with coefficient 1 goes first and costs nothing beyond its operand
        std::vector<std::pair<std::string, double>> hterms;
        if (s.fh[E] != 0.0) hterms.push_back({"U(0)", s.fh[E]});
        for (int d = 1; d <= E; ++d) {
            const double a = s.fh[E - d], b = s.fh[E + d];
            if (a != 0.0 && a == b) hterms.push_back({"radd(U(" + std::to_string(-d) + "), U(" + std::to_string(d) + "))", a});
            else {
                if (a != 0.0) hterms.push_back({"U(" + std::to_string(-d) + ")", a});
                if (b != 0.0) hterms.push_back({"U(" + std::to_string(d) + ")", b});
            }
        }
        for (size_t q = 0; q < hterms.size(); ++q)
            if (hterms[q].second == 1.0) { std::swap(hterms[0], hterms[q]); break; }
        for (size_t q = 0; q < hterms.size(); ++q) {
            const std::string& operand = hterms[q].first;
            const double c = hterms[q].second;
            if (q == 0) {
                if (c == 1.0) o << " \\\n    hacc = " << operand << ";";
                else o << " \\\n    hacc = rmul(" << operand << ", (real)(" << lit17(c) << "));";
            } else if (c == 1.0) o << " \\\n    hacc = radd(hacc, " << operand << ");";
            else o << " \\\n    hacc = rfma(" << operand << ", (real)(" << lit17(c) << "), hacc);";
        }
        o << "\n";
    }
    o << "#define DRS_SCATTER(P, U)";
    for (int dj = -RJ; dj <= RJ; ++dj) {
        const std::string P = "P(" + std::to_string(dj) + ")";
        bool started = dj != -RJ;     // rows after the first accumulate into an existing sum
        auto add_term = [&](const std::string& operand, double c) {
            if (!started) {
                if (c == 1.0) o << " \\\n    " << P << " = " << operand << ";";
                else o << " \\\n    " << P << " = rmul(" << operand << ", (real)(" << lit17(c) << "));";
            } else if (c == 1.0) o << " \\\n    " << P << " = radd(" << P << ", " << operand << ");";
            else o << " \\\n    " << P << " = rfma(" << operand << ", (real)(" << lit17(c) << "), " << P << ");";
            started = true;
        };
        if (s.factored) {
            if (s.fw[dj + RJ] != 0.0) add_term("hacc", s.fw[dj + RJ]);
            for (const Term& t : s.fres)
                if (t.dj == dj) add_term("U(" + std::to_string(t.di) + ")", t.coef);
        } else {
            for (const Term& t : s.chain)      // (un-factorised: the chain's coefficients divided by the deferred scale)
                if (t.dj == dj) add_term("U(" + std::to_string(t.di) + ")", t.coef / s.fscale);
        }
        if (!started) o << " \\\n    " << P << " = (real)0;";
    }
    o << "\n";
}

// 3D scatter (drs_sweep3d_t.cuh): P(dk) is the partial sum of the output plane that sees the source
// plane at k-offset dk; U(dj, di) is the source plane at row/column offsets.
inline void emit_scatter3(std::ostringstream& o, const KernelSpec& s) {
    o << "#define DRS_SCATTER3(P, U)";
    for (int dk = -s.rk; dk <= s.rk; ++dk) {
        const std::string P = "P(" + std::to_string(dk) + ")";
        bool started = dk != -s.rk;
        for (const Term& t : s.chain) {
            if (t.dk != dk) continue;
            const std::string U = "U(" + std::to_string(t.dj) + ", " + std::to_string(t.di) + ")";
            const double c = t.coef / s.fscale;         // deferred scale: a coefficient of 1 costs no multiply
            if (!started) {
                if (c == 1.0) o << " \\\n    " << P << " = " << U << ";";
                else o << " \\\n    " << P << " = rmul(" << U << ", (real)(" << lit17(c) << "));";
            } else if (c == 1.0) o << " \\\n    " << P << " = radd(" << P << ", " << U << ");";
            else o << " \\\n    " << P << " = rfma(" << U << ", (real)(" << lit17(c) << "), " << P << ");";
            started = true;
        }
        if (!started) o << " \\\n    " << P << " = (real)0;";
    }
    o << "\n";
}

inline void emit_chain(std::ostringstream& o, const char* macro, const std::vector<Term>& terms) {
    // nvcc contracts t1 + t2 + ... + tP (gold order) into mul(t2), fma(t1), fma(t3) ... fma(tP);
    // the chain is emitted in that order so that results match the reference's gold kernel bit
    // for bit (SURVEY.md section 8c).  P == 1 is a single product.
    o << "#define " << macro << "(MUL, FMA)";
    std::vector<int> order;
    if (terms.size() == 1) order = {0};
    else { order = {1, 0}; for (int q = 2; q < (int)terms.size(); ++q) order.push_back(q); }
    bool first = true;
    for (int q : order) {
        const Term& t = terms[q];
        o << " \\\n    " << (first ? "MUL" : "FMA") << "(" << t.dk << ", " << t.dj << ", " << t.di << ", "
          << coef_literal_text(t.coef) << ")";
        first = false;
    }
    o << "\n";
}

// The specialised translation unit (kernel templates are #included by name and resolved from
// the headers embedded in libdrstencil.so, or from -I .../csrc/kernels for emitted programs).
inline std::string generate_tu(const KernelSpec& s) {
    std::ostringstream o;
    o << "// generated by drstencil-b200 for sm_100a -- stencil '" << s.name << "', " << (s.dim == 3 ? "3D" : "2D")
      << ", " << (s.dtype == DRS_F64 ? "fp64" : "fp32") << ", step " << s.step << " ("
      << (s.reuse ? "forward/backward data reuse" : s.ts > 1 ? "temporal" : (s.step > 1 ? "algebraic" : "single")) << ")\n";
    o << "#define DRS_DIM " << s.dim << "\n";
    o << "#define DRS_T " << (s.dtype == DRS_F64 ? "double" : "float") << "\n";
    o << "#define DRS_NAME dr_" << s.name << "\n";
    o << "#define DRS_SLAB_NAME drslab_" << s.name << "\n";
    o << "#define DRS_GOLD_NAME gold_" << s.name << "\n";
    o << "#define DRS_CHECK_NAME check_" << s.name << "\n";
    o << "#define DRS_SIGNAL_NAME signal_" << s.name << "\n";
    o << "#define DRS_WAIT_NAME wait_" << s.name << "\n";
    o << "#define DRS_HALO " << s.halo << "\n";
    o << "#define DRS_TS " << s.ts << "\n";
    o << "#define DRS_RK " << s.rk << "\n#define DRS_RJ " << s.rj << "\n#define DRS_E " << s.e << "\n";
    o << "#define DRS_NW " << s.nw << "\n#define DRS_ST " << s.st << "\n#define DRS_RB " << s.rb << "\n";
    o << "#define DRS_RY " << s.ry << "\n#define DRS_VT " << s.vt << "\n#define DRS_MINB " << s.minb << "\n";
    if (s.share3d) o << "#define DRS_SX " << s.sx << "\n#define DRS_SY " << s.sy << "\n";
    if (s.flat) o << "#define DRS_FLAT " << s.flat << "\n";
    // development aid: DRS_EXTRA_DEFINES="A=1;B=2" adds `#define A 1` ... to the translation unit
    // (tools/probe_shape.py experiments; part of the source, hence of the cubin cache key)
    if (const char* xd = std::getenv("DRS_EXTRA_DEFINES")) {
        std::string all = xd, item;
        std::istringstream is(all);
        while (std::getline(is, item, ';')) {
            if (item.empty()) continue;
            const size_t eq = item.find('=');
            o << "#define " << item.substr(0, eq) << " " << (eq == std::string::npos ? "1" : item.substr(eq + 1)) << "\n";
        }
    }
    if (s.keep_planes) o << "#ifndef DRS_LD_HINT\n#define DRS_LD_HINT 1\n#endif\n";
    if (s.reuse) {
        o << "#define DRS_DIST " << s.dist << "\n#define DRS_RBX " << s.rbx << "\n#define DRS_RBY " << s.rby << "\n";
        emit_chain(o, "DRS_FWD_SLOW", s.fwd_slow);
        o << "#define DRS_HAS_BWD " << (s.bwd.empty() ? 0 : 1) << "\n";
        if (!s.bwd.empty()) emit_chain(o, "DRS_BWD", s.bwd);
        o << "#define DRS_HAS_FWD_MID " << (s.fwd_mid.empty() ? 0 : 1) << "\n";
        if (!s.fwd_mid.empty()) emit_chain(o, "DRS_FWD_MID", s.fwd_mid);
        o << "#define DRS_HAS_FWD_FAST " << (s.fwd_fast.empty() ? 0 : 1) << "\n";
        if (!s.fwd_fast.empty()) emit_chain(o, "DRS_FWD_FAST", s.fwd_fast);
    }
    emit_chain(o, "DRS_CHAIN", s.chain);
    if (s.ts > 1 && s.dim == 2) emit_scatter(o, s);
    if (s.fused3d) emit_scatter3(o, s);
    if (s.ts > 1 && s.fscale != 1.0) o << "#define DRS_OUT_SCALE (" << lit17(std::pow(s.fscale, s.ts)) << ")\n";
    emit_chain(o, "DRS_GOLD_CHAIN", s.gold);
    if (s.reuse) o << "#include \"drs_reuse.cuh\"\n";
    else if (s.tma_ok)
        o << "#include \"" << (s.fused3d ? "drs_sweep3d_t.cuh" : s.share3d ? "drs_sweep3d_cta.cuh" : s.dim == 3 ? "drs_sweep3d.cuh" : "drs_sweep2d.cuh") << "\"\n";
    o << "#include \"drs_gold.cuh\"\n";
    return o.str();
}

inline uint64_t fnv1a(const std::string& s, uint64_t h = 1469598103934665603ull) {
    for (unsigned char c : s) { h ^= c; h *= 1099511628211ull; }
    return h;
}

}  // namespace drs
