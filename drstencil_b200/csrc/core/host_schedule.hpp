// Time-skewed block schedule of the host-buffer runs (drs_run_host, drs_run_host_slab): pure host logic, no CUDA.
//
// The emitted main() of the reference copies the grid in, runs the ping-pong loop, copies it out
// (/root/reference/codegen_2d.hpp:572-583,604-619,647).  This planner orders the same work so that
// the three phases can overlap.  The run is a list of K launches, launch k advancing d_k = 1 level (a single
// sweep) or d_k = 2 levels (an exact pair launch); odd launches read A and write B, even ones read B and write A,
// the launch sequence of drs_run.  The planes a device holds along the slow axis are cut into blocks; block b
// runs ALL K launches before block b+1 starts, its output range sliding down by R_k at launch k:
//
//     launch k (1-based) of block b produces  [edge[b] - R_k, edge[b+1] - R_k)  clamped to [out_lo, out_hi)
//     R_1 = d_1*H,   R_k = R_{k-1} + max(d_k, d_{k-1})*H
//
// (the first block is pinned to out_lo at the bottom, the last one to out_hi at the top).  With single sweeps only,
// R_k = k*H.  With every block at least max_k (R_k - R_{k-1} + d_k*H) thick (min_block: 2*H for single sweeps
// only, 4*H once the list has a pair launch) this order honours each dependency of the plain schedule in place,
// on the same two buffers:
//   * what launch k reads -- [edge[b] - R_k - d_k*H, edge[b+1] - R_k + d_k*H) of its input buffer -- was produced
//     at launch k-1 by block b (up to edge[b+1] - R_{k-1}, as R_k >= R_{k-1} + d_k*H) and block b-1 (down to
//     edge[b-1] - R_{k-1}, by the thickness floor), and block b-1's later writes to that buffer (launches k+1,
//     k+3, ...) all lie below edge[b] - R_{k+1} <= edge[b] - R_k - d_k*H;
//   * what it overwrites (launch k-1's input) is no longer needed: block b+1's launch k-1 reads it only from
//     edge[b+1] - R_{k-1} - d_{k-1}*H upwards, and R_k >= R_{k-1} + d_{k-1}*H.
// The second term of the max matters at one place only, the first single sweep after the last pair launch: a
// slide of H there would overwrite H planes of B that block b+1's last pair launch still reads.
// A launch is a pure function of its input array and of the ring cells of A (level 0 of a pair launch) and B
// (level 1), which no launch writes and which are uploaded with the planes the launch reads, so the result
// equals the plain schedule bit for bit.  Block b needs nothing above edge[b+1] on the device, and its final
// planes never change afterwards: the upload of later blocks and the download of earlier ones can run under
// the launches.
//
// A single-device run (whole_grid) owns every plane and has no neighbours.  One rank of a slab-decomposed
// run may have a face to a neighbour below and one above.  Its array holds `local` planes, of which
// [own_lo, own_hi) are its own (host slab, uploaded / downloaded) and [out_lo, out_hi) are swept (out_lo >
// own_lo only where the global frozen ring lies inside the slab); the rest are ghost planes a neighbour fills.
// A face is fixed in space, so the blocks cannot slide past it: neighbouring ranks skew in OPPOSITE
// directions (even ranks down, odd ranks up, processing their blocks top-down).  Then the two blocks that
// meet at a face are both processed first, or both processed last, and run their sweeps in lockstep through
// the step flags:
//   wait   before a launch that reads ghost planes of a face: flag of that face >= sweep
//          (the neighbour has produced -- and pushed -- level sweep-1, and has finished reading what
//          this launch's own push will overwrite);
//   signal after the launch that completes the face planes of a level: flag := sweep + 1;
//   init   after the upload that brings the face planes of level 0: push them to the neighbour's
//          ghost, flag := 1.
// When a block's range has slid off a face the next block inherits the lockstep at the same sweep on
// both sides (mirror symmetry), so no rank ever waits for a level its neighbour produces later than
// it needs it itself.  Without neighbours every step's `faces` is 0.
//
// Slab runs use single sweeps only: the step flags count sweeps.
//
// tests/test_host_schedule.py and tests/test_host_pairs_schedule.py replay the single-device step list on the CPU
// (not-yet-uploaded planes poisoned) for both extreme interleavings of the copies and compare with the plain
// schedule; tests/test_slab_schedule.py runs the step lists of all ranks against each other, with random
// interleavings, ghost planes and flags.
#pragma once
#include <algorithm>
#include <vector>

namespace drs {

enum HostFace {
    WAIT_LOWER = 1, WAIT_UPPER = 2, SIGNAL_LOWER = 4, SIGNAL_UPPER = 8, INIT_LOWER = 16, INIT_UPPER = 32
};

struct HostStep {
    enum Kind { UPLOAD = 0, SWEEP = 1, DOWNLOAD = 2, PAIR = 3 };
    int kind, block, launch;    // launch: 1..K for SWEEP / PAIR (odd: A -> B, even: B -> A), else 0
    long long lo, hi;           // slow-axis range [lo, hi): planes copied / output planes the launch stores
    int faces;                  // HostFace bits
};

struct SlabSide {
    long long local, own_lo, own_hi, out_lo, out_hi;
    bool has_lower, has_upper;   // neighbours below / above
    bool up_skew;                // mirror image: blocks processed top-down, ranges slide up
};

// A grid of `slow` planes on one device: every plane is owned, the outer H on each side are the frozen ring.
inline SlabSide whole_grid(long long slow, long long H) { return {slow, 0, slow, H, slow - H, false, false, false}; }

// The least block thickness the argument above needs for the launch depths `depth`.
inline long long min_block(const std::vector<int>& depth, long long H) {
    long long m = 2 * H;
    for (size_t k = 0; k < depth.size(); ++k) {
        const long long slide = std::max(depth[k], k ? depth[k - 1] : 0) * H;
        m = std::max(m, slide + depth[k] * H);
    }
    return std::max<long long>(m, 1);
}

// H = halo of one sweep, S = nominal block thickness, depth = levels of each launch (1 or 2; all 1 on slabs).  Per
// block: UPLOAD, its non-empty SWEEP / PAIR launches in order, DOWNLOAD.  The first and the last block are thin (a
// quarter of S, at least min_block): the first one's upload and the last one's download (its thickness + R_K planes)
// are the only copies that nothing overlaps.
inline std::vector<HostStep> plan_block_schedule(SlabSide g, long long H, long long S, const std::vector<int>& depth) {
    const long long L = g.local;
    if (g.up_skew) {            // plan the mirror image, reflect the result
        SlabSide m = g;
        m.up_skew = false;
        m.own_lo = L - g.own_hi; m.own_hi = L - g.own_lo;
        m.out_lo = L - g.out_hi; m.out_hi = L - g.out_lo;
        m.has_lower = g.has_upper; m.has_upper = g.has_lower;
        std::vector<HostStep> r = plan_block_schedule(m, H, S, depth);
        for (HostStep& st : r) {
            const long long lo = L - st.hi, hi = L - st.lo;
            st.lo = lo; st.hi = hi;
            const int f = st.faces;
            st.faces = ((f & WAIT_LOWER) ? WAIT_UPPER : 0) | ((f & WAIT_UPPER) ? WAIT_LOWER : 0) |
                       ((f & SIGNAL_LOWER) ? SIGNAL_UPPER : 0) | ((f & SIGNAL_UPPER) ? SIGNAL_LOWER : 0) |
                       ((f & INIT_LOWER) ? INIT_UPPER : 0) | ((f & INIT_UPPER) ? INIT_LOWER : 0);
        }
        return r;
    }
    const int K = (int)depth.size();
    std::vector<long long> R(K + 1, 0);          // R[k]: slide of launch k
    for (int k = 1; k <= K; ++k) R[k] = R[k - 1] + std::max(depth[k - 1], k > 1 ? depth[k - 2] : 0) * H;
    const long long least = min_block(depth, H);
    S = std::max(S, least);
    const long long thin = std::max<long long>(least, S / 4);
    std::vector<long long> edge;
    edge.push_back(g.own_lo);
    long long at = std::min(g.own_lo + thin, g.own_hi);
    while (at < g.own_hi) {
        edge.push_back(at);
        const long long left = g.own_hi - at;
        at += (left - thin > S) ? S : ((left > 2 * thin) ? left - thin : left);
    }
    edge.push_back(g.own_hi);
    // every block must be at least `least` thick (see above): a thinner remainder joins its predecessor
    while (edge.size() > 2 && edge.back() - edge[edge.size() - 2] < least) edge.erase(edge.end() - 2);
    const int B = (int)edge.size() - 1;
    auto cut = [&](int b, int k) -> long long {   // first output plane of block b at launch k
        if (b <= 0) return g.out_lo;
        if (b >= B) return g.out_hi;
        return std::min(std::max(edge[b] - R[k], g.out_lo), g.out_hi);
    };
    std::vector<HostStep> steps;
    for (int b = 0; b < B; ++b) {
        HostStep up{};
        up.kind = HostStep::UPLOAD; up.block = b; up.launch = 0; up.lo = edge[b]; up.hi = edge[b + 1];
        up.faces = (g.has_lower && b == 0 ? INIT_LOWER : 0) | (g.has_upper && b == B - 1 ? INIT_UPPER : 0);
        steps.push_back(up);
        for (int k = 1; k <= K; ++k) {
            const long long lo = cut(b, k), hi = cut(b + 1, k);
            if (hi <= lo) continue;
            HostStep sw{};
            sw.kind = depth[k - 1] == 2 ? HostStep::PAIR : HostStep::SWEEP;
            sw.block = b; sw.launch = k; sw.lo = lo; sw.hi = hi;
            if (g.has_lower && lo < g.own_lo + H) {
                sw.faces |= WAIT_LOWER;
                if (hi >= g.own_lo + H) sw.faces |= SIGNAL_LOWER;    // completes the face planes of level k
            }
            if (g.has_upper && hi > g.own_hi - H) {
                sw.faces |= WAIT_UPPER;
                if (lo <= g.own_hi - H) sw.faces |= SIGNAL_UPPER;
            }
            steps.push_back(sw);
        }
        HostStep dn{};
        dn.kind = HostStep::DOWNLOAD; dn.block = b; dn.launch = 0;
        dn.lo = b == 0 ? g.own_lo : cut(b, K);
        dn.hi = std::max(dn.lo, b == B - 1 ? g.own_hi : cut(b + 1, K));
        dn.faces = 0;
        steps.push_back(dn);
    }
    return steps;
}

}  // namespace drs
