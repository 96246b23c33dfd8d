// Time-skewed block schedule of the host-buffer runs (drs_run_host, drs_run_host_slab): pure host logic, no CUDA.
//
// The emitted main() of the reference copies the grid in, runs the ping-pong loop, copies it out
// (/root/reference/codegen_2d.hpp:572-583,604-619,647).  This planner orders the same work so that
// the three phases can overlap.  The planes a device holds along the slow axis are cut into blocks;
// block b runs ALL n sweeps before block b+1 starts, its output range sliding down one halo per sweep:
//
//     sweep s (1-based) of block b produces  [edge[b] - s*H, edge[b+1] - s*H)  clamped to [out_lo, out_hi)
//
// (the first block is pinned to out_lo at the bottom, the last one to out_hi at the top).  With every
// block at least 2*H thick this order honours each dependency of the plain schedule in place, on the
// same two buffers:
//   * what sweep s reads -- [edge[b] - s*H - H, edge[b+1] - s*H + H) of level s-1 -- was produced by
//     blocks b-1 and b at sweep s-1, and block b-1's later sweeps (s+1, s+3, ...) write strictly below;
//   * what it overwrites (level s-2) is no longer needed: block b+1 reads level s-2 only from
//     edge[b+1] - s*H upwards.
// A sweep is a pure function of its input array, so the result equals the plain schedule bit for bit.
// Block b needs nothing above edge[b+1] on the device, and its final planes never change afterwards:
// the upload of later blocks and the download of earlier ones can run under the sweeps.
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
// tests/test_host_schedule.py replays the single-device step list on the CPU (not-yet-uploaded planes
// poisoned) for both extreme interleavings of the copies and compares with the plain schedule;
// tests/test_slab_schedule.py runs the step lists of all ranks against each other, with random
// interleavings, ghost planes and flags.
#pragma once
#include <algorithm>
#include <vector>

namespace drs {

enum HostFace {
    WAIT_LOWER = 1, WAIT_UPPER = 2, SIGNAL_LOWER = 4, SIGNAL_UPPER = 8, INIT_LOWER = 16, INIT_UPPER = 32
};

struct HostStep {
    enum Kind { UPLOAD = 0, SWEEP = 1, DOWNLOAD = 2 };
    int kind, block, sweep;     // sweep: 1..n for SWEEP (odd: A -> B, even: B -> A), else 0
    long long lo, hi;           // slow-axis range [lo, hi): planes copied / output planes of the launch
    int faces;                  // HostFace bits
};

struct SlabSide {
    long long local, own_lo, own_hi, out_lo, out_hi;
    bool has_lower, has_upper;   // neighbours below / above
    bool up_skew;                // mirror image: blocks processed top-down, ranges slide up
};

// A grid of `slow` planes on one device: every plane is owned, the outer H on each side are the frozen ring.
inline SlabSide whole_grid(long long slow, long long H) { return {slow, 0, slow, H, slow - H, false, false, false}; }

// H = halo of one sweep, S = nominal block thickness (>= 2*H), n = sweeps (even).  Per block: UPLOAD, its
// non-empty SWEEPs in order, DOWNLOAD.  The first and the last block are thin (a quarter of S, at least 2*H):
// the first one's upload and the last one's download (its thickness + n*H planes) are the only copies that
// nothing overlaps.
inline std::vector<HostStep> plan_block_schedule(SlabSide g, long long H, long long S, int n) {
    const long long L = g.local;
    if (g.up_skew) {            // plan the mirror image, reflect the result
        SlabSide m = g;
        m.up_skew = false;
        m.own_lo = L - g.own_hi; m.own_hi = L - g.own_lo;
        m.out_lo = L - g.out_hi; m.out_hi = L - g.out_lo;
        m.has_lower = g.has_upper; m.has_upper = g.has_lower;
        std::vector<HostStep> r = plan_block_schedule(m, H, S, n);
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
    S = std::max<long long>(S, std::max<long long>(2 * H, 1));
    const long long thin = std::max<long long>(2 * H, std::max<long long>(S / 4, 1));
    std::vector<long long> edge;
    edge.push_back(g.own_lo);
    long long at = std::min(g.own_lo + thin, g.own_hi);
    while (at < g.own_hi) {
        edge.push_back(at);
        const long long left = g.own_hi - at;
        at += (left - thin > S) ? S : ((left > 2 * thin) ? left - thin : left);
    }
    edge.push_back(g.own_hi);
    // every block must be at least 2*H thick (see above): a thinner remainder joins its predecessor
    while (edge.size() > 2 && edge.back() - edge[edge.size() - 2] < 2 * H) edge.erase(edge.end() - 2);
    const int B = (int)edge.size() - 1;
    auto cut = [&](int b, int s) -> long long {   // first output plane of block b at sweep s
        if (b <= 0) return g.out_lo;
        if (b >= B) return g.out_hi;
        return std::min(std::max(edge[b] - (long long)s * H, g.out_lo), g.out_hi);
    };
    std::vector<HostStep> steps;
    for (int b = 0; b < B; ++b) {
        HostStep up{};
        up.kind = HostStep::UPLOAD; up.block = b; up.sweep = 0; up.lo = edge[b]; up.hi = edge[b + 1];
        up.faces = (g.has_lower && b == 0 ? INIT_LOWER : 0) | (g.has_upper && b == B - 1 ? INIT_UPPER : 0);
        steps.push_back(up);
        for (int s = 1; s <= n; ++s) {
            const long long lo = cut(b, s), hi = cut(b + 1, s);
            if (hi <= lo) continue;
            HostStep sw{};
            sw.kind = HostStep::SWEEP; sw.block = b; sw.sweep = s; sw.lo = lo; sw.hi = hi;
            if (g.has_lower && lo < g.own_lo + H) {
                sw.faces |= WAIT_LOWER;
                if (hi >= g.own_lo + H) sw.faces |= SIGNAL_LOWER;    // completes the face planes of level s
            }
            if (g.has_upper && hi > g.own_hi - H) {
                sw.faces |= WAIT_UPPER;
                if (lo <= g.own_hi - H) sw.faces |= SIGNAL_UPPER;
            }
            steps.push_back(sw);
        }
        HostStep dn{};
        dn.kind = HostStep::DOWNLOAD; dn.block = b; dn.sweep = 0;
        dn.lo = b == 0 ? g.own_lo : cut(b, n);
        dn.hi = std::max(dn.lo, b == B - 1 ? g.own_hi : cut(b + 1, n));
        dn.faces = 0;
        steps.push_back(dn);
    }
    return steps;
}

}  // namespace drs
