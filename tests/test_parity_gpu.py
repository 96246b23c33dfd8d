"""Parity of the CUDA sweep (through the C ABI) against the CPU oracle on seeded inputs.

Bars (BASELINE.json north_star): fp64 with the FMA order matched -> bit-exact; temporal depth > 1
-> max relative error <= 1e-12 (fp64) / <= 1e-5 (fp32) after the whole schedule."""
import numpy as np
import pytest

from helpers import SHIPPED, max_rel, oracle_run, oracle_terms, pointwise_rel, stc_path

pytestmark = pytest.mark.gpu

SHAPES_2D = [(200, 264), (130, 150), (67, 64), (33, 1000), (1030, 36)]
SHAPES_3D = [(40, 48, 72), (19, 21, 66), (70, 9, 130)]


def _dev(a):
    import torch
    return torch.from_numpy(a).cuda()


def _plan(name, shape, **kn):
    import drstencil_b200 as drs
    st = drs.Stencil.from_file(stc_path(name)).set_size(shape)
    return drs.Plan(st, drs.Knobs(**kn))


def _sweeps(plan, A, B, n):
    bufs = [A, B]
    for s in range(n):
        plan.sweep(bufs[s & 1], bufs[(s & 1) ^ 1])
    plan.sync_check()


@pytest.mark.parametrize("name", SHIPPED)
def test_single_step_fp64_bit_exact(built, name):
    from oracle import oracle
    shapes = SHAPES_3D if name.startswith("3d") else SHAPES_2D
    for shape in shapes:
        plan = _plan(name, shape)
        assert plan.info.kernel_name.startswith("dr_")
        a0 = oracle.rand_array(shape)
        A, B = _dev(a0), _dev(np.full(shape, -3.0))
        _sweeps(plan, A, B, 2)
        refA, refB = a0.copy(), np.full(shape, -3.0)
        offs, coefs, halo = oracle_terms(name, 1)
        oracle.sweep(refA, refB, offs, coefs, halo)
        oracle.sweep(refB, refA, offs, coefs, halo)
        assert np.array_equal(B.cpu().numpy(), refB), (name, shape, "sweep 1")
        assert np.array_equal(A.cpu().numpy(), refA), (name, shape, "sweep 2")


@pytest.mark.parametrize("name,step", [("2d5pt_star", 2), ("2d9pt_box", 2), ("2d9pt_box", 4), ("2d5pt_cross", 2),
                                       ("2d25pt_box", 2), ("3d7pt_star", 2), ("3d9pt_cross", 2)])
def test_algebraic_fusion_fp64_bit_exact(built, name, step):
    """--fuse algebraic evaluates the composed operator literally: same chain as the reference's
    emitted gold kernel, hence bit-exact."""
    shape = (40, 48, 72) if name.startswith("3d") else (200, 264)
    plan = _plan(name, shape, step=step, fuse="algebraic")
    from oracle import oracle
    a0 = oracle.rand_array(shape)
    A, B = _dev(a0), _dev(np.zeros(shape))
    _sweeps(plan, A, B, 2)
    refA, refB = oracle_run(name, step, shape, 2)
    assert np.array_equal(B.cpu().numpy(), refB)
    assert np.array_equal(A.cpu().numpy(), refA)


@pytest.mark.parametrize("name,step", [("2d5pt_star", 2), ("2d5pt_star", 3), ("2d9pt_box", 2), ("2d9pt_box", 4),
                                       ("2d9pt_star", 2), ("2d25pt_box", 2), ("2d5pt_cross", 2), ("2d9pt_cross", 2)])
def test_temporal_blocking_fp64_within_1e12(built, name, step):
    for shape in [(200, 264), (131, 70), (64, 600)]:
        plan = _plan(name, shape, step=step)
        assert plan.note == ""
        assert "#define DRS_TS %d" % step in plan.source
        from oracle import oracle
        a0 = oracle.rand_array(shape)
        A, B = _dev(a0), _dev(np.zeros(shape))
        n = plan.run(A, B, iterations=4 * step)
        plan.sync_check()
        assert n == 4
        refA, refB = oracle_run(name, step, shape, 4)
        H = plan.halo
        inner = (slice(H, -H), slice(H, -H))
        assert max_rel(A.cpu().numpy()[inner], refA[inner]) <= 1e-12, (name, step, shape)
        # the frozen ring keeps the reference's alternating contents
        got = A.cpu().numpy()
        ring = np.ones(shape, bool)
        ring[inner] = False
        assert np.array_equal(got[ring], refA[ring])


@pytest.mark.parametrize("name", ["2d5pt_star", "2d9pt_box", "2d25pt_box", "2d9pt_star", "3d7pt_star"])
def test_fp32_bit_exact_and_within_1e5_of_fp64(built, name):
    from oracle import oracle
    shape = (40, 48, 72) if name.startswith("3d") else (200, 264)
    plan = _plan(name, shape, dtype="f32")
    a64 = oracle.rand_array(shape)
    a0 = a64.astype(np.float32)
    A, B = _dev(a0), _dev(np.zeros(shape, np.float32))
    _sweeps(plan, A, B, 4)
    ref32, _ = oracle_run(name, 1, shape, 4, np.float32, a0=a0)
    assert np.array_equal(A.cpu().numpy(), ref32)
    ref64, _ = oracle_run(name, 1, shape, 4, np.float64, a0=a64)
    H = plan.halo
    inner = tuple(slice(H, -H) for _ in shape)
    assert max_rel(A.cpu().numpy()[inner], ref64[inner]) <= 1e-5


def test_fp32_temporal_within_1e5(built):
    from oracle import oracle
    shape = (300, 520)
    plan = _plan("2d25pt_box", shape, dtype="f32", step=2)
    a64 = oracle.rand_array(shape)
    A, B = _dev(a64.astype(np.float32)), _dev(np.zeros(shape, np.float32))
    plan.run(A, B, iterations=4)
    plan.sync_check()
    ref64, _ = oracle_run("2d25pt_box", 2, shape, 2, np.float64, a0=a64)
    H = plan.halo
    inner = (slice(H, -H), slice(H, -H))
    assert max_rel(A.cpu().numpy()[inner], ref64[inner]) <= 1e-5


@pytest.mark.parametrize("name,step", [("3d7pt_star", 2), ("3d9pt_cross", 2), ("3d7pt_star", 3)])
def test_fp32_3d_temporal_within_1e5(built, name, step):
    """The fused 3D temporal kernel in fp32 (four columns per lane, shuffled column halo)."""
    from oracle import oracle
    shape = (30, 70, 264)
    plan = _plan(name, shape, dtype="f32", step=step)
    assert "drs_sweep3d_t.cuh" in plan.source
    a64 = oracle.rand_array(shape)
    A, B = _dev(a64.astype(np.float32)), _dev(np.zeros(shape, np.float32))
    plan.run(A, B, iterations=2 * step)
    plan.sync_check()
    ref64, _ = oracle_run(name, step, shape, 2, np.float64, a0=a64)
    H = plan.halo
    inner = tuple(slice(H, -H) for _ in shape)
    got = A.cpu().numpy()
    assert max_rel(got[inner], ref64[inner]) <= 1e-5
    ring = np.ones(shape, bool)
    ring[inner] = False
    assert np.array_equal(got[ring], a64.astype(np.float32)[ring])


@pytest.mark.parametrize("name,kn", [
    ("2d5pt_star", dict(sn=7)), ("2d5pt_star", dict(sn=1000, stages=2, rows_per_stage=1)),
    ("2d9pt_box", dict(step=3, sn=16, warps=4, stages=8, rows_per_stage=8)),
    ("2d25pt_box", dict(streaming=1, bx=128, sn=33, prefetch=1)),
    ("2d5pt_star", dict(block_merge_x=2, sn=50)), ("2d9pt_box", dict(step=4, vectors=2, sn=40)),
    ("2d9pt_star", dict(step=2, vectors=2)), ("2d25pt_box", dict(vectors=2, sn=19)),
    ("3d7pt_star", dict(sn=5, rows_3d=4)), ("3d7pt_star", dict(sn=64, rows_3d=16, warps=1, stages=8)),
    ("3d9pt_cross", dict(bx=32, by=4, sn=9)),
])
def test_knob_variants_keep_parity(built, name, kn):
    from oracle import oracle
    shape = (40, 48, 72) if name.startswith("3d") else (150, 200)
    plan = _plan(name, shape, **kn)
    step = kn.get("step", 1)
    a0 = oracle.rand_array(shape)
    A, B = _dev(a0), _dev(np.zeros(shape))
    _sweeps(plan, A, B, 2)
    refA, refB = oracle_run(name, step, shape, 2)
    if step == 1:
        assert np.array_equal(A.cpu().numpy(), refA)
    else:
        assert max_rel(A.cpu().numpy(), refA) <= 1e-12


@pytest.mark.parametrize("name,shape,kn", [
    ("2d9pt_box", (50, 63), dict()), ("2d5pt_star", (131, 257), dict()), ("2d5pt_star", (90, 1001), dict(sn=7)),
    ("2d25pt_box", (77, 133), dict()), ("2d9pt_cross", (64, 95), dict()), ("2d9pt_star", (200, 265), dict(vectors=2)),
    ("2d25pt_box", (130, 262), dict(dtype="f32")), ("2d25pt_box", (130, 263), dict(dtype="f32")),
    ("2d5pt_star", (130, 261), dict(dtype="f32", sn=9)),
    ("3d7pt_star", (40, 48, 73), dict()), ("3d7pt_star", (19, 21, 67), dict(sn=5)), ("3d9pt_cross", (30, 33, 131), dict()),
    ("3d7pt_star", (24, 40, 129), dict(dtype="f32")), ("3d7pt_star", (24, 41, 130), dict(dtype="f32", rows_3d=6)),
    ("3d7pt_star", (24, 40, 131), dict(share_x=2, share_y=2)),      # shared ring has no flat form: private rings
])
@pytest.mark.parametrize("mode", [1, 2])
def test_unaligned_row_pitch_stays_on_the_tma_kernels_bit_exact(built, name, shape, kn, mode, monkeypatch):
    """Rows that are not a multiple of 16 bytes (odd N in fp64, N % 4 != 0 in fp32) cannot be described to TMA by rows,
    and a TMA box must start on a 16-byte boundary.  The sweep kernels then fetch a tile as one TMA request per row
    from the 16-byte boundary below the row's start, the consumers adding the row's shift (DRS_FLAT 1), or -- arrays
    beyond 2^31 elements, forced here with DRS_FLAT_MODE=2 -- fill the same ring with element-sized cp.async
    (DRS_FLAT 2), instead of falling back to the naive kernel: the reference's emitted kernels handle any N at full
    speed through their i_ok guards (codegen_2d.hpp:192-207).  Same chain, same bits; the frozen ring stays untouched."""
    from oracle import oracle
    if mode == 2:
        monkeypatch.setenv("DRS_FLAT_MODE", "2")
    plan = _plan(name, shape, **kn)
    assert plan.info.kernel_name.startswith("dr_") and "#define DRS_FLAT %d" % mode in plan.source
    f32 = kn.get("dtype") == "f32"
    dt = np.float32 if f32 else np.float64
    a0 = oracle.rand_array(shape, dt)
    A, B = _dev(a0), _dev(np.full(shape, -3.0, dt))
    _sweeps(plan, A, B, 2)
    offs, coefs, halo = oracle_terms(name, 1)
    refA, refB = a0.copy(), np.full(shape, -3.0, dt)
    oracle.sweep(refA, refB, offs, coefs, halo)
    oracle.sweep(refB, refA, offs, coefs, halo)
    assert np.array_equal(B.cpu().numpy(), refB), "sweep 1"
    assert np.array_equal(A.cpu().numpy(), refA), "sweep 2"


@pytest.mark.parametrize("name,shape,kn", [
    ("2d9pt_box", (300, 263), dict(step=4)), ("2d5pt_star", (200, 1001), dict(step=2)), ("2d25pt_box", (150, 263), dict(step=2)),
    ("2d9pt_box", (300, 262), dict(step=2, dtype="f32")),
    ("3d7pt_star", (40, 48, 131), dict(step=2)), ("3d9pt_cross", (36, 40, 67), dict(step=2)), ("3d7pt_star", (48, 50, 129), dict(step=3)),
    ("3d7pt_star", (40, 44, 131), dict(step=5)),                     # per-sub-step launches through scratch buffers
])
@pytest.mark.parametrize("mode", [1, 2])
def test_unaligned_row_pitch_temporal_kernels(built, name, shape, kn, mode, monkeypatch):
    from oracle import oracle
    if mode == 2:
        monkeypatch.setenv("DRS_FLAT_MODE", "2")
    plan = _plan(name, shape, **kn)
    fused3d = "drs_sweep3d_t.cuh" in plan.source       # the fused 3D temporal kernel only has the cp.async form
    assert plan.info.kernel_name.startswith("dr_") and "#define DRS_FLAT %d" % (2 if fused3d else mode) in plan.source
    step = kn["step"]
    f32 = kn.get("dtype") == "f32"
    a64 = oracle.rand_array(shape)
    a0 = a64.astype(np.float32) if f32 else a64
    A, B = _dev(a0), _dev(np.zeros(shape, a0.dtype))
    _sweeps(plan, A, B, 2)
    refA, _ = oracle_run(name, step, shape, 2)
    assert max_rel(A.cpu().numpy(), refA) <= (1e-5 if f32 else 1e-12)
    ring = np.ones(shape, bool)
    H = plan.info.halo
    ring[tuple(slice(H, n - H) for n in shape)] = False
    assert np.array_equal(A.cpu().numpy()[ring], a0[ring])


@pytest.mark.parametrize("name,odd,even,kn,bar", [
    ("2d5pt_star", (8191, 8191), (8192, 8192), dict(), 1.15),          # measured 0.97 - 1.07
    ("3d7pt_star", (767, 767, 767), (768, 768, 768), dict(), 1.30),    # measured 1.14 - 1.18
    ("2d9pt_box", (8191, 8191), (8192, 8192), dict(step=4), 1.40),     # measured 1.21 - 1.27
])
def test_unaligned_row_pitch_is_no_performance_cliff(built, name, odd, even, kn, bar):
    """VERDICT r01 item 8: an odd N must stay close to the aligned size next to it (round 1: the naive kernel, ~10x
    slower; the cp.async form: 1.3x - 1.6x; per-row TMA: 0.97x / 1.14x / 1.21x, profiles/r02_unaligned_pitch.md).
    The bursts of the two sizes alternate, so that both are timed under the same clocks and the same neighbours."""
    import torch
    runs = []
    for shape in (odd, even):
        plan = _plan(name, shape, **kn)
        A = torch.rand(shape, dtype=torch.float64, device="cuda")
        B = torch.zeros_like(A)
        _sweeps(plan, A, B, 4)
        runs.append((plan, A, B, float(np.prod(shape))))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    per_point = [None, None]
    for _ in range(5):
        for q, (plan, A, B, points) in enumerate(runs):
            e0.record()
            _sweeps(plan, A, B, 20)
            e1.record()
            torch.cuda.synchronize()
            t = e0.elapsed_time(e1) / points
            per_point[q] = t if per_point[q] is None else min(per_point[q], t)
    del runs
    print("unaligned / aligned time per point: %.3f" % (per_point[0] / per_point[1]))
    assert per_point[0] <= bar * per_point[1], per_point


@pytest.mark.parametrize("name,step", [("2d9pt_box", 4), ("3d7pt_star", 2), ("2d25pt_box", 1)])
def test_gold_kernel_is_the_oracle_chain(built, name, step):
    """drs_gold_sweep (K4/K5 stand-in) == oracle, bit for bit, for the composed operator."""
    from oracle import oracle
    shape = (40, 48, 72) if name.startswith("3d") else (120, 136)
    plan = _plan(name, shape, step=step)
    a0 = oracle.rand_array(shape)
    A, B = _dev(a0), _dev(np.zeros(shape))
    n = plan.gold_run(A, B, iterations=2 * step)
    assert n == 2
    refA, _ = oracle_run(name, step, shape, 2)
    assert np.array_equal(A.cpu().numpy(), refA)


def test_check_error_matches_common_hpp(built):
    from oracle import oracle
    shape = (90, 100)
    plan = _plan("2d5pt_star", shape)
    rng = np.random.default_rng(5)
    x = rng.random(shape)
    y = x + rng.normal(0, 1e-9, shape)
    mx, rms = plan.check_error(_dev(x), _dev(y))
    emx, erms, _ = oracle.check_error(x, y, 1)
    assert abs(mx - emx) <= 1e-18 and abs(rms - erms) <= 1e-6 * erms
    mx, rms = plan.check_error(_dev(x), _dev(x))
    assert mx == 1e-13 and rms == 0.0


def test_run_host_round_trip(built):
    """The emitted main()'s data path on host buffers == oracle schedule."""
    import torch
    from oracle import oracle
    shape = (256, 320)
    plan = _plan("2d5pt_star", shape)
    a = torch.from_numpy(oracle.rand_array(shape)).pin_memory()
    b = torch.zeros(shape, dtype=torch.float64).pin_memory()
    ms = plan.run_host(a, b, iterations=10)
    assert ms > 0
    refA, _ = oracle_run("2d5pt_star", 1, shape, 10)
    assert np.array_equal(a.numpy(), refA)


def test_linearity_and_idempotence_at_scale(built):
    """Size-independent properties at a BASELINE size (4096^2): sweep(a*x + y) == a*sweep(x) + sweep(y)
    up to rounding, and a sweep is idempotent on its destination."""
    import torch
    shape = (4096, 4096)
    plan = _plan("2d5pt_star", shape)
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.rand(shape, dtype=torch.float64, device="cuda", generator=g)
    y = torch.rand(shape, dtype=torch.float64, device="cuda", generator=g)
    ox, oy, oz = (torch.zeros_like(x) for _ in range(3))
    plan.sweep(x, ox); plan.sweep(y, oy); plan.sweep(2.0 * x + y, oz)
    plan.sync_check()
    assert torch.max(torch.abs(oz - (2.0 * ox + oy))).item() < 1e-14 * 4
    o2 = ox.clone()
    plan.sweep(x, o2)
    plan.sync_check()
    assert torch.equal(o2, ox)
    # checksum against the gold kernel on the same input
    og = torch.zeros_like(x)
    plan.gold_sweep(x, og)
    assert torch.equal(og, ox)


@pytest.mark.parametrize("name,shape,kn", [
    ("2d5pt_star", (70, 136), dict(sn=16)), ("2d9pt_box", (90, 264), dict(step=4, vectors=2, sn=24)),
    ("2d25pt_box", (61, 200), dict(step=2)), ("3d7pt_star", (14, 21, 70), dict(sn=5, rows_3d=4)),
    ("3d9pt_cross", (12, 18, 66), dict()),
])
def test_no_write_outside_the_interior(built, name, shape, kn):
    """Guard bands (compute-sanitizer is closed on this pool): the destination sits inside a larger
    poisoned allocation; a sweep may change nothing but the interior -- neither the guard bands
    before/after the array nor the frozen Halo ring."""
    import torch
    plan = _plan(name, shape, **kn)
    n = int(np.prod(shape))
    pad = 4096
    src = torch.rand(n + 2 * pad, dtype=torch.float64, device="cuda")
    dst = torch.full((n + 2 * pad,), -777.0, dtype=torch.float64, device="cuda")
    a = src[pad:pad + n].view(shape)
    b = dst[pad:pad + n].view(shape)
    assert a.data_ptr() % 16 == 0 and b.is_contiguous()
    plan.sweep(a, b)
    plan.sync_check()
    H = plan.halo
    assert torch.all(dst[:pad] == -777.0) and torch.all(dst[pad + n:] == -777.0)
    ring = torch.ones(shape, dtype=torch.bool, device="cuda")
    ring[tuple(slice(H, -H) for _ in shape)] = False
    assert torch.all(b[ring] == -777.0)
    assert not torch.any(b[~ring] == -777.0)


def test_degenerate_grids(built):
    """Grids with an empty interior, or thinner than one tile, are legal and write nothing / little."""
    import torch
    for name, shape in [("2d9pt_star", (4, 64)), ("2d5pt_star", (3, 8)), ("3d7pt_star", (2, 8, 8)), ("2d25pt_box", (5, 6))]:
        plan = _plan(name, shape)
        a = torch.rand(shape, dtype=torch.float64, device="cuda")
        b = torch.full(shape, -5.0, dtype=torch.float64, device="cuda")
        plan.sweep(a, b)
        plan.sync_check()
        from oracle import oracle
        offs, coefs, halo = oracle_terms(name, 1)
        ref = np.full(shape, -5.0)
        if all(n > 2 * halo for n in shape):
            oracle.sweep(a.cpu().numpy(), ref, offs, coefs, halo)
        assert np.array_equal(b.cpu().numpy(), ref), (name, shape)


@pytest.mark.parametrize("preset,bar", [("c1", 0.0), ("c2", 1e-12), ("c3", 0.0), ("c4", 0.0), ("c5", 0.0)])
def test_baseline_sizes_against_the_gold_kernel(built, preset, bar):
    """BASELINE.json sizes (4096^2, 16384^2 depth 4, 16384^2 fp32, 768^3, and 1536^3 = 3.6e9 points, beyond
    32-bit indexing: three 27 GiB arrays on one 180 GB GPU): one sweep of the tuned
    plan against the device gold kernel (itself bit-exact against the oracle at small sizes) --
    bit-identical for depth 1, <= 1e-12 relative for the temporally fused config."""
    import torch
    import drstencil_b200 as drs
    from drstencil_b200.presets import PRESETS
    path, kn = PRESETS[preset]
    st = drs.Stencil.from_file(path)
    plan = drs.Plan(st, kn)
    dt = torch.float32 if kn.dtype == drs.F32 else torch.float64
    g = torch.Generator(device="cuda").manual_seed(7)
    a = torch.rand(st.shape, dtype=dt, device="cuda", generator=g)
    b = torch.zeros_like(a)
    ref = torch.zeros_like(a)
    plan.sweep(a, b)
    plan.gold_sweep(a, ref)
    plan.sync_check()
    if bar == 0.0:
        assert torch.equal(b, ref)
    else:
        mx, rms = plan.check_error(b, ref)
        assert mx / float(ref.abs().max()) <= bar
    # checksum of checksums: row sums of the result, summed, equal in both
    assert abs(float(b.double().sum()) - float(ref.double().sum())) <= 1e-9 * abs(float(ref.double().sum()))


def test_streams_many_plans_and_argument_errors(built):
    import torch
    import drstencil_b200 as drs
    from oracle import oracle
    shape = (96, 128)
    a0 = oracle.rand_array(shape)
    refA, refB = oracle_run("2d9pt_box", 1, shape, 1)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    outs = []
    for k in range(6):                                # several live plans, alternating streams
        plan = _plan("2d9pt_box", shape, sn=8 + 4 * k)
        A, B = _dev(a0), _dev(np.zeros(shape))
        torch.cuda.synchronize()
        st = s1 if k % 2 == 0 else s2
        with torch.cuda.stream(st):
            plan.sweep(A, B)                          # picks up torch's current stream
        plan.sync_check(st)
        outs.append(B.cpu().numpy())
        del plan
    assert all(np.array_equal(o, refB) for o in outs)
    plan = _plan("2d9pt_box", shape)
    A = _dev(a0)
    with pytest.raises(drs.DrsError) as e:
        plan.sweep(A, A)                              # in-place is not allowed (the reference requires in != out too)
    assert e.value.code == drs.E_ARG
    flat = torch.zeros(shape[0] * shape[1] + 1, dtype=torch.float64, device="cuda")
    with pytest.raises(drs.DrsError) as e:
        plan.sweep(flat[1:].view(shape), _dev(np.zeros(shape)))   # 8-byte aligned only: no TMA descriptor
    assert e.value.code == drs.E_ARG


@pytest.mark.parametrize("name", ["2d5pt_cross", "2d9pt_cross", "2d9pt_star", "2d25pt_box"])
def test_fp32_temporal_all_shapes(built, name):
    from oracle import oracle
    shape = (160, 264)
    plan = _plan(name, shape, dtype="f32", step=2)
    a64 = oracle.rand_array(shape)
    A, B = _dev(a64.astype(np.float32)), _dev(np.zeros(shape, np.float32))
    plan.run(A, B, iterations=4)
    plan.sync_check()
    ref64, _ = oracle_run(name, 2, shape, 2, np.float64, a0=a64)
    H = plan.halo
    inner = (slice(H, -H), slice(H, -H))
    assert max_rel(A.cpu().numpy()[inner], ref64[inner]) <= 1e-5


@pytest.mark.parametrize("name,step,kn", [
    ("3d7pt_star", 2, dict()), ("3d7pt_star", 3, dict()), ("3d9pt_cross", 2, dict()),
    ("3d7pt_star", 2, dict(warps=4, sn=7)), ("3d7pt_star", 4, dict(warps=8, rows_3d=2, sn=9, stages=4)),
    ("3d7pt_star", 2, dict(no_fused3d=1)), ("3d9pt_cross", 3, dict(no_fused3d=1)),
])
def test_3d_temporal_depth(built, name, step, kn):
    """3D `--step n` (temporal): n sub-steps fused in one kernel (drs_sweep3d_t.cuh), or -- with the
    engine override no_fused3d -- n single-step launches through scratch buffers.  Either way ==
    the composed operator within 1e-12, and the frozen ring of width n*r is untouched."""
    from oracle import oracle
    for shape in [(40, 48, 72), (23, 37, 130), (9 + 2 * step, 70, 64)]:
        plan = _plan(name, shape, step=step, **kn)
        fused = not kn.get("no_fused3d")
        assert ("drs_sweep3d_t.cuh" in plan.source) == fused
        a0 = oracle.rand_array(shape)
        A, B = _dev(a0), _dev(np.full(shape, -9.0))
        n = plan.run(A, B, iterations=2 * step)
        plan.sync_check()
        assert n == 2 and plan.launch_count == (2 if fused else 2 * step)
        refA, refB = a0.copy(), np.full(shape, -9.0)
        offs, coefs, halo = oracle_terms(name, step)
        oracle.sweep(refA, refB, offs, coefs, halo)
        oracle.sweep(refB, refA, offs, coefs, halo)
        assert halo == plan.halo
        inner = tuple(slice(halo, -halo) for _ in shape)
        got = A.cpu().numpy()
        assert max_rel(got[inner], refA[inner]) <= 1e-12, (name, step, shape, kn)
        ring = np.ones(shape, bool)
        ring[inner] = False
        assert np.array_equal(got[ring], refA[ring])
        assert np.array_equal(B.cpu().numpy()[ring], refB[ring])


def _synthetic(kind):
    """Synthetic descriptions that none of the shipped files cover: asymmetric coefficient values,
    one-sided rows, radius 3, a full 3D box."""
    rng = np.random.default_rng(11)
    if kind == "2d_asym_box":          # 3x3 with nine different coefficients
        offs = [(j, i) for j in (-1, 0, 1) for i in (-1, 0, 1)]
    elif kind == "2d_star_r3":         # 13-point star, radius 3
        offs = [(0, 0)] + [(d, 0) for d in (-3, -2, -1, 1, 2, 3)] + [(0, d) for d in (-3, -2, -1, 1, 2, 3)]
    elif kind == "2d_forward_rows":    # rows j and j+1 only (no dj = -1 terms), upwind in i
        offs = [(0, -1), (0, 0), (1, -1), (1, 0), (1, 1)]
    elif kind == "2d_rank1":           # separable 3x3: every row a multiple of (1, 2, 1)
        offs = [(j, i) for j in (-1, 0, 1) for i in (-1, 0, 1)]
        w = {-1: 0.05, 0: 0.1, 1: 0.075}
        h = {-1: 1.0, 0: 2.0, 1: 1.0}
        return offs, [w[j] * h[i] for j, i in offs]
    elif kind == "3d_box27":
        offs = [(k, j, i) for k in (-1, 0, 1) for j in (-1, 0, 1) for i in (-1, 0, 1)]
    elif kind == "3d_star_r2":
        offs = [(0, 0, 0)] + [tuple(d if a == ax else 0 for a in range(3)) for ax in range(3) for d in (-2, -1, 1, 2)]
    else:
        raise KeyError(kind)
    coefs = [round(float(c), 4) for c in rng.uniform(0.01, 0.2, len(offs))]
    return offs, coefs


@pytest.mark.parametrize("kind,shape", [
    ("2d_asym_box", (90, 136)), ("2d_star_r3", (80, 200)), ("2d_forward_rows", (70, 132)), ("2d_rank1", (64, 128)),
    ("3d_box27", (18, 20, 68)), ("3d_star_r2", (20, 22, 70)),
])
def test_synthetic_stencils(built, kind, shape):
    """from_points path: single step bit-exact, temporal depth 2/3 within 1e-12 (factorised and not)."""
    import drstencil_b200 as drs
    from oracle import oracle
    offs, coefs = _synthetic(kind)
    dim = len(shape)
    pts = {((0,) + tuple(o)) if dim == 2 else tuple(o): c for o, c in zip(offs, coefs)}
    a0 = oracle.rand_array(shape)
    for step, kn in [(1, dict()), (2, dict()), (2, dict(fuse="temporal")), (3, dict(fuse="temporal", no_factor=1)),
                     (2, dict(fuse="temporal", vectors=1, sn=11))]:
        st = drs.Stencil.from_points(offs, coefs, shape, 2 * step, name="syn_" + kind)
        plan = drs.Plan(st, drs.Knobs(step=step, **kn))
        A, B = _dev(a0), _dev(np.zeros(shape))
        plan.run(A, B, 2 * step)
        plan.sync_check()
        comp = oracle.compose(pts, step)
        halo, _ = oracle.order_dist(comp, dim)
        explicit_temporal = kn.get("fuse") == "temporal"
        literal = "#define DRS_TS 1\n" in plan.source and "drs_sweep3d_t" not in plan.source   # gather chain of literals
        if not literal:
            # sub-steps follow the exact composed operator (the 6-digit literals of the reference would
            # perturb these many-digit coefficients by ~1e-7, which plan.note reports)
            keys = sorted(comp)
            o = np.array(keys, dtype=np.int32)
            c = np.array([comp[k] for k in keys])
        else:
            o, c = oracle.terms(comp)
        refA, refB = a0.copy(), np.zeros(shape)
        oracle.run(refA, refB, o, c, halo, 2 * step, step)
        assert halo == plan.halo
        got = A.cpu().numpy()
        assert literal == (not explicit_temporal) or kind == "2d_rank1"
        if literal:
            # parity first: single step, or the composed operator evaluated literally
            assert np.array_equal(got, refA), (kind, step)
            if step > 1:
                assert "composed operator used for parity" in plan.note
        else:
            assert max_rel(got, refA) <= 1e-12, (kind, step, kn, max_rel(got, refA))


def test_tuner_smoke(built, tmp_path, monkeypatch):
    """The tuner end to end on a small grid: search, confirmation, result record."""
    from drstencil_b200.tuner import tune
    monkeypatch.chdir(tmp_path)
    res = tune.tune(stc_path("2d9pt_box"), step=2, size=(1024, 1024), budget_s=20.0, top=1, log=lambda *a: None)
    assert res["tried"] >= 3 and res["winners"] and res["winners"][0]["ms_confirmed"] > 0
    assert res["winners"][0]["name"].startswith("fu2d0bx")


def test_run_as_cuda_graph_equals_plain_launches(built):
    """drs_run replays its launches as a CUDA graph by default: same kernels, same count, same
    bits as plain launches; different sweep counts and buffer pairs get their own graphs; a stream
    that the caller is capturing gets plain launches (and the caller's graph replays correctly)."""
    import torch
    from oracle import oracle
    shape = (300, 264)
    plan = _plan("2d5pt_star", shape)
    a0 = oracle.rand_array(shape)
    outs = {}
    for mode in (False, True):
        plan.set_graph(mode)
        for iters in (10, 4, 10):
            A, B = _dev(a0), _dev(np.zeros(shape))
            l0 = plan.launch_count
            n = plan.run(A, B, iterations=iters)
            plan.sync_check()
            assert n == iters and plan.launch_count - l0 == iters
            if (iters, False) in outs:
                assert np.array_equal(A.cpu().numpy(), outs[(iters, False)])
            outs[(iters, mode)] = A.cpu().numpy()
    refA, _ = oracle_run("2d5pt_star", 1, shape, 10)
    assert np.array_equal(outs[(10, True)], refA)
    # the same plan inside the caller's own graph
    A, B = _dev(a0), _dev(np.zeros(shape))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        plan.run(A, B, iterations=2)
    torch.cuda.current_stream().wait_stream(s)
    A.copy_(torch.from_numpy(a0)); B.zero_()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        plan.run(A, B, iterations=10)
    g.replay()
    plan.sync_check()
    assert np.array_equal(A.cpu().numpy(), refA)


@pytest.mark.parametrize("preset,timesteps,tol,ptol", [
    ("c2", 128, 1e-12, 1e-11),     # 2d9pt_box fp64, temporal depth 4: bench.py's whole step (32 sweeps)
    ("c3", 8, None, None),         # 2d25pt_box fp32, depth 1: bench.py's whole step (8 sweeps), bit-exact vs the fp32 oracle
    ("c1", 10, None, None),        # 2d5pt_star fp64: 10 sweeps, bit-exact
    ("c1t2", 20, 1e-12, 1e-11),
])
def test_whole_bench_schedules_against_the_oracle(built, preset, timesteps, tol, ptol):
    """The schedules bench.py times (same knobs, same timesteps per step), on a 1024^2 grid the oracle finishes in
    seconds: global AND floored pointwise relative error after the WHOLE schedule (VERDICT r01: temporal tests
    stopped at 4 sweeps while the bench runs 32)."""
    import drstencil_b200 as drs
    from drstencil_b200.presets import PRESETS
    from oracle import oracle
    path, kn = PRESETS[preset]
    shape = (1024, 1024)
    st = drs.Stencil.from_file(path).set_size(shape)
    plan = drs.Plan(st, kn)
    f32 = kn.dtype == drs.F32
    a64 = oracle.rand_array(shape)
    a0 = a64.astype(np.float32) if f32 else a64
    A, B = _dev(a0), _dev(np.zeros(shape, a0.dtype))
    n = plan.run(A, B, timesteps)
    plan.sync_check()
    name = [s_ for s_ in SHIPPED if s_ in path][0]
    assert n == drs.sweep_count(timesteps, kn.step)
    got = A.cpu().numpy()
    if tol is None:
        ref, _ = oracle_run(name, kn.step, shape, n, a0.dtype, a0=a0)
        assert np.array_equal(got, ref)
        if f32:
            ref64, _ = oracle_run(name, kn.step, shape, n, np.float64, a0=a64)
            H = plan.halo
            inner = (slice(H, -H), slice(H, -H))
            assert max_rel(got[inner], ref64[inner]) <= 1e-5 and pointwise_rel(got[inner], ref64[inner]) <= 1e-4
    else:
        ref, _ = oracle_run(name, kn.step, shape, n, np.float64, a0=a64)
        assert max_rel(got, ref) <= tol and pointwise_rel(got, ref) <= ptol, (max_rel(got, ref), pointwise_rel(got, ref))


@pytest.mark.parametrize("preset,timesteps", [("c4", 16), ("c5", 10), ("c4t2", 16)])
def test_whole_3d_bench_schedules_against_the_oracle(built, preset, timesteps):
    import drstencil_b200 as drs
    from drstencil_b200.presets import PRESETS
    from oracle import oracle
    path, kn = PRESETS[preset]
    shape = (72, 200, 264)
    st = drs.Stencil.from_file(path).set_size(shape)
    plan = drs.Plan(st, kn)
    a0 = oracle.rand_array(shape)
    A, B = _dev(a0), _dev(np.zeros(shape))
    n = plan.run(A, B, timesteps)
    plan.sync_check()
    ref, _ = oracle_run("3d7pt_star", kn.step, shape, n, a0=a0)
    got = A.cpu().numpy()
    if kn.step == 1:
        assert np.array_equal(got, ref)
    else:
        assert max_rel(got, ref) <= 1e-12 and pointwise_rel(got, ref) <= 1e-11


@pytest.mark.parametrize("name,shape,kn", [
    ("2d5pt_star", (200, 264), dict()), ("2d9pt_star", (130, 150), dict()), ("2d9pt_box", (200, 265), dict(step=2)),
    ("2d25pt_box", (150, 200), dict(bx=64, sn=7)), ("2d9pt_box", (120, 136), dict(step=4, merge_forward=30)),
    ("2d5pt_cross", (100, 120), dict(step=2)), ("2d25pt_box", (130, 262), dict(dtype="f32")),
    ("3d7pt_star", (40, 48, 72), dict()), ("3d7pt_star", (30, 41, 67), dict(step=2, merge_forward=1, bx=16, by=16, sn=5)),
    ("3d9pt_cross", (30, 40, 64), dict(step=2)), ("3d7pt_star", (24, 40, 64), dict(dtype="f32", step=2)),
])
def test_data_reuse_mode_against_its_oracle(built, name, shape, kn):
    """`--fuse reuse` (SURVEY 8f-4): the reference's forward/backward evaluation as an A/B mode -- equal, bit for bit,
    to the oracle's restatement of that scheme, within the reference's own bar of the gold expression, ring untouched."""
    from oracle import oracle
    plan = _plan(name, shape, fuse="reuse", **kn)
    assert "drs_reuse.cuh" in plan.source and plan.info.kernel_name.startswith("dr_")
    step = kn.get("step", 1)
    f32 = kn.get("dtype") == "f32"
    dt = np.float32 if f32 else np.float64
    is3d = name.startswith("3d")
    s = oracle.parse_stc(stc_path(name), is3d)
    pts = oracle.compose(s.points, step)
    a0 = oracle.rand_array(shape, dt)
    A, B = _dev(a0), _dev(np.full(shape, -3.0, dt))
    _sweeps(plan, A, B, 2)
    ra, rb = a0.copy(), np.full(shape, -3.0, dt)
    assert oracle.sweep_reuse(ra, rb, pts, s.dim, 0, kn.get("merge_forward", 5))
    assert oracle.sweep_reuse(rb, ra, pts, s.dim, 0, kn.get("merge_forward", 5))
    assert np.array_equal(B.cpu().numpy(), rb) and np.array_equal(A.cpu().numpy(), ra)
    # within the reference's own bar of the gold expression (same schedule, same initial buffers)
    offs, coefs, halo = oracle_terms(name, step)
    ga, gb = a0.copy(), np.full(shape, -3.0, dt)
    oracle.sweep(ga, gb, offs, coefs, halo)
    oracle.sweep(gb, ga, offs, coefs, halo)
    assert max_rel(A.cpu().numpy(), ga) <= (1e-5 if f32 else 1e-13)
