"""Host-side logic of the 2D slab path (drstencil_b200/slab.py on row slabs) with world_size 2 and 3 over gloo on CPU:
SlabGeometry over rows, SlabRunner's ping-pong schedule and halo_exchange on (rows, N) slices.  The sweep is a stand-in
supplied by the test (the CPU oracle restricted to the rank's output rows), so what is checked is that decomposed ==
undecomposed, bit for bit, including the frozen global ring."""
import os
import socket

import numpy as np
import pytest

from helpers import oracle_terms


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, name, step, shape, timesteps, out_dir):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from oracle import oracle
    from drstencil_b200.slab import SlabGeometry, SlabRunner, halo_exchange
    offs, coefs, halo = oracle_terms(name, step)
    M, N = shape
    geom = SlabGeometry(M, world, rank, halo)
    a_glob = oracle.rand_array(shape)
    A = np.zeros((geom.local_planes, N))
    B = np.zeros_like(A)
    for yl in range(geom.local_planes):
        yg = geom.origin + yl
        if 0 <= yg < M:
            A[yl] = a_glob[yg]
    tA, tB = torch.from_numpy(A), torch.from_numpy(B)

    def sweep(src, dst):
        s, d = src.numpy(), dst.numpy()
        keep = d.copy()
        oracle.sweep(s, d, offs, coefs, halo)            # writes local rows [halo, local_rows - halo)
        d[:geom.out_lo] = keep[:geom.out_lo]             # only the rank's output rows may change
        d[geom.out_hi:] = keep[geom.out_hi:]

    runner = SlabRunner(geom, [tA, tB], sweep, lambda dst, s: halo_exchange(dst, geom))
    n = runner.run(timesteps, step)
    np.save(os.path.join(out_dir, "rank%d.npy" % rank), tA.numpy()[geom.ghost:geom.ghost + geom.hi - geom.lo])
    np.save(os.path.join(out_dir, "n%d.npy" % rank), np.array([n]))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world,name,step,shape,timesteps", [
    (2, "2d5pt_star", 1, (23, 40), 6),
    (3, "2d9pt_box", 2, (31, 36), 8),
    (3, "2d25pt_box", 1, (14, 30), 4),          # Halo 2: rows [0, 4), [4, 9), [9, 14) -- a middle rank 5 rows thick
])
def test_decomposed_rows_equal_global(built, tmp_path, world, name, step, shape, timesteps):
    import torch.multiprocessing as mp
    from oracle import oracle
    port = _free_port()
    ctx = mp.get_context("spawn")
    procs = [ctx.Process(target=_worker, args=(r, world, port, name, step, shape, timesteps, str(tmp_path)))
             for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    got = np.concatenate([np.load(tmp_path / ("rank%d.npy" % r)) for r in range(world)], axis=0)
    offs, coefs, halo = oracle_terms(name, step)
    A = oracle.rand_array(shape)
    B = np.zeros(shape)
    n = oracle.run(A, B, offs, coefs, halo, timesteps, step)
    assert int(np.load(tmp_path / "n0.npy")[0]) == n
    assert np.array_equal(got, A)


def test_row_geometry():
    """SlabGeometry over the rows of c1's 4096^2 grid at N = 8: 512 rows per rank, one ghost row per side."""
    from drstencil_b200.slab import SlabGeometry
    g = SlabGeometry(4096, 8, 3, 1)
    assert (g.lo, g.hi, g.local_planes, g.out_lo, g.out_hi) == (1536, 2048, 514, 1, 513)
    assert (g.send_lower(), g.recv_lower(), g.send_upper(), g.recv_upper()) == ((1, 2), (0, 1), (512, 513), (513, 514))
    g = SlabGeometry(16384, 8, 0, 4)             # c2: 16384^2, Halo 4 (depth 4)
    assert (g.out_lo, g.out_hi, g.lower, g.upper) == (8, 2052, None, 1)
