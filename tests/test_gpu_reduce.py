"""The final reduction through the C ABI: pdmpflux_moments_reduce against numpy, and (with >= 2 GPUs) the library-owned
NCCL communicator: pdmpflux_comm_* + pdmpflux_moments_allreduce from two ranks."""
import ctypes as C
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def p():
    import pdmpflux_b200
    n = C.c_int(0)
    pdmpflux_b200.lib().pdmpflux_device_count(C.byref(n))
    assert n.value > 0, "GPU tests need a CUDA device"
    return pdmpflux_b200


@pytest.mark.parametrize("C_,d", [(1, 1), (37, 5), (4096, 50), (70000, 33), (513, 1000)])
def test_moments_reduce_matches_numpy(p, C_, d):
    from pdmpflux_b200 import _lib
    g = np.random.default_rng(C_ + d)
    m1 = g.standard_normal((C_, d)); m2 = 1.0 + g.random((C_, d)); T = 1.0 + g.random(C_)
    out = np.empty((4, d))
    _lib.check(p.lib().pdmpflux_moments_reduce(d, C_, m1.ctypes.data, m2.ctypes.data, T.ctypes.data, out.ctypes.data, 0, None))
    mean, sec = m1 / T[:, None], m2 / T[:, None]
    ref = p.dist.moment_sums(mean, sec)
    scale = np.abs(mean).sum(0).max() + C_
    assert np.abs(out - ref).max() < 1e-13 * scale
    assert np.all(out[3] == C_)
    # T = NULL: the inputs are already time averages; device pointers: same numbers bit for bit (fixed summation order)
    out2 = np.empty((4, d))
    _lib.check(p.lib().pdmpflux_moments_reduce(d, C_, mean.ctypes.data, sec.ctypes.data, None, out2.ctypes.data, 0, None))
    assert np.abs(out2 - ref).max() < 1e-13 * scale
    import torch
    dm, ds = torch.from_numpy(mean).cuda(), torch.from_numpy(sec).cuda()
    dout = torch.empty((4, d), dtype=torch.float64, device="cuda")
    p.dist.moment_sums_device(dm, ds, None, dout, torch.cuda.current_stream().cuda_stream)
    assert np.array_equal(dout.cpu().numpy(), out2)
    st = p.dist.ess_from_sums(dout)
    assert np.allclose(st["mean"], mean.mean(0), atol=1e-12)


def _rank(rank, world, port, q):
    import torch
    import torch.distributed as dist

    import pdmpflux_b200 as p
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    p.lib().pdmpflux_set_device(rank)
    dist.init_process_group("gloo", rank=rank, world_size=world)   # only carries the 128-byte unique id
    comm = p.dist.Comm()
    x = torch.full((4, 7), float(rank + 1), dtype=torch.float64, device="cuda")
    p.dist.all_reduce_sums(x, comm, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    q.put((rank, x.cpu().numpy()))
    dist.barrier()
    comm.close()
    dist.destroy_process_group()


def test_two_rank_nccl_allreduce_through_the_c_abi(p):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + os.getpid() % 2000
    procs = [ctx.Process(target=_rank, args=(r, 2, port, q)) for r in range(2)]
    for pr in procs:
        pr.start()
    got = dict(q.get(timeout=180) for _ in range(2))
    for pr in procs:
        pr.join(timeout=180)
        assert pr.exitcode == 0
    for r in range(2):
        assert np.all(got[r] == 3.0)
