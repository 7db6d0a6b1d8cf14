"""GPU tests of the channel-sharded f-k filter (BASELINE config 4 path, das4whales_b200/dist.py) with the REAL CUDA backend:
d4w_fk_apply_pass_ex on time slabs (passes 1 / 5) and on kept-row ranges (passes 2-4).

* one GPU: G rank objects stepped through the schedule in one process (dist.run_local_group), which exercises the
  slab / slot arithmetic of the C entry point and the two-level / pipelined column kernels on slab plans;
* >= 2 GPUs: the same through torch.distributed all_to_all_single over NCCL, one process per GPU."""
import os
import sys

import numpy as np
import pytest

from conftest import rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DX, FS = 2.0419046878814697, 200.0


@pytest.fixture(scope="module")
def dw():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import das4whales_b200 as dw
    from das4whales_b200 import _lib
    _lib.lib()
    return dw


def _mask(dw, kind, nx, ns):
    if kind == "fan":
        return dw.dsp.fk_filter_design((nx, ns), [0, nx, 1], DX, FS)
    return dw.dsp.hybrid_ninf_filter_design((nx, ns), [0, nx, 1], DX, FS, 1350., 1450., 3300, 3450, 14., 30.)


@pytest.mark.parametrize("nx,ns,world,kind,taper,nsub", [
    (1000, 4800, 2, "fan", False, 1),        # 25 x 40: two-level, engine level B, separate launches
    (10000, 4800, 2, "fan", True, 1),        # 25 x 400: the pipelined kernels of the headline configuration, on 2400-sample slabs
    (10000, 4800, 4, "hybrid", False, 1),    # nothing pruned, 4 ranks, uneven row split (5001 rows)
    (600, 3600, 3, "fan", False, 1),         # 3 ranks
    (20000, 1920, 4, "fan", False, 1),       # config-4 channel count (25 x 800): two-level with the three-stage level B
    (10000, 9600, 2, "fan", True, 3),        # three sub-slabs of 1600 samples per rank (the overlapped schedule's slicing)
    (20000, 3840, 4, "fan", False, 2),       # config-4 channel count, two sub-slabs
])
def test_sharded_cuda_backend_local_group(dw, nx, ns, world, kind, taper, nsub):
    import torch
    from das4whales_b200 import dist as d4wdist
    from das4whales_b200.fk import FkFilter
    gen = torch.Generator(device="cuda").manual_seed(nx + ns)
    x = torch.randn((nx, ns), device="cuda", generator=gen)
    mask = _mask(dw, kind, nx, ns)
    ref = FkFilter(mask)(x, tapering=taper)                       # single-GPU path (checked against the oracle elsewhere)
    be = d4wdist.CudaBackend(mask, nx, ns, world, nsub=nsub)
    filters = [d4wdist.ShardedFkFilter(nx, ns, be, rank=r, world=world) for r in range(world)]
    cpr = nx // world
    ys = d4wdist.run_local_group(filters, [x[r * cpr:(r + 1) * cpr].contiguous() for r in range(world)], tapering=taper)
    got = torch.cat(ys, dim=0)
    e = rel_err(got.cpu().numpy(), ref.cpu().numpy())
    assert e[0] <= 5e-6 and e[1] <= 5e-6, e
    if nx * ns <= 5_000_000:
        from oracle import dsp_oracle as O
        xo = x.cpu().numpy().astype(np.float64)
        mo = (O.fk_filter_design((nx, ns), [0, nx, 1], DX, FS) if kind == "fan" else
              O.hybrid_ninf_filter_design((nx, ns), [0, nx, 1], DX, FS, 1350., 1450., 3300, 3450, 14., 30.))
        eo = rel_err(got.cpu().numpy(), O.fk_filter_filt(xo, mo, tapering=taper))
        assert eo[0] <= 2e-5, eo


def _nccl_worker(rank, world, port, nx, ns, q):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    import das4whales_b200 as dw
    from das4whales_b200 import dist as d4wdist
    from das4whales_b200.fk import FkFilter
    gen = torch.Generator(device="cuda").manual_seed(5)
    x = torch.randn((nx, ns), device="cuda", generator=gen)        # same matrix on every rank
    mask = dw.dsp.fk_filter_design((nx, ns), [0, nx, 1], DX, FS)
    ref = FkFilter(mask)(x)
    cpr = nx // world
    r = ref[rank * cpr:(rank + 1) * cpr]
    err = 0.0
    for nsub in (1, 3):                                            # serial schedule and the overlapped one (async all-to-alls)
        y = d4wdist.fk_filter_filt_sharded(x[rank * cpr:(rank + 1) * cpr].contiguous(), mask, nx, nsub=nsub)
        err = max(err, float((y - r).abs().max() / ref.abs().max()))
    q.put((rank, err))
    dist.destroy_process_group()


def test_sharded_two_gpus_nccl(dw):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29700 + os.getpid() % 200
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, 10000, 24000, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for rank, err in res:
        assert err <= 5e-6, (rank, err)
