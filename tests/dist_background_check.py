"""Background fields on the slab decomposition, run under torchrun (one rank per GPU):
    torchrun --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29536 tests/dist_background_check.py
A y-dependent background U(y) on u and B = N² z on b: every rank tabulates the backgrounds at its own slab's nodes and halos
(no exchange), and the decomposed model must reproduce the single-process oracle with the same backgrounds to <= 1e-12 per step."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "clima-oceananigans.jl_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)


def main():
    import torch
    import torch.distributed as dist
    import oracle as O
    import ocean_b200 as ob
    from background_reference import BackgroundNonhydrostaticModel

    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    rank, R = dist.get_rank(), dist.get_world_size()
    arch = ob.MultiArch.from_torch_distributed(local_rank)
    N = (64, 16 * R if 16 * R >= 32 else 32, 32)
    L = (1.0, 2.0, 1.5)
    topo = ("Periodic",) * 3
    bg = {"u": lambda x, y, z, t: 0.2 * np.sin(np.pi * y), "b": lambda x, y, z, t: 0.5 * z}
    go = O.RectilinearGrid(np.float64, size=N, extent=L, topology=topo)
    gb = ob.RectilinearGrid(arch, np.float64, size=N, extent=L, topology=topo)
    mo = BackgroundNonhydrostaticModel(go, background_fields=bg, advection=O.WENO5(), tracers=("b",),
                                       buoyancy=O.BuoyancyTracer(), timestepper="RungeKutta3")
    mb = ob.NonhydrostaticModel(gb, advection=ob.WENO5(), tracers=("b",), buoyancy=ob.BuoyancyTracer(),
                                timestepper="RungeKutta3", background_fields=bg)
    rng = np.random.default_rng(7)
    vals = {}
    for n in "uvw":
        a = rng.uniform(-1, 1, N)
        vals[n] = a - a.mean()
    vals["b"] = 0.1 * rng.uniform(-1, 1, N)
    mo.set(**vals)
    sl = mb.grid.local_slice()
    ob.set_model(mb, **{n: v[sl] for n, v in vals.items()})
    worst = 0.0
    for step in range(3):
        mo.time_step(2e-3)
        ob.time_step(mb, 2e-3)
        for n in mo.names:
            a, b = mb.fields[n].interior(), mo.fields[n].interior[sl]
            e = float(np.max(np.abs(a - b)) / np.max(np.abs(mo.fields[n].interior)))
            worst = max(worst, e)
            assert e < 1e-12, (rank, step, n, e)
    t = torch.tensor([worst], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        print(f"DIST_BACKGROUND_OK ranks={R} global={N} worst_rel_err={t[0].item():.3e}")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
