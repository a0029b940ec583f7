"""Worker of tests/test_gpu_surface.py::test_multi_gpu_surface_matches_single_gpu (also usable directly):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        tests/nccl_surface_worker.py OUT.json [--mode p2p|nccl] [--steps K]

Every rank drives one z slab of the small dense energized pore (cuts inside the end caps) on its own GPU with surface
recording on -- --mode p2p: amc_slab_step; --mode nccl: the step-wise entry points over NCCL -- and the accumulators
are summed over the processes (DistTransport.allreduce_u64).  Rank 0 then runs the same job as a single domain and
compares the raw accumulators word for word.  Exit code 0 only if they are identical."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--mode", default="p2p", choices=["p2p", "nccl"])
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    from argon_monte_carlo_b200 import amc, config, init_state, slab
    world, rank, local = int(os.environ["WORLD_SIZE"]), int(os.environ["RANK"]), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cfg = config.pore_config(True, scale=0.5)
    state = init_state.synthetic_pore_state(cfg, seed=11)
    nz = cfg.grid.nc[2]
    cuts = {2: [0, 2, nz], 3: [0, 1, nz - 2, nz], 4: [0, 1, 2, nz - 1, nz]}.get(world)
    if cuts is None:
        cuts = [0, 1, 2, 3] + [nz - (world - 3) + k for k in range(world - 3)]
    cuts = np.array(cuts, dtype=np.int32)
    sim = slab.SlabSimulation(cfg, world, state[2], transport=slab.DistTransport(), local_ranks=[rank], devices=[local],
                              cuts=cuts, seed=17, p2p=args.mode == "p2p")
    layer = slab.owner_layer(state[2], cfg.grid.edge[2])
    m = (layer >= cuts[rank]) & (layer < cuts[rank + 1])
    sim.set_local_state(np.nonzero(m)[0], *[a[m] for a in state], n_global=len(state[0]))
    sim.surface_enable()
    dist.barrier()
    if args.mode == "p2p":
        sim.step_fused(args.steps)
    else:
        sim.step(args.steps)
    acc, ns, no = sim.surface_raw()
    sim.close()
    result = {"world": world, "mode": args.mode, "steps": args.steps, "cuts": [int(c) for c in cuts], "ok": True, "mismatch": []}
    if rank == 0:
        one = amc.Simulation(cfg, seed=17, device=local, max_particles=len(state[0]))
        one.set_state(*state)
        one.surface_enable()
        one.step(args.steps)
        ref = one.surface_raw()
        one.close()
        if ref[1] != ns or not np.array_equal(ref[2], no):
            result["mismatch"].append("n_steps / outside: single %s %s, %d ranks %s %s" % (ref[1], ref[2], world, ns, no))
        bad = int(np.count_nonzero(np.any(ref[0] != acc, axis=1)))
        if bad:
            result["mismatch"].append("%d elements differ" % bad)
        result.update(ok=not result["mismatch"], n_steps=ns, hits=int(acc[:, 0].sum()))
        with open(args.out, "w") as f:
            json.dump(result, f)
        print(json.dumps(result))
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if result["ok"] else 1)


if __name__ == "__main__":
    main()
