"""Worker of tests/test_gpu_vdf.py::test_multi_gpu_vdf_matches_single_gpu (also usable directly):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        tests/nccl_vdf_worker.py OUT.json [--steps K]

Every rank drives one z slab of the small dense pore (cuts inside the end caps) on its own GPU with amc_slab_step,
field sampling every second step and the velocity distribution on, and the histograms are summed over the processes
(DistTransport.allreduce_u64).  Rank 0 then runs the same job as a single domain and compares the words one by one.
Exit code 0 only if they are identical."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
BINS, VMAX = 200, 1650.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--steps", type=int, default=6)
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    from argon_monte_carlo_b200 import amc, config, init_state, slab
    world, rank, local = int(os.environ["WORLD_SIZE"]), int(os.environ["RANK"]), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cfg = config.pore_config(False, scale=0.5)
    state = init_state.synthetic_pore_state(cfg, seed=11)
    nz = cfg.grid.nc[2]
    cuts = {2: [0, 2, nz], 3: [0, 1, nz - 2, nz], 4: [0, 1, 2, nz - 1, nz]}.get(world)
    if cuts is None:
        cuts = [0, 1, 2, 3] + [nz - (world - 3) + k for k in range(world - 3)]
    cuts = np.array(cuts, dtype=np.int32)
    sim = slab.SlabSimulation(cfg, world, state[2], transport=slab.DistTransport(), local_ranks=[rank], devices=[local],
                              cuts=cuts, seed=17, p2p=True)
    layer = slab.owner_layer(state[2], cfg.grid.edge[2])
    m = (layer >= cuts[rank]) & (layer < cuts[rank + 1])
    sim.set_local_state(np.nonzero(m)[0], *[a[m] for a in state], n_global=len(state[0]))
    sim.sample_enable(2, 1)
    sim.vdf_enable(BINS, VMAX)
    dist.barrier()
    sim.step_fused(args.steps)
    vdf = sim.vdf_raw()
    ns = sim.sample_raw()[1]
    sim.close()
    result = {"world": world, "steps": args.steps, "cuts": [int(c) for c in cuts], "ok": True, "mismatch": []}
    if rank == 0:
        one = amc.Simulation(cfg, seed=17, device=local, max_particles=len(state[0]))
        one.set_state(*state)
        one.sample_enable(2, 1)
        one.vdf_enable(BINS, VMAX)
        one.step(args.steps)
        ref, ref_ns = one.vdf_raw(), one.sample_raw()[1]
        one.close()
        if ref_ns != ns:
            result["mismatch"].append("samples: single %s, %d ranks %s" % (ref_ns, world, ns))
        bad = int(np.count_nonzero(ref != vdf))
        if bad:
            result["mismatch"].append("%d words differ" % bad)
        result.update(ok=not result["mismatch"], samples=ns, particles_binned=int(vdf[:, 0].sum()))
        with open(args.out, "w") as f:
            json.dump(result, f)
        print(json.dumps(result))
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if result["ok"] else 1)


if __name__ == "__main__":
    main()
