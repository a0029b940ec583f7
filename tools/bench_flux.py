#!/usr/bin/env python
"""Cost of plane flux recording (amc_flux_*) on the 12.5 M-particle energized-pore workload of bench.py (one GPU).

Two arms on the same seeded synthetic gas -- recording off and recording on -- run alternately in one process after a
warm-up, each from its own copy of the initial state; reported per arm: device time per step (CUDA events of amc_step)
and the share of it after the pair kernels ([3] of amc_last_timing: the closing recapture and, with recording on, the
flux kernel; recording closes every step with its own recapture launch).  The card's name and power limit are read in
the same run.  The state digests of the two arms must agree (recording changes nothing).  Prints one JSON line; --out
writes it to a file as well.

    python tools/bench_flux.py [--particles 12500000] [--steps 20] [--rounds 4] [--out FILE]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True     # importing bench.py leaves no cache in the tree


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--particles", type=int, default=12_500_000)
    ap.add_argument("--steps", type=int, default=20, help="timed steps per arm and round")
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out")
    args = ap.parse_args()
    import bench
    from bench_sampling import card
    from argon_monte_carlo_b200 import amc, init_state
    info = card()
    cfg, _ = bench.scaled_temp_config(args.particles)
    n = cfg.num_molecules
    sims = {}
    for name in ("off", "on"):
        sim = amc.Simulation(cfg, seed=17, max_particles=n)
        sim.init_synthetic(init_state.pore_spec(cfg, seed=17))
        if name == "on":
            sim.flux_enable()
        sim.step_quiet(args.warmup)
        sims[name] = sim
    res = {name: {"ms_per_step": [], "tail_ms_per_step": []} for name in sims}
    for _ in range(args.rounds):
        for name, sim in sims.items():
            sim.step_quiet(args.steps)
            ms, _ = sim.last_timing()
            res[name]["ms_per_step"].append(ms[4] / args.steps)
            res[name]["tail_ms_per_step"].append(ms[3] / args.steps)
    acc, n_steps = sims["on"].flux_raw()
    digests = {name: ["%016x" % d for d in sim.state_digest()[:2]] for name, sim in sims.items()}
    for sim in sims.values():
        sim.close()
    crossings = int(acc[:, 0].sum() + acc[:, 1].sum())
    out = {"tool": "bench_flux", "card": info, "particles": n, "planes": int(acc.shape[0]), "steps_per_round": args.steps,
           "rounds": args.rounds, "recorded_steps": n_steps, "plane_crossings_per_step": crossings / max(n_steps, 1),
           "digests_equal": digests["off"] == digests["on"], "digests": digests, "arms": {}}
    for name, r in res.items():
        out["arms"][name] = {k: {"median": float(np.median(v)), "min": float(min(v)), "max": float(max(v)), "all": [float(x) for x in v]}
                             for k, v in r.items()}
    off, on = out["arms"]["off"]["ms_per_step"]["median"], out["arms"]["on"]["ms_per_step"]["median"]
    out["step_overhead"] = on / off - 1.0
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    if not out["digests_equal"]:
        sys.exit("state digests differ between the arms: recording changed the state")


if __name__ == "__main__":
    main()
