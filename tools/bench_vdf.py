#!/usr/bin/env python
"""Cost of the velocity distribution (amc_vdf_*) on the 12.5 M-particle energized-pore workload of bench.py (one GPU).

Three arms on the same seeded synthetic gas -- sampling off, field sampling every 10th step, field sampling + VDF
(200 bins, the drivers' default range) every 10th step -- run alternately in one process after a warm-up, each from its
own copy of the initial state.  Reported per arm: device time per step (CUDA events of amc_step) and, for the sampled
arms, the sampling kernel's time per sample (amc_last_sample_ms: k_sample<false> against k_sample<true>) and that time
against the byte floor of one sample (56 bytes per particle at the project's copy peak).  The card's name and power
limit are read in the same run.  The state digests of the three arms must agree.  Prints one JSON line; --out writes
it to a file as well.

    python tools/bench_vdf.py [--particles 12500000] [--steps 20] [--rounds 3] [--bins 200] [--out FILE]
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
from bench_sampling import BYTES_PER_PARTICLE, COPY_PEAK_GBS, card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--particles", type=int, default=12_500_000)
    ap.add_argument("--steps", type=int, default=20, help="timed steps per arm and round")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--bins", type=int, default=200)
    ap.add_argument("--out")
    args = ap.parse_args()
    import bench
    from argon_monte_carlo_b200 import amc, driver_common, init_state
    info = card()
    cfg, _ = bench.scaled_temp_config(args.particles)
    n = cfg.num_molecules
    v_max = driver_common.vdf_default_vmax(cfg)
    arms = {"off": (None, False), "fields_every_10": (10, False), "fields_vdf_every_10": (10, True)}
    sims = {}
    for name, (every, vdf) in arms.items():
        sim = amc.Simulation(cfg, seed=17, max_particles=n)
        sim.init_synthetic(init_state.pore_spec(cfg, seed=17))
        if every:
            sim.sample_enable(every, 0)
        if vdf:
            sim.vdf_enable(args.bins, v_max)
        sim.step_quiet(args.warmup)
        sims[name] = sim
    res = {name: {"ms_per_step": [], "sample_ms": [], "samples": 0} for name in arms}
    for _ in range(args.rounds):
        for name, sim in sims.items():
            before = sim.sample_raw()[1] if arms[name][0] else 0
            sim.step_quiet(args.steps)
            ms, _ = sim.last_timing()
            res[name]["ms_per_step"].append(ms[4] / args.steps)
            if arms[name][0]:
                k = sim.sample_raw()[1] - before
                res[name]["samples"] += k
                res[name]["sample_ms"].append(sim.last_sample_ms() / max(k, 1))
    digests = {name: ["%016x" % d for d in sim.state_digest()[:2]] for name, sim in sims.items()}
    for sim in sims.values():
        sim.close()
    floor_ms = n * BYTES_PER_PARTICLE / (COPY_PEAK_GBS * 1e9) * 1e3
    out = {"tool": "bench_vdf", "card": info, "particles": n, "steps_per_round": args.steps, "rounds": args.rounds,
           "vdf_bins": args.bins, "vdf_vmax": v_max, "sample_floor_ms": floor_ms, "copy_peak_gbs": COPY_PEAK_GBS,
           "arms": {}, "digests_equal": len({tuple(d) for d in digests.values()}) == 1, "digests": digests}
    for name, r in res.items():
        a = {"ms_per_step": float(np.median(r["ms_per_step"])), "ms_per_step_min": float(min(r["ms_per_step"])),
             "ms_per_step_max": float(max(r["ms_per_step"]))}
        if r["sample_ms"]:
            s = float(np.median(r["sample_ms"]))
            a.update(samples=r["samples"], sample_kernel_ms=s, sample_vs_floor=s / floor_ms)
        out["arms"][name] = a
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    if not out["digests_equal"]:
        sys.exit("state digests differ between the arms: the VDF or sampling changed the state")


if __name__ == "__main__":
    main()
