#!/usr/bin/env python
"""Drop-in driver for the open-air cube stage on one B200.

Same entry point, constants, seed (127), progress lines and result files (8 hist_*_data.txt) as the
reference script of this name; the per-timestep work -- drift, six specular plane walls and the
serial lexicographic cell sweep with write-back after every cell (reference lines 175-338) -- runs in
libamc.so.  The reference's curve_fit of the histograms only feeds a plot label and is skipped.
"""
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from argon_monte_carlo_b200 import amc, config, driver_common, init_state, outputs  # noqa: E402

cfg = config.cube_config()
print(cfg.num_molecules)

if __name__ == "__main__":
    args = driver_common.parse_args(cfg.num_timesteps, __doc__)
    state = init_state.cube_initial_state(cfg)
    sim = amc.Simulation(cfg, device=args.device)
    sim.set_state(*state)
    driver_common.sampling_begin(sim, args)
    done = 0
    while done < args.steps:
        chunk = driver_common.flux_chunk(sim, args, done, driver_common.surface_chunk(sim, args, done, min(args.chunk, args.steps - done)))
        for k, s in enumerate(sim.step(chunk)):
            print('  timestep', done + k, 'of', cfg.num_timesteps, '  (sim', 1, '/', 1, ')')
            print('    ', s["pp_collisions"], ' collisions')
        done += chunk
    counts, n_paths, sums = sim.histograms()
    means = sums / n_paths if n_paths else sums * float("nan")
    for lab, m in zip(("mean free path: ", "mean x free path: ", "mean y free path: ", "mean z free path: "), means):
        print('Simulation 1 ' + lab + str(m))
    print('Num of collisions total: ' + str(n_paths))
    outputs.write_histograms(counts, args.outdir)
    driver_common.sampling_finish(sim, cfg, args)
    driver_common.surface_finish(sim, cfg, args)
    driver_common.flux_finish(sim, cfg, args)
    sim.close()
    driver_common.maybe_show(args.show)
