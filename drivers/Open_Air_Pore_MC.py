#!/usr/bin/env python
"""Drop-in driver for the thruster-pore stage (specular walls) on one B200.

Same entry point, constants, seeds, progress lines and result files (8 hist_*_data.txt in the
working directory) as the reference script of this name; the per-timestep work -- drift, the six
wall cases, out-of-bounds recapture, the 8-colour-group particle-particle pass and the mean-free-path
bookkeeping (reference lines 416-557) -- runs in libamc.so through argon_monte_carlo_b200.amc.
Differences: optional --steps/--outdir/--device flags (the reference has no CLI; without flags the
run is the reference's 20,000 steps), the every-100-steps "missed case" census is not printed, and
the two per-phase runtimes are device times.
"""
import os
import sys
from time import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from argon_monte_carlo_b200 import amc, config, driver_common, init_state  # noqa: E402

start = time()
cfg = config.pore_config(temperature=False)

if __name__ == "__main__":
    args = driver_common.parse_args(cfg.num_timesteps, __doc__)
    state = init_state.pore_initial_state(cfg)          # seeds 17 / 17, reference draw order
    sim = amc.Simulation(cfg, device=args.device)
    sim.set_state(*state)
    driver_common.sampling_begin(sim, args)
    print('Initialization Runtime: ' + str(time() - start) + ' seconds')
    print('  There are {} particles out of bounds after initialization.'.format(sim.recapture()))
    total_cols = total_errs = 0
    done = 0
    while done < args.steps:
        chunk = driver_common.flux_chunk(sim, args, done, driver_common.surface_chunk(sim, args, done, min(args.chunk, args.steps - done)))
        stats = sim.step(chunk)
        ms, _ = sim.last_timing()
        for k, s in enumerate(stats):
            print('  timestep', done + k, 'of', cfg.num_timesteps, '  (sim', 1, '/', 1, ')')
            print('    There are {} particles out of bounds after handling wall collisions.'.format(s["oob_after_walls"]))
            print('    Wall Step Runtime: ' + str(ms[0] / chunk * 1e-3) + ' seconds')
            print('    Num collisions from walls: ' + str(s["wall_collisions"]))
            print('    There are {} particles out of bounds after particle-particle collisions.'.format(s["oob_after_pp"]))
            print('    Particle-Particle step Runtime: ' + str((ms[1] + ms[2] + ms[3]) / chunk * 1e-3) + ' seconds')
            total_cols += s["collisions"]
            total_errs += s["errors"]
            print('   ', s["collisions"], ' collisions from this timestep')
        done += chunk
    driver_common.final_report(sim, total_errs, total_cols, start, args.outdir)
    driver_common.sampling_finish(sim, cfg, args)
    driver_common.surface_finish(sim, cfg, args)
    driver_common.flux_finish(sim, cfg, args)
    print('Runtime: ' + str((time() - start) / 60.0) + ' minutes')
    sim.close()
    driver_common.maybe_show(args.show)
