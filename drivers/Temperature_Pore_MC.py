#!/usr/bin/env python
"""Drop-in driver for the energized-wall stage on one B200.

Same entry point, constants, seeds, progress lines and result files (8 hist_*_data.txt and
momentum_energy.csv in the working directory) as the reference script of this name; the
per-timestep work (reference lines 662-853) runs in libamc.so.

--rng host (default) keeps the reference's two Mersenne-Twister streams on the host and feeds the
directions to the device case by case, in the reference's order, so momentum_energy.csv comes out
as the reference writes it (rows 0-1 of the shipped file digit for digit; later rows to the
floating-point noise of NumPy-scalar pow).  --rng device draws on the GPU (Philox) with no host
round trips: same physics, different random stream.
"""
import os
import sys
from time import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from argon_monte_carlo_b200 import amc, config, driver_common, init_state, outputs  # noqa: E402

start = time()
cfg = config.pore_config(temperature=True)


def census_after_init(x, y, z, g):
    """num_out_of_bounds() right after initialisation (report only; reference lines 560-592)."""
    r2 = x**2 + y**2
    masks = [z < 0, z > g.H, (r2 > g.R_oa_sq) & (z >= 0) & (z <= g.oah), (r2 > g.R_oa_sq) & (z >= g.z_cold) & (z <= g.H),
             (r2 > g.R_g_sq) & (z >= g.z_gb) & (z <= g.z_gt), (r2 > g.R_p_sq) & (z > g.oah) & (z < g.z_gb),
             (r2 > g.R_p_sq) & (z > g.z_gt) & (z < g.z_cold)]
    return int(sum(m.sum() for m in masks))


if __name__ == "__main__":
    args = driver_common.parse_args(cfg.num_timesteps, __doc__, temp=True)
    state = init_state.pore_initial_state(cfg)          # seeds 17 / 17, reference draw order
    host = args.rng == "host"
    sim = amc.Simulation(cfg, device=args.device, rng_mode=amc.RNG_HOST if host else amc.RNG_DEVICE)
    sim.set_state(*state)
    driver_common.sampling_begin(sim, args)
    print('Initialization Runtime: ' + str(time() - start) + ' seconds')
    print('  There are {} particles out of bounds after initialization.'.format(census_after_init(*state[:3], cfg.geom)))
    momentum, e_hot, e_cold = [], [], []
    total_cols = total_errs = 0
    done = 0
    while done < args.steps:
        chunk = driver_common.flux_chunk(sim, args, done, driver_common.surface_chunk(sim, args, done, 1 if host else min(args.chunk, args.steps - done)))
        t0 = time()
        stats = [sim.step_host_rng()] if host else sim.step(chunk)
        wall_dt = (time() - t0) / chunk
        ms = None if host else sim.last_timing()[0]
        for k, s in enumerate(stats):
            print('  timestep', done + k, 'of', cfg.num_timesteps, '  (sim', 1, '/', 1, ')')
            print('    There are {} particles out of bounds after handling wall collisions.'.format(s["oob_after_walls"]))
            print('    There are {} particles out of bounds after post wall collision recapture.'.format(s["oob_after_walls_recapture"]))
            print('    Wall Step Runtime: ' + str(wall_dt if host else ms[0] / chunk * 1e-3) + ' seconds')
            print('    Num collisions from walls: ' + str(s["wall_collisions"]))
            print('    There are {} particles out of bounds after particle-particle collisions.'.format(s["oob_after_pp"]))
            print('    There are {} particles out of bounds after post particle-particle recapture.'.format(s["oob_after_pp_recapture"]))
            print('    Particle-Particle step Runtime: ' + str(wall_dt if host else (ms[1] + ms[2] + ms[3]) / chunk * 1e-3) + ' seconds')
            total_cols += s["collisions"]
            total_errs += s["errors"]
            print('   ', s["collisions"], ' collisions from this timestep')
            print(' ', total_errs, ' errors/warnings so far')
            momentum.append(s["dpz"]); e_hot.append(s["e_hot"]); e_cold.append(s["e_cold"])
        done += chunk
    driver_common.final_report(sim, total_errs, total_cols, start, args.outdir)
    driver_common.sampling_finish(sim, cfg, args)
    driver_common.surface_finish(sim, cfg, args)
    driver_common.flux_finish(sim, cfg, args)
    outputs.write_momentum_energy_csv(momentum, e_cold, e_hot, os.path.join(args.outdir, "momentum_energy.csv"))
    import mpmath
    for series in (momentum, e_cold, e_hot):
        print(sum(mpmath.mpf(float(v)) if not isinstance(v, int) else v for v in series))
    print('Runtime: ' + str((time() - start) / 60.0) + ' minutes')
    sim.close()
    driver_common.maybe_show(args.show)
