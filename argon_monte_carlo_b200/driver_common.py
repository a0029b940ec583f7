"""Shared pieces of the three drop-in driver scripts (drivers/*.py): the optional command line the
reference does not have, the end-of-run report and the output files."""
from __future__ import annotations

import argparse
import os
from time import time

import numpy as np

from . import outputs


VDF_VMAX_SIGMAS = 6.0   # default VDF range: this many thermal speeds; P(|v_a - u_a| > 6 sigma) = 2e-9 per component


def vdf_default_vmax(cfg):
    """VDF_VMAX_SIGMAS * sqrt(k_B T / m) at the hottest wall temperature of the config (the ambient temperature where the
    walls have none of their own)."""
    t = max(float(getattr(cfg, k)) for k in ("temp_ambient", "t_cold", "t_hot") if hasattr(cfg, k))
    return VDF_VMAX_SIGMAS * float(np.sqrt(float(cfg.boltzman) * t / float(cfg.argon_mass)))


def parse_args(default_steps, description, temp=False, argv=None):
    ap = argparse.ArgumentParser(description=description)
    ap.add_argument("--steps", type=int, default=int(os.environ.get("AMC_STEPS", default_steps)),
                    help="number of timesteps (default: the script's own num_timesteps = %d)" % default_steps)
    ap.add_argument("--outdir", default=os.environ.get("AMC_OUTDIR", "."), help="where the result files go (default: CWD)")
    ap.add_argument("--device", type=int, default=int(os.environ.get("AMC_DEVICE", 0)))
    ap.add_argument("--chunk", type=int, default=100, help="timesteps per device call (device-RNG / specular runs)")
    if temp:
        ap.add_argument("--rng", choices=["host", "device"], default=os.environ.get("AMC_RNG", "host"),
                        help="host: the reference's Mersenne-Twister draws in its order (reproduces "
                             "momentum_energy.csv); device: Philox on the GPU, no host round trips")
    ap.add_argument("--show", action="store_true", help="plt.show() at the end if matplotlib is installed")
    ap.add_argument("--sample-every", type=int, default=0, metavar="K",
                    help="sample density, flow velocity and temperature per collision cell after every K-th timestep "
                         "and write profile_z.csv (default 0: off)")
    ap.add_argument("--sample-start", type=int, default=0, metavar="S", help="first timestep sampled (default 0)")
    ap.add_argument("--surface-start", type=int, default=None, metavar="S",
                    help="record wall pressure, shear stress and heat flux per wall element from timestep S to the end "
                         "and write surface.csv (default: off)")
    ap.add_argument("--flux-start", type=int, default=None, metavar="S",
                    help="count the particles crossing every z plane of the sampling grid, with their momentum and "
                         "energy, from timestep S to the end and write flux_z.csv (default: off)")
    ap.add_argument("--vdf-bins", type=int, default=0, metavar="N",
                    help="with --sample-every: also histogram vx, vy, vz and the speed per z layer on the sampled steps, "
                         "N bins each, and write vdf_z.csv (default 0: off)")
    ap.add_argument("--vdf-vmax", type=float, default=None, metavar="V",
                    help="range of the VDF in m/s: [-V, V] for the components, [0, V] for the speed (default: "
                         "%g times the thermal speed sqrt(k_B T / m) at the config's hottest wall temperature)" % VDF_VMAX_SIGMAS)
    args = ap.parse_args(argv)
    if args.sample_every < 0 or args.sample_start < 0:
        ap.error("--sample-every and --sample-start must be >= 0")
    if args.vdf_bins:
        if args.sample_every <= 0:
            ap.error("--vdf-bins extends the field sample: it needs --sample-every")
        if not 1 <= args.vdf_bins <= 4096:
            ap.error("--vdf-bins must be in [1, 4096]")
    if args.vdf_vmax is not None and (args.vdf_bins <= 0 or not (np.isfinite(args.vdf_vmax) and args.vdf_vmax > 0)):
        ap.error("--vdf-vmax needs --vdf-bins and must be finite and > 0")
    if args.surface_start is not None and args.surface_start < 0:
        ap.error("--surface-start must be >= 0")
    if args.flux_start is not None and args.flux_start < 0:
        ap.error("--flux-start must be >= 0")
    return args


def surface_chunk(sim, args, done, chunk):
    """The number of timesteps to take from timestep `done` on, at most `chunk`: a batch never straddles
    --surface-start, and recording starts when the run reaches it."""
    s = args.surface_start
    if s is None:
        return chunk
    if done >= s and not sim.surface_on:
        sim.surface_enable()
    return s - done if done < s < done + chunk else chunk


def surface_finish(sim, cfg, args):
    """Write surface.csv (one row per wall element) into --outdir if --surface-start was given."""
    if args.surface_start is None:
        return
    if not sim.surface_on:      # the run ended before timestep S: nothing recorded
        sim.surface_enable()
    grid = getattr(sim, "sample_grid", cfg.grid)
    outputs.write_surface_csv(os.path.join(args.outdir, "surface.csv"), outputs.surface_fields(sim.surface_raw(), cfg, grid, sim.kind))


def flux_chunk(sim, args, done, chunk):
    """The number of timesteps to take from timestep `done` on, at most `chunk`: a batch never straddles
    --flux-start, and recording starts when the run reaches it."""
    s = args.flux_start
    if s is None:
        return chunk
    if done >= s and not sim.flux_on:
        sim.flux_enable()
    return s - done if done < s < done + chunk else chunk


def flux_finish(sim, cfg, args):
    """Write flux_z.csv (one row per z plane) into --outdir if --flux-start was given."""
    if args.flux_start is None:
        return
    if not sim.flux_on:         # the run ended before timestep S: nothing recorded
        sim.flux_enable()
    grid = getattr(sim, "sample_grid", cfg.grid)
    outputs.write_flux_csv(os.path.join(args.outdir, "flux_z.csv"), outputs.flux_fields(sim.flux_raw(), cfg, grid, sim.kind))


def sampling_begin(sim, args):
    """Enable field sampling on `sim` if --sample-every asks for it, and the VDF if --vdf-bins does."""
    if args.sample_every > 0:
        sim.sample_enable(args.sample_every, args.sample_start)
        if args.vdf_bins:
            sim.vdf_enable(args.vdf_bins, args.vdf_vmax or vdf_default_vmax(sim.cfg))


def sampling_finish(sim, cfg, args):
    """Write profile_z.csv (one row per z layer) and, with --vdf-bins, vdf_z.csv into --outdir if sampling was on."""
    if args.sample_every > 0:
        raw = sim.sample_raw()
        outputs.write_axial_profile(os.path.join(args.outdir, "profile_z.csv"), outputs.axial_profile(raw, cfg))
        if args.vdf_bins:
            fields = outputs.vdf_fields(sim.vdf_raw(), sim.vdf_layout(), raw, cfg)
            outputs.write_vdf_csv(os.path.join(args.outdir, "vdf_z.csv"), fields)


def final_report(sim, total_errs, total_cols, start, outdir, show=False, labels=("Simulation mean free path: ",
                 "Simulation mean x free path: ", "Simulation mean y free path: ", "Simulation mean z free path: ")):
    counts, n_paths, sums = sim.histograms()
    print(' ', total_errs, ' errors/warnings - potential lost particles')
    print(' ', total_cols, ' collisions')
    print(' ', n_paths, ' completed paths')
    with np.errstate(invalid="ignore", divide="ignore"):
        means = sums / n_paths if n_paths else np.full(4, np.nan)
    for lab, m in zip(labels, means):
        print(lab + str(m))
    print('Num of measured full paths total: ' + str(n_paths))
    print('Runtime: ' + str((time() - start) / 60.0) + ' minutes (pre histogram data rewrite)')
    outputs.write_histograms(counts, outdir)
    return counts, n_paths, means


def maybe_show(show):
    if not show:
        return
    try:
        import matplotlib.pyplot as plt
        plt.show()
    except Exception:
        pass
