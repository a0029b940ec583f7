"""Output writers of the three drivers: the eight histogram text files and momentum_energy.csv,
byte-compatible with what the reference scripts write (SURVEY Appendix D).

  hist_x_axis_*_data.txt = str(bins[0:200])    (Open_Air_Pore_MC.py:607-630, same in Cube / Temp)
  hist_y_axis_*_data.txt = str(n) with n = np.histogram(..., density=True)   (Pore:575-596)
  momentum_energy.csv    = pandas.DataFrame.from_dict({...}).to_csv          (Temperature_Pore_MC.py:929-933)

The device keeps the histogram *counts* (integers, exact); the density normalisation is the one
np.histogram applies: counts / diff(edges) / counts.sum().
"""
from __future__ import annotations

import os
import sys

import numpy as np

from .config import HIST_RANGE, NUM_BINS

SUFFIXES = ("total", "x", "y", "z")


def bin_edges():
    return np.linspace(HIST_RANGE[0], HIST_RANGE[1], NUM_BINS + 1)


def density(counts):
    """np.histogram(..., density=True) from integer counts (numpy/lib/_histograms_impl.py:873-875)."""
    counts = np.asarray(counts)
    db = np.array(np.diff(bin_edges()), float)
    with np.errstate(divide="ignore", invalid="ignore"):
        return counts / db / counts.sum()


def write_histograms(counts4, directory="."):
    """counts4: [4][200] integer counts in the order total, x, y, z."""
    edges = bin_edges()
    old = np.get_printoptions()
    np.set_printoptions(threshold=sys.maxsize)      # the reference sets this at import (Pore:12)
    try:
        for j, suffix in enumerate(SUFFIXES):
            n = density(counts4[j])
            with open(os.path.join(directory, "hist_x_axis_%s_data.txt" % suffix), "w") as f:
                f.write(str(edges[0:len(n)]))
            with open(os.path.join(directory, "hist_y_axis_%s_data.txt" % suffix), "w") as f:
                f.write(str(n))
    finally:
        np.set_printoptions(**old)


def write_momentum_energy_csv(momentum, energy_cold, energy_hot, path="momentum_energy.csv"):
    """Per-step series as the reference prints them: mpf values through pandas, i.e. 15 significant
    digits (a step without an energized hit stays the Python int 0, as in the reference)."""
    import mpmath
    import pandas as pd

    def conv(v):
        if isinstance(v, (int,)) and v == 0:
            return 0
        return v if isinstance(v, mpmath.mpf) else mpmath.mpf(float(v))
    data = {"Momentum": [conv(v) for v in momentum],
            "EnergyCold": [conv(v) for v in energy_cold],
            "EnergyHot": [conv(v) for v in energy_hot]}
    pd.DataFrame.from_dict(data).to_csv(path)


# ---------------------------------------------------------------- sampled fields (amc_sample_*)
PROFILE_COLUMNS = ("z_lo", "z_hi", "samples", "particles_per_sample", "number_density", "vz_mean", "temperature",
                   "temperature_x", "temperature_y", "temperature_z")


def decode_sample_sums(acc):
    """acc [cells][13] uint64 (Simulation.sample_raw) -> (count [cells], sum v [cells, 3], sum v^2 [cells, 3]) as
    float64: every sum is high * 2^-S1 + low * 2^-S2 of its two signed limbs (include/amc.h)."""
    from .amc import SAMPLE_Q1, SAMPLE_Q2, SAMPLE_V1, SAMPLE_V2
    w = np.ascontiguousarray(acc, dtype=np.uint64).reshape(-1, 13).view(np.int64)
    dec = lambda j, s1, s2: np.ldexp(w[:, j].astype(np.float64), -s1) + np.ldexp(w[:, j + 1].astype(np.float64), -s2)
    count = w[:, 0].view(np.uint64).astype(np.float64)
    sv = np.stack([dec(1 + 2 * a, SAMPLE_V1, SAMPLE_V2) for a in range(3)], axis=1)
    sq = np.stack([dec(7 + 2 * a, SAMPLE_Q1, SAMPLE_Q2) for a in range(3)], axis=1)
    return count, sv, sq


def _moments_to_fields(count, sv, sq, n_samples, cfg):
    """Means and temperatures from particle counts and sums; T_a = m / k_B (<v_a^2> - <v_a>^2), T = mean of the three."""
    m, kb = float(cfg.argon_mass), float(cfg.boltzman)
    with np.errstate(invalid="ignore", divide="ignore"):
        mean = sv / count[:, None]
        t_axes = m / kb * (sq / count[:, None] - mean * mean)
        pps = count / n_samples if n_samples else np.full_like(count, np.nan)
    return {"count": count, "particles_per_sample": pps, "v_mean": mean, "temperature_axes": t_axes,
            "temperature": t_axes.mean(axis=1)}


def sample_fields(raw, cfg):
    """Per-cell fields of raw = (acc, n_samples, n_outside): particles per sample, mean velocity [cells, 3],
    temperature T = m / (3 k_B) (<v^2> - |<v>|^2) and its axis parts [cells, 3], with the config's own argon_mass and
    boltzman.  Cells without a particle give NaN means."""
    acc, n_samples, _ = raw
    count, sv, sq = decode_sample_sums(acc)
    return _moments_to_fields(count, sv, sq, int(n_samples), cfg)


def _overlap(lo, hi, a, b):
    return np.maximum(0.0, np.minimum(hi, b) - np.maximum(lo, a))


def layer_volumes(cfg, z_edges):
    """Volume each z layer [z_edges[k], z_edges[k+1]) offers to particle centres.  Pore: the piecewise cylinder of
    collision radii -- open air R_oa_c on [0, oah] and [z_cold, H], coated pore R_p_c on [oah, z_gb] and [z_gt, z_cold],
    gap R_g_c on [z_gb, z_gt] -- with layers that straddle a boundary split exactly.  Cube: the layer's box."""
    lo, hi = np.asarray(z_edges[:-1], dtype=np.float64), np.asarray(z_edges[1:], dtype=np.float64)
    if cfg.kind == "cube":
        return float(cfg.cube_x) * float(cfg.cube_y) * _overlap(lo, hi, 0.0, float(cfg.cube_z))
    g = cfg.geom
    regions = ((0.0, g.oah, g.R_oa_c), (g.oah, g.z_gb, g.R_p_c), (g.z_gb, g.z_gt, g.R_g_c), (g.z_gt, g.z_cold, g.R_p_c),
               (g.z_cold, g.H, g.R_oa_c))
    return sum(np.pi * float(r) ** 2 * _overlap(lo, hi, float(a), float(b)) for a, b, r in regions)


def axial_profile(raw, cfg, grid=None):
    """Fields of every z layer of the sampling grid (default cfg.grid): the per-cell sums of the layer added up, then
    the number density over the layer's centre-accessible volume (layer_volumes).  Returns a dict of the
    PROFILE_COLUMNS arrays."""
    grid = grid or cfg.grid
    acc, n_samples, _ = raw
    nx, ny, nz = (int(v) for v in grid.nc)
    count, sv, sq = decode_sample_sums(acc)
    layer = lambda a: a.reshape(nx * ny, nz, *a.shape[1:]).sum(axis=0)
    f = _moments_to_fields(layer(count), layer(sv), layer(sq), int(n_samples), cfg)
    z = np.asarray(grid.edge[2], dtype=np.float64)
    vol = layer_volumes(cfg, z)
    with np.errstate(invalid="ignore", divide="ignore"):
        density = f["particles_per_sample"] / vol
    return {"z_lo": z[:-1], "z_hi": z[1:], "samples": np.full(nz, int(n_samples), dtype=np.int64),
            "particles_per_sample": f["particles_per_sample"], "number_density": density, "vz_mean": f["v_mean"][:, 2],
            "temperature": f["temperature"], "temperature_x": f["temperature_axes"][:, 0],
            "temperature_y": f["temperature_axes"][:, 1], "temperature_z": f["temperature_axes"][:, 2]}


def write_axial_profile(path, profile):
    """profile_z.csv: one row per z layer, the PROFILE_COLUMNS (number density in particles per m^3, velocities in
    m/s, temperatures in K), floats with 17 significant digits."""
    with open(path, "w") as f:
        f.write(",".join(PROFILE_COLUMNS) + "\n")
        for k in range(len(profile["z_lo"])):
            f.write(",".join(str(int(profile[c][k])) if c == "samples" else "%.17g" % float(profile[c][k])
                             for c in PROFILE_COLUMNS) + "\n")
