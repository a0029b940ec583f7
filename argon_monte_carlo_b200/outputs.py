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


# ---------------------------------------------------------------- velocity distribution (amc_vdf_*)
VDF_NAMES = ("vx", "vy", "vz", "speed")
VDF_COLUMNS = ("z_lo", "z_hi", "histogram", "bin", "v_lo", "v_hi", "count", "pdf", "maxwellian", "under_fraction",
               "over_fraction", "l1")


def maxwell_component_cdf(v, u, sigma):
    """CDF of one velocity component of a Maxwellian with drift u and sigma = sqrt(k_B T / m)."""
    from scipy.special import erf
    return 0.5 * (1.0 + erf((np.asarray(v, dtype=np.float64) - u) / (sigma * np.sqrt(2.0))))


def maxwell_speed_cdf(c, u, sigma):
    """CDF of the speed |v| of a Maxwellian with drift speed u = |<v>| and sigma = sqrt(k_B T / m):
    (erf((c-u)/(s sqrt2)) + erf((c+u)/(s sqrt2))) / 2 - s / (u sqrt(2 pi)) (exp(-(c-u)^2/2s^2) - exp(-(c+u)^2/2s^2)),
    at u = 0 the Maxwell-Boltzmann speed CDF erf(c/(s sqrt2)) - sqrt(2/pi) (c/s) exp(-c^2/2s^2)."""
    from scipy.special import erf
    c = np.asarray(c, dtype=np.float64)
    r2 = sigma * np.sqrt(2.0)
    if u <= 1e-6 * sigma:
        return erf(c / r2) - np.sqrt(2.0 / np.pi) * (c / sigma) * np.exp(-c * c / (2 * sigma * sigma))
    return (0.5 * (erf((c - u) / r2) + erf((c + u) / r2))
            - sigma / (u * np.sqrt(2 * np.pi)) * (np.exp(-(c - u) ** 2 / (2 * sigma * sigma)) - np.exp(-(c + u) ** 2 / (2 * sigma * sigma))))


def vdf_fields(raw, layout, sample_raw, cfg, grid=None):
    """Per z layer and histogram (vx, vy, vz, speed) of the VDF words raw [ncz][4][n_bins + 2] (Simulation.vdf_raw)
    with layout (ncz, n_bins, v_max) and the field sample sample_raw = (acc, n_samples, n_outside) taken with it:
      pdf         the measured pdf over the in-range counts (np.histogram's density=True), [ncz, 4, n_bins]
      under_fraction, over_fraction   the share of the layer's particles below / above the range, [ncz, 4]
      maxwellian  the Maxwellian at the layer's sampled drift velocity and temperature (axial_profile), averaged over
                  each bin: (CDF(v_hi) - CDF(v_lo)) / width; not renormalised to the range, [ncz, 4, n_bins]
      l1          sum over bins of |pdf - maxwellian| * width, [ncz, 4]
    with the config's own argon_mass and boltzman.  Layers without a particle give NaN."""
    from .amc import vdf_edges
    grid = grid or cfg.grid
    ncz, nb, vmax = int(layout[0]), int(layout[1]), float(layout[2])
    words = np.asarray(raw, dtype=np.uint64).reshape(ncz, 4, nb + 2)
    acc = words.astype(np.float64)
    prof = axial_profile(sample_raw, cfg, grid)
    acc_s = np.asarray(sample_raw[0], dtype=np.uint64).reshape(-1, 13)
    nx, ny = int(grid.nc[0]), int(grid.nc[1])
    count, sv, _ = decode_sample_sums(acc_s)
    with np.errstate(invalid="ignore", divide="ignore"):
        drift = sv.reshape(nx * ny, ncz, 3).sum(axis=0) / count.reshape(nx * ny, ncz).sum(axis=0)[:, None]
        sigma = np.sqrt(float(cfg.boltzman) * prof["temperature"] / float(cfg.argon_mass))
    ec, es = vdf_edges(nb, vmax)
    edges = [ec, ec, ec, es]
    width = np.stack([np.diff(e) for e in edges])                       # [4, n_bins]
    bins, total = acc[:, :, 1:-1], acc.sum(axis=2)
    inside = bins.sum(axis=2)
    maxw = np.full((ncz, 4, nb), np.nan)
    for k in range(ncz):
        if not (np.isfinite(sigma[k]) and sigma[k] > 0):
            continue
        for j in range(3):
            cdf = maxwell_component_cdf(ec, drift[k, j], sigma[k])
            maxw[k, j] = np.diff(cdf) / width[j]
        maxw[k, 3] = np.diff(maxwell_speed_cdf(es, float(np.sqrt(np.sum(drift[k] ** 2))), sigma[k])) / width[3]
    with np.errstate(invalid="ignore", divide="ignore"):
        pdf = bins / (inside[:, :, None] * width[None])
        under, over = acc[:, :, 0] / total, acc[:, :, -1] / total
        l1 = np.sum(np.abs(pdf - maxw) * width[None], axis=2)
    l1[inside == 0] = np.nan
    z = np.asarray(grid.edge[2], dtype=np.float64)
    return {"z_lo": z[:-1], "z_hi": z[1:], "n_bins": nb, "v_max": vmax, "edges": edges, "counts": words[:, :, 1:-1],
            "particles": total, "temperature": prof["temperature"], "drift": drift, "pdf": pdf, "maxwellian": maxw,
            "under_fraction": under, "over_fraction": over, "l1": l1}


def write_vdf_csv(path, fields):
    """vdf_z.csv: one row per z layer, histogram (vx, vy, vz, speed) and bin, the VDF_COLUMNS of vdf_fields (velocities in
    m/s, pdfs in s/m; the per-histogram under / over fractions and l1 repeated on every bin row), floats with 17
    significant digits."""
    nb = fields["n_bins"]
    with open(path, "w") as f:
        f.write(",".join(VDF_COLUMNS) + "\n")
        for k in range(len(fields["z_lo"])):
            for j, name in enumerate(VDF_NAMES):
                e = fields["edges"][j]
                tail = "%.17g,%.17g,%.17g" % (fields["under_fraction"][k, j], fields["over_fraction"][k, j], fields["l1"][k, j])
                for b in range(nb):
                    f.write("%.17g,%.17g,%s,%d,%.17g,%.17g,%d,%.17g,%.17g,%s\n" % (
                        fields["z_lo"][k], fields["z_hi"][k], name, b, e[b], e[b + 1], int(fields["counts"][k, j, b]),
                        fields["pdf"][k, j, b], fields["maxwellian"][k, j, b], tail))


# ---------------------------------------------------------------- wall surfaces (amc_surface_*)
SURFACE_COLUMNS = ("element", "case", "lo1", "hi1", "lo2", "hi2", "area", "hits", "number_flux", "pressure", "shear_1",
                   "shear_2", "heat_flux")


def decode_surface_sums(acc):
    """acc [elements][9] uint64 (Simulation.surface_raw) -> (hits [elements], sums [elements, 4]: dv.n, dv.t1, dv.t2
    in m/s and dE in J) as float64, each sum high * 2^-S1 + low * 2^-S2 of its signed limbs (include/amc.h)."""
    from .amc import SURF_E1, SURF_E2, SURF_V1, SURF_V2, SURF_WORDS
    w = np.ascontiguousarray(acc, dtype=np.uint64).reshape(-1, SURF_WORDS).view(np.int64)
    dec = lambda j, s1, s2: np.ldexp(w[:, j].astype(np.float64), -s1) + np.ldexp(w[:, j + 1].astype(np.float64), -s2)
    sums = np.stack([dec(1, SURF_V1, SURF_V2), dec(3, SURF_V1, SURF_V2), dec(5, SURF_V1, SURF_V2), dec(7, SURF_E1, SURF_E2)], axis=1)
    return w[:, 0].view(np.uint64).astype(np.float64), sums


def wall_extents(cfg, kind):
    """Per case the extent of its contact surface along the binned coordinate: cylinders (radius, [(z_lo, z_hi), ...]),
    planes (z, r_lo, r_hi), from the z and radial conditions of the case masks (Pore:442-485, Temp:693-753).  The
    open-air side wall has no z condition; particles reach it in the two open-air regions only."""
    from .amc import KIND_PORE
    g = cfg.geom
    oa = [(0.0, g.oah), (g.z_cold, g.H)]
    if kind == KIND_PORE:
        return {0: ("side", g.R_oa_c, oa), 1: ("plane", 0.0, 0.0, g.R_oa_c), 2: ("plane", g.H, 0.0, g.R_oa_c),
                3: ("plane", g.z_cold, g.R_p, g.R_oa_c), 4: ("plane", g.oah, g.R_p, g.R_oa_c),
                5: ("side", g.R_g_c, [(g.z_gb, g.z_gt_pore)]), 6: ("plane", g.z_gb, g.R_p, g.R_g_c),
                7: ("plane", g.z_gt_pore, g.R_p, g.R_g_c), 8: ("side", g.R_p_c, [(g.oah, g.z_gb), (g.z_gt_pore, g.z_cold)])}
    return {0: ("side", g.R_oa_c, oa), 1: ("plane", 0.0, 0.0, g.R_oa_c), 2: ("plane", g.H, 0.0, g.R_oa_c),
            3: ("plane", g.zc3, g.R_p, g.R_oa_c), 4: ("plane", g.zh3, g.R_p, g.R_oa_c), 5: ("side", g.R_g_c, [(g.zgb_p, g.zgt_m)]),
            6: ("plane", g.zgb_p, g.R_p_c, g.R_g_c), 7: ("plane", g.zgt_m, g.R_p_c, g.R_g_c),
            8: ("side", g.R_p_c, [(g.zh3, g.zgb_p)]), 9: ("side", g.R_p_c, [(g.zgt_m, g.zc3)])}


def surface_geometry(cfg, layout):
    """Per element: case, coordinate ranges (lo1, hi1, lo2, hi2: z for cylinders, r for annuli, the two in-plane
    axes for cube faces; lo2 / hi2 NaN where there is one coordinate) and the area of the contact surface the element
    covers: radius Rc for cylinders, the shifted planes (zc3 etc.), each clipped to its wall's extent."""
    n = layout.n_elements
    case = np.zeros(n, dtype=np.int64)
    rng = np.full((n, 4), np.nan)
    area = np.zeros(n)
    ext = None if layout.kind == 0 else wall_extents(cfg, layout.kind)
    for c in range(len(layout.types)):
        a0, a1 = int(layout.offsets[c]), int(layout.offsets[c + 1])
        if a1 == a0:
            continue
        case[a0:a1] = c
        t = layout.types[c]
        if t == "face":
            _, b1, b2 = layout.face_axes(c)
            L = (cfg.cube_x, cfg.cube_y, cfg.cube_z)
            e1, e2 = layout.edges[b1], layout.edges[b2]
            w1 = _overlap(e1[:-1], e1[1:], 0.0, float(L[b1]))
            w2 = _overlap(e2[:-1], e2[1:], 0.0, float(L[b2]))
            rng[a0:a1] = np.stack([np.repeat(e1[:-1], len(w2)), np.repeat(e1[1:], len(w2)),
                                   np.tile(e2[:-1], len(w1)), np.tile(e2[1:], len(w1))], axis=1)
            area[a0:a1] = np.outer(w1, w2).ravel()
        elif t == "side":
            _, Rc, spans = ext[c]
            z = layout.zedge
            rng[a0:a1, 0], rng[a0:a1, 1] = z[:-1], z[1:]
            area[a0:a1] = 2.0 * np.pi * float(Rc) * sum(_overlap(z[:-1], z[1:], float(lo), float(hi)) for lo, hi in spans)
        else:
            _, _, rlo, rhi = ext[c]
            r = np.sqrt(layout.rsq)
            rng[a0:a1, 0], rng[a0:a1, 1] = r[:-1], r[1:]
            lo, hi = np.maximum(r[:-1], float(rlo)), np.minimum(r[1:], float(rhi))
            area[a0:a1] = np.where(hi > lo, np.pi * (hi * hi - lo * lo), 0.0)
    return case, rng, area


def surface_fields(raw, cfg, grid, kind):
    """Per wall element of raw = (acc, n_steps, outside) (Simulation.surface_raw) on `grid` for a handle of `kind`: the
    SURFACE_COLUMNS -- case, coordinate ranges and area (surface_geometry), hits, number flux hits / (A n_steps dt)
    (1 / (m^2 s)), pressure m sum(dv.n) / (A n_steps dt) and the shear components m sum(dv.t) / (A n_steps dt) (Pa),
    heat flux into the wall -sum(dE) / (A n_steps dt) (W / m^2).  Elements of zero area give NaN rates."""
    from .amc import surface_layout_of
    acc, n_steps, _ = raw
    layout = surface_layout_of(cfg, kind, grid)
    case, rng, area = surface_geometry(cfg, layout)
    hits, sums = decode_surface_sums(acc)
    m = float(cfg.argon_mass)
    with np.errstate(invalid="ignore", divide="ignore"):
        denom = np.where(area > 0, area, np.nan) * (float(n_steps) * float(cfg.dt))
        return {"element": np.arange(layout.n_elements), "case": case, "lo1": rng[:, 0], "hi1": rng[:, 1], "lo2": rng[:, 2],
                "hi2": rng[:, 3], "area": area, "hits": acc[:, 0].astype(np.uint64), "number_flux": hits / denom,
                "pressure": m * sums[:, 0] / denom, "shear_1": m * sums[:, 1] / denom, "shear_2": m * sums[:, 2] / denom,
                "heat_flux": -sums[:, 3] / denom, "n_steps": int(n_steps)}


def write_surface_csv(path, fields):
    """surface.csv: one row per wall element, the SURFACE_COLUMNS (lengths in m, areas in m^2, number flux in
    1 / (m^2 s), pressure and shear in Pa, heat flux into the wall in W / m^2), floats with 17 significant digits."""
    ints = ("element", "case", "hits")
    with open(path, "w") as f:
        f.write(",".join(SURFACE_COLUMNS) + "\n")
        for k in range(len(fields["element"])):
            f.write(",".join(str(int(fields[c][k])) if c in ints else "%.17g" % float(fields[c][k]) for c in SURFACE_COLUMNS) + "\n")


# ---------------------------------------------------------------- plane fluxes (amc_flux_*)
FLUX_COLUMNS = ("plane", "z", "area", "up", "down", "up_rate", "down_rate", "particle_flux", "mass_flux", "p_xz", "p_yz",
                "p_zz", "energy_flux")


def decode_flux_sums(acc):
    """acc [planes][10] uint64 (Simulation.flux_raw) -> (up [planes], down [planes], sums [planes, 4]: sum s*vx, s*vy,
    s*vz in m/s and sum s*v^2 in m^2/s^2) as float64, each sum high * 2^-S1 + low * 2^-S2 of its signed limbs
    (include/amc.h)."""
    from .amc import FLUX_Q1, FLUX_Q2, FLUX_V1, FLUX_V2, FLUX_WORDS
    w = np.ascontiguousarray(acc, dtype=np.uint64).reshape(-1, FLUX_WORDS).view(np.int64)
    dec = lambda j, s1, s2: np.ldexp(w[:, j].astype(np.float64), -s1) + np.ldexp(w[:, j + 1].astype(np.float64), -s2)
    sums = np.stack([dec(2, FLUX_V1, FLUX_V2), dec(4, FLUX_V1, FLUX_V2), dec(6, FLUX_V1, FLUX_V2), dec(8, FLUX_Q1, FLUX_Q2)], axis=1)
    u = w.view(np.uint64)
    return u[:, 0].astype(np.float64), u[:, 1].astype(np.float64), sums


def plane_areas(cfg, kind, z):
    """Cross-section pi R^2 of the pore at each plane z, R the wall radius of the section the plane lies in: R_oa in the
    open air, R_p in the coated sections, R_g in the gap (the z bounds of the wall masks: the gap ends at z_gt_pore in
    Pore, at z_gt in Temp); a plane on a section boundary takes the smaller radius, a plane outside [0, H] the open-air
    one.  Cube (kind 0): cube_x * cube_y."""
    from .amc import KIND_CUBE, KIND_PORE
    z = np.asarray(z, dtype=np.float64)
    if kind == KIND_CUBE:
        return np.full(z.shape, float(cfg.cube_x) * float(cfg.cube_y))
    g = cfg.geom
    z_top = g.z_gt_pore if kind == KIND_PORE else g.z_gt
    sections = ((0.0, g.oah, g.R_oa), (g.oah, g.z_gb, g.R_p), (g.z_gb, z_top, g.R_g), (z_top, g.z_cold, g.R_p),
                (g.z_cold, g.H, g.R_oa))
    r = np.full(z.shape, float(g.R_oa))
    inside = np.zeros(z.shape, dtype=bool)
    for lo, hi, R in sections:
        m = (z >= float(lo)) & (z <= float(hi))
        r = np.where(m, np.where(inside, np.minimum(r, float(R)), float(R)), r)
        inside |= m
    return np.pi * r * r


def flux_fields(raw, cfg, grid, kind):
    """Per plane of raw = (acc, n_steps) (Simulation.flux_raw) on the z edges of `grid` for a handle of `kind`: the
    FLUX_COLUMNS -- plane index, z, cross-section A (plane_areas), crossings up / down and their rates per second,
    the net particle flux (up - down) / (A n_steps dt) (1 / (m^2 s)) and mass flux m times it (kg / (m^2 s)), the
    momentum fluxes m sum(s v_a) / (A n_steps dt) for a = x, y, z (P_xz, P_yz, P_zz in Pa) and the energy flux
    m/2 sum(s v^2) / (A n_steps dt) (W / m^2), with the config's own argon_mass and dt.  No record point: NaN rates."""
    acc, n_steps = raw
    z = np.asarray(grid.edge[2], dtype=np.float64)
    area = plane_areas(cfg, kind, z)
    up, down, sums = decode_flux_sums(acc)
    m, t = float(cfg.argon_mass), float(n_steps) * float(cfg.dt)
    with np.errstate(invalid="ignore", divide="ignore"):
        tt = t if t > 0 else np.nan
        net = (up - down) / (area * tt)
        words = np.asarray(acc, dtype=np.uint64).reshape(len(z), -1)
        return {"plane": np.arange(len(z)), "z": z, "area": area, "up": words[:, 0], "down": words[:, 1],
                "up_rate": up / tt, "down_rate": down / tt, "particle_flux": net, "mass_flux": m * net,
                "p_xz": m * sums[:, 0] / (area * tt), "p_yz": m * sums[:, 1] / (area * tt), "p_zz": m * sums[:, 2] / (area * tt),
                "energy_flux": 0.5 * m * sums[:, 3] / (area * tt), "n_steps": int(n_steps)}


def write_flux_csv(path, fields):
    """flux_z.csv: one row per z plane, the FLUX_COLUMNS (z in m, area in m^2, rates in 1 / s, particle flux in
    1 / (m^2 s), mass flux in kg / (m^2 s), momentum fluxes in Pa, energy flux in W / m^2), floats with 17 significant
    digits."""
    ints = ("plane", "up", "down")
    with open(path, "w") as f:
        f.write(",".join(FLUX_COLUMNS) + "\n")
        for k in range(len(fields["plane"])):
            f.write(",".join(str(int(fields[c][k])) if c in ints else "%.17g" % float(fields[c][k]) for c in FLUX_COLUMNS) + "\n")
