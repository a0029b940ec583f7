"""Velocity distribution (amc_vdf_*), host side, no GPU needed: the constants and entry points of include/amc.h against
the Python mirror, the NumPy restatement's bin rule against np.histogram on values at and around every edge, the
under / over words and the per-layer totals against the field sample, additivity, the Maxwellian pdfs of
outputs.vdf_fields, the vdf_z.csv format and the drivers' --vdf-bins / --vdf-vmax flags."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_vdf_constants_and_entry_points_match_the_header(tmp_path):
    from argon_monte_carlo_b200 import amc
    src = tmp_path / "probe.c"
    src.write_text('#include <stdio.h>\n#include "amc.h"\n'
                   'int main(void){printf("%d %d\\n", AMC_VDF_HISTS, AMC_VDF_MAX_BINS); return 0;}\n'
                   'int (*e)(amc_handle *, int32_t, double) = amc_vdf_enable;\n'
                   'int (*d)(amc_handle *) = amc_vdf_disable;\n'
                   'int (*l)(amc_handle *, int32_t *, int32_t *, double *) = amc_vdf_layout;\n'
                   'int (*g)(amc_handle *, uint64_t *) = amc_vdf_get_raw;\n'
                   'int (*s)(amc_handle *, const uint64_t *) = amc_vdf_set_raw;\n')
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-Wl,--unresolved-symbols=ignore-all", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert got == [amc.VDF_HISTS, amc.VDF_MAX_BINS]
    for name in ("amc_vdf_enable", "amc_vdf_disable", "amc_vdf_layout", "amc_vdf_get_raw", "amc_vdf_set_raw"):
        assert name in amc.EXPORTS


def _one_layer_grid():
    from argon_monte_carlo_b200 import config
    return config.Grid(nc=(1, 1, 1), c0=(-1, -1, 0), d=(2.0, 2.0, 1.0), band=(0, 0, 0))


def _state_with_velocities(vx, vy, vz):
    n = len(vx)
    return dict(x=np.full(n, -1.0), y=np.full(n, -1.0), z=np.full(n, 0.5), vx=np.asarray(vx, float), vy=np.asarray(vy, float),
                vz=np.asarray(vz, float))


@pytest.mark.parametrize("n_bins,v_max", [(200, 1500.0), (7, 3.0), (1, 1.0), (4096, 0.1)])
def test_bin_rule_equals_np_histogram_on_edges(n_bins, v_max):
    from argon_monte_carlo_b200 import amc
    ec, es = amc.vdf_edges(n_bins, v_max)
    assert np.array_equal(ec, np.linspace(-v_max, v_max, n_bins + 1)) and np.array_equal(es, np.linspace(0, v_max, n_bins + 1))
    vals = np.concatenate([ec, np.nextafter(ec, -np.inf), np.nextafter(ec, np.inf), [-v_max, v_max, 0.0, -0.0],
                           [1e300, -1e300, 10 * v_max, -10 * v_max, np.inf, -np.inf]])
    words = amc.vdf_of_arrays(_state_with_velocities(vals, vals, vals), _one_layer_grid(), n_bins, v_max)
    assert words.shape == (1, amc.VDF_HISTS, n_bins + 2)
    ref, _ = np.histogram(vals, bins=n_bins, range=(-v_max, v_max))
    for j in range(3):
        assert np.array_equal(words[0, j, 1:-1], ref)
        assert int(words[0, j, 0]) == np.count_nonzero(vals < -v_max)
        assert int(words[0, j, -1]) == np.count_nonzero(vals > v_max)
    with np.errstate(over="ignore"):
        speed = np.sqrt((vals * vals + vals * vals) + vals * vals)
    ref_s, _ = np.histogram(speed, bins=n_bins, range=(0, v_max))
    assert np.array_equal(words[0, 3, 1:-1], ref_s)
    assert int(words[0, 3, 0]) == 0 and int(words[0, 3, -1]) == np.count_nonzero(speed > v_max)
    # the speeds on the speed edges themselves: vx = edge, vy = vz = 0
    z = np.zeros(len(es) * 3)
    sv = np.concatenate([es, np.nextafter(es, -np.inf), np.nextafter(es, np.inf)])
    w = amc.vdf_of_arrays(_state_with_velocities(sv, z, z), _one_layer_grid(), n_bins, v_max)
    ref_s, _ = np.histogram(np.abs(sv), bins=n_bins, range=(0, v_max))
    assert np.array_equal(w[0, 3, 1:-1], ref_s)


def test_nan_goes_to_over():
    from argon_monte_carlo_b200 import amc
    w = amc.vdf_of_arrays(_state_with_velocities([np.nan, 1.0], [0.0, 0.0], [0.0, 0.0]), _one_layer_grid(), 10, 5.0)
    assert w[0, 0, -1] == 1 and w[0, 3, -1] == 1 and w[0, 0].sum() == 2 and w[0, 1].sum() == 2


def _gas(n, seed, grid, T=298.0, m=6.63e-26, kb=1.38e-23, drift=(0.0, 0.0, 0.0)):
    rng = np.random.default_rng(seed)
    lo = [float(grid.edge[a][0]) for a in range(3)]
    hi = [float(grid.edge[a][-1]) for a in range(3)]
    span = [h - l for l, h in zip(lo, hi)]
    pos = [rng.uniform(lo[a] - 0.02 * span[a], hi[a] + 0.02 * span[a], n) for a in range(3)]   # some outside the grid
    sig = np.sqrt(kb * T / m)
    vel = [rng.normal(drift[a], sig, n) for a in range(3)]
    return dict(zip(("x", "y", "z", "vx", "vy", "vz"), pos + vel))


@pytest.fixture(scope="module")
def small_grid():
    from argon_monte_carlo_b200 import config
    return config.pore_config(False, scale=0.5).grid


def test_totals_equal_the_field_sample_count_and_parts_add_up(small_grid):
    from argon_monte_carlo_b200 import amc
    st = _gas(50000, 1, small_grid)
    n_bins, v_max = 50, 800.0                       # about 3 sigma: under and over are well populated
    acc = amc.vdf_of_arrays(st, small_grid, n_bins, v_max)
    sample, _, outside = amc.sample_moments_of_arrays(st, small_grid)
    nx, ny, nz = small_grid.nc
    per_layer = sample[:, 0].reshape(nx * ny, nz).sum(axis=0)
    assert outside > 0
    for j in range(amc.VDF_HISTS):
        assert np.array_equal(acc[:, j].sum(axis=1), per_layer)
    assert acc[:, :3, 0].sum() > 0 and acc[:, :, -1].sum() > 0
    perm = np.random.default_rng(2).permutation(50000)
    parts = [amc.vdf_of_arrays(st, small_grid, n_bins, v_max, ids=p) for p in np.array_split(perm, 3)]
    assert np.array_equal(parts[0] + parts[1] + parts[2], acc)


@pytest.mark.parametrize("drift", [(0.0, 0.0, 0.0), (30.0, -50.0, 200.0), (1e-9, 0.0, 0.0)])
def test_maxwellian_pdfs_integrate_to_one(drift):
    from argon_monte_carlo_b200 import outputs
    sigma = 250.0
    e = np.linspace(-6000, 6000, 4001)
    for a in range(3):
        assert abs(np.diff(outputs.maxwell_component_cdf(e, drift[a], sigma)).sum() - 1) < 1e-12
    u = float(np.sqrt(np.sum(np.square(drift))))
    c = np.linspace(0, 6000, 3001)
    cdf = outputs.maxwell_speed_cdf(c, u, sigma)
    assert abs(cdf[0]) < 1e-12 and abs(cdf[-1] - 1) < 1e-12 and np.all(np.diff(cdf) >= -1e-15)
    # the speed pdf agrees with a histogram of sampled speeds
    rng = np.random.default_rng(4)
    v = np.stack([rng.normal(d, sigma, 400000) for d in drift])
    h, edges = np.histogram(np.sqrt((v * v).sum(axis=0)), bins=60, range=(0, 1500), density=True)
    model = np.diff(outputs.maxwell_speed_cdf(edges, u, sigma)) / np.diff(edges)
    assert np.sum(np.abs(h - model) * np.diff(edges)) < 0.02


def test_vdf_fields_of_a_maxwellian():
    from argon_monte_carlo_b200 import amc, config, outputs
    cfg = config.pore_config(True)
    grid = config.Grid(nc=(2, 2, 3), c0=(-1, -1, 0), d=(cfg.dx * 7, cfg.dy * 7, cfg.dz * 37), band=(0, 0, 0))
    st = _gas(300000, 5, grid, T=298.0, m=cfg.argon_mass, kb=cfg.boltzman, drift=(0.0, 0.0, 60.0))
    n_bins, v_max = 80, 2000.0
    f = outputs.vdf_fields(amc.vdf_of_arrays(st, grid, n_bins, v_max), (3, n_bins, v_max),
                           amc.sample_moments_of_arrays(st, grid), cfg, grid)
    width = np.stack([np.diff(e) for e in f["edges"]])
    assert np.allclose((f["pdf"] * width).sum(axis=2), 1.0)
    assert np.allclose((f["maxwellian"] * width).sum(axis=2), 1.0, atol=1e-6)
    assert np.all(f["l1"] < 0.05) and np.all(f["under_fraction"] == 0) and np.all(f["over_fraction"] < 1e-4)
    assert np.allclose(f["drift"][:, 2], 60.0, atol=5.0) and np.all(np.abs(f["temperature"] / 298.0 - 1) < 0.02)


def test_vdf_csv_format(tmp_path):
    from argon_monte_carlo_b200 import amc, config, outputs
    cfg = config.pore_config(False, scale=0.5)
    st = _gas(20000, 7, cfg.grid)
    nz, n_bins, v_max = cfg.grid.nc[2], 5, 1500.0
    f = outputs.vdf_fields(amc.vdf_of_arrays(st, cfg.grid, n_bins, v_max), (nz, n_bins, v_max),
                           amc.sample_moments_of_arrays(st, cfg.grid), cfg)
    path = tmp_path / "vdf_z.csv"
    outputs.write_vdf_csv(str(path), f)
    lines = path.read_text().splitlines()
    assert lines[0] == "z_lo,z_hi,histogram,bin,v_lo,v_hi,count,pdf,maxwellian,under_fraction,over_fraction,l1"
    assert len(lines) == 1 + nz * 4 * n_bins
    rows = [r.split(",") for r in lines[1:]]
    assert all(len(r) == 12 for r in rows)
    assert [r[2] for r in rows[:4 * n_bins:n_bins]] == ["vx", "vy", "vz", "speed"]
    assert [int(r[3]) for r in rows[:n_bins]] == list(range(n_bins))
    assert float(rows[0][4]) == -v_max and float(rows[n_bins - 1][5]) == v_max and float(rows[3 * n_bins][4]) == 0.0
    assert float(rows[0][0]) == cfg.grid.edge[2][0] and float(rows[-1][1]) == cfg.grid.edge[2][-1]
    total = sum(int(r[6]) for r in rows if r[2] == "vx")
    assert total <= 20000 and total > 0


def test_driver_flags():
    from argon_monte_carlo_b200 import config, driver_common
    a = driver_common.parse_args(10, "x", argv=[])
    assert a.vdf_bins == 0 and a.vdf_vmax is None
    a = driver_common.parse_args(10, "x", argv=["--sample-every", "5", "--vdf-bins", "100", "--vdf-vmax", "1200"])
    assert (a.vdf_bins, a.vdf_vmax) == (100, 1200.0)
    for bad in (["--vdf-bins", "100"], ["--sample-every", "5", "--vdf-bins", "0", "--vdf-vmax", "3"],
                ["--sample-every", "5", "--vdf-bins", "4097"], ["--sample-every", "5", "--vdf-bins", "-1"],
                ["--sample-every", "5", "--vdf-bins", "10", "--vdf-vmax", "0"],
                ["--sample-every", "5", "--vdf-bins", "10", "--vdf-vmax", "nan"]):
        with pytest.raises(SystemExit):
            driver_common.parse_args(10, "x", argv=bad)
    temp, pore = config.pore_config(True), config.pore_config(False)
    sig = lambda t, c: np.sqrt(c.boltzman * t / c.argon_mass)
    assert driver_common.vdf_default_vmax(temp) == pytest.approx(driver_common.VDF_VMAX_SIGMAS * sig(353.0, temp))
    assert driver_common.vdf_default_vmax(pore) == pytest.approx(driver_common.VDF_VMAX_SIGMAS * sig(298.0, pore))
