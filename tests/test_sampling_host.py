"""Field sampling, host side, no GPU needed: the constants of include/amc.h against the Python mirror (gcc probe), the
NumPy restatement of the sampling kernel (binning, fixed-point limbs, order independence, additivity), the layer
volumes and fields of outputs.py, the profile_z.csv format and the drivers' command-line flags."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sample_constants_match_the_header(tmp_path):
    from argon_monte_carlo_b200 import amc
    src = tmp_path / "probe.c"
    src.write_text('#include <stdio.h>\n#include "amc.h"\nint main(void){printf("%d %d %d %d %d %d\\n", AMC_SAMPLE_WORDS,'
                   ' AMC_SAMPLE_V1, AMC_SAMPLE_V2, AMC_SAMPLE_Q1, AMC_SAMPLE_Q2, AMC_ABI_VERSION); return 0;}\n')
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert got == [amc.SAMPLE_WORDS, amc.SAMPLE_V1, amc.SAMPLE_V2, amc.SAMPLE_Q1, amc.SAMPLE_Q2, 1]
    assert amc.ABI_VERSION == 1


def test_new_entry_points_are_exported_names():
    from argon_monte_carlo_b200 import amc
    for name in ("amc_sample_enable", "amc_sample_disable", "amc_sample_now", "amc_sample_get_raw", "amc_sample_set_raw",
                 "amc_last_sample_ms"):
        assert name in amc.EXPORTS


def _gas(n, seed, grid, T=298.0, m=6.63e-26, kb=1.38e-23, drift=(0.0, 0.0, 0.0)):
    rng = np.random.default_rng(seed)
    lo = [float(grid.edge[a][0]) for a in range(3)]
    hi = [float(grid.edge[a][-1]) for a in range(3)]
    pos = [rng.uniform(lo[a], hi[a], n) for a in range(3)]
    sig = np.sqrt(kb * T / m)
    vel = [rng.normal(drift[a], sig, n) for a in range(3)]
    return dict(zip(("x", "y", "z", "vx", "vy", "vz"), pos + vel))


@pytest.fixture(scope="module")
def small_grid():
    from argon_monte_carlo_b200 import config
    return config.pore_config(False, scale=0.5).grid


def test_restatement_is_order_independent_and_additive(small_grid):
    from argon_monte_carlo_b200 import amc
    st = _gas(40000, 1, small_grid)
    acc, ns, no = amc.sample_moments_of_arrays(st, small_grid)
    assert ns == 1 and acc.shape == (int(np.prod(small_grid.nc)), amc.SAMPLE_WORDS) and acc.dtype == np.uint64
    perm = np.random.default_rng(2).permutation(40000)
    acc_p, _, no_p = amc.sample_moments_of_arrays({k: v[perm] for k, v in st.items()}, small_grid)
    assert np.array_equal(acc, acc_p) and no == no_p
    parts = np.array_split(perm, 3)
    raws = [amc.sample_moments_of_arrays(st, small_grid, ids=p) for p in parts]
    merged = amc.merge_sample_ranks(raws)
    assert np.array_equal(merged[0], acc) and merged[1] == 1 and merged[2] == no
    assert int(acc[:, 0].sum()) + no == 40000


def test_limbs_decode_to_the_float_sums():
    from argon_monte_carlo_b200 import amc, config, outputs
    cfg = config.pore_config(False)
    grid = config.Grid(nc=(2, 2, 6), c0=(-1, -1, 0), d=(cfg.dx * 7, cfg.dy * 7, cfg.dz * 25), band=(0, 0, 0))
    st = _gas(60000, 3, grid, drift=(50.0, -20.0, 300.0))
    acc, _, _ = amc.sample_moments_of_arrays(st, grid)
    count, sv, sq = outputs.decode_sample_sums(acc)
    cell, inside = amc.sample_cells_of(st["x"], st["y"], st["z"], grid)
    ncell = int(np.prod(grid.nc))
    for a, k in enumerate(("vx", "vy", "vz")):
        v = st[k][inside]
        ref = np.zeros(ncell)
        np.add.at(ref, cell[inside], v)
        ref_sq = np.zeros(ncell)
        np.add.at(ref_sq, cell[inside], v * v)
        scale = np.abs(np.zeros(ncell))
        np.add.at(scale, cell[inside], np.abs(v))
        m = count > 0
        assert np.all(np.abs(sv[m, a] - ref[m]) <= 1e-12 * scale[m])
        assert np.all(np.abs(sq[m, a] - ref_sq[m]) <= 1e-12 * ref_sq[m])
    # limbs of one value are exact: high * 2^-S1 + low * 2^-S2 reproduces v to the low limb's resolution
    v = np.array([0.0, 1.0, -1.0, 399.123456789, -1234.5e-3, 9999.999999, 1e-9])
    i1, i2 = amc.sample_limbs(v, amc.SAMPLE_V1, amc.SAMPLE_V2)
    assert np.all(np.abs(np.ldexp(i1.astype(float), -amc.SAMPLE_V1) + np.ldexp(i2.astype(float), -amc.SAMPLE_V2) - v)
                  <= 2.0 ** -amc.SAMPLE_V2)


def test_binning_matches_searchsorted_on_edges_nan_and_outside(small_grid):
    from argon_monte_carlo_b200 import amc
    g = small_grid
    ex, ey, ez = (np.asarray(g.edge[a]) for a in range(3))
    x = np.array([ex[0], ex[1], ex[-1], np.nextafter(ex[-1], -np.inf), np.nextafter(ex[0], -np.inf), np.nan, 0.0, ex[3], 0.0])
    y = np.array([ey[0], ey[2], 0.0, ey[1], 0.0, 0.0, np.nan, ey[-2], 0.0])
    z = np.array([ez[0], ez[5], ez[1], np.nextafter(ez[-1], -np.inf), ez[2], ez[3], ez[4], ez[7], ez[-1]])
    cell, inside = amc.sample_cells_of(x, y, z, g)
    nx, ny, nz = g.nc
    for i in range(len(x)):
        k = [np.searchsorted(e, v, side="right") - 1 for e, v in ((ex, x[i]), (ey, y[i]), (ez, z[i]))]
        ok = all(0 <= kk < n for kk, n in zip(k, (nx, ny, nz)))
        assert inside[i] == ok, i
        if ok:
            assert cell[i] == (k[0] * ny + k[1]) * nz + k[2]
    assert inside.tolist() == [True, True, False, True, False, False, False, True, False]
    st = dict(x=x, y=y, z=z, vx=np.ones(len(x)), vy=np.zeros(len(x)), vz=np.zeros(len(x)))
    acc, _, no = amc.sample_moments_of_arrays(st, g)
    assert no == 5 and int(acc[:, 0].sum()) == 4


@pytest.mark.parametrize("temperature", [False, True])
def test_layer_volumes_sum_to_the_centre_accessible_volume(temperature):
    from argon_monte_carlo_b200 import config, outputs
    for scale in (1.0, 0.5):
        cfg = config.pore_config(temperature, scale=scale)
        g = cfg.geom
        vol = outputs.layer_volumes(cfg, cfg.grid.edge[2])
        total = (config.cylinder_volume(g.R_oa_c, g.oah) + config.cylinder_volume(g.R_p_c, g.z_gb - g.oah)
                 + config.cylinder_volume(g.R_g_c, g.z_gt - g.z_gb) + config.cylinder_volume(g.R_p_c, g.z_cold - g.z_gt)
                 + config.cylinder_volume(g.R_oa_c, g.H - g.z_cold))
        assert abs(vol.sum() - total) <= 1e-12 * total
        assert np.all(vol > 0)
    cube = config.cube_config()
    v = outputs.layer_volumes(cube, cube.grid.edge[2])
    assert abs(v.sum() - cube.cube_x * cube.cube_y * cube.cube_z) <= 1e-12 * cube.cube_volume


def test_fields_of_a_maxwellian_give_its_temperature():
    from argon_monte_carlo_b200 import amc, config, outputs
    cfg = config.pore_config(True)
    grid = config.Grid(nc=(2, 2, 4), c0=(-1, -1, 0), d=(cfg.dx * 7, cfg.dy * 7, cfg.dz * 37), band=(0, 0, 0))
    n = 400000
    st = _gas(n, 5, grid, T=298.0, m=cfg.argon_mass, kb=cfg.boltzman, drift=(0.0, 0.0, 40.0))
    raw = amc.sample_moments_of_arrays(st, grid)
    f = outputs.sample_fields(raw, cfg)
    # the whole gas within 0.5 %; every cell (25,000 particles: 0.5 % standard deviation) within 2.5 %
    assert abs(np.sum(f["temperature"] * f["count"]) / f["count"].sum() / 298.0 - 1) < 0.005
    assert np.all(np.abs(f["temperature"] / 298.0 - 1) < 0.025)
    assert np.all(np.abs(f["temperature_axes"] / 298.0 - 1) < 0.04)
    assert np.allclose(f["v_mean"][:, 2], 40.0, atol=3.0)
    assert abs(f["particles_per_sample"].sum() - n) < 1e-6
    # two samples of the same state: particles per sample unchanged, the same temperature
    acc2 = raw[0] + raw[0]
    f2 = outputs.sample_fields((acc2, 2, 0), cfg)
    assert np.allclose(f2["particles_per_sample"], f["particles_per_sample"])
    assert np.allclose(f2["temperature"], f["temperature"], rtol=1e-12)
    prof = outputs.axial_profile(raw, cfg, grid)
    assert np.all(np.abs(prof["temperature"] / 298.0 - 1) < 0.01)


def test_profile_csv_format(tmp_path):
    from argon_monte_carlo_b200 import amc, config, outputs
    cfg = config.pore_config(False, scale=0.5)
    st = _gas(20000, 7, cfg.grid)
    prof = outputs.axial_profile(amc.sample_moments_of_arrays(st, cfg.grid), cfg)
    path = tmp_path / "profile_z.csv"
    outputs.write_axial_profile(str(path), prof)
    lines = path.read_text().splitlines()
    assert lines[0] == ("z_lo,z_hi,samples,particles_per_sample,number_density,vz_mean,temperature,temperature_x,"
                        "temperature_y,temperature_z")
    assert len(lines) == 1 + cfg.grid.nc[2]
    for k, row in enumerate(lines[1:]):
        vals = row.split(",")
        assert len(vals) == 10 and vals[2] == "1"
        assert float(vals[0]) == cfg.grid.edge[2][k] and float(vals[1]) == cfg.grid.edge[2][k + 1]


def test_driver_flags_parse():
    from argon_monte_carlo_b200 import driver_common
    a = driver_common.parse_args(10, "x", argv=[])
    assert a.sample_every == 0 and a.sample_start == 0
    a = driver_common.parse_args(10, "x", temp=True, argv=["--sample-every", "5", "--sample-start", "100", "--steps", "7"])
    assert (a.sample_every, a.sample_start, a.steps) == (5, 100, 7)
    with pytest.raises(SystemExit):
        driver_common.parse_args(10, "x", argv=["--sample-every", "-1"])


def test_transport_sums_sample_arrays():
    from argon_monte_carlo_b200 import slab
    a = np.array([[1, 2], [3, 2 ** 64 - 1]], dtype=np.uint64)
    out = slab.LocalTransport().allreduce_u64(a)
    assert isinstance(out, np.ndarray) and np.array_equal(out, a)
    assert slab.LocalTransport().allreduce_u64((1, 2)) == (1, 2)
