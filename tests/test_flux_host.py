"""Plane flux recording (amc_flux_*), host side, no GPU needed: the constants and entry points of include/amc.h against
the Python mirror, the NumPy restatement against a brute-force loop over planes (positions on the planes, one ulp
either side, NaN, infinities and jumps over several planes), the decoded limbs against the float sums, the worst-case
headroom of the limbs, the cross-sections and columns of outputs.flux_fields / flux_z.csv and the drivers'
--flux-start flag and batching."""
import os
import subprocess
from types import SimpleNamespace

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_flux_constants_and_entry_points_match_the_header(tmp_path):
    from argon_monte_carlo_b200 import amc
    src = tmp_path / "probe.c"
    src.write_text('#include <stdio.h>\n#include "amc.h"\n'
                   'int main(void){printf("%d %d %d %d %d\\n", AMC_FLUX_WORDS, AMC_FLUX_V1, AMC_FLUX_V2, AMC_FLUX_Q1, '
                   'AMC_FLUX_Q2); return 0;}\n'
                   'int (*e)(amc_handle *) = amc_flux_enable;\n'
                   'int (*d)(amc_handle *) = amc_flux_disable;\n'
                   'int (*w)(amc_handle *) = amc_flux_now;\n'
                   'int (*l)(amc_handle *, int32_t *) = amc_flux_layout;\n'
                   'int (*g)(amc_handle *, uint64_t *, uint64_t *) = amc_flux_get_raw;\n'
                   'int (*s)(amc_handle *, const uint64_t *, uint64_t) = amc_flux_set_raw;\n')
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-Wl,--unresolved-symbols=ignore-all", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert got == [amc.FLUX_WORDS, amc.FLUX_V1, amc.FLUX_V2, amc.FLUX_Q1, amc.FLUX_Q2]
    for name in ("amc_flux_enable", "amc_flux_disable", "amc_flux_now", "amc_flux_layout", "amc_flux_get_raw", "amc_flux_set_raw"):
        assert name in amc.EXPORTS


def brute_force(z0, z1, v, edges):
    """Per plane k and particle: crossed upward if z0 < e_k <= z1 in the cnt sense, i.e. cnt(z0) <= k < cnt(z1)."""
    from argon_monte_carlo_b200 import amc

    def cnt(z):
        if z != z:
            return len(edges)
        return sum(1 for e in edges if e <= z)
    acc = np.zeros((len(edges), amc.FLUX_WORDS), dtype=np.uint64)
    for i in range(len(z0)):
        c0, c1 = cnt(z0[i]), cnt(z1[i])
        s = 1.0 if c1 > c0 else -1.0
        with np.errstate(over="ignore", invalid="ignore"):
            q = (v[0][i] * v[0][i] + v[1][i] * v[1][i]) + v[2][i] * v[2][i]
        limbs = []
        for val, s1, s2 in ((v[0][i], amc.FLUX_V1, amc.FLUX_V2), (v[1][i], amc.FLUX_V1, amc.FLUX_V2),
                            (v[2][i], amc.FLUX_V1, amc.FLUX_V2), (q, amc.FLUX_Q1, amc.FLUX_Q2)):
            i1, i2 = amc.sample_limbs(np.array([s * val]), s1, s2)
            limbs += [int(i1[0]), int(i2[0])]
        for k in range(min(c0, c1), max(c0, c1)):
            acc[k, 0 if c1 > c0 else 1] += np.uint64(1)
            for j, w in enumerate(limbs):
                acc[k, 2 + j] = np.uint64((int(acc[k, 2 + j]) + w) & ((1 << 64) - 1))
    return acc


def _edges():
    from argon_monte_carlo_b200 import config
    return np.asarray(config.pore_config(False, scale=0.5).grid.edge[2], dtype=np.float64)


def test_plane_count_is_searchsorted_right_on_every_edge():
    from argon_monte_carlo_b200 import amc
    e = _edges()
    z = np.concatenate([e, np.nextafter(e, -np.inf), np.nextafter(e, np.inf), [np.nan, np.inf, -np.inf, -0.0, 0.0, -1.0, 1.0]])
    c = amc.flux_counts_of(z, e)
    for zz, cc in zip(z, c):
        assert cc == (len(e) if zz != zz else sum(1 for x in e if x <= zz)), zz


def test_restatement_equals_brute_force():
    from argon_monte_carlo_b200 import amc
    e = _edges()
    rng = np.random.default_rng(5)
    n = 3000
    pool = np.concatenate([e, np.nextafter(e, -np.inf), np.nextafter(e, np.inf), [np.nan, np.inf, -np.inf, -1e-6, 1e-3]])
    z0 = rng.choice(pool, n)
    z1 = np.where(rng.random(n) < 0.5, z0, rng.choice(pool, n))            # half stay, the rest jump anywhere
    z1[:50] = z0[:50] + rng.normal(0, 3 * (e[1] - e[0]), 50)                # short moves over a few planes
    v = [rng.normal(0, 300, n) for _ in range(3)]
    v[0][7] = 2e4
    v[2][9] = -1e4
    st0, st1 = dict(z=z0), dict(z=z1, vx=v[0], vy=v[1], vz=v[2])
    acc = amc.flux_of_states(st0, st1, e)
    assert acc.shape == (len(e), amc.FLUX_WORDS)
    assert np.array_equal(acc, brute_force(z0, z1, v, e))
    assert acc[:, 0].sum() > 0 and acc[:, 1].sum() > 0
    assert int(acc[:, 0].astype(np.int64).max()) > 0
    # the way back cancels: every count word swaps up and down, every sum word changes sign
    back = amc.flux_of_states(dict(z=z1), dict(z=z0, vx=v[0], vy=v[1], vz=v[2]), e)
    assert np.array_equal(back[:, 0], acc[:, 1]) and np.array_equal(back[:, 1], acc[:, 0])
    with np.errstate(over="ignore"):
        assert not (back[:, 2:] + acc[:, 2:]).any()


def test_conservation_over_a_sequence_of_states():
    """up - down of a plane summed over the record points = particles at or above it at the end minus at the start."""
    from argon_monte_carlo_b200 import amc
    e = _edges()
    rng = np.random.default_rng(8)
    n = 20000
    z = rng.uniform(e[0] - 1e-8, e[-1] + 1e-8, n)
    start = z.copy()
    total = np.zeros((len(e), amc.FLUX_WORDS), dtype=np.uint64)
    for _ in range(5):
        znew = z + rng.normal(0, 2 * (e[1] - e[0]), n)
        with np.errstate(over="ignore"):
            total += amc.flux_of_states(dict(z=z), dict(z=znew, vx=np.ones(n), vy=np.ones(n), vz=np.ones(n)), e)
        z = znew
    net = total[:, 0].astype(np.int64) - total[:, 1].astype(np.int64)
    above = lambda zz: np.array([np.count_nonzero(zz >= x) for x in e])
    assert np.array_equal(net, above(z) - above(start))


def test_decoded_limbs_equal_the_float_sums():
    from argon_monte_carlo_b200 import amc, outputs
    e = np.array([0.0, 1.0, 2.0])
    rng = np.random.default_rng(3)
    n = 100000
    z0, z1 = rng.uniform(-0.5, 2.5, n), rng.uniform(-0.5, 2.5, n)
    v = [rng.normal(0, 400, n) for _ in range(3)]
    acc = amc.flux_of_states(dict(z=z0), dict(z=z1, vx=v[0], vy=v[1], vz=v[2]), e)
    up, down, sums = outputs.decode_flux_sums(acc)
    c0, c1 = np.searchsorted(e, z0, "right"), np.searchsorted(e, z1, "right")
    q = (v[0] * v[0] + v[1] * v[1]) + v[2] * v[2]
    for k in range(len(e)):
        upk, dnk = (c0 <= k) & (k < c1), (c1 <= k) & (k < c0)
        assert up[k] == np.count_nonzero(upk) and down[k] == np.count_nonzero(dnk)
        s = upk.astype(float) - dnk.astype(float)
        for j, val in enumerate((v[0], v[1], v[2], q)):
            ref = float(np.sum(s * val))
            scale = float(np.sum(np.abs(s * val)))
            assert abs(sums[k, j] - ref) <= 1e-12 * scale + 1e-9, (k, j, sums[k, j], ref)


def test_worst_case_headroom():
    """10^10 crossings per plane at speeds <= 10^4 m/s stay inside the signed 64-bit limbs (include/amc.h)."""
    from argon_monte_carlo_b200 import amc
    n, vmax = 1e10, 1e4
    v_hi = n * vmax * 2.0 ** amc.FLUX_V1
    q_hi = n * vmax * vmax * 2.0 ** amc.FLUX_Q1
    lo = n * max(2.0 ** (amc.FLUX_V2 - amc.FLUX_V1 - 1), 2.0 ** (amc.FLUX_Q2 - amc.FLUX_Q1 - 1))
    assert (round(v_hi / 1e18, 1), round(q_hi / 1e18, 1), round(lo / 1e18, 1)) == (6.6, 4.0, 5.4)
    assert max(v_hi, q_hi, lo) < 2.0 ** 63
    # one crossing at the extremes: the limbs a particle adds are what the bound assumes
    i1, i2 = amc.sample_limbs(np.array([vmax, -vmax, vmax * (1 - 2 ** -40)]), amc.FLUX_V1, amc.FLUX_V2)
    assert np.all(np.abs(i1) <= vmax * 2.0 ** amc.FLUX_V1) and np.all(np.abs(i2) <= 2.0 ** (amc.FLUX_V2 - amc.FLUX_V1 - 1))
    i1, i2 = amc.sample_limbs(np.array([vmax * vmax, vmax * vmax * (1 - 2 ** -40)]), amc.FLUX_Q1, amc.FLUX_Q2)
    assert np.all(np.abs(i1) <= vmax * vmax * 2.0 ** amc.FLUX_Q1) and np.all(np.abs(i2) <= 2.0 ** (amc.FLUX_Q2 - amc.FLUX_Q1 - 1))


def test_plane_areas_follow_the_sections():
    from argon_monte_carlo_b200 import amc, config, outputs
    for kind, temp in ((amc.KIND_PORE, False), (amc.KIND_TEMP, True)):
        cfg = config.pore_config(temp)
        g = cfg.geom
        z_top = g.z_gt_pore if kind == amc.KIND_PORE else g.z_gt
        z = np.array([0.0, 0.5 * g.oah, g.oah, 0.5 * (g.oah + g.z_gb), g.z_gb, 0.5 * (g.z_gb + z_top), z_top,
                      0.5 * (z_top + g.z_cold), g.z_cold, g.H, -1e-9, 2 * g.H])
        lo = lambda a, b: min(float(a), float(b))       # a plane on a section boundary: the smaller radius
        R = np.array([g.R_oa, g.R_oa, lo(g.R_oa, g.R_p), g.R_p, lo(g.R_p, g.R_g), g.R_g, lo(g.R_g, g.R_p), g.R_p,
                      lo(g.R_p, g.R_oa), g.R_oa, g.R_oa, g.R_oa])
        assert np.array_equal(outputs.plane_areas(cfg, kind, z), np.pi * R * R)
    cube = config.cube_config()
    assert np.all(outputs.plane_areas(cube, amc.KIND_CUBE, cube.grid.edge[2]) == cube.cube_x * cube.cube_y)


def test_flux_fields_and_csv_format(tmp_path):
    from argon_monte_carlo_b200 import amc, config, outputs
    cfg = config.pore_config(True, scale=0.5)
    e = np.asarray(cfg.grid.edge[2], dtype=np.float64)
    rng = np.random.default_rng(1)
    n = 50000
    z0 = rng.uniform(e[0], e[-1], n)
    z1 = z0 + rng.normal(0, e[1] - e[0], n)
    v = [rng.normal(0, 300, n) for _ in range(2)] + [np.full(n, 150.0)]
    acc = amc.flux_of_states(dict(z=z0), dict(z=z1, vx=v[0], vy=v[1], vz=v[2]), e)
    n_steps = 4
    f = outputs.flux_fields((acc, n_steps), cfg, cfg.grid, amc.KIND_TEMP)
    t = n_steps * cfg.dt
    up, down, sums = outputs.decode_flux_sums(acc)
    area = outputs.plane_areas(cfg, amc.KIND_TEMP, e)
    m = cfg.argon_mass
    assert np.array_equal(f["up"], acc[:, 0]) and np.array_equal(f["down"], acc[:, 1])
    assert np.allclose(f["up_rate"], up / t) and np.allclose(f["down_rate"], down / t)
    assert np.allclose(f["particle_flux"], (up - down) / (area * t)) and np.allclose(f["mass_flux"], m * (up - down) / (area * t))
    assert np.allclose(f["p_zz"], m * sums[:, 2] / (area * t)) and np.allclose(f["energy_flux"], 0.5 * m * sums[:, 3] / (area * t))
    path = tmp_path / "flux_z.csv"
    outputs.write_flux_csv(str(path), f)
    lines = path.read_text().splitlines()
    assert lines[0] == "plane,z,area,up,down,up_rate,down_rate,particle_flux,mass_flux,p_xz,p_yz,p_zz,energy_flux"
    assert len(lines) == 1 + len(e)
    rows = [r.split(",") for r in lines[1:]]
    assert all(len(r) == 13 for r in rows)
    assert [int(r[0]) for r in rows] == list(range(len(e)))
    assert [float(r[1]) for r in rows] == list(e)
    assert [int(r[3]) for r in rows] == [int(x) for x in acc[:, 0]]
    assert float(rows[5][11]) == pytest.approx(f["p_zz"][5], rel=1e-15)
    empty = outputs.flux_fields((np.zeros_like(acc), 0), cfg, cfg.grid, amc.KIND_TEMP)
    assert np.all(np.isnan(empty["up_rate"])) and np.all(empty["up"] == 0)


def test_driver_flag_and_batches():
    from argon_monte_carlo_b200 import driver_common
    assert driver_common.parse_args(10, "x", argv=[]).flux_start is None
    assert driver_common.parse_args(10, "x", argv=["--flux-start", "5"]).flux_start == 5
    assert driver_common.parse_args(10, "x", argv=["--flux-start", "0"]).flux_start == 0
    with pytest.raises(SystemExit):
        driver_common.parse_args(10, "x", argv=["--flux-start", "-1"])

    class FakeSim:
        flux_on = False

        def flux_enable(self):
            self.flux_on = True
    sim = FakeSim()
    args = SimpleNamespace(flux_start=150)
    assert driver_common.flux_chunk(sim, args, 0, 100) == 100 and not sim.flux_on
    assert driver_common.flux_chunk(sim, args, 100, 100) == 50 and not sim.flux_on     # stops at S
    assert driver_common.flux_chunk(sim, args, 150, 100) == 100 and sim.flux_on        # records from S on
    sim = FakeSim()
    assert driver_common.flux_chunk(sim, SimpleNamespace(flux_start=None), 0, 7) == 7 and not sim.flux_on
    # together with --surface-start: a batch straddles neither
    both = SimpleNamespace(flux_start=30, surface_start=70)
    sim = FakeSim()
    sim.surface_on = False
    sim.surface_enable = lambda: setattr(sim, "surface_on", True)
    done, batches = 0, []
    while done < 100:
        c = driver_common.flux_chunk(sim, both, done, driver_common.surface_chunk(sim, both, done, min(25, 100 - done)))
        batches.append((done, c, sim.flux_on, sim.surface_on))
        done += c
    assert batches == [(0, 25, False, False), (25, 5, False, False), (30, 25, True, False), (55, 15, True, False),
                       (70, 25, True, True), (95, 5, True, True)]
