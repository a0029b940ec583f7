"""Surface recording, host side: header constants and exports, the layout restatement, element areas, the fixed-point
limbs, the NumPy restatement of the accumulators on oracle hit lists, the CSV format and the driver flag."""
import os
import re

import numpy as np
import pytest

from argon_monte_carlo_b200 import amc, config, driver_common, outputs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header():
    return open(os.path.join(ROOT, "include", "amc.h")).read()


def test_header_constants_and_exports():
    h = header()
    for name, v in (("AMC_SURF_WORDS", amc.SURF_WORDS), ("AMC_SURF_V1", amc.SURF_V1), ("AMC_SURF_V2", amc.SURF_V2),
                    ("AMC_SURF_E1", amc.SURF_E1), ("AMC_SURF_E2", amc.SURF_E2)):
        assert int(re.search(r"#define %s (\d+)" % name, h).group(1)) == v
    assert "#define AMC_ABI_VERSION 1" in h
    for name in ("amc_surface_enable", "amc_surface_disable", "amc_surface_layout", "amc_surface_get_raw", "amc_surface_set_raw"):
        assert name in amc.EXPORTS and re.search(r"int %s\(" % name, h)
    # headroom stated in amc.h: 10^9 hits at |dv| <= 2*10^4 m/s and |dE| <= 3.4e-18 J stay inside int64
    assert 1e9 * 2e4 * 2.0 ** amc.SURF_V1 < 2.0 ** 63 and 1e9 * 3.4e-18 * 2.0 ** amc.SURF_E1 < 2.0 ** 63
    assert 1e9 * 2.0 ** (amc.SURF_V2 - amc.SURF_V1 - 1) < 2.0 ** 63 and 1e9 * 2.0 ** (amc.SURF_E2 - amc.SURF_E1 - 1) < 2.0 ** 63


@pytest.mark.parametrize("which", ["pore", "temp", "cube"])
def test_layout_restatement(which):
    cfg = {"pore": config.pore_config(False), "temp": config.pore_config(True), "cube": config.cube_config()}[which]
    kind = {"pore": amc.KIND_PORE, "temp": amc.KIND_TEMP, "cube": amc.KIND_CUBE}[which]
    L = amc.surface_layout_of(cfg, kind, cfg.grid)
    nx, ny, nz = (int(v) for v in cfg.grid.nc)
    n = np.diff(L.offsets)
    if kind == amc.KIND_CUBE:
        assert list(n) == [ny * nz, ny * nz, nx * nz, nx * nz, nx * ny, nx * ny, 0, 0, 0, 0]
        return
    e = np.asarray(cfg.grid.edge[0])
    dr = (e[-1] - e[0]) / nx
    nann = int(np.ceil(cfg.geom.R_oa / dr))
    assert L.nann == nann and L.rsq[0] == 0.0 and L.rsq[-1] >= cfg.geom.R_oa ** 2
    assert np.all(np.diff(L.rsq) > 0)
    sides = (0, 5, 8) if kind == amc.KIND_PORE else (0, 5, 8, 9)
    for c in range(amc.NUM_CASES):
        want = nz if c in sides else (0 if (kind == amc.KIND_PORE and c == 9) else nann)
        assert n[c] == want, c


@pytest.mark.parametrize("which", ["pore", "temp", "cube"])
def test_element_areas_sum_to_the_contact_surface(which):
    cfg = {"pore": config.pore_config(False), "temp": config.pore_config(True), "cube": config.cube_config()}[which]
    kind = {"pore": amc.KIND_PORE, "temp": amc.KIND_TEMP, "cube": amc.KIND_CUBE}[which]
    L = amc.surface_layout_of(cfg, kind, cfg.grid)
    case, _, area = outputs.surface_geometry(cfg, L)
    tot = np.bincount(case, weights=area, minlength=amc.NUM_CASES)
    if kind == amc.KIND_CUBE:
        a = (cfg.cube_x, cfg.cube_y, cfg.cube_z)
        want = [a[1] * a[2]] * 2 + [a[0] * a[2]] * 2 + [a[0] * a[1]] * 2 + [0] * 4
    else:
        want = []
        for c, e in sorted(outputs.wall_extents(cfg, kind).items()):
            if e[0] == "side":
                want.append(2 * np.pi * e[1] * sum(hi - lo for lo, hi in e[2]))
            else:
                want.append(np.pi * (e[3] ** 2 - e[2] ** 2))
        want += [0.0] * (amc.NUM_CASES - len(want))
    assert np.allclose(tot, want, rtol=1e-12, atol=0)


def test_limbs_and_additivity():
    rng = np.random.default_rng(3)
    v = rng.normal(0, 600, 1000)
    i1, i2 = amc.sample_limbs(v, amc.SURF_V1, amc.SURF_V2)
    dec = np.ldexp(i1.astype(np.float64), -amc.SURF_V1) + np.ldexp(i2.astype(np.float64), -amc.SURF_V2)
    assert np.all(np.abs(dec - v) <= 2.0 ** -(amc.SURF_V2 + 1))
    g = config.pore_config(False)
    L = amc.surface_layout_of(g, amc.KIND_PORE, g.grid)
    n = 500
    hits = {"case": rng.integers(0, 9, n), "col": np.stack([rng.uniform(-1.6e-7, 1.6e-7, n), rng.uniform(-1.6e-7, 1.6e-7, n),
                                                           rng.uniform(0, g.geom.H, n)], 1),
            "v_in": rng.normal(0, 300, (n, 3)), "v_out": rng.normal(0, 300, (n, 3)), "dE": rng.normal(0, 1e-21, n)}
    whole = amc.surface_moments_of_hits(hits, L, g.geom)
    a = amc.surface_moments_of_hits({k: v[:200] for k, v in hits.items()}, L, g.geom)
    b = amc.surface_moments_of_hits({k: v[200:] for k, v in hits.items()}, L, g.geom)
    merged = amc.merge_surface_ranks([(a[0], 4, a[1]), (b[0], 4, b[1])])
    assert np.array_equal(merged[0], whole[0]) and np.array_equal(merged[2], whole[1]) and merged[1] == 4
    assert whole[0][:, 0].sum() + whole[1].sum() == n
    hits["col"][:3] = np.nan
    assert amc.surface_moments_of_hits(hits, L, g.geom)[1].sum() >= 3


def _run_hits(kind, nsteps=3):
    import surface_oracle as SO
    from oracle import oracle as O
    from oracle import steps
    from argon_monte_carlo_b200 import init_state
    O.lib()
    O.set_ref_mode(False)
    cfg = {"pore": config.pore_config(False), "temp": config.pore_config(True), "cube": config.cube_config()}[kind]
    init = init_state.cube_initial_state(cfg) if kind == "cube" else init_state.pore_initial_state(cfg)
    st, ref = O.ParticleState(*init), O.ParticleState(*init)
    sink = SO.HitSink()
    counts = np.zeros(amc.NUM_CASES, dtype=np.int64)
    cheb = config.gap_energy_chebyshev(cfg, 16) if kind == "temp" else None
    for k in range(nsteps):
        if kind == "pore":
            SO.pore_step(st, cfg, sink)
            r = steps.pore_step(ref, cfg)
        elif kind == "cube":
            SO.cube_step(st, cfg, sink)
            r = steps.cube_step(ref, cfg)
        else:
            SO.temp_step_philox(st, cfg, 17, k, cheb, sink)
            r = steps.temp_step_philox(ref, cfg, 17, k, cheb)
        counts[:len(r["wall_counts"])] += r["wall_counts"]
    for f in SO.FIELDS:
        assert np.array_equal(getattr(st, f).view(np.uint64), getattr(ref, f).view(np.uint64)), f
    return cfg, sink.hits(), counts


@pytest.mark.parametrize("which", ["pore", "temp", "cube"])
def test_restatement_on_oracle_hit_lists(which):
    cfg, hits, counts = _run_hits(which)
    kind = {"pore": amc.KIND_PORE, "temp": amc.KIND_TEMP, "cube": amc.KIND_CUBE}[which]
    L = amc.surface_layout_of(cfg, kind, cfg.grid)
    acc, out = amc.surface_moments_of_hits(hits, L, None if which == "cube" else cfg.geom)
    per_case = np.array([acc[L.offsets[c]:L.offsets[c + 1], 0].sum() for c in range(amc.NUM_CASES)], dtype=np.int64)
    assert np.array_equal(per_case + out.astype(np.int64), counts)
    assert counts.sum() > 0
    if which == "pore":     # all specular: the tangential sums vanish against the normal one
        _, sums = outputs.decode_surface_sums(acc)
        assert np.all(sums[:, 0] >= 0)
        assert np.abs(sums[:, 1:3]).sum() <= 1e-9 * np.abs(sums[:, 0]).sum()


def test_csv_format(tmp_path):
    cfg = config.pore_config(True)
    L = amc.surface_layout_of(cfg, amc.KIND_TEMP, cfg.grid)
    acc = np.zeros((L.n_elements, amc.SURF_WORDS), dtype=np.uint64)
    e = L.offsets[4] - 1                # outermost annulus of case 3C
    acc[e, 0] = 5
    acc[e, 1] = np.uint64(1000 << amc.SURF_V1)
    f = outputs.surface_fields((acc, 10, np.zeros(amc.NUM_CASES, dtype=np.uint64)), cfg, cfg.grid, amc.KIND_TEMP)
    p = str(tmp_path / "surface.csv")
    outputs.write_surface_csv(p, f)
    lines = open(p).read().splitlines()
    assert lines[0] == ",".join(outputs.SURFACE_COLUMNS) and len(lines) == L.n_elements + 1
    row = dict(zip(outputs.SURFACE_COLUMNS, lines[1 + e].split(",")))
    assert row["case"] == "3" and row["hits"] == "5"
    a = float(row["area"])
    assert a > 0
    assert float(row["pressure"]) == pytest.approx(cfg.argon_mass * 1000 / (a * 10 * cfg.dt), rel=1e-14)


def test_driver_flags():
    a = driver_common.parse_args(10, "x", argv=[])
    assert a.surface_start is None
    a = driver_common.parse_args(10, "x", argv=["--surface-start", "4"])
    assert a.surface_start == 4
    with pytest.raises(SystemExit):
        driver_common.parse_args(10, "x", argv=["--surface-start", "-1"])

    class Fake:
        surface_on = False

        def surface_enable(self):
            self.surface_on = True
    sim = Fake()
    assert driver_common.surface_chunk(sim, a, 0, 8) == 4 and not sim.surface_on
    assert driver_common.surface_chunk(sim, a, 4, 8) == 8 and sim.surface_on
