"""The builders of tests/pair_edges.py check themselves on the CPU: every coordinate is the boundary it claims, every
pair has the claimed squared distance, the worst placements for the fp32 filter are where they should be, and the
oracle resolves exactly the pairs each state was built to collide."""
import math

import numpy as np
import pytest

import pair_edges as pe


def oracle_pairs(oracle, b, grid, cfg, sweep=False):
    st = oracle.ParticleState(*b.arrays())
    sink = oracle.PairSink()
    run = oracle.cube_pp_sweep if sweep else oracle.pp_groups
    ncol, checks, errs = run(st, grid, cfg.collision_range, cfg.argon_mass, None, sink)
    hi, lo, _, _ = sink.arrays()
    return set(zip(hi.tolist(), lo.tolist())), ncol, errs


def check_pairs(b):
    osq = b.osq
    for i, j in b.collide:
        assert pe.d2_kernel(b.pos[i], b.pos[j]) == pe.down(osq) or pe.d2_kernel(b.pos[i], b.pos[j]) < osq, b.label[j]
    for i, j in b.miss:
        assert pe.d2_kernel(b.pos[i], b.pos[j]) >= osq, b.label[j]
    # the constructed pairs are the only ones within two collision ranges: nothing else can interact
    assert pe.close_pairs(b, 2.0 * b.cr) == b.pair_keys("collide") | b.pair_keys("miss")


def test_boundary_values_are_what_they_claim(pore_cfg, cube_cfg):
    for cfg in (pore_cfg, cube_cfg):
        for a in range(3):
            vals = pe.boundary_values(cfg.grid, a)
            pe.check_boundary_values(cfg.grid, a, vals)
            assert len(vals) >= 6 * cfg.grid.nc[a]
    zeros = [lab for v, lab in pe.boundary_values(pore_cfg.grid, 0) if v == 0.0 and math.copysign(1.0, v) < 0]
    assert zeros == ["-0.0 (edge[7])"]
    with pytest.raises(AssertionError):
        pe.check_boundary_values(pore_cfg.grid, 2, [(pe.up(pore_cfg.grid.edge[2][5]), "edge[5]")])


def test_owner_estimate_misses_where_the_fallback_decides(pore_cfg, cube_cfg):
    """The fast owner estimate is wrong on 97 of the 147 interior z edges of the Pore grid, one double below 10 of the
    13 interior x and y edges, and one double below every interior edge of the cube grid; owner_exact is the rule."""
    m = [pe.estimate_misses(pore_cfg.grid, a) for a in range(3)]
    assert len(m[2]["on"]) == 97 and len(m[0]["below"]) == 10 and len(m[1]["below"]) == 10
    assert all(len(pe.estimate_misses(cube_cfg.grid, a)["below"]) == cube_cfg.grid.nc[a] - 1 for a in range(3))
    g = pore_cfg.grid
    e = g.edge[2]
    assert np.array_equal(pe.owner_exact(g, 2, e[1:-1]), np.arange(1, g.nc[2]))
    assert np.array_equal(pe.owner_exact(g, 2, pe.down(e[1:-1])), np.arange(0, g.nc[2] - 1))
    assert pe.owner_exact(g, 0, -0.0) == 7 and pe.owner_exact(g, 0, pe.down(g.edge[0][0])) == -1


def test_partner_at_hits_the_exact_squared_distance(pore_cfg):
    rng = np.random.default_rng(5)
    osq = pe.overlap_sq(pore_cfg.collision_range)
    assert osq == pore_cfg.collision_range * pore_cfg.collision_range
    found = 0
    for _ in range(200):
        a = rng.uniform(-1.5e-7, 1.5e-7, 3) * np.array([1.0, 1.0, 20.0])
        a[2] = abs(a[2])
        for target in (pe.down(osq), osq):
            p = pe.partner_at(a, rng.normal(size=3), target)
            if p is not None:
                found += 1
                assert pe.d2_kernel(a, p) == target
                assert (math.sqrt(pe.d2_kernel(a, p)) < pore_cfg.collision_range) == (target < osq)   # Pore:173-174
    assert found > 150         # far from the origin a single start often has no exact hit; Builder.pair tilts and retries


def test_drift_preimages_land_on_the_boundaries(oracle, pore_cfg):
    b = pe.pore_lattice(pore_cfg)
    want = np.array(b.pos)
    n0 = len(b.pos)
    dropped, keep = b.drift_preimages(pore_cfg.dt)
    assert dropped < 0.1 * n0
    st = oracle.ParticleState(*b.arrays())
    oracle.drift(st, pore_cfg.dt, True)
    got = np.stack([st.x, st.y, st.z], axis=1)
    assert np.array_equal(got, want[keep])            # by value: a drift gives +0.0 where -0.0 was placed


@pytest.mark.parametrize("which", ["pore", "cube", "cube 14"])
def test_lattice_resolves_exactly_the_intended_pairs(oracle, pore_cfg, cube_cfg, which):
    cfg = {"pore": pore_cfg, "cube": cube_cfg}.get(which) or pe.cube_groups_config()
    b = (pe.pore_lattice if which == "pore" else pe.cube_lattice)(cfg)
    attempted = len(b.collide) + len(b.miss) + b.skipped
    assert b.skipped < 0.02 * attempted and len(b.collide) > 500
    check_pairs(b)
    pairs, ncol, errs = oracle_pairs(oracle, b, cfg.grid, cfg)
    want = b.expected(cfg.grid)
    assert pairs == want and errs == 0 and len(b.pair_keys("collide") - want) < 50   # only pairs outside the grid drop out
    if which != "pore":
        assert oracle_pairs(oracle, b, cfg.grid, cfg, sweep=True)[0] == want
    # every boundary value of the z axis (pore) / every axis (cube) carries an anchor exactly
    axes = (2,) if which == "pore" else (0, 1, 2)
    pos = np.array(b.pos)
    for a in axes:
        vals = pe.boundary_values(cfg.grid, a)
        have = set(pos[:, a].view(np.int64).tolist())
        missing = [lab for v, lab in vals if np.float64(v).view(np.int64) not in have]
        assert len(missing) <= 0.02 * len(vals), missing[:5]


@pytest.mark.parametrize("which", ["pore", "cube 2.0/8"])
def test_threshold_cells(oracle, pore_cfg, which):
    from argon_monte_carlo_b200 import config
    cfg = pore_cfg if which == "pore" else config.cube_config(2.0, 8)
    b, used = pe.threshold_cells(cfg, background=0 if which == "pore" else 60000)
    check_pairs(b)
    g = cfg.grid
    thr = float(pe.det_thr(g, b.cr))
    for i, j in b.collide:
        cell = tuple(int(pe.owner_exact(g, a, b.pos[i][a])) for a in range(3))
        assert float(pe.filter_d2(b.pos[i], b.pos[j], pe.cell_lo(g, cell))) < thr          # the filter keeps every true pair
    far = [(i, j) for i, j in b.collide if b.label[i].startswith(("far corner", "1 filter", "8 filter", "9 filter"))]
    assert len(far) == len(used["worst"]) + len(used["hits"])
    for i, j in far:
        cell = tuple(int(pe.owner_exact(g, a, b.pos[i][a])) for a in range(3))
        rel = (b.pos[i] - pe.cell_lo(g, cell)) / np.array([g.edge[a][cell[a] + 1] - g.lo[a][cell[a]] for a in range(3)])
        assert np.all(rel > 0.8), rel                                # the far corner of the cell
        assert pe.missed_by_rounded_down_filter(g, b.cr, b.pos[i], b.pos[j], cell)
    for c, h in used["hits"]:                                        # filter hits per cell: exactly h
        inside = [(i, j) for i, j in b.collide + b.miss
                  if tuple(int(pe.owner_exact(g, a, b.pos[i][a])) for a in range(3)) == c
                  and float(pe.filter_d2(b.pos[i], b.pos[j], pe.cell_lo(g, c))) < thr]
        assert len(inside) == h
    if which == "cube 2.0/8":
        nb = pe.det_bins(g, b.cr, 0, 3)[0]
        assert nb == 64 and math.floor(float(np.float32(g.edge[0][4] - g.lo[0][3]) / pe.det_w(g, b.cr))) > 64   # the clamp
        assert len(b.pos) > 50000
    pairs, _, errs = oracle_pairs(oracle, b, g, cfg)
    assert pairs == b.expected(g) == b.pair_keys("collide") and errs == 0


@pytest.mark.parametrize("case", list(pe.CAPACITY_CASES))
def test_capacity_cells(oracle, pore_cfg, case):
    b = pe.capacity_cell(pore_cfg, case)
    n_lat, n_pair, triple = pe.CAPACITY_CASES[case]
    assert len(b.pos) == n_lat + n_pair + 2 * int(triple)
    g = pore_cfg.grid
    pos = np.array(b.pos)
    for a in range(3):                                                # all in the owner cell, outside every band
        assert np.all(pe.owner_exact(g, a, pos[:, a]) == (9, 9, 40)[a])
        assert np.all(pos[:, a] < g.lo[a][(9, 9, 40)[a] + 1]) and np.all(pos[:, a] > g.edge[a][(9, 9, 40)[a]])
    pairs, ncol, errs = oracle_pairs(oracle, b, g, pore_cfg)
    assert pairs == b.pair_keys("collide") and errs == 0
    moved = {p for q in pairs for p in q}
    if case.startswith("moved"):
        assert len(moved) == int(case.split()[1])
    if case.startswith("overlapping"):
        assert ncol == int(case.split()[2])


def test_degenerate_pair_counts_an_error(oracle, pore_cfg, cube_cfg):
    for cfg, sweep in ((pore_cfg, False), (cube_cfg, True)):
        b = pe.degenerate_pair(cfg, cell=(9, 9, 40) if not sweep else (4, 5, 6))
        pairs, ncol, errs = oracle_pairs(oracle, b, cfg.grid, cfg, sweep=sweep)
        assert pairs == b.pair_keys("collide") and ncol == 1 and errs >= 1
