"""The pair pass at its floating-point boundaries (states from tests/pair_edges.py) against the oracle, bit for bit:
particles on cell edges, band edges and the doubles next to them, pairs at exactly prev(overlap_sq) and overlap_sq,
pairs only the slack of the fp32 filter keeps, cells with 1, 8 and 9 filter hits, capacities at their switch points,
a degenerate pair, and the same lattice through the cube's serial sweep and emulated slab ranks."""
import numpy as np
import pytest

import pair_edges as pe

pytestmark = pytest.mark.gpu

KEYS = ("x", "y", "z", "vx", "vy", "vz", "dist", "dist_x", "dist_y", "dist_z")


def pair_set(hi, lo, grp, cell):
    return sorted(zip(hi.tolist(), lo.tolist(), grp.tolist(), cell.tolist()))


def assert_same(got, st, labels, what):
    msg = pe.first_difference(got, st.arrays(), labels, KEYS + ("flag",))
    assert msg is None, "%s: %s" % (what, msg)


def assert_counters(g, ncol, checks, errs, what):
    assert (g["pp_collisions"], g["pair_checks_ref"], g["errors"]) == (ncol, checks, errs), what


def run_pairs(oracle, cfg, b, labels=None, sweep=False, grid=None, extra=None, **kw):
    """sim.pairs() against oracle.pp_groups (or cube_pp_sweep) from the same state: counters, state and pair multiset."""
    from argon_monte_carlo_b200 import amc
    grid = grid or cfg.grid
    arrs = b.arrays()
    labels = list(b.label)
    if extra is not None:
        arrs = tuple(np.concatenate([a, [e]]) for a, e in zip(arrs, extra))
        labels.append("fast particle")
    st = oracle.ParticleState(*arrs)
    sink = oracle.PairSink()
    run = oracle.cube_pp_sweep if sweep else oracle.pp_groups
    ncol, checks, errs = run(st, grid, cfg.collision_range, cfg.argon_mass, None, sink)
    sim = amc.Simulation(cfg, taps=amc.TAP_PAIRS, max_particles=len(arrs[0]), grid=grid, **kw)
    sim.set_state(*arrs)
    g = sim.pairs()
    assert_counters(g, ncol, checks, errs, "pair pass counters")
    assert_same(sim.get_state(), st, labels, "pair pass")
    assert pair_set(*sim.pair_list()) == pair_set(*sink.arrays())
    return sim, st, ncol, errs


@pytest.mark.parametrize("which", ["pore", "cube"])
def test_lattice_colour_groups(oracle, pore_cfg, which):
    """Every boundary value with partners at prev(overlap_sq) and overlap_sq on both sides, and 2- and 3-axis corners,
    through the phase-level pair pass (colour groups).  On the Pore grid the sampling kernel bins the same state by the
    owner rule, with one particle fast enough for its per-particle fallback."""
    from argon_monte_carlo_b200 import amc
    cfg = pore_cfg if which == "pore" else pe.cube_groups_config()
    b = (pe.pore_lattice if which == "pore" else pe.cube_lattice)(cfg)
    kw = {} if which == "pore" else {"kind": amc.KIND_CUBE, "pp_mode": amc.PP_GROUPS}
    extra = None
    if which == "pore":
        p, v = pe.fast_particle(cfg)
        extra = tuple(p) + tuple(v)
    sim, st, ncol, _ = run_pairs(oracle, cfg, b, extra=extra, **kw)
    assert ncol >= len(b.expected(cfg.grid))
    if which == "pore":
        built = tuple(np.concatenate([a, [e]]) for a, e in zip(b.arrays(), extra))
        for what in ("after the pair pass", "as built"):
            if what == "as built":
                sim.set_state(*built)
            state = sim.get_state()
            sim.sample_enable(0)
            sim.sample_now()
            acc, ns, outside = sim.sample_raw()
            ref, _, ref_out = amc.sample_moments_of_arrays(state, cfg.grid)
            bad = np.nonzero(np.any(acc != ref, axis=1))[0]
            assert len(bad) == 0 and outside == ref_out, "sample %s: cell %d differs" % (what, bad[0] if len(bad) else -1)
            sim.sample_disable()
    sim.close()


@pytest.mark.parametrize("which", ["pore", "cube"])
def test_lattice_one_step(oracle, pore_cfg, which):
    """The same lattice reached by a drift: start positions that one drift maps exactly onto the boundaries, then
    step(1) (k_keys, k_scatter_advect, k_detect_tma, k_pairs_group) against the oracle's timestep."""
    from argon_monte_carlo_b200 import amc
    from oracle import steps
    cfg = pore_cfg if which == "pore" else pe.cube_groups_config()
    b = (pe.pore_lattice if which == "pore" else pe.cube_lattice)(cfg)
    b.drift_preimages(cfg.dt)
    st = oracle.ParticleState(*b.arrays())
    pairs = oracle.PairSink()
    if which == "pore":
        r = steps.pore_step(st, cfg, None, pairs)
        ncol, checks, errs = r["pp_collisions"], r["checks"], r["errors"]
        sim = amc.Simulation(cfg, taps=amc.TAP_PAIRS, max_particles=st.n)
    else:
        oracle.drift(st, cfg.dt, False)
        oracle.cube_walls(st, cfg.cube_x, cfg.cube_y, cfg.cube_z)
        ncol, checks, errs = oracle.pp_groups(st, cfg.grid, cfg.collision_range, cfg.argon_mass, None, pairs)
        sim = amc.Simulation(cfg, kind=amc.KIND_CUBE, pp_mode=amc.PP_GROUPS, taps=amc.TAP_PAIRS, max_particles=st.n)
    sim.set_state(*b.arrays())
    g = sim.step(1)[0]
    assert ncol > 500
    assert_counters(g, ncol, checks, errs, "step counters")
    assert_same(sim.get_state(), st, b.label, "one step")
    assert pair_set(*sim.pair_list()) == pair_set(*pairs.arrays())
    sim.close()


@pytest.mark.parametrize("which", ["pore", "cube 2.0/8"])
def test_threshold_pairs(oracle, pore_cfg, which):
    """Pairs at prev(overlap_sq) / overlap_sq: far-corner pairs that only the slack of det_thr keeps, random places and
    directions, across detection bin boundaries, and cells with 1, 8 and 9 filter hits (one true pair each).  The
    cube grid carries a background gas so every cell fits the detection tile and is hashed into 64 x bins."""
    from argon_monte_carlo_b200 import amc, config
    if which == "pore":
        cfg, kw = pore_cfg, {}
        b, used = pe.threshold_cells(cfg)
    else:
        cfg, kw = config.cube_config(2.0, 8), {"kind": amc.KIND_CUBE, "pp_mode": amc.PP_GROUPS}
        b, used = pe.threshold_cells(cfg, background=60000)
    sim, st, ncol, _ = run_pairs(oracle, cfg, b, **kw)
    assert ncol == len(b.pair_keys("collide"))
    sim.close()


@pytest.mark.parametrize("case", list(pe.CAPACITY_CASES))
def test_capacity_switch_points(oracle, pore_cfg, case):
    """One reference cell at each capacity switch point: 384 / 385 candidates (detection tile or flagged unseen),
    64 / 65 overlapping pairs (candidate list or scan mode), 32 / 33 moved particles (on chip or spilled), 512 members
    (accepted) and 513 (AmcError)."""
    from argon_monte_carlo_b200 import amc
    b = pe.capacity_cell(pore_cfg, case)
    if case == "members 513":
        sim = amc.Simulation(pore_cfg, max_particles=len(b.pos))
        sim.set_state(*b.arrays())
        with pytest.raises(amc.AmcError, match="AMC_MAX_MEMBERS"):
            sim.pairs()
        sim.close()
        return
    sim, _, ncol, _ = run_pairs(oracle, pore_cfg, b)
    assert ncol == len(b.collide)
    sim.close()


@pytest.mark.parametrize("path", ["colour groups", "cube sweep"])
def test_degenerate_pair(oracle, pore_cfg, cube_cfg, path):
    """Two overlapping particles with equal velocities (a == 0): the error is counted and the pair skipped, as the
    oracle does, next to an ordinary collision in the same cell."""
    if path == "colour groups":
        b = pe.degenerate_pair(pore_cfg)
        _, _, ncol, errs = run_pairs(oracle, pore_cfg, b)
    else:
        b = pe.degenerate_pair(cube_cfg, cell=(4, 5, 6))
        _, _, ncol, errs = run_pairs(oracle, cube_cfg, b, sweep=True)
    assert ncol == 1 and errs >= 1


@pytest.mark.parametrize("sweep", ["events", "handover"])
def test_lattice_cube_sweep(oracle, cube_cfg, sweep, monkeypatch):
    """The cube lattice through the serial cell sweep (PP_SWEEP against oracle.cube_pp_sweep): the event-driven sweep,
    and column lists of 16 so every pass is handed to the plain walk."""
    if sweep == "handover":
        monkeypatch.setenv("AMC_SWEEP_COLCAP", "16")
    b = pe.cube_lattice(cube_cfg)
    sim, _, ncol, _ = run_pairs(oracle, cube_cfg, b, sweep=True)
    assert ncol >= len(b.expected(cube_cfg.grid))
    sim.close()


def run_single(cfg, init, steps, **kw):
    from argon_monte_carlo_b200 import amc
    sim = amc.Simulation(cfg, taps=amc.TAP_PAIRS, max_particles=len(init[0]), **kw)
    sim.set_state(*init)
    stats = sim.step(steps)
    out = sim.get_state(), stats, sim.pair_list(), sim.histograms()
    sim.close()
    return out


def run_slabs(cfg, init, steps, nranks, cuts=None, **kw):
    from argon_monte_carlo_b200 import amc, slab
    sim = slab.SlabSimulation(cfg, nranks, init[2], taps=amc.TAP_PAIRS, cuts=cuts, **kw)
    sim.set_state(*init)
    stats = sim.step(steps)
    out = sim.get_state(), stats, sim.pair_list(), sim.histograms(), sim.cuts
    sim.close()
    return out


def compare(single, slabs, n, labels):
    (st1, stats1, pairs1, hist1), (st2, stats2, pairs2, hist2, cuts) = single, slabs
    assert st2["_owned_total"] == n, "particles lost or duplicated across ranks (cuts %s)" % cuts
    for a, b in zip(stats1, stats2):
        for k in ("wall_collisions", "pp_collisions", "pair_checks_ref", "oob_after_walls", "oob_after_pp", "errors"):
            assert a[k] == b[k], (k, a[k], b[k], cuts)
    msg = pe.first_difference(st2, st1, labels, KEYS + ("flag",))
    assert msg is None, "cuts %s: %s" % (cuts, msg)
    key = lambda p: sorted(zip(p[0].tolist(), p[1].tolist(), p[2].tolist()))
    assert key(pairs1) == key(pairs2)
    assert np.array_equal(hist1[0], hist2[0]) and hist1[1] == hist2[1]


def test_lattice_slab_ranks(pore_cfg):
    """The Pore lattice reached by a drift, stepped on emulated slab ranks with cuts at the z layers it occupies
    (one-layer slabs included): equal to the single-domain run bit for bit, no particle lost or duplicated."""
    b = pe.pore_lattice(pore_cfg)
    b.drift_preimages(pore_cfg.dt)
    init = b.arrays()
    nz = pore_cfg.grid.nc[2]
    single = run_single(pore_cfg, init, 2)
    for cuts in ([0, 1, 2, 3, 74, nz - 1, nz], [0, 40, 41, 42, nz]):
        compare(single, run_slabs(pore_cfg, init, 2, len(cuts) - 1, cuts), len(init[0]), b.label)
