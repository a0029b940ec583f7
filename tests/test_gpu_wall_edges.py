"""The drift / wall / recapture half of the timestep at its floating-point boundaries (states from tests/wall_edges.py)
against the oracle, bit for bit, through every copy of the per-particle step: k_keys (dry run) + k_scatter_advect (live
run, calm shortcut, closing recapture fused into the next step), k_advect and the cube sweep, the phase-level entry
points (advect_body), the surface-recording instantiations, the host-RNG case kernels, and the slab path (k_keys<SLAB>,
slab_pack) with one-layer slabs.  Each geometry at scale 1 and at the timed 12.5 M-particle scale, as built and inside a
background gas."""
import random

import numpy as np
import pytest

import wall_edges as we

pytestmark = pytest.mark.gpu

KEYS = ("x", "y", "z", "vx", "vy", "vz", "dist", "dist_x", "dist_y", "dist_z")
SEED = 17
GAS = 20000
PORE_CASES = [(k, s, gas) for k in ("pore", "temp") for s in ("1", "bench") for gas in (False, True)]
_STATES = {}


def edge_state(oracle, kind, scale, gas):
    """(cfg, arrays, labels) of the edge particles of one geometry and scale, optionally inside a gas."""
    key = (kind, scale, gas)
    if key not in _STATES:
        from argon_monte_carlo_b200 import init_state
        if kind == "cube":
            cfg = we.cube_cfg_of(scale)
            b = we.cube_edges(cfg)
            gas_arrs = init_state.synthetic_cube_state(cfg, GAS, seed=5) if gas else None
        else:
            cfg, s = we.pore_cfg_of(kind, scale)
            b = we.pore_edges(oracle, cfg, s)
            gas_arrs = init_state.synthetic_pore_state(cfg, seed=5, n=GAS) if gas else None
        arrs, labels = we.with_gas(b, gas_arrs) if gas else (b.arrays(), list(b.label))
        _STATES[key] = (cfg, arrs, labels)
    return _STATES[key]


def bits64(d):
    return {k: np.asarray(d[k]).view(np.int64) if k != "flag" else np.asarray(d[k]) for k in d}


def assert_state(got, st, labels, what):
    ref = {k: getattr(st, k) for k in KEYS}
    ref["flag"] = st.flag
    msg = we.first_difference(bits64({k: got[k] for k in KEYS + ("flag",)}), bits64(ref), labels, KEYS + ("flag",))
    assert msg is None, "%s: %s (int64 views)" % (what, msg)


def assert_bits(got, ref, labels, what):
    bad = np.nonzero(np.asarray(got, dtype=np.int64) != np.asarray(ref, dtype=np.int64))[0]
    assert len(bad) == 0, "%s: wall bits differ for %d particles; first %d (%s): %d vs %d" % (
        what, len(bad), bad[0], labels[bad[0]], got[bad[0]], ref[bad[0]])


def close(a, b):
    return abs(a - b) <= 1e-12 * abs(b) + 1e-40


def assert_stats(g, r, what):
    nc = len(r["wall_hits"])
    assert np.array_equal(np.asarray(g["wall_hits"][:nc]), r["wall_hits"]), (what, g["wall_hits"], r["wall_hits"])
    for k in ("errors", "oob_after_walls", "oob_after_pp", "oob_after_walls_recapture", "oob_after_pp_recapture", "pp_collisions"):
        if k in r:
            assert g[k] == r[k], (what, k, g[k], r[k])
    for k in ("dpz", "e_cold", "e_hot"):
        if k in r:
            assert close(g[k], r[k]), (what, k, g[k], r[k])


def ref_step(oracle, st, cfg, k, cheb, sink=None):
    """One timestep of the oracle with every counter the device reports (steps.pore_step / temp_step_philox, with the
    census after each recapture)."""
    g = cfg.geom
    if cfg.kind == "pore":
        from oracle import steps
        r = steps.pore_step(st, cfg, sink, None, want_bits=True)
        return dict(wall_hits=r["wall_counts"], errors=r["errors"], oob_after_walls=r["oob_after_walls"],
                    oob_after_pp=r["oob_after_pp"], pp_collisions=r["pp_collisions"], bits=r["hit_bits"])
    oracle.drift(st, cfg.dt, True)
    counts, sums, errs, bits = oracle.temp_walls_philox(st, g, SEED, k, cheb, sink, True)
    r = dict(wall_hits=counts, bits=bits, dpz=sums[0], e_cold=sums[1], e_hot=sums[2])
    r["oob_after_walls"] = oracle.temp_oob_count(st, g)
    oracle.temp_recapture(st, g)
    r["oob_after_walls_recapture"] = oracle.temp_oob_count(st, g)      # only moved particles can still be out
    r["pp_collisions"], _, perr = oracle.pp_groups(st, cfg.grid, cfg.collision_range, cfg.argon_mass, sink)
    r["errors"] = errs + perr
    r["oob_after_pp"] = oracle.temp_oob_count(st, g)
    oracle.temp_recapture(st, g)
    r["oob_after_pp_recapture"] = oracle.temp_oob_count(st, g)
    return r


def sim_of(cfg, n, **kw):
    from argon_monte_carlo_b200 import amc
    cheb = we.cheb_of(cfg) if cfg.kind == "temp" else None
    return amc.Simulation(cfg, seed=SEED, cheb=cheb, max_particles=n, **kw), cheb


def path_rows(p):
    return sorted(zip(*[np.asarray(a).view(np.int64).tolist() for a in p]))


@pytest.mark.parametrize("kind,scale,gas", PORE_CASES)
def test_pore_step3(oracle, kind, scale, gas):
    """step(3) in one call (k_keys DRY + k_scatter_advect LIVE, calm shortcut, closing recapture fused into steps 2 and
    3) against three oracle steps: state, counters, census, wall bits of the last step, completed paths."""
    from argon_monte_carlo_b200 import amc
    cfg, arrs, labels = edge_state(oracle, kind, scale, gas)
    sim, cheb = sim_of(cfg, len(arrs[0]), taps=amc.TAP_WALL_BITS | amc.TAP_PATHS)
    sim.set_state(*arrs)
    st = oracle.ParticleState(*arrs)
    sink = oracle.PathSink()
    refs = [ref_step(oracle, st, cfg, k, cheb, sink) for k in range(3)]
    got = sim.step(3)
    for k in range(3):
        assert_stats(got[k], refs[k], "step %d" % k)
    assert_bits(sim.wall_bits(), refs[2]["bits"], labels, "step 2")
    assert_state(sim.get_state(), st, labels, "after step(3)")
    assert path_rows(sim.completed_paths()) == path_rows(sink.arrays())
    assert sum(r["wall_hits"].sum() for r in refs) > 1000
    sim.close()


@pytest.mark.parametrize("kind,scale,gas", PORE_CASES)
def test_pore_phases(oracle, kind, scale, gas):
    """drift() / walls() / recapture(True) (advect_body: no calm shortcut) against the oracle's phases, state compared
    after each.  Temp: every case 4 hit that nothing else touched gives Es back from the device's speed after the
    walls, which must be mpmath's surface_energy_gap at the device's contact height to 1e-12.  (An applied energized hit
    leaves the particle at the contact point with its path lengths reset.)"""
    from argon_monte_carlo_b200 import amc, config
    cfg, arrs, labels = edge_state(oracle, kind, scale, gas)
    g = cfg.geom
    sim, cheb = sim_of(cfg, len(arrs[0]), taps=amc.TAP_WALL_BITS)
    sim.set_state(*arrs)
    st = oracle.ParticleState(*arrs)
    oracle.drift(st, cfg.dt, True)
    sim.drift()
    assert_state(sim.get_state(), st, labels, "drift")
    before = sim.get_state()
    d = sim.walls()
    if kind == "temp":
        counts, _, errs, bits = oracle.temp_walls_philox(st, g, SEED, 0, cheb, None, True)
    else:
        counts, errs, bits = oracle.pore_walls(st, g, None, True)
    assert np.array_equal(np.asarray(d["wall_hits"][:len(counts)]), counts) and d["errors"] == errs, (d["wall_hits"], counts, d["errors"], errs)
    dev_bits = sim.wall_bits()
    assert_bits(dev_bits, bits, labels, "walls")
    after = sim.get_state()
    assert_state(after, st, labels, "walls")
    if kind == "temp":
        only4 = np.nonzero((dev_bits == (1 << 5)) & (after["dist"] == 0.0))[0]     # applied (not the error path)
        assert len(only4) > 20
        m = g.argon_mass
        for i in only4:
            v = np.sqrt((before["vx"][i] ** 2 + before["vy"][i] ** 2) + before["vz"][i] ** 2)
            w2 = (after["vx"][i] ** 2 + after["vy"][i] ** 2) + after["vz"][i] ** 2
            E, Enew = (0.5 * m) * (v * v), (0.5 * m) * w2
            Es = E + (Enew - E) / g.alpha_g
            ref = float(config.surface_energy_gap(cfg, after["z"][i]))
            assert abs(Es - ref) <= 1e-12 * ref, (labels[i], after["z"][i], Es, ref)
        cnt = oracle.temp_oob_count(st, g)
        oracle.temp_recapture(st, g)
        assert sim.recapture(True) == (cnt, oracle.temp_oob_count(st, g))
    else:
        assert sim.recapture() == oracle.pore_recapture(st, g)
    assert_state(sim.get_state(), st, labels, "recapture")
    sim.close()


@pytest.mark.parametrize("scale,gas", [(s, gas) for s in ("1", "2") for gas in (False, True)])
@pytest.mark.parametrize("pp", ["groups", "sweep"])
def test_cube_step3(oracle, scale, gas, pp):
    """Cube faces, edges and corners: step(3) with the colour groups (k_keys + k_scatter_advect) and with the serial
    sweep (k_advect), and the phase-level drift() / walls()."""
    from argon_monte_carlo_b200 import amc
    from oracle import steps
    cfg, arrs, labels = edge_state(oracle, "cube", scale, gas)
    L = (cfg.cube_x, cfg.cube_y, cfg.cube_z)
    mode = amc.PP_GROUPS if pp == "groups" else amc.PP_SWEEP
    sim = amc.Simulation(cfg, kind=amc.KIND_CUBE, pp_mode=mode, max_particles=len(arrs[0]))
    sim.set_state(*arrs)
    st = oracle.ParticleState(*arrs)
    got = sim.step(3)
    for k in range(3):
        if pp == "groups":
            oracle.drift(st, cfg.dt, False)
            counts = oracle.cube_walls(st, *L)
            ncol, _, errs = oracle.pp_groups(st, cfg.grid, cfg.collision_range, cfg.argon_mass)
        else:
            r = steps.cube_step(st, cfg)
            counts, ncol, errs = r["wall_counts"], r["pp_collisions"], r["errors"]
        assert np.array_equal(np.asarray(got[k]["wall_hits"][:6]), counts) and got[k]["pp_collisions"] == ncol and got[k]["errors"] == errs
    assert_state(sim.get_state(), st, labels, "cube %s step(3)" % pp)
    sim.set_state(*arrs)
    st = oracle.ParticleState(*arrs)
    oracle.drift(st, cfg.dt, False)
    sim.drift()
    counts = oracle.cube_walls(st, *L)
    d = sim.walls()
    assert np.array_equal(np.asarray(d["wall_hits"][:6]), counts) and counts[0] > 0
    assert_state(sim.get_state(), st, labels, "cube phases")
    sim.close()


SURF = [(k, s) for k in ("pore", "temp", "cube") for s in ("1", "bench" if k != "cube" else "2")]


@pytest.mark.parametrize("kind,scale", SURF)
def test_surface_recording(oracle, kind, scale):
    """Surface recording on (k_scatter_advect_surf / k_advect_surf): the state equals the plain run bit for bit, and the
    words equal amc.surface_moments_of_hits of the oracle's hit records, the outside counts of the error-path hits
    included; once for step(3) and once for the phase-level walls()."""
    import surface_oracle as SO
    from argon_monte_carlo_b200 import amc
    cfg, arrs, labels = edge_state(oracle, kind, scale, True)
    kid = {"pore": amc.KIND_PORE, "temp": amc.KIND_TEMP, "cube": amc.KIND_CUBE}[kind]
    layout = amc.surface_layout_of(cfg, kid, cfg.grid)
    geom = None if kind == "cube" else cfg.geom
    runs = []
    for surf in (False, True):
        sim, cheb = sim_of(cfg, len(arrs[0]))
        sim.set_state(*arrs)
        if surf:
            sim.surface_enable()
        sim.step(3)
        runs.append(sim.get_state())
        if surf:
            raw = sim.surface_raw()
        sim.close()
    for k in KEYS:
        assert np.array_equal(runs[0][k].view(np.int64), runs[1][k].view(np.int64)), k
    sink = SO.HitSink()
    st = oracle.ParticleState(*arrs)
    for k in range(3):
        if kind == "pore":
            SO.pore_step(st, cfg, sink)
        elif kind == "temp":
            SO.temp_step_philox(st, cfg, SEED, k, cheb, sink)
        else:
            SO.cube_step(st, cfg, sink)
    acc, out = amc.surface_moments_of_hits(sink.hits(), layout, geom)
    assert_raw(raw, acc, out)
    if kind != "cube":
        assert out.sum() > 0                                   # error-path hits are in the words
    # phase level
    sim, cheb = sim_of(cfg, len(arrs[0]))
    sim.set_state(*arrs)
    sim.surface_enable()
    sim.drift()
    sim.walls()
    raw = sim.surface_raw()
    sim.close()
    sink = SO.HitSink()
    st = oracle.ParticleState(*arrs)
    oracle.drift(st, cfg.dt, kind != "cube")
    if kind == "pore":
        SO.pore_wall_hits(st, cfg.geom, sink)
    elif kind == "temp":
        SO.temp_walls_philox_hits(st, cfg.geom, SEED, 0, cheb, sink)
    else:
        SO.cube_wall_hits(st, (cfg.cube_x, cfg.cube_y, cfg.cube_z), sink)
    acc, out = amc.surface_moments_of_hits(sink.hits(), layout, geom)
    assert_raw(raw, acc, out)


def assert_raw(raw, acc, out):
    assert np.array_equal(np.asarray(raw[2], dtype=np.uint64), np.asarray(out, dtype=np.uint64)), ("outside", raw[2], out)
    bad = np.nonzero(np.any(raw[0] != acc, axis=1))[0]
    assert len(bad) == 0, "%d surface elements differ (first %d: %s vs %s)" % (len(bad), bad[0], raw[0][bad[0]], acc[bad[0]])
    assert acc[:, 0].sum() > 0


@pytest.mark.parametrize("scale", ["1", "bench"])
def test_temp_host_rng(oracle, scale):
    """step_host_rng() twice (k_case_specular / detect / apply, NaN normals of failed contacts included) against
    steps.temp_step_host_rng with the same Mersenne-Twister states."""
    from argon_monte_carlo_b200 import amc
    from oracle import steps
    cfg, arrs, labels = edge_state(oracle, "temp", scale, True)
    np.random.seed(23)
    random.seed(23)
    state_np, state_py = np.random.get_state(), random.getstate()
    st = oracle.ParticleState(*arrs)
    refs = [steps.temp_step_host_rng(st, cfg) for _ in range(2)]
    np.random.set_state(state_np)
    random.setstate(state_py)
    sim = amc.Simulation(cfg, rng_mode=amc.RNG_HOST, max_particles=len(arrs[0]))
    sim.set_state(*arrs)
    for k in range(2):
        g = sim.step_host_rng()
        r = refs[k]
        assert np.array_equal(np.asarray(g["wall_hits"]), r["wall_counts"]), (k, g["wall_hits"], r["wall_counts"])
        for key in ("errors", "oob_after_walls", "oob_after_pp", "pp_collisions", "dpz", "e_cold", "e_hot"):
            assert g[key] == r[key], (k, key, g[key], r[key])
    assert refs[0]["errors"] > 0
    assert_state(sim.get_state(), st, labels, "host rng")
    sim.close()


def slab_cuts(cfg):
    """One-layer slabs at the layers of the end plates, the recapture targets and the wall planes, the rest in between."""
    from argon_monte_carlo_b200 import slab
    g, e = cfg.geom, cfg.grid.edge[2]
    nz = cfg.grid.nc[2]
    lay = lambda z: int(slab.owner_layer(np.array([z]), e)[0])
    singles = {0, 1, nz - 1, lay(g.recap_lo), lay(g.recap_hi), lay(g.oah), lay(g.zh3), lay(g.zgb_p), lay(g.zgt_m), lay(g.z_cold), lay(g.zc3)}
    cuts = set()
    for l in singles:
        cuts |= {max(0, min(nz, l)), max(0, min(nz, l + 1))}
    return sorted(cuts | {0, nz})


@pytest.mark.parametrize("kind,scale", [("temp", "1"), ("temp", "bench"), ("pore", "1")])
def test_slab_ranks(oracle, kind, scale):
    """SlabSimulation with one-layer slabs at the layers of the edge particles, the wall planes and the recapture targets
    (k_keys<SLAB>, slab_pack, the far transfer of a recaptured particle) against the single-domain run, and a 1-rank
    p2p step_fused run: state, counters, no particle lost or duplicated."""
    from argon_monte_carlo_b200 import amc, slab
    cfg, arrs, labels = edge_state(oracle, kind, scale, True)
    n = len(arrs[0])
    one, _ = sim_of(cfg, n)
    one.set_state(*arrs)
    ref = one.step(3)
    ref_state = one.get_state()
    ref_digest = one.state_digest()
    one.close()
    cuts = slab_cuts(cfg)
    assert len(cuts) > 10
    sim = slab.SlabSimulation(cfg, len(cuts) - 1, arrs[2], seed=SEED, cuts=cuts)
    sim.set_state(*arrs)
    got = sim.step(3)
    st = sim.get_state()
    sim.close()
    assert st["_owned_total"] == n, "particles lost or duplicated across ranks (cuts %s)" % cuts
    counters = ("wall_collisions", "pp_collisions", "pair_checks_ref", "oob_after_walls", "oob_after_pp", "errors")
    for a, b in zip(ref, got):
        for k in counters:
            assert a[k] == b[k], (k, a[k], b[k], cuts)
        assert np.array_equal(a["wall_hits"], b["wall_hits"])
    msg = we.first_difference(bits64({k: st[k] for k in KEYS + ("flag",)}), bits64({k: ref_state[k] for k in KEYS + ("flag",)}),
                              labels, KEYS + ("flag",))
    assert msg is None, "cuts %s: %s" % (cuts, msg)
    p2p = slab.SlabSimulation(cfg, 1, arrs[2], seed=SEED, p2p=True)
    p2p.set_state(*arrs)
    got = p2p.step_fused(3)
    for a, b in zip(ref, got):
        for k in counters:
            assert a[k] == b[k], (k, a[k], b[k])
    assert p2p.state_digest() == ref_digest
    p2p.close()
