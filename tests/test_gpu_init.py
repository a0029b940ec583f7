"""Device-side synthetic initial state (amc_init_synthetic, SURVEY 8f): agreement with the NumPy restatement of the
generator, region populations, Maxwellian velocities, slab selection."""
import numpy as np
import pytest

from synthetic_ref import generate

pytestmark = pytest.mark.gpu


def test_pore_spec_matches_numpy_restatement(temp_cfg):
    from argon_monte_carlo_b200 import amc, init_state
    spec = init_state.pore_spec(temp_cfg, seed=17)
    sim = amc.Simulation(temp_cfg)
    n = sim.init_synthetic(spec)
    assert n == temp_cfg.num_molecules
    got = sim.get_state()
    x, y, z, vx, vy, vz, reg = generate(spec, np.arange(n))
    # tolerance: CUDA's and glibc's sin / cos / log differ in the last ulp; positions are ~1e-7 m, speeds ~1e2 m/s
    for k, ref, scale in (("x", x, 1e-7), ("y", y, 1e-7), ("z", z, 1e-5), ("vx", vx, 1e3), ("vy", vy, 1e3), ("vz", vz, 1e3)):
        assert np.max(np.abs(got[k] - ref)) <= 1e-12 * scale, k
    assert not got["dist"].any() and not got["flag"].any()
    # region populations follow the volumes (Pore:79-83) within 5 sigma of the multinomial
    cum = np.array(spec.cum_weight[:5]); pr = np.diff(np.concatenate([[0.0], cum]))
    counts = np.bincount(reg, minlength=5)
    assert np.all(np.abs(counts - n * pr) <= 5 * np.sqrt(n * pr * (1 - pr)) + 1)
    # Maxwellian: component mean 0, variance a_shape^2 (5 sigma of the sampling error)
    for k in ("vx", "vy", "vz"):
        assert abs(got[k].mean()) <= 5 * temp_cfg.a_shape / np.sqrt(n)
        assert abs(got[k].var() / temp_cfg.a_shape ** 2 - 1) <= 5 * np.sqrt(2.0 / n)
    # every particle inside its region, one argon radius off the walls it touches
    r2 = got["x"] ** 2 + got["y"] ** 2
    assert np.all(r2 <= (np.array(spec.radius[:5])[reg] * (1 + 1e-12)) ** 2)
    # and the state is usable: the energized pore steps without anomalies
    st = sim.step(2)
    assert all(s["errors"] == 0 and s["oob_after_walls_recapture"] == 0 for s in st)
    sim.close()


def test_slabs_generate_their_own_particles_and_run_like_the_single_domain(temp_cfg):
    """Three ranks (one GPU, local transport) each generate their slab of the same job; together they hold every
    particle exactly once, equal to the single-domain state, and three steps later the runs are still
    bit-identical (ids are global, Philox is keyed by id)."""
    from argon_monte_carlo_b200 import amc, init_state, slab
    make = lambda kz: init_state.pore_spec(temp_cfg, seed=5, keep_z=kz)
    one = amc.Simulation(temp_cfg, seed=5)
    n = one.init_synthetic(make(None))
    ref0 = one.get_state()
    sl = slab.SlabSimulation(temp_cfg, 3, ref0["z"], seed=5)
    sl.init_synthetic(make)
    got0 = sl.get_state()
    assert got0["_owned_total"] == n
    for k in ("x", "y", "z", "vx", "vy", "vz"):
        assert np.array_equal(got0[k], ref0[k]), k
    s1, s2 = one.step(3), sl.step(3)
    assert [a["collisions"] for a in s1] == [b["collisions"] for b in s2]
    a, b = one.get_state(), sl.get_state()
    for k in ("x", "y", "z", "vx", "vy", "vz", "dist"):
        assert np.array_equal(a[k], b[k]), k
    one.close(); sl.close()


def test_cube_spec_and_bad_arguments(cube_cfg):
    from argon_monte_carlo_b200 import amc, init_state
    sim = amc.Simulation(cube_cfg, max_particles=200000)
    spec = init_state.cube_spec(cube_cfg, 150000, seed=127)
    assert sim.init_synthetic(spec) == 150000
    got = sim.get_state()
    x, y, z, vx, vy, vz, _ = generate(spec, np.arange(150000))
    assert np.array_equal(got["x"], x) and np.array_equal(got["y"], y) and np.array_equal(got["z"], z)   # no transcendental functions in a box
    assert np.max(np.abs(got["vx"] - vx)) <= 1e-9
    spec.n_total = 300000
    with pytest.raises(amc.AmcError):
        sim.init_synthetic(spec)
    spec.n_total, spec.n_regions = 1000, 0
    with pytest.raises(amc.AmcError):
        sim.init_synthetic(spec)
    sim.close()


def test_overlap_free_seeding(oracle):
    """amc_seed_relax: the synthetic state starts with ~0.2 % of its particles overlapping a neighbour, like the
    reference's own (1,051 pairs at 557,649 particles); after relaxing, a census with a KD-tree finds no pair closer
    than the collision range, untouched particles keep their positions, velocities are untouched, and the first
    timestep resolves (almost) no particle-particle collision instead of the initial burst."""
    from scipy.spatial import cKDTree
    from argon_monte_carlo_b200 import amc, config, init_state
    cfg = config.pore_config(True)
    n = cfg.num_molecules
    sim = amc.Simulation(cfg, seed=17, max_particles=n)
    sim.init_synthetic(init_state.pore_spec(cfg, 17))
    before = sim.get_state()
    pairs0 = cKDTree(np.column_stack([before["x"], before["y"], before["z"]])).query_pairs(cfg.collision_range)
    assert 800 < len(pairs0) < 1400                      # the reference's initial state: 1,051
    redrawn, left = sim.seed_relax(8)
    after = sim.get_state()
    assert left == 0 and len(pairs0) * 0.9 <= redrawn <= len(pairs0) * 1.2
    pts = np.column_stack([after["x"], after["y"], after["z"]])
    assert len(cKDTree(pts).query_pairs(cfg.collision_range)) == 0
    moved = (after["x"] != before["x"]) | (after["y"] != before["y"]) | (after["z"] != before["z"])
    assert moved.sum() <= redrawn and moved.sum() >= 0.9 * len(pairs0) * 0.95
    hi = np.array([max(a, b) for a, b in pairs0])
    assert moved[hi].all()                               # in every overlapping pair the higher index was re-drawn
    for k in ("vx", "vy", "vz"):
        assert np.array_equal(after[k], before[k])
    r = np.hypot(after["x"], after["y"])
    assert r.max() <= cfg.open_air_radius and after["z"].min() > 0 and after["z"].max() < cfg.total_height
    first = sim.step(1)[0]
    assert first["pp_collisions"] < 600                  # steady state ~260 per step; the un-relaxed start resolves ~1,070
    sim.close()


def test_seed_relax_pinned():
    """amc_seed_relax at 557,649 particles, seed 17: positions re-drawn and the state digest afterwards.  The values were
    recorded on a B200 with the earlier seeding kernel, which loaded the candidates with the threads; the seeding variant
    of the bulk-copy detection kernel has to mark the same particles in every round."""
    from argon_monte_carlo_b200 import amc, config, init_state
    cfg = config.pore_config(True)
    n = cfg.num_molecules
    assert n == 557649
    sim = amc.Simulation(cfg, seed=17, max_particles=n)
    sim.init_synthetic(init_state.pore_spec(cfg, 17))
    assert sim.seed_relax(8) == (1115, 0)
    assert sim.state_digest() == (6298284287226869198, 17013363693960920395, 557649)
    sim.close()
