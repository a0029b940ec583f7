"""GPU parity tests proper: the CUDA path (through the C ABI, via ctypes) against the CPU oracle
from identical input states.  Bar (BASELINE.json north_star): collision-pair sets and wall-hit
flags bit-exact, velocities within 1e-6 relative.  The oracle's plain arithmetic mode performs the
same IEEE operations in the same order as the kernels, so these tests assert the stronger
property: the whole particle state is bit-identical."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KEYS = ("x", "y", "z", "vx", "vy", "vz", "dist", "dist_x", "dist_y", "dist_z")


def assert_state_equal(got, st, what=""):
    for k in KEYS:
        a, b = got[k], getattr(st, k)
        bad = np.nonzero(a != b)[0]
        assert len(bad) == 0, "%s: %s differs for %d particles, first id %d: %r vs %r" % (
            what, k, len(bad), bad[0], a[bad[0]], b[bad[0]])
    assert np.array_equal(got["flag"].astype(bool), st.flag.astype(bool)), what + ": flag differs"


def pair_set(hi, lo, grp, cell):
    return sorted(zip(hi.tolist(), lo.tolist(), grp.tolist(), cell.tolist()))


def test_pore_three_steps_bit_exact(oracle, pore_cfg, pore_init):
    from argon_monte_carlo_b200 import amc
    from oracle import steps
    st = oracle.ParticleState(*pore_init)
    sim = amc.Simulation(pore_cfg, taps=amc.TAP_PAIRS | amc.TAP_WALL_BITS | amc.TAP_PATHS)
    sim.set_state(*pore_init)
    expected_collisions = (1069, 261, 414)   # printed by the unmodified reference (tests/golden/ref_pore_3steps.json)
    sink = oracle.PathSink()
    for k in range(3):
        pairs = oracle.PairSink()
        r = steps.pore_step(st, pore_cfg, sink, pairs, want_bits=True)
        g = sim.step(1)[0]
        assert g["collisions"] == r["collisions"] == expected_collisions[k]
        assert np.array_equal(g["wall_hits"][:9], r["wall_counts"])
        assert g["pp_collisions"] == r["pp_collisions"]
        assert g["pair_checks_ref"] == r["checks"]
        assert g["oob_after_walls"] == r["oob_after_walls"] and g["oob_after_pp"] == r["oob_after_pp"]
        assert g["errors"] == r["errors"] == 0
        assert np.array_equal(sim.wall_bits(), r["hit_bits"]), "wall-hit flags differ at step %d" % k
        hi, lo, grp, cell = sim.pair_list()
        assert len(hi) == sum(1 for _ in hi)  # tap readable every step
        assert_state_equal(sim.get_state(), st, "pore step %d" % k)
    # pair list over the three steps vs the oracle's (same (hi, lo, group, cell) multiset)
    st2 = oracle.ParticleState(*pore_init)
    allpairs = oracle.PairSink()
    for k in range(3):
        steps.pore_step(st2, pore_cfg, None, allpairs)
    assert pair_set(*sim.pair_list()) == pair_set(*allpairs.arrays())
    # completed free paths: same multiset in all four lists, histograms = np.histogram of them
    got = sim.completed_paths()
    exp = sink.arrays()
    for a, b in zip(got, exp):
        assert np.array_equal(np.sort(a), np.sort(b))
    counts, npaths, sums = sim.histograms()
    assert npaths == len(sink)
    for j in range(4):
        ref_counts, _ = np.histogram(exp[j], bins=200, range=(0, 10 ** -6))
        assert np.array_equal(counts[j].astype(np.int64), ref_counts)
        assert abs(sums[j] - exp[j].sum()) <= 1e-12 * abs(exp[j].sum())
    sim.close()


def test_temp_host_rng_matches_oracle_and_shipped_csv(oracle, temp_cfg):
    """Parity mode: host Mersenne-Twister draws in the reference's order.  Rows 0-1 of the shipped
    momentum_energy.csv must come out digit for digit (15 significant digits, str(mpf))."""
    import os
    import mpmath
    from argon_monte_carlo_b200 import amc, init_state
    from oracle import steps
    init = init_state.pore_initial_state(temp_cfg)           # seeds both generators (Temp:108-109)
    import random
    state_np, state_py = np.random.get_state(), random.getstate()
    st = oracle.ParticleState(*init)
    ref = [steps.temp_step_host_rng(st, temp_cfg) for _ in range(2)]
    np.random.set_state(state_np)
    random.setstate(state_py)
    sim = amc.Simulation(temp_cfg, rng_mode=amc.RNG_HOST)
    sim.set_state(*init)
    rows = open(os.path.join(os.path.dirname(__file__), "golden", "shipped_momentum_energy.csv")).read().split("\n")[1:3]
    for k in range(2):
        g = sim.step_host_rng()
        r = ref[k]
        assert np.array_equal(g["wall_hits"], r["wall_counts"])
        assert g["collisions"] == r["collisions"] == (1402, 563)[k]
        assert g["dpz"] == r["dpz"] and g["e_cold"] == r["e_cold"] and g["e_hot"] == r["e_hot"]
        line = "%d,%s,%s,%s" % (k, mpmath.mpf(g["dpz"]), mpmath.mpf(g["e_cold"]), mpmath.mpf(g["e_hot"]))
        assert line == rows[k]
    assert_state_equal(sim.get_state(), st, "temp host-rng")
    sim.close()


def test_temp_device_rng_bit_exact(oracle, temp_cfg, temp_init):
    """Energized pore with the device RNG, three timesteps against the oracle."""
    from argon_monte_carlo_b200 import amc, config
    from oracle import steps
    cheb = config.gap_energy_chebyshev(temp_cfg, 16)
    st = oracle.ParticleState(*temp_init)
    sim = amc.Simulation(temp_cfg, taps=amc.TAP_WALL_BITS | amc.TAP_PAIRS, seed=17, cheb=cheb)
    sim.set_state(*temp_init)
    allpairs = oracle.PairSink()
    for k in range(3):
        r = steps.temp_step_philox(st, temp_cfg, 17, k, cheb, None, allpairs, want_bits=True)
        g = sim.step(1)[0]
        assert np.array_equal(g["wall_hits"], r["wall_counts"])
        assert g["collisions"] == r["collisions"]
        assert np.array_equal(sim.wall_bits(), r["hit_bits"])
        for key in ("dpz", "e_cold", "e_hot"):
            assert abs(g[key] - r[key]) <= 1e-12 * abs(r[key]), key
        assert g["oob_after_walls"] == r["oob_after_walls"] and g["oob_after_pp"] == r["oob_after_pp"]
        assert_state_equal(sim.get_state(), st, "temp philox step %d" % k)
    assert pair_set(*sim.pair_list()) == pair_set(*allpairs.arrays())
    sim.close()


@pytest.mark.parametrize("sweep", ["events", "handover"])
def test_cube_steps_bit_exact(oracle, cube_cfg, cube_init, sweep, monkeypatch):
    """Open_Air_Cube_MC.py as shipped, serial cell sweep (Cube:232-336).  events: the event-driven sweep
    (k_sweep_detect / k_sweep_events); handover: column lists too small for the gas, so every pass is handed to the
    plain one-CTA walk over all 3,375 cells (k_cube_sweep)."""
    from argon_monte_carlo_b200 import amc
    from oracle import steps
    if sweep == "handover":
        monkeypatch.setenv("AMC_SWEEP_COLCAP", "16")
    st = oracle.ParticleState(*cube_init)
    sim = amc.Simulation(cube_cfg, taps=amc.TAP_PAIRS | amc.TAP_PATHS)
    sim.set_state(*cube_init)
    allpairs, sink = oracle.PairSink(), oracle.PathSink()
    ncol = []
    for k in range(6):
        r = steps.cube_step(st, cube_cfg, sink, allpairs)
        g = sim.step(1)[0]
        assert g["pp_collisions"] == r["pp_collisions"]
        assert np.array_equal(g["wall_hits"][:6], r["wall_counts"])
        assert g["pair_checks_ref"] == r["checks"]
        ncol.append(g["pp_collisions"])
        assert_state_equal(sim.get_state(), st, "cube step %d" % k)
    assert ncol[:6] == [31, 41, 36, 50, 44, 45]   # printed by the unmodified Open_Air_Cube_MC.py (SURVEY F.6)
    assert pair_set(*sim.pair_list()) == pair_set(*allpairs.arrays())
    for a, b in zip(sim.completed_paths(), sink.arrays()):
        assert np.array_equal(np.sort(a), np.sort(b))
    sim.close()


def test_multi_step_call_equals_single_steps(oracle, temp_cfg, temp_init):
    """amc_step(h, 5) fuses the closing recapture of each step into the next step's advect kernel;
    results and per-step counters must equal five amc_step(h, 1) calls and the oracle."""
    from argon_monte_carlo_b200 import amc, config
    from oracle import steps
    cheb = config.gap_energy_chebyshev(temp_cfg, 16)
    a = amc.Simulation(temp_cfg, seed=5, cheb=cheb)
    b = amc.Simulation(temp_cfg, seed=5, cheb=cheb)
    a.set_state(*temp_init)
    b.set_state(*temp_init)
    sa = a.step(5)
    sb = [b.step(1)[0] for _ in range(5)]
    st = oracle.ParticleState(*temp_init)
    so = [steps.temp_step_philox(st, temp_cfg, 5, k, cheb) for k in range(5)]
    for x, y, o in zip(sa, sb, so):
        for k in ("collisions", "oob_after_walls", "oob_after_pp", "oob_after_pp_recapture", "completed_paths", "dpz", "e_cold"):
            assert x[k] == y[k], k
        assert x["collisions"] == o["collisions"] and x["oob_after_pp"] == o["oob_after_pp"]
    ga, gb = a.get_state(), b.get_state()
    for k in KEYS:
        assert np.array_equal(ga[k], gb[k]) and np.array_equal(ga[k], getattr(st, k)), k
    a.close(); b.close()
