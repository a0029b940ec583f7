"""Plane flux recording on the device (amc_flux_*): the words must equal the NumPy restatement of the sequence of states
word for word (device-RNG steps of Pore, Temp and Cube one at a time and in one call, a host-RNG step), conserve
particles exactly across the 256-step chunk, change nothing else, resume exactly from a checkpoint, refuse slab
handles, show the kinetic-theory crossing rate and the ideal-gas momentum flux in an equilibrium cube, and the
drivers must add flux_z.csv without touching their other output files."""
import hashlib
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
AMC_E_INVALID, AMC_E_STATE = -1, -5         # include/amc.h
COUNTERS = ("wall_collisions", "pp_collisions", "pair_checks_ref", "pair_checks_exec", "oob_after_walls", "oob_after_pp",
            "oob_after_walls_recapture", "oob_after_pp_recapture", "errors", "completed_paths", "dpz", "e_cold", "e_hot")


def assert_words_equal(a, b):
    assert a.shape == b.shape, (a.shape, b.shape)
    bad = np.argwhere(a != b)
    assert len(bad) == 0, "%d words differ (first %s: %s vs %s)" % (len(bad), bad[0], a[tuple(bad[0])], b[tuple(bad[0])])


def _case(which, pore_cfg, pore_init, temp_cfg, temp_init, cube_cfg, cube_init):
    return {"pore": (pore_cfg, pore_init), "temp": (temp_cfg, temp_init), "cube": (cube_cfg, cube_init)}[which]


def _edges(cfg):
    return np.asarray(cfg.grid.edge[2], dtype=np.float64)


@pytest.mark.parametrize("which", ["pore", "temp", "cube"])
def test_device_words_equal_restatement(which, pore_cfg, pore_init, temp_cfg, temp_init, cube_cfg, cube_init):
    """5 steps one at a time with get_state between them: the words equal flux_of_states over the sequence; the same
    run as one step(5) call gives the same words."""
    from argon_monte_carlo_b200 import amc
    cfg, init = _case(which, pore_cfg, pore_init, temp_cfg, temp_init, cube_cfg, cube_init)
    e = _edges(cfg)
    sim = amc.Simulation(cfg, seed=17)
    sim.set_state(*init)
    sim.flux_enable()
    assert sim.flux_layout() == cfg.grid.nc[2] + 1
    prev = sim.get_state()
    ref = np.zeros((len(e), amc.FLUX_WORDS), dtype=np.uint64)
    for _ in range(5):
        sim.step(1)
        cur = sim.get_state()
        with np.errstate(over="ignore"):
            ref += amc.flux_of_states(prev, cur, e)
        prev = cur
    acc, ns = sim.flux_raw()
    assert ns == 5
    assert ref[:, :2].sum() > 0
    assert_words_equal(acc, ref)
    digest = sim.state_digest()
    sim.flux_enable()                   # re-enabling starts from zero
    assert not sim.flux_raw()[0].any() and sim.flux_raw()[1] == 0
    sim.close()
    one = amc.Simulation(cfg, seed=17)
    one.set_state(*init)
    one.flux_enable()
    one.step(5)
    acc1, ns1 = one.flux_raw()
    assert ns1 == 5 and one.state_digest() == digest
    assert_words_equal(acc1, ref)
    one.close()


def test_host_rng_step_and_flux_now(temp_cfg, temp_init):
    from argon_monte_carlo_b200 import amc
    e = _edges(temp_cfg)
    sim = amc.Simulation(temp_cfg, rng_mode=amc.RNG_HOST)
    sim.set_state(*temp_init)
    sim.flux_enable()
    prev = sim.get_state()
    ref = np.zeros((len(e), amc.FLUX_WORDS), dtype=np.uint64)
    for _ in range(2):
        sim.step_host_rng()             # calls flux_now after the timestep
        cur = sim.get_state()
        with np.errstate(over="ignore"):
            ref += amc.flux_of_states(prev, cur, e)
        prev = cur
    acc, ns = sim.flux_raw()
    assert ns == 2 and ref[:, :2].sum() > 0
    assert_words_equal(acc, ref)
    sim.close()


def test_conservation_is_exact_across_the_chunk(temp_cfg, temp_init):
    """Energized pore, 300 steps in one call: for every plane, up - down equals the particles at or above it at the end
    minus those at the start."""
    from argon_monte_carlo_b200 import amc
    e = _edges(temp_cfg)
    sim = amc.Simulation(temp_cfg, seed=17)
    sim.set_state(*temp_init)
    sim.flux_enable()
    z0 = sim.get_state()["z"]
    sim.step(300)
    acc, ns = sim.flux_raw()
    z1 = sim.get_state()["z"]
    sim.close()
    assert ns == 300
    net = acc[:, 0].astype(np.int64) - acc[:, 1].astype(np.int64)
    above = lambda z: np.array([np.count_nonzero(amc.flux_counts_of(z, e) > k) for k in range(len(e))])
    assert np.array_equal(net, above(z1) - above(z0))
    assert acc[1:-1, 0].min() > 0       # every interior plane is crossed


@pytest.mark.parametrize("which", ["pore", "temp", "cube"])
def test_recording_does_not_perturb(which, pore_cfg, pore_init, temp_cfg, temp_init, cube_cfg, cube_init):
    from argon_monte_carlo_b200 import amc
    cfg, init = _case(which, pore_cfg, pore_init, temp_cfg, temp_init, cube_cfg, cube_init)
    runs = []
    for flux in (False, True):
        sim = amc.Simulation(cfg, seed=17)
        sim.set_state(*init)
        sim.sample_enable(2, 0)
        sim.vdf_enable(50, 1500.0)
        sim.surface_enable()
        if flux:
            sim.flux_enable()
        stats = sim.step(10)
        runs.append((sim.state_digest(), stats, sim.histograms(), sim.sample_raw(), sim.vdf_raw(), sim.surface_raw(),
                     sim.lib.amc_get_step_index(sim.h)))
        sim.close()
    (d0, s0, h0, r0, v0, f0, i0), (d1, s1, h1, r1, v1, f1, i1) = runs
    assert d0 == d1 and i0 == i1
    for a, b in zip(s0, s1):
        for k in COUNTERS:
            assert a[k] == b[k], k
        assert np.array_equal(a["wall_hits"], b["wall_hits"])
    assert np.array_equal(h0[0], h1[0]) and h0[1] == h1[1] and np.array_equal(h0[2], h1[2])
    assert np.array_equal(r0[0], r1[0]) and r0[1:] == r1[1:]
    assert np.array_equal(v0, v1)
    assert np.array_equal(f0[0], f1[0]) and f0[1] == f1[1] and np.array_equal(f0[2], f1[2])


def test_checkpoint_resumes_exactly(pore_cfg, pore_init, tmp_path):
    from argon_monte_carlo_b200 import amc
    one = amc.Simulation(pore_cfg)
    one.set_state(*pore_init)
    one.flux_enable()
    one.step(40)
    ref, ns = one.flux_raw()
    digest = one.state_digest()
    one.close()
    first = amc.Simulation(pore_cfg)
    first.set_state(*pore_init)
    first.flux_enable()
    first.step(20)
    path = str(tmp_path / "ck.npz")
    first.checkpoint(path)
    first.close()
    second = amc.Simulation(pore_cfg)
    second.restore(path)
    assert second.flux_on
    second.step(20)
    acc, ns2 = second.flux_raw()
    assert ns2 == ns == 40 and second.state_digest() == digest
    assert_words_equal(acc, ref)
    second.close()
    plain = amc.Simulation(pore_cfg)
    plain.set_state(*pore_init)
    ck = plain.checkpoint()
    assert not any(k.startswith("flux_") for k in ck)
    plain.close()


def test_set_state_retakes_the_snapshot(pore_cfg, pore_init):
    """A new state replaces the snapshot: a record point right after set_state counts nothing."""
    from argon_monte_carlo_b200 import amc
    sim = amc.Simulation(pore_cfg)
    sim.set_state(*pore_init)
    sim.flux_enable()
    st = list(pore_init)
    st[2] = np.asarray(st[2]) + 3 * (pore_cfg.grid.edge[2][1] - pore_cfg.grid.edge[2][0])
    sim.set_state(*st)
    sim.flux_now()
    acc, ns = sim.flux_raw()
    assert ns == 1 and not acc.any()
    sim.close()


def test_error_paths(pore_cfg, pore_init):
    from argon_monte_carlo_b200 import amc, config, init_state, slab
    sim = amc.Simulation(pore_cfg)
    sim.set_state(*pore_init)
    L = sim.lib
    assert L.amc_flux_now(sim.h) == AMC_E_STATE
    assert L.amc_flux_layout(sim.h, None) == AMC_E_STATE
    sim.flux_enable()
    with pytest.raises(amc.AmcError):
        sim.flux_set_raw(np.zeros((sim.flux_layout() + 1, amc.FLUX_WORDS), dtype=np.uint64), 0)
    # amc_slab_enable while recording is on
    holder = SimpleNamespace(nranks=1)
    nz = pore_cfg.grid.nc[2]
    c = slab.SlabRank._slab_config(holder, pore_cfg.grid, [0, nz], 0, 1024, 512, 1024)
    assert L.amc_slab_enable(sim.h, amc.C.byref(c)) == AMC_E_STATE
    ids = np.arange(sim.n, dtype=np.int64)
    assert L.amc_set_ids(sim.h, ids.ctypes.data_as(amc.c_int64_p)) == AMC_E_STATE
    sim.step(3)
    assert sim.flux_raw()[0].any()
    sim.flux_disable()
    assert L.amc_flux_get_raw(sim.h, None, None) == AMC_E_STATE
    sim.flux_enable()                   # disable then enable: zeros
    acc, ns = sim.flux_raw()
    assert ns == 0 and not acc.any()
    sim.close()
    # ids other than 0 .. n-1 (a single-domain handle given ids of a larger job)
    odd = amc.Simulation(pore_cfg)
    odd.set_state(*pore_init)
    ids = np.arange(odd.n, dtype=np.int64) * 2
    odd._check(odd.lib.amc_set_ids(odd.h, ids.ctypes.data_as(amc.c_int64_p)), "amc_set_ids")
    assert odd.lib.amc_flux_enable(odd.h) == AMC_E_INVALID
    assert odd.lib.amc_flux_now(odd.h) == AMC_E_STATE
    odd.close()
    # amc_flux_enable on a slab handle
    cfg = config.pore_config(False, scale=0.5)
    init = init_state.synthetic_pore_state(cfg, seed=11)
    fused = slab.SlabSimulation(cfg, 1, init[2], seed=17, p2p=True)
    r = fused.ranks[0].sim
    assert r.lib.amc_flux_enable(r.h) == AMC_E_STATE
    fused.close()


def test_equilibrium_cube_rates_and_momentum_flux(cube_cfg, cube_init):
    """A 298 K cube over 200 steps, interior planes: the upward crossing rate is n sqrt(k T / (2 pi m)) A, P_zz is
    n k T (both within 3 %), and the net particle flux is within 5 sigma of zero."""
    from argon_monte_carlo_b200 import amc, outputs
    sim = amc.Simulation(cube_cfg, seed=17)
    sim.set_state(*cube_init)
    sim.flux_enable()
    sim.step(200)
    raw = sim.flux_raw()
    st = sim.get_state()
    sim.close()
    assert raw[1] == 200
    n = len(cube_init[0]) / (cube_cfg.cube_x * cube_cfg.cube_y * cube_cfg.cube_z)
    m, kb = cube_cfg.argon_mass, cube_cfg.boltzman
    T = m * np.mean(st["vx"] ** 2 + st["vy"] ** 2 + st["vz"] ** 2) / (3 * kb)
    f = outputs.flux_fields(raw, cube_cfg, cube_cfg.grid, amc.KIND_CUBE)
    inner = slice(1, len(f["z"]) - 1)
    rate = n * np.sqrt(kb * T / (2 * np.pi * m)) * f["area"][inner]
    assert np.all(np.abs(f["up_rate"][inner] / rate - 1) < 0.03), f["up_rate"][inner] / rate
    assert np.all(np.abs(f["p_zz"][inner] / (n * kb * T) - 1) < 0.03), f["p_zz"][inner] / (n * kb * T)
    t = raw[1] * cube_cfg.dt
    sigma = np.sqrt(f["up"][inner].astype(float) + f["down"][inner].astype(float)) / (f["area"][inner] * t)
    assert np.all(np.abs(f["particle_flux"][inner]) < 5 * sigma)


def _md5(path):
    return hashlib.md5(open(path, "rb").read()).hexdigest()


@pytest.mark.parametrize("script,extra", [("Temperature_Pore_MC.py", ["--rng", "device"]), ("Open_Air_Cube_MC.py", [])])
def test_driver_writes_flux_and_leaves_other_outputs_alone(tmp_path, script, extra, temp_cfg, cube_cfg):
    outs = {}
    for tag, flag in (("plain", []), ("flux", ["--flux-start", "5"])):
        d = tmp_path / tag
        d.mkdir()
        r = subprocess.run([sys.executable, os.path.join(ROOT, "drivers", script), "--steps", "20", *extra, *flag],
                           cwd=str(d), capture_output=True, text=True, timeout=1500)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        outs[tag] = d
    plain = sorted(os.listdir(outs["plain"]))
    assert sorted(os.listdir(outs["flux"])) == sorted(plain + ["flux_z.csv"])
    for f in plain:
        assert _md5(outs["plain"] / f) == _md5(outs["flux"] / f), f
    cfg = temp_cfg if script.startswith("Temperature") else cube_cfg
    rows = (outs["flux"] / "flux_z.csv").read_text().splitlines()
    assert len(rows) == 1 + cfg.grid.nc[2] + 1
    up = np.array([int(r.split(",")[3]) for r in rows[1:]])
    assert up.sum() > 0
