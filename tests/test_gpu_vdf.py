"""Velocity distribution on the device (amc_vdf_*): the histograms must equal the NumPy restatement of the sampled
states word for word (after device-RNG steps, a host-RNG step, and states with velocities on the bin edges), the VDF
must change nothing else, follow the field sample's schedule across the 256-step chunk and checkpoint / restore, merge
over slab ranks to the single-domain words, reject bad arguments, show a Maxwellian in an equilibrium cube, and the
drivers must add vdf_z.csv without touching their other output files."""
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BINS, VMAX = 200, 1650.0
AMC_E_INVALID, AMC_E_STATE = -1, -5         # include/amc.h
COUNTERS = ("wall_collisions", "pp_collisions", "pair_checks_ref", "pair_checks_exec", "oob_after_walls", "oob_after_pp",
            "oob_after_walls_recapture", "oob_after_pp_recapture", "errors", "completed_paths", "dpz", "e_cold", "e_hot")


def assert_words_equal(a, b):
    assert a.shape == b.shape, (a.shape, b.shape)
    bad = np.argwhere(a != b)
    assert len(bad) == 0, "%d words differ (first %s: %s vs %s)" % (len(bad), bad[0], a[tuple(bad[0])], b[tuple(bad[0])])


def restate(sim, n_bins=BINS, v_max=VMAX):
    from argon_monte_carlo_b200 import amc
    return amc.vdf_of_arrays(sim.get_state(), sim.sample_grid, n_bins, v_max)


def _case(which, pore_cfg, pore_init, temp_cfg, temp_init, cube_cfg, cube_init):
    return {"pore": (pore_cfg, pore_init), "temp": (temp_cfg, temp_init), "cube": (cube_cfg, cube_init)}[which]


@pytest.mark.parametrize("which", ["pore", "temp", "cube"])
def test_device_words_equal_restatement(which, pore_cfg, pore_init, temp_cfg, temp_init, cube_cfg, cube_init):
    from argon_monte_carlo_b200 import amc
    cfg, init = _case(which, pore_cfg, pore_init, temp_cfg, temp_init, cube_cfg, cube_init)
    sim = amc.Simulation(cfg, seed=17)
    sim.set_state(*init)
    sim.sample_enable()
    sim.vdf_enable(BINS, VMAX)
    assert sim.vdf_layout() == (cfg.grid.nc[2], BINS, VMAX)
    sim.step(3)
    sim.sample_now()
    vdf = sim.vdf_raw()
    assert_words_equal(vdf, restate(sim))
    nx, ny, nz = cfg.grid.nc
    per_layer = sim.sample_raw()[0][:, 0].reshape(nx * ny, nz).sum(axis=0)
    for j in range(amc.VDF_HISTS):
        assert np.array_equal(vdf[:, j].sum(axis=1), per_layer)
    assert sim.last_sample_ms() > 0
    sim.vdf_enable(BINS, VMAX)          # re-enabling starts from zero
    assert not sim.vdf_raw().any()
    sim.close()


def test_host_rng_step_follows_the_schedule(temp_cfg, temp_init):
    from argon_monte_carlo_b200 import amc
    sim = amc.Simulation(temp_cfg, rng_mode=amc.RNG_HOST)
    sim.set_state(*temp_init)
    sim.sample_enable(2, 1)
    sim.vdf_enable(BINS, VMAX)
    sim.step_host_rng()                 # step 0: not sampled
    assert not sim.vdf_raw().any()
    sim.step_host_rng()                 # step 1: sampled (amc_sample_now)
    assert_words_equal(sim.vdf_raw(), restate(sim))
    sim.close()


@pytest.mark.parametrize("n_bins,v_max", [(BINS, VMAX), (7, 3.0), (1, 1.0), (3000, 500.0)])
def test_velocities_on_bin_edges(n_bins, v_max, pore_cfg, pore_init):
    """A state whose velocities sit on the bin edges, one ulp either side, on +-v_max, far beyond and at NaN."""
    from argon_monte_carlo_b200 import amc
    ec, es = amc.vdf_edges(n_bins, v_max)
    pool = np.concatenate([ec, np.nextafter(ec, -np.inf), np.nextafter(ec, np.inf), es, np.nextafter(es, np.inf),
                           [0.0, -0.0, v_max, -v_max, 1e300, -1e300, 10 * v_max, np.inf, -np.inf, np.nan]])
    n = len(pore_init[0])
    rng = np.random.default_rng(3)
    state = list(pore_init)
    for a in (3, 4, 5):
        v = rng.choice(pool, n)
        v[rng.random(n) < 0.5] = 0.0        # vx = edge, vy = vz = 0 puts speeds on the speed edges
        state[a] = v
    sim = amc.Simulation(pore_cfg, seed=17)
    sim.set_state(*state)
    sim.sample_enable()
    sim.vdf_enable(n_bins, v_max)
    sim.sample_now()
    assert_words_equal(sim.vdf_raw(), restate(sim, n_bins, v_max))
    sim.close()


@pytest.mark.parametrize("which", ["pore", "temp", "cube"])
def test_vdf_does_not_perturb(which, pore_cfg, pore_init, temp_cfg, temp_init, cube_cfg, cube_init):
    from argon_monte_carlo_b200 import amc
    cfg, init = _case(which, pore_cfg, pore_init, temp_cfg, temp_init, cube_cfg, cube_init)
    runs = []
    for vdf in (False, True):
        sim = amc.Simulation(cfg, seed=17)
        sim.set_state(*init)
        sim.sample_enable(2, 0)
        if vdf:
            sim.vdf_enable(BINS, VMAX)
        stats = sim.step(10)
        runs.append((sim.state_digest(), stats, sim.histograms(), sim.sample_raw(), sim.lib.amc_get_step_index(sim.h)))
        sim.close()
    (d0, s0, h0, r0, i0), (d1, s1, h1, r1, i1) = runs
    assert d0 == d1 and i0 == i1
    for a, b in zip(s0, s1):
        for k in COUNTERS:
            assert a[k] == b[k], k
        assert np.array_equal(a["wall_hits"], b["wall_hits"])
    assert np.array_equal(h0[0], h1[0]) and h0[1] == h1[1] and np.array_equal(h0[2], h1[2])
    assert np.array_equal(r0[0], r1[0]) and r0[1:] == r1[1:]


def test_schedule_across_chunks_and_checkpoint(pore_cfg, pore_init, tmp_path):
    """every=3 from step 2 over 300 steps: one amc_step call (crosses the 256-step chunk) = explicit sample_now after
    each due step(1) = a run split by checkpoint / restore at an unsampled step (150) into a fresh handle."""
    from argon_monte_carlo_b200 import amc
    one = amc.Simulation(pore_cfg)
    one.set_state(*pore_init)
    one.sample_enable(3, 2)
    one.vdf_enable(BINS, VMAX)
    one.step(300)
    ref = one.vdf_raw()
    digest = one.state_digest()
    one.close()

    single = amc.Simulation(pore_cfg)
    single.set_state(*pore_init)
    single.sample_enable(0, 0)
    single.vdf_enable(BINS, VMAX)
    acc = np.zeros_like(ref)
    for s in range(300):
        single.step(1)
        if s >= 2 and (s - 2) % 3 == 0:
            acc += restate(single)
            single.sample_now()
    assert_words_equal(ref, single.vdf_raw())
    assert_words_equal(ref, acc)
    assert single.state_digest() == digest
    single.close()

    first = amc.Simulation(pore_cfg)
    first.set_state(*pore_init)
    first.sample_enable(3, 2)
    first.vdf_enable(BINS, VMAX)
    first.step(151)                     # last step taken: 150, (150 - 2) % 3 != 0
    path = str(tmp_path / "ck.npz")
    first.checkpoint(path)
    first.close()
    second = amc.Simulation(pore_cfg)
    second.restore(path)
    assert second.vdf == (BINS, VMAX)
    second.step(149)
    assert_words_equal(ref, second.vdf_raw())
    assert second.state_digest() == digest
    second.close()


def test_checkpoint_without_vdf_restores_without_it(pore_cfg, pore_init):
    from argon_monte_carlo_b200 import amc
    sim = amc.Simulation(pore_cfg)
    sim.set_state(*pore_init)
    sim.sample_enable(2, 0)
    ck = sim.checkpoint()
    assert not any(k.startswith("vdf_") for k in ck)
    sim.close()
    again = amc.Simulation(pore_cfg)
    again.restore(ck)
    assert again.vdf is None and again.sampling == (2, 0)
    again.close()


def test_slabs_merge_to_the_single_domain_words():
    """The dense small pore with cuts inside the end caps, 1-layer slabs included: the merged histograms of 2, 3 and
    4 emulated ranks (LocalTransport, one GPU) and of a 1-rank amc_slab_step run equal the single-domain ones."""
    from argon_monte_carlo_b200 import amc, config, init_state, slab
    cfg = config.pore_config(False, scale=0.5)
    init = init_state.synthetic_pore_state(cfg, seed=11)
    nz = cfg.grid.nc[2]
    one = amc.Simulation(cfg, seed=17)
    one.set_state(*init)
    one.sample_enable(2, 1)
    one.vdf_enable(BINS, VMAX)
    one.step(6)
    ref = one.vdf_raw()
    digest = one.state_digest()
    one.close()
    assert ref.sum() > 0
    for nranks, cuts in ((2, [0, nz // 2, nz]), (3, [0, 1, nz - 2, nz]), (4, [0, 1, 2, nz - 1, nz])):
        sim = slab.SlabSimulation(cfg, nranks, init[2], cuts=cuts, seed=17)
        sim.set_state(*init)
        sim.sample_enable(2, 1)
        sim.vdf_enable(BINS, VMAX)
        sim.step(6)
        assert sim.state_digest() == digest
        assert_words_equal(ref, sim.vdf_raw())
        sim.close()
    fused = slab.SlabSimulation(cfg, 1, init[2], seed=17, p2p=True)
    fused.set_state(*init)
    fused.sample_enable(2, 1)
    fused.vdf_enable(BINS, VMAX)
    fused.step_fused(4)
    fused.step_fused(2)
    assert fused.state_digest() == digest
    assert_words_equal(ref, fused.vdf_raw())
    fused.close()


def test_error_paths(pore_cfg, pore_init):
    from argon_monte_carlo_b200 import amc
    sim = amc.Simulation(pore_cfg)
    sim.set_state(*pore_init)
    L = sim.lib
    assert L.amc_vdf_enable(sim.h, amc.C.c_int32(10), amc.C.c_double(1000.0)) == AMC_E_STATE
    sim.sample_enable()
    for nb, vm in ((0, 1000.0), (4097, 1000.0), (-1, 1000.0), (10, 0.0), (10, -5.0), (10, float("nan")),
                   (10, float("inf"))):
        assert L.amc_vdf_enable(sim.h, amc.C.c_int32(nb), amc.C.c_double(vm)) == AMC_E_INVALID, (nb, vm)
    assert L.amc_vdf_layout(sim.h, None, None, None) == AMC_E_STATE
    sim.vdf_enable(amc.VDF_MAX_BINS, 1000.0)
    assert sim.vdf_layout()[1] == amc.VDF_MAX_BINS
    sim.sample_disable()                # frees the VDF too
    assert sim.vdf is None
    assert L.amc_vdf_layout(sim.h, None, None, None) == AMC_E_STATE
    sim.close()


def test_equilibrium_cube_is_maxwellian(cube_cfg, cube_init):
    """A 298 K cube over 200 steps, sampled every 10th: the vx, vy, vz histograms summed over the layers against the
    Maxwellian at the sampled temperature and zero drift.  The 20 samples hold the same particles, so the counts are
    divided by the number of samples before the chi-square; the bound is chi2 / dof < 1 + 6 sqrt(2 / dof)."""
    from argon_monte_carlo_b200 import amc, outputs
    sim = amc.Simulation(cube_cfg, seed=17)
    sim.set_state(*cube_init)
    sim.sample_enable(10, 9)
    sigma0 = np.sqrt(cube_cfg.boltzman * 298.0 / cube_cfg.argon_mass)
    n_bins, v_max = 60, 5 * sigma0
    sim.vdf_enable(n_bins, v_max)
    sim.step(200)
    raw, (acc, ns, _) = sim.vdf_raw(), sim.sample_raw()
    sim.close()
    assert ns == 20
    count, sv, sq = outputs.decode_sample_sums(acc)
    n = count.sum()
    t = cube_cfg.argon_mass / cube_cfg.boltzman * (sq.sum(axis=0) / n - (sv.sum(axis=0) / n) ** 2).mean()
    assert abs(t / 298.0 - 1) < 0.03
    sigma = np.sqrt(cube_cfg.boltzman * t / cube_cfg.argon_mass)
    ec, _ = amc.vdf_edges(n_bins, v_max)
    expect = np.diff(outputs.maxwell_component_cdf(ec, 0.0, sigma)) * (n / ns)
    for j in range(3):
        obs = raw[:, j, 1:-1].sum(axis=0).astype(float) / ns
        m = expect >= 5
        chi2, dof = float(np.sum((obs[m] - expect[m]) ** 2 / expect[m])), int(m.sum()) - 1
        assert chi2 / dof < 1 + 6 * np.sqrt(2.0 / dof), (j, chi2, dof)


def _md5(path):
    return hashlib.md5(open(path, "rb").read()).hexdigest()


def test_driver_writes_vdf_and_leaves_other_outputs_alone(tmp_path, pore_cfg):
    outs = {}
    for tag, extra in (("plain", ["--sample-every", "5"]), ("vdf", ["--sample-every", "5", "--vdf-bins", "50"])):
        d = tmp_path / tag
        d.mkdir()
        r = subprocess.run([sys.executable, os.path.join(ROOT, "drivers", "Open_Air_Pore_MC.py"), "--steps", "10", *extra],
                           cwd=str(d), capture_output=True, text=True, timeout=1500)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        outs[tag] = d
    plain = sorted(os.listdir(outs["plain"]))
    assert sorted(os.listdir(outs["vdf"])) == sorted(plain + ["vdf_z.csv"])
    for f in plain:
        assert _md5(outs["plain"] / f) == _md5(outs["vdf"] / f), f
    rows = (outs["vdf"] / "vdf_z.csv").read_text().splitlines()
    assert len(rows) == 1 + pore_cfg.grid.nc[2] * 4 * 50
    l1 = np.array([float(r.split(",")[11]) for r in rows[1:]])
    assert np.nanmedian(l1) < 0.5


def test_multi_gpu_vdf_matches_single_gpu(tmp_path):
    """One process per GPU (torch.distributed.run, amc_slab_step): the histograms summed over the ranks equal rank 0's
    single-domain run (tests/nccl_vdf_worker.py).  Needs >= 2 GPUs."""
    import json
    import socket
    import torch
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("needs >= 2 GPUs (found %d)" % ngpu)
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = tmp_path / "vdf.json"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(min(ngpu, 4)), "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "nccl_vdf_worker.py"), str(out), "--steps", "6"]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    res = json.loads(out.read_text())
    assert res["ok"] and res["samples"] == 3
