"""Surface recording on the device (amc_surface_*): the accumulators must equal the NumPy restatement of the oracle's
hit records bit for bit, recording must not change anything else, it must agree with the per-step wall series, give the
ideal-gas pressure in the cube, survive the 256-step chunk and checkpoint / restore, merge across slab ranks, and the
drivers must write surface.csv without touching their other output files."""
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COUNTERS = ("wall_collisions", "pp_collisions", "pair_checks_ref", "pair_checks_exec", "oob_after_walls", "oob_after_pp",
            "oob_after_walls_recapture", "oob_after_pp_recapture", "errors", "completed_paths", "dpz", "e_cold", "e_hot")
KINDS = {"pore": 1, "temp": 2, "cube": 0}


def assert_raw_equal(a, b):
    assert a[1] == b[1], ("n_steps", a[1], b[1])
    assert np.array_equal(np.asarray(a[2], dtype=np.uint64), np.asarray(b[2], dtype=np.uint64)), ("outside", a[2], b[2])
    bad = np.nonzero(np.any(a[0] != b[0], axis=1))[0]
    assert len(bad) == 0, "%d elements differ (first %d: %s vs %s)" % (len(bad), bad[0], a[0][bad[0]], b[0][bad[0]])


@pytest.mark.parametrize("which", ["pore", "temp", "cube", "temp_host"])
def test_device_raw_equals_restatement_of_oracle_hits(which, oracle, pore_cfg, pore_init, temp_cfg, temp_init, cube_cfg, cube_init):
    import random
    import surface_oracle as SO
    from argon_monte_carlo_b200 import amc, config, init_state
    base = which.split("_")[0]
    cfg, init = {"pore": (pore_cfg, pore_init), "temp": (temp_cfg, temp_init), "cube": (cube_cfg, cube_init)}[base]
    kind = KINDS[base]
    layout = amc.surface_layout_of(cfg, kind, cfg.grid)
    sink = SO.HitSink()
    if which == "temp_host":
        init = init_state.pore_initial_state(cfg)       # seeds both host generators
        state_np, state_py = np.random.get_state(), random.getstate()
        st = oracle.ParticleState(*init)
        SO.temp_step_host_rng(st, cfg, sink)
        np.random.set_state(state_np)
        random.setstate(state_py)
        sim = amc.Simulation(cfg, rng_mode=amc.RNG_HOST)
        sim.set_state(*init)
        sim.surface_enable()
        sim.step_host_rng()
        n_steps = 1
    else:
        cheb = config.gap_energy_chebyshev(cfg, 16) if base == "temp" else None
        st = oracle.ParticleState(*init)
        for k in range(3):
            if base == "pore":
                SO.pore_step(st, cfg, sink)
            elif base == "cube":
                SO.cube_step(st, cfg, sink)
            else:
                SO.temp_step_philox(st, cfg, 17, k, cheb, sink)
        sim = amc.Simulation(cfg, seed=17, cheb=cheb)
        sim.set_state(*init)
        sim.surface_enable()
        sim.step(3)
        n_steps = 3
    assert np.array_equal(sim.surface_layout(), layout.offsets)
    acc, out = amc.surface_moments_of_hits(sink.hits(), layout, None if base == "cube" else cfg.geom)
    raw = sim.surface_raw()
    assert acc[:, 0].sum() > 0
    assert_raw_equal(raw, (acc, n_steps, out))
    sim.close()


@pytest.mark.parametrize("which", ["pore", "temp", "cube"])
def test_recording_does_not_perturb(which, pore_cfg, pore_init, temp_cfg, temp_init, cube_cfg, cube_init):
    from argon_monte_carlo_b200 import amc
    cfg, init = {"pore": (pore_cfg, pore_init), "temp": (temp_cfg, temp_init), "cube": (cube_cfg, cube_init)}[which]
    runs = []
    for surf, sample in ((False, False), (True, False), (True, True)):
        sim = amc.Simulation(cfg, seed=17)
        sim.set_state(*init)
        if surf:
            sim.surface_enable()
        if sample:
            sim.sample_enable(1, 0)
        stats = sim.step(10)
        runs.append((sim.state_digest(), stats, sim.histograms(), sim.surface_raw()[1] if surf else 10))
        sim.close()
    d0, s0, h0, _ = runs[0]
    for d1, s1, h1, n1 in runs[1:]:
        assert d0 == d1 and n1 == 10
        for a, b in zip(s0, s1):
            for k in COUNTERS:
                assert a[k] == b[k], k
            assert np.array_equal(a["wall_hits"], b["wall_hits"])
        assert np.array_equal(h0[0], h1[0]) and h0[1] == h1[1] and np.array_equal(h0[2], h1[2])


def test_consistent_with_the_wall_series(temp_cfg, temp_init):
    """Temp, device RNG, 50 steps: hits + outside = wall_hits per case; sum dE over the cold / hot coated cases = the
    e_cold / e_hot series; m sum dv_z over the energized cases = the dpz series."""
    from argon_monte_carlo_b200 import amc, config, outputs
    cheb = config.gap_energy_chebyshev(temp_cfg, 16)
    sim = amc.Simulation(temp_cfg, seed=17, cheb=cheb)
    sim.set_state(*temp_init)
    sim.surface_enable()
    stats = sim.step(50)
    acc, n_steps, out = sim.surface_raw()
    off = sim.surface_layout()
    sim.close()
    assert n_steps == 50
    wall = np.sum([s["wall_hits"] for s in stats], axis=0)
    hits = np.array([acc[off[c]:off[c + 1], 0].sum() for c in range(amc.NUM_CASES)], dtype=np.int64)
    assert np.array_equal(hits + out.astype(np.int64), wall)
    _, sums = outputs.decode_surface_sums(acc)
    per_case = lambda j: np.array([sums[off[c]:off[c + 1], j].sum() for c in range(amc.NUM_CASES)])
    per_case_abs = lambda j: np.array([np.abs(sums[off[c]:off[c + 1], j]).sum() for c in range(amc.NUM_CASES)])
    dE, dEa = per_case(3), per_case_abs(3)
    e_cold, e_hot = sum(s["e_cold"] for s in stats), sum(s["e_hot"] for s in stats)
    assert abs(dE[[3, 7, 9]].sum() - e_cold) <= 1e-12 * dEa[[3, 7, 9]].sum()
    assert abs(dE[[4, 6, 8]].sum() - e_hot) <= 1e-12 * dEa[[4, 6, 8]].sum()
    # dv_z: planes dv.n = +-dv_z (2A / 3C / 5B: +), cylinders dv.t1 = dv_z
    dvn, dvt1 = per_case(0), per_case(1)
    dvz = sum(dvt1[c] for c in (5, 8, 9)) + sum(dvn[c] if c in (3, 6) else -dvn[c] for c in (3, 4, 6, 7))
    scale = sum(per_case_abs(1)[c] for c in (5, 8, 9)) + sum(per_case_abs(0)[c] for c in (3, 4, 6, 7))
    dpz = sum(s["dpz"] for s in stats)
    m = temp_cfg.argon_mass
    assert abs(m * dvz - dpz) <= 1e-12 * m * scale


def test_cube_pressure_is_the_ideal_gas_pressure(cube_cfg, cube_init):
    from argon_monte_carlo_b200 import amc, outputs
    sim = amc.Simulation(cube_cfg)
    sim.set_state(*cube_init)
    sim.surface_enable()
    sim.step(200)
    raw = sim.surface_raw()
    st = sim.get_state()
    sim.close()
    n = len(cube_init[0]) / (cube_cfg.cube_x * cube_cfg.cube_y * cube_cfg.cube_z)
    v2 = np.mean(st["vx"] ** 2 + st["vy"] ** 2 + st["vz"] ** 2)
    T = cube_cfg.argon_mass * v2 / (3 * cube_cfg.boltzman)
    p_ideal = n * cube_cfg.boltzman * T
    f = outputs.surface_fields(raw, cube_cfg, cube_cfg.grid, amc.KIND_CUBE)
    for c in range(6):
        m = f["case"] == c
        p = np.sum(f["pressure"][m] * f["area"][m]) / np.sum(f["area"][m])
        assert abs(p / p_ideal - 1) < 0.03, (c, p, p_ideal)


def test_long_call_equals_single_steps_and_checkpoint(pore_cfg, pore_init, tmp_path):
    from argon_monte_carlo_b200 import amc
    one = amc.Simulation(pore_cfg)
    one.set_state(*pore_init)
    one.surface_enable()
    one.step(300)
    ref = one.surface_raw()
    digest = one.state_digest()
    one.close()
    assert ref[1] == 300
    single = amc.Simulation(pore_cfg)
    single.set_state(*pore_init)
    single.surface_enable()
    for _ in range(300):
        single.step(1)
    assert_raw_equal(ref, single.surface_raw())
    assert single.state_digest() == digest
    single.close()
    first = amc.Simulation(pore_cfg)
    first.set_state(*pore_init)
    first.surface_enable()
    first.step(151)
    path = str(tmp_path / "ck.npz")
    first.checkpoint(path)
    first.close()
    second = amc.Simulation(pore_cfg)
    second.restore(path)
    assert second.surface_on
    second.step(149)
    assert_raw_equal(ref, second.surface_raw())
    assert second.state_digest() == digest
    second.close()
    old = amc.Simulation(pore_cfg)          # a checkpoint without recording restores without it
    old.set_state(*pore_init)
    ck = old.checkpoint()
    assert not any(k.startswith("surface_") for k in ck)
    old.restore(ck)
    assert not old.surface_on
    old.close()


def test_slabs_merge_to_the_single_domain_raw():
    """The dense small energized pore, emulated 2, 3 and 4 ranks on one GPU (1-layer slabs included) and a 1-rank
    amc_slab_step run: the merged accumulators equal the single-domain ones bit for bit."""
    from argon_monte_carlo_b200 import amc, config, init_state, slab
    cfg = config.pore_config(True, scale=0.5)
    init = init_state.synthetic_pore_state(cfg, seed=11)
    nz = cfg.grid.nc[2]
    one = amc.Simulation(cfg, seed=17)
    one.set_state(*init)
    one.surface_enable()
    one.step(6)
    ref = one.surface_raw()
    digest = one.state_digest()
    one.close()
    assert ref[0][:, 0].sum() > 0
    for nranks, cuts in ((2, None), (3, [0, 1, nz - 2, nz]), (4, [0, 1, 2, nz - 1, nz])):
        sim = slab.SlabSimulation(cfg, nranks, init[2], cuts=cuts, seed=17)
        sim.set_state(*init)
        sim.surface_enable()
        sim.step(6)
        assert sim.state_digest() == digest
        assert_raw_equal(ref, sim.surface_raw())
        sim.close()
    fused = slab.SlabSimulation(cfg, 1, init[2], seed=17, p2p=True)
    fused.set_state(*init)
    fused.surface_enable()
    fused.step_fused(4)
    fused.step_fused(2)
    assert fused.state_digest() == digest
    assert_raw_equal(ref, fused.surface_raw())
    fused.close()


def _md5(path):
    return hashlib.md5(open(path, "rb").read()).hexdigest()


@pytest.mark.parametrize("script", ["Temperature_Pore_MC.py", "Open_Air_Cube_MC.py"])
def test_driver_writes_surface_and_leaves_other_outputs_alone(tmp_path, script):
    outs = {}
    for tag, extra in (("plain", []), ("surface", ["--surface-start", "5"])):
        d = tmp_path / tag
        d.mkdir()
        r = subprocess.run([sys.executable, os.path.join(ROOT, "drivers", script), "--steps", "20", *extra],
                           cwd=str(d), capture_output=True, text=True, timeout=1500)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        outs[tag] = d
    plain = sorted(os.listdir(outs["plain"]))
    assert sorted(os.listdir(outs["surface"])) == sorted(plain + ["surface.csv"])
    for f in plain:
        assert _md5(outs["plain"] / f) == _md5(outs["surface"] / f), f
    rows = (outs["surface"] / "surface.csv").read_text().splitlines()
    assert len(rows) > 1 and all(len(r.split(",")) == 13 for r in rows)
    assert sum(int(r.split(",")[7]) for r in rows[1:]) > 0


@pytest.mark.parametrize("mode", ["p2p", "nccl"])
def test_multi_gpu_surface_matches_single_gpu(tmp_path, mode):
    """One process per GPU (torch.distributed.run): the accumulators summed over the ranks equal rank 0's
    single-domain run (tests/nccl_surface_worker.py).  Needs >= 2 GPUs."""
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
    out = tmp_path / "surface.json"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(min(ngpu, 4)), "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "nccl_surface_worker.py"), str(out),
           "--mode", mode, "--steps", "6"]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    res = json.loads(out.read_text())
    assert res["ok"] and res["n_steps"] == 6 and res["hits"] > 0
