"""Field sampling on the device (amc_sample_*): the accumulators must equal the NumPy restatement of the state they
sampled bit for bit, sampling must not change anything else, the schedule inside amc_step must equal explicit samples
between single steps and survive checkpoint / restore, slab runs must merge to the single-domain accumulators, and
the drivers must write profile_z.csv without touching their other output files."""
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


def assert_raw_equal(a, b):
    assert a[1] == b[1], ("samples", a[1], b[1])
    assert a[2] == b[2], ("outside", a[2], b[2])
    bad = np.nonzero(np.any(a[0] != b[0], axis=1))[0]
    assert len(bad) == 0, "%d cells differ (first %d: %s vs %s)" % (len(bad), bad[0], a[0][bad[0]], b[0][bad[0]])


def restate(sim):
    from argon_monte_carlo_b200 import amc
    return amc.sample_moments_of_arrays(sim.get_state(), sim.sample_grid)


@pytest.mark.parametrize("which", ["pore", "temp", "cube"])
def test_device_raw_equals_restatement(which, pore_cfg, pore_init, temp_cfg, temp_init, cube_cfg, cube_init):
    from argon_monte_carlo_b200 import amc
    cfg, init = {"pore": (pore_cfg, pore_init), "temp": (temp_cfg, temp_init), "cube": (cube_cfg, cube_init)}[which]
    sim = amc.Simulation(cfg, seed=17)
    sim.set_state(*init)
    sim.sample_enable()
    sim.sample_now()
    assert_raw_equal(sim.sample_raw(), restate(sim))
    sim.step(3)
    sim.sample_enable()                 # zeroes the accumulators
    sim.sample_now()
    raw = sim.sample_raw()
    assert raw[0][:, 0].sum() + raw[2] == len(init[0])
    assert_raw_equal(raw, restate(sim))
    assert sim.last_sample_ms() > 0
    sim.close()


def test_host_rng_steps_follow_the_schedule(temp_cfg, temp_init):
    from argon_monte_carlo_b200 import amc
    sim = amc.Simulation(temp_cfg, rng_mode=amc.RNG_HOST)
    sim.set_state(*temp_init)
    sim.sample_enable(2, 1)
    sim.step_host_rng()                 # step 0: not sampled
    assert sim.sample_raw()[1] == 0
    sim.step_host_rng()                 # step 1: sampled
    assert_raw_equal(sim.sample_raw(), restate(sim))
    sim.close()


@pytest.mark.parametrize("which", ["pore", "temp", "cube"])
def test_sampling_does_not_perturb(which, pore_cfg, pore_init, temp_cfg, temp_init, cube_cfg, cube_init):
    from argon_monte_carlo_b200 import amc
    cfg, init = {"pore": (pore_cfg, pore_init), "temp": (temp_cfg, temp_init), "cube": (cube_cfg, cube_init)}[which]
    runs = []
    for every in (None, 1):
        sim = amc.Simulation(cfg, seed=17)
        sim.set_state(*init)
        if every:
            sim.sample_enable(every, 0)
        stats = sim.step(10)
        runs.append((sim.state_digest(), stats, sim.histograms(), sim.sample_raw()[1] if every else 0))
        sim.close()
    (d0, s0, h0, _), (d1, s1, h1, n1) = runs
    assert d0 == d1 and n1 == 10
    for a, b in zip(s0, s1):
        for k in COUNTERS:
            assert a[k] == b[k], k
        assert np.array_equal(a["wall_hits"], b["wall_hits"])
    assert np.array_equal(h0[0], h1[0]) and h0[1] == h1[1] and np.array_equal(h0[2], h1[2])


def test_schedule_across_chunks_matches_single_steps_and_checkpoint(pore_cfg, pore_init, tmp_path):
    """every=3 from step 2 over 300 steps: one amc_step call (crosses the 256-step chunk of the library) = explicit
    sample_now after each due step(1) = a run split by checkpoint / restore into a fresh handle."""
    from argon_monte_carlo_b200 import amc
    one = amc.Simulation(pore_cfg)
    one.set_state(*pore_init)
    one.sample_enable(3, 2)
    one.step(300)
    raw_one = one.sample_raw()
    digest = one.state_digest()
    one.close()
    assert raw_one[1] == len(range(2, 300, 3))

    single = amc.Simulation(pore_cfg)
    single.set_state(*pore_init)
    single.sample_enable(0, 0)
    for s in range(300):
        single.step(1)
        if s >= 2 and (s - 2) % 3 == 0:
            single.sample_now()
    assert_raw_equal(raw_one, single.sample_raw())
    assert single.state_digest() == digest
    single.close()

    first = amc.Simulation(pore_cfg)
    first.set_state(*pore_init)
    first.sample_enable(3, 2)
    first.step(151)
    path = str(tmp_path / "ck.npz")
    first.checkpoint(path)
    first.close()
    second = amc.Simulation(pore_cfg)
    second.restore(path)
    assert second.sampling == (3, 2)
    second.step(149)
    assert_raw_equal(raw_one, second.sample_raw())
    assert second.state_digest() == digest
    second.close()


def test_old_checkpoint_restores_without_sampling(pore_cfg, pore_init):
    from argon_monte_carlo_b200 import amc
    sim = amc.Simulation(pore_cfg)
    sim.set_state(*pore_init)
    ck = sim.checkpoint()
    assert not any(k.startswith("sample_") for k in ck)
    sim.close()
    again = amc.Simulation(pore_cfg)
    again.restore(ck)
    assert again.sampling is None
    again.close()


def test_slabs_merge_to_the_single_domain_raw():
    """The dense small pore with cuts inside the end caps, 1-layer slabs included: the merged accumulators of the
    ranks (LocalTransport, one GPU) and of a 1-rank amc_slab_step run equal the single-domain ones bit for bit."""
    from argon_monte_carlo_b200 import amc, config, init_state, slab
    cfg = config.pore_config(False, scale=0.5)
    init = init_state.synthetic_pore_state(cfg, seed=11)
    nz = cfg.grid.nc[2]
    one = amc.Simulation(cfg, seed=17)
    one.set_state(*init)
    one.sample_enable(2, 1)
    one.step(6)
    ref = one.sample_raw()
    digest = one.state_digest()
    one.close()
    assert ref[1] == 3
    for nranks, cuts in ((3, [0, 1, nz - 2, nz]), (4, [0, 1, 2, nz - 1, nz])):
        sim = slab.SlabSimulation(cfg, nranks, init[2], cuts=cuts, seed=17)
        sim.set_state(*init)
        sim.sample_enable(2, 1)
        sim.step(6)
        assert sim.state_digest() == digest
        assert_raw_equal(ref, sim.sample_raw())
        sim.close()
    fused = slab.SlabSimulation(cfg, 1, init[2], seed=17, p2p=True)
    fused.set_state(*init)
    fused.sample_enable(2, 1)
    fused.step_fused(4)
    fused.step_fused(2)
    assert fused.state_digest() == digest
    assert_raw_equal(ref, fused.sample_raw())
    fused.close()


def _md5(path):
    return hashlib.md5(open(path, "rb").read()).hexdigest()


def test_driver_writes_profile_and_leaves_other_outputs_alone(tmp_path, pore_cfg):
    outs = {}
    for tag, extra in (("plain", []), ("sampled", ["--sample-every", "5"])):
        d = tmp_path / tag
        d.mkdir()
        r = subprocess.run([sys.executable, os.path.join(ROOT, "drivers", "Open_Air_Pore_MC.py"), "--steps", "10", *extra],
                           cwd=str(d), capture_output=True, text=True, timeout=1500)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        outs[tag] = d
    plain = sorted(os.listdir(outs["plain"]))
    assert sorted(os.listdir(outs["sampled"])) == sorted(plain + ["profile_z.csv"])
    for f in plain:
        assert _md5(outs["plain"] / f) == _md5(outs["sampled"] / f), f
    rows = (outs["sampled"] / "profile_z.csv").read_text().splitlines()
    assert len(rows) == 1 + pore_cfg.grid.nc[2]
    vals = [r.split(",") for r in rows[1:]]
    assert all(len(v) == 10 and v[2] == "2" for v in vals)
    t = np.array([float(v[6]) for v in vals])
    assert 250 < np.nanmedian(t) < 350


@pytest.mark.parametrize("mode", ["p2p", "nccl"])
def test_multi_gpu_sampling_matches_single_gpu(tmp_path, mode):
    """One process per GPU (torch.distributed.run): the accumulators summed over the ranks equal rank 0's
    single-domain run (tests/nccl_sampling_worker.py).  Needs >= 2 GPUs."""
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
    out = tmp_path / "sampling.json"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(min(ngpu, 4)), "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "nccl_sampling_worker.py"), str(out),
           "--mode", mode, "--steps", "6"]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    res = json.loads(out.read_text())
    assert res["ok"] and res["samples"] == 3
