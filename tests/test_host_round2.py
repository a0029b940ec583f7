"""Host-side pieces added in round 2, no GPU needed: the ctypes mirrors against the C header (sizes taken from gcc),
the state checksum restatement, the reference-baseline runner's parsing, the clock sampler's row selection."""
import ctypes as C
import datetime
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_ctypes_structures_have_the_sizes_of_the_c_header(tmp_path):
    """Every struct that crosses the C ABI is declared twice (include/amc.h and the ctypes classes): compile a probe
    against the header and compare sizeof and a few offsets."""
    from argon_monte_carlo_b200 import amc, slab
    src = tmp_path / "probe.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "amc.h"\nint main(void){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu\\n",'
                   "sizeof(amc_geom), sizeof(amc_config), sizeof(amc_step_stats), sizeof(amc_init_spec), sizeof(amc_slab_config),"
                   "sizeof(amc_slab_p2p_desc), offsetof(amc_config, max_particles), offsetof(amc_slab_p2p_desc, off_flags),"
                   "offsetof(amc_step_stats, dpz));return 0;}\n")
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    want = [C.sizeof(amc.AmcGeom), C.sizeof(amc.AmcConfig), C.sizeof(amc.AmcStepStats), C.sizeof(amc.AmcInitSpec),
            C.sizeof(slab.AmcSlabConfig), C.sizeof(slab.AmcSlabP2PDesc), amc.AmcConfig.max_particles.offset,
            slab.AmcSlabP2PDesc.off_flags.offset, amc.AmcStepStats.dpz.offset]
    assert got == want


def test_state_digest_restatement_is_order_independent_and_additive():
    from argon_monte_carlo_b200 import amc
    rng = np.random.default_rng(7)
    n = 5000
    st = {k: rng.normal(size=n) for k in ("x", "y", "z", "vx", "vy", "vz", "dist", "dist_x", "dist_y", "dist_z")}
    st["flag"] = rng.integers(0, 2, n).astype(np.uint8)
    ids = rng.permutation(10 * n)[:n]
    d = amc.digest_of_arrays(ids, st)
    perm = rng.permutation(n)
    assert amc.digest_of_arrays(ids[perm], {k: v[perm] for k, v in st.items()}) == d
    cut = [0, 17, 1234, n]
    parts = [amc.digest_of_arrays(ids[a:b], {k: v[a:b] for k, v in st.items()}) for a, b in zip(cut, cut[1:])]
    assert amc.combine_digests(parts) == d and d[2] == n
    # one flipped bit anywhere changes both sums
    st2 = {k: v.copy() for k, v in st.items()}
    st2["vz"][123] = np.nextafter(st2["vz"][123], np.inf)
    d2 = amc.digest_of_arrays(ids, st2)
    assert d2[0] != d[0] and d2[1] != d[1]
    # ... and so does attaching a state to another particle id
    ids2 = ids.copy()
    ids2[[5, 6]] = ids2[[6, 5]]
    assert amc.digest_of_arrays(ids2, st) != d


def test_reference_runner_parses_the_scripts_own_timing_prints(monkeypatch, tmp_path):
    """baseline/stage.py takes the per-step times from the lines the upstream scripts print (Pore:517, 554 / Temp:810, 849);
    fed a canned transcript, it returns particle-steps/s from the steps after the initial-overlap transient."""
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import stage
    text = ("Initialization Runtime: 11.5 seconds\n  timestep 0 of 20000   (sim 1 / 1 )\n    Wall Step Runtime: 0.25 seconds\n"
            "    Num collisions from walls: 333\n    Particle-Particle step Runtime: 80.0 seconds\n    1402  collisions from this timestep\n"
            "  timestep 1 of 20000   (sim 1 / 1 )\n    Wall Step Runtime: 0.2 seconds\n    Particle-Particle step Runtime: 39.8 seconds\n"
            "    563  collisions from this timestep\n")
    monkeypatch.setattr(stage, "staged", lambda: True)
    monkeypatch.setattr(stage, "_run_script", lambda kind, k, timeout: (text, 140.0))
    r = stage.run("temp", 2)
    assert r["kind"] == "reference" and r["cores"] == os.cpu_count()
    assert abs(r["ms_per_step"] - 40000.0) < 1e-6 and abs(r["value"] - 557649 / 40.0) < 1e-6      # step 0 dropped
    assert r["detail"]["collisions_per_step"] == [1402, 563]
    # staging copies the upstream files byte for byte (a stand-in upstream tree with distinct contents per file)
    src, dst = tmp_path / "upstream", tmp_path / "_ref"
    src.mkdir()
    for k, f in enumerate(stage.FILES):
        (src / f).write_bytes(bytes(range(k, 256)) + b"\r\n" + f.encode())
    monkeypatch.setattr(stage, "REF_DIR", str(dst))
    assert stage.stage(str(src))
    for f in stage.FILES:
        assert (dst / f).read_bytes() == (src / f).read_bytes()
    assert not stage.stage(str(tmp_path / "missing"))


def test_clock_sampler_selects_rows_by_timestamp():
    sys.path.insert(0, ROOT)
    import bench
    cs = bench.ClockSampler(0)
    t0 = datetime.datetime(2026, 10, 18, 12, 0, 0)
    fmt = lambda t: t.strftime("%Y/%m/%d %H:%M:%S.%f")[:-3]
    rows = []
    for k in range(100):                                    # one row every 10 ms; rows 40-59 run hot and capped
        t = t0 + datetime.timedelta(milliseconds=10 * k)
        rows.append([fmt(t), "1965" if 40 <= k < 60 else "345", "1965", "700.0", "Not Active", "Not Active", "Not Active",
                     "Active" if 50 <= k < 55 else "Not Active"])
    cs.rows = rows

    class P:                                               # a finished nvidia-smi
        def terminate(self): pass
        def wait(self, timeout=None): pass
    cs.proc = P()
    cs.t_warm = t0 + datetime.timedelta(milliseconds=300)
    cs.t_start = t0 + datetime.timedelta(milliseconds=400)
    real_now = datetime.datetime.now

    class FakeDT(datetime.datetime):
        @classmethod
        def now(cls):
            return t0 + datetime.timedelta(milliseconds=590)
    datetime.datetime = FakeDT
    try:
        out = cs.stop()
    finally:
        datetime.datetime = FakeDT.__mro__[1]
    assert out["window"] == "timed region" and out["sm_mhz"] == 1965.0 and out["sm_max_mhz"] == 1965.0
    assert out["samples"] >= 19 and out["reasons"] == ["sw_power_cap"]


def test_event_driven_cube_sweep_model_equals_the_serial_sweep(oracle, cube_cfg, cube_init):
    """k_sweep_detect / k_sweep_events walk only the cells that can hold a collision (~60 of 3,375 per timestep) and
    reproduce the reference's stale layer masks through per-particle snapshots.  Their Python restatement
    (tests/cube_events_model.py) must give the oracle's serial sweep (Cube:232-336) bit for bit: state, collision
    count, reference-equivalent test counter, completed paths, pair list."""
    import cube_events_model as M
    from oracle import steps
    names = ("x", "y", "z", "vx", "vy", "vz", "dist", "dist_x", "dist_y", "dist_z", "flag")
    st, mine = oracle.ParticleState(*cube_init), oracle.ParticleState(*cube_init)
    visits = 0
    for k in range(8):
        sink, pairs = oracle.PathSink(), oracle.PairSink()
        r = steps.cube_step(st, cube_cfg, sink, pairs)
        oracle.drift(mine, cube_cfg.dt, False)
        oracle.cube_walls(mine, cube_cfg.cube_x, cube_cfg.cube_y, cube_cfg.cube_z)
        d = {nm: getattr(mine, nm) for nm in names}
        ncol, checks, paths, prs, v = M.sweep_events(d, cube_cfg.grid, cube_cfg.collision_range, cube_cfg.argon_mass)
        assert (ncol, checks) == (r["pp_collisions"], r["checks"]), k
        for nm in names:
            assert np.array_equal(getattr(mine, nm), getattr(st, nm)), (k, nm)
        ref_paths = np.array(sink.arrays()).T.reshape(-1, 4)
        assert np.array_equal(np.sort(np.array(paths).reshape(-1, 4), axis=0), np.sort(ref_paths, axis=0))
        hi, lo, _, cell = pairs.arrays()
        assert [(int(a), int(b), int(c)) for a, b, c in zip(hi, lo, cell)] == prs     # same pairs, same order, same cells
        visits += v
    assert visits < 8 * 150            # the point of the exercise: a few dozen cell visits per step, not 3,375
