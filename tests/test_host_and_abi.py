"""Host-side logic and the C-ABI library, without a GPU: constants, exported symbols, loud failure
when no device is present, the product never touching the oracle, output formats."""
import ctypes
import math
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def test_constants_match_the_reference_scripts(pore_cfg, temp_cfg, cube_cfg):
    assert pore_cfg.num_molecules == temp_cfg.num_molecules == 557649 and cube_cfg.num_molecules == 24627
    assert pore_cfg.collision_range == 3.385137501286538e-10
    assert (pore_cfg.open_air_particles, pore_cfg.hot_pore_particles, pore_cfg.gap_particles,
            pore_cfg.cold_pore_particles, pore_cfg.remaining_particles) == (174079, 2088, 2683, 204717, 3)
    assert pore_cfg.geom.z_gb == 1.3000000000000003e-07          # open_air_height + hot_coating_height
    assert abs(pore_cfg.dt - 1.84808e-13) < 1e-18 and abs(temp_cfg.dt - 1.84895e-13) < 1e-18
    assert abs(cube_cfg.dt - 7.39234e-12) < 1e-17
    assert pore_cfg.grid.nc == (14, 14, 148) and pore_cfg.grid.c0 == (-7, -7, 0)
    assert cube_cfg.grid.nc == (15, 15, 15) and cube_cfg.min_num_particles_per_cell == 7 and cube_cfg.remaining_particles == 1002
    assert float(temp_cfg.surface_energy_cold) == 1.7463480823716586e-21
    assert float(temp_cfg.surface_energy_hot) == 3.2454458503944502e-21


def test_grid_tables_use_the_reference_expressions(pore_cfg):
    g, c = pore_cfg.grid, pore_cfg
    for grp in range(2):
        for layer in range(7):
            k = 2 * layer + grp
            assert g.lo[0][k] == (2 * layer + grp - c.num_x_subdivions) * c.dx - c.collision_range
            assert g.edge[0][k + 1] == (2 * layer + grp - c.num_x_subdivions + 1) * c.dx
        for layer in range(74):
            k = 2 * layer + grp
            assert g.lo[2][k] == (2 * layer + grp) * c.dz - c.collision_range
            assert g.edge[2][k + 1] == (2 * layer + grp + 1) * c.dz


def test_scaled_configs_keep_density_and_even_grids():
    from argon_monte_carlo_b200 import config
    base = config.pore_config(True)
    for scale in (0.5, 2.82, 5.64):
        c = config.pore_config(True, scale=scale)
        assert all(n % 2 == 0 for n in c.grid.nc)
        assert abs(c.num_molecules / base.num_molecules / scale**3 - 1) < 1e-3
        assert 18e-9 < c.dx < 26e-9 and 18e-9 < c.dz < 26e-9


def test_overlap_threshold_is_the_exact_sqrt_boundary(pore_cfg):
    import math
    from argon_monte_carlo_b200 import amc
    cr = float(pore_cfg.collision_range)
    t = amc.overlap_threshold(cr)
    assert math.sqrt(t) >= cr and math.sqrt(math.nextafter(t, 0.0)) < cr
    rng = np.random.default_rng(0)
    d2 = t * (1 + rng.uniform(-4, 4, 20000) * 2.220446049250313e-16)
    assert np.array_equal(np.sqrt(d2) < cr, d2 < t)


def test_library_exports_every_symbol_of_the_header():
    from argon_monte_carlo_b200 import amc, build
    header = open(os.path.join(ROOT, "include", "amc.h")).read()
    declared = sorted(set(re.findall(r"\b(amc_[a-z_0-9]+)\s*\(", header)))
    assert declared == sorted(amc.EXPORTS)
    lib = ctypes.CDLL(build.build_library())
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.amc_abi_version() == amc.ABI_VERSION


def test_ctypes_structs_match_the_header_layout():
    from argon_monte_carlo_b200 import amc
    header = open(os.path.join(ROOT, "include", "amc.h")).read()
    geom = re.search(r"typedef struct amc_geom \{(.*?)\} amc_geom;", header, re.S).group(1)
    names = re.findall(r"\b([A-Za-z_0-9]+)\s*[,;]", re.sub(r"/\*.*?\*/", "", geom, flags=re.S))
    assert tuple(n for n in names if n != "double") == amc.GEOM_FIELDS
    assert ctypes.sizeof(amc.AmcGeom) == 8 * len(amc.GEOM_FIELDS)
    assert ctypes.sizeof(amc.AmcStepStats) == 8 * (10 + 10 + 3)


def test_no_cpu_fallback_without_a_device():
    """In a process that sees no device (CUDA_VISIBLE_DEVICES empty, so this runs on GPU machines too) creating a
    simulation raises AmcError instead of computing anywhere else."""
    import subprocess
    import sys
    code = ("from argon_monte_carlo_b200 import amc, config\n"
            "try:\n    amc.Simulation(config.pore_config(False))\nexcept amc.AmcError as e:\n    print('AmcError', e)\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.startswith("AmcError"), r.stdout + r.stderr


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "argon_monte_carlo_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.lower().replace("the cpu oracle", "").replace("oracle)", "") or \
                    "import oracle" not in text and "from oracle" not in text, f
                assert "from oracle" not in text and "import oracle" not in text, f
    for f in os.listdir(os.path.join(ROOT, "drivers")):
        text = open(os.path.join(ROOT, "drivers", f)).read()
        assert "from oracle" not in text and "import oracle" not in text, f


def test_host_rng_consumes_the_streams_like_the_reference():
    """random_inbounds_direction (Temperature_Pore_MC.py:132-141) draws np.random.uniform,
    random.uniform, np.random.choice per attempt; check the stream positions and the cone."""
    import random
    from argon_monte_carlo_b200 import host_rng
    np.random.seed(3); random.seed(3)
    norm = np.array([0.0, 0.0, -1.0])
    d = host_rng.inbound_direction(norm)
    assert abs(np.dot(d, d) - 1) < 1e-15 and np.dot(d, norm) >= host_rng.COS85
    after_np, after_py = np.random.uniform(), random.random()
    # replay by hand
    np.random.seed(3); random.seed(3)
    import math
    while True:
        ct = np.random.uniform(low=-1.0, high=1.0); phi = random.uniform(0, math.pi); th = math.acos(ct)
        v = np.array([math.cos(phi) * math.sin(th), math.sin(phi) * math.sin(th) * np.random.choice([-1, 1]), math.cos(th)])
        if abs(np.dot(v, norm)) < host_rng.COS85:
            continue
        if np.dot(v, norm) < host_rng.COS85:
            v = -v
        break
    assert np.array_equal(v, d) and np.random.uniform() == after_np and random.random() == after_py


def test_output_writers_formats(tmp_path):
    from argon_monte_carlo_b200 import outputs
    counts = np.zeros((4, 200), dtype=np.int64)
    counts[:, 0], counts[:, 3] = 7, 1
    outputs.write_histograms(counts, str(tmp_path))
    x = open(os.path.join(str(tmp_path), "hist_x_axis_z_data.txt")).read()
    assert x == open(os.path.join(GOLD, "shipped_hist_x_axis_z_data.txt")).read()
    y = open(os.path.join(str(tmp_path), "hist_y_axis_total_data.txt")).read()
    assert y.startswith("[1.75e+08 0.00e+00 0.00e+00 2.50e+07") and y.endswith("]")
    ref = np.histogram([1e-9] * 7 + [1.6e-8], bins=200, range=(0, 10 ** -6), density=True)[0]
    assert np.array_equal(outputs.density(counts[0]), ref)
    outputs.write_momentum_energy_csv([-4.06031315107044e-22, 0], [-1.81678728388749e-18, 0], [-1.4427412763244e-19, 0],
                                      os.path.join(str(tmp_path), "m.csv"))
    lines = open(os.path.join(str(tmp_path), "m.csv")).read().split("\n")
    shipped = open(os.path.join(GOLD, "shipped_momentum_energy.csv")).read().split("\n")
    assert lines[0] == shipped[0] and lines[1] == shipped[1] and lines[2] == "1,0,0,0"


def test_shipped_histograms_are_consistent_with_the_density_rule():
    """The four shipped hist_y files all come from 30,828 completed paths (SURVEY section 4)."""
    from argon_monte_carlo_b200 import outputs
    for s in ("total", "x", "y", "z"):
        dens = np.array(open(os.path.join(GOLD, "shipped_hist_y_axis_%s_data.txt" % s)).read().strip("[]").split(), dtype=float)
        assert len(dens) == 200
        counts = np.rint(dens * 5e-9 * 30828).astype(np.int64)
        assert counts.sum() == 30828
        assert np.allclose(outputs.density(counts), dens, rtol=2e-8)


def test_calm_regions_never_hide_a_wall_event(oracle, temp_cfg):
    """advance_particle (amc_kernels.cuh) skips the wall masks, the recapture and the out-of-bounds census for
    particles whose positions before and after the drift lie in one of three 'calm' regions whose bounds are the
    min / max of the geometry's thresholds (amc_api.cu).  Property checked here against the oracle, on particles
    thrown at every wall from both sides with displacements of up to several nanometres per step: for every particle
    the predicate calls calm, the reference's step is the drift and nothing else."""
    import math
    from wall_edges import calm_bounds
    g, dt = temp_cfg.geom, temp_cfg.dt
    zs = [g.oah, g.zh3, g.z_gb, g.zgb_p, g.z_gt, g.zgt_m, g.z_cold, g.zc3]
    zA, zB, rA, rC = calm_bounds(g)
    assert 0 < zA < zB < g.H and 0 < rC < rA

    rng = np.random.default_rng(42)
    n = 600000
    # z: uniform over the domain and a bit beyond, plus clusters within 2 nm of every threshold
    z = rng.uniform(-3e-9, g.H + 3e-9, n)
    k = rng.integers(0, len(zs) + 2, n)
    near = np.array(zs + [0.0, g.H])[k] + rng.uniform(-2e-9, 2e-9, n)
    z = np.where(rng.random(n) < 0.5, near, z)
    radii = np.array([g.R_oa, math.sqrt(g.R_p_sq), math.sqrt(g.R_g_sq), math.sqrt(g.R_p_c_sq), math.sqrt(g.R_g_c_sq)])
    r = np.where(rng.random(n) < 0.5, radii[rng.integers(0, 5, n)] + rng.uniform(-2e-9, 2e-9, n),
                 g.R_oa * 1.02 * np.sqrt(rng.random(n)))
    r = np.abs(r)
    th = rng.uniform(0, 2 * np.pi, n)
    x, y = r * np.cos(th), r * np.sin(th)
    disp = rng.normal(0.0, 1.5e-9, (3, n))                     # ~20 x the thermal displacement of one step
    vx, vy, vz = disp / dt
    nx, ny, nz = x + dt * vx, y + dt * vy, z + dt * vz         # the device's drift, operation for operation
    rmax = np.maximum(x * x + y * y, nx * nx + ny * ny)
    zmin, zmax = np.minimum(z, nz), np.maximum(z, nz)
    calm = ((rmax <= rA) & (((zmin >= 0.0) & (zmax < zA)) | ((zmin > zB) & (zmax <= g.H)))) | \
           ((rmax < rC) & (zmin >= 0.0) & (zmax <= g.H))
    assert 0.1 < calm.mean() < 0.9                              # the sample exercises both sides of the predicate
    c = np.nonzero(calm)[0]
    st = oracle.ParticleState(x[c], y[c], z[c], vx[c], vy[c], vz[c])
    # closing recapture of the previous step on the pre-drift position: nothing to do
    assert oracle.temp_oob_count(st, g) == 0 and oracle.temp_recapture(st, g) == 0
    oracle.drift(st, dt, True)
    from argon_monte_carlo_b200 import config
    cheb = config.gap_energy_chebyshev(temp_cfg, 16)
    counts, sums, errs, bits = oracle.temp_walls_philox(st, g, 1, 0, cheb, None, True)
    assert counts.sum() == 0 and errs == 0 and not bits.any()
    assert oracle.temp_oob_count(st, g) == 0 and oracle.temp_recapture(st, g) == 0
    assert np.array_equal(st.x, nx[c]) and np.array_equal(st.y, ny[c]) and np.array_equal(st.z, nz[c])
    assert np.array_equal(st.vx, vx[c]) and np.array_equal(st.vz, vz[c])
    # and the predicate is not vacuous about the rest: the others do hit walls or leave the domain
    o = np.nonzero(~calm)[0]
    st2 = oracle.ParticleState(x[o], y[o], z[o], vx[o], vy[o], vz[o])
    oracle.drift(st2, dt, True)
    counts2, _, _, _ = oracle.temp_walls_philox(st2, g, 1, 0, cheb, None, True)
    assert counts2.sum() > 1000


def test_detection_filter_threshold_is_conservative(pore_cfg):
    """k_detect decides in fp32 on cell-relative coordinates whether a pair may overlap; det_thr (amc_api.cu) widens
    the threshold by the rounding bound so that no pair the exact fp64 test accepts is ever filtered out.  Emulated
    here in NumPy float32 (both summation orders; the kernel's fused multiply-adds round less, not more) on pairs
    placed within +-1e-4 relative of the collision range, anywhere in a cell, along random directions."""
    from argon_monte_carlo_b200 import amc
    g = pore_cfg.grid
    cr = pore_cfg.collision_range
    overlap_sq = amc.overlap_threshold(cr)
    wmax = max(float(np.max(g.edge[a][1:] - g.lo[a])) for a in range(3))
    e_abs = 6.0 * math.ldexp(wmax, -24)
    r_f = math.sqrt(overlap_sq) * (1.0 + 1e-9) + 2.0 * e_abs
    thr = np.nextafter(np.float32(r_f * r_f * (1.0 + math.ldexp(1.0, -20))), np.float32(np.inf))
    rng = np.random.default_rng(7)
    n = 2000000
    lo = np.array([g.lo[a][3] for a in range(3)])
    a = lo[:, None] + rng.uniform(0, wmax, (3, n))
    d = rng.normal(size=(3, n)); d /= np.linalg.norm(d, axis=0)
    b = a + d * cr * (1.0 + rng.uniform(-1e-4, 1e-4, n))
    dd = b - a
    exact = (dd[0] * dd[0] + dd[1] * dd[1]) + dd[2] * dd[2] < overlap_sq          # Pore:173-174 as the kernels evaluate it
    fa, fb = (a - lo[:, None]).astype(np.float32), (b - lo[:, None]).astype(np.float32)
    e = fb - fa
    d2a = (e[0] * e[0] + e[1] * e[1]) + e[2] * e[2]
    d2b = e[2] * e[2] + (e[1] * e[1] + e[0] * e[0])
    assert exact.sum() > 500000
    assert np.all(d2a[exact] < thr) and np.all(d2b[exact] < thr)
    # the filter is not sloppy either: it widens the radius by ~5e-5 relative (a quarter of this +-1e-4 sample,
    # 1.4e-4 of the true pairs of a uniform gas)
    assert np.mean((d2a < thr) & ~exact) < 0.3 and math.sqrt(float(thr)) / cr - 1 < 1e-4
