"""The builders of tests/wall_edges.py check themselves on the CPU: every particle lands exactly where its label says,
the threshold relations the kernels rely on hold at the configs used, the reference's own radial decision equals the
squared-threshold one, the oracle's hit bits show every wall case, corner, error path, recapture condition and both
sides of every calm bound, and the Chebyshev table of the gap energy matches mpmath at every case 4 contact height."""
import math

import numpy as np
import pytest

import wall_edges as we

CONFIGS = [("pore", "1"), ("pore", "bench"), ("temp", "1"), ("temp", "0.5"), ("temp", "bench")]
_BUILT = {}


def built(oracle, kind, scale):
    if (kind, scale) not in _BUILT:
        cfg, s = we.pore_cfg_of(kind, scale)
        _BUILT[(kind, scale)] = (cfg, s, we.pore_edges(oracle, cfg, s))
    return _BUILT[(kind, scale)]


def same_bits(a, b):
    return np.array_equal(we.bits_of(a), we.bits_of(b))


@pytest.mark.parametrize("kind,scale", CONFIGS)
def test_builders_land_on_what_they_claim(oracle, kind, scale):
    cfg, s, b = built(oracle, kind, scale)
    assert len(b.pos) > 4000 and b.skipped < 0.1 * len(b.pos)
    pre, post, vel = np.array(b.pos), np.array(b.post), np.array(b.vel)
    drift = pre + cfg.dt * vel                                   # the kernels' drift, operation for operation
    assert same_bits(drift, post)
    st = oracle.ParticleState(*b.arrays())
    oracle.drift(st, cfg.dt, True)
    assert same_bits(np.stack([st.x, st.y, st.z], 1), post)
    for i, c in enumerate(b.claims):
        got = {"r2": we.r2k(post[i, 0], post[i, 1]), "pr2": we.r2k(pre[i, 0], pre[i, 1]), "z": post[i, 2], "pz": pre[i, 2]}
        for k, v in c.items():
            assert same_bits(got[k], v), (b.label[i], k, got[k], v)


def test_cube_builder_lands_on_every_face_value(oracle):
    from pair_edges import cube_groups_config
    for cfg in (cube_groups_config(), we.cube_cfg_of("2")):
        b = we.cube_edges(cfg)
        pre, post, vel = np.array(b.pos), np.array(b.post), np.array(b.vel)
        assert same_bits(pre + cfg.dt * vel, post)
        L = (cfg.cube_x, cfg.cube_y, cfg.cube_z)
        for a in range(3):
            have = set(we.bits_of(post[:, a]).tolist())
            for v in (L[a], we.up(L[a]), 0.0, -0.0, we.down(0.0)):
                assert int(we.bits_of(v)) in have, (a, v)
        st = oracle.ParticleState(*b.arrays())
        oracle.drift(st, cfg.dt, False)
        counts = oracle.cube_walls(st, *L)
        assert np.all(counts > 0)
        assert b.skipped < 0.02 * len(b.pos)


def test_threshold_relations_of_the_configs_used():
    """At scale 1 the open-air threshold gt_R_oa is R_oa_sq + 1 ulp (the recapture sees one double the wall does not);
    at the timed 12.5 M-particle geometry gt_R == R_sq for all three radii; the calm bounds are zh3 and zc3."""
    for kind, scale in CONFIGS:
        cfg, _ = we.pore_cfg_of(kind, scale)
        g = cfg.geom
        rel = {nm: int(we.bits_of(we.sq_threshold_gt(R)) - we.bits_of(Rsq))
               for nm, R, Rsq in (("R_oa", g.R_oa, g.R_oa_sq), ("R_p", g.R_p, g.R_p_sq), ("R_g", g.R_g, g.R_g_sq))}
        if scale == "1":
            assert rel["R_oa"] == 1
        if scale == "bench":
            assert rel == {"R_oa": 0, "R_p": 0, "R_g": 0}
        zA, zB, rA, rC = we.calm_bounds(g)
        assert zA == g.zh3 and zB == g.zc3 and rA == min(g.R_oa_sq, we.sq_threshold_gt(g.R_oa)) and rC == g.R_p_c_sq


@pytest.mark.parametrize("kind,scale", CONFIGS)
def test_reference_radial_decision_equals_the_squared_threshold(kind, scale):
    """math.sqrt(r2) > R (the reference's expression, correctly rounded) == r2 > gt_R, and < R == r2 < lt_R, for every
    radial value of the builders and every double within 16 ulps of R*R and of gt_R / lt_R."""
    cfg, _ = we.pore_cfg_of(kind, scale)
    g = cfg.geom
    vals = [v for v, _ in we.radial_values(g)]
    for R in (g.R_oa, g.R_p, g.R_g):
        gt, lt = we.sq_threshold_gt(R), we.sq_threshold_lt(R)
        around = [float(we.nudge(c, k)) for c in (R * R, gt, lt) for k in range(-16, 17)]
        for v in vals + around:
            assert (math.sqrt(v) > R) == (v > gt), (R, v)
            assert (math.sqrt(v) < R) == (v < lt), (R, v)


def oracle_bits(oracle, cfg, b):
    _, bits, _, _ = we.oracle_walls(oracle, cfg, b)
    return bits.astype(np.int64)


@pytest.mark.parametrize("kind,scale", [c for c in CONFIGS if c[1] != "0.5"])
def test_coverage_by_the_oracle(oracle, kind, scale):
    cfg, s, b = built(oracle, kind, scale)
    g = cfg.geom
    bits = oracle_bits(oracle, cfg, b)
    ncase = 10 if kind == "temp" else 9
    boundary = np.array([lab.split(":")[0] in ("radial", "z", "calm", "gap energy") for lab in b.label])
    for c in range(ncase):                                   # every case from a particle placed on a boundary
        assert np.any(boundary & ((bits >> c) & 1).astype(bool)), "case bit %d never hit from a boundary value" % c
    for name, m in we.corner_kinds(kind, bits):
        assert m.sum() > 0, name
    if kind == "pore":                                       # no corner at the pore mouth of the open-air pore
        assert not np.any(((bits & 0b11000) != 0) & (((bits >> 8) & 1) == 1))
    # the error path: a == 0 and disc < 0, alone
    for what in ("a == 0", "disc < 0"):
        sub = b.subset([i for i, lab in enumerate(b.label) if what in lab])
        _, _, counts, errs = we.oracle_walls(oracle, cfg, sub)
        assert len(sub.pos) > 0 and errs == counts[0] == len(sub.pos), what
    # every recapture condition fires after the walls or after the pair pass
    st, _, _, _ = we.oracle_walls(oracle, cfg, b)
    fired = recapture_conditions(g, st)
    (oracle.temp_recapture if kind == "temp" else oracle.pore_recapture)(st, g)
    oracle.pp_groups(st, cfg.grid, cfg.collision_range, cfg.argon_mass)
    after_pp = recapture_conditions(g, st)
    for k in fired:
        assert fired[k].any() or after_pp[k].any(), k
    assert after_pp["z < 0"].any() and after_pp["z > H"].any()
    # the one-double window at scale 1: r2 == gt_R_oa is no open-air hit, but the recapture moves it to the axis
    if scale == "1":
        gt = we.sq_threshold_gt(g.R_oa)
        on = np.array([c.get("r2") == gt for c in b.claims])
        post = np.array(b.post)
        assert on.any() and not np.any(bits[on] & 1)
        assert np.all(we.r2k(post[on, 0], post[on, 1]) > g.R_oa_sq)


def recapture_conditions(g, st):
    x, y, z = st.x, st.y, st.z
    r2 = we.r2k(x, y)
    return {"z < 0": z < 0, "z > H": z > g.H, "R_oa": r2 > g.R_oa_sq, "R_g": (r2 > g.R_g_sq) & (z > g.oah) & (z < g.z_cold),
            "R_p": (r2 > g.R_p_sq) & (((z > g.oah) & (z < g.z_gb)) | ((z > g.z_gt) & (z < g.z_cold)))}


@pytest.mark.parametrize("scale", ["1", "bench"])
def test_both_sides_of_every_calm_bound(oracle, scale):
    """Particles the calm predicate accepts on each bound, and particles one double outside it that do hit a wall or
    leave the domain: 6H at z == zh3 == calm_zA is one of them."""
    cfg, s, b = built(oracle, "temp", scale)
    g = cfg.geom
    zA, zB, rA, rC = we.calm_bounds(g)
    pre, post = np.array(b.pos), np.array(b.post)
    calm = we.is_calm(g, pre, post)
    bits = oracle_bits(oracle, cfg, b)
    st, _, _, _ = we.oracle_walls(oracle, cfg, b)
    oob = we.oob_rows(g, "temp", st.x, st.y, st.z)
    event = (bits != 0) | oob
    assert not np.any(calm & event)                     # the predicate never hides a wall event
    zmax, zmin = np.maximum(pre[:, 2], post[:, 2]), np.minimum(pre[:, 2], post[:, 2])
    rmax = np.maximum(we.r2k(pre[:, 0], pre[:, 1]), we.r2k(post[:, 0], post[:, 1]))
    sides = {"zmax == prev(calm_zA)": zmax == we.down(zA), "zmax == calm_zA": zmax == zA,
             "zmin == calm_zB": zmin == zB, "zmin == next(calm_zB)": zmin == we.up(zB),
             "zmin == 0": zmin == 0.0, "zmin == prev(0)": zmin == we.down(0.0), "zmax == H": zmax == g.H, "zmax == next(H)": zmax == we.up(g.H),
             "rmax == calm_rA": rmax == rA, "rmax == next(calm_rA)": rmax == we.up(rA),
             "rmax == prev(calm_rC)": rmax == we.down(rC), "rmax == calm_rC": rmax == rC}
    inside = ("zmax == prev(calm_zA)", "zmin == next(calm_zB)", "zmin == 0", "zmax == H", "rmax == calm_rA", "rmax == prev(calm_rC)")
    for k, m in sides.items():
        if k in inside:
            assert np.any(m & calm), k
        elif k == "zmin == prev(0)":          # only a start can be there: no drift from inside ends on the smallest negative
            assert np.any(m & ~calm), k
        else:
            assert np.any(m & ~calm & event), k
    six_h = (post[:, 2] == g.zh3) & (((bits >> 8) & 1) == 1)
    assert np.any(six_h & (zmax == zA))


@pytest.mark.parametrize("scale", ["1", "bench"])
def test_gap_energy_table_at_every_case4_contact(oracle, scale):
    """The device's Chebyshev table (cheb_eval) against mpmath's surface_energy_gap at the contact height of every
    case 4 hit of the built states, contacts outside [z_gb, z_gt] included, to 1e-13 relative."""
    import surface_oracle as SO
    from argon_monte_carlo_b200 import config
    cfg, s, b = built(oracle, "temp", scale)
    cheb = we.cheb_of(cfg)
    st = oracle.ParticleState(*b.arrays())
    oracle.drift(st, cfg.dt, True)
    sink = SO.HitSink()
    SO.temp_walls_philox_hits(st, cfg.geom, 17, 0, cheb, sink)
    h = sink.hits()
    zc = h["col"][h["case"] == 5, 2]
    zc = zc[np.isfinite(zc)]
    assert len(zc) > 50
    assert np.any(zc < cfg.gap_bottom_height) and np.any(zc > cfg.gap_top_height)
    for z in zc:
        ref = float(config.surface_energy_gap(cfg, z))
        assert abs(oracle.cheb_eval(cheb, z) - ref) <= 1e-13 * ref, z
