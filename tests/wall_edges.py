"""States placed on the floating-point boundaries of the per-particle step (test infrastructure only; NumPy and the oracle).

Every decision of the drift / wall / recapture half of a timestep is a comparison with a threshold: the radial masks
(`np.sqrt(x**2 + y**2) > R` in the reference and the oracle, `x*x + y*y > gt_R` in the kernels, with gt_R / lt_R found
by a nextafter search in amc_api.cu), the z planes of the masks, the recapture and the out-of-bounds census, the cube
faces, and the bounds of the calm regions with which advance_particle skips all wall work.  Gas states reach these
values with a probability close to zero; the builders here put particles on them exactly, before and after the drift,
and label each particle with what it was placed on.

- ``radial_values`` / ``z_planes``: the thresholds of a geometry and the doubles next to them, labelled.
- ``on_r2``: a point (x, y) with x*x + y*y equal to a given double, evaluated in the kernels' order.
- ``velocity_for``: a velocity with which the drift maps one coordinate exactly onto another.
- ``Edges``: a State whose particles are placed by (pre-drift, post-drift) targets, with the claims recorded.
- the builders (radial, z, calm bounds, corners, contact degeneracies, recapture, pair-pass pushes, gap energy, cube
  faces), ``pore_edges`` / ``cube_edges`` that collect them, and ``with_gas`` to interleave them with a gas.
"""
from __future__ import annotations

import itertools
import math

import numpy as np

from pair_edges import State, down, first_difference, nudge, preimage, up  # noqa: F401  (first_difference: re-exported)

NM = 1e-9


# ------------------------------------------------------------------ thresholds
def sq_threshold_gt(R):
    """amc_api.cu: largest double t with sqrt(t) <= R, so sqrt(v) > R <=> v > t."""
    t = R * R
    while math.sqrt(t) <= R:
        t = float(np.nextafter(t, np.inf))
    while math.sqrt(t) > R:
        t = float(np.nextafter(t, 0.0))
    return float(t)


def sq_threshold_lt(R):
    """amc_api.cu: smallest double t with sqrt(t) >= R, so sqrt(v) < R <=> v < t."""
    t = R * R
    while math.sqrt(t) >= R:
        t = float(np.nextafter(t, 0.0))
    while math.sqrt(t) < R:
        t = float(np.nextafter(t, np.inf))
    return float(t)


def calm_bounds(g):
    """(calm_zA, calm_zB, calm_rA, calm_rC) as amc_api.cu computes them for the energized pore."""
    zs = [g.oah, g.zh3, g.z_gb, g.zgb_p, g.z_gt, g.zgt_m, g.z_cold, g.zc3]
    zA, zB = min(zs + [g.H]), max(zs + [0.0])
    rA = min(sq_threshold_gt(g.R_oa), g.R_oa_sq)
    rC = min(rA, g.R_p_sq, g.R_g_c_sq, g.R_p_c_sq, g.R_g_sq)
    return zA, zB, rA, rC


def is_calm(g, pre, post):
    """advance_particle's calm predicate on (x, y, z) before and after the drift (arrays of shape (n, 3))."""
    zA, zB, rA, rC = calm_bounds(g)
    pre, post = np.asarray(pre), np.asarray(post)
    rmax = np.maximum(r2k(pre[:, 0], pre[:, 1]), r2k(post[:, 0], post[:, 1]))
    zmin, zmax = np.minimum(pre[:, 2], post[:, 2]), np.maximum(pre[:, 2], post[:, 2])
    return ((rmax <= rA) & (((zmin >= 0.0) & (zmax < zA)) | ((zmin > zB) & (zmax <= g.H)))) | \
        ((rmax < rC) & (zmin >= 0.0) & (zmax <= g.H))


def r2k(x, y):
    """x*x + y*y in the kernels' order (no fused multiply-add)."""
    x, y = np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64)
    return x * x + y * y


def radial_families(g):
    """{family: [(value, label)]}: for R_oa, R_p and R_g the values R*R, gt_R, lt_R and R_*_sq, for R_p_c and R_g_c the
    squared contact radii of the config, each with the doubles -1, +1 and +2 ulp away; duplicates dropped."""
    fam = {}
    for nm, R, Rsq in (("R_oa", g.R_oa, g.R_oa_sq), ("R_p", g.R_p, g.R_p_sq), ("R_g", g.R_g, g.R_g_sq)):
        fam[nm] = {"%s*%s" % (nm, nm): R * R, "gt_%s" % nm: sq_threshold_gt(R), "lt_%s" % nm: sq_threshold_lt(R),
                   "%s_sq" % nm: float(Rsq)}
    fam["R_p_c"] = {"R_p_c_sq": float(g.R_p_c_sq)}
    fam["R_g_c"] = {"R_g_c_sq": float(g.R_g_c_sq)}
    out = {}
    for f, base in fam.items():
        seen, vals = set(), []
        for lab, T in base.items():
            for k in (-1, 0, 1, 2):
                v = float(nudge(T, k))
                if v not in seen:
                    seen.add(v)
                    vals.append((v, lab + ("" if k == 0 else "%+dulp" % k)))
        out[f] = vals
    return out


def radial_values(g):
    return [vl for vals in radial_families(g).values() for vl in vals]


def z_planes(g):
    """[(value, label)]: every z that a wall mask, the recapture or the census of either pore script compares with."""
    return [(0.0, "0"), (float(g.H), "H"), (g.oah, "oah"), (g.z_cold, "z_cold"), (g.z_gb, "z_gb"),
            (g.z_gt_pore, "z_gt_pore"), (g.z_gt, "z_gt"), (g.zh3, "zh3"), (g.zc3, "zc3"), (g.zgb_p, "zgb_p"),
            (g.zgt_m, "zgt_m")]


def z_values(g):
    """Each plane and the doubles on either side, -0.0 beside 0."""
    out = []
    for P, lab in z_planes(g):
        out += [(float(down(P)), "prev(%s)" % lab), (float(P), lab), (float(up(P)), "next(%s)" % lab)]
        if P == 0.0:
            out.append((-0.0, "-0.0"))
    return out


# ------------------------------------------------------------------ exact placements
def on_r2(T, theta, reach=48):
    """(x, y) near sqrt(T) (cos theta, sin theta) with x*x + y*y == T exactly, or None."""
    r = math.sqrt(T)
    x0, s = r * math.cos(theta), math.copysign(1.0, math.sin(theta))
    X = nudge(np.full(2 * reach + 1, x0), np.arange(-reach, reach + 1))
    Y0 = s * np.sqrt(np.maximum(T - X * X, 0.0))
    for dk in (0, -1, 1, -2, 2, -3, 3):
        Y = nudge(Y0, dk)
        hit = np.flatnonzero(r2k(X, Y) == T)
        if len(hit):
            h = hit[np.argmin(np.abs(hit - reach))]
            return float(X[h]), float(Y[h])
    return None


def velocity_for(p0, p1, dt, reach=48):
    """v with fl(p0 + fl(dt * v)) == p1 (the drift of the oracle and the kernels), or None."""
    p0, p1 = float(p0), float(p1)
    if np.float64(p0).view(np.int64) == np.float64(p1).view(np.int64):
        return -0.0 if math.copysign(1.0, p0) < 0 else 0.0
    v0 = (p1 - p0) / dt
    if v0 == 0.0:
        return None
    for k in range(reach + 1):
        for v in {float(nudge(v0, k)), float(nudge(v0, -k))}:
            if p0 + dt * v == p1 and math.copysign(1.0, p0 + dt * v) == math.copysign(1.0, p1):
                return v
    return None


def bits_of(v):
    return np.asarray(v, dtype=np.float64).view(np.int64)


class Edges(State):
    """Particles placed by their position before and after one drift.  `claims[i]` holds what particle i was placed on
    (any of 'r2', 'pr2', 'z', 'pz', 'x', 'y' -> the intended double), checked bit for bit by the host tests."""

    def __init__(self, cfg, tag):
        super().__init__()
        self.cfg, self.dt, self.tag = cfg, float(cfg.dt), tag
        self.claims, self.post = [], []
        self.skipped = 0

    def move(self, pre, post, label, claims=None):
        """pre is taken as given; post exactly on the axes a claim names ('r2': x and y, 'z'), on the others the
        double the drift gives if no velocity lands exactly."""
        claims = dict(claims or {})
        fixed = ({0, 1} if "r2" in claims else set()) | ({2} if "z" in claims else set())
        post = [float(c) for c in post]
        v = [velocity_for(pre[a], post[a], self.dt) for a in range(3)]
        for a in range(3):
            if v[a] is None and a not in fixed and pre[a] != post[a]:
                v[a] = (post[a] - pre[a]) / self.dt
                post[a] = pre[a] + self.dt * v[a]
        if any(c is None for c in v):
            self.skipped += 1
            return None
        i = self.add(pre, v, "%s: %s" % (self.tag, label))
        self.post.append(np.asarray(post, dtype=np.float64))
        self.claims.append(dict(claims or {}))
        return i

    def land(self, post, v, label, claims=None):
        """A particle with velocity v whose drift ends exactly on post (pre-drift position from pair_edges.preimage)."""
        pre = [preimage(post[a], v[a], self.dt) for a in range(3)]
        if any(c is None for c in pre) or \
                not np.array_equal(bits_of([p + self.dt * u for p, u in zip(pre, v)]), bits_of(post)):   # -0.0 is not 0.0
            self.skipped += 1
            return None
        i = self.add(pre, v, "%s: %s" % (self.tag, label))
        self.post.append(np.asarray(post, dtype=np.float64))
        self.claims.append(dict(claims or {}))
        return i

    def extend(self, other):
        for k in ("pos", "vel", "label", "claims", "post"):
            getattr(self, k).extend(getattr(other, k))
        self.skipped += other.skipped

    def subset(self, keep):
        out = Edges(self.cfg, self.tag)
        for i in keep:
            for k in ("pos", "vel", "label", "claims", "post"):
                getattr(out, k).append(getattr(self, k)[i])
        return out


class Angles:
    """Golden-angle sequence: particles on one ring stay far apart."""

    def __init__(self, start=0.3):
        self.t = start

    def __call__(self):
        self.t = (self.t + 2.399963229728653) % (2 * math.pi)
        if min(abs(math.sin(self.t)), abs(math.cos(self.t))) < 0.05:   # keep both coordinates away from 0
            return self()
        return self.t


def _ring_point(r, theta):
    return r * math.cos(theta), r * math.sin(theta)


def _xy_exact_or_ring(r2, r, theta):
    if r2 is not None:
        return on_r2(r2, theta)
    return _ring_point(r, theta)


def _pair_move(b, r2_pre, r_pre, r2_post, r_post, pz, z, theta, label, claims):
    """Pre-drift (x, y) on r2_pre (exact) or radius r_pre at angle theta, post-drift on r2_post / r_post a little further
    round the ring (so the path is not radial), z from pz to z."""
    step = 0.04 * NM * 30e-9 / max(r_post if r_post else math.sqrt(r2_post), 1e-12)
    a = _xy_exact_or_ring(r2_pre, r_pre, theta)
    c = _xy_exact_or_ring(r2_post, r_post, theta + step)
    if a is None or c is None:
        b.skipped += 1
        return None
    return b.move((a[0], a[1], pz), (c[0], c[1], z), label, claims)


# ------------------------------------------------------------------ pore builders
def z_scenarios(g, s):
    """(label, pz, z): heights at which the radial masks' other conditions hold and at which they do not."""
    d = 0.05 * NM * s
    zgt_hi = max(g.z_gt, g.z_gt_pore)
    return [("bottom cap", 0.5 * g.oah, 0.5 * g.oah + 0.3 * d), ("top cap", 0.5 * (g.z_cold + g.H), 0.5 * (g.z_cold + g.H) - 0.3 * d),
            ("hot pore", 0.5 * (g.oah + g.z_gb), 0.5 * (g.oah + g.z_gb) + 0.3 * d),
            ("gap", 0.5 * (g.z_gb + g.z_gt), 0.5 * (g.z_gb + g.z_gt) - 0.3 * d),
            ("cold pore", 0.5 * (g.z_gt + g.z_cold), 0.5 * (g.z_gt + g.z_cold) + 0.3 * d),
            ("up across oah", g.oah - d, g.oah + d), ("up across zh3", g.zh3 - d, g.zh3 + d),
            ("down across z_cold", g.z_cold + d, g.z_cold - d), ("down across zc3", g.zc3 + d, g.zc3 - d),
            ("down out of the gap", g.zgb_p + d, g.z_gb - d), ("up out of the gap", g.zgt_m - d, zgt_hi + d)]


def radial_edges(cfg, s):
    """Post-drift r2 and pre-drift pr2 on every radial value, at every z scenario, moving out and in; and (pr2, r2)
    pairs both on values of one family (the masks that read both)."""
    g = cfg.geom
    b = Edges(cfg, "radial")
    ang = Angles(0.1)
    dr = 0.04 * NM * s
    fams = radial_families(g)
    for zl, pz, z in z_scenarios(g, s):
        for fam, vals in fams.items():
            for T, lab in vals:
                R = math.sqrt(T)
                for sgn, way in ((1, "out"), (-1, "in")):
                    _pair_move(b, None, R - sgn * dr, T, None, pz, z, ang(), "r2=%s (moving %s), %s" % (lab, way, zl),
                               {"r2": T})
                    _pair_move(b, T, None, None, R + sgn * dr, pz, z, ang(), "pr2=%s (moving %s), %s" % (lab, way, zl),
                               {"pr2": T})
            for i, (T0, l0) in enumerate(vals):
                for T1, l1 in vals[i + 1:]:
                    lo, hi = (T0, l0), (T1, l1)
                    if T1 < T0:
                        lo, hi = hi, lo
                    for (A, la), (B, lb) in ((lo, hi), (hi, lo)):
                        _pair_move(b, A, None, B, None, pz, z, ang(), "pr2=%s, r2=%s, %s" % (la, lb, zl), {"pr2": A, "r2": B})
    return b


def radii_options(g, s):
    """(label, r_pre, r_post) for z-threshold particles: static radii between the walls and paths across each wall."""
    d = 0.03 * NM * s
    Rpc, Rgc = math.sqrt(g.R_p_c_sq), math.sqrt(g.R_g_c_sq)
    static = [("axis", 0.3 * Rpc), ("R_p_c..R_p", 0.5 * (Rpc + g.R_p)), ("R_p..R_g_c", 0.5 * (g.R_p + Rgc)),
              ("R_g_c..R_g", 0.5 * (Rgc + g.R_g)), ("R_g..R_oa", 2.0 * g.R_p)]
    out = [(lab, r, r) for lab, r in static]
    for lab, R in (("R_p_c", Rpc), ("R_p", g.R_p), ("R_g_c", Rgc), ("R_g", g.R_g), ("R_oa", g.R_oa)):
        out += [("out across " + lab, R - d, R + d), ("in across " + lab, R + d, R - d)]
    return out


def z_edges(cfg, s):
    """Post-drift z and pre-drift pz on every z value (z_values), each from above and from below, at every radius option."""
    g = cfg.geom
    b = Edges(cfg, "z")
    ang = Angles(0.7)
    d = 0.05 * NM * s
    for zv, zl in z_values(g):
        for side, sg in (("from above", 1.0), ("from below", -1.0)):
            other = zv + sg * d
            for rl, r0, r1 in radii_options(g, s):
                _pair_move(b, None, r0, None, r1, other, zv, ang(), "z=%s %s, %s" % (zl, side, rl), {"z": zv})
                _pair_move(b, None, r0, None, r1, zv, zv - sg * d, ang(), "pz=%s moving %s, %s" % (zl, "down" if sg > 0 else "up", rl),
                           {"pz": zv})
    return b


def calm_edges(cfg, s):
    """Temp: pre- and post-drift z on calm_zA, calm_zB, 0 and H and the doubles next to them, with rmax on calm_rA and
    calm_rC and the doubles next to them, crossing R_p_c (so 6H / 6C can fire) or staying on one radius."""
    g = cfg.geom
    zA, zB, rA, rC = calm_bounds(g)
    b = Edges(cfg, "calm")
    ang = Angles(1.3)
    d = 0.05 * NM * s
    zs = []
    for P, lab in ((zA, "calm_zA"), (zB, "calm_zB"), (0.0, "0"), (float(g.H), "H")):
        zs += [(float(down(P)), "prev(%s)" % lab), (P, lab), (float(up(P)), "next(%s)" % lab)]
    rs = []
    for T, lab in ((rA, "calm_rA"), (rC, "calm_rC")):
        rs += [(float(down(T)), "prev(%s)" % lab), (T, lab), (float(up(T)), "next(%s)" % lab)]
    for zv, zl in zs:
        inside = zv - d if zv > 0.5 * g.H else zv + d        # the other end of the path inside the domain
        for T, rl in rs:
            R = math.sqrt(T)
            for pre_z, post_z, how in ((inside, zv, "z"), (zv, inside, "pz")):
                _pair_move(b, None, R - 0.03 * NM * s, T, None, pre_z, post_z, ang(), "%s=%s, r2=%s" % (how, zl, rl),
                           {how: zv, "r2": T})
                _pair_move(b, T, None, None, R - 0.03 * NM * s, pre_z, post_z, ang(), "%s=%s, pr2=%s" % (how, zl, rl),
                           {how: zv, "pr2": T})
        # the same heights crossing the pore's contact radius: 6H at z == zh3 == calm_zA is one of these
        Rpc = math.sqrt(g.R_p_c_sq)
        for pre_z, post_z, how in ((inside, zv, "z"), (zv, inside, "pz")):
            _pair_move(b, g.R_p_c_sq, None, None, Rpc + 0.03 * NM * s, pre_z, post_z, ang(), "%s=%s, out across R_p_c" % (how, zl),
                       {how: zv, "pr2": g.R_p_c_sq})
    return b


def degenerate_edges(cfg, s):
    """Side-wall hits the contact cannot be found for, and rewind times outside [0, dt]:
    - vx = vy = 0 outside the open-air radius (a == 0), on r2 = gt_Roa + 1ulp and further out;
    - tangential paths outside the open-air radius whose line never meets R_oa_c (disc < 0);
    - paths starting exactly on a contact radius (pr2 == R_g_c_sq / R_p_c_sq) and leaving it tangentially: disc at
      the rounding limit, in the gap (case 4) and at the hot / cold coatings (6H / 6C);
    - particles outside R_oa moving inwards (both rewind roots negative) and crossing R_oa from between R_oa_c and
      R_oa (rewind time beyond dt)."""
    g = cfg.geom
    b = Edges(cfg, "degenerate")
    ang = Angles(2.1)
    s_nm = NM * s
    zs = [("bottom cap", 0.5 * g.oah), ("top cap", 0.5 * (g.z_cold + g.H)), ("gap", 0.5 * (g.z_gb + g.z_gt)),
          ("hot coating", 0.5 * (g.zh3 + g.zgb_p)), ("cold coating", 0.5 * (g.zgt_m + g.zc3))]
    gt_oa = sq_threshold_gt(g.R_oa)
    for zl, z in zs:
        for T, lab in ((float(up(gt_oa)), "gt_R_oa+1ulp"), ((g.R_oa + 0.5 * s_nm) ** 2, "R_oa+0.5nm")):
            p = on_r2(T, ang())
            if p is not None:
                b.move((p[0], p[1], z), (p[0], p[1], z + 0.01 * s_nm), "a == 0, r2=%s, %s" % (lab, zl), {"r2": T, "pr2": T})
        for frac in (0.3, 0.6, 0.9):           # closest approach between R_oa_c and R_oa: the line misses R_oa_c
            dist = g.R_oa_c + frac * (g.R_oa - g.R_oa_c)
            th = ang()
            n = np.array([math.cos(th), math.sin(th)])
            t = np.array([-n[1], n[0]])
            along = math.sqrt(g.R_oa ** 2 - dist ** 2) + 0.02 * s_nm
            post = dist * n + along * t
            pre = post - 0.05 * s_nm * t
            b.move((pre[0], pre[1], z), (post[0], post[1], z), "disc < 0, closest approach %.1f of R_oa - R_oa_c, %s" % (frac, zl))
        for T, lab in ((g.R_g_c_sq, "R_g_c_sq"), (g.R_p_c_sq, "R_p_c_sq")):
            p = on_r2(T, ang())
            if p is None:
                continue
            r = math.sqrt(T)
            tang = np.array([-p[1], p[0]]) / r
            for k in (0.01, 0.05):
                post = np.array(p) + k * s_nm * tang
                b.move((p[0], p[1], z), (post[0], post[1], z - 0.01 * s_nm), "tangential from pr2=%s by %.2f nm, %s" % (lab, k, zl),
                       {"pr2": T})
        th = ang()
        out = _ring_point(g.R_oa + 1.0 * s_nm, th)
        inw = _ring_point(g.R_oa + 0.9 * s_nm, th + 1e-4)
        b.move((out[0], out[1], z), (inw[0], inw[1], z), "outside R_oa moving inwards (t < 0), %s" % zl)
        th = ang()
        a0 = _ring_point(0.5 * (g.R_oa_c + g.R_oa), th)
        a1 = _ring_point(g.R_oa + 0.02 * s_nm, th + 1e-4)
        b.move((a0[0], a0[1], z), (a1[0], a1[1], z), "from between R_oa_c and R_oa (t > dt), %s" % zl)
    return b


def recapture_edges(cfg, s):
    """Particles at rest (nothing for the walls to do) on the recapture's and the census's thresholds: r2 on R_oa_sq,
    R_g_sq, R_p_sq (and the doubles next to them) at every z value, and at the heights between."""
    g = cfg.geom
    b = Edges(cfg, "recapture")
    ang = Angles(2.9)
    rs = []
    for T, lab in ((g.R_oa_sq, "R_oa_sq"), (g.R_g_sq, "R_g_sq"), (g.R_p_sq, "R_p_sq")):
        rs += [(float(down(T)), "prev(%s)" % lab), (float(T), lab), (float(up(T)), "next(%s)" % lab)]
    zs = [(z, l) for z, l in z_values(g) if 0.0 <= z <= g.H] + [(0.5 * (g.oah + g.z_gb), "hot pore"), (0.5 * (g.z_gb + g.z_gt), "gap"),
                                                               (0.5 * (g.z_gt + g.z_cold), "cold pore"), (0.5 * g.oah, "bottom cap")]
    for z, zl in zs:
        for T, rl in rs:
            p = on_r2(T, ang())
            if p is not None:
                b.move((p[0], p[1], z), (p[0], p[1], z), "at rest, r2=%s, z=%s" % (rl, zl), {"r2": T, "pr2": T, "z": z, "pz": z})
    return b


def gap_energy_edges(cfg, s):
    """Case 4 (Temp) hits with contact heights next to zgb_p and zgt_m, down to z_gb - 0.9a and up to z_gt + 0.9a: a
    radial path across the contact radius R_g_c, pz inside the open gap interval, z chosen so the contact falls on the
    target height."""
    g = cfg.geom
    b = Edges(cfg, "gap energy")
    ang = Angles(0.45)
    a = g.argon_radius
    Rgc = math.sqrt(g.R_g_c_sq)
    d = 0.02 * NM * s
    targets = [(g.zgb_p, "zgb_p"), (float(up(g.zgb_p)), "next(zgb_p)"), (g.zgb_p - 0.5 * a, "zgb_p - a/2"), (g.z_gb, "z_gb"),
               (g.z_gb - 0.9 * a, "z_gb - 0.9a"), (g.zgt_m, "zgt_m"), (float(down(g.zgt_m)), "prev(zgt_m)"),
               (g.zgt_m + 0.5 * a, "zgt_m + a/2"), (g.z_gt, "z_gt"), (g.z_gt + 0.9 * a, "z_gt + 0.9a")]
    for zc, lab in targets:
        for pz, how in ((float(up(g.zgb_p)), "pz=next(zgb_p)"), (g.zgb_p + 0.05 * a, "pz above zgb_p"),
                        (float(down(g.zgt_m)), "pz=prev(zgt_m)"), (g.zgt_m - 0.05 * a, "pz below zgt_m")):
            # radial path Rgc - d -> Rgc + d crosses the contact radius halfway: contact height = (pz + z) / 2
            z = 2.0 * zc - pz
            if abs(z - pz) > 6 * a:
                continue
            th = ang()
            p0, p1 = _ring_point(Rgc - d, th), _ring_point(Rgc + d, th)
            b.move((p0[0], p0[1], pz), (p1[0], p1[1], z), "case 4 contact near %s, %s" % (lab, how), {"pz": pz})
    return b


def corner_candidates(cfg, s, rng, n=160):
    """Paths aimed through the places where two or more wall cases can fire in one step: (label, pre-drift radius
    range, post-drift radius range, plane); each path crosses the plane or starts / ends on it."""
    g = cfg.geom
    b = Edges(cfg, "corner")
    d = 0.12 * NM * s
    Rpc, Rgc = math.sqrt(g.R_p_c_sq), math.sqrt(g.R_g_c_sq)
    corners = [("open-air rim, bottom", (g.R_oa - d, g.R_oa), (g.R_oa, g.R_oa + d), 0.0),
               ("open-air rim, top", (g.R_oa - d, g.R_oa), (g.R_oa, g.R_oa + d), g.H),
               ("gap lip, bottom", (Rgc - d, Rgc), (Rgc, g.R_g + d), g.zgb_p), ("gap lip, top", (Rgc - d, Rgc), (Rgc, g.R_g + d), g.zgt_m),
               ("gap lip R_g, bottom", (g.R_g - d, g.R_g), (g.R_g, g.R_g + d), g.z_gb),
               ("gap lip R_g, top", (g.R_g - d, g.R_g), (g.R_g, g.R_g + d), g.z_gt_pore),
               ("pore mouth, bottom", (Rpc - d, Rpc), (g.R_p, g.R_p + d), g.zh3), ("pore mouth, top", (Rpc - d, Rpc), (g.R_p, g.R_p + d), g.zc3),
               ("pore mouth oah", (g.R_p - d, g.R_p), (g.R_p, g.R_p + d), g.oah),
               ("pore mouth z_cold", (g.R_p - d, g.R_p), (g.R_p, g.R_p + d), g.z_cold)]
    ang = Angles(0.9)
    for lab, (a0, a1), (c0, c1), Z in corners:
        for _ in range(n):
            th = ang()
            r0, r1 = rng.uniform(a0, a1), rng.uniform(c0, c1)
            z0, z1 = Z + rng.uniform(-1.0, 1.0) * d, Z + rng.uniform(-1.0, 1.0) * d
            if rng.random() < 0.3:     # start or end exactly on the plane
                if rng.random() < 0.5:
                    z0 = Z
                else:
                    z1 = Z
            p0, p1 = _ring_point(r0, th), _ring_point(r1, th + rng.uniform(-2, 2) * d / r1)
            b.move((p0[0], p0[1], z0), (p1[0], p1[1], z1), lab)
    return b


def pp_push_candidates(cfg, s, rng, n=120):
    """Overlapping, approaching pairs next to the end plates and the cylinder walls (each pair far from every other):
    the pair pass can push one of them out of bounds."""
    g = cfg.geom
    b = Edges(cfg, "pair push")
    cr = g.collision_range
    ang = Angles(1.7)
    places = [("z=0", lambda th, u: (0.4 * g.R_oa * math.cos(th), 0.4 * g.R_oa * math.sin(th), u * cr), (0, 0, -1)),
              ("z=H", lambda th, u: (0.4 * g.R_oa * math.cos(th), 0.4 * g.R_oa * math.sin(th), g.H - u * cr), (0, 0, 1)),
              ("R_oa", lambda th, u: ((g.R_oa - u * cr) * math.cos(th), (g.R_oa - u * cr) * math.sin(th), 0.5 * g.oah), None),
              ("R_p hot", lambda th, u: ((g.R_p - u * cr) * math.cos(th), (g.R_p - u * cr) * math.sin(th), 0.5 * (g.oah + g.z_gb)), None),
              ("R_g gap", lambda th, u: ((g.R_g - u * cr) * math.cos(th), (g.R_g - u * cr) * math.sin(th), 0.5 * (g.z_gb + g.z_gt)), None),
              ("R_p cold", lambda th, u: ((g.R_p - u * cr) * math.cos(th), (g.R_p - u * cr) * math.sin(th), 0.5 * (g.z_gt + g.z_cold)), None)]
    for lab, where, normal in places:
        for k in range(n):
            th = ang()
            u = rng.uniform(0.05, 1.2)
            p = np.array(where(th, u))
            out = np.array(normal, dtype=np.float64) if normal else np.array([math.cos(th), math.sin(th), 0.0])
            dvec = rng.normal(size=3)
            dvec = dvec / np.linalg.norm(dvec)
            q = p + 0.6 * cr * dvec
            speed = rng.uniform(300.0, 1500.0)
            va = speed * out + rng.normal(size=3) * 100.0
            vb = va - 400.0 * dvec                  # b approaches a
            for pos, v, who in ((p, va, "a"), (q, vb, "b")):
                b.add(pos, v, "%s: %s, pair %d (%s)" % (b.tag, lab, k, who))
                b.post.append(pos + cfg.dt * v)
                b.claims.append({})
    return b


def cube_edges(cfg):
    """Cube: post-drift coordinates on L, 0, -0.0 and one double beyond each face, one axis at a time, on edges (two
    axes) and corners (three axes), each reached by an outward (or, on the face, resting) velocity."""
    b = Edges(cfg, "cube")
    L = [cfg.cube_x, cfg.cube_y, cfg.cube_z]
    rng = np.random.default_rng(5)

    def face_values(a):
        return [(float(L[a]), "L", 1), (float(up(L[a])), "next(L)", 1), (0.0, "0", -1), (-0.0, "-0.0", -1), (float(down(0.0)), "prev(0)", -1),
                (-1e-3 * NM, "-1e-12", -1), (L[a] + 1e-3 * NM, "L+1e-12", 1)]
    for na in (1, 2, 3):
        for axes in itertools.combinations(range(3), na):
            choices = [face_values(a) for a in axes]
            for combo in itertools.product(*choices):
                for rep in range(2 if na < 3 else 1):
                    post = [rng.uniform(0.2, 0.8) * L[a] for a in range(3)]
                    v = list(rng.normal(size=3) * 300.0)
                    lab = []
                    for a, (val, vl, sgn) in zip(axes, combo):
                        post[a] = val
                        v[a] = sgn * abs(v[a]) * (1 + rep)
                        lab.append("%s=%s" % ("xyz"[a], vl))
                    i = b.land(post, v, ", ".join(lab), {"xyz"[a]: val for a, (val, _, _) in zip(axes, combo)})
                    if i is None:           # no pre-image from inside: start on the face itself (0, -0.0 or L)
                        b.skipped -= 1
                        pre = [preimage(post[a], v[a], cfg.dt) for a in range(3)]
                        for a, (val, _, sgn) in zip(axes, combo):
                            pre[a] = float(L[a]) if sgn > 0 else math.copysign(0.0, val)
                            v[a] = velocity_for(pre[a], val, cfg.dt)
                        if any(c is None for c in pre + v):
                            b.skipped += 1
                            continue
                        b.add(pre, v, "%s: %s (from the face)" % (b.tag, ", ".join(lab)))
                        b.post.append(np.asarray(post, dtype=np.float64))
                        b.claims.append({"xyz"[a]: val for a, (val, _, _) in zip(axes, combo)})
    return b


# ------------------------------------------------------------------ oracle filters
CORNERS = {
    # Open-air pore: a case 3 plane hit reflects the particle back out of the z range of case 6, so the pore mouth is
    # no corner there (corner_candidates aims at it all the same)
    "pore": {"open-air rim (1 + 2A/2B)": (0, (1, 2)), "gap lip (4 + 5/6)": (5, (6, 7, 8))},
    "temp": {"open-air rim (1 + 2A/2B)": (0, (1, 2)), "gap lip (4 + 5B/5T)": (5, (6, 7)), "pore mouth (3C/3H + 6C/6H)": ((3, 4), (8, 9))},
}


def corner_kinds(kind, bits):
    """Names of the CORNERS combinations present in each hit-bit word."""
    out = []
    for name, (a, bb) in CORNERS[kind].items():
        a = (a,) if isinstance(a, int) else a
        ma = sum(1 << c for c in a)
        mb = sum(1 << c for c in bb)
        out.append((name, ((bits & ma) != 0) & ((bits & mb) != 0)))
    return out


def oracle_walls(oracle, cfg, b, seed=17, step=0, cheb=None):
    """Drift and wall phase of the oracle on the built state: (state, hit bits, counts, errors)."""
    st = oracle.ParticleState(*b.arrays())
    oracle.drift(st, cfg.dt, True)
    if cfg.kind == "temp":
        counts, _, errs, bits = oracle.temp_walls_philox(st, cfg.geom, seed, step, cheb if cheb is not None else cheb_of(cfg), None, True)
    else:
        counts, errs, bits = oracle.pore_walls(st, cfg.geom, None, True)
    return st, bits, counts, errs


_CHEB = {}


def cheb_of(cfg):
    from argon_monte_carlo_b200 import config
    key = (cfg.kind, float(cfg.pore_coated_radius))
    if key not in _CHEB:
        _CHEB[key] = config.gap_energy_chebyshev(cfg, 16)
    return _CHEB[key]


def keep_corners(oracle, cfg, b):
    """The candidates whose oracle hit bits have two or more bits set."""
    _, bits, _, _ = oracle_walls(oracle, cfg, b)
    keep = [i for i in range(len(b.pos)) if bin(int(bits[i])).count("1") >= 2]
    return b.subset(keep)


def oob_rows(g, kind, x, y, z):
    """Per particle: is it out of bounds for the recapture of the script (Pore: num_out_of_bounds, Temp: its census)."""
    r2 = r2k(x, y)
    if kind == "temp":
        return (z < 0) | (z > g.H) | ((r2 > g.R_oa_sq) & (z >= 0) & (z <= g.oah)) | ((r2 > g.R_oa_sq) & (z >= g.z_cold) & (z <= g.H)) | \
            ((r2 > g.R_g_sq) & (z >= g.z_gb) & (z <= g.z_gt)) | ((r2 > g.R_p_sq) & (z > g.oah) & (z < g.z_gb)) | \
            ((r2 > g.R_p_sq) & (z > g.z_gt) & (z < g.z_cold))
    return (z < 0) | (z > g.H) | (r2 > g.R_oa_sq) | ((r2 > g.R_g_sq) & (z > g.oah) & (z < g.z_cold)) | \
        ((r2 > g.R_p_sq) & (((z > g.oah) & (z < g.z_gb)) | ((z > g.z_gt) & (z < g.z_cold))))


def keep_pp_pushes(oracle, cfg, b):
    """The pairs one of which is out of bounds after the oracle's pair pass (before the closing recapture)."""
    g = cfg.geom
    st, _, _, _ = oracle_walls(oracle, cfg, b)
    (oracle.temp_recapture if cfg.kind == "temp" else oracle.pore_recapture)(st, g)
    oracle.pp_groups(st, cfg.grid, cfg.collision_range, cfg.argon_mass)
    bad = oob_rows(g, cfg.kind, st.x, st.y, st.z)
    keep = []
    for i in range(0, len(b.pos), 2):
        if bad[i] or bad[i + 1]:
            keep += [i, i + 1]
    return b.subset(keep)


# ------------------------------------------------------------------ whole states
def pore_edges(oracle, cfg, scale):
    """Every pore builder for one config (Pore or Temp), concatenated."""
    rng = np.random.default_rng(11)
    b = Edges(cfg, "all")
    parts = [radial_edges(cfg, scale), z_edges(cfg, scale), degenerate_edges(cfg, scale), recapture_edges(cfg, scale)]
    if cfg.kind == "temp":
        parts += [calm_edges(cfg, scale), gap_energy_edges(cfg, scale)]
    parts += [keep_corners(oracle, cfg, corner_candidates(cfg, scale, rng)), keep_pp_pushes(oracle, cfg, pp_push_candidates(cfg, scale, rng))]
    for p in parts:
        b.extend(p)
    return b


def with_gas(b, gas, every=2):
    """(arrays, labels): the edge particles of b interleaved by id with the gas (x, y, z, vx, vy, vz): edge particle i
    at id every*i, gas particles in the slots between and after."""
    arrs = b.arrays()
    ne, ng = len(arrs[0]), len(gas[0])
    n = ne + ng
    is_edge = np.zeros(n, dtype=bool)
    is_edge[np.arange(ne) * every if ne * every <= n else np.linspace(0, n - 1, ne).astype(np.int64)] = True
    out = []
    for e, gv in zip(arrs, gas):
        a = np.empty(n)
        a[is_edge] = e
        a[~is_edge] = np.asarray(gv)[:ng]
        out.append(a)
    labels = np.empty(n, dtype=object)
    labels[is_edge] = b.label
    labels[~is_edge] = "gas"
    return tuple(out), list(labels)


def bench_scale():
    import bench
    return bench.scaled_temp_config(12_500_000)[1]


def pore_cfg_of(kind, scale_name):
    """(config, scale) for kind 'pore' / 'temp' and scale '1' / 'bench' / '0.5'."""
    from argon_monte_carlo_b200 import config
    if kind == "temp" and scale_name == "bench":
        import bench
        return bench.scaled_temp_config(12_500_000)
    s = {"1": 1.0, "0.5": 0.5}.get(scale_name) or bench_scale()
    return config.pore_config(kind == "temp", scale=s), s


def cube_cfg_of(scale_name):
    """Cube configs on grids with an even cell count (colour groups and the serial sweep both run on them): 14 cells of
    7.1 nm at scale 1, 8 cells of 25 nm at scale 2."""
    from argon_monte_carlo_b200 import config
    return config.cube_config(1.0, 14) if scale_name == "1" else config.cube_config(2.0, 8)
