"""States placed on the floating-point boundaries of the pair pass (test infrastructure only; plain NumPy plus the oracle).

Every decision the pair pass makes is a comparison with a table value or a threshold: the owner cell
(edge[k] <= v < edge[k+1], a division estimate checked against the table), the membership of a reference cell
(lo[k] < v < edge[k+1], strict on both sides, Pore:527-529), the band prefix of the sort (v > lo[k+1]) and the overlap
test (d2 < overlap_sq, Pore:173-174) behind an fp32 filter (det_thr).  Gas states reach these boundaries with a
probability close to zero; the builders here put particles on them exactly and check that they did.

- ``boundary_values``: edge[k], lo[k] and the doubles next to each, the virtual layer below edge[0], the last double
  of the grid, -0.0 where 0.0 is an edge, labelled.
- ``estimate_misses``: the edges at which the kernels' fast owner estimate floor((v - e0) * inv_d) is wrong.
- ``partner_at``: a partner at an exact squared distance (evaluated in the kernels' order) from an anchor.
- ``preimage``: a start position that the drift (x += dt * v) maps exactly onto a target.
- lattices, threshold-pair cells and capacity cells built from these, each with the pairs it means to collide.
"""
from __future__ import annotations

import math

import numpy as np

from argon_monte_carlo_b200 import amc

V_APPROACH = 200.0   # m/s: relative speed of a constructed pair, along the line of centres, approaching


# ------------------------------------------------------------------ scalars
def d2_kernel(a, b):
    """Squared distance as the kernels and the oracle evaluate it: (dx*dx + dy*dy) + dz*dz, d = b - a."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    d = b - a
    return (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]


def overlap_sq(cr):
    return amc.overlap_threshold(cr)


def det_thr(grid, cr):
    """fp32 threshold of the detection filter, restated from amc_api.cu (as test_detection_filter_threshold_is_conservative)."""
    wmax = max(float(np.max(grid.edge[a][1:] - grid.lo[a])) for a in range(3))
    e_abs = 6.0 * math.ldexp(wmax, -24)
    r_f = math.sqrt(overlap_sq(cr)) * (1.0 + 1e-9) + 2.0 * e_abs
    return np.nextafter(np.float32(r_f * r_f * (1.0 + math.ldexp(1.0, -20))), np.float32(np.inf))


def filter_d2(a, b, lo):
    """fp32 squared distance of the detection filter on cell-relative coordinates (k_detect_tma: fmaf(ez, ez,
    fmaf(ey, ey, ex * ex))).  Each fused step is emulated as an exact product plus a double-precision add, then one
    rounding to fp32; that can differ from the hardware by one fp32 ulp at a tie, which callers leave margin for."""
    fa = (np.asarray(a, dtype=np.float64) - lo).astype(np.float32)
    fb = (np.asarray(b, dtype=np.float64) - lo).astype(np.float32)
    e = (fb - fa).astype(np.float64)
    s = (e[..., 0] * e[..., 0]).astype(np.float32).astype(np.float64)
    s = (e[..., 1] * e[..., 1] + s).astype(np.float32).astype(np.float64)
    return (e[..., 2] * e[..., 2] + s).astype(np.float32)


def nudge(v, k):
    """v moved by k doubles (k > 0: towards +inf); v and every step stay on one side of zero."""
    v = np.asarray(v, dtype=np.float64)
    k = np.asarray(k, dtype=np.int64)
    iv = v.view(np.int64)
    return np.where(v > 0, iv + k, iv - k).view(np.float64)


def up(v):
    return np.nextafter(v, np.inf)


def down(v):
    return np.nextafter(v, -np.inf)


# ------------------------------------------------------------------ boundaries
def owner_estimate(grid, a, v):
    """The kernels' fast owner estimate (owner_axis): floor((v - e0) * inv_d), clamped to the grid."""
    e = grid.edge[a]
    nc = grid.nc[a]
    inv_d = float(nc) / (e[nc] - e[0])
    est = np.floor((np.asarray(v, dtype=np.float64) - e[0]) * inv_d).astype(np.int64)
    return np.clip(est, 0, nc - 1)


def owner_exact(grid, a, v):
    """edge[k] <= v < edge[k+1]: -1 below edge[0], nc at or above edge[nc]."""
    return np.searchsorted(grid.edge[a], np.asarray(v, dtype=np.float64), side="right") - 1


def estimate_misses(grid, a):
    """{'on': edges k (0 < k < nc) where v = edge[k] gets an estimate != k, 'below': where v = prev(edge[k]) gets an
    estimate != k - 1}: the coordinates at which owner_axis has to fall back to owner_axis_slow."""
    e, nc = grid.edge[a], grid.nc[a]
    k = np.arange(1, nc)
    on = k[owner_estimate(grid, a, e[1:nc]) != k]
    below = k[owner_estimate(grid, a, down(e[1:nc])) != k - 1]
    return {"on": on.tolist(), "below": below.tolist()}


def boundary_values(grid, a, ks=None):
    """[(value, label)] on axis a: for every edge k in ks (default: all), edge[k], lo[k] (k < nc) and the doubles on
    either side of each; plus the virtual owner layer (edge[0], lo[0] and between), prev(edge[nc]) and -0.0 where 0.0
    is an edge."""
    e, lo, nc = grid.edge[a], grid.lo[a], grid.nc[a]
    ks = range(nc + 1) if ks is None else ks
    out = []
    for k in ks:
        out += [(e[k], "edge[%d]" % k), (down(e[k]), "prev(edge[%d])" % k), (up(e[k]), "next(edge[%d])" % k)]
        if k < nc:
            out += [(lo[k], "lo[%d]" % k), (down(lo[k]), "prev(lo[%d])" % k), (up(lo[k]), "next(lo[%d])" % k)]
        if e[k] == 0.0:
            out.append((-0.0, "-0.0 (edge[%d])" % k))
    if 0 in ks:
        out.append((0.5 * (lo[0] + e[0]), "virtual layer below edge[0]"))
    return out


def check_boundary_values(grid, a, vals):
    """Every value is the boundary its label names (raises AssertionError otherwise)."""
    e, lo = grid.edge[a], grid.lo[a]
    for v, lab in vals:
        if lab.startswith("virtual"):
            assert lo[0] < v < e[0], lab
            continue
        if lab.startswith("-0.0"):
            assert v == 0.0 and math.copysign(1.0, v) < 0, lab
            continue
        tab, k = (e, int(lab.split("[")[1].split("]")[0]))
        if "lo[" in lab:
            tab = lo
        ref = tab[k]
        want = {"prev": down(ref), "next": up(ref)}.get(lab.split("(")[0], ref)
        assert v == want and np.float64(v).view(np.int64) == np.float64(want).view(np.int64), lab


def member_cells(grid, p):
    """Reference cells (kx, ky, kz) that position p is a member of: lo[k] < v < edge[k+1] on every axis."""
    ks = [[k for k in range(grid.nc[a]) if grid.lo[a][k] < p[a] < grid.edge[a][k + 1]] for a in range(3)]
    return {(i, j, k) for i in ks[0] for j in ks[1] for k in ks[2]}


# ------------------------------------------------------------------ pairs
def unit(v):
    v = np.asarray(v, dtype=np.float64)
    return v / np.linalg.norm(v)


def partner_at(anchor, direction, target, reach=20):
    """Partner p near anchor + sqrt(target) * direction with d2_kernel(anchor, p) == target exactly, or None.

    One double more or less in a coordinate moves d2 by about 2 |d_i| ulp(p_i), which can be thousands of ulps of d2
    far from the origin.  So the two coarser coordinates are moved by up to `reach` doubles each, and for every such
    choice the finest coordinate is solved for and its neighbours tried; the hit closest to the start wins."""
    anchor = np.asarray(anchor, dtype=np.float64)
    p0 = anchor + math.sqrt(target) * unit(direction)
    d0 = p0 - anchor
    ulp = np.abs(np.spacing(p0))
    step = np.abs(2.0 * d0 * ulp) / np.spacing(np.float64(target))      # ulps of d2 per double of each coordinate
    usable = [i for i in range(3) if p0[i] != 0.0 and step[i] > 0.05]
    if not usable:
        return None
    f = min(usable, key=lambda i: step[i])
    others = [i for i in range(3) if i != f]
    r = np.arange(-reach, reach + 1)
    offs = [r if (p0[i] != 0.0 and step[i] > 0.05) else np.zeros(1, dtype=np.int64) for i in others]
    A, B = np.meshgrid(offs[0], offs[1], indexing="ij")
    A, B = A.ravel(), B.ravel()
    P = np.repeat(p0[None, :], len(A), axis=0)
    P[:, others[0]] = nudge(np.full(len(A), p0[others[0]]), A)
    P[:, others[1]] = nudge(np.full(len(A), p0[others[1]]), B)
    base = d2_kernel(anchor, P)
    sign = np.sign(d0[f]) * np.sign(p0[f])                      # d2 grows with +k when |d_f| grows
    kf = np.rint((target - base) / (step[f] * np.spacing(np.float64(target))) * sign).astype(np.int64)
    best, best_cost = None, None
    for dk in (0, -1, 1, -2, 2, -3, 3):
        Q = P.copy()
        Q[:, f] = nudge(np.full(len(A), p0[f]), kf + dk)
        hit = np.flatnonzero(d2_kernel(anchor, Q) == target)
        if len(hit):
            cost = np.abs(A[hit]) + np.abs(B[hit]) + np.abs(kf[hit] + dk)
            h = hit[np.argmin(cost)]
            if best is None or cost.min() < best_cost:
                best, best_cost = Q[h].copy(), cost.min()
    return best


def approaching(v_anchor, anchor, partner, speed=V_APPROACH):
    """Velocity of the partner: the anchor's minus `speed` along the line of centres (the pair closes in)."""
    return np.asarray(v_anchor, dtype=np.float64) - speed * unit(np.asarray(partner) - np.asarray(anchor))


# ------------------------------------------------------------------ drift pre-images
def preimage(target, v, dt, reach=6):
    """x0 with fl(x0 + fl(dt * v)) == target (the oracle's and the kernels' drift), the closest such double to
    target - dt * v; None if none within `reach` doubles of it works."""
    ax = dt * v
    lo = hi = target - ax
    cands = [lo]
    for _ in range(reach):
        lo, hi = float(down(lo)), float(up(hi))
        cands += [lo, hi]
    for c in cands:
        if c + ax == target:
            return c
    return None


class State:
    """Particles under construction: positions, velocities, a label per particle and the pairs meant to collide."""

    def __init__(self):
        self.pos, self.vel, self.label = [], [], []
        self.collide, self.miss = [], []   # (i, j) index pairs: meant to overlap / meant to sit at exactly overlap_sq

    def add(self, p, v, label):
        self.pos.append(np.asarray(p, dtype=np.float64))
        self.vel.append(np.asarray(v, dtype=np.float64))
        self.label.append(label)
        return len(self.pos) - 1

    def add_pair(self, anchor, direction, target, v_anchor, label, collide):
        """Anchor plus a partner at squared distance `target` (the caller picks prev(overlap_sq) or overlap_sq)."""
        p = partner_at(anchor, direction, target)
        if p is None:
            return None
        i = self.add(anchor, v_anchor, label + " (anchor)")
        j = self.add(p, approaching(v_anchor, anchor, p), label + " (partner)")
        (self.collide if collide else self.miss).append((i, j))
        return i, j

    def arrays(self):
        pos = np.array(self.pos).reshape(-1, 3)
        vel = np.array(self.vel).reshape(-1, 3)
        return (pos[:, 0].copy(), pos[:, 1].copy(), pos[:, 2].copy(), vel[:, 0].copy(), vel[:, 1].copy(), vel[:, 2].copy())

    def pair_keys(self, which):
        return {(max(i, j), min(i, j)) for i, j in (self.collide if which == "collide" else self.miss)}

    def expected(self, grid):
        """The pairs meant to collide that share a reference cell (lo[k] < v < edge[k+1] on every axis, Pore:527-529):
        a pair placed outside the grid is never tested."""
        return {k for k in self.pair_keys("collide") if member_cells(grid, self.pos[k[0]]) & member_cells(grid, self.pos[k[1]])}

    def drift_preimages(self, dt):
        """Replace every position by its drift pre-image so that one drift lands on the constructed position exactly.
        A pair with a particle that has no pre-image is dropped (with both its particles).  Returns the number of
        particles dropped and the original indices of those kept."""
        n = len(self.pos)
        pre = [None] * n
        for i in range(n):
            q = [preimage(self.pos[i][a], self.vel[i][a], dt) for a in range(3)]
            pre[i] = None if any(c is None for c in q) else np.array(q)
        bad = {i for i in range(n) if pre[i] is None}
        for i, j in self.collide + self.miss:
            if i in bad or j in bad:
                bad |= {i, j}
        keep = [i for i in range(n) if i not in bad]
        remap = {old: new for new, old in enumerate(keep)}
        self.pos = [pre[i] for i in keep]
        self.vel = [self.vel[i] for i in keep]
        self.label = [self.label[i] for i in keep]
        self.collide = [(remap[i], remap[j]) for i, j in self.collide if i in remap and j in remap]
        self.miss = [(remap[i], remap[j]) for i, j in self.miss if i in remap and j in remap]
        if hasattr(self, "_grid"):
            self._grid = {}
            for i, p in enumerate(self.pos):
                self._grid.setdefault(self._key(p), []).append(i)
        return len(bad), keep


# ------------------------------------------------------------------ lattices
KINDS = (("+", True), ("+", False), ("-", True), ("-", False))   # (side of the boundary, partner at prev(osq) or at osq)


class Builder(State):
    """State with a clearance rule: a pair is only added if both its particles keep 2.5 collision ranges from every
    particle already placed, so the constructed pairs are the only ones that can interact."""

    def __init__(self, cr):
        super().__init__()
        self.cr = cr
        self.osq = overlap_sq(cr)
        self.skipped = 0
        self._grid = {}

    def _key(self, p):
        return tuple(np.floor(np.asarray(p) / (2.5 * self.cr)).astype(np.int64).tolist())

    def _clear(self, pts):
        for p in pts:
            k = self._key(p)
            for dx in (-1, 0, 1):
                for dy in (-1, 0, 1):
                    for dz in (-1, 0, 1):
                        for q in self._grid.get((k[0] + dx, k[1] + dy, k[2] + dz), ()):
                            if np.linalg.norm(self.pos[q] - p) <= 2.5 * self.cr:
                                return False
        return True

    def add(self, p, v, label):
        i = super().add(p, v, label)
        self._grid.setdefault(self._key(p), []).append(i)
        return i

    def pair(self, anchor, direction, kind, v, label):
        side, collide = kind
        target = down(self.osq) if collide else self.osq
        p = None
        for t in range(8):           # no exact hit from this start: tilt the direction a little and search again
            direction = unit(np.asarray(direction) + 0.02 * t * np.array([0.3, -0.5, 0.7]))
            p = partner_at(anchor, direction, target)
            if p is not None:
                break
        if p is None or not self._clear([anchor, p]):
            self.skipped += 1
            return None
        return self.add_pair(anchor, direction, target, v, "%s, side %s, %s" % (label, side, "prev(overlap_sq)" if collide else "overlap_sq"),
                             collide)


def _side_dir(a, side, rng):
    d = rng.normal(size=3)
    d[a] = 0.0
    d = 0.6 * unit(d)
    d[a] = 1.0 if side == "+" else -1.0
    return unit(d)


def _group(b, fixed, origins, rng, v_scale, tag):
    """The four pairs (KINDS) of one boundary coordinate combination `fixed` ({axis: (value, label)}); origins[q] is the
    position of anchor q before its fixed coordinates are set; the side is taken along the first fixed axis."""
    a0 = min(fixed)
    for q, kind in enumerate(KINDS):
        p = np.array(origins[q], dtype=np.float64)
        for a, (v, _) in fixed.items():
            p[a] = v
        lab = "%s %s" % (tag, ", ".join("%s=%s" % ("xyz"[a], fixed[a][1]) for a in sorted(fixed)))
        b.pair(p, _side_dir(a0, kind[0], rng), kind, rng.normal(size=3) * v_scale, lab)


def _corner(b, fixed, rng, v_scale, tag):
    """One pair at a point on a boundary in all three axes (no free coordinate for more): random kind and direction."""
    p = np.array([fixed[a][0] for a in range(3)])
    kind = KINDS[rng.integers(4)]
    b.pair(p, unit(rng.normal(size=3)), kind, rng.normal(size=3) * v_scale,
           "%s %s" % (tag, ", ".join("%s=%s" % ("xyz"[a], fixed[a][1]) for a in range(3))))


def _variants(grid, a, k, table, rng=None):
    """edge[k] or lo[k] and the doubles on either side, labelled (a random one if rng is given)."""
    v = grid.edge[a][k] if table == "edge" else grid.lo[a][k]
    out = [(v, "%s[%d]" % (table, k)), (down(v), "prev(%s[%d])" % (table, k)), (up(v), "next(%s[%d])" % (table, k))]
    return out if rng is None else out[rng.integers(3)]


def pore_lattice(cfg, seed=0, v_scale=300.0):
    """Pairs on the boundaries of the Pore grid, where the Pore walls touch nothing in one step (inside the pore and the
    open-air caps):
    - every z boundary value (all 149 edges, the 97 on which the owner estimate misses among them) in a column inside
      the pore;
    - every interior x and y boundary value in the bottom cap (the edges one double below which the estimate misses
      among them);
    - x-y corners in the bottom cap, edge and lo variants;
    - x-y-z corners where the bands of 8 cells meet, in both caps.
    Each boundary value gets the four KINDS of pair; each corner one."""
    g = cfg.grid
    rng = np.random.default_rng(seed)
    b = Builder(cfg.collision_range)
    nm = 1e-9
    for k in range(g.nc[2] + 1):
        vals = [(v, lab) for v, lab in boundary_values(g, 2, [k])]
        for s, val in enumerate(vals):
            origins = [((2.0 + 1.2 * ((4 * s + q) % 8)) * nm, (2.0 + 1.2 * ((4 * s + q) // 8)) * nm, 0.0) for q in range(4)]
            _group(b, {2: val}, origins, rng, v_scale, "z")
    for a in (0, 1):
        for k in range(1, g.nc[a]):
            for s, val in enumerate(boundary_values(g, a, [k])):
                origins = []
                for q in range(4):
                    o = [0.0, 0.0, (45.0 + 7.0 * a + 1.2 * ((4 * s + q) // 7)) * nm]
                    o[1 - a] = (2.0 + 1.2 * ((4 * s + q) % 7)) * nm
                    origins.append(o)
                _group(b, {a: val}, origins, rng, v_scale, "xy"[a])
    for kx in (3, 5, 7, 9, 11):
        for ky in (5, 7, 9):
            q0 = 0
            for table in ("edge", "lo"):
                for xv in _variants(g, 0, kx, table):
                    for yv in _variants(g, 1, ky, table):
                        origins = [(0.0, 0.0, (3.0 + 1.2 * (q0 + q)) * nm) for q in range(4)]
                        q0 += 4
                        _group(b, {0: xv, 1: yv}, origins, rng, v_scale, "xy")
    for kx in (4, 6, 8, 10):
        for ky in (4, 6, 8, 10):
            for kz in (1, 2, 3, 4, g.nc[2] - 4, g.nc[2] - 3, g.nc[2] - 2, g.nc[2] - 1):
                fixed = {a: _variants(g, a, k, ("edge", "lo")[rng.integers(2)], rng) for a, k in ((0, kx), (1, ky), (2, kz))}
                _corner(b, fixed, rng, v_scale, "xyz")
    return b


def cube_lattice(cfg, seed=1, v_scale=300.0):
    """Pairs on every boundary value of each axis of a cube grid (the four KINDS each, the other coordinates inside
    cells), x-y corners with their edge and lo variants, and x-y-z corners."""
    g = cfg.grid
    rng = np.random.default_rng(seed)
    b = Builder(cfg.collision_range)
    nm = 1e-9
    for a in range(3):
        bb, cc = [q for q in range(3) if q != a]
        for k in range(g.nc[a] + 1):
            cb, ccell = (3 + k + 5 * a) % (g.nc[bb] - 1), (7 + 2 * k + a) % g.nc[cc]
            for s, val in enumerate(boundary_values(g, a, [k])):
                origins = []
                for q in range(4):
                    t = 4 * s + q
                    o = [0.0, 0.0, 0.0]
                    o[bb] = g.edge[bb][cb + t // 16] + (1.0 + 1.2 * (t % 4)) * nm
                    o[cc] = g.edge[cc][ccell] + (1.0 + 1.2 * ((t // 4) % 4)) * nm
                    origins.append(o)
                _group(b, {a: val}, origins, rng, v_scale, "xyz"[a])
    for kx, ky in ((4, 4), (4, 10), (10, 4), (10, 10)):
        q0 = 0
        for table in ("edge", "lo"):
            for xv in _variants(g, 0, kx, table):
                for yv in _variants(g, 1, ky, table):
                    origins = [(0.0, 0.0, (2.0 + 1.2 * (q0 + q)) * nm) for q in range(4)]
                    q0 += 4
                    _group(b, {0: xv, 1: yv}, origins, rng, v_scale, "xy")
    for kx in (2, 7, 12):
        for ky in (2, 7, 12):
            for kz in (2, 7, 12):
                fixed = {a: _variants(g, a, k, ("edge", "lo")[rng.integers(2)], rng) for a, k in ((0, kx), (1, ky), (2, kz))}
                _corner(b, fixed, rng, v_scale, "xyz")
    return b


def cube_groups_config():
    """The cube stage on an even grid (14 cells of 7.1 nm per axis, bands of a tenth of a cell): colour groups need
    both parities on every axis, which the shipped 15-cell grid of cube_config() does not have."""
    from argon_monte_carlo_b200 import config
    return config.cube_config(1.0, 14)


def fast_particle(cfg, speed=2.0e5):
    """One particle with |v| > 2^17 m/s in the middle of a cell of the pore column (the per-particle fallback of the
    sampling kernel's fixed-point sums)."""
    g = cfg.grid
    p = [0.5 * (g.edge[a][g.nc[a] // 2 + 2] + g.edge[a][g.nc[a] // 2 + 3]) for a in range(3)]
    return np.array(p), np.array([speed, -0.3 * speed, 0.1 * speed])


# ------------------------------------------------------------------ the fp32 filter, cell by cell
def det_w(grid, cr):
    """Minimal bin width of the detection pass (amc_api.cu): 1.05 filter radii, rounded up in fp32."""
    return np.nextafter(np.float32(1.05 * math.sqrt(float(det_thr(grid, cr)))), np.float32(np.inf))


def det_bins(grid, cr, a, k):
    """(bins, fp32 inverse bin width) of reference cell k on axis a (x: up to 64 bins; y: up to 32, twice as wide)."""
    wd = np.float32(grid.edge[a][k + 1] - grid.lo[a][k])
    w = det_w(grid, cr) * (np.float32(1.0) if a == 0 else np.float32(2.0))
    nb = max(1, int(min(64.0 if a == 0 else 32.0, math.floor(float(wd / w)))))
    return nb, np.float32(nb) / wd


def interior(grid, a, k, cr, margin=2.0):
    """The part of owner cell k on axis a outside every band, less `margin` collision ranges on each side."""
    return grid.edge[a][k] + margin * cr, grid.lo[a][k + 1] - margin * cr


def cell_lo(grid, cell):
    return np.array([grid.lo[a][cell[a]] for a in range(3)])


def missed_by_rounded_down_filter(grid, cr, a, b, cell):
    """True when the fp32 filter of cell `cell` puts the pair (a, b) at or above fp32(overlap_sq) rounded down by a
    margin of 3 fp32 ulps: a filter without its rounding slack would drop it."""
    osq32 = np.float32(overlap_sq(cr))
    if float(osq32) > overlap_sq(cr):
        osq32 = np.nextafter(osq32, np.float32(0))
    return float(filter_d2(a, b, cell_lo(grid, cell))) >= float(osq32) * (1.0 + 3 * 2.0 ** -23)


def worst_pair(b, grid, cell, rng, v_scale=300.0, label="far corner"):
    """A pair at prev(overlap_sq) in the far corner of cell `cell` (largest cell-relative coordinates, so the largest
    fp32 rounding), chosen so that the filter evaluates it above fp32(overlap_sq): only the slack of det_thr keeps it."""
    cr = b.cr
    for _ in range(400):
        hi = np.array([interior(grid, a, cell[a], cr)[1] for a in range(3)])
        anchor = hi - rng.uniform(0.0, 1.0, 3) * cr
        direction = -np.abs(rng.normal(size=3))
        p = partner_at(anchor, direction, down(b.osq))
        if p is not None and missed_by_rounded_down_filter(grid, cr, anchor, p, cell) and b._clear([anchor, p]):
            return b.add_pair(anchor, direction, down(b.osq), rng.normal(size=3) * v_scale,
                              "%s, cell %s, prev(overlap_sq)" % (label, tuple(cell)), True)
    raise AssertionError("no far-corner pair found in cell %s" % (tuple(cell),))


def false_positive_pair(b, grid, cell, slot, rng, v_scale=300.0):
    """A pair the exact test rejects (d2 >= overlap_sq (1 + 1e-5)) that the fp32 filter of the cell passes (below
    det_thr by a margin), near the low corner of the owner cell's interior; slot spaces such pairs 1.2 nm apart."""
    cr = b.cr
    thr = float(det_thr(grid, cr))
    lo = np.array([interior(grid, a, cell[a], cr)[0] for a in range(3)])
    for _ in range(200):
        anchor = lo + np.array([1.2e-9 * (slot % 4), 1.2e-9 * (slot // 4), 0.5e-9]) + rng.uniform(0.0, 0.2, 3) * cr
        direction = unit(rng.normal(size=3))
        p = anchor + math.sqrt(b.osq * (1.0 + 2.5e-5)) * direction
        if d2_kernel(anchor, p) >= b.osq * (1.0 + 1e-5) and float(filter_d2(anchor, p, cell_lo(grid, cell))) < thr * (1.0 - 4e-7) \
                and b._clear([anchor, p]):
            i = b.add(anchor, rng.normal(size=3) * v_scale, "false positive, cell %s (anchor)" % (tuple(cell),))
            j = b.add(p, approaching(b.vel[i], anchor, p), "false positive, cell %s (partner)" % (tuple(cell),))
            b.miss.append((i, j))
            return i, j
    raise AssertionError("no false-positive pair found in cell %s" % (tuple(cell),))


def threshold_cells(cfg, grid=None, seed=2, n_worst=24, n_random=48, n_straddle=16, hits=(1, 8, 9), background=0):
    """Pairs at the overlap threshold, one scenario per reference cell:
    - far-corner pairs that only the slack of det_thr keeps in the filter (worst_pair);
    - pairs at prev(overlap_sq) or overlap_sq at random places and directions;
    - pairs straddling a detection bin boundary in x or in y (y bins are twice as wide);
    - cells with 1, 8 and 9 filter hits: one far-corner true pair plus false positives (listed on either side of
      AMC_MAX_HITS, then searched).
    background: particles of a uniform gas added around them (every one 2.5 collision ranges clear of every other), so
    the detection pass really hashes full cells.  Returns (builder, {scenario: [cells]})."""
    grid = grid or cfg.grid
    rng = np.random.default_rng(seed)
    b = Builder(cfg.collision_range)
    cr = b.cr
    cells = [(int(rng.integers(1, grid.nc[0] - 1)), int(rng.integers(1, grid.nc[1] - 1)), int(rng.integers(1, grid.nc[2] - 1)))
             for _ in range(4 * (n_worst + n_random + n_straddle + len(hits)))]
    cells = list(dict.fromkeys(cells))
    it = iter(cells)
    used = {"worst": [], "random": [], "straddle": [], "hits": []}
    for _ in range(n_worst):
        c = next(it)
        worst_pair(b, grid, c, rng)
        used["worst"].append(c)
    for t in range(n_random):
        c = next(it)
        lo_hi = [interior(grid, a, c[a], cr) for a in range(3)]
        anchor = np.array([rng.uniform(*lo_hi[a]) for a in range(3)])
        if b.pair(anchor, unit(rng.normal(size=3)), KINDS[t % 4], rng.normal(size=3) * 300.0, "random, cell %s" % (c,)) is not None:
            used["random"].append(c)
    for t in range(n_straddle):
        c = next(it)
        a = t % 2
        nb, inv_w = det_bins(grid, cr, a, c[a])
        m = max(1, nb // 2 + (t // 2) % 3 - 1)
        anchor = np.array([0.5 * sum(interior(grid, q, c[q], cr)) for q in range(3)])
        anchor[a] = grid.lo[a][c[a]] + float(m / inv_w) - 0.3 * cr        # just below the bin boundary m
        direction = np.zeros(3)
        direction[a] = 1.0
        direction[(a + 1) % 3] = 0.3
        if b.pair(anchor, direction, KINDS[t % 4], rng.normal(size=3) * 300.0, "bin boundary %d along %s, cell %s" % (m, "xy"[a], c)) is not None:
            used["straddle"].append(c)
    for h in hits:
        c = next(it)
        worst_pair(b, grid, c, rng, label="%d filter hits" % h)
        for s in range(h - 1):
            false_positive_pair(b, grid, c, s, rng)
        used["hits"].append((c, h))
    if background:
        add_background(b, grid, background, rng)
    return b, used


def add_background(b, grid, n, rng, v_scale=300.0):
    """n particles uniformly over the grid, kept only where they stay 2.5 collision ranges clear of every other one."""
    from scipy.spatial import cKDTree
    lo = np.array([grid.edge[a][0] for a in range(3)])
    hi = np.array([grid.edge[a][-1] for a in range(3)])
    pts = lo + rng.uniform(0.0, 1.0, (n, 3)) * (hi - lo)
    have = np.array(b.pos)
    near = cKDTree(have).query_ball_point(pts, 2.5 * b.cr) if len(have) else [[] for _ in range(n)]
    keep = np.array([len(q) == 0 for q in near])
    pts = pts[keep]
    bad = set()
    for i, j in cKDTree(pts).query_pairs(2.5 * b.cr):
        bad.add(max(i, j))
    pts = pts[[i for i in range(len(pts)) if i not in bad]]
    for p in pts:
        b.pos.append(p)
        b.vel.append(rng.normal(size=3) * v_scale)
        b.label.append("background")
    return len(pts)


# ------------------------------------------------------------------ capacities
CAPACITY_CASES = {                       # (lattice points, partners at 0.5 cr, triple) -> particles in one reference cell
    "candidates 384": (383, 1, False), "candidates 385": (384, 1, False),
    "overlapping pairs 64": (64, 64, False), "overlapping pairs 65": (65, 65, False),
    "moved 32": (16, 16, False), "moved 33": (16, 15, True),
    "members 512": (511, 1, False), "members 513": (512, 1, False),
}


def capacity_cell(cfg, case, cell=(9, 9, 40), seed=3, v_scale=300.0):
    """One reference cell of the Pore grid at a capacity switch point (CAPACITY_CASES): lattice points 2.8 nm apart in
    the interior of the owner cell (outside every band, so candidates == members == particles), the first ones with
    a partner half a collision range away, approaching; 'moved 33' turns lattice point 15 into a collinear triple
    (A-B and B-C overlap, A-C not), so one visit moves 33 particles."""
    g = cfg.grid
    n_lat, n_pair, triple = CAPACITY_CASES[case]
    rng = np.random.default_rng(seed)
    b = Builder(cfg.collision_range)
    cr = b.cr
    lo_hi = [interior(g, a, cell[a], cr) for a in range(3)]
    ticks = [np.linspace(lo_hi[a][0], lo_hi[a][1], 8) for a in range(3)]
    pts = np.array([(ticks[0][i], ticks[1][j], ticks[2][k]) for i in range(8) for j in range(8) for k in range(8)])
    order = rng.permutation(len(pts))
    for t in range(n_lat):
        p = pts[order[t]]
        v = rng.normal(size=3) * v_scale
        i = b.add(p, v, "%s: lattice point %d" % (case, t))
        if t < n_pair or (triple and t == n_pair):
            u = unit(rng.normal(size=3))
            step = 0.6 * cr if triple and t == n_pair else 0.5 * cr
            j = b.add(p + step * u, v - V_APPROACH * u, "%s: partner of %d" % (case, t))
            b.collide.append((i, j))
            if triple and t == n_pair:
                k = b.add(p + 2 * step * u, v - 2 * V_APPROACH * u, "%s: third of %d" % (case, t))
                b.collide.append((j, k))
    return b


def degenerate_pair(cfg, grid=None, cell=(9, 9, 40), seed=4):
    """Two overlapping particles with identical velocities (a == 0: the reference raises, the oracle counts an error and
    skips the pair) in one owner cell's interior, and an ordinary overlapping pair in the same cell."""
    g = grid or cfg.grid
    rng = np.random.default_rng(seed)
    b = Builder(cfg.collision_range)
    cr = b.cr
    lo = np.array([interior(g, a, cell[a], cr)[0] for a in range(3)])
    v = rng.normal(size=3) * 300.0
    u = unit(rng.normal(size=3))
    b.add(lo + 1e-9, v, "degenerate (a)")
    b.add(lo + 1e-9 + 0.5 * cr * u, v.copy(), "degenerate (b)")
    i = b.add(lo + 4e-9, v, "ordinary (a)")
    j = b.add(lo + 4e-9 + 0.5 * cr * u, v - V_APPROACH * u, "ordinary (b)")
    b.collide.append((i, j))
    return b


# ------------------------------------------------------------------ checks shared by the host and GPU tests
def close_pairs(b, r):
    """Index pairs (hi, lo) of the state within distance r of each other."""
    from scipy.spatial import cKDTree
    return {(max(i, j), min(i, j)) for i, j in cKDTree(np.array(b.pos)).query_pairs(r)}


def first_difference(got, ref, labels, keys):
    """Message naming the first particle whose state differs and the boundary it was placed on, or None."""
    for k in keys:
        a, c = np.asarray(got[k]), np.asarray(ref[k])
        bad = np.nonzero(a != c)[0] if k != "flag" else np.nonzero(a.astype(bool) != c.astype(bool))[0]
        if len(bad):
            i = int(bad[0])
            return "%s differs for %d particles; first %d (%s): %r vs %r" % (k, len(bad), i, labels[i], a[i], c[i])
    return None
