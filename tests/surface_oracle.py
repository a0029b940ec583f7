"""Hit records of the oracle's wall phases, for the surface-recording tests (test infrastructure only).

Every wall interaction a phase applies gives one record: case, particle index, contact point, v_in, v_out and dE (the
energy the gas gained); a hit the reference counts but applies nothing to (its floating-point error path) has a NaN
contact point.  Pore and Cube walls are restated case by case in NumPy on a copy of the state (elementwise IEEE
operations in the oracle's plain-mode order) and the copy is checked bit for bit against the oracle's own wall pass;
the Temp cases run through the oracle itself (temp_case_detect / temp_case_apply), with the state read before and
after every case.  The whole timesteps below compose these with the oracle's other phases exactly as oracle/steps.py
does."""
from __future__ import annotations

import numpy as np

from argon_monte_carlo_b200 import amc
from oracle import oracle as O

FIELDS = ("x", "y", "z", "vx", "vy", "vz")
ENERGIZED = (3, 4, 5, 6, 7, 8, 9)


class HitSink:
    def __init__(self):
        self.parts = []

    def add(self, case, pid, col, v_in, v_out, dE):
        n = len(pid)
        if n:
            self.parts.append((np.full(n, case, dtype=np.int64), np.asarray(pid, dtype=np.int64), np.asarray(col, dtype=np.float64).reshape(n, 3),
                               np.asarray(v_in, dtype=np.float64).reshape(n, 3), np.asarray(v_out, dtype=np.float64).reshape(n, 3),
                               np.broadcast_to(np.asarray(dE, dtype=np.float64), (n,)).copy()))

    def hits(self):
        if not self.parts:
            return {"case": np.zeros(0, np.int64), "pid": np.zeros(0, np.int64), "col": np.zeros((0, 3)), "v_in": np.zeros((0, 3)),
                    "v_out": np.zeros((0, 3)), "dE": np.zeros(0)}
        cols = list(zip(*self.parts))
        return {k: np.concatenate(v) for k, v in zip(("case", "pid", "col", "v_in", "v_out", "dE"), cols)}

    def wall_counts(self):
        return np.bincount(self.hits()["case"], minlength=amc.NUM_CASES)


def _arrays(st):
    return {k: getattr(st, k).copy() for k in FIELDS + ("px", "py", "pz")}


def _side_t(x, y, vx, vy, Rc):
    """side_quadratic (Pore:312-315) elementwise; ok = False on the floating-point error path."""
    with np.errstate(invalid="ignore", divide="ignore"):
        a = (-vx) * (-vx) + (-vy) * (-vy)
        b = 2 * (x * (-vx) + y * (-vy))
        c = (x * x + y * y) - Rc * Rc
        disc = b * b - (4 * a) * c
        ok = (disc >= 0.0) & (a != 0.0)
        r = np.sqrt(np.where(ok, disc, 0.0))
        t1, t2 = (-b + r) / (2 * a), (-b - r) / (2 * a)
    return np.where(t1 < t2, t1, t2), ok


def _side(s, m, Rc, case, sink):
    i = np.flatnonzero(m)
    x, y, z, vx, vy, vz = (s[k][i] for k in FIELDS)
    t, ok = _side_t(x, y, vx, vy, Rc)
    with np.errstate(invalid="ignore"):
        cx, cy, cz = x - vx * t, y - vy * t, z - vz * t
        nx, ny = cx / Rc, cy / Rc
        sc = vx * nx + vy * ny
        nvx, nvy = vx - (2 * sc) * nx, vy - (2 * sc) * ny
    col = np.where(ok[:, None], np.stack([cx, cy, cz], axis=1), np.nan)
    sink.add(case, i, col, np.stack([vx, vy, vz], 1), np.stack([np.where(ok, nvx, vx), np.where(ok, nvy, vy), vz], 1), 0.0)
    j = i[ok]
    s["x"][j], s["y"][j] = (cx + nvx * t)[ok], (cy + nvy * t)[ok]
    s["vx"][j], s["vy"][j] = nvx[ok], nvy[ok]


def _plane(s, m, zp, case, sink):
    i = np.flatnonzero(m)
    x, y, z, vx, vy, vz = (s[k][i] for k in FIELDS)
    t = (z - zp) / vz
    sink.add(case, i, np.stack([x - vx * t, y - vy * t, np.full(len(i), zp)], 1), np.stack([vx, vy, vz], 1), np.stack([vx, vy, -vz], 1), 0.0)
    s["vz"][i] = -vz
    s["z"][i] = zp + t * (-vz)


def pore_wall_hits(st, g, sink):
    """Open_Air_Pore_MC wall cases (Pore:442-485) on the oracle state st: records into sink, leaves st unchanged."""
    s = _arrays(st)
    r = lambda: np.sqrt(s["x"] * s["x"] + s["y"] * s["y"])
    pr = np.sqrt(s["px"] * s["px"] + s["py"] * s["py"])
    pz = s["pz"]
    _side(s, r() > g.R_oa, g.R_oa_c, 0, sink)
    _plane(s, s["z"] < 0, 0.0, 1, sink)
    _plane(s, s["z"] > g.H, g.H, 2, sink)
    _plane(s, (pz > g.z_cold) & (s["z"] < g.z_cold) & (r() > g.R_p), g.z_cold, 3, sink)
    _plane(s, (pz < g.oah) & (s["z"] > g.oah) & (r() > g.R_p), g.oah, 4, sink)
    _side(s, (pz < g.z_gt_pore) & (pz > g.z_gb) & (pr < g.R_g) & (r() > g.R_g), g.R_g_c, 5, sink)
    _plane(s, (pr > g.R_p) & (s["z"] < g.z_gb) & (pz < g.z_gt_pore) & (pz > g.z_gb), g.z_gb, 6, sink)
    _plane(s, (pr > g.R_p) & (s["z"] > g.z_gt_pore) & (pz < g.z_gt_pore) & (pz > g.z_gb), g.z_gt_pore, 7, sink)
    z = s["z"]
    _side(s, (pr < g.R_p) & (r() > g.R_p) & (((z < g.z_cold) & (z > g.z_gt_pore)) | ((z < g.z_gb) & (z > g.oah))), g.R_p_c, 8, sink)
    return s


def cube_wall_hits(st, L, sink):
    """Open_Air_Cube_MC walls (Cube:192-226): x then y then z, the face at L before the face at 0."""
    s = _arrays(st)
    pos, vel = ("x", "y", "z"), ("vx", "vy", "vz")
    for a in range(3):
        for c, face in ((2 * a, float(L[a])), (2 * a + 1, 0.0)):
            i = np.flatnonzero(s[pos[a]] > face if c == 2 * a else s[pos[a]] < 0)
            v = np.stack([s[k][i] for k in vel], 1)
            t = (s[pos[a]][i] - face) / v[:, a] if c == 2 * a else s[pos[a]][i] / v[:, a]
            col = np.stack([np.full(len(i), face) if b == a else s[pos[b]][i] - v[:, b] * t for b in range(3)], 1)
            vout = v.copy()
            vout[:, a] = -v[:, a]
            sink.add(c, i, col, v, vout, 0.0)
            s[vel[a]][i] = -v[:, a]
            s[pos[a]][i] = (face + t * (-v[:, a])) if c == 2 * a else t * (-v[:, a])
    return s


def _check_same(s, st, what):
    for k in FIELDS:
        assert np.array_equal(s[k].view(np.uint64), getattr(st, k).view(np.uint64)), (what, k)


def temp_case_hits(st, g, case, idx, normal, dirs, surf_e, sink):
    """Apply one Temp case through the oracle (temp_case_apply) and record its hits (Temp:311-553)."""
    pre = _arrays(st)
    res = O.temp_case_apply(st, g, case, idx, dirs, surf_e)
    i = np.asarray(idx, dtype=np.int64)
    x, y, z, vx, vy, vz = (pre[k][i] for k in FIELDS)
    v_in = np.stack([vx, vy, vz], 1)
    v_out = np.stack([getattr(st, k)[i] for k in ("vx", "vy", "vz")], 1)
    dE = np.zeros(len(i))
    with np.errstate(invalid="ignore", divide="ignore"):
        if case in (1, 2):
            zp = 0.0 if case == 1 else float(g.H)
            t = (z - zp) / vz
            col = np.stack([x - vx * t, y - vy * t, np.full(len(i), zp)], 1)
        elif case == 0:
            t, ok = _side_t(x, y, vx, vy, float(g.R_oa_c))
            col = np.where(ok[:, None], np.stack([x - vx * t, y - vy * t, z - vz * t], 1), np.nan)
        else:
            ok = normal[:, 0] == normal[:, 0]
            col = np.where(ok[:, None], np.stack([getattr(st, k)[i] for k in ("x", "y", "z")], 1), np.nan)
            m = float(g.argon_mass)
            Es = np.asarray(surf_e, dtype=np.float64)[:len(i)] if case == 5 else np.full(len(i), float(g.E_cold if case in (3, 7, 9) else g.E_hot))
            alpha = float(g.alpha_g if case == 5 else g.alpha_c)
            v_mag = np.sqrt((vx * vx + vy * vy) + vz * vz)
            E = (0.5 * m) * (v_mag * v_mag)
            Enew = E + (Es - E) * alpha
            dE = np.where(ok, Enew - E, 0.0)
    sink.add(case, i, col, v_in, v_out, dE)
    return res


def temp_walls_philox_hits(st, g, seed, step, cheb, sink):
    """The device-RNG wall phase (what orc_temp_walls_philox does), case by case with hit records."""
    counts = np.zeros(amc.NUM_CASES, dtype=np.int64)
    for c in range(amc.NUM_CASES):
        idx, normal, colz = O.temp_case_detect(st, g, c)
        counts[c] = len(idx)
        dirs, se = np.zeros((max(len(idx), 1), 3)), np.zeros(max(len(idx), 1))
        if c in ENERGIZED:
            for k in range(len(idx)):
                if normal[k, 0] == normal[k, 0]:
                    dirs[k] = O.philox_direction(seed, int(idx[k]), step, c, normal[k], g.cos85)
                    if c == 5:
                        se[k] = O.cheb_eval(cheb, colz[k])
        temp_case_hits(st, g, c, idx, normal, dirs, se, sink)
    return counts


def pore_step(st, cfg, sink):
    O.drift(st, cfg.dt, True)
    s = pore_wall_hits(st, cfg.geom, sink)
    O.pore_walls(st, cfg.geom)
    _check_same(s, st, "pore walls")
    O.pore_recapture(st, cfg.geom)
    O.pp_groups(st, cfg.grid, cfg.collision_range, cfg.argon_mass)
    O.pore_recapture(st, cfg.geom)


def cube_step(st, cfg, sink):
    O.drift(st, cfg.dt, False)
    s = cube_wall_hits(st, (cfg.cube_x, cfg.cube_y, cfg.cube_z), sink)
    O.cube_walls(st, cfg.cube_x, cfg.cube_y, cfg.cube_z)
    _check_same(s, st, "cube walls")
    O.cube_pp_sweep(st, cfg.grid, cfg.collision_range, cfg.argon_mass)


def _temp_close(st, cfg):
    O.temp_recapture(st, cfg.geom)
    O.pp_groups(st, cfg.grid, cfg.collision_range, cfg.argon_mass)
    O.temp_recapture(st, cfg.geom)


def temp_step_philox(st, cfg, seed, step, cheb, sink):
    O.drift(st, cfg.dt, True)
    temp_walls_philox_hits(st, cfg.geom, seed, step, cheb, sink)
    _temp_close(st, cfg)


def temp_step_host_rng(st, cfg, sink):
    """steps.temp_step_host_rng with hit records (the same Mersenne-Twister draws in the same order)."""
    from argon_monte_carlo_b200 import host_rng
    from argon_monte_carlo_b200.config import surface_energy_gap as seg
    O.drift(st, cfg.dt, True)
    for c in range(amc.NUM_CASES):
        idx, normal, colz = O.temp_case_detect(st, cfg.geom, c)
        dirs = surf = None
        if c in ENERGIZED:
            if c == 5:
                dirs, surf = np.zeros((len(idx), 3)), np.zeros(len(idx))
                for k in range(len(idx)):
                    if normal[k, 0] == normal[k, 0]:
                        dirs[k] = host_rng.inbound_direction(normal[k])
                        surf[k] = float(seg(cfg, colz[k]))
            else:
                dirs = host_rng.directions_for_hits(normal)
        temp_case_hits(st, cfg.geom, c, idx, normal, dirs, surf if surf is not None else np.zeros(max(len(idx), 1)), sink)
    _temp_close(st, cfg)
