"""ctypes binding of libamc.so (include/amc.h) and the host-side mirror of the reference's
per-timestep interface.

The reference keeps its particle state in module globals and advances it with a script-level
loop (Open_Air_Pore_MC.py:416-557, Temperature_Pore_MC.py:662-853, Open_Air_Cube_MC.py:175-338);
`Simulation` owns the same state on one B200 and exposes that loop body as `step()`, plus the
phase-level operators the parity tests compare one by one.  There is no CPU fallback: if the CUDA
library is missing or no device is present, construction raises.
"""
from __future__ import annotations

import ctypes as C
import math
import os

import numpy as np

from . import build as _build
from .config import HIST_RANGE, NUM_BINS

KIND_CUBE, KIND_PORE, KIND_TEMP = 0, 1, 2
PP_GROUPS, PP_SWEEP = 0, 1
RNG_DEVICE, RNG_HOST = 0, 1
TAP_PAIRS, TAP_WALL_BITS, TAP_PATHS = 1, 2, 4
NUM_CASES = 10
ABI_VERSION = 1

GEOM_FIELDS = ("argon_mass", "argon_radius", "collision_range", "R_oa", "R_oa_c", "R_p", "R_p_c", "R_g", "R_g_c",
               "H", "oah", "z_cold", "z_gb", "z_gt_pore", "z_gt", "ten_a", "R_oa_sq", "R_g_sq", "R_p_sq",
               "zc3", "zh3", "zgt_m", "zgb_p", "R_g_c_sq", "R_p_c_sq", "recap_lo", "recap_hi",
               "E_cold", "E_hot", "alpha_c", "alpha_g", "cos85")

c_double_p = C.POINTER(C.c_double)
c_int64_p = C.POINTER(C.c_int64)
c_uint8_p = C.POINTER(C.c_uint8)


class AmcGeom(C.Structure):
    _fields_ = [(k, C.c_double) for k in GEOM_FIELDS]


class AmcConfig(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("kind", C.c_int32), ("pp_mode", C.c_int32), ("rng_mode", C.c_int32),
                ("taps", C.c_int32), ("dt", C.c_double), ("cube", C.c_double * 3), ("geom", AmcGeom),
                ("nc", C.c_int32 * 3), ("c0", C.c_int32 * 3), ("edge", c_double_p * 3), ("lo", c_double_p * 3),
                ("overlap_sq", C.c_double), ("seed", C.c_uint64), ("cheb_coef", c_double_p), ("cheb_n", C.c_int32),
                ("cheb_zmid", C.c_double), ("cheb_inv_half", C.c_double), ("hist_first", C.c_double),
                ("hist_last", C.c_double), ("hist_edges", c_double_p), ("max_particles", C.c_int64),
                ("pair_capacity", C.c_int64), ("path_capacity", C.c_int64)]


class AmcStepStats(C.Structure):
    _fields_ = [("wall_hits", C.c_int64 * NUM_CASES), ("wall_collisions", C.c_int64), ("pp_collisions", C.c_int64),
                ("pair_checks_ref", C.c_int64), ("pair_checks_exec", C.c_int64), ("oob_after_walls", C.c_int64),
                ("oob_after_pp", C.c_int64), ("oob_after_walls_recapture", C.c_int64),
                ("oob_after_pp_recapture", C.c_int64), ("errors", C.c_int64), ("completed_paths", C.c_int64),
                ("dpz", C.c_double), ("e_cold", C.c_double), ("e_hot", C.c_double)]

    def as_dict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_ if k != "wall_hits"}
        d["wall_hits"] = np.array(self.wall_hits[:], dtype=np.int64)
        d["collisions"] = d["wall_collisions"] + d["pp_collisions"]
        return d


INIT_MAX_REGIONS = 8


class AmcInitSpec(C.Structure):
    """struct amc_init_spec (include/amc.h): synthetic Maxwellian state generated on the device."""
    _fields_ = [("n_total", C.c_int64), ("seed", C.c_uint64), ("n_regions", C.c_int32), ("shape", C.c_int32),
                ("cum_weight", C.c_double * INIT_MAX_REGIONS), ("radius", C.c_double * INIT_MAX_REGIONS),
                ("bx", C.c_double * INIT_MAX_REGIONS), ("by", C.c_double * INIT_MAX_REGIONS),
                ("z_lo", C.c_double * INIT_MAX_REGIONS), ("z_hi", C.c_double * INIT_MAX_REGIONS),
                ("sigma", C.c_double), ("keep_z_lo", C.c_double), ("keep_z_hi", C.c_double)]


class AmcError(RuntimeError):
    pass


_lib = None

# every exported symbol of include/amc.h (tests check the built library against this list)
EXPORTS = ("amc_create", "amc_destroy", "amc_last_error", "amc_abi_version", "amc_set_state", "amc_get_state",
           "amc_num_particles", "amc_step", "amc_drift", "amc_walls", "amc_recapture", "amc_pairs", "amc_wall_case",
           "amc_wall_hits_pending", "amc_wall_apply_directions", "amc_get_histograms", "amc_get_pair_list",
           "amc_get_wall_bits", "amc_get_completed_paths", "amc_clear_taps", "amc_set_step_index", "amc_last_timing",
           "amc_last_detect_ms", "amc_init_synthetic",
           "amc_get_outputs_raw", "amc_set_outputs_raw", "amc_get_step_index",
           "amc_slab_enable", "amc_set_stream", "amc_set_ids", "amc_slab_advect", "amc_slab_sort", "amc_slab_pairs_begin",
           "amc_slab_group", "amc_slab_apply", "amc_slab_finish", "amc_slab_get_owned", "amc_state_digest",
           "amc_slab_p2p_setup", "amc_slab_p2p_connect", "amc_slab_step", "amc_wall_operator", "amc_seed_relax", "amc_last_scatter_ms",
           "amc_sample_enable", "amc_sample_disable", "amc_sample_now", "amc_sample_get_raw", "amc_sample_set_raw",
           "amc_last_sample_ms", "amc_surface_enable", "amc_surface_disable", "amc_surface_layout", "amc_surface_get_raw",
           "amc_surface_set_raw", "amc_vdf_enable", "amc_vdf_disable", "amc_vdf_layout", "amc_vdf_get_raw", "amc_vdf_set_raw",
           "amc_flux_enable", "amc_flux_disable", "amc_flux_now", "amc_flux_layout", "amc_flux_get_raw", "amc_flux_set_raw")

# field sampling (include/amc.h): words per cell and the binary scales of the fixed-point limbs
SAMPLE_WORDS = 13
SAMPLE_V1, SAMPLE_V2 = 19, 49     # velocity sums: high / low limb
SAMPLE_Q1, SAMPLE_Q2 = 6, 36      # sums of squares: high / low limb

# velocity distribution (include/amc.h): histograms per z layer (vx, vy, vz, speed) and the largest bin count
VDF_HISTS = 4
VDF_MAX_BINS = 4096

# plane flux recording (include/amc.h): words per plane and the binary scales of the fixed-point limbs
FLUX_WORDS = 10
FLUX_V1, FLUX_V2 = 16, 46         # velocity sums: high / low limb
FLUX_Q1, FLUX_Q2 = 2, 32          # sums of v^2: high / low limb

# surface recording (include/amc.h): words per wall element and the binary scales of the fixed-point limbs
SURF_WORDS = 9
SURF_V1, SURF_V2 = 16, 46         # velocity-change sums: high / low limb
SURF_E1, SURF_E2 = 90, 120        # energy sums: high / low limb
SIDE_CASES = (0, 5, 8, 9)         # cylinder slots of Pore (0, 5, 8) and Temp (1, 4, 6H, 6C)
PLUS_Z_CASES = (1, 3, 6)          # planes whose normal into the gas is +z (2A / 3C / 5B, Pore 1 / 3 / 6); others: -z


def load_library():
    """dlopen libamc.so (building it in-tree with nvcc first if it is missing)."""
    global _lib
    if _lib is None:
        path = _build.library_path()
        if not os.environ.get("AMC_LIBRARY"):
            try:
                _build.build_library()       # returns at once unless a source is newer than the library
            except Exception:
                if not os.path.isfile(path):
                    raise                    # no nvcc and no library: nothing to run (there is no CPU fallback)
        L = C.CDLL(path)
        L.amc_last_error.restype = C.c_char_p
        L.amc_last_error.argtypes = [C.c_void_p]
        L.amc_num_particles.restype = C.c_int64
        L.amc_num_particles.argtypes = [C.c_void_p]
        L.amc_get_step_index.restype = C.c_int64
        L.amc_get_step_index.argtypes = [C.c_void_p]
        if L.amc_abi_version() != ABI_VERSION:
            raise AmcError("libamc.so ABI version mismatch")
        _lib = L
    return _lib


def overlap_threshold(collision_range: float) -> float:
    """Smallest double t with sqrt(t) >= collision_range, so that the reference's predicate
    ``sqrt(d2) < collision_range`` (Pore:173-174) equals ``d2 < t`` exactly (sqrt is correctly
    rounded and monotone)."""
    cr = float(collision_range)
    t = cr * cr
    while math.sqrt(t) >= cr:
        t = math.nextafter(t, 0.0)
    while math.sqrt(t) < cr:
        t = math.nextafter(t, math.inf)
    return t


def _dp(a):
    return a.ctypes.data_as(c_double_p) if a is not None else None


_M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def _mix64(z):
    z = z + np.uint64(0x9E3779B97F4A7C15)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def digest_of_arrays(ids, state):
    """NumPy restatement of amc_state_digest (include/amc.h): (sum0, sum1, count) over the given particles.
    ids: global particle indices; state: mapping with the ten float64 arrays and 'flag'."""
    keys = ("x", "y", "z", "vx", "vy", "vz", "dist", "dist_x", "dist_y", "dist_z")
    ids = np.asarray(ids).astype(np.uint64)
    s0 = s1 = np.uint64(0)
    with np.errstate(over="ignore"):
        for f, k in enumerate(keys + ("flag",)):
            if k == "flag":
                bits = (np.asarray(state[k]).astype(np.uint64) & np.uint64(1))
            else:
                bits = np.ascontiguousarray(state[k], dtype=np.float64).view(np.uint64)
            a = _mix64(bits ^ _mix64(np.uint64(16) * ids + np.uint64(f)))
            s0 = s0 + a.sum(dtype=np.uint64)
            s1 = s1 + _mix64(a + np.uint64(0xD6E8FEB86659FD93)).sum(dtype=np.uint64)
    return int(s0), int(s1), int(len(ids))


def sample_grid_shape(grid):
    """(nx, ny, nz) cells of the sampling grid of a handle on `grid` (a slab run: the global grid)."""
    return tuple(int(v) for v in grid.nc)


def sample_cells_of(x, y, z, grid):
    """Sampling cell of every particle (x-major, z-minor) and a mask of the particles inside the grid: the owner-cell
    rule edge[a][k] <= v < edge[a][k+1] of the sort; NaN and anything outside the grid on any axis is outside."""
    idx, inside = [], None
    for a, v in enumerate((x, y, z)):
        e = np.asarray(grid.edge[a], dtype=np.float64)
        k = np.searchsorted(e, np.asarray(v, dtype=np.float64), side="right") - 1
        ok = (k >= 0) & (k < len(e) - 1)
        inside = ok if inside is None else inside & ok
        idx.append(k)
    nx, ny, nz = sample_grid_shape(grid)
    cell = (idx[0] * ny + idx[1]) * nz + idx[2]
    return np.where(inside, cell, -1), inside


def sample_limbs(v, s1, s2):
    """The two fixed-point limbs one value adds (acc_add's scheme, include/amc.h), as int64 arrays."""
    v = np.asarray(v, dtype=np.float64)
    with np.errstate(invalid="ignore"):
        i1 = np.rint(v * 2.0 ** s1).astype(np.int64)
        rem = v - i1.astype(np.float64) * 2.0 ** -s1
        i2 = np.rint(rem * 2.0 ** s2).astype(np.int64)
    return i1, i2


def sample_moments_of_arrays(state, grid, ids=None):
    """NumPy restatement of one amc_sample_now on `state` (mapping with 'x', 'y', 'z', 'vx', 'vy', 'vz'):
    (acc [cells][SAMPLE_WORDS] uint64, 1, n_outside), the layout of Simulation.sample_raw.  ids: optional indices
    into the arrays selecting the particles (default: all).  Integer sums: the result does not depend on the order of
    the particles, and the raw arrays of disjoint parts add up (mod 2^64) to the raw array of the whole."""
    sel = (lambda a: np.asarray(a)) if ids is None else (lambda a: np.asarray(a)[np.asarray(ids)])
    cell, inside = sample_cells_of(sel(state["x"]), sel(state["y"]), sel(state["z"]), grid)
    ncell = int(np.prod(sample_grid_shape(grid)))
    acc = np.zeros((ncell, SAMPLE_WORDS), dtype=np.uint64)
    c = cell[inside]
    order = np.argsort(c, kind="stable")
    cs = c[order]
    starts = np.flatnonzero(np.concatenate([[True], cs[1:] != cs[:-1]])) if len(cs) else np.zeros(0, dtype=np.int64)
    acc[:, 0] = np.bincount(c, minlength=ncell).astype(np.uint64)
    words = []
    for k in ("vx", "vy", "vz"):
        words += list(sample_limbs(sel(state[k])[inside], SAMPLE_V1, SAMPLE_V2))
    for k in ("vx", "vy", "vz"):
        v = np.asarray(sel(state[k]), dtype=np.float64)[inside]
        words += list(sample_limbs(v * v, SAMPLE_Q1, SAMPLE_Q2))
    if len(cs):
        for j, w in enumerate(words):       # per-cell sums of the sorted words (uint64 adds wrap mod 2^64)
            acc[cs[starts], 1 + j] = np.add.reduceat(w.view(np.uint64)[order], starts)
    return acc, 1, int(np.count_nonzero(~inside))


def merge_sample_ranks(parts):
    """Raw samples of the ranks of one run (each (acc, n_samples, n_outside)): element-wise sums mod 2^64; every rank
    took the same samples."""
    parts = list(parts)
    ns = {int(p[1]) for p in parts}
    if len(ns) != 1:
        raise AmcError("ranks disagree on the number of samples taken: %s" % sorted(ns))
    acc = parts[0][0].copy()
    with np.errstate(over="ignore"):
        for p in parts[1:]:
            acc += p[0]
    return acc, ns.pop(), sum(int(p[2]) for p in parts) & ((1 << 64) - 1)


class SurfaceLayout:
    """The wall elements of a handle (amc_surface_layout): per case its bin type -- "side" (z layers of `zedge`),
    "annulus" (bounds `rsq`), "face" (cube face: in-plane owner cells) or None (no elements) -- and the case-major
    offsets[NUM_CASES + 1]."""

    def __init__(self, kind, grid, R_oa=None):
        self.kind = kind
        self.edges = [np.asarray(e, dtype=np.float64) for e in grid.edge]
        self.nc = tuple(len(e) - 1 for e in self.edges)
        self.zedge = self.edges[2]
        x = self.edges[0]
        self.dr = float((x[-1] - x[0]) / float(len(x) - 1))
        self.nann = 0 if kind == KIND_CUBE else int(math.ceil(float(R_oa) / self.dr))
        k = np.arange(self.nann + 1, dtype=np.float64)
        self.rsq = (k * self.dr) * (k * self.dr)
        self.types, counts = [], []
        for c in range(NUM_CASES):
            if kind == KIND_CUBE:
                t = "face" if c < 6 else None
                n = self.nc[self.face_axes(c)[1]] * self.nc[self.face_axes(c)[2]] if t else 0
            elif kind == KIND_PORE and c == 9:
                t, n = None, 0
            elif c in SIDE_CASES:
                t, n = "side", self.nc[2]
            else:
                t, n = "annulus", self.nann
            self.types.append(t)
            counts.append(n)
        self.offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)

    @staticmethod
    def face_axes(c):
        """(normal axis a, in-plane axes b1 < b2) of cube case c."""
        a = c >> 1
        return a, (1 if a == 0 else 0), (1 if a == 2 else 2)

    @property
    def n_elements(self):
        return int(self.offsets[-1])


def surface_layout_of(cfg, kind, grid):
    """NumPy restatement of amc_surface_layout for a handle of `kind` on `grid` (a slab run: the global grid)."""
    return SurfaceLayout(kind, grid, None if kind == KIND_CUBE else cfg.geom.R_oa)


def _bin_of(tab, v):
    """k with tab[k] <= v < tab[k+1], or -1 (NaN and anything outside the table)."""
    tab = np.asarray(tab, dtype=np.float64)
    k = np.searchsorted(tab, v, side="right") - 1
    with np.errstate(invalid="ignore"):
        ok = (v >= tab[0]) & (v < tab[-1])
    return np.where(ok, k, -1)


def surface_moments_of_hits(hits, layout, geom=None):
    """NumPy restatement of the surface accumulators: hits = dict of arrays "case", "col" [n, 3] (contact point),
    "v_in", "v_out" [n, 3], "dE" (the energy the gas gained), one entry per hit the wall phases applied, plus hits
    that apply nothing (col NaN: the reference's floating-point error path).  geom: the config's geometry (cylinder
    radii; not needed for the cube).  Returns (acc [elements][SURF_WORDS] uint64, outside [NUM_CASES] uint64) with
    the binning and the IEEE expressions of include/amc.h."""
    case = np.asarray(hits["case"], dtype=np.int64)
    col = np.asarray(hits["col"], dtype=np.float64).reshape(-1, 3)
    dv = np.asarray(hits["v_out"], dtype=np.float64).reshape(-1, 3) - np.asarray(hits["v_in"], dtype=np.float64).reshape(-1, 3)
    dE = np.asarray(hits["dE"], dtype=np.float64)
    n = len(case)
    elem = np.full(n, -1, dtype=np.int64)
    w = np.zeros((n, 3), dtype=np.float64)
    cx, cy, cz = col[:, 0], col[:, 1], col[:, 2]
    dvx, dvy, dvz = dv[:, 0], dv[:, 1], dv[:, 2]
    with np.errstate(invalid="ignore", divide="ignore"):
        for c in range(NUM_CASES):
            m = case == c
            t = layout.types[c]
            if not m.any() or t is None:
                continue
            if t == "face":
                a, b1, b2 = layout.face_axes(c)
                w[m, 0] = dv[m, a] if c & 1 else -dv[m, a]
                w[m, 1], w[m, 2] = dv[m, b1], dv[m, b2]
                o1, o2 = _bin_of(layout.edges[b1], col[m, b1]), _bin_of(layout.edges[b2], col[m, b2])
                e = np.where((o1 >= 0) & (o2 >= 0), o1 * layout.nc[b2] + o2, -1)
            elif t == "side":
                Rc = float(geom.R_oa_c if c == 0 else (geom.R_g_c if c == 5 else geom.R_p_c))
                ex, ey = cx[m] / Rc, cy[m] / Rc
                w[m, 0] = -(dvx[m] * ex + dvy[m] * ey)
                w[m, 1] = dvz[m]
                w[m, 2] = dvy[m] * ex - dvx[m] * ey
                e = _bin_of(layout.zedge, cz[m])
            else:
                r2 = cx[m] * cx[m] + cy[m] * cy[m]
                r = np.sqrt(r2)
                ex = np.where(r > 0.0, cx[m] / r, 1.0)
                ey = np.where(r > 0.0, cy[m] / r, 0.0)
                w[m, 0] = dvz[m] if c in PLUS_Z_CASES else -dvz[m]
                w[m, 1] = dvx[m] * ex + dvy[m] * ey
                w[m, 2] = dvy[m] * ex - dvx[m] * ey
                e = _bin_of(layout.rsq, r2)
            elem[m] = np.where(e >= 0, layout.offsets[c] + e, -1)
    inside = elem >= 0
    outside = np.bincount(case[~inside], minlength=NUM_CASES).astype(np.uint64)
    acc = np.zeros((layout.n_elements, SURF_WORDS), dtype=np.uint64)
    el = elem[inside]
    acc[:, 0] = np.bincount(el, minlength=layout.n_elements).astype(np.uint64)
    cols = [sample_limbs(w[inside, j], SURF_V1, SURF_V2) for j in range(3)] + [sample_limbs(dE[inside], SURF_E1, SURF_E2)]
    with np.errstate(over="ignore"):
        for j, (i1, i2) in enumerate(cols):
            np.add.at(acc[:, 1 + 2 * j], el, i1.view(np.uint64))
            np.add.at(acc[:, 2 + 2 * j], el, i2.view(np.uint64))
    return acc, outside


def merge_surface_ranks(parts):
    """Raw surface arrays of the ranks of one run (each (acc, n_steps, outside)): element-wise sums mod 2^64; every
    rank recorded the same wall phases."""
    parts = list(parts)
    ns = {int(p[1]) for p in parts}
    if len(ns) != 1:
        raise AmcError("ranks disagree on the number of wall phases recorded: %s" % sorted(ns))
    acc, out = parts[0][0].copy(), parts[0][2].copy()
    with np.errstate(over="ignore"):
        for p in parts[1:]:
            acc += p[0]
            out += p[2]
    return acc, ns.pop(), out


def vdf_edges(n_bins, v_max):
    """Bin edges of the velocity components and of the speed (amc_vdf_enable computes the same on the host)."""
    v = float(v_max)
    return np.linspace(-v, v, int(n_bins) + 1), np.linspace(0.0, v, int(n_bins) + 1)


def vdf_words_of(values, n_bins, lo, hi):
    """[under, bin 0 .. bin n_bins-1, over] of one histogram: np.histogram over [lo, hi] (last bin closed), values below
    lo in under, above hi or NaN in over."""
    values = np.asarray(values, dtype=np.float64)
    inside, _ = np.histogram(values, bins=int(n_bins), range=(lo, hi))
    under = int(np.count_nonzero(values < lo))
    over = len(values) - under - int(inside.sum())
    return np.concatenate([[under], inside, [over]]).astype(np.uint64)


def vdf_of_arrays(state, grid, n_bins, v_max, ids=None):
    """NumPy restatement of the VDF words one amc_sample_now adds for `state` (mapping with 'x', 'y', 'z', 'vx', 'vy',
    'vz'): acc [ncz][VDF_HISTS][n_bins + 2] uint64, the layout of Simulation.vdf_raw.  The particles are those of the
    field sample (sample_cells_of: inside the grid), the region is the z layer of their cell.  ids: optional indices
    into the arrays selecting the particles (default: all)."""
    sel = (lambda a: np.asarray(a, dtype=np.float64)) if ids is None else (lambda a: np.asarray(a, dtype=np.float64)[np.asarray(ids)])
    cell, inside = sample_cells_of(sel(state["x"]), sel(state["y"]), sel(state["z"]), grid)
    nz = sample_grid_shape(grid)[2]
    layer = cell[inside] % nz
    vx, vy, vz = (sel(state[k])[inside] for k in ("vx", "vy", "vz"))
    with np.errstate(over="ignore", invalid="ignore"):
        speed = np.sqrt((vx * vx + vy * vy) + vz * vz)
    v = float(v_max)
    acc = np.zeros((nz, VDF_HISTS, int(n_bins) + 2), dtype=np.uint64)
    order = np.argsort(layer, kind="stable")
    bounds = np.searchsorted(layer[order], np.arange(nz + 1))
    cols = [(a[order], lo) for a, lo in ((vx, -v), (vy, -v), (vz, -v), (speed, 0.0))]
    for k in range(nz):
        if bounds[k] < bounds[k + 1]:
            for j, (vals, lo) in enumerate(cols):
                acc[k, j] = vdf_words_of(vals[bounds[k]:bounds[k + 1]], n_bins, lo, v)
    return acc


def flux_counts_of(z, edge_z):
    """Plane count of every position: the number of planes edge_z[k] <= z (NaN: len(edge_z)), as amc_flux_* counts."""
    return np.searchsorted(np.asarray(edge_z, dtype=np.float64), np.asarray(z, dtype=np.float64), side="right")


def flux_of_states(state_prev, state_cur, edge_z):
    """NumPy restatement of the flux words one record point adds (include/amc.h): acc [planes][FLUX_WORDS] uint64 for
    the move from state_prev to state_cur (mappings with 'z' and, for state_cur, 'vx', 'vy', 'vz', indexed by particle
    id), planes edge_z.  Integer sums: the words of consecutive record points add up (mod 2^64) to those of the run."""
    c0, c1 = flux_counts_of(state_prev["z"], edge_z), flux_counts_of(state_cur["z"], edge_z)
    acc = np.zeros((len(edge_z), FLUX_WORDS), dtype=np.uint64)
    moved = np.flatnonzero(c0 != c1)
    if len(moved) == 0:
        return acc
    a, b = c0[moved], c1[moved]
    lo, n_planes = np.minimum(a, b), np.abs(b - a)
    sign = np.where(b > a, 1.0, -1.0)
    vx, vy, vz = (np.asarray(state_cur[k], dtype=np.float64)[moved] for k in ("vx", "vy", "vz"))
    with np.errstate(over="ignore", invalid="ignore"):
        q = (vx * vx + vy * vy) + vz * vz
    words = []
    for v, s1, s2 in ((vx, FLUX_V1, FLUX_V2), (vy, FLUX_V1, FLUX_V2), (vz, FLUX_V1, FLUX_V2), (q, FLUX_Q1, FLUX_Q2)):
        words += list(sample_limbs(sign * v, s1, s2))
    # one row per crossed plane: particle j crosses planes lo[j] .. lo[j] + n_planes[j] - 1
    j = np.repeat(np.arange(len(moved)), n_planes)
    plane = lo[j] + (np.arange(len(j)) - np.repeat(np.cumsum(n_planes) - n_planes, n_planes))
    up = b[j] > a[j]
    acc[:, 0] = np.bincount(plane[up], minlength=len(edge_z)).astype(np.uint64)
    acc[:, 1] = np.bincount(plane[~up], minlength=len(edge_z)).astype(np.uint64)
    with np.errstate(over="ignore"):
        for k, w in enumerate(words):
            np.add.at(acc[:, 2 + k], plane, w.view(np.uint64)[j])
    return acc


def combine_digests(parts):
    """Sum of per-rank digests (mod 2^64 per component)."""
    m = (1 << 64) - 1
    return tuple(sum(p[i] for p in parts) & m for i in range(3))


class Simulation:
    """One simulation domain resident on one GPU.

    cfg: a namespace from ``config.cube_config`` / ``config.pore_config``.
    kind / pp_mode default to the script the config belongs to (cube: six planes + serial sweep;
    pore / temp: pore walls + 8 colour groups)."""

    def __init__(self, cfg, *, kind=None, pp_mode=None, rng_mode=RNG_DEVICE, taps=0, device=0, seed=None,
                 max_particles=None, pair_capacity=1 << 20, path_capacity=1 << 22, grid=None, cheb=None):
        self.lib = load_library()
        self.cfg = cfg
        default_kind = {"cube": KIND_CUBE, "pore": KIND_PORE, "temp": KIND_TEMP}[cfg.kind]
        self.kind = default_kind if kind is None else kind
        self.pp_mode = (PP_SWEEP if cfg.kind == "cube" else PP_GROUPS) if pp_mode is None else pp_mode
        self.rng_mode = rng_mode
        grid = grid or cfg.grid
        c = AmcConfig()
        c.abi_version = ABI_VERSION
        c.kind, c.pp_mode, c.rng_mode, c.taps = self.kind, self.pp_mode, rng_mode, taps
        c.dt = float(cfg.dt)
        self._keep = []
        if cfg.kind == "cube":
            c.cube[0], c.cube[1], c.cube[2] = cfg.cube_x, cfg.cube_y, cfg.cube_z
            c.geom.argon_mass, c.geom.argon_radius = cfg.argon_mass, cfg.argon_radius
            c.geom.collision_range = cfg.collision_range
        else:
            for k in GEOM_FIELDS:
                setattr(c.geom, k, float(getattr(cfg.geom, k)))
        for a in range(3):
            c.nc[a], c.c0[a] = grid.nc[a], grid.c0[a]
            e, lo = np.ascontiguousarray(grid.edge[a], dtype=np.float64), np.ascontiguousarray(grid.lo[a], dtype=np.float64)
            self._keep += [e, lo]
            c.edge[a], c.lo[a] = _dp(e), _dp(lo)
        c.overlap_sq = overlap_threshold(cfg.collision_range)
        c.seed = int(cfg.seed if seed is None else seed)
        if self.kind == KIND_TEMP and rng_mode == RNG_DEVICE:
            if cheb is None:
                from .config import gap_energy_chebyshev
                cheb = gap_energy_chebyshev(cfg, 16)
            coef = np.ascontiguousarray(cheb[0], dtype=np.float64)
            self._keep.append(coef)
            c.cheb_coef, c.cheb_n, c.cheb_zmid, c.cheb_inv_half = _dp(coef), len(coef), cheb[1], cheb[2]
        self.cheb = cheb
        edges = np.linspace(HIST_RANGE[0], HIST_RANGE[1], NUM_BINS + 1)
        self._keep.append(edges)
        self.hist_edges = edges
        c.hist_first, c.hist_last, c.hist_edges = float(HIST_RANGE[0]), float(HIST_RANGE[1]), _dp(edges)
        c.max_particles = int(max_particles if max_particles is not None else cfg.num_molecules)
        c.pair_capacity, c.path_capacity = int(pair_capacity), int(path_capacity)
        self._c = c
        self.h = C.c_void_p()
        rc = self.lib.amc_create(C.byref(c), int(device), C.byref(self.h))
        if rc != 0:
            msg = self.lib.amc_last_error(None)
            self.h = None
            raise AmcError("amc_create failed (%d): %s" % (rc, msg.decode() if msg else "?"))
        self.n = 0
        self.sample_grid = grid     # a slab rank's handle samples the global grid (slab.SlabRank sets it)
        self.sampling = None    # (every, first_step) while field sampling is enabled
        self.host_steps = 0     # timesteps taken by step_host_rng (the index the sampling schedule of that path uses)
        self.surface_on = False  # surface recording enabled (amc_surface_enable)
        self.vdf = None         # (n_bins, v_max) while the velocity distribution is enabled
        self.flux_on = False    # plane flux recording enabled (amc_flux_enable)

    # ------------------------------------------------------------------ plumbing
    def _check(self, rc, what):
        if rc != 0:
            msg = self.lib.amc_last_error(self.h)
            raise AmcError("%s failed (%d): %s" % (what, rc, msg.decode() if msg else "?"))

    def close(self):
        if getattr(self, "h", None):
            self.lib.amc_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ------------------------------------------------------------------ state
    def set_state(self, x, y, z, vx, vy, vz, dist=None, dist_x=None, dist_y=None, dist_z=None, flag=None):
        f = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)
        arrs = [f(a) for a in (x, y, z, vx, vy, vz, dist, dist_x, dist_y, dist_z)]
        fl = None if flag is None else np.ascontiguousarray(np.asarray(flag).astype(np.uint8))
        n = len(arrs[0])
        rc = self.lib.amc_set_state(self.h, C.c_int64(n), *[_dp(a) for a in arrs],
                                    fl.ctypes.data_as(c_uint8_p) if fl is not None else None)
        self._check(rc, "amc_set_state")
        self.n = n

    def init_synthetic(self, spec):
        """Generate the synthetic Maxwellian state described by an AmcInitSpec on the device (init_state.pore_spec /
        cube_spec build one); returns the number of particles this handle holds afterwards."""
        n = C.c_int64(0)
        self._check(self.lib.amc_init_synthetic(self.h, C.byref(spec), C.byref(n)), "amc_init_synthetic")
        self.n = int(n.value)
        return self.n

    def seed_relax(self, max_rounds=8):
        """Overlap-free seeding after init_synthetic (amc_seed_relax): returns (positions re-drawn, particles still
        overlapping a neighbour afterwards)."""
        a, b = C.c_int64(0), C.c_int64(0)
        self._check(self.lib.amc_seed_relax(self.h, C.c_int32(max_rounds), C.byref(a), C.byref(b)), "amc_seed_relax")
        return int(a.value), int(b.value)

    def get_state(self, out=None):
        """dict of the ten float64 arrays and the uint8 flag, original particle index order.
        `out`: optional dict of preallocated (e.g. pinned) arrays to fill."""
        keys = ("x", "y", "z", "vx", "vy", "vz", "dist", "dist_x", "dist_y", "dist_z")
        if out is None:
            out = {k: np.empty(self.n, dtype=np.float64) for k in keys}
            out["flag"] = np.empty(self.n, dtype=np.uint8)
        rc = self.lib.amc_get_state(self.h, *[_dp(out[k]) for k in keys], out["flag"].ctypes.data_as(c_uint8_p))
        self._check(rc, "amc_get_state")
        return out

    # ------------------------------------------------------------------ stepping
    def step(self, n_steps=1):
        """n_steps whole timesteps on the device; returns a list of per-step counter dicts."""
        st = (AmcStepStats * n_steps)()
        self._check(self.lib.amc_step(self.h, C.c_int32(n_steps), st), "amc_step")
        return [s.as_dict() for s in st]

    def step_quiet(self, n_steps=1):
        self._check(self.lib.amc_step(self.h, C.c_int32(n_steps), None), "amc_step")

    def drift(self):
        self._check(self.lib.amc_drift(self.h), "amc_drift")

    def walls(self):
        st = AmcStepStats()
        self._check(self.lib.amc_walls(self.h, C.byref(st)), "amc_walls")
        return st.as_dict()

    def recapture(self, with_after=False):
        cnt, after = C.c_int64(0), C.c_int64(0)
        self._check(self.lib.amc_recapture(self.h, C.byref(cnt), C.byref(after)), "amc_recapture")
        return (int(cnt.value), int(after.value)) if with_after else int(cnt.value)

    def pairs(self):
        st = AmcStepStats()
        self._check(self.lib.amc_pairs(self.h, C.byref(st)), "amc_pairs")
        return st.as_dict()

    def set_step_index(self, step):
        self._check(self.lib.amc_set_step_index(self.h, C.c_int64(step)), "amc_set_step_index")

    # ------------------------------------------------------------------ host-RNG parity mode
    def wall_case(self, case):
        n = C.c_int64(0)
        self._check(self.lib.amc_wall_case(self.h, int(case), C.byref(n)), "amc_wall_case")
        return int(n.value)

    def wall_hits_pending(self, case, cap=None):
        cap = int(cap or max(self.n, 1))
        idx = np.zeros(cap, dtype=np.int64)
        nrm = np.zeros(3 * cap)
        colz = np.zeros(cap)
        n = C.c_int64(0)
        rc = self.lib.amc_wall_hits_pending(self.h, int(case), C.c_int64(cap), C.byref(n), idx.ctypes.data_as(c_int64_p),
                                            _dp(nrm), _dp(colz))
        self._check(rc, "amc_wall_hits_pending")
        k = int(n.value)
        return idx[:k].copy(), nrm[:3 * k].reshape(k, 3).copy(), colz[:k].copy()

    def wall_apply_directions(self, case, idx, dirs, surf_e=None):
        k = len(idx)
        idx = np.ascontiguousarray(idx, dtype=np.int64)
        dirs = np.ascontiguousarray(dirs, dtype=np.float64).reshape(-1) if k else np.zeros(3)
        se = np.ascontiguousarray(surf_e, dtype=np.float64) if surf_e is not None else None
        dpz, de = np.zeros(max(k, 1)), np.zeros(max(k, 1))
        errs = C.c_int64(0)
        rc = self.lib.amc_wall_apply_directions(self.h, int(case), C.c_int64(k), idx.ctypes.data_as(c_int64_p), _dp(dirs),
                                                _dp(se), _dp(dpz), _dp(de), C.byref(errs))
        self._check(rc, "amc_wall_apply_directions")
        return dpz[:k], de[:k], int(errs.value)

    def step_host_rng(self, surface_energy_gap=None):
        """One Temperature_Pore_MC timestep with the reference's host Mersenne-Twister draws
        (Temp:662-853): walls case by case, directions drawn on the host in the reference's order,
        per-hit contributions summed sequentially like the reference's mpf accumulators."""
        from . import host_rng
        from .config import surface_energy_gap as seg
        cfg = self.cfg
        self.drift()
        dpz = e_hot = e_cold = 0
        counts = np.zeros(NUM_CASES, dtype=np.int64)
        errors = 0
        for case in range(NUM_CASES):
            if case <= 2:
                counts[case] = self.wall_case(case)
                continue
            idx, nrm, colz = self.wall_hits_pending(case)
            counts[case] = len(idx)
            surf = None
            if case == 5:
                dirs = np.zeros((len(idx), 3))
                surf = np.zeros(len(idx))
                for k in range(len(idx)):
                    if nrm[k, 0] == nrm[k, 0]:
                        dirs[k] = host_rng.inbound_direction(nrm[k])
                        surf[k] = float((surface_energy_gap or (lambda z: seg(cfg, z)))(colz[k]))
            else:
                dirs = host_rng.directions_for_hits(nrm)
            p, e, er = self.wall_apply_directions(case, idx, dirs, surf)
            errors += er
            sp = se = 0
            for k in range(len(idx)):      # sequential sums, ascending particle index (Temp:385,389)
                sp = sp + p[k]
                se = se + e[k]
            dpz = dpz + sp
            if case in (3, 7, 9):
                e_cold = e_cold + se
            elif case in (4, 6, 8):
                e_hot = e_hot + se
        oob_walls, oob_walls_after = self.recapture(True)
        st = self.pairs()
        oob_pp, oob_pp_after = self.recapture(True)
        wall_hits = int(counts[3:].sum())
        st.update(wall_hits=counts, wall_collisions=wall_hits, oob_after_walls=oob_walls, oob_after_pp=oob_pp,
                  oob_after_walls_recapture=oob_walls_after, oob_after_pp_recapture=oob_pp_after,
                  dpz=dpz, e_cold=e_cold, e_hot=e_hot, collisions=wall_hits + st["pp_collisions"],
                  errors=st["errors"] + errors)
        self.host_steps += 1
        if self.sample_due(self.host_steps - 1):
            self.sample_now()
        if self.flux_on:
            self.flux_now()
        return st

    # ------------------------------------------------------------------ field sampling
    def sample_enable(self, every=0, first_step=0):
        """Accumulate per-cell moments of the state (amc_sample_enable): after every timestep s with s >= first_step
        and (s - first_step) % every == 0 (every = 0: only on sample_now()).  Zeroes the accumulators."""
        self._check(self.lib.amc_sample_enable(self.h, C.c_int32(int(every)), C.c_int64(int(first_step))), "amc_sample_enable")
        self.sampling = (int(every), int(first_step))

    def sample_disable(self):
        self._check(self.lib.amc_sample_disable(self.h), "amc_sample_disable")
        self.sampling = None
        self.vdf = None         # amc_sample_disable frees the VDF too

    def sample_due(self, step):
        if self.sampling is None or self.sampling[0] <= 0:
            return False
        every, first = self.sampling
        return step >= first and (step - first) % every == 0

    def sample_now(self):
        """One sample of the current state."""
        self._check(self.lib.amc_sample_now(self.h), "amc_sample_now")

    def sample_cells(self):
        return int(np.prod(sample_grid_shape(self.sample_grid)))

    def sample_raw(self):
        """(acc [cells][SAMPLE_WORDS] uint64, samples taken, particles found outside the grid)."""
        acc = np.zeros((self.sample_cells(), SAMPLE_WORDS), dtype=np.uint64)
        ns, no = C.c_uint64(0), C.c_uint64(0)
        self._check(self.lib.amc_sample_get_raw(self.h, acc.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(ns), C.byref(no)),
                    "amc_sample_get_raw")
        return acc, int(ns.value), int(no.value)

    def sample_set_raw(self, acc, n_samples, n_outside):
        acc = np.ascontiguousarray(acc, dtype=np.uint64)
        if acc.size != self.sample_cells() * SAMPLE_WORDS:
            raise AmcError("sample accumulators of %d words for a grid of %d cells" % (acc.size, self.sample_cells()))
        self._check(self.lib.amc_sample_set_raw(self.h, acc.ctypes.data_as(C.POINTER(C.c_uint64)), C.c_uint64(int(n_samples)),
                                                C.c_uint64(int(n_outside))), "amc_sample_set_raw")

    def last_sample_ms(self):
        """Device time (ms) of the sampling kernel, summed over the samples of the last step() / sample_now() call."""
        v = C.c_double(0.0)
        self._check(self.lib.amc_last_sample_ms(self.h, C.byref(v)), "amc_last_sample_ms")
        return float(v.value)

    # ------------------------------------------------------------------ velocity distribution
    def vdf_enable(self, n_bins, v_max):
        """Histogram vx, vy, vz over [-v_max, v_max] and the speed over [0, v_max] per z layer of the sampling grid,
        on the samples of the field sample (amc_vdf_enable; field sampling must be on).  Zeroes the histograms."""
        self._check(self.lib.amc_vdf_enable(self.h, C.c_int32(int(n_bins)), C.c_double(float(v_max))), "amc_vdf_enable")
        self.vdf = (int(n_bins), float(v_max))

    def vdf_disable(self):
        self._check(self.lib.amc_vdf_disable(self.h), "amc_vdf_disable")
        self.vdf = None

    def vdf_layout(self):
        """(layers, bins, v_max) of the enabled VDF."""
        ncz, nb, vm = C.c_int32(0), C.c_int32(0), C.c_double(0.0)
        self._check(self.lib.amc_vdf_layout(self.h, C.byref(ncz), C.byref(nb), C.byref(vm)), "amc_vdf_layout")
        return int(ncz.value), int(nb.value), float(vm.value)

    def vdf_raw(self):
        """acc [layers][VDF_HISTS][n_bins + 2] uint64: [under, bins, over] of vx, vy, vz and the speed per layer."""
        ncz, nb, _ = self.vdf_layout()
        acc = np.zeros((ncz, VDF_HISTS, nb + 2), dtype=np.uint64)
        self._check(self.lib.amc_vdf_get_raw(self.h, acc.ctypes.data_as(C.POINTER(C.c_uint64))), "amc_vdf_get_raw")
        return acc

    def vdf_set_raw(self, acc):
        ncz, nb, _ = self.vdf_layout()
        acc = np.ascontiguousarray(acc, dtype=np.uint64)
        if acc.size != ncz * VDF_HISTS * (nb + 2):
            raise AmcError("VDF histograms of %d words for a layout of %d layers x %d bins" % (acc.size, ncz, nb))
        self._check(self.lib.amc_vdf_set_raw(self.h, acc.ctypes.data_as(C.POINTER(C.c_uint64))), "amc_vdf_set_raw")

    # ------------------------------------------------------------------ surface recording
    def surface_enable(self):
        """Record every wall interaction into per-element accumulators (amc_surface_enable); zeroes them."""
        self._check(self.lib.amc_surface_enable(self.h), "amc_surface_enable")
        self.surface_on = True

    def surface_disable(self):
        self._check(self.lib.amc_surface_disable(self.h), "amc_surface_disable")
        self.surface_on = False

    def surface_layout(self):
        """offsets[NUM_CASES + 1] int64: the elements of case c are offsets[c] .. offsets[c+1]."""
        off = np.zeros(NUM_CASES + 1, dtype=np.int64)
        self._check(self.lib.amc_surface_layout(self.h, off.ctypes.data_as(c_int64_p)), "amc_surface_layout")
        return off

    def surface_raw(self):
        """(acc [elements][SURF_WORDS] uint64, wall phases recorded, outside [NUM_CASES] uint64)."""
        acc = np.zeros((int(self.surface_layout()[-1]), SURF_WORDS), dtype=np.uint64)
        out = np.zeros(NUM_CASES, dtype=np.uint64)
        ns = C.c_uint64(0)
        u64 = C.POINTER(C.c_uint64)
        self._check(self.lib.amc_surface_get_raw(self.h, acc.ctypes.data_as(u64), C.byref(ns), out.ctypes.data_as(u64)),
                    "amc_surface_get_raw")
        return acc, int(ns.value), out

    def surface_set_raw(self, acc, n_steps, outside):
        acc = np.ascontiguousarray(acc, dtype=np.uint64)
        outside = np.ascontiguousarray(outside, dtype=np.uint64)
        if acc.size != int(self.surface_layout()[-1]) * SURF_WORDS or outside.size != NUM_CASES:
            raise AmcError("surface accumulators of %d words for a layout of %d elements" % (acc.size, int(self.surface_layout()[-1])))
        u64 = C.POINTER(C.c_uint64)
        self._check(self.lib.amc_surface_set_raw(self.h, acc.ctypes.data_as(u64), C.c_uint64(int(n_steps)), outside.ctypes.data_as(u64)),
                    "amc_surface_set_raw")

    # ------------------------------------------------------------------ plane flux recording
    def flux_enable(self):
        """Count the particles crossing the z planes of the sampling grid, and what they carry, at every timestep of
        step() and at every flux_now() (amc_flux_enable); zeroes the words and takes the snapshot of the current state."""
        self._check(self.lib.amc_flux_enable(self.h), "amc_flux_enable")
        self.flux_on = True

    def flux_disable(self):
        self._check(self.lib.amc_flux_disable(self.h), "amc_flux_disable")
        self.flux_on = False

    def flux_now(self):
        """One record point: the crossings since the previous one (step_host_rng calls it after its timestep)."""
        self._check(self.lib.amc_flux_now(self.h), "amc_flux_now")

    def flux_layout(self):
        """Number of planes (z edges of the sampling grid)."""
        n = C.c_int32(0)
        self._check(self.lib.amc_flux_layout(self.h, C.byref(n)), "amc_flux_layout")
        return int(n.value)

    def flux_raw(self):
        """(acc [planes][FLUX_WORDS] uint64, record points taken)."""
        acc = np.zeros((self.flux_layout(), FLUX_WORDS), dtype=np.uint64)
        ns = C.c_uint64(0)
        self._check(self.lib.amc_flux_get_raw(self.h, acc.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(ns)), "amc_flux_get_raw")
        return acc, int(ns.value)

    def flux_set_raw(self, acc, n_steps):
        acc = np.ascontiguousarray(acc, dtype=np.uint64)
        n = self.flux_layout()
        if acc.size != n * FLUX_WORDS:
            raise AmcError("flux words of %d words for a layout of %d planes" % (acc.size, n))
        self._check(self.lib.amc_flux_set_raw(self.h, acc.ctypes.data_as(C.POINTER(C.c_uint64)), C.c_uint64(int(n_steps))),
                    "amc_flux_set_raw")

    # ------------------------------------------------------------------ outputs
    def histograms(self):
        """(counts[4, 200] uint64 in the order total/x/y/z, number of completed paths, sums[4])."""
        counts = np.zeros((4, NUM_BINS), dtype=np.uint64)
        n = C.c_uint64(0)
        sums = np.zeros(4)
        rc = self.lib.amc_get_histograms(self.h, counts.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(n), _dp(sums))
        self._check(rc, "amc_get_histograms")
        return counts, int(n.value), sums

    def pair_list(self, cap=1 << 20):
        hi, lo = np.zeros(cap, dtype=np.int64), np.zeros(cap, dtype=np.int64)
        grp, cell = np.zeros(cap, dtype=np.int32), np.zeros(cap, dtype=np.int32)
        n = C.c_int64(0)
        rc = self.lib.amc_get_pair_list(self.h, C.c_int64(cap), C.byref(n), hi.ctypes.data_as(c_int64_p),
                                        lo.ctypes.data_as(c_int64_p), grp.ctypes.data_as(C.POINTER(C.c_int32)),
                                        cell.ctypes.data_as(C.POINTER(C.c_int32)))
        self._check(rc, "amc_get_pair_list")
        k = int(n.value)
        return hi[:k].copy(), lo[:k].copy(), grp[:k].copy(), cell[:k].copy()

    def wall_bits(self):
        bits = np.zeros(max(self.n, 1), dtype=np.uint16)
        self._check(self.lib.amc_get_wall_bits(self.h, bits.ctypes.data_as(C.POINTER(C.c_uint16))), "amc_get_wall_bits")
        return bits[:self.n]

    def completed_paths(self, cap=1 << 22):
        arrs = [np.zeros(cap) for _ in range(4)]
        n = C.c_int64(0)
        rc = self.lib.amc_get_completed_paths(self.h, C.c_int64(cap), C.byref(n), *[_dp(a) for a in arrs])
        self._check(rc, "amc_get_completed_paths")
        k = int(n.value)
        return tuple(a[:k].copy() for a in arrs)

    # ------------------------------------------------------------------ checkpoint / resume
    def checkpoint(self, path=None):
        """Everything needed to continue the run exactly: particle state, histograms, free-path sums
        (raw fixed-point limbs) and the step index that keys the device RNG.  Returns the dict and, if
        `path` is given, writes it with np.savez."""
        st = self.get_state()
        counts = np.zeros((4, NUM_BINS), dtype=np.uint64)
        n = C.c_uint64(0)
        limbs = np.zeros(8, dtype=np.uint64)
        rc = self.lib.amc_get_outputs_raw(self.h, counts.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(n),
                                          limbs.ctypes.data_as(C.POINTER(C.c_uint64)))
        self._check(rc, "amc_get_outputs_raw")
        st.update(hist_counts=counts, n_paths=np.uint64(n.value), path_limbs=limbs,
                  step_index=np.int64(self.lib.amc_get_step_index(self.h)))
        if self.rng_mode == RNG_HOST:
            # parity mode draws from the two global Mersenne-Twister streams (host_rng.py): part of the state
            import pickle
            import random
            st["host_rng"] = np.frombuffer(pickle.dumps((np.random.get_state(), random.getstate())), dtype=np.uint8)
        if self.sampling is not None:
            acc, ns, no = self.sample_raw()
            st.update(sample_acc=acc, sample_n=np.uint64(ns), sample_outside=np.uint64(no),
                      sample_schedule=np.array(self.sampling, dtype=np.int64), host_steps=np.int64(self.host_steps))
        if self.vdf is not None:
            st.update(vdf_acc=self.vdf_raw(), vdf_bins=np.int64(self.vdf[0]), vdf_vmax=np.float64(self.vdf[1]))
        if self.surface_on:
            acc, ns, out = self.surface_raw()
            st.update(surface_acc=acc, surface_n_steps=np.uint64(ns), surface_outside=out)
        if self.flux_on:
            acc, ns = self.flux_raw()
            st.update(flux_acc=acc, flux_n_steps=np.uint64(ns))
        if path is not None:
            np.savez(path, **st)
        return st

    def restore(self, ck):
        """ck: dict from checkpoint() or the path of an .npz written by it."""
        if isinstance(ck, (str, bytes)) or hasattr(ck, "__fspath__"):
            ck = dict(np.load(ck))
        self.set_state(*[ck[k] for k in ("x", "y", "z", "vx", "vy", "vz", "dist", "dist_x", "dist_y", "dist_z")], flag=ck["flag"])
        counts = np.ascontiguousarray(ck["hist_counts"], dtype=np.uint64)
        limbs = np.ascontiguousarray(ck["path_limbs"], dtype=np.uint64)
        rc = self.lib.amc_set_outputs_raw(self.h, counts.ctypes.data_as(C.POINTER(C.c_uint64)), C.c_uint64(int(ck["n_paths"])),
                                          limbs.ctypes.data_as(C.POINTER(C.c_uint64)))
        self._check(rc, "amc_set_outputs_raw")
        self.set_step_index(int(ck["step_index"]))
        if self.rng_mode == RNG_HOST:
            if "host_rng" not in ck:
                raise AmcError("checkpoint of a host-RNG run without the Mersenne-Twister states: exact resume impossible")
            import pickle
            import random
            np_state, py_state = pickle.loads(np.asarray(ck["host_rng"], dtype=np.uint8).tobytes())
            np.random.set_state(np_state)
            random.setstate(py_state)
        if "sample_acc" in ck:          # checkpoints written without sampling have none of these keys
            every, first = (int(v) for v in ck["sample_schedule"])
            self.sample_enable(every, first)
            self.sample_set_raw(ck["sample_acc"], int(ck["sample_n"]), int(ck["sample_outside"]))
            self.host_steps = int(ck["host_steps"])
        if "vdf_acc" in ck:             # checkpoints written without the VDF have none of these keys
            self.vdf_enable(int(ck["vdf_bins"]), float(ck["vdf_vmax"]))
            self.vdf_set_raw(ck["vdf_acc"])
        if "surface_acc" in ck:         # checkpoints written without surface recording have none of these keys
            self.surface_enable()
            self.surface_set_raw(ck["surface_acc"], int(ck["surface_n_steps"]), ck["surface_outside"])
        if "flux_acc" in ck:            # checkpoints written without flux recording have none of these keys
            self.flux_enable()          # the snapshot of the restored state: the one the checkpointed handle held
            self.flux_set_raw(ck["flux_acc"], int(ck["flux_n_steps"]))

    def state_digest(self):
        """(sum0, sum1, count): order-independent checksum of the owned particle state, computed on the device
        (amc_state_digest); equals digest_of_arrays(arange(n), get_state()) for a single-domain handle."""
        out = (C.c_uint64 * 3)()
        self._check(self.lib.amc_state_digest(self.h, out), "amc_state_digest")
        return int(out[0]), int(out[1]), int(out[2])

    def clear_taps(self):
        self._check(self.lib.amc_clear_taps(self.h), "amc_clear_taps")

    def last_timing(self):
        """(ms[5], launches) of the last step() call: advect+walls, cell sort, pair kernels,
        recapture, total -- CUDA events on the handle's stream."""
        ms = (C.c_double * 5)()
        n = C.c_int64(0)
        self._check(self.lib.amc_last_timing(self.h, ms, C.byref(n)), "amc_last_timing")
        return list(ms), int(n.value)

    def last_scatter_ms(self):
        """Device time (ms) of k_scatter_advect alone, summed over the steps of the last step() call."""
        v = C.c_double(0.0)
        self._check(self.lib.amc_last_scatter_ms(self.h, C.byref(v)), "amc_last_scatter_ms")
        return float(v.value)

    def last_detect_ms(self):
        """Device time (ms) of the detection kernel alone, summed over the steps of the last step() call."""
        v = C.c_double(0.0)
        self._check(self.lib.amc_last_detect_ms(self.h, C.byref(v)), "amc_last_detect_ms")
        return float(v.value)
