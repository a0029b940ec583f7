// amc_device.cuh -- device-side types and per-particle physics of libamc.so.
//
// Arithmetic contract (SURVEY Appendix E): everything that decides a flag (wall masks, cell
// membership, the overlap test) and everything that updates particle state is IEEE fp64 in the
// reference's operation order with separate multiply / add roundings.  This translation unit is
// compiled with -fmad=false, so no contraction happens unless an explicit __fma_rn is written.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "amc.h"

#define AMC_FLAG_PATH 1u /* full_path_traveled (Pore:392) */
#define AMC_FLAG_ESC 2u  /* transient: particle left its sorted owner cell during the pair pass */
/* slab decomposition (multi-GPU), all transient within one timestep */
#define AMC_FLAG_GHOST 4u     /* copy of a particle owned by a neighbouring rank */
#define AMC_FLAG_REL_UP 8u    /* the rank above holds a copy of / owns this particle */
#define AMC_FLAG_REL_DOWN 16u /* the rank below holds a copy of / owns this particle */
#define AMC_FLAG_LATE_UP 32u  /* immigrant that landed in the top band: export it before the first group */
#define AMC_FLAG_DIRTY_UP 64u  /* already queued for the boundary exchange of the current group */
#define AMC_FLAG_DIRTY_DOWN 128u
#define AMC_FLAG_KEEP (AMC_FLAG_PATH | AMC_FLAG_GHOST | AMC_FLAG_REL_UP | AMC_FLAG_REL_DOWN)
#define AMC_REC 12            /* doubles per exchanged particle record: 10 state, id, flags */

#define AMC_MAX_MEMBERS 512  /* particles per reference cell incl. overlap band (reference: <= 308) */
#define AMC_MAX_CAND 64     /* simultaneously overlapping pairs per cell visit */
#define AMC_WI 32            /* ints per work item: cell, kx, ky, kz, beg[8], len[8], 6 doubles of bounds = 128 bytes */
#define AMC_MAX_HITS 8      /* filter hits of one cell that k_detect hands to the resolution as a list */
#define AMC_HIT_REC (1 + 2 * AMC_MAX_HITS) /* ints per work item in wl_hit: count (-1: search the cell), then slot pairs */
#define AMC_CELL_DIRTY 0x40000000 /* bit of cell_n: a particle entered / left the cell after k_detect looked at it */
#define AMC_WL_COUNTERS 24 /* wl_count[8], wl_next[8], dl_count, padding */
#define AMC_XBINS 64         /* slabs along x of the neighbour search inside a flagged cell, at most */

/* how much of a timestep's per-particle work a kernel carries out (advance_particle and the wall helpers):
   DRY: only what decides the final position; LIVE: everything; QUIET: the full state update, but no counters,
   completed paths or accumulators (the live run of the same particle records them) */
enum { AMC_DRY = 0, AMC_LIVE = 1, AMC_QUIET = 2 };
enum { PH_DRIFT = 1, PH_WALLS = 2, PH_RECAP = 4, PH_KEYS = 8, PH_SAVE_PRIOR = 16, PH_LOAD_PRIOR = 32, PH_RECAP_POST = 64 };

// Position record: what the neighbour search, the membership tests and the sort read together is stored together --
// one 32-byte, 32-byte-aligned record per particle, moved with single 256-bit accesses (LDG.E.256 / STG.E.256) and,
// being contiguous per owner cell, with bulk copies (cp.async.bulk) into shared memory by the detection pass.
// Velocities and the four path accumulators stay structure-of-arrays: only the streaming passes and the (rare)
// collisions touch them.
struct __align__(32) PosRec {
    double x, y, z;
    int32_t id;    /* original particle index */
    uint32_t flag; /* AMC_FLAG_* */
};
struct Arrays {
    PosRec *pos;
    double *vx, *vy, *vz, *d, *dx, *dy, *dz;
};
// separate x / y / z / id / flag arrays laid over an idle record array of `cap` records (29 of its 32 bytes per particle):
// staging between the C ABI's arrays and the records
struct SoaView {
    double *x, *y, *z;
    int32_t *id;
    uint8_t *flag;
};
__host__ __device__ __forceinline__ SoaView soa_view(PosRec *base, int64_t cap)
{
    SoaView v;
    v.x = reinterpret_cast<double *>(base); v.y = v.x + cap; v.z = v.y + cap;
    v.id = reinterpret_cast<int32_t *>(v.z + cap); v.flag = reinterpret_cast<uint8_t *>(v.id + cap);
    return v;
}
// the whole record with one 256-bit store (sm_100: st.global.v4.b64 -> STG.E.256; the compiler emits the 256-bit LOAD
// for a plain record read by itself, but splits a store whose fields come from different registers)
__device__ __forceinline__ void st_pos(PosRec *p, const double x, const double y, const double z, const int32_t id, const uint32_t flag)
{
    const unsigned long long w = (unsigned long long)(uint32_t)id | ((unsigned long long)flag << 32);
    asm volatile("st.global.v4.b64 [%0], {%1, %2, %3, %4};" ::"l"(p), "d"(x), "d"(y), "d"(z), "l"(w) : "memory");
}
// a position record past L1 (producer -> consumer edges inside one launch, see k_pairs_group)
__device__ __forceinline__ PosRec ldcg_pos(const PosRec *p)
{
    PosRec r;
    unsigned long long w;
    asm volatile("ld.global.cg.v2.b64 {%0, %1}, [%2];" : "=d"(r.x), "=d"(r.y) : "l"(p));
    asm volatile("ld.global.cg.v2.b64 {%0, %1}, [%2];" : "=d"(r.z), "=l"(w) : "l"(reinterpret_cast<const char *>(p) + 16));
    r.id = (int32_t)(uint32_t)w; r.flag = (uint32_t)(w >> 32);
    return r;
}

struct StatsDev {
    unsigned long long wall_hits[AMC_NUM_CASES];
    unsigned long long pp, checks_ref, checks_exec, oob_walls, oob_pp, oob_walls_after, oob_pp_after, errors, paths;
    unsigned long long cell_overflow, cand_overflow, esc_overflow;
    unsigned long long dpz[2], ecold[2], ehot[2]; /* two-limb fixed point, see acc_add */
};

struct P {
    int64_t n;
    int64_t cap;          /* slots of every per-particle array */
    Arrays a, b;
    double *px, *py, *pz;
    int32_t *key, *rank;
    int32_t *band_count, *rest_count; /* per owner cell: particles inside / outside a low-side band of a next cell */
    int32_t *cell_start;
    int32_t ncell_pad;
    int32_t pnc[3];
    int32_t kind, pp_mode;
    double dt;
    double cube[3];
    amc_geom g;
    int32_t nc[3];
    const double *edge[3];
    const double *lo[3];
    double e0[3], inv_d[3];
    double overlap_sq, cr, mass;
    /* exact squared-radius thresholds: sqrt(v) > R <=> v > gt_*,  sqrt(v) < R <=> v < lt_* (sqrt is monotone and
       correctly rounded; the values are found on the host by stepping through neighbouring doubles) */
    double gt_Roa, gt_Rp, gt_Rg, lt_Rp, lt_Rg;
    /* calm regions of the energized pore (advance_particle): below calm_zA / above calm_zB no z comparison of the wall
       masks, the recapture or the out-of-bounds census can fire; inside calm_rA (squared) the open-air wall cannot,
       inside calm_rC no radial comparison at all */
    double calm_zA, calm_zB, calm_rA, calm_rC;
    int32_t calm_ok;
    uint32_t key0, key1;
    int64_t step;
    const double *cheb;
    int32_t cheb_n;
    double cheb_zmid, cheb_inv_half;
    const double *hist_edges;
    double hist_first, hist_last;
    unsigned long long *hist;       /* [4][AMC_NUM_BINS] */
    unsigned long long *path_count; /* cumulative */
    unsigned long long *path_sums;  /* [4][2] limbs */
    int64_t pair_cap;
    unsigned long long *pair_count;
    int64_t *pair_hi, *pair_lo;
    int32_t *pair_group, *pair_cell;
    int64_t path_cap;
    unsigned long long *tap_path_count;
    double *tap_paths[4];
    uint16_t *wall_bits;
    int32_t *wl;          /* [8][wl_stride][AMC_WI] work items: the cells of each colour group that can hold a pair */
    int32_t *wl_count;    /* [8] */
    int32_t *wl_next;     /* [8] ticket counters of the persistent pair kernel */
    int32_t *wl_hit;      /* [8][wl_stride][AMC_HIT_REC] per work item: the pairs k_detect found (as slots), see AMC_HIT_REC */
    int32_t *dl;          /* [cells][AMC_WI] work items of the detection pass: every reference cell with >= 2 candidates */
    int32_t *dl_count;    /* [1] */
    int32_t *cell_n;      /* [8][wl_stride] members counted by the detection pass for cells it did not flag (0 otherwise) */
    float det_thr;        /* fp32 squared distance below which the detection pass treats a pair as overlapping (conservative) */
    float det_w;          /* minimal bin width of the detection pass: 1.05 * sqrt(det_thr) */
    double *mv_spill;     /* [CTAs of the pair kernel][AMC_MAX_MEMBERS][3]: pre-visit positions of moved members beyond AMC_MV_CAP */
    int32_t det_own_is_member; /* lo[k] < edge[k] everywhere: a particle of owner cell k is a member of reference cell k */
    int32_t *cell_active; /* [8][wl_stride] 0: not on its group's worklist, 1: on it, e + 2: on it and escaped entry e heads its list (esc_link) */
    int32_t wl_stride;    /* reference cells per colour group */
    int32_t nh[3];        /* reference cells per axis and parity class: (nc+1)/2 */
    /* ---- slab decomposition along z (multi-GPU); slab == 0: single domain */
    int32_t slab, srank, nranks; /* srank: this handle's rank in the slab decomposition */
    int32_t zoff;             /* global z index of local cell layer 0 */
    const int32_t *cuts;      /* [nranks+1] global layer cuts */
    const double *gz_edge;    /* global z edges [gncz+1] */
    int32_t gncz;
    double g_e0z, g_inv_dz;
    double up_thr, down_thr;  /* lo_global[Z_{r+1}] (+inf on the last rank), edge_global[Z_r] (-inf on rank 0) */
    double down_band;         /* lo_global[Z_r]: above it a particle of the rank below is a band member of this rank's cells */
    double *xf_send;          /* per peer d: records [xf_off[d], xf_off[d] + xf_capv[d]], the first one = header (count) */
    const double *xf_recv;
    int32_t *xf_count;        /* [nranks] */
    int2 *xf_pack;            /* same block layout as the records: {slot, flag bits} of every particle k_keys found to travel; k_slab_pack makes the records */
    int32_t xf_cap;           /* largest per-peer capacity */
    int32_t xf_cap_nb, xf_cap_far; /* capacity of the blocks exchanged with rank +-1 / with every other rank */
    const int32_t *xf_off, *xf_capv; /* [nranks] record offset / capacity of each peer's block (same layout for send and recv) */
    int32_t *n_in;            /* particles unpacked from xf_recv in this step */
    int32_t *bnd_dirty[2];    /* [0] = up, [1] = down: slots moved in the current group that the neighbour must see */
    int32_t *bnd_n;           /* [2] */
    int32_t bnd_cap;
    double *bnd_send[2];
    const double *bnd_recv[2];
    int32_t *rel_id, *rel_slot, *rel_count; /* open-addressing hash: particles a neighbour may send updates for, id -> slot */
    int32_t rel_cap;          /* power of two; rel_id[] == -1: empty */
    uint8_t *aux;             /* per slot, k_keys -> k_scatter_advect: AUX_* bits of the slab protocol */
    int32_t *n_foreign;       /* foreign copies appended after the sort */
    int32_t foreign_cap;
    int32_t group_done;       /* last finished colour group (-1 before the first) */
    /* device-resident stepping (amc_slab_step): the particle count lives on the device, the exchange buffers of the
       other ranks are mapped peer-to-peer and every transfer is a kernel that writes the records straight into the
       receiver's buffer, then a sequence number into the receiver's flag word (release / acquire at system scope) */
    int32_t *n_dev;           /* [0] particles in the arrays (null: p.n is authoritative) */
    int64_t n_hint;           /* host-side upper bound of the count during this call: the grids are sized by it */
    int32_t parity;           /* buffer half used by this step's all-to-all */
    uint32_t xf_seq;          /* sequence number of this step's all-to-all */
    uint32_t bnd_seq;         /* sequence number of the hand-over round being packed / applied */
    uint32_t bnd_seq_apply;   /* fused hand-over (k_pairs_group): round whose records are applied at the head of the launch, 0 = none */
    uint32_t *applied;        /* [2] fused hand-over: bnd_seq of the launch whose head has finished applying direction d */
    int32_t *pg_done;         /* fused hand-over: CTAs of the current k_pairs_group launch that have finished */
    double *const *peer_xf;   /* [nranks] base of every rank's xfer_recv (both halves); [srank] = own */
    const int64_t *peer_xf_stride; /* [nranks] doubles per half of that rank's xfer_recv (end ranks have one big block, inner ranks two) */
    const int64_t *peer_xf_off;    /* [nranks] record offset of THIS rank's block inside that rank's xfer_recv */
    uint32_t *const *peer_flag; /* [nranks] base of every rank's flag words */
    double *peer_bnd[2];      /* [0] bnd_recv_down of the rank above, [1] bnd_recv_up of the rank below (both halves) */
    const uint32_t *flags;    /* own flag words: [0..nranks) all-to-all from rank r, [nranks] hand-over from above, [nranks+1] from below */
    int32_t bnd_stride;       /* doubles per half of a hand-over buffer */
    int32_t xf_stride;        /* doubles per half of xfer_recv */
    unsigned long long *slab_overflow;
    int32_t *touched;         /* slots the closing recapture of this step has to look at (touch_slot) */
    int32_t *touched_n;       /* lives behind the last band counter: cleared with them at the start of a step */
    int32_t *touch_mark;      /* [cap] step tag of the last listing of each slot */
    int32_t touched_cap;
    int32_t esc_cap;
    int32_t *esc_count;
    int32_t *esc_slot;
    int32_t *esc_cell; /* [esc_cap][8] member cell per colour group, -1 = none */
    int32_t *esc_next; /* [esc_cap][8] next entry (+ 2) on the list of that cell, < 2 = end */
    StatsDev *stats;
    StatsDev *stats_prev; /* counters of the previous step (recapture fused into the next step's k_advect) */
    /* ---- event-driven serial sweep of the cube stage (k_sweep_detect / k_sweep_events); null: the plain serial sweep */
    int32_t *sw_col;      /* [columns][sw_colcap] particles inside the x and y masks of each (x layer, y layer) column before the sweep */
    int32_t *sw_col_n;    /* [columns] */
    int32_t sw_colcap;
    int32_t sw_pass;      /* tag of the current pass (sw_tag) */
    int32_t *sw_tag;      /* [cap] == sw_pass: a collision of this pass has moved the particle */
    int32_t *sw_ml;       /* [cap] the moved particles of this pass */
    double *sw_xs, *sw_ys; /* [cap] moved particles: the x the current layer's mask saw, the y the current column's mask saw */
    unsigned long long *sw_state; /* [0] != 0: a column list overflowed, the plain sweep takes over; [1] pair tests of pass 1 */
};

// surface recording (amc_surface_*): a kernel parameter of its own, passed only to the recording kernels
// (k_advect_surf, k_scatter_advect_surf, the host-RNG case kernels), so that P and every other kernel stay as they are
struct SurfP {
    unsigned long long *acc; /* [elements][AMC_SURF_WORDS], then outside[AMC_NUM_CASES]; null: not recording */
    int32_t off[AMC_NUM_CASES + 1]; /* first element of every case (case-major numbering) */
    const double *rsq;       /* annulus bounds (k * dr) * (k * dr), k = 0 .. nann */
    int32_t nann;
    double inv_dr;
    const double *zedge;     /* z edges of the layout (a slab handle: the global ones) */
    int32_t ncz;
    double ze0, zinv;
};

// ---------------------------------------------------------------- deterministic accumulation
// Sums that feed printed outputs (momentum / energy per step, free-path means) are accumulated as
// two 64-bit integer limbs at fixed binary scales: integer adds are associative, so the result does
// not depend on thread order, and the low limb keeps ~40 bits below the high limb's resolution.
#define SC_P1 0x1p116
#define SC_P1I 0x1p-116
#define SC_P2 0x1p156
#define SC_E1 0x1p108
#define SC_E1I 0x1p-108
#define SC_E2 0x1p148
#define SC_L1 0x1p49
#define SC_L1I 0x1p-49
#define SC_L2 0x1p89

__device__ __forceinline__ void acc_add(unsigned long long *acc, double v, double s1, double s1inv, double s2)
{
    long long i1 = __double2ll_rn(v * s1);
    double rem = v - (double)i1 * s1inv;
    long long i2 = __double2ll_rn(rem * s2);
    atomicAdd(&acc[0], (unsigned long long)i1);
    atomicAdd(&acc[1], (unsigned long long)i2);
}

// surface recording (defined below, after the owner-cell helpers it uses)
__device__ __noinline__ void surf_record(const P &p, const SurfP &sp, const int c, const double cx, const double cy, const double cz,
                                         const double dvx, const double dvy, const double dvz, const double dE);
__device__ __noinline__ void surf_outside(const SurfP &sp, const int c);

// ---------------------------------------------------------------- completed free paths
// One completed path = one append to each of the reference's four lists (Pore:187-190).  The
// histogram index follows np.histogram's uniform-bin rule with its two edge corrections
// (numpy/lib/_histograms_impl.py:851-863) as reached through Axes.hist at Pore:575.
__device__ __forceinline__ void hist_add(const P &p, int which, double x)
{
    if (!(x >= p.hist_first && x <= p.hist_last)) return;
    double f = ((x - p.hist_first) / (p.hist_last - p.hist_first)) * (double)AMC_NUM_BINS;
    long long idx = (long long)f;
    if (idx == AMC_NUM_BINS) idx--;
    if (x < p.hist_edges[idx]) idx--;
    else if (x >= p.hist_edges[idx + 1] && idx != AMC_NUM_BINS - 1) idx++;
    atomicAdd(&p.hist[which * AMC_NUM_BINS + idx], 1ull);
}

__device__ __noinline__ void emit_path(const P &p, double t, double cx, double cy, double cz)
{
    hist_add(p, 0, t); hist_add(p, 1, cx); hist_add(p, 2, cy); hist_add(p, 3, cz);
    atomicAdd(p.path_count, 1ull);
    atomicAdd(&p.stats->paths, 1ull);
    acc_add(p.path_sums + 0, t, SC_L1, SC_L1I, SC_L2);
    acc_add(p.path_sums + 2, cx, SC_L1, SC_L1I, SC_L2);
    acc_add(p.path_sums + 4, cy, SC_L1, SC_L1I, SC_L2);
    acc_add(p.path_sums + 6, cz, SC_L1, SC_L1I, SC_L2);
    if (p.tap_path_count) {
        unsigned long long k = atomicAdd(p.tap_path_count, 1ull);
        if ((int64_t)k < p.path_cap) { p.tap_paths[0][k] = t; p.tap_paths[1][k] = cx; p.tap_paths[2][k] = cy; p.tap_paths[3][k] = cz; }
    }
}

// ---------------------------------------------------------------- one particle in registers
struct Part {
    double x, y, z, vx, vy, vz, d, dx, dy, dz;
    double px, py, pz;
    uint32_t flag;
};

// MFP bookkeeping shared by walls and pair collisions (Pore:274-284, 324-335, 186-199): a particle
// that already finished a first collision completes a path of |path - |speed*t||, else it is flagged.
template <int MODE = 1>
__device__ __forceinline__ void mfp_record(const P &p, double d, double dx, double dy, double dz, uint32_t &flag,
                                           double vx, double vy, double vz, double t)
{
    if (MODE == AMC_DRY) return;                             /* only the final position matters */
    if (MODE == AMC_QUIET) { flag |= AMC_FLAG_PATH; return; } /* state as in the live run, nothing recorded */
    if (flag & AMC_FLAG_PATH) {
        double sp = sqrt((vx * vx + vy * vy) + vz * vz);
        emit_path(p, fabs(d - fabs(sp * t)), fabs(dx - fabs(vx * t)), fabs(dy - fabs(vy * t)), fabs(dz - fabs(vz * t)));
    } else {
        flag |= AMC_FLAG_PATH;
    }
}

// rewind time onto a coaxial cylinder of radius Rc (Pore:312-315).  false: the reference's
// try/except path (invalid sqrt or division by zero under np.seterr(all='raise')).
__device__ __forceinline__ bool side_quadratic(double x, double y, double vx, double vy, double Rc, double &t)
{
    double a = (-vx) * (-vx) + (-vy) * (-vy);
    double b = 2 * (x * (-vx) + y * (-vy));
    double c = (x * x + y * y) - Rc * Rc;
    double disc = b * b - (4 * a) * c;
    if (!(disc >= 0.0) || a == 0.0) return false;
    double r = sqrt(disc);
    double t1 = (-b + r) / (2 * a), t2 = (-b - r) / (2 * a);
    t = t1 < t2 ? t1 : t2;
    return true;
}

// specular reflection in the xy plane about the contact normal (Pore:316-323)
__device__ __forceinline__ void reflect_xy(Part &q, double Rc, double t)
{
    double col_x = q.x - q.vx * t, col_y = q.y - q.vy * t;
    double nx = col_x / Rc, ny = col_y / Rc;
    double scalar = q.vx * nx + q.vy * ny;
    double nvx = q.vx - (2 * scalar) * nx, nvy = q.vy - (2 * scalar) * ny;
    q.x = col_x + nvx * t; q.y = col_y + nvy * t; q.vx = nvx; q.vy = nvy;
}

// hit_cylinder_side_wall, Pore:294-348.  SURF: record the hit as wall case c (surf_record)
template <int MODE = 1, bool SURF = false>
__device__ __forceinline__ void pore_side_wall(const P &p, Part &q, double Rc, int c = 0, const SurfP *sp = nullptr)
{
    double t;
    if (!side_quadratic(q.x, q.y, q.vx, q.vy, Rc, t)) {
        if (MODE == AMC_LIVE) atomicAdd(&p.stats->errors, 1ull);
        if (SURF && MODE == AMC_LIVE) surf_outside(*sp, c);
        return;
    }
    double vx = q.vx, vy = q.vy, vz = q.vz;
    mfp_record<MODE>(p, q.d, q.dx, q.dy, q.dz, q.flag, vx, vy, vz, t);
    const double cx = q.x - vx * t, cy = q.y - vy * t, cz = q.z - vz * t; /* contact point (the col_x, col_y of reflect_xy) */
    reflect_xy(q, Rc, t);
    if (SURF && MODE == AMC_LIVE) surf_record(p, *sp, c, cx, cy, cz, q.vx - vx, q.vy - vy, 0.0, 0.0);
    q.d = fabs(sqrt((q.vx * q.vx + q.vy * q.vy) + vz * vz) * t);
    q.dx = fabs(q.vx * t); q.dy = fabs(q.vy * t); q.dz = fabs(vz * t);
}

// hit_vertical_wall, Pore:257-292
template <int MODE = 1, bool SURF = false>
__device__ __forceinline__ void pore_plane_wall(const P &p, Part &q, double zp, int c = 0, const SurfP *sp = nullptr)
{
    double t = (q.z - zp) / q.vz;
    if (SURF && MODE == AMC_LIVE) surf_record(p, *sp, c, q.x - q.vx * t, q.y - q.vy * t, zp, 0.0, 0.0, -q.vz - q.vz, 0.0);
    mfp_record<MODE>(p, q.d, q.dx, q.dy, q.dz, q.flag, q.vx, q.vy, q.vz, t);
    q.d = fabs(sqrt((q.vx * q.vx + q.vy * q.vy) + q.vz * q.vz) * t);
    q.dx = fabs(q.vx * t); q.dy = fabs(q.vy * t); q.dz = fabs(q.vz * t);
    q.vz = -q.vz;
    q.z = zp + t * q.vz;
}

// Pore wall cases 1..6 against the progressively mutated particle (Pore:442-485); returns hit bits.
// `np.sqrt(x**2 + y**2) > R` is evaluated as `x*x + y*y > gt_R` (exactly equivalent, see P).
template <int MODE = 1, bool SURF = false>
__device__ __forceinline__ uint32_t pore_walls(const P &p, Part &q, const SurfP *sp = nullptr)
{
    const amc_geom &g = p.g;
    uint32_t bits = 0;
    if (q.x * q.x + q.y * q.y > p.gt_Roa) { bits |= 1u << 0; pore_side_wall<MODE, SURF>(p, q, g.R_oa_c, 0, sp); }
    if (q.z < 0) { bits |= 1u << 1; pore_plane_wall<MODE, SURF>(p, q, 0.0, 1, sp); }
    if (q.z > g.H) { bits |= 1u << 2; pore_plane_wall<MODE, SURF>(p, q, g.H, 2, sp); }
    if (q.pz > g.z_cold && q.z < g.z_cold && q.x * q.x + q.y * q.y > p.gt_Rp) { bits |= 1u << 3; pore_plane_wall<MODE, SURF>(p, q, g.z_cold, 3, sp); }
    if (q.pz < g.oah && q.z > g.oah && q.x * q.x + q.y * q.y > p.gt_Rp) { bits |= 1u << 4; pore_plane_wall<MODE, SURF>(p, q, g.oah, 4, sp); }
    double pr2 = q.px * q.px + q.py * q.py;
    bool pz_in_gap = q.pz < g.z_gt_pore && q.pz > g.z_gb;
    if (pz_in_gap && pr2 < p.lt_Rg && q.x * q.x + q.y * q.y > p.gt_Rg) { bits |= 1u << 5; pore_side_wall<MODE, SURF>(p, q, g.R_g_c, 5, sp); }
    if (pr2 > p.gt_Rp && q.z < g.z_gb && pz_in_gap) { bits |= 1u << 6; pore_plane_wall<MODE, SURF>(p, q, g.z_gb, 6, sp); }
    if (pr2 > p.gt_Rp && q.z > g.z_gt_pore && pz_in_gap) { bits |= 1u << 7; pore_plane_wall<MODE, SURF>(p, q, g.z_gt_pore, 7, sp); }
    if (pr2 < p.lt_Rp && q.x * q.x + q.y * q.y > p.gt_Rp &&
        ((q.z < g.z_cold && q.z > g.z_gt_pore) || (q.z < g.z_gb && q.z > g.oah))) { bits |= 1u << 8; pore_side_wall<MODE, SURF>(p, q, g.R_p_c, 8, sp); }
    return bits;
}

// Pore num_out_of_bounds(): count and teleport (Pore:354-375)
__device__ __forceinline__ int pore_recapture(const amc_geom &g, Part &q)
{
    int cnt = 0;
    if (q.z < 0) { q.z += g.ten_a; cnt++; }
    if (q.z > g.H) { q.z -= g.ten_a; cnt++; }
    if (q.x * q.x + q.y * q.y > g.R_oa_sq) { q.x = 0; q.y = 0; cnt++; }
    if (q.x * q.x + q.y * q.y > g.R_g_sq && q.z > g.oah && q.z < g.z_cold) { q.x = 0; q.y = 0; cnt++; }
    if (q.x * q.x + q.y * q.y > g.R_p_sq && ((q.z > g.oah && q.z < g.z_gb) || (q.z > g.z_gt && q.z < g.z_cold))) { q.x = 0; q.y = 0; cnt++; }
    return cnt;
}

// ---------------------------------------------------------------- Temp walls
__device__ __forceinline__ bool temp_mask(const P &p, int c, const Part &q)
{
    const amc_geom &g = p.g;
    double r2 = q.x * q.x + q.y * q.y, pr2 = q.px * q.px + q.py * q.py;
    switch (c) {
    case AMC_CASE_1: return r2 > p.gt_Roa;   /* np.sqrt(x**2 + y**2) > open_air_radius */                /* Temp:693 */
    case AMC_CASE_2A: return q.z < 0;                                                                 /* Temp:699 */
    case AMC_CASE_2B: return q.z > g.H;                                                               /* Temp:702 */
    case AMC_CASE_3C: return q.pz >= g.zc3 && q.z < g.zc3 && r2 > g.R_p_sq;                           /* Temp:708 */
    case AMC_CASE_3H: return q.pz <= g.zh3 && q.z > g.zh3 && r2 > g.R_p_sq;                           /* Temp:713 */
    case AMC_CASE_4: return q.pz < g.zgt_m && q.pz > g.zgb_p && pr2 <= g.R_g_c_sq && r2 > g.R_g_c_sq; /* Temp:720 */
    case AMC_CASE_5B: return pr2 >= g.R_p_c_sq && q.z < g.zgb_p && q.pz <= g.zgt_m && q.pz >= g.zgb_p; /* Temp:728 */
    case AMC_CASE_5T: return pr2 >= g.R_p_c_sq && q.z > g.zgt_m && q.pz <= g.zgt_m && q.pz >= g.zgb_p; /* Temp:734 */
    case AMC_CASE_6H: return pr2 <= g.R_p_c_sq && r2 > g.R_p_c_sq && q.z <= g.zgb_p && q.z >= g.zh3;  /* Temp:743 */
    case AMC_CASE_6C: return pr2 <= g.R_p_c_sq && r2 > g.R_p_c_sq && q.z < g.zc3 && q.z > g.zgt_m;    /* Temp:749 */
    }
    return false;
}
__device__ __forceinline__ bool temp_is_side(int c) { return c == AMC_CASE_1 || c == AMC_CASE_4 || c == AMC_CASE_6H || c == AMC_CASE_6C; }
__device__ __forceinline__ bool temp_is_cold(int c) { return c == AMC_CASE_3C || c == AMC_CASE_5T || c == AMC_CASE_6C; }
__device__ __forceinline__ double temp_plane(const amc_geom &g, int c)
{
    switch (c) {
    case AMC_CASE_2B: return g.H;
    case AMC_CASE_3C: return g.zc3;
    case AMC_CASE_3H: return g.zh3;
    case AMC_CASE_5B: return g.zgb_p;
    case AMC_CASE_5T: return g.zgt_m;
    }
    return 0.0;
}
__device__ __forceinline__ double temp_radius(const amc_geom &g, int c)
{
    return c == AMC_CASE_1 ? g.R_oa_c : (c == AMC_CASE_4 ? g.R_g_c : g.R_p_c);
}

// contact geometry of an energized hit: rewind time, contact point and the vector the reference
// passes to random_inbounds_direction (Temp:372-375, 440-444).  false = floating-point error path.
__device__ __forceinline__ bool temp_contact(const amc_geom &g, int c, const Part &q, double &t, double col[3], double nrm[3])
{
    if (temp_is_side(c)) {
        double Rc = temp_radius(g, c);
        if (!side_quadratic(q.x, q.y, q.vx, q.vy, Rc, t)) return false;
        col[0] = q.x - q.vx * t; col[1] = q.y - q.vy * t; col[2] = q.z - q.vz * t;
        nrm[0] = -(col[0] / Rc); nrm[1] = -(col[1] / Rc); nrm[2] = -(0.0 / Rc);
    } else {
        double zp = temp_plane(g, c);
        t = (q.z - zp) / q.vz;
        col[0] = q.x - q.vx * t; col[1] = q.y - q.vy * t; col[2] = zp;
        nrm[0] = 0.0; nrm[1] = 0.0; nrm[2] = (c == AMC_CASE_3C || c == AMC_CASE_5B) ? 1.0 : -1.0;
    }
    return true;
}

// energy accommodation at an energized wall (Temp:377-389, 402-403); leaves the particle at the
// contact point with paths reset (Temp:398-401)
template <int MODE = 1>
__device__ __forceinline__ void temp_energized(const P &p, Part &q, double t, const double col[3], const double dir[3],
                                               double Es, double alpha, double &dpz, double &dE)
{
    double m = p.g.argon_mass;
    double v_mag = sqrt((q.vx * q.vx + q.vy * q.vy) + q.vz * q.vz);
    double old_pz = m * q.vz;
    double E = (0.5 * m) * (v_mag * v_mag);
    double ediff = Es - E;
    double Enew = E + ediff * alpha;
    double new_mag = sqrt((Enew * 2) / m);
    dE = Enew - E;
    double nvx = dir[0] * new_mag, nvy = dir[1] * new_mag, nvz = dir[2] * new_mag;
    dpz = m * nvz - old_pz;
    mfp_record<MODE>(p, q.d, q.dx, q.dy, q.dz, q.flag, q.vx, q.vy, q.vz, t);
    q.d = 0; q.dx = 0; q.dy = 0; q.dz = 0;
    q.x = col[0]; q.y = col[1]; q.z = col[2];
    q.vx = nvx; q.vy = nvy; q.vz = nvz;
}

// specular Temp cases: no MFP bookkeeping (Temp:311-347)
template <int MODE = 1, bool SURF = false>
__device__ __forceinline__ void temp_specular(const P &p, int c, Part &q, const SurfP *sp = nullptr)
{
    if (c == AMC_CASE_1) {
        double t;
        if (!side_quadratic(q.x, q.y, q.vx, q.vy, p.g.R_oa_c, t)) {
            if (MODE == AMC_LIVE) atomicAdd(&p.stats->errors, 1ull);
            if (SURF && MODE == AMC_LIVE) surf_outside(*sp, c);
            return;
        }
        const double vx = q.vx, vy = q.vy, cx = q.x - vx * t, cy = q.y - vy * t, cz = q.z - q.vz * t;
        reflect_xy(q, p.g.R_oa_c, t);
        if (SURF && MODE == AMC_LIVE) surf_record(p, *sp, c, cx, cy, cz, q.vx - vx, q.vy - vy, 0.0, 0.0);
    } else {
        double zp = temp_plane(p.g, c);
        double t = (q.z - zp) / q.vz;
        if (SURF && MODE == AMC_LIVE) surf_record(p, *sp, c, q.x - q.vx * t, q.y - q.vy * t, zp, 0.0, 0.0, -q.vz - q.vz, 0.0);
        q.vz = -q.vz;
        q.z = zp + t * q.vz;
    }
}

// recapture_out_of_bounds, Temp:594-616
__device__ __forceinline__ int temp_recapture(const amc_geom &g, Part &q)
{
    int cnt = 0;
    if (q.z < 0) { q.z = g.recap_lo; cnt++; }
    if (q.z > g.H) { q.z = g.recap_hi; cnt++; }
    if (q.x * q.x + q.y * q.y > g.R_oa_sq) { q.x = 0; q.y = 0; cnt++; }
    if (q.x * q.x + q.y * q.y > g.R_g_sq && q.z > g.oah && q.z < g.z_cold) { q.x = 0; q.y = 0; cnt++; }
    if (q.x * q.x + q.y * q.y > g.R_p_sq && ((q.z > g.oah && q.z < g.z_gb) || (q.z > g.z_gt && q.z < g.z_cold))) { q.x = 0; q.y = 0; cnt++; }
    return cnt;
}
// num_out_of_bounds (report), Temp:560-592
__device__ __forceinline__ int temp_oob(const amc_geom &g, const Part &q)
{
    double r2 = q.x * q.x + q.y * q.y, z = q.z;
    int cnt = 0;
    cnt += z < 0;
    cnt += z > g.H;
    cnt += r2 > g.R_oa_sq && z >= 0 && z <= g.oah;
    cnt += r2 > g.R_oa_sq && z >= g.z_cold && z <= g.H;
    cnt += r2 > g.R_g_sq && z >= g.z_gb && z <= g.z_gt;
    cnt += r2 > g.R_p_sq && z > g.oah && z < g.z_gb;
    cnt += r2 > g.R_p_sq && z > g.z_gt && z < g.z_cold;
    return cnt;
}

// ---------------------------------------------------------------- device RNG (throughput mode)
// Philox4x32-10, counter = (particle id, case, step, attempt); isotropic direction by Marsaglia's
// disc method (+ - * sqrt only, bit-reproducible against the CPU oracle); then the reference's
// acceptance rule about the inward normal (Temp:136-139).
__device__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1)
{
#pragma unroll
    for (int r = 0; r < 10; r++) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
        c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}
__device__ __forceinline__ double u53(uint32_t hi, uint32_t lo)
{
    return ((double)(hi >> 5) * 67108864.0 + (double)(lo >> 6)) * (1.0 / 9007199254740992.0);
}
__device__ __noinline__ void philox_direction(const P &p, int64_t id, int c, const double nrm[3], double dir[3])
{
    for (uint32_t attempt = 0;; attempt++) {
        uint32_t r[4] = {(uint32_t)id, (uint32_t)((uint64_t)id >> 32) ^ ((uint32_t)c << 24), (uint32_t)p.step, attempt};
        philox4x32_10(r, p.key0, p.key1);
        double u = 2.0 * u53(r[0], r[1]) - 1.0, v = 2.0 * u53(r[2], r[3]) - 1.0;
        double ss = u * u + v * v;
        if (!(ss < 1.0) || ss == 0.0) continue;
        double root = sqrt(1.0 - ss);
        double d0 = (2.0 * u) * root, d1 = (2.0 * v) * root, d2 = 1.0 - 2.0 * ss;
        double dn = (d0 * nrm[0] + d1 * nrm[1]) + d2 * nrm[2];
        if (fabs(dn) < p.g.cos85) continue;
        if (dn < p.g.cos85) { d0 = -d0; d1 = -d1; d2 = -d2; }
        dir[0] = d0; dir[1] = d1; dir[2] = d2;
        return;
    }
}
// Chebyshev/Clenshaw evaluation of surface_energy_gap(z) (Temp:143-152), coefficients fitted on the
// host with mpmath
__device__ __forceinline__ double cheb_eval(const P &p, double z)
{
    double u = (z - p.cheb_zmid) * p.cheb_inv_half, u2 = 2.0 * u, b1 = 0.0, b2 = 0.0;
    for (int k = p.cheb_n - 1; k >= 1; k--) {
        double b0 = (p.cheb[k] + u2 * b1) - b2;
        b2 = b1; b1 = b0;
    }
    return (p.cheb[0] + u * b1) - b2;
}

// true when at least one of the ten wall masks holds for the (unmutated) particle.  The cases only
// change a particle they hit, so when this is false the sequential case loop is a no-op: 99.9 % of the
// particles skip it.
__device__ __forceinline__ bool temp_any_mask(const P &p, const Part &q)
{
    const amc_geom &g = p.g;
    double r2 = q.x * q.x + q.y * q.y, pr2 = q.px * q.px + q.py * q.py, z = q.z, pz = q.pz;
    bool pz_gap_open = pz < g.zgt_m && pz > g.zgb_p, pz_gap_closed = pz <= g.zgt_m && pz >= g.zgb_p;
    bool crossed_p = pr2 <= g.R_p_c_sq && r2 > g.R_p_c_sq;
    return r2 > p.gt_Roa || z < 0 || z > g.H ||
           (pz >= g.zc3 && z < g.zc3 && r2 > g.R_p_sq) || (pz <= g.zh3 && z > g.zh3 && r2 > g.R_p_sq) ||
           (pz_gap_open && pr2 <= g.R_g_c_sq && r2 > g.R_g_c_sq) ||
           (pr2 >= g.R_p_c_sq && pz_gap_closed && (z < g.zgb_p || z > g.zgt_m)) ||
           (crossed_p && ((z <= g.zgb_p && z >= g.zh3) || (z < g.zc3 && z > g.zgt_m)));
}

// all ten Temp cases on one particle with device RNG (Temp:693-753)
template <int MODE = 1, bool SURF = false>
__device__ __forceinline__ uint32_t temp_walls_device(const P &p, Part &q, int64_t id, const SurfP *sp = nullptr)
{
    uint32_t bits = 0;
    if (!temp_any_mask(p, q)) return 0;
#pragma unroll 1
    for (int c = 0; c < AMC_NUM_CASES; c++) {
        if (!temp_mask(p, c, q)) continue;
        bits |= 1u << c;
        if (c <= AMC_CASE_2B) { temp_specular<MODE, SURF>(p, c, q, sp); continue; }
        double t, col[3], nrm[3], dir[3], dpz, dE;
        if (!temp_contact(p.g, c, q, t, col, nrm)) {
            if (MODE == AMC_LIVE) atomicAdd(&p.stats->errors, 1ull);
            if (SURF && MODE == AMC_LIVE) surf_outside(*sp, c);
            continue;
        }
        philox_direction(p, id, c, nrm, dir);
        double Es = c == AMC_CASE_4 ? cheb_eval(p, col[2]) : (temp_is_cold(c) ? p.g.E_cold : p.g.E_hot);
        double alpha = c == AMC_CASE_4 ? p.g.alpha_g : p.g.alpha_c;
        const double vx = q.vx, vy = q.vy, vz = q.vz;
        temp_energized<MODE>(p, q, t, col, dir, Es, alpha, dpz, dE);
        if (MODE != AMC_LIVE) continue;
        if (SURF) surf_record(p, *sp, c, col[0], col[1], col[2], q.vx - vx, q.vy - vy, q.vz - vz, dE);
        acc_add(p.stats->dpz, dpz, SC_P1, SC_P1I, SC_P2);
        if (c != AMC_CASE_4) acc_add(temp_is_cold(c) ? p.stats->ecold : p.stats->ehot, dE, SC_E1, SC_E1I, SC_E2);
    }
    return bits;
}

// contact point of a cube face hit (face of case c on axis c / 2 at coordinate L): (x, y, z) - v * t with the face's own
// coordinate set to L
__device__ __forceinline__ void cube_record(const P &p, const SurfP &sp, const int c, const Part &q, const double t, const double L, const double dva)
{
    const int a = c >> 1;
    const double cx = a == 0 ? L : q.x - q.vx * t, cy = a == 1 ? L : q.y - q.vy * t, cz = a == 2 ? L : q.z - q.vz * t;
    surf_record(p, sp, c, cx, cy, cz, a == 0 ? dva : 0.0, a == 1 ? dva : 0.0, a == 2 ? dva : 0.0, 0.0);
}

// Cube: six specular planes, x then y then z, max wall before min wall (Cube:192-226).  SURF (live runs only): record
// every hit at the contact point the same rewind gives, taken on the particle as it stands when its axis is handled
template <int MODE = 1, bool SURF = false>
__device__ __forceinline__ uint32_t cube_walls(const P &p, Part &q, const SurfP *sp = nullptr)
{
    uint32_t bits = 0;
    double *pos[3] = {&q.x, &q.y, &q.z}, *vel[3] = {&q.vx, &q.vy, &q.vz};
#pragma unroll
    for (int a = 0; a < 3; a++) {
        double L = p.cube[a];
        if (*pos[a] > L) {
            double t = (*pos[a] - L) / *vel[a];
            if (SURF && MODE == AMC_LIVE) cube_record(p, *sp, 2 * a, q, t, L, -*vel[a] - *vel[a]);
            *vel[a] = -*vel[a]; *pos[a] = L + t * *vel[a]; bits |= 1u << (2 * a);
        }
        if (*pos[a] < 0) {
            double t = *pos[a] / *vel[a];
            if (SURF && MODE == AMC_LIVE) cube_record(p, *sp, 2 * a + 1, q, t, 0.0, -*vel[a] - *vel[a]);
            *vel[a] = -*vel[a]; *pos[a] = t * *vel[a]; bits |= 1u << (2 * a + 1);
        }
    }
    return bits;
}

// ---------------------------------------------------------------- owner cell of a coordinate
// Owner k: edge[k] <= v < edge[k+1].  Returns -1 below edge[0] (only the low band of cell 0 can
// contain it) and nc for v >= edge[nc] or NaN (member of no cell).  The division is only an
// estimate; the table comparisons decide.
__device__ __noinline__ int owner_axis_slow(const double *edge, int nc, double e0, double inv_d, double v)
{
    if (!(v < edge[nc])) return nc;
    if (v < edge[0]) return -1;
    double f = (v - e0) * inv_d;
    int o = f >= (double)(nc - 1) ? nc - 1 : (int)f;
    if (o < 0) o = 0;
    while (v < edge[o]) --o;
    while (v >= edge[o + 1]) ++o;
    return o;
}
// the estimate is right for all but the particles within a rounding error of an edge: one pair of table
// entries decides; everything else (outside the grid, NaN, off by one) takes the slow path
__device__ __forceinline__ int owner_axis(const double *edge, int nc, double e0, double inv_d, double v)
{
    int o = __double2int_rd((v - e0) * inv_d);
    o = min(max(o, 0), nc - 1);
    if (edge[o] <= v && v < edge[o + 1]) return o;
    return owner_axis_slow(edge, nc, e0, inv_d, v);
}
// padded owner key: each axis shifted by +1 so the virtual layer below edge[0] is index 0;
// anything outside on the high side (or NaN) goes to the trailing OUT bucket ncell_pad
__device__ __forceinline__ int32_t owner_key(const P &p, double x, double y, double z, int o[3])
{
    o[0] = owner_axis(p.edge[0], p.nc[0], p.e0[0], p.inv_d[0], x);
    o[1] = owner_axis(p.edge[1], p.nc[1], p.e0[1], p.inv_d[1], y);
    o[2] = owner_axis(p.edge[2], p.nc[2], p.e0[2], p.inv_d[2], z);
    if (o[0] == p.nc[0] || o[1] == p.nc[1] || o[2] == p.nc[2]) return p.ncell_pad;
    return ((o[0] + 1) * p.pnc[1] + (o[1] + 1)) * p.pnc[2] + (o[2] + 1);
}
// ---------------------------------------------------------------- surface recording (amc_surface_*)
// One wall interaction of case c: contact point (cx, cy, cz), velocity change dv = v_out - v_in of the particle, energy
// dE the gas gained.  The binning, the wall-local components and the limbs are defined in include/amc.h (a NumPy
// restatement mirrors every expression).  Out of line: the recording instantiations carry one call per wall helper, the
// streaming kernels none.
// bin k of v with tab[k] <= v < tab[k+1], 0 <= k < n, or -1 (NaN included); est: estimate of k.  Self-contained rather
// than owner_axis: a call from here with a pointer of the SurfP parameter would turn the global loads of the shared
// owner_axis_slow into generic ones in every kernel of the library.
__device__ __forceinline__ int surf_bin(const double *tab, const int n, const double est, const double v)
{
    if (!(v >= tab[0] && v < tab[n])) return -1;
    int k = min(max(__double2int_rd(est), 0), n - 1);
    while (v < tab[k]) --k;
    while (v >= tab[k + 1]) ++k;
    return k;
}
// bin of coordinate v on axis a of the layout's grid (z: the global edges on a slab handle)
__device__ __forceinline__ int surf_axis_bin(const P &p, const SurfP &sp, const int a, const double v)
{
    return a == 2 ? surf_bin(sp.zedge, sp.ncz, (v - sp.ze0) * sp.zinv, v) : surf_bin(p.edge[a], p.nc[a], (v - p.e0[a]) * p.inv_d[a], v);
}
__device__ __forceinline__ bool surf_is_side(const int kind, const int c)
{
    return kind != AMC_KIND_CUBE && (c == AMC_CASE_1 || c == AMC_CASE_4 || c == AMC_CASE_6H || c == AMC_CASE_6C);
}
__device__ __noinline__ void surf_record(const P &p, const SurfP &sp, const int c, const double cx, const double cy, const double cz,
                                         const double dvx, const double dvy, const double dvz, const double dE)
{
    static_assert(AMC_SURF_WORDS == 9 && AMC_SURF_V1 == 16 && AMC_SURF_V2 == 46 && AMC_SURF_E1 == 90 && AMC_SURF_E2 == 120,
                  "scales of surf_record");
    int e = -1; /* element inside the case, -1: outside every bin */
    double dn, d1, d2;
    if (p.kind == AMC_KIND_CUBE) {
        const int a = c >> 1, b1 = a == 0 ? 1 : 0, b2 = a == 2 ? 1 : 2;
        const double col[3] = {cx, cy, cz}, dv[3] = {dvx, dvy, dvz};
        dn = (c & 1) ? dv[a] : -dv[a]; /* even case: the face at cube[a], normal -e_a; odd: the face at 0, normal +e_a */
        d1 = dv[b1]; d2 = dv[b2];
        const int o1 = surf_axis_bin(p, sp, b1, col[b1]), o2 = surf_axis_bin(p, sp, b2, col[b2]);
        if (o1 >= 0 && o2 >= 0) e = o1 * (b2 == 2 ? sp.ncz : p.nc[b2]) + o2;
    } else if (surf_is_side(p.kind, c)) {
        const double Rc = c == AMC_CASE_1 ? p.g.R_oa_c : (c == AMC_CASE_4 ? p.g.R_g_c : p.g.R_p_c);
        const double ex = cx / Rc, ey = cy / Rc;
        dn = -(dvx * ex + dvy * ey); d1 = dvz; d2 = dvy * ex - dvx * ey;
        e = surf_axis_bin(p, sp, 2, cz);
    } else {
        const double r2 = cx * cx + cy * cy, r = sqrt(r2);
        const double ex = r > 0.0 ? cx / r : 1.0, ey = r > 0.0 ? cy / r : 0.0;
        dn = (c == AMC_CASE_2A || c == AMC_CASE_3C || c == AMC_CASE_5B) ? dvz : -dvz;
        d1 = dvx * ex + dvy * ey; d2 = dvy * ex - dvx * ey;
        e = surf_bin(sp.rsq, sp.nann, r * sp.inv_dr, r2);
    }
    if (e < 0) { surf_outside(sp, c); return; }
    unsigned long long *w = sp.acc + (int64_t)(sp.off[c] + e) * AMC_SURF_WORDS;
    atomicAdd(w, 1ull);
    acc_add(w + 1, dn, 0x1p16, 0x1p-16, 0x1p46);
    acc_add(w + 3, d1, 0x1p16, 0x1p-16, 0x1p46);
    acc_add(w + 5, d2, 0x1p16, 0x1p-16, 0x1p46);
    acc_add(w + 7, dE, 0x1p90, 0x1p-90, 0x1p120);
}
// a hit the case counts but applies nothing to (the reference's floating-point error path)
__device__ __noinline__ void surf_outside(const SurfP &sp, const int c)
{
    atomicAdd(sp.acc + (int64_t)sp.off[AMC_NUM_CASES] * AMC_SURF_WORDS + c, 1ull);
}

// true when the coordinate lies inside the low-side band of the next cell up on this axis, i.e. the
// particle can be a member of a reference cell other than its owner cell (Pore:527-529)
__device__ __forceinline__ bool in_next_band(const double *lo, int nc, int owner, double v)
{
    return owner + 1 < nc && v > lo[owner + 1];
}
__device__ __forceinline__ bool any_band(const P &p, double x, double y, double z, const int o[3])
{
    return in_next_band(p.lo[0], p.nc[0], o[0], x) || in_next_band(p.lo[1], p.nc[1], o[1], y) || in_next_band(p.lo[2], p.nc[2], o[2], z);
}
// member cell (0-based) of coordinate v on one axis for parity `par`, or -1 (strict inequalities
// lo[k] < v < edge[k+1], Pore:527-529)
__device__ __forceinline__ int member_axis(const double *edge, const double *lo, int nc, int owner, int par, double v)
{
    if (owner >= nc) return -1;
    int k = owner < 0 ? 0 : owner;
    for (int kk = k; kk <= k + 1 && kk < nc; kk++)
        if ((kk & 1) == par && lo[kk] < v && v < edge[kk + 1]) return kk;
    return -1;
}

// One work item of the pair pass = everything a CTA needs to start on a reference cell, in one 128-byte
// record: cell id, cell indices, the 8 candidate ranges (owner cell: all of it; 7 low-side neighbours:
// their band prefix) and the cell's membership bounds (Pore:527-529).
__device__ __forceinline__ void write_work_item(const P &p, int32_t *w, int cell, int kx, int ky, int kz)
{
    w[0] = cell; w[1] = kx; w[2] = ky; w[3] = kz;
#pragma unroll
    for (int nb = 0; nb < 8; nb++) {
        int oc = ((kx + 1 - (nb >> 2)) * p.pnc[1] + (ky + 1 - ((nb >> 1) & 1))) * p.pnc[2] + (kz + 1 - (nb & 1));
        int beg = p.cell_start[oc];
        w[4 + nb] = beg;
        w[12 + nb] = nb == 0 ? p.cell_start[oc + 1] - beg : p.band_count[oc];
    }
    double *d = reinterpret_cast<double *>(w + 20);
    d[0] = p.lo[0][kx]; d[1] = p.edge[0][kx + 1];
    d[2] = p.lo[1][ky]; d[3] = p.edge[1][ky + 1];
    d[4] = p.lo[2][kz]; d[5] = p.edge[2][kz + 1];
}

// relation table of the slab decomposition: id -> slot, open addressing with linear probing
__device__ __forceinline__ uint32_t rel_hash(int32_t id) { return (uint32_t)id * 2654435761u; }
__device__ __forceinline__ void rel_insert(const P &p, int32_t id, int32_t slot)
{
    if (atomicAdd(p.rel_count, 1) >= p.rel_cap / 2) { atomicAdd(p.slab_overflow + 1, 1ull); return; }
    uint32_t mask = (uint32_t)p.rel_cap - 1, h = rel_hash(id) & mask;
    while (true) {
        int32_t prev = atomicCAS(&p.rel_id[h], -1, id);
        if (prev == -1 || prev == id) { p.rel_slot[h] = slot; return; }
        h = (h + 1) & mask;
    }
}
__device__ __forceinline__ int32_t rel_find(const P &p, int32_t id)
{
    uint32_t mask = (uint32_t)p.rel_cap - 1, h = rel_hash(id) & mask;
    while (true) {
        int32_t k = p.rel_id[h];
        if (k == id) return p.rel_slot[h];
        if (k == -1) return -1;
        h = (h + 1) & mask;
    }
}

__device__ __forceinline__ int64_t cur_n(const P &p) { return p.n_dev ? (int64_t)*p.n_dev : p.n; }

// flag words of the peer-to-peer exchange: the writer publishes with a release store at system scope after its data
// stores, the reader spins with acquire loads; sequence numbers only grow (compare as signed differences)
__device__ __forceinline__ void flag_publish(uint32_t *f, const uint32_t seq)
{
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f), "r"(seq) : "memory");
}
// A rank that never publishes (it crashed, or the ranks disagree about the protocol) must not hang the others: after
// AMC_FLAG_TIMEOUT_NS of waiting the wait gives up and counts itself in g_flag_timeouts; amc_slab_step reads the counter
// after the call and fails with AMC_E_STATE (the state of the handle is then undefined).
#define AMC_FLAG_TIMEOUT_NS 20000000000ull /* 20 s */
__device__ unsigned int g_flag_timeouts;
__device__ __forceinline__ void flag_wait(const uint32_t *f, const uint32_t seq)
{
    uint32_t v;
    unsigned long long t0 = 0;
    for (unsigned int spins = 0;; spins++) {
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
        if ((int32_t)(v - seq) >= 0) break;
        __nanosleep(64);
        if ((spins & 0xfffu) == 0xfffu) { /* look at the clock every 4096 polls (~0.5 ms) */
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (t0 == 0) t0 = now;
            else if (now - t0 > AMC_FLAG_TIMEOUT_NS) { atomicAdd(&g_flag_timeouts, 1u); break; }
        }
    }
}

// see k_recapture_list (amc_kernels.cuh)
// One round trip: the call sits at the tail of a cell visit, which is what a launch of k_pairs_group waits for.  A slot
// moved in several visits of one step is listed several times; the reader (k_recapture_list) takes each slot once.
__device__ __forceinline__ void touch_slot(const P &p, const int32_t s)
{
    int i = atomicAdd(p.touched_n, 1);
    if (i < p.touched_cap) p.touched[i] = s;
}
