/*
 * amc.h -- C ABI of libamc.so, the B200 (sm_100a) implementation of Argon_Monte_Carlo's
 * per-timestep hot path (drift -> wall collisions -> recapture -> cell-binned particle-particle
 * collisions -> mean-free-path / momentum bookkeeping).
 *
 * The upstream project is pure Python and has no FFI layer; its de-facto operator boundary is
 *   (1) the worker entry point  pairwise_particles_in_cell(...)      Open_Air_Pore_MC.py:160-255
 *       dispatched by pool.starmap over the cells of a colour group  Open_Air_Pore_MC.py:522-549
 *   (2) the wall operators taking an N-long boolean mask             Open_Air_Pore_MC.py:257-348,
 *                                                                    Temperature_Pore_MC.py:311-553
 *   (3) the step loop of each script                                 Open_Air_Pore_MC.py:416-557,
 *       Temperature_Pore_MC.py:662-853, Open_Air_Cube_MC.py:175-338
 * Each entry point below names the reference code it replaces.  Plain pointers and sizes only;
 * host arrays are owned by the caller and copied in/out, all device memory is owned by the handle
 * and no pointer is retained after a call returns.  Every function returns 0 on success or a
 * negative AMC_E_* code; amc_last_error() gives the message.  A handle is not thread-safe.
 * INTEGRATION.md shows the ctypes binding a maintainer of the reference would add.
 */
#ifndef AMC_H
#define AMC_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AMC_ABI_VERSION 1

enum { AMC_OK = 0, AMC_E_INVALID = -1, AMC_E_CUDA = -2, AMC_E_NOMEM = -3, AMC_E_CAPACITY = -4, AMC_E_STATE = -5 };

/* wall geometry (amc_config.kind) */
enum { AMC_KIND_CUBE = 0,  /* six specular planes, no MFP bookkeeping     Open_Air_Cube_MC.py:192-226 */
       AMC_KIND_PORE = 1,  /* specular pore walls with MFP bookkeeping    Open_Air_Pore_MC.py:442-485 */
       AMC_KIND_TEMP = 2   /* specular + energized (accommodating) walls  Temperature_Pore_MC.py:693-753 */ };
/* particle-particle schedule (amc_config.pp_mode) */
enum { AMC_PP_GROUPS = 0,  /* 8 colour groups, cells of a group independent   Open_Air_Pore_MC.py:522-549 */
       AMC_PP_SWEEP = 1    /* serial lexicographic sweep, write-back per cell  Open_Air_Cube_MC.py:232-336 */ };
/* random directions at energized walls (amc_config.rng_mode) */
enum { AMC_RNG_DEVICE = 0, /* counter-based Philox4x32-10 on the device (throughput mode) */
       AMC_RNG_HOST = 1    /* parity mode: host draws via amc_wall_hits_pending / amc_wall_apply_directions */ };
/* debug taps (amc_config.taps, OR-ed) */
enum { AMC_TAP_PAIRS = 1, AMC_TAP_WALL_BITS = 2, AMC_TAP_PATHS = 4 };

/* Temp wall cases in evaluation order (Temperature_Pore_MC.py:693-753).  Pore uses the first nine
 * slots in its own order 1, 2a, 2b, 3cold, 3hot, 4, 5bottom, 5top, 6 (Open_Air_Pore_MC.py:442-485);
 * Cube uses six: +x, -x, +y, -y, +z, -z (Open_Air_Cube_MC.py:192-226). */
enum { AMC_CASE_1 = 0, AMC_CASE_2A, AMC_CASE_2B, AMC_CASE_3C, AMC_CASE_3H, AMC_CASE_4, AMC_CASE_5B, AMC_CASE_5T,
       AMC_CASE_6H, AMC_CASE_6C, AMC_NUM_CASES };

#define AMC_NUM_BINS 200

/* Thresholds of the wall masks, evaluated on the host with the reference's own expressions. */
typedef struct amc_geom {
    double argon_mass, argon_radius, collision_range;
    double R_oa, R_oa_c;   /* open_air_radius, open_air_collision_radius                  Pore:35,67 */
    double R_p, R_p_c;     /* pore_coated_radius, pore_collision_radius                   Pore:25,69 */
    double R_g, R_g_c;     /* gap_radius, gap_collision_radius                            Pore:26,68 */
    double H, oah;         /* total_height, open_air_height                               Pore:39,36 */
    double z_cold;         /* total_height - open_air_height                              Pore:457 */
    double z_gb;           /* open_air_height + hot_coating_height                        Pore:465 */
    double z_gt_pore;      /* total_height - open_air_height - cold_coating_height        Pore:465 */
    double z_gt;           /* open_air_height + hot_coating_height + gap_height           Pore:371 */
    double ten_a;          /* 10*argon_radius                                             Pore:358 */
    double R_oa_sq, R_g_sq, R_p_sq;     /* radii ** 2                                     Pore:363-371 */
    double zc3, zh3;       /* (H - oah) + a, oah - a                                      Temp:708,713 */
    double zgt_m, zgb_p;   /* gap_top_height - a, gap_bottom_height + a                   Temp:720 */
    double R_g_c_sq, R_p_c_sq;          /* collision radii ** 2                           Temp:721,728 */
    double recap_lo, recap_hi;          /* 50e-9, H - 50e-9                               Temp:599,602 */
    double E_cold, E_hot;  /* surface_energy_cold / _hot (Debye integrals, host mpmath)   Temp:83-84 */
    double alpha_c, alpha_g;            /* accommodation coefficients                     Temp:76-77 */
    double cos85;          /* cos(85*pi/180)                                              Temp:136 */
} amc_geom;

typedef struct amc_config {
    int32_t abi_version;   /* AMC_ABI_VERSION */
    int32_t kind, pp_mode, rng_mode, taps;
    double dt;             /* timestep                                                    Pore:76 */
    double cube[3];        /* cube_x, cube_y, cube_z (AMC_KIND_CUBE)                      Cube:26-28 */
    amc_geom geom;
    /* collision-cell grid: axis a has nc[a] cells, first cell index c0[a];
     * edge[a][k] = (c0+k)*d (nc+1 entries) and lo[a][k] = edge[a][k] - band (nc entries) are the two
     * sides of the reference's strict layer masks                      Pore:527-529, Cube:233-237 */
    int32_t nc[3], c0[3];
    const double *edge[3];
    const double *lo[3];
    double overlap_sq;     /* smallest double t with sqrt(t) >= collision_range: `sqrt(d2) < cr` <=> `d2 < t` */
    uint64_t seed;         /* Philox key (AMC_RNG_DEVICE) */
    const double *cheb_coef; /* Chebyshev fit of surface_energy_gap(z)  Temp:143-152 (AMC_RNG_DEVICE) */
    int32_t cheb_n;
    double cheb_zmid, cheb_inv_half;
    double hist_first, hist_last; /* histogram range (0, 1e-6)                            Pore:575 */
    const double *hist_edges;     /* np.linspace(first, last, AMC_NUM_BINS+1) */
    int64_t max_particles;
    int64_t pair_capacity; /* AMC_TAP_PAIRS: max logged collisions between two amc_clear_taps() calls */
    int64_t path_capacity; /* AMC_TAP_PATHS: max logged completed paths */
} amc_config;

/* per-timestep counters: the numbers the reference prints every step (Pore:512-557, Temp:803-853) */
typedef struct amc_step_stats {
    int64_t wall_hits[AMC_NUM_CASES]; /* hits per wall case */
    int64_t wall_collisions;  /* "Num collisions from walls" (Pore: all cases; Temp: energized only) */
    int64_t pp_collisions;    /* particle-particle collisions resolved */
    int64_t pair_checks_ref;  /* reference-equivalent distance tests: sum over visited cells of n(n-1)/2 */
    int64_t pair_checks_exec; /* distance tests actually executed on the device */
    int64_t oob_after_walls;  /* "particles out of bounds after handling wall collisions" */
    int64_t oob_after_pp;     /* "... after particle-particle collisions" */
    int64_t oob_after_walls_recapture; /* Temp: "... after post wall collision recapture"        Temp:805 */
    int64_t oob_after_pp_recapture;    /* Temp: "... after post particle-particle recapture"     Temp:845 */
    int64_t errors;           /* floating-point anomalies (negative discriminant, zero relative speed) */
    int64_t completed_paths;  /* free paths completed during this step */
    double dpz, e_cold, e_hot; /* momentum_z_change / energy_transfer_{cold,hot} of this step  Temp:756-758 */
} amc_step_stats;

typedef struct amc_handle amc_handle;

/* lifetime.  `device`: CUDA ordinal. */
int amc_create(const amc_config *cfg, int device, amc_handle **out);
int amc_destroy(amc_handle *h);
const char *amc_last_error(const amc_handle *h); /* h may be NULL: last error of a failed amc_create */
int amc_abi_version(void);

/* particle state = the reference's module-global arrays (Pore:385-400), original index order.
 * dist*, flag may be NULL in amc_set_state (zeros); any output may be NULL in amc_get_state. */
int amc_set_state(amc_handle *h, int64_t n, const double *x, const double *y, const double *z, const double *vx,
                  const double *vy, const double *vz, const double *dist, const double *dist_x,
                  const double *dist_y, const double *dist_z, const uint8_t *flag);
int amc_get_state(amc_handle *h, double *x, double *y, double *z, double *vx, double *vy, double *vz, double *dist,
                  double *dist_x, double *dist_y, double *dist_z, uint8_t *flag);
int64_t amc_num_particles(const amc_handle *h);

/* production entry point: n_steps whole timesteps (body of the loops Pore:416-557 / Temp:662-853 /
 * Cube:175-338) without host round trips.  stats: n_steps entries or NULL.  AMC_RNG_HOST handles
 * must be stepped phase by phase instead (see below). */
int amc_step(amc_handle *h, int32_t n_steps, amc_step_stats *stats);

/* phase-level entry points, for per-phase parity checks (each is synchronous):
 *   amc_drift      Pore:427-437 / Temp:673-683 / Cube:180-187
 *   amc_walls      all wall cases in order: Pore:442-485 / Temp:693-753 (device RNG) / Cube:192-226
 *   amc_recapture  Pore num_out_of_bounds() 354-375 / Temp num_out_of_bounds()+recapture 560-616;
 *                  *count = Pore: particles teleported; Temp: the report count taken before recapture;
 *                  *count_after (nullable) = Temp: the report count taken again after recapture
 *   amc_pairs      the whole particle-particle pass Pore:522-549 / Temp:815-842 / Cube:232-336
 * stats (nullable) receives the counters the phase produces; other fields are zero. */
int amc_drift(amc_handle *h);
int amc_walls(amc_handle *h, amc_step_stats *stats);
int amc_recapture(amc_handle *h, int64_t *count, int64_t *count_after);
int amc_pairs(amc_handle *h, amc_step_stats *stats);

/* operator-level entry point: ONE wall operator of the reference applied to the particles selected by an N-long
 * boolean mask (indexed by particle), the way the reference's functions are called:
 *   AMC_OP_PLANE_MFP       hit_vertical_wall(hits, z_plane, 4 lists)              Open_Air_Pore_MC.py:257-292
 *   AMC_OP_SIDE_MFP        hit_cylinder_side_wall(hits, collision_radius, ...)    Open_Air_Pore_MC.py:294-348
 *   AMC_OP_PLANE_SPECULAR  hit_vertical_specular_wall(hits, z_plane)              Temperature_Pore_MC.py:311-315
 *   AMC_OP_SIDE_SPECULAR   hit_cylinder_specular_side_wall(hits, R, total_errs)   Temperature_Pore_MC.py:317-347
 * param = z_plane or collision_radius.  *n_hits = particles processed, *errors = floating-point error path taken
 * (the reference's try/except).  Completed free paths go to the handle's histograms / AMC_TAP_PATHS as usual.
 * (The energized operators Temp:349-553 are reached through amc_wall_hits_pending / amc_wall_apply_directions.) */
enum { AMC_OP_PLANE_MFP = 0, AMC_OP_SIDE_MFP = 1, AMC_OP_PLANE_SPECULAR = 2, AMC_OP_SIDE_SPECULAR = 3 };
int amc_wall_operator(amc_handle *h, int32_t op, const uint8_t *mask, double param, int64_t *n_hits, int64_t *errors);

/* parity hooks for the energized walls (AMC_KIND_TEMP): one wall case at a time, in AMC_CASE_*
 * order, after amc_drift.  Specular cases (AMC_CASE_1, _2A, _2B): call amc_wall_case (*errors: AMC_CASE_1 hits that
 * took the reference's floating-point error path).
 * Energized cases: amc_wall_hits_pending reports the hits in ascending particle index with the
 * vector the reference hands to random_inbounds_direction (Temp:375,444,514; NaN = the hit raised a
 * floating-point error in the reference and draws nothing) and the contact height (argument of
 * surface_energy_gap for AMC_CASE_4, Temp:519); the host draws one direction per valid hit from
 * its Mersenne-Twister streams (Temp:132-141) and calls amc_wall_apply_directions, which returns
 * per-hit momentum / energy contributions (dpz[k], de[k]) so the host can sum them in the
 * reference's sequential order (Temp:385,389).  surf_e: per-hit surface energy, AMC_CASE_4 only. */
int amc_wall_case(amc_handle *h, int32_t case_id, int64_t *n_hits, int64_t *errors);
int amc_wall_hits_pending(amc_handle *h, int32_t case_id, int64_t cap, int64_t *n_hits, int64_t *idx, double *normal3,
                          double *col_z);
int amc_wall_apply_directions(amc_handle *h, int32_t case_id, int64_t n_hits, const int64_t *idx, const double *dir3,
                              const double *surf_e, double *dpz, double *de, int64_t *errors);

/* Synthetic Maxwellian initial state generated on the device (replaces init_positions / init_velocities,
 * Pore:106-158, for the synthetic configurations of BASELINE.json: 10 M-particle cube, 100 M-particle pore, where
 * the host-side generators take minutes).  Particle i depends only on (seed, i): Philox4x32-10 with counter
 * (i, stream) gives its region (cumulative weights), a uniform position inside the region (cylinder about the z axis
 * or box) and velocity components ~ N(0, sigma^2) (Box-Muller).  keep_z_lo <= z < keep_z_hi selects the particles
 * that stay on this handle (one slab of a multi-GPU run; -inf / +inf: all of them, stored with slot == i);
 * ids (amc_set_ids) are set to i.  Path accumulators and flags start at zero. */
#define AMC_INIT_MAX_REGIONS 8
typedef struct amc_init_spec {
    int64_t n_total;                           /* particles of the whole job */
    uint64_t seed;
    int32_t n_regions;                         /* 1 .. AMC_INIT_MAX_REGIONS */
    int32_t shape;                             /* 0: cylinders about the z axis (radius, z_lo, z_hi); 1: boxes [0,bx] x [0,by] x [z_lo,z_hi] */
    double cum_weight[AMC_INIT_MAX_REGIONS];   /* cumulative region probabilities, last one 1.0 */
    double radius[AMC_INIT_MAX_REGIONS];
    double bx[AMC_INIT_MAX_REGIONS], by[AMC_INIT_MAX_REGIONS];
    double z_lo[AMC_INIT_MAX_REGIONS], z_hi[AMC_INIT_MAX_REGIONS];
    double sigma;                              /* sqrt(k_B T / m), Cube:56 */
    double keep_z_lo, keep_z_hi;
} amc_init_spec;
int amc_init_synthetic(amc_handle *h, const amc_init_spec *spec, int64_t *n_kept);

/* Overlap-free seeding for the state amc_init_synthetic just generated on a single-domain handle: the reference's own
 * random initial state leaves ~0.2 % of the particles overlapping a neighbour (1,051 pairs at 557,649 particles,
 * Pore:106-158) and resolves them as a transient burst of collisions in the first timesteps.  Up to max_rounds times:
 * find every overlapping pair (the detection pass of the step, exact test Pore:173-174), re-draw the position of its
 * higher-index particle from the same generator (attempt counter in the Philox counter).  *n_redrawn = positions
 * re-drawn in total, *n_left = particles still marked after the last round (0 = no overlapping pair left). */
int amc_seed_relax(amc_handle *h, int32_t max_rounds, int64_t *n_redrawn, int64_t *n_left);

/* outputs: completed free paths (the four lists Pore:410-413) as device-side histograms with
 * np.histogram's uniform-bin rule (Pore:575-596), their count and sums (for the printed means
 * Pore:565-568).  counts: [4][AMC_NUM_BINS] in the order total, x, y, z. */
int amc_get_histograms(amc_handle *h, uint64_t *counts, uint64_t *n_paths, double *sums4);

/* debug taps (enabled through amc_config.taps) */
int amc_get_pair_list(amc_handle *h, int64_t cap, int64_t *n, int64_t *hi, int64_t *lo, int32_t *group, int32_t *cell);
int amc_get_wall_bits(amc_handle *h, uint16_t *bits);  /* bit c set: AMC_CASE c hit in the last wall phase */
int amc_get_completed_paths(amc_handle *h, int64_t cap, int64_t *n, double *total, double *cx, double *cy, double *cz);
int amc_clear_taps(amc_handle *h);

/* checkpoint / resume (the reference keeps everything in module globals and cannot restart a run): together with
 * amc_get_state / amc_set_state and the step index these restore a handle exactly.  limbs8: the four free-path
 * sums as two 64-bit fixed-point limbs each (see amc_get_histograms for their decoded value). */
int amc_get_outputs_raw(amc_handle *h, uint64_t *counts, uint64_t *n_paths, uint64_t *limbs8);
int amc_set_outputs_raw(amc_handle *h, const uint64_t *counts, uint64_t n_paths, const uint64_t *limbs8);
int64_t amc_get_step_index(const amc_handle *h);

/* Order-independent checksum of the particle state this handle owns (slab handles: ghost copies excluded), computed
 * on the device: out[0], out[1] = two 64-bit sums over all (particle id, field, value bits) triples of the ten state
 * arrays and the full_path_traveled flag (Pore:385-400), out[2] = number of particles counted.  Sums of the values of
 * all ranks of a slab run (mod 2^64) equal the value of the single-domain run of the same job iff the id-ordered
 * states are bit-identical -- the check that replaces reading 8 GB of state back at 100 M particles. */
int amc_state_digest(amc_handle *h, uint64_t out[3]);

/* Field sampling: per-cell moments of the particle state, accumulated on the device.  The sampling grid is the
 * handle's collision-cell grid (a slab handle: the global grid, x and y of its own tables, z of gz_edge); a particle
 * goes to the cell with edge[a][k] <= v < edge[a][k+1] on every axis (the owner cell of the sort), cells are numbered
 * x-major, z-minor, and a particle outside the grid on any axis only counts in n_outside.  Ghost copies of a slab
 * handle are skipped, so the element-wise sum (mod 2^64) of the raw arrays of all ranks equals the single-domain
 * run's array bit for bit.  Per cell AMC_SAMPLE_WORDS uint64 words:
 *   [0] particles;  [1..6] sum vx, sum vy, sum vz;  [7..12] sum vx^2, sum vy^2, sum vz^2 (fp64 products)
 * every sum as two signed 64-bit fixed-point limbs (high, low): one particle adds i1 = rint(v * 2^S1) to the high
 * limb and i2 = rint((v - i1 * 2^-S1) * 2^S2) to the low limb (round half to even), S1/S2 = AMC_SAMPLE_V1/_V2 for
 * the velocities and AMC_SAMPLE_Q1/_Q2 for the squares; the sum decodes as high * 2^-S1 + low * 2^-S2.  Integer
 * adds make the words independent of thread order and of the split of the particles over ranks.  Headroom: 10^6
 * samples x 10^3 particles per cell at |v| <= 10^4 m/s keep every limb inside the signed 64-bit range (worst case:
 * 5.2e18 in a velocity high limb, 6.4e18 in a square high limb, 5.4e17 in a low limb).
 * A sample is taken on the state at the end of a timestep (what amc_get_state returns after amc_step): by amc_step /
 * amc_slab_step after every step whose index s (amc_get_step_index numbering) has s >= first_step and
 * (s - first_step) % every == 0, and by amc_sample_now.  Sampling changes no state, counter, histogram or digest;
 * while it is disabled (the default) no launch and no memory is added.  Memory: 8 * AMC_SAMPLE_WORDS bytes per cell.
 *   amc_sample_enable   allocate and zero the accumulators; every = 0: on demand only (amc_sample_now)
 *   amc_sample_disable  free them
 *   amc_sample_get_raw  acc: [cells][AMC_SAMPLE_WORDS] (nullable), samples taken, particles outside the grid
 *   amc_sample_set_raw  resume from amc_sample_get_raw's values (sampling must be enabled)
 *   amc_last_sample_ms  device time of the sampling kernel, summed over the samples of the last amc_step /
 *                       amc_slab_step / amc_sample_now call (the sample is part of [3] of amc_last_timing) */
#define AMC_SAMPLE_WORDS 13
#define AMC_SAMPLE_V1 19
#define AMC_SAMPLE_V2 49
#define AMC_SAMPLE_Q1 6
#define AMC_SAMPLE_Q2 36
int amc_sample_enable(amc_handle *h, int32_t every, int64_t first_step);
int amc_sample_disable(amc_handle *h);
int amc_sample_now(amc_handle *h);
int amc_sample_get_raw(amc_handle *h, uint64_t *acc, uint64_t *n_samples, uint64_t *n_outside);
int amc_sample_set_raw(amc_handle *h, const uint64_t *acc, uint64_t n_samples, uint64_t n_outside);
int amc_last_sample_ms(amc_handle *h, double *ms);

/* Velocity distribution (VDF): an extension of the field sample.  It covers the particles of the field sample (owned,
 * inside the sampling grid) on the steps of the field sample (the schedule of amc_sample_enable, and amc_sample_now).
 * One region per z layer k of the sampling grid (a slab handle: the global z edges), the rows of profile_z.csv.  Per
 * layer AMC_VDF_HISTS histograms, in the order vx, vy, vz, speed: the components over [lo, hi] = [-v_max, v_max], the
 * speed sqrt((vx*vx + vy*vy) + vz*vz) (fp64, separate roundings, correctly rounded sqrt) over [0, v_max].  Each
 * histogram has n_bins + 2 uint64 words [under, bin 0 .. bin n_bins-1, over]: x < lo counts in under, x > hi or NaN in
 * over, and lo <= x <= hi in the bin of np.histogram(x, bins=n_bins, range=(lo, hi)) -- the last bin closed on the
 * right -- found as in np.histogram against edges = np.linspace(lo, hi, n_bins + 1) computed on the host at enable time:
 *   i = (int64)(((x - lo) / (hi - lo)) * n_bins);  i == n_bins: i - 1;  then x < edges[i]: i - 1, else
 *   x >= edges[i+1] and i != n_bins - 1: i + 1
 * Every histogram of a layer, under and over included, therefore sums to the particle counts (word 0) of the field
 * sample's cells of that layer.  Layout [ncz][AMC_VDF_HISTS][n_bins + 2]; all counts are integer adds, so the words do
 * not depend on thread order or on the split over ranks, and merging ranks is an element-wise sum (mod 2^64).  The
 * number of samples is the one amc_sample_get_raw reports; amc_last_sample_ms covers the VDF too.  The VDF changes no
 * state, counter, histogram, digest or field-sampling word; while it is disabled (the default) nothing is added.
 * Memory: ncz * AMC_VDF_HISTS * (n_bins + 2) * 8 bytes.
 *   amc_vdf_enable   allocate and zero the histograms; AMC_E_STATE without field sampling, AMC_E_INVALID for n_bins
 *                    outside [1, AMC_VDF_MAX_BINS] or v_max not finite and > 0; re-enabling starts from zero
 *   amc_vdf_disable  free them (amc_sample_disable does too)
 *   amc_vdf_layout   layers, bins and v_max of the enabled VDF
 *   amc_vdf_get_raw  acc: [ncz][AMC_VDF_HISTS][n_bins + 2]
 *   amc_vdf_set_raw  resume from amc_vdf_get_raw's words (the VDF must be enabled with the same layout) */
#define AMC_VDF_HISTS 4
#define AMC_VDF_MAX_BINS 4096
int amc_vdf_enable(amc_handle *h, int32_t n_bins, double v_max);
int amc_vdf_disable(amc_handle *h);
int amc_vdf_layout(amc_handle *h, int32_t *ncz, int32_t *n_bins, double *v_max);
int amc_vdf_get_raw(amc_handle *h, uint64_t *acc);
int amc_vdf_set_raw(amc_handle *h, const uint64_t *acc);

/* Surface recording: what the gas does to the walls, per wall element, accumulated on the device as every wall
 * interaction happens.  The walls are the AMC_CASE_* slots of the handle's kind (Pore 9, Temp 10, Cube 6; a case the
 * kind does not have has no element), each cut into bins on the handle's sampling grid (that of amc_sample_*; a slab
 * handle: the global z edges).  c = (cx, cy, cz) is the contact point of a hit:
 *   cylinders (Pore 0, 5, 8; Temp 1, 4, 6H, 6C; radius Rc = R_oa_c, R_g_c, R_p_c): the z layer k of cz with
 *     edge[k] <= cz < edge[k+1] (the rows of profile_z.csv)
 *   planes of Pore / Temp: the annulus k with rsq[k] <= cx*cx + cy*cy < rsq[k+1], rsq[k] = (k*dr) * (k*dr) in fp64,
 *     dr = (edge_x[nc_x] - edge_x[0]) / nc_x, k < ceil(R_oa / dr)
 *   cube faces (case 2a: the face x = cube[a], 2a+1: the face x_a = 0): the pair of owner cells (o1, o2) of the two
 *     in-plane axes b1 < b2, element o1 * nc[b2] + o2
 * Elements are numbered case-major (amc_surface_layout: offsets[c] .. offsets[c+1]).  A hit in no bin -- a NaN contact,
 * a contact outside the grid, or the reference's floating-point error path (the case counts a hit and applies nothing)
 * -- counts in outside[c] instead, so per case the hits of the elements plus outside[c] equal the sum of wall_hits[c].
 * Contact points: planes (x - vx*t, y - vy*t, zp) with t = (z - zp) / vz before the reflection; cylinders
 * (x - vx*t, y - vy*t, z - vz*t) with t from the side-wall quadratic; energized cases the contact point of the reference
 * (Temp:372-375, 440-444); cube faces the same rewind on the particle as it stands when its axis is handled, with the
 * face's own coordinate set to the face.  With dv = v_out - v_in (fp64, per component) and with n the unit normal from
 * the wall into the gas, every hit adds, in IEEE fp64 with separate roundings:
 *   cylinders  ex = cx / Rc, ey = cy / Rc;  dv.n = -(dvx*ex + dvy*ey);  dv.t1 = dvz (t1 = z);  dv.t2 = dvy*ex - dvx*ey
 *              (t2 = azimuth (-ey, ex, 0))
 *   annuli     r = sqrt(cx*cx + cy*cy);  ex = cx / r, ey = cy / r (r = 0: ex = 1, ey = 0);  dv.n = s * dvz with
 *              s = +1 for 2A / 3C / 5B (Pore 1, 3, 6) and -1 for 2B / 3H / 5T (Pore 2, 4, 7);  dv.t1 = dvx*ex + dvy*ey
 *              (radial);  dv.t2 = dvy*ex - dvx*ey (azimuth)
 *   cube faces dv.n = -dv_a on the face at cube[a], +dv_a on the face at 0;  dv.t1 = dv_b1, dv.t2 = dv_b2
 * and dE, the energy the gas gained: the dE of the energized exchange (Temp:377-389) on energized cases -- case 4
 * included, which the e_cold / e_hot series of amc_step_stats leave out -- and 0 on specular ones.  Per element
 * AMC_SURF_WORDS uint64 words:
 *   [0] hits;  [1..2] sum dv.n;  [3..4] sum dv.t1;  [5..6] sum dv.t2 (m/s);  [7..8] sum dE (J)
 * every sum as two signed 64-bit fixed-point limbs, the scheme of amc_sample_*: S1 / S2 = AMC_SURF_V1 / _V2 for the
 * velocities, AMC_SURF_E1 / _E2 for the energy.  Headroom: 10^9 hits per element at |v| <= 10^4 m/s (|dv| <= 2*10^4,
 * |dE| <= 3.4e-18 J for argon) keep every limb inside the signed 64-bit range (worst case: 1.4e18 in a velocity high
 * limb, 4.2e18 in the energy high limb, 5.4e17 in a low limb).
 * Recorded wall phases: every timestep of amc_step and amc_slab_step, every amc_slab_advect and amc_walls call, and
 * every amc_wall_case(h, AMC_CASE_1) (the first case of a host-RNG wall phase); *n_steps counts them, so that rates
 * are sums / (n_steps * dt).  Not recorded: amc_wall_operator (operator-level parity entry point), and the recapture
 * (a teleport, not a wall interaction).  A slab handle records a hit on the rank that owns the particle at the start
 * of the step, so the element-wise sum (mod 2^64) of the raw arrays of all ranks equals the single-domain run's.
 * Recording changes no state, counter, histogram or digest; while it is disabled (the default) no launch and no memory
 * is added.  Memory: 8 * AMC_SURF_WORDS bytes per element.
 *   amc_surface_enable   allocate, zero and start recording (a slab handle: after amc_slab_enable)
 *   amc_surface_disable  free the accumulators
 *   amc_surface_layout   offsets[AMC_NUM_CASES + 1]: first element of every case, offsets[AMC_NUM_CASES] = elements
 *   amc_surface_get_raw  acc: [elements][AMC_SURF_WORDS] (nullable), wall phases recorded, outside (nullable)
 *   amc_surface_set_raw  resume from amc_surface_get_raw's values (recording must be enabled) */
#define AMC_SURF_WORDS 9
#define AMC_SURF_V1 16
#define AMC_SURF_V2 46
#define AMC_SURF_E1 90
#define AMC_SURF_E2 120
int amc_surface_enable(amc_handle *h);
int amc_surface_disable(amc_handle *h);
int amc_surface_layout(amc_handle *h, int64_t offsets[AMC_NUM_CASES + 1]);
int amc_surface_get_raw(amc_handle *h, uint64_t *acc, uint64_t *n_steps, uint64_t outside[AMC_NUM_CASES]);
int amc_surface_set_raw(amc_handle *h, const uint64_t *acc, uint64_t n_steps, const uint64_t outside[AMC_NUM_CASES]);

/* Plane flux recording: particles and what they carry through the z planes of the sampling grid, counted on the
 * device.  Planes: the ncz + 1 z edges edge_z[0..ncz] of the handle's sampling grid (that of amc_sample_*), the
 * boundaries of the rows of profile_z.csv.  The plane count of a position is cnt(z) = the number of planes with
 * edge_z[k] <= z (np.searchsorted(edge_z, z, side='right'); NaN counts ncz + 1, as in NumPy).  At every record point
 * each particle's cnt(z) (c1) is compared with the one stored at the previous record point (c0, a per-particle int32
 * snapshot indexed by particle id): c1 > c0 crossed planes c0 .. c1-1 upward (s = +1), c1 < c0 crossed planes
 * c1 .. c0-1 downward (s = -1); every crossed plane gets one full contribution, then the snapshot becomes c1.  The
 * carried quantities use the particle's velocity in the current state (the end of the step).  Per plane
 * AMC_FLUX_WORDS uint64 words:
 *   [0] upward crossings;  [1] downward crossings;  [2..3] sum s*vx;  [4..5] sum s*vy;  [6..7] sum s*vz;
 *   [8..9] sum s*((vx*vx + vy*vy) + vz*vz) (fp64, separate roundings)
 * every sum as two signed 64-bit fixed-point limbs, the scheme of amc_sample_*: S1 / S2 = AMC_FLUX_V1 / _V2 for the
 * velocities, AMC_FLUX_Q1 / _Q2 for the squares.  Headroom: 10^10 crossings per plane at speeds <= 10^4 m/s keep every
 * limb inside the signed 64-bit range (worst case: 6.6e18 in a velocity high limb, 4.0e18 in a square high limb,
 * 5.4e18 in a low limb).  Rates are sums / (n_steps * dt), n_steps = record points.
 * The words count net crossings between consecutive record points: a particle that crosses and comes back in between
 * counts nothing, and everything that moves a particle counts -- drift, wall reflections, collision moves, and the
 * recapture's z teleports (at most 10*a in Pore, to 50 nm from an end in Temp: only planes that close to z = 0 or
 * z = H see those).  The words are a function of the sequence of states at the record points alone.
 * Record points: the end of every timestep of amc_step, and every amc_flux_now.  amc_set_state, amc_init_synthetic
 * and amc_seed_relax re-take the snapshot from the state they leave; the other phase-level calls do not (their moves
 * are recorded at the next record point).  Single-domain handles only: a migrant between slab ranks would have to
 * carry its plane count.  Recording changes no state, counter, histogram, digest or sample / VDF / surface word;
 * while it is disabled (the default) no launch and no memory is added.  Memory: 8 * AMC_FLUX_WORDS bytes per plane and
 * 4 bytes per particle slot (max_particles).
 *   amc_flux_enable   allocate and zero the accumulators, take the snapshot of the current state; re-enabling starts
 *                     from zero.  AMC_E_STATE on a slab handle (and amc_slab_enable / amc_set_ids return AMC_E_STATE
 *                     while recording is on), AMC_E_INVALID unless the particle ids are 0 .. n-1
 *   amc_flux_disable  free everything
 *   amc_flux_now      one record point (the host-RNG / phase-level paths call it after a timestep)
 *   amc_flux_layout   number of planes (ncz + 1)
 *   amc_flux_get_raw  acc: [planes][AMC_FLUX_WORDS] (nullable), record points taken
 *   amc_flux_set_raw  resume from amc_flux_get_raw's values (recording must be enabled) */
#define AMC_FLUX_WORDS 10
#define AMC_FLUX_V1 16
#define AMC_FLUX_V2 46
#define AMC_FLUX_Q1 2
#define AMC_FLUX_Q2 32
int amc_flux_enable(amc_handle *h);
int amc_flux_disable(amc_handle *h);
int amc_flux_now(amc_handle *h);
int amc_flux_layout(amc_handle *h, int32_t *n_planes);
int amc_flux_get_raw(amc_handle *h, uint64_t *acc, uint64_t *n_steps);
int amc_flux_set_raw(amc_handle *h, const uint64_t *acc, uint64_t n_steps);

/* set the step counter that keys the device RNG (default: counts amc_step / amc_walls calls from 0) */
int amc_set_step_index(amc_handle *h, int64_t step);

/* device time (ms, CUDA events on the handle's stream) of the kernels of the last amc_step call:
 * [0] advect+walls  [1] cell sort (scan+scatter)  [2] pair kernels  [3] recapture/other  [4] whole call.
 * launches: number of kernel launches in that call. */
int amc_last_timing(amc_handle *h, double ms[5], int64_t *launches);

/* device time (ms, summed over the steps of the last amc_step call) of the detection kernel alone (k_detect: the
 * neighbour search over every reference cell, Pore:168-174); the rest of [2] above is the ordered resolution.
 * Handles driven through the amc_slab_* entry points accumulate this time over steps instead. */
int amc_last_detect_ms(amc_handle *h, double *ms);
/* the same for k_scatter_advect, the kernel that carries out the timestep on the way to the sorted slot (the longest
 * kernel of a step: reads 93 B and writes 85 B per particle) */
int amc_last_scatter_ms(amc_handle *h, double *ms);

/* ------------------------------------------------------------------------------------------------
 * Slab decomposition along z over several GPUs (one handle = one rank = the reference cells of the
 * global z layers [cuts[rank], cuts[rank+1]); no counterpart in the reference, results are identical
 * to the single-domain run).  The handle is created with the z tables of its own layers; the exchange
 * buffers are device memory owned by the caller (e.g. torch tensors), who also moves them between
 * ranks (NCCL all-to-all / neighbour send-recv) between the calls below.  Record = 12 doubles
 * (10 state values, particle id, flag bits); every buffer starts with one header record (count).
 *   per step:  amc_slab_advect -> [all-to-all xfer_send -> xfer_recv] -> amc_slab_sort
 *              -> amc_slab_pairs_begin(pre_round) -> if pre_round: [neighbour exchange] -> amc_slab_apply(-1)
 *              -> for g in 0..7: amc_slab_group(g) -> [neighbour exchange] -> amc_slab_apply(g)
 *              -> amc_slab_finish */
typedef struct amc_slab_config {
    int32_t rank, nranks;
    const int32_t *cuts;     /* nranks+1 global z-layer cuts, cuts[0] = 0, cuts[nranks] = global cell count in z */
    int32_t gncz;            /* global number of cells in z */
    const double *gz_edge;   /* global z edges, gncz+1 */
    const double *gz_lo;     /* global z low-side bounds, gncz */
    int32_t xfer_capacity;   /* records per neighbouring rank (rank +-1): migrants and ghost copies */
    int32_t xfer_capacity_far; /* records per non-neighbouring rank (teleports across several slabs: rare) */
    int32_t bnd_capacity;    /* records per neighbour and colour group */
    void *xfer_send, *xfer_recv;                 /* sum over peers of (capacity+1) * 96 bytes each; block of peer d starts at
                                                    record sum_{e<d} (capacity_e + 1), capacity_e = xfer_capacity if |e-rank|==1 else _far */
    void *bnd_send_up, *bnd_send_down;           /* (bnd_capacity+1) * 96 bytes each */
    void *bnd_recv_up, *bnd_recv_down;           /* received from the rank above / below */
} amc_slab_config;

int amc_slab_enable(amc_handle *h, const amc_slab_config *cfg);
int amc_set_stream(amc_handle *h, void *cuda_stream);   /* run on the caller's stream (e.g. torch's current stream) */
int amc_set_ids(amc_handle *h, const int64_t *ids);     /* global particle indices of the state set by amc_set_state */
int amc_slab_advect(amc_handle *h);
int amc_slab_sort(amc_handle *h, int64_t *n_resident);
int amc_slab_pairs_begin(amc_handle *h, int32_t pre_round); /* pre_round != 0: pack the late exports now (needed when a cut is even) */
int amc_slab_group(amc_handle *h, int32_t group);
int amc_slab_apply(amc_handle *h, int32_t group_done);
int amc_slab_finish(amc_handle *h, amc_step_stats *stats);
int amc_slab_get_owned(amc_handle *h, int64_t cap, int64_t *n, int64_t *ids, double *x, double *y, double *z, double *vx,
                       double *vy, double *vz, double *dist, double *dist_x, double *dist_y, double *dist_z, uint8_t *flag);

/* Device-resident multi-GPU stepping (one rank per GPU, e.g. one process per GPU under torchrun).  The step-wise
 * entry points above leave the transport to the caller (NCCL through torch.distributed) and return to the host
 * after every phase; here the handle owns the exchange buffers, maps the other ranks' buffers peer-to-peer over
 * NVLink (cudaIpc across processes) and amc_slab_step enqueues whole timesteps: every transfer is a kernel that
 * writes the records straight into the receiver's buffer and then a sequence number into the receiver's flag word;
 * the receiving kernel spins on that word.  No NCCL call, no host synchronisation and no host code between the
 * colour groups.  Results are identical to the step-wise path and to the single-domain run.
 *   amc_slab_enable (buffer pointers of amc_slab_config may be NULL) -> amc_slab_p2p_setup on every rank
 *   -> exchange the descriptors between the ranks (all-gather) -> amc_slab_p2p_connect -> amc_slab_step ...
 * Ranks that wait on one another must run on different GPUs (kernels of two ranks on one GPU are not guaranteed to
 * run at the same time); emulated ranks on one GPU use the step-wise entry points. */
typedef struct amc_slab_p2p_desc {
    int64_t pid;             /* process that owns the allocation */
    int32_t device, rank;
    uint64_t base;           /* device address of the allocation in that process */
    uint8_t ipc[64];         /* cudaIpcMemHandle_t of the allocation */
    int64_t off_flags, off_xfer, off_bnd_up, off_bnd_down; /* byte offsets inside the allocation */
    int64_t xfer_stride, bnd_stride;                       /* doubles per buffer half */
} amc_slab_p2p_desc;
int amc_slab_p2p_setup(amc_handle *h, amc_slab_p2p_desc *out);
int amc_slab_p2p_connect(amc_handle *h, const amc_slab_p2p_desc *all_ranks); /* nranks descriptors, indexed by rank */
/* n_steps whole timesteps of this rank's slab; pre_round as in amc_slab_pairs_begin (the same value on every rank).
 * stats: n_steps entries (this rank's share of every counter) or NULL. */
int amc_slab_step(amc_handle *h, int32_t n_steps, int32_t pre_round, amc_step_stats *stats);

#ifdef __cplusplus
}
#endif
#endif /* AMC_H */
