// amc_api.cu -- host side of libamc.so: handle, memory, kernel sequencing, the C ABI of include/amc.h.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -fmad=false -shared -Xcompiler -fPIC
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <string>
#include <vector>
#include <algorithm>
#include <unistd.h>
#include "amc_kernels.cuh"

static thread_local std::string g_create_error;

struct amc_handle {
    amc_config cfg;
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    cudaStream_t aux = nullptr;          // second stream of amc_step: pair-pass bookkeeping beside the scatter
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    bool slab = false;
    int32_t xf_total = 0;
    // peer-to-peer exchange (amc_slab_p2p_*): one allocation = flag words + both halves of every receive buffer
    char *p2p_base = nullptr;
    bool p2p = false;
    std::vector<void *> p2p_opened;  // cudaIpcOpenMemHandle mappings, closed in amc_destroy
    uint32_t xf_seq = 0, bnd_seq = 0;
    int32_t *d_n = nullptr;          // device-resident particle count of amc_slab_step
    amc_slab_p2p_desc p2p_desc;
    std::vector<cudaEvent_t> grp_events; // amc_slab_step with AMC_SLAB_TRACE: around every colour-group launch of the last step of a chunk
    double group_ms[10] = {0};           // [0..7] group launches, [8] closing hand-over, [9] steps accumulated
    amc_init_spec init_spec;         // of the last amc_init_synthetic call (amc_seed_relax re-draws from it)
    bool have_init_spec = false;
    int32_t *d_counters = nullptr; // slab mode: xf_count[nranks], n_in, bnd_n[2], rel_count, n_foreign, compact count
    unsigned long long *d_slab_overflow = nullptr;
    P p;                        // kernel parameter block (device pointers)
    int64_t cap = 0, n = 0;
    std::vector<void *> allocs; // every cudaMalloc, freed in amc_destroy
    StatsDev *d_stats = nullptr; // [stats_cap]
    int stats_cap = 0;
    StatsDev *h_stats = nullptr; // pinned
    int32_t *d_tile_sums = nullptr;
    int n_buckets = 0;          // padded owner cells + OUT
    bool have_prior = false;
    int64_t step_index = 0;
    int pair_grid = 148 * 5;    // persistent CTAs of k_pairs_group: SMs x resident CTAs per SM
    int pair_grid_fused = 148;  // the same for the fused (in-kernel hand-over) variant
    int det_grid_tma = 148 * 4; // persistent CTAs of k_detect_tma
    int32_t sweep_pass = 0;     // tag of the last pass of the event-driven cube sweep (P::sw_pass)
    // host-RNG parity mode: pending hits of the last amc_wall_hits_pending call
    int32_t *d_pend_count = nullptr, *d_pend_slot = nullptr, *d_pend_id = nullptr;
    double *d_pend_nrm = nullptr, *d_pend_colz = nullptr, *d_pend_dirs = nullptr, *d_pend_se = nullptr, *d_pend_dpz = nullptr, *d_pend_de = nullptr;
    int32_t pend_cap = 0;
    std::vector<int32_t> pend_slot;
    std::vector<int64_t> pend_id;
    int pend_case = -1;
    // timing
    std::vector<cudaEvent_t> events;
    double last_ms[5] = {0, 0, 0, 0, 0};
    std::vector<cudaEvent_t> det_events; // two per step of the last amc_step chunk: around k_detect_tma
    int det_slot = -1;                   // step of the chunk run_pairs is recording for (-1: none)
    int slab_phase = 0;                  // slab mode: PH_* bits of the step between amc_slab_advect and amc_slab_sort
    bool slab_det_pending = false;       // slab mode: events around k_detect_tma recorded, not yet read
    double last_detect_ms = 0;
    std::vector<cudaEvent_t> sc_events;  // two per step of the last amc_step chunk: around k_scatter_advect
    double last_scatter_ms = 0;
    int64_t last_launches = 0;
    // field sampling (amc_sample_*): accumulators [cells][AMC_SAMPLE_WORDS] + the outside counter; null: disabled
    unsigned long long *d_sample = nullptr;
    int64_t sample_cells = 0;
    int32_t sample_every = 0;
    int64_t sample_first = 0;
    uint64_t n_samples = 0;
    std::vector<cudaEvent_t> sample_events; // two per sample of the last call: around k_sample
    int sample_slot = 0;                    // samples recorded into sample_events by the current call
    double last_sample_ms = 0;
    // velocity distribution (amc_vdf_*): histograms [ncz][AMC_VDF_HISTS][n_bins + 2]; null: disabled
    unsigned long long *d_vdf = nullptr;
    double *d_vdf_edges = nullptr; // VdfArgs::edges
    VdfArgs va = {};               // kernel parameter of k_sample<true> (va.acc = d_vdf)
    int32_t vdf_ncz = 0;
    double vdf_vmax = 0;
    // surface recording (amc_surface_*): accumulators [elements][AMC_SURF_WORDS] + outside[AMC_NUM_CASES]; null: off
    unsigned long long *d_surf = nullptr;
    double *d_surf_rsq = nullptr; // annulus bounds, SurfP::rsq
    SurfP sp = {};                // kernel parameter of the recording kernels (sp.acc = d_surf)
    uint64_t surf_steps = 0;      // wall phases recorded
    double surf_dr = 0;           // x cell width of the grid: (edge[0][nc] - edge[0][0]) / nc
    // plane flux recording (amc_flux_*): accumulators [ncz + 1][AMC_FLUX_WORDS] + FluxArgs::bad, the snapshot [cap];
    // null: off
    unsigned long long *d_flux = nullptr;
    int32_t *d_flux_snap = nullptr;
    uint64_t flux_steps = 0;      // record points taken
    std::string error;

    int fail(int code, const std::string &msg)
    {
        error = msg;
        return code;
    }
};

#define CK(call)                                                                                              \
    do {                                                                                                      \
        cudaError_t e_ = (call);                                                                              \
        if (e_ != cudaSuccess)                                                                                \
            return h->fail(AMC_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));                   \
    } while (0)

template <typename T> static int dev_alloc(amc_handle *h, T **ptr, size_t count)
{
    void *q = nullptr;
    cudaError_t e = cudaMalloc(&q, std::max<size_t>(count, 1) * sizeof(T));
    if (e != cudaSuccess) return h->fail(AMC_E_NOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e));
    h->allocs.push_back(q);
    *ptr = (T *)q;
    return AMC_OK;
}
#define ALLOC(ptr, count)                                 \
    do {                                                  \
        int rc_ = dev_alloc(h, &(ptr), (size_t)(count));  \
        if (rc_ != AMC_OK) return rc_;                    \
    } while (0)

static int alloc_arrays(amc_handle *h, Arrays &a, int64_t n)
{
    ALLOC(a.pos, n); /* cudaMalloc returns 256-byte aligned blocks: every record is 32-byte aligned */
    ALLOC(a.vx, n); ALLOC(a.vy, n); ALLOC(a.vz, n);
    ALLOC(a.d, n); ALLOC(a.dx, n); ALLOC(a.dy, n); ALLOC(a.dz, n);
    return AMC_OK;
}

// largest double t with sqrt(t) <= R: then sqrt(v) > R <=> v > t for every double v
static double sq_threshold_gt(double R)
{
    double t = R * R;
    while (std::sqrt(t) <= R) t = std::nextafter(t, INFINITY);
    while (std::sqrt(t) > R) t = std::nextafter(t, 0.0);
    return t;
}
// smallest double t with sqrt(t) >= R: then sqrt(v) < R <=> v < t
static double sq_threshold_lt(double R)
{
    double t = R * R;
    while (std::sqrt(t) >= R) t = std::nextafter(t, 0.0);
    while (std::sqrt(t) < R) t = std::nextafter(t, INFINITY);
    return t;
}

static inline unsigned grid_for(int64_t n, int threads) { return (unsigned)((n + threads - 1) / threads); }

static void stats_to_host(const amc_handle *h, const StatsDev &s, amc_step_stats *o)
{
    memset(o, 0, sizeof(*o));
    int64_t all = 0, energized = 0;
    for (int c = 0; c < AMC_NUM_CASES; c++) {
        o->wall_hits[c] = (int64_t)s.wall_hits[c];
        all += o->wall_hits[c];
        if (c >= AMC_CASE_3C) energized += o->wall_hits[c];
    }
    o->wall_collisions = h->cfg.kind == AMC_KIND_TEMP ? energized : all;
    o->pp_collisions = (int64_t)s.pp;
    o->pair_checks_ref = (int64_t)s.checks_ref;
    o->pair_checks_exec = (int64_t)s.checks_exec;
    o->oob_after_walls = (int64_t)s.oob_walls;
    o->oob_after_pp = (int64_t)s.oob_pp;
    o->oob_after_walls_recapture = (int64_t)s.oob_walls_after;
    o->oob_after_pp_recapture = (int64_t)s.oob_pp_after;
    o->errors = (int64_t)s.errors;
    o->completed_paths = (int64_t)s.paths;
    o->dpz = ldexp((double)(long long)s.dpz[0], -116) + ldexp((double)(long long)s.dpz[1], -156);
    o->e_cold = ldexp((double)(long long)s.ecold[0], -108) + ldexp((double)(long long)s.ecold[1], -148);
    o->e_hot = ldexp((double)(long long)s.ehot[0], -108) + ldexp((double)(long long)s.ehot[1], -148);
}

static int check_overflow(amc_handle *h, const StatsDev &s)
{
    if (s.cell_overflow) return h->fail(AMC_E_CAPACITY, "a collision cell holds more than AMC_MAX_MEMBERS particles");
    if (s.cand_overflow) return h->fail(AMC_E_CAPACITY, "internal: candidate bookkeeping overflow in one cell visit");
    if (s.esc_overflow) return h->fail(AMC_E_CAPACITY, "escaped-particle list overflow");
    return AMC_OK;
}

extern "C" int amc_abi_version(void) { return AMC_ABI_VERSION; }

extern "C" const char *amc_last_error(const amc_handle *h) { return h ? h->error.c_str() : g_create_error.c_str(); }

extern "C" int64_t amc_num_particles(const amc_handle *h) { return h ? h->n : 0; }

extern "C" int amc_destroy(amc_handle *h)
{
    if (!h) return AMC_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (void *q : h->p2p_opened) cudaIpcCloseMemHandle(q);
    for (void *q : h->allocs) cudaFree(q);
    for (cudaEvent_t e : h->events) cudaEventDestroy(e);
    for (cudaEvent_t e : h->det_events) cudaEventDestroy(e);
    for (cudaEvent_t e : h->sc_events) cudaEventDestroy(e);
    for (cudaEvent_t e : h->sample_events) cudaEventDestroy(e);
    if (h->d_sample) cudaFree(h->d_sample);
    if (h->d_vdf) cudaFree(h->d_vdf);
    if (h->d_vdf_edges) cudaFree(h->d_vdf_edges);
    if (h->d_surf) cudaFree(h->d_surf);
    if (h->d_surf_rsq) cudaFree(h->d_surf_rsq);
    if (h->d_flux) cudaFree(h->d_flux);
    if (h->d_flux_snap) cudaFree(h->d_flux_snap);
    if (h->h_stats) cudaFreeHost(h->h_stats);
    if (h->aux) { cudaStreamSynchronize(h->aux); cudaStreamDestroy(h->aux); }
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    if (h->stream && h->own_stream) cudaStreamDestroy(h->stream);
    delete h;
    return AMC_OK;
}

static int create_impl(amc_handle *h, const amc_config *cfg, int device)
{
    if (cfg->abi_version != AMC_ABI_VERSION) return h->fail(AMC_E_INVALID, "amc_config.abi_version mismatch");
    if (cfg->kind < AMC_KIND_CUBE || cfg->kind > AMC_KIND_TEMP) return h->fail(AMC_E_INVALID, "bad kind");
    if (cfg->pp_mode != AMC_PP_GROUPS && cfg->pp_mode != AMC_PP_SWEEP) return h->fail(AMC_E_INVALID, "bad pp_mode");
    if (cfg->max_particles <= 0 || cfg->max_particles > 0x7fffffffLL) return h->fail(AMC_E_INVALID, "max_particles out of range");
    for (int a = 0; a < 3; a++) {
        if (cfg->nc[a] < 1 || !cfg->edge[a] || !cfg->lo[a]) return h->fail(AMC_E_INVALID, "grid tables missing");
        if (cfg->pp_mode == AMC_PP_GROUPS && a < 2 && (cfg->nc[a] & 1)) return h->fail(AMC_E_INVALID, "colour groups need an even cell count in x and y");
    }
    if (!cfg->hist_edges) return h->fail(AMC_E_INVALID, "hist_edges missing");
    if (cfg->kind == AMC_KIND_TEMP && cfg->rng_mode == AMC_RNG_DEVICE && (!cfg->cheb_coef || cfg->cheb_n < 1))
        return h->fail(AMC_E_INVALID, "device RNG mode needs the Chebyshev table of surface_energy_gap");
    h->cfg = *cfg;
    h->device = device;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) return h->fail(AMC_E_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(e));
    CK(cudaSetDevice(device));
    CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->aux, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    P &p = h->p;
    memset(&p, 0, sizeof(p));
    h->cap = cfg->max_particles;
    p.cap = h->cap;
    int rc;
    if ((rc = alloc_arrays(h, p.a, h->cap)) != AMC_OK) return rc;
    if ((rc = alloc_arrays(h, p.b, h->cap)) != AMC_OK) return rc;
    ALLOC(p.key, h->cap); ALLOC(p.rank, h->cap);
    p.kind = cfg->kind; p.pp_mode = cfg->pp_mode; p.dt = cfg->dt;
    for (int a = 0; a < 3; a++) p.cube[a] = cfg->cube[a];
    p.g = cfg->geom;
    p.cr = cfg->geom.collision_range; p.mass = cfg->geom.argon_mass; p.overlap_sq = cfg->overlap_sq;
    if (cfg->kind != AMC_KIND_CUBE) {
        p.gt_Roa = sq_threshold_gt(cfg->geom.R_oa); p.gt_Rp = sq_threshold_gt(cfg->geom.R_p); p.gt_Rg = sq_threshold_gt(cfg->geom.R_g);
        p.lt_Rp = sq_threshold_lt(cfg->geom.R_p); p.lt_Rg = sq_threshold_lt(cfg->geom.R_g);
    }
    if (cfg->kind == AMC_KIND_TEMP) {
        const amc_geom &g = cfg->geom;
        const double zs[8] = {g.oah, g.zh3, g.z_gb, g.zgb_p, g.z_gt, g.zgt_m, g.z_cold, g.zc3};
        double zA = g.H, zB = 0.0;
        for (double v : zs) { zA = std::min(zA, v); zB = std::max(zB, v); }
        p.calm_zA = zA; p.calm_zB = zB;
        p.calm_rA = std::min(p.gt_Roa, g.R_oa_sq);
        p.calm_rC = std::min(std::min(std::min(p.calm_rA, g.R_p_sq), std::min(g.R_g_c_sq, g.R_p_c_sq)), g.R_g_sq);
        p.calm_ok = zA > 0.0 && zB < g.H && p.calm_rA > 0.0 && p.calm_rC > 0.0;
    }
    int64_t ncell = 1;
    for (int a = 0; a < 3; a++) {
        p.nc[a] = cfg->nc[a]; p.pnc[a] = cfg->nc[a] + 1;
        ncell *= p.pnc[a];
        double *de = nullptr, *dl = nullptr;
        ALLOC(de, cfg->nc[a] + 1); ALLOC(dl, cfg->nc[a]);
        CK(cudaMemcpy(de, cfg->edge[a], (cfg->nc[a] + 1) * sizeof(double), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(dl, cfg->lo[a], cfg->nc[a] * sizeof(double), cudaMemcpyHostToDevice));
        p.edge[a] = de; p.lo[a] = dl;
        p.e0[a] = cfg->edge[a][0];
        p.inv_d[a] = (double)cfg->nc[a] / (cfg->edge[a][cfg->nc[a]] - cfg->edge[a][0]);
    }
    h->surf_dr = (cfg->edge[0][cfg->nc[0]] - cfg->edge[0][0]) / (double)cfg->nc[0];
    if (ncell + 2 > 0x7fffffffLL) return h->fail(AMC_E_INVALID, "too many cells");
    p.ncell_pad = (int32_t)ncell;
    for (int a = 0; a < 3; a++) p.nh[a] = (cfg->nc[a] + 1) / 2;
    h->n_buckets = (int)ncell + 2; /* padded owner cells + OUT + GONE (slab mode: emigrants and dropped ghosts) */
    ALLOC(p.band_count, h->n_buckets + 2); ALLOC(p.rest_count, h->n_buckets + 1); ALLOC(p.cell_start, h->n_buckets + 1);
    p.touched_n = p.band_count + (h->n_buckets + 1);
    p.touched_cap = (int32_t)std::min<int64_t>(std::max<int64_t>(h->cap / 32, 8192), 1 << 22);
    ALLOC(p.touched, p.touched_cap); ALLOC(p.touch_mark, h->cap);
    CK(cudaMemset(p.touch_mark, 0, h->cap * sizeof(int32_t)));
    CK(cudaMemset(p.band_count, 0, (h->n_buckets + 2) * sizeof(int32_t)));
    ALLOC(h->d_tile_sums, (h->n_buckets + SCAN_TILE - 1) / SCAN_TILE + 1);
    p.key0 = (uint32_t)cfg->seed; p.key1 = (uint32_t)(cfg->seed >> 32);
    if (cfg->cheb_coef && cfg->cheb_n > 0) {
        double *dc = nullptr;
        ALLOC(dc, cfg->cheb_n);
        CK(cudaMemcpy(dc, cfg->cheb_coef, cfg->cheb_n * sizeof(double), cudaMemcpyHostToDevice));
        p.cheb = dc; p.cheb_n = cfg->cheb_n; p.cheb_zmid = cfg->cheb_zmid; p.cheb_inv_half = cfg->cheb_inv_half;
    }
    {
        double *dh = nullptr;
        ALLOC(dh, AMC_NUM_BINS + 1);
        CK(cudaMemcpy(dh, cfg->hist_edges, (AMC_NUM_BINS + 1) * sizeof(double), cudaMemcpyHostToDevice));
        p.hist_edges = dh; p.hist_first = cfg->hist_first; p.hist_last = cfg->hist_last;
    }
    ALLOC(p.hist, 4 * AMC_NUM_BINS); ALLOC(p.path_count, 1); ALLOC(p.path_sums, 8 + 3); /* + scratch of amc_state_digest */
    CK(cudaMemset(p.hist, 0, 4 * AMC_NUM_BINS * sizeof(unsigned long long)));
    CK(cudaMemset(p.path_count, 0, sizeof(unsigned long long)));
    CK(cudaMemset(p.path_sums, 0, 8 * sizeof(unsigned long long)));
    if (cfg->taps & AMC_TAP_PAIRS) {
        p.pair_cap = std::max<int64_t>(cfg->pair_capacity, 1);
        ALLOC(p.pair_count, 1); ALLOC(p.pair_hi, p.pair_cap); ALLOC(p.pair_lo, p.pair_cap);
        ALLOC(p.pair_group, p.pair_cap); ALLOC(p.pair_cell, p.pair_cap);
        CK(cudaMemset(p.pair_count, 0, sizeof(unsigned long long)));
    }
    if (cfg->taps & AMC_TAP_PATHS) {
        p.path_cap = std::max<int64_t>(cfg->path_capacity, 1);
        ALLOC(p.tap_path_count, 1);
        for (int k = 0; k < 4; k++) ALLOC(p.tap_paths[k], p.path_cap);
        CK(cudaMemset(p.tap_path_count, 0, sizeof(unsigned long long)));
    }
    if (cfg->taps & AMC_TAP_WALL_BITS) {
        ALLOC(p.wall_bits, h->cap);
        CK(cudaMemset(p.wall_bits, 0, h->cap * sizeof(uint16_t)));
    }
    {
        int64_t per_group = (int64_t)(cfg->nc[0] / 2 + 1) * (cfg->nc[1] / 2 + 1) * (cfg->nc[2] / 2 + 1);
        p.wl_stride = (int32_t)per_group;
        ALLOC(p.wl, (size_t)per_group * 8 * AMC_WI); ALLOC(p.wl_count, AMC_WL_COUNTERS); ALLOC(p.cell_active, per_group * 8);
        p.wl_next = p.wl_count + 8;
        p.dl_count = p.wl_count + 16;
        ALLOC(p.dl, (size_t)cfg->nc[0] * cfg->nc[1] * cfg->nc[2] * AMC_WI); ALLOC(p.cell_n, per_group * 8);
        ALLOC(p.wl_hit, (size_t)per_group * 8 * AMC_HIT_REC);
        CK(cudaMemset(p.wl_count, 0, AMC_WL_COUNTERS * sizeof(int32_t)));
        CK(cudaMemset(p.cell_active, 0, per_group * 8 * sizeof(int32_t)));
        CK(cudaMemset(p.cell_n, 0, per_group * 8 * sizeof(int32_t)));
        // fp32 filter of the detection pass.  Coordinates relative to the cell's low corner lie in (0, W) and are
        // rounded to fp32 with an error <= 2^-24 W each; a coordinate difference is then off by e <= 3 * 2^-24 W
        // (two roundings plus its own), the distance by <= sqrt(3) e, and the fused square sum by a relative
        // 4 * 2^-24.  Every pair the exact test (Pore:173-174) accepts therefore has an fp32 squared distance
        // below ((cr + sqrt(3) e)^2) (1 + 2^-21); the factors used here are twice as generous.
        double wmax = 0.0;
        p.det_own_is_member = 1;
        for (int a = 0; a < 3; a++)
            for (int k = 0; k < cfg->nc[a]; k++) {
                wmax = std::max(wmax, cfg->edge[a][k + 1] - cfg->lo[a][k]);
                if (!(cfg->lo[a][k] < cfg->edge[a][k])) p.det_own_is_member = 0;
            }
        double e_abs = 6.0 * std::ldexp(wmax, -24);
        double r_f = std::sqrt(cfg->overlap_sq) * (1.0 + 1e-9) + 2.0 * e_abs;
        double thr = r_f * r_f * (1.0 + std::ldexp(1.0, -20));
        p.det_thr = std::nextafterf((float)thr, INFINITY);
        p.det_w = std::nextafterf((float)(1.05 * std::sqrt((double)p.det_thr)), INFINITY);
    }
    if (cfg->pp_mode == AMC_PP_SWEEP) {
        // event-driven serial sweep of the cube stage; the plain one-CTA walk over every cell (k_cube_sweep) takes
        // over a pass in which a column overflows its list
        const int64_t ncols = (int64_t)cfg->nc[0] * cfg->nc[1];
        p.sw_colcap = (int32_t)std::min<int64_t>(h->cap, std::max<int64_t>(512, 6 * h->cap / ncols + 64));
        if (const char *cc = getenv("AMC_SWEEP_COLCAP")) p.sw_colcap = std::max(1, atoi(cc)); /* tests: force the hand-over to the plain sweep */
        ALLOC(p.sw_col, (size_t)ncols * p.sw_colcap); ALLOC(p.sw_col_n, ncols);
        ALLOC(p.sw_tag, h->cap); ALLOC(p.sw_ml, h->cap); ALLOC(p.sw_xs, h->cap); ALLOC(p.sw_ys, h->cap);
        ALLOC(p.sw_state, 2);
        CK(cudaMemset(p.sw_tag, 0, h->cap * sizeof(int32_t)));
    }
    p.esc_cap = (int32_t)std::min<int64_t>(std::max<int64_t>(h->cap / 64, 4096), 1 << 22);
    ALLOC(p.esc_count, 1); ALLOC(p.esc_slot, p.esc_cap); ALLOC(p.esc_cell, (size_t)p.esc_cap * 8); ALLOC(p.esc_next, (size_t)p.esc_cap * 8);
    CK(cudaMemset(p.esc_count, 0, sizeof(int32_t)));
    CK(cudaMemset(p.esc_cell, 0xff, (size_t)p.esc_cap * 8 * sizeof(int32_t)));
    h->stats_cap = 256;
    ALLOC(h->d_stats, h->stats_cap);
    CK(cudaMallocHost((void **)&h->h_stats, h->stats_cap * sizeof(StatsDev)));
    p.stats = h->d_stats;
    if (cfg->kind == AMC_KIND_TEMP && cfg->rng_mode == AMC_RNG_HOST) {
        h->pend_cap = (int32_t)std::min<int64_t>(h->cap, 1 << 22);
        ALLOC(h->d_pend_count, 1); ALLOC(h->d_pend_slot, h->pend_cap); ALLOC(h->d_pend_id, h->pend_cap);
        ALLOC(h->d_pend_nrm, (size_t)h->pend_cap * 3); ALLOC(h->d_pend_colz, h->pend_cap);
        ALLOC(h->d_pend_dirs, (size_t)h->pend_cap * 3); ALLOC(h->d_pend_se, h->pend_cap);
        ALLOC(h->d_pend_dpz, h->pend_cap); ALLOC(h->d_pend_de, h->pend_cap);
    }
    {
        int sms = 0, per_sm = 0;
        CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
        CK(cudaFuncSetAttribute(k_pairs_group<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        CK(cudaFuncSetAttribute(k_pairs_group<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        {
            int per_sm_fused = 0; /* the fused variant waits inside the kernel: every CTA of its grid must be resident */
            CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_fused, k_pairs_group<true>, PAIR_THREADS, 0));
            h->pair_grid_fused = std::max(1, sms * std::max(per_sm_fused, 1));
        }
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_pairs_group<false>, PAIR_THREADS, 0));
        h->pair_grid = std::max(1, sms * std::max(per_sm, 1));
        CK(cudaFuncSetAttribute(k_detect_tma<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_detect_tma<false>, DET_THREADS, 0));
        h->det_grid_tma = std::max(1, sms * std::max(per_sm, 1));
        ALLOC(p.mv_spill, (size_t)std::max(h->pair_grid, 1) * AMC_MAX_MEMBERS * 3);
    }
    CK(cudaDeviceSynchronize());
    return AMC_OK;
}

extern "C" int amc_create(const amc_config *cfg, int device, amc_handle **out)
{
    if (!cfg || !out) { g_create_error = "null argument"; return AMC_E_INVALID; }
    amc_handle *h = new amc_handle();
    int rc = create_impl(h, cfg, device);
    if (rc != AMC_OK) {
        g_create_error = h->error;
        amc_destroy(h);
        *out = nullptr;
        return rc;
    }
    *out = h;
    return AMC_OK;
}

static int flux_retake(amc_handle *h);

static int ensure_prior(amc_handle *h)
{
    if (h->have_prior) return AMC_OK;
    ALLOC(h->p.px, h->cap); ALLOC(h->p.py, h->cap); ALLOC(h->p.pz, h->cap);
    h->have_prior = true;
    return AMC_OK;
}

extern "C" int amc_set_state(amc_handle *h, int64_t n, const double *x, const double *y, const double *z,
                             const double *vx, const double *vy, const double *vz, const double *dist,
                             const double *dist_x, const double *dist_y, const double *dist_z, const uint8_t *flag)
{
    if (!h) return AMC_E_INVALID;
    if (n < 0 || n > h->cap) return h->fail(AMC_E_INVALID, "n exceeds max_particles");
    if (n && (!x || !y || !z || !vx || !vy || !vz)) return h->fail(AMC_E_INVALID, "null position/velocity array");
    CK(cudaSetDevice(h->device));
    Arrays &a = h->p.a;
    // positions and flags arrive as separate arrays: staged in the SoaView over the idle b records, then packed
    const SoaView v = soa_view(h->p.b.pos, h->cap);
    const double *src[10] = {x, y, z, vx, vy, vz, dist, dist_x, dist_y, dist_z};
    double *dst[10] = {v.x, v.y, v.z, a.vx, a.vy, a.vz, a.d, a.dx, a.dy, a.dz};
    for (int k = 0; k < 10; k++) {
        if (src[k]) CK(cudaMemcpyAsync(dst[k], src[k], n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        else CK(cudaMemsetAsync(dst[k], 0, n * sizeof(double), h->stream));
    }
    if (flag) CK(cudaMemcpyAsync(v.flag, flag, n, cudaMemcpyHostToDevice, h->stream));
    else CK(cudaMemsetAsync(v.flag, 0, n, h->stream));
    h->n = n;
    h->p.n = n;
    if (n) k_pack_pos<<<grid_for(n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(h->p, 0); // slot == particle index
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(h->stream));
    return flux_retake(h);
}

extern "C" int amc_init_synthetic(amc_handle *h, const amc_init_spec *spec, int64_t *n_kept)
{
    if (!h || !spec) return AMC_E_INVALID;
    if (spec->n_total < 0 || spec->n_total > 0x7fffffffLL) return h->fail(AMC_E_INVALID, "n_total out of range");
    if (spec->n_regions < 1 || spec->n_regions > AMC_INIT_MAX_REGIONS) return h->fail(AMC_E_INVALID, "n_regions out of range");
    if (spec->shape != 0 && spec->shape != 1) return h->fail(AMC_E_INVALID, "bad shape");
    if (!(spec->sigma >= 0.0)) return h->fail(AMC_E_INVALID, "bad sigma");
    const bool keep_all = std::isinf(spec->keep_z_lo) && spec->keep_z_lo < 0 && std::isinf(spec->keep_z_hi) && spec->keep_z_hi > 0;
    if (keep_all && spec->n_total > h->cap) return h->fail(AMC_E_INVALID, "n_total exceeds max_particles");
    CK(cudaSetDevice(h->device));
    int32_t *cnt = h->p.wl_count + 20; /* spare counter of the pair-pass block */
    CK(cudaMemsetAsync(cnt, 0, sizeof(int32_t), h->stream));
    if (spec->n_total)
        k_init_synthetic<<<148 * 8, ADVECT_THREADS, 0, h->stream>>>(h->p, *spec, keep_all ? 1 : 0, cnt, h->cap);
    CK(cudaGetLastError());
    int32_t c = 0;
    CK(cudaMemcpyAsync(&c, cnt, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    int64_t n = keep_all ? spec->n_total : c;
    if (n > h->cap) return h->fail(AMC_E_CAPACITY, "max_particles too small for the particles of this slab");
    h->n = n;
    h->p.n = n;
    h->init_spec = *spec;
    h->have_init_spec = keep_all;
    if (n_kept) *n_kept = n;
    return flux_retake(h);
}

// bring the state back to original index order (slot == id); b arrays are scratch between phases
static int unsort(amc_handle *h)
{
    if (h->n == 0) return AMC_OK;
    k_inverse_perm<<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(h->p);
    k_unsort<<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(h->p);
    CK(cudaGetLastError());
    std::swap(h->p.a, h->p.b);
    return AMC_OK;
}

extern "C" int amc_get_state(amc_handle *h, double *x, double *y, double *z, double *vx, double *vy, double *vz,
                             double *dist, double *dist_x, double *dist_y, double *dist_z, uint8_t *flag)
{
    if (!h) return AMC_E_INVALID;
    if (h->slab) return h->fail(AMC_E_STATE, "slab handles hold global particle ids: read them with amc_slab_get_owned");
    CK(cudaSetDevice(h->device));
    int rc = unsort(h);
    if (rc != AMC_OK) return rc;
    Arrays &a = h->p.a;
    // the records leave as separate arrays: unpacked into the SoaView over the b records (scratch after the unsort)
    const SoaView v = soa_view(h->p.b.pos, h->cap);
    if (h->n) k_unpack_pos<<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(h->p);
    CK(cudaGetLastError());
    double *dst[10] = {x, y, z, vx, vy, vz, dist, dist_x, dist_y, dist_z};
    const double *src[10] = {v.x, v.y, v.z, a.vx, a.vy, a.vz, a.d, a.dx, a.dy, a.dz};
    for (int k = 0; k < 10; k++)
        if (dst[k]) CK(cudaMemcpyAsync(dst[k], src[k], h->n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (flag) CK(cudaMemcpyAsync(flag, v.flag, h->n, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return AMC_OK;
}

// counting sort of the state into owner-cell order; keys/ranks/cell_count must be filled
static int sort_scatter(amc_handle *h, int64_t *launches)
{
    P &p = h->p;
    int m = h->n_buckets;
    int ntiles = (m + SCAN_TILE - 1) / SCAN_TILE;
    k_scan_tiles<<<ntiles, SCAN_THREADS, 0, h->stream>>>(p.band_count, p.rest_count, p.cell_start, h->d_tile_sums, m);
    k_scan_sums<<<1, SCAN_THREADS, 0, h->stream>>>(h->d_tile_sums, ntiles);
    k_scan_add<<<ntiles, SCAN_THREADS, 0, h->stream>>>(p.cell_start, h->d_tile_sums, m, (int32_t)h->n);
    k_scatter<<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(p);
    CK(cudaGetLastError());
    std::swap(p.a, p.b);
    if (launches) *launches += 4;
    return AMC_OK;
}

// bookkeeping of one pair pass that depends on the sorted layout only through cell_start / band_count (not on the
// particle arrays): reset of the escaped list and of the worklists, list of the cells k_detect_tma has to look at
static int prepare_pairs(amc_handle *h, cudaStream_t st)
{
    P &p = h->p;
    k_pp_begin<<<1, 256, 0, st>>>(p);
    CK(cudaMemsetAsync(p.wl_count, 0, AMC_WL_COUNTERS * sizeof(int32_t), st));
    int ncell = p.nc[0] * p.nc[1] * p.nc[2];
    CK(cudaMemsetAsync(p.cell_active, 0, (size_t)p.wl_stride * 8 * sizeof(int32_t), st));
    CK(cudaMemsetAsync(p.cell_n, 0, (size_t)p.wl_stride * 8 * sizeof(int32_t), st));
    k_build_worklist<<<grid_for(ncell, ADVECT_THREADS), ADVECT_THREADS, 0, st>>>(p);
    CK(cudaGetLastError());
    return AMC_OK;
}

// the detection pass of a timestep: candidates staged by bulk copies (DESIGN section 5)
static void launch_detect(amc_handle *h)
{
    k_detect_tma<false><<<h->det_grid_tma, DET_THREADS, 0, h->stream>>>(h->p);
}

// launch `kernel` programmatically dependent on the kernel before it in the stream (griddepcontrol, see pdl_trigger /
// pdl_wait in amc_kernels.cuh): its CTAs may become resident while that kernel still runs
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, cudaStream_t stream, Args &&...args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = 0; cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

static int run_pairs(amc_handle *h, int64_t *launches, bool prepared = false)
{
    P &p = h->p;
    if (p.pp_mode == AMC_PP_SWEEP) { /* event-driven sweep: detection over all columns, then the flagged cells in sweep order */
        if (h->sweep_pass == 0x7fffffff) { /* pass tags exhausted: start over with clean tags */
            CK(cudaMemsetAsync(p.sw_tag, 0, h->cap * sizeof(int32_t), h->stream));
            h->sweep_pass = 0;
        }
        p.sw_pass = ++h->sweep_pass;
        const int ncell = p.nc[0] * p.nc[1] * p.nc[2];
        CK(cudaMemsetAsync(p.cell_active, 0, (size_t)((ncell + 31) / 32) * sizeof(int32_t), h->stream));
        CK(cudaMemsetAsync(p.sw_state, 0, 2 * sizeof(unsigned long long), h->stream));
        k_sweep_detect<<<p.nc[0] * p.nc[1], SWD_THREADS, 0, h->stream>>>(p);
        k_sweep_events<<<1, SWE_THREADS, 0, h->stream>>>(p);
        k_cube_sweep<<<1, SWEEP_THREADS, 0, h->stream>>>(p); /* returns at once unless a column list overflowed */
        if (launches) *launches += 3;
    } else {
        if (!prepared) {
            int rc = prepare_pairs(h, h->stream);
            if (rc != AMC_OK) return rc;
        }
        int ncell = p.nc[0] * p.nc[1] * p.nc[2];
        if (h->det_slot >= 0) CK(cudaEventRecord(h->det_events[2 * h->det_slot], h->stream));
        launch_detect(h);
        if (h->det_slot >= 0) CK(cudaEventRecord(h->det_events[2 * h->det_slot + 1], h->stream));
        unsigned grid = (unsigned)std::min<int64_t>((int64_t)h->pair_grid, std::max<int64_t>(ncell / 8, 1));
        k_pairs_group<false><<<grid, PAIR_THREADS, 0, h->stream>>>(p, 0);
        for (int g = 1; g < 8; g++) CK(launch_pdl(k_pairs_group<false>, dim3(grid), dim3(PAIR_THREADS), h->stream, p, g));
        if (launches) *launches += 11;
    }
    CK(cudaGetLastError());
    return AMC_OK;
}

// grow one of the handle's event pools to `count` events
static int ensure_events(amc_handle *h, std::vector<cudaEvent_t> &pool, size_t count)
{
    while (pool.size() < count) {
        cudaEvent_t e;
        CK(cudaEventCreate(&e));
        pool.push_back(e);
    }
    return AMC_OK;
}

// ---- field sampling --------------------------------------------------------------------------------
static bool sample_due(const amc_handle *h, int64_t step)
{
    return h->d_sample && h->sample_every > 0 && step >= h->sample_first && (step - h->sample_first) % h->sample_every == 0;
}

static void sample_reset_timing(amc_handle *h)
{
    h->sample_slot = 0;
    h->last_sample_ms = 0;
}

// one sample of the state in h->p.a on h->stream (count: p.n, or the device-resident count inside amc_slab_step);
// grid_n: slots the launch covers; launches (nullable) counts the kernel launch
static int launch_sample(amc_handle *h, int64_t grid_n, int64_t *launches)
{
    int rc = ensure_events(h, h->sample_events, (size_t)(2 * h->sample_slot + 2));
    if (rc != AMC_OK) return rc;
    const P &p = h->p;
    SampleArgs sa;
    sa.acc = h->d_sample;
    sa.outside = h->d_sample + h->sample_cells * AMC_SAMPLE_WORDS;
    if (p.slab) { sa.zedge = p.gz_edge; sa.ncz = p.gncz; sa.ze0 = p.g_e0z; sa.zinv = p.g_inv_dz; }
    else { sa.zedge = p.edge[2]; sa.ncz = p.nc[2]; sa.ze0 = p.e0[2]; sa.zinv = p.inv_d[2]; }
    CK(cudaEventRecord(h->sample_events[2 * h->sample_slot], h->stream));
    if (grid_n > 0) {
        if (h->d_vdf) k_sample<true><<<grid_for(grid_n, SAMPLE_THREADS), SAMPLE_THREADS, 0, h->stream>>>(p, sa, h->va);
        else k_sample<false><<<grid_for(grid_n, SAMPLE_THREADS), SAMPLE_THREADS, 0, h->stream>>>(p, sa, VdfArgs{});
        if (launches) *launches += 1;
    }
    CK(cudaEventRecord(h->sample_events[2 * h->sample_slot + 1], h->stream));
    CK(cudaGetLastError());
    h->sample_slot++;
    h->n_samples++;
    return AMC_OK;
}

// after a synchronisation: add the kernel times of the samples recorded since the last call
static int sample_collect_timing(amc_handle *h)
{
    for (int k = 0; k < h->sample_slot; k++) {
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, h->sample_events[2 * k], h->sample_events[2 * k + 1]));
        h->last_sample_ms += ms;
    }
    h->sample_slot = 0;
    return AMC_OK;
}

extern "C" int amc_sample_enable(amc_handle *h, int32_t every, int64_t first_step)
{
    if (!h) return AMC_E_INVALID;
    if (every < 0) return h->fail(AMC_E_INVALID, "every < 0");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    const int64_t ncz = h->slab ? h->p.gncz : h->cfg.nc[2];
    const int64_t cells = (int64_t)h->cfg.nc[0] * h->cfg.nc[1] * ncz;
    if (h->d_sample && cells != h->sample_cells) { cudaFree(h->d_sample); h->d_sample = nullptr; }
    const size_t bytes = ((size_t)cells * AMC_SAMPLE_WORDS + 1) * sizeof(unsigned long long);
    if (!h->d_sample) {
        cudaError_t e = cudaMalloc(&h->d_sample, bytes);
        if (e != cudaSuccess) { h->d_sample = nullptr; return h->fail(AMC_E_NOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e)); }
    }
    CK(cudaMemset(h->d_sample, 0, bytes));
    h->sample_cells = cells;
    h->sample_every = every;
    h->sample_first = first_step;
    h->n_samples = 0;
    return AMC_OK;
}

extern "C" int amc_sample_disable(amc_handle *h)
{
    if (!h) return AMC_E_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    if (h->d_sample) CK(cudaFree(h->d_sample));
    h->d_sample = nullptr;
    h->sample_cells = 0; h->sample_every = 0; h->sample_first = 0; h->n_samples = 0;
    return amc_vdf_disable(h); // the VDF is part of the field sample
}

extern "C" int amc_sample_now(amc_handle *h)
{
    if (!h) return AMC_E_INVALID;
    if (!h->d_sample) return h->fail(AMC_E_STATE, "sampling is not enabled (amc_sample_enable)");
    CK(cudaSetDevice(h->device));
    sample_reset_timing(h);
    int rc = launch_sample(h, h->n, nullptr);
    if (rc != AMC_OK) return rc;
    CK(cudaStreamSynchronize(h->stream));
    return sample_collect_timing(h);
}

extern "C" int amc_sample_get_raw(amc_handle *h, uint64_t *acc, uint64_t *n_samples, uint64_t *n_outside)
{
    if (!h) return AMC_E_INVALID;
    if (!h->d_sample) return h->fail(AMC_E_STATE, "sampling is not enabled (amc_sample_enable)");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    if (acc) CK(cudaMemcpy(acc, h->d_sample, (size_t)h->sample_cells * AMC_SAMPLE_WORDS * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    if (n_outside) CK(cudaMemcpy(n_outside, h->d_sample + h->sample_cells * AMC_SAMPLE_WORDS, sizeof(uint64_t), cudaMemcpyDeviceToHost));
    if (n_samples) *n_samples = h->n_samples;
    return AMC_OK;
}

extern "C" int amc_sample_set_raw(amc_handle *h, const uint64_t *acc, uint64_t n_samples, uint64_t n_outside)
{
    if (!h || !acc) return AMC_E_INVALID;
    if (!h->d_sample) return h->fail(AMC_E_STATE, "sampling is not enabled (amc_sample_enable)");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(h->d_sample, acc, (size_t)h->sample_cells * AMC_SAMPLE_WORDS * sizeof(uint64_t), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->d_sample + h->sample_cells * AMC_SAMPLE_WORDS, &n_outside, sizeof(uint64_t), cudaMemcpyHostToDevice));
    h->n_samples = n_samples;
    return AMC_OK;
}

extern "C" int amc_last_sample_ms(amc_handle *h, double *ms)
{
    if (!h || !ms) return AMC_E_INVALID;
    *ms = h->last_sample_ms;
    return AMC_OK;
}

// ---- velocity distribution -------------------------------------------------------------------------
static size_t vdf_words(const amc_handle *h)
{
    return (size_t)h->vdf_ncz * AMC_VDF_HISTS * (h->va.n_bins + 2);
}

// np.linspace(lo, hi, n + 1): lo + k * ((hi - lo) / n), the last edge hi itself.  The volatile keeps the host compiler
// from fusing the multiply and the add, which NumPy does not.
static void linspace_edges(double lo, double hi, int n, double *e)
{
    const double step = (hi - lo) / n;
    for (int k = 0; k < n; k++) {
        volatile double t = (double)k * step;
        e[k] = t + lo;
    }
    e[n] = hi;
}

extern "C" int amc_vdf_enable(amc_handle *h, int32_t n_bins, double v_max)
{
    if (!h) return AMC_E_INVALID;
    if (!h->d_sample) return h->fail(AMC_E_STATE, "the VDF extends the field sample: enable sampling first (amc_sample_enable)");
    if (n_bins < 1 || n_bins > AMC_VDF_MAX_BINS) return h->fail(AMC_E_INVALID, "n_bins outside [1, AMC_VDF_MAX_BINS]");
    if (!(std::isfinite(v_max) && v_max > 0)) return h->fail(AMC_E_INVALID, "v_max must be finite and > 0");
    int rc = amc_vdf_disable(h);
    if (rc != AMC_OK) return rc;
    h->vdf_ncz = (int32_t)(h->sample_cells / ((int64_t)h->cfg.nc[0] * h->cfg.nc[1]));
    h->vdf_vmax = v_max;
    VdfArgs &va = h->va;
    va.n_bins = n_bins;
    va.lo[0] = -v_max; va.hi[0] = v_max;
    va.lo[1] = 0.0; va.hi[1] = v_max;
    std::vector<double> edges(2 * (size_t)(n_bins + 1));
    linspace_edges(va.lo[0], va.hi[0], n_bins, edges.data());
    linspace_edges(va.lo[1], va.hi[1], n_bins, edges.data() + n_bins + 1);
    cudaError_t e = cudaMalloc(&h->d_vdf, vdf_words(h) * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMalloc(&h->d_vdf_edges, edges.size() * sizeof(double));
    if (e != cudaSuccess) {
        amc_vdf_disable(h);
        return h->fail(AMC_E_NOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e));
    }
    CK(cudaMemset(h->d_vdf, 0, vdf_words(h) * sizeof(unsigned long long)));
    CK(cudaMemcpy(h->d_vdf_edges, edges.data(), edges.size() * sizeof(double), cudaMemcpyHostToDevice));
    va.acc = h->d_vdf;
    va.edges = h->d_vdf_edges;
    return AMC_OK;
}

extern "C" int amc_vdf_disable(amc_handle *h)
{
    if (!h) return AMC_E_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    if (h->d_vdf) CK(cudaFree(h->d_vdf));
    if (h->d_vdf_edges) CK(cudaFree(h->d_vdf_edges));
    h->d_vdf = nullptr; h->d_vdf_edges = nullptr;
    h->va = VdfArgs{};
    h->vdf_ncz = 0; h->vdf_vmax = 0;
    return AMC_OK;
}

extern "C" int amc_vdf_layout(amc_handle *h, int32_t *ncz, int32_t *n_bins, double *v_max)
{
    if (!h) return AMC_E_INVALID;
    if (!h->d_vdf) return h->fail(AMC_E_STATE, "the VDF is not enabled (amc_vdf_enable)");
    if (ncz) *ncz = h->vdf_ncz;
    if (n_bins) *n_bins = h->va.n_bins;
    if (v_max) *v_max = h->vdf_vmax;
    return AMC_OK;
}

extern "C" int amc_vdf_get_raw(amc_handle *h, uint64_t *acc)
{
    if (!h || !acc) return AMC_E_INVALID;
    if (!h->d_vdf) return h->fail(AMC_E_STATE, "the VDF is not enabled (amc_vdf_enable)");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(acc, h->d_vdf, vdf_words(h) * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return AMC_OK;
}

extern "C" int amc_vdf_set_raw(amc_handle *h, const uint64_t *acc)
{
    if (!h || !acc) return AMC_E_INVALID;
    if (!h->d_vdf) return h->fail(AMC_E_STATE, "the VDF is not enabled (amc_vdf_enable)");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(h->d_vdf, acc, vdf_words(h) * sizeof(uint64_t), cudaMemcpyHostToDevice));
    return AMC_OK;
}

// ---- surface recording ---------------------------------------------------------------------------
// elements of every wall case (include/amc.h): z layers for the cylinders, annuli for the planes of Pore / Temp, the
// in-plane cell pairs for the cube faces; rsq (nullable) receives the annulus bounds
static void surf_layout(const amc_handle *h, int64_t off[AMC_NUM_CASES + 1], std::vector<double> *rsq)
{
    const int64_t nc[3] = {h->cfg.nc[0], h->cfg.nc[1], h->slab ? h->p.gncz : h->cfg.nc[2]};
    const int32_t kind = h->cfg.kind;
    const int64_t nann = kind == AMC_KIND_CUBE ? 0 : (int64_t)ceil(h->cfg.geom.R_oa / h->surf_dr);
    off[0] = 0;
    for (int c = 0; c < AMC_NUM_CASES; c++) {
        int64_t n = 0;
        if (kind == AMC_KIND_CUBE) {
            const int a = c >> 1;
            if (c < 6) n = nc[a == 0 ? 1 : 0] * nc[a == 2 ? 1 : 2];
        } else if (kind == AMC_KIND_PORE && c == AMC_CASE_6C) {
            n = 0;
        } else {
            const bool side = c == AMC_CASE_1 || c == AMC_CASE_4 || c == AMC_CASE_6H || c == AMC_CASE_6C;
            n = side ? nc[2] : nann;
        }
        off[c + 1] = off[c] + n;
    }
    if (rsq) {
        rsq->resize((size_t)nann + 1);
        for (int64_t k = 0; k <= nann; k++) (*rsq)[k] = ((double)k * h->surf_dr) * ((double)k * h->surf_dr);
    }
}

extern "C" int amc_surface_layout(amc_handle *h, int64_t offsets[AMC_NUM_CASES + 1])
{
    if (!h || !offsets) return AMC_E_INVALID;
    surf_layout(h, offsets, nullptr);
    return AMC_OK;
}

extern "C" int amc_surface_disable(amc_handle *h)
{
    if (!h) return AMC_E_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    if (h->d_surf) CK(cudaFree(h->d_surf));
    if (h->d_surf_rsq) CK(cudaFree(h->d_surf_rsq));
    h->d_surf = nullptr; h->d_surf_rsq = nullptr;
    h->sp = SurfP{};
    h->surf_steps = 0;
    return AMC_OK;
}

extern "C" int amc_surface_enable(amc_handle *h)
{
    if (!h) return AMC_E_INVALID;
    int rc = amc_surface_disable(h);
    if (rc != AMC_OK) return rc;
    P &p = h->p;
    int64_t off[AMC_NUM_CASES + 1];
    std::vector<double> rsq;
    surf_layout(h, off, &rsq);
    if (off[AMC_NUM_CASES] > 0x7fffffffLL / AMC_SURF_WORDS) return h->fail(AMC_E_INVALID, "too many surface elements");
    const size_t words = (size_t)off[AMC_NUM_CASES] * AMC_SURF_WORDS + AMC_NUM_CASES;
    cudaError_t e = cudaMalloc(&h->d_surf, words * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMalloc(&h->d_surf_rsq, rsq.size() * sizeof(double));
    if (e != cudaSuccess) {
        amc_surface_disable(h);
        return h->fail(AMC_E_NOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e));
    }
    CK(cudaMemsetAsync(h->d_surf, 0, words * sizeof(unsigned long long), h->stream));
    CK(cudaMemcpyAsync(h->d_surf_rsq, rsq.data(), rsq.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    SurfP &sp = h->sp;
    for (int c = 0; c <= AMC_NUM_CASES; c++) sp.off[c] = (int32_t)off[c];
    sp.rsq = h->d_surf_rsq;
    sp.nann = (int32_t)(rsq.size() - 1);
    sp.inv_dr = 1.0 / h->surf_dr;
    if (p.slab) { sp.zedge = p.gz_edge; sp.ncz = p.gncz; sp.ze0 = p.g_e0z; sp.zinv = p.g_inv_dz; }
    else { sp.zedge = p.edge[2]; sp.ncz = p.nc[2]; sp.ze0 = p.e0[2]; sp.zinv = p.inv_d[2]; }
    sp.acc = h->d_surf;
    h->surf_steps = 0;
    return AMC_OK;
}

static size_t surf_acc_words(const amc_handle *h) { return (size_t)h->sp.off[AMC_NUM_CASES] * AMC_SURF_WORDS; }

extern "C" int amc_surface_get_raw(amc_handle *h, uint64_t *acc, uint64_t *n_steps, uint64_t outside[AMC_NUM_CASES])
{
    if (!h) return AMC_E_INVALID;
    if (!h->d_surf) return h->fail(AMC_E_STATE, "surface recording is not enabled (amc_surface_enable)");
    CK(cudaSetDevice(h->device));
    const size_t nw = surf_acc_words(h);
    if (acc) CK(cudaMemcpyAsync(acc, h->d_surf, nw * sizeof(uint64_t), cudaMemcpyDeviceToHost, h->stream));
    if (outside) CK(cudaMemcpyAsync(outside, h->d_surf + nw, AMC_NUM_CASES * sizeof(uint64_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (n_steps) *n_steps = h->surf_steps;
    return AMC_OK;
}

extern "C" int amc_surface_set_raw(amc_handle *h, const uint64_t *acc, uint64_t n_steps, const uint64_t outside[AMC_NUM_CASES])
{
    if (!h || !acc || !outside) return AMC_E_INVALID;
    if (!h->d_surf) return h->fail(AMC_E_STATE, "surface recording is not enabled (amc_surface_enable)");
    CK(cudaSetDevice(h->device));
    const size_t nw = surf_acc_words(h);
    CK(cudaMemcpyAsync(h->d_surf, acc, nw * sizeof(uint64_t), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_surf + nw, outside, AMC_NUM_CASES * sizeof(uint64_t), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->surf_steps = n_steps;
    return AMC_OK;
}

// ---- plane flux recording ------------------------------------------------------------------------
static size_t flux_words(const amc_handle *h)
{
    return (size_t)(h->cfg.nc[2] + 1) * AMC_FLUX_WORDS;
}

static FluxArgs flux_args(const amc_handle *h)
{
    return FluxArgs{h->d_flux, h->d_flux_snap, h->d_flux + flux_words(h)};
}

// one record point on h->stream; launches (nullable) counts the kernel launch
static int launch_flux(amc_handle *h, int64_t *launches)
{
    if (h->n) {
        k_flux<<<grid_for(h->n, FLUX_THREADS), FLUX_THREADS, 0, h->stream>>>(h->p, flux_args(h));
        if (launches) *launches += 1;
    }
    CK(cudaGetLastError());
    h->flux_steps++;
    return AMC_OK;
}

// the snapshot of the current state; AMC_E_INVALID unless the ids are 0 .. n-1 (the snapshot is indexed by id)
static int flux_snapshot(amc_handle *h)
{
    const FluxArgs fa = flux_args(h);
    CK(cudaMemsetAsync(fa.bad, 0, sizeof(unsigned long long), h->stream));
    CK(cudaMemsetAsync(fa.snap, 0xff, h->n * sizeof(int32_t), h->stream));
    if (h->n) k_flux_snap<<<grid_for(h->n, FLUX_THREADS), FLUX_THREADS, 0, h->stream>>>(h->p, fa);
    CK(cudaGetLastError());
    unsigned long long bad = 0;
    CK(cudaMemcpyAsync(&bad, fa.bad, sizeof(bad), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (bad) return h->fail(AMC_E_INVALID, "flux recording indexes its snapshot by particle id: the ids must be 0 .. n-1");
    return AMC_OK;
}

// after a call that replaced the state: a new snapshot while recording is on.  A state the snapshot cannot index
// ends the recording, so that no later record point reads outside it.
static int flux_retake(amc_handle *h)
{
    if (!h->d_flux) return AMC_OK;
    const int rc = flux_snapshot(h);
    if (rc != AMC_OK) {
        const std::string msg = h->error;
        amc_flux_disable(h);
        h->error = msg + " (flux recording disabled)";
    }
    return rc;
}

extern "C" int amc_flux_enable(amc_handle *h)
{
    if (!h) return AMC_E_INVALID;
    if (h->slab) return h->fail(AMC_E_STATE, "flux recording needs a single-domain handle (a migrant between slab ranks would have to carry its plane count)");
    int rc = amc_flux_disable(h);
    if (rc != AMC_OK) return rc;
    cudaError_t e = cudaMalloc(&h->d_flux, (flux_words(h) + 1) * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMalloc(&h->d_flux_snap, (size_t)h->cap * sizeof(int32_t));
    if (e != cudaSuccess) {
        amc_flux_disable(h);
        return h->fail(AMC_E_NOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e));
    }
    CK(cudaMemsetAsync(h->d_flux, 0, flux_words(h) * sizeof(unsigned long long), h->stream));
    if ((rc = flux_snapshot(h)) != AMC_OK) {
        const std::string msg = h->error;
        amc_flux_disable(h);
        h->error = msg;
    }
    return rc;
}

extern "C" int amc_flux_disable(amc_handle *h)
{
    if (!h) return AMC_E_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    if (h->d_flux) CK(cudaFree(h->d_flux));
    if (h->d_flux_snap) CK(cudaFree(h->d_flux_snap));
    h->d_flux = nullptr; h->d_flux_snap = nullptr;
    h->flux_steps = 0;
    return AMC_OK;
}

extern "C" int amc_flux_now(amc_handle *h)
{
    if (!h) return AMC_E_INVALID;
    if (!h->d_flux) return h->fail(AMC_E_STATE, "flux recording is not enabled (amc_flux_enable)");
    CK(cudaSetDevice(h->device));
    int rc = launch_flux(h, nullptr);
    if (rc != AMC_OK) return rc;
    CK(cudaStreamSynchronize(h->stream));
    return AMC_OK;
}

extern "C" int amc_flux_layout(amc_handle *h, int32_t *n_planes)
{
    if (!h) return AMC_E_INVALID;
    if (!h->d_flux) return h->fail(AMC_E_STATE, "flux recording is not enabled (amc_flux_enable)");
    if (n_planes) *n_planes = h->cfg.nc[2] + 1;
    return AMC_OK;
}

extern "C" int amc_flux_get_raw(amc_handle *h, uint64_t *acc, uint64_t *n_steps)
{
    if (!h) return AMC_E_INVALID;
    if (!h->d_flux) return h->fail(AMC_E_STATE, "flux recording is not enabled (amc_flux_enable)");
    CK(cudaSetDevice(h->device));
    if (acc) CK(cudaMemcpyAsync(acc, h->d_flux, flux_words(h) * sizeof(uint64_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (n_steps) *n_steps = h->flux_steps;
    return AMC_OK;
}

extern "C" int amc_flux_set_raw(amc_handle *h, const uint64_t *acc, uint64_t n_steps)
{
    if (!h || !acc) return AMC_E_INVALID;
    if (!h->d_flux) return h->fail(AMC_E_STATE, "flux recording is not enabled (amc_flux_enable)");
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync(h->d_flux, acc, flux_words(h) * sizeof(uint64_t), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->flux_steps = n_steps;
    return AMC_OK;
}

extern "C" int amc_step(amc_handle *h, int32_t n_steps, amc_step_stats *stats)
{
    if (!h) return AMC_E_INVALID;
    if (n_steps < 0) return h->fail(AMC_E_INVALID, "n_steps < 0");
    if (h->slab) return h->fail(AMC_E_STATE, "slab handles are stepped through the amc_slab_* entry points");
    if (h->cfg.kind == AMC_KIND_TEMP && h->cfg.rng_mode == AMC_RNG_HOST)
        return h->fail(AMC_E_STATE, "host-RNG handles are stepped through the phase-level entry points");
    CK(cudaSetDevice(h->device));
    P &p = h->p;
    const bool sweep = p.pp_mode == AMC_PP_SWEEP;
    const bool has_recap = p.kind != AMC_KIND_CUBE;
    memset(h->last_ms, 0, sizeof(h->last_ms));
    h->last_detect_ms = 0;
    h->last_scatter_ms = 0;
    h->last_launches = 0;
    sample_reset_timing(h);
    const bool flux = h->d_flux != nullptr; // every step is a record point
    int done = 0;
    if (sweep && h->n) { // the sweep kernel addresses particles by id: keep slot == id
        int rc = unsort(h);
        if (rc != AMC_OK) return rc;
    }
    while (done < n_steps) {
        int chunk = std::min(n_steps - done, h->stats_cap);
        int rc;
        if ((rc = ensure_events(h, h->events, (size_t)chunk * 4 + 1)) != AMC_OK) return rc;
        if ((rc = ensure_events(h, h->det_events, (size_t)chunk * 2)) != AMC_OK) return rc;
        if ((rc = ensure_events(h, h->sc_events, (size_t)chunk * 2)) != AMC_OK) return rc;
        CK(cudaMemsetAsync(h->d_stats, 0, chunk * sizeof(StatsDev), h->stream));
        CK(cudaEventRecord(h->events[0], h->stream));
        bool closed_prev = true; // the step before this one ended with its own recapture launch
        for (int s = 0; s < chunk; s++) {
            p.stats = h->d_stats + s;
            p.step = h->step_index++;
            if (h->sp.acc) h->surf_steps++;
            // a sampled or recorded step is closed like the last step of a chunk, so the sample and the flux
            // recording see the state at its end
            const bool sample = sample_due(h, p.step);
            if (h->n > 0) {
                // the recapture that closes step s-1's pair pass rides along in step s's advect kernel
                const bool fuse_prev = has_recap && !closed_prev;
                p.stats_prev = fuse_prev ? h->d_stats + (s - 1) : h->d_stats + s;
                int phase = PH_DRIFT | PH_WALLS | (has_recap ? PH_RECAP : 0) | (fuse_prev ? PH_RECAP_POST : 0);
                if (sweep) {
                    if (h->sp.acc) k_advect_surf<<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(p, phase, h->sp);
                    else k_advect<<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(p, phase);
                    h->last_launches += 1;
                    CK(cudaEventRecord(h->events[4 * s + 1], h->stream));
                } else { // fused: keys of the post-step positions, then the step itself on the way to the sorted slot
                    CK(cudaMemsetAsync(p.band_count, 0, (h->n_buckets + 2) * sizeof(int32_t), h->stream));
                    CK(cudaMemsetAsync(p.rest_count, 0, (h->n_buckets + 1) * sizeof(int32_t), h->stream));
                    k_keys<false><<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(p, phase);
                    CK(cudaEventRecord(h->events[4 * s + 1], h->stream));
                    int m = h->n_buckets, ntiles = (m + SCAN_TILE - 1) / SCAN_TILE;
                    k_scan_tiles<<<ntiles, SCAN_THREADS, 0, h->stream>>>(p.band_count, p.rest_count, p.cell_start, h->d_tile_sums, m);
                    CK(launch_pdl(k_scan_sums, dim3(1), dim3(SCAN_THREADS), h->stream, h->d_tile_sums, ntiles));
                    CK(launch_pdl(k_scan_add, dim3(ntiles), dim3(SCAN_THREADS), h->stream, p.cell_start, (const int32_t *)h->d_tile_sums, m, (int32_t)h->n));
                    // the bookkeeping of the pair pass needs the scan, not the scattered particles: it runs beside the scatter
                    CK(cudaEventRecord(h->ev_fork, h->stream));
                    CK(cudaStreamWaitEvent(h->aux, h->ev_fork, 0));
                    if ((rc = prepare_pairs(h, h->aux)) != AMC_OK) return rc;
                    CK(cudaEventRecord(h->ev_join, h->aux));
                    CK(cudaEventRecord(h->sc_events[2 * s], h->stream));
                    if (h->sp.acc) k_scatter_advect_surf<false><<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(p, phase, h->sp);
                    else k_scatter_advect<false><<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(p, phase);
                    CK(cudaEventRecord(h->sc_events[2 * s + 1], h->stream));
                    CK(cudaGetLastError());
                    CK(cudaStreamWaitEvent(h->stream, h->ev_join, 0));
                    std::swap(p.a, p.b);
                    h->last_launches += 5;
                }
                CK(cudaEventRecord(h->events[4 * s + 2], h->stream));
                h->det_slot = sweep ? -1 : s;
                rc = run_pairs(h, &h->last_launches, !sweep);
                h->det_slot = -1;
                if (rc != AMC_OK) return rc;
                CK(cudaEventRecord(h->events[4 * s + 3], h->stream));
                closed_prev = s == chunk - 1 || sample || flux;
                if (has_recap && closed_prev) { // last step of the call (or a sampled / recorded step): close it now
                    if (sweep) k_recapture_post<<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(p);
                    else k_recapture_list<<<148, ADVECT_THREADS, 0, h->stream>>>(p);
                    h->last_launches += 1;
                }
                if (sample && (rc = launch_sample(h, h->n, &h->last_launches)) != AMC_OK) return rc;
                if (flux && (rc = launch_flux(h, &h->last_launches)) != AMC_OK) return rc;
                CK(cudaEventRecord(h->events[4 * s + 4], h->stream));
            } else {
                if (sample && (rc = launch_sample(h, 0, nullptr)) != AMC_OK) return rc;
                if (flux && (rc = launch_flux(h, nullptr)) != AMC_OK) return rc;
            }
        }
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(h->h_stats, h->d_stats, chunk * sizeof(StatsDev), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        if ((rc = sample_collect_timing(h)) != AMC_OK) return rc;
        if (h->n > 0)
            for (int s = 0; s < chunk; s++) {
                float ms;
                for (int k = 0; k < 4; k++) {
                    CK(cudaEventElapsedTime(&ms, h->events[4 * s + k], h->events[4 * s + k + 1]));
                    h->last_ms[k] += ms;
                }
                if (!sweep) {
                    CK(cudaEventElapsedTime(&ms, h->det_events[2 * s], h->det_events[2 * s + 1]));
                    h->last_detect_ms += ms;
                    CK(cudaEventElapsedTime(&ms, h->sc_events[2 * s], h->sc_events[2 * s + 1]));
                    h->last_scatter_ms += ms;
                }
            }
        for (int s = 0; s < chunk; s++) {
            rc = check_overflow(h, h->h_stats[s]);
            if (rc != AMC_OK) return rc;
            if (stats) stats_to_host(h, h->h_stats[s], stats + done + s);
        }
        done += chunk;
    }
    h->last_ms[4] = h->last_ms[0] + h->last_ms[1] + h->last_ms[2] + h->last_ms[3];
    p.stats = h->d_stats;
    return AMC_OK;
}

// ---- phase-level entry points -------------------------------------------------------------------
static int phase_begin(amc_handle *h)
{
    CK(cudaSetDevice(h->device));
    h->p.stats = h->d_stats;
    CK(cudaMemsetAsync(h->d_stats, 0, sizeof(StatsDev), h->stream));
    return AMC_OK;
}
static int phase_end(amc_handle *h, amc_step_stats *stats)
{
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h->h_stats, h->d_stats, sizeof(StatsDev), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    int rc = check_overflow(h, h->h_stats[0]);
    if (rc != AMC_OK) return rc;
    if (stats) stats_to_host(h, h->h_stats[0], stats);
    return AMC_OK;
}

extern "C" int amc_drift(amc_handle *h)
{
    if (!h) return AMC_E_INVALID;
    int rc = phase_begin(h);
    if (rc != AMC_OK) return rc;
    if ((rc = ensure_prior(h)) != AMC_OK) return rc;
    if (h->n) k_advect<<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(h->p, PH_DRIFT | PH_SAVE_PRIOR);
    if (h->p.wall_bits) CK(cudaMemsetAsync(h->p.wall_bits, 0, h->cap * sizeof(uint16_t), h->stream));
    return phase_end(h, nullptr);
}

extern "C" int amc_walls(amc_handle *h, amc_step_stats *stats)
{
    if (!h) return AMC_E_INVALID;
    if (h->cfg.kind == AMC_KIND_TEMP && h->cfg.rng_mode == AMC_RNG_HOST)
        return h->fail(AMC_E_STATE, "host-RNG handles apply walls case by case (amc_wall_case / amc_wall_hits_pending)");
    int rc = phase_begin(h);
    if (rc != AMC_OK) return rc;
    if ((rc = ensure_prior(h)) != AMC_OK) return rc;
    h->p.step = h->step_index++;
    if (h->sp.acc) h->surf_steps++;
    if (h->n) {
        if (h->sp.acc) k_advect_surf<<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(h->p, PH_WALLS | PH_LOAD_PRIOR, h->sp);
        else k_advect<<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(h->p, PH_WALLS | PH_LOAD_PRIOR);
    }
    return phase_end(h, stats);
}

extern "C" int amc_recapture(amc_handle *h, int64_t *count, int64_t *count_after)
{
    if (!h) return AMC_E_INVALID;
    int rc = phase_begin(h);
    if (rc != AMC_OK) return rc;
    if (h->n && h->cfg.kind != AMC_KIND_CUBE)
        k_recapture_post<<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(h->p);
    amc_step_stats st;
    rc = phase_end(h, &st);
    if (count) *count = st.oob_after_pp;
    if (count_after) *count_after = st.oob_after_pp_recapture;
    return rc;
}

extern "C" int amc_pairs(amc_handle *h, amc_step_stats *stats)
{
    if (!h) return AMC_E_INVALID;
    if (h->slab) return h->fail(AMC_E_STATE, "slab handles are stepped through the amc_slab_* entry points");
    int rc = phase_begin(h);
    if (rc != AMC_OK) return rc;
    P &p = h->p;
    if (h->n) {
        if (p.pp_mode == AMC_PP_SWEEP) {
            if ((rc = unsort(h)) != AMC_OK) return rc;
        } else {
            CK(cudaMemsetAsync(p.band_count, 0, (h->n_buckets + 2) * sizeof(int32_t), h->stream));
            CK(cudaMemsetAsync(p.rest_count, 0, (h->n_buckets + 1) * sizeof(int32_t), h->stream));
            k_advect<<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(p, PH_KEYS);
            if ((rc = sort_scatter(h, nullptr)) != AMC_OK) return rc;
        }
        if ((rc = run_pairs(h, nullptr)) != AMC_OK) return rc;
    }
    return phase_end(h, stats);
}

// Overlap-free seeding (SURVEY 8f rank 4): the reference's random initial state leaves ~0.2 % of the particles
// overlapping a neighbour (1,051 pairs at 557,649 particles, Open_Air_Pore_MC.py:106-158), which the first timesteps
// resolve as a burst of unphysical collisions.  Each round sorts the particles into cells, runs the detection pass in
// seed mode (exact overlap test on the pairs its filter finds; the particle with the higher index of every
// overlapping pair is marked) and gives the marked particles a fresh position from the same generator.
extern "C" int amc_seed_relax(amc_handle *h, int32_t max_rounds, int64_t *n_redrawn, int64_t *n_left)
{
    if (!h) return AMC_E_INVALID;
    if (!h->have_init_spec) return h->fail(AMC_E_STATE, "amc_seed_relax follows amc_init_synthetic on a single-domain handle");
    if (h->slab || h->cfg.pp_mode != AMC_PP_GROUPS) return h->fail(AMC_E_STATE, "amc_seed_relax needs a single-domain handle with the colour-group schedule");
    P &p = h->p;
    int64_t total = 0, left = 0;
    for (int round = 0; round <= max_rounds; round++) { /* the last round only counts */
        int rc = phase_begin(h);
        if (rc != AMC_OK) return rc;
        if (h->n == 0) break;
        CK(cudaMemsetAsync(p.band_count, 0, (h->n_buckets + 2) * sizeof(int32_t), h->stream));
        CK(cudaMemsetAsync(p.rest_count, 0, (h->n_buckets + 1) * sizeof(int32_t), h->stream));
        k_advect<<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(p, PH_KEYS);
        if ((rc = sort_scatter(h, nullptr)) != AMC_OK) return rc;
        if ((rc = prepare_pairs(h, h->stream)) != AMC_OK) return rc;
        CK(cudaMemsetAsync(p.rank, 0, h->n * sizeof(int32_t), h->stream));
        k_detect_tma<true><<<h->det_grid_tma, DET_THREADS, 0, h->stream>>>(p);
        if (round < max_rounds) k_seed_redraw<<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(p, h->init_spec, (uint32_t)(round + 1));
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(h->h_stats, h->d_stats, sizeof(StatsDev), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        left = (int64_t)h->h_stats[0].pp;
        if (left == 0 || round == max_rounds) break;
        total += left;
    }
    // worklists built by the seed-mode passes are reset by the next pair pass (prepare_pairs)
    if (n_redrawn) *n_redrawn = total;
    if (n_left) *n_left = left;
    return flux_retake(h);
}

extern "C" int amc_wall_operator(amc_handle *h, int32_t op, const uint8_t *mask, double param, int64_t *n_hits, int64_t *errors)
{
    if (!h) return AMC_E_INVALID;
    if (op < AMC_OP_PLANE_MFP || op > AMC_OP_SIDE_SPECULAR) return h->fail(AMC_E_INVALID, "unknown wall operator");
    if (h->n && !mask) return h->fail(AMC_E_INVALID, "null mask");
    if (h->slab) return h->fail(AMC_E_STATE, "operator-level entry points work on single-domain handles");
    int rc = phase_begin(h);
    if (rc != AMC_OK) return rc;
    if (h->n) {
        uint8_t *dm = reinterpret_cast<uint8_t *>(h->p.key); /* scratch until the next sort: n bytes of the n-int key array */
        CK(cudaMemcpyAsync(dm, mask, h->n, cudaMemcpyHostToDevice, h->stream));
        k_wall_operator<<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(h->p, op, dm, param);
    }
    amc_step_stats st;
    rc = phase_end(h, &st);
    if (n_hits) *n_hits = st.wall_hits[0];
    if (errors) *errors = st.errors;
    return rc;
}

// ---- host-RNG parity hooks ----------------------------------------------------------------------
extern "C" int amc_wall_case(amc_handle *h, int32_t c, int64_t *n_hits)
{
    if (!h) return AMC_E_INVALID;
    if (h->cfg.kind != AMC_KIND_TEMP) return h->fail(AMC_E_STATE, "amc_wall_case: AMC_KIND_TEMP only");
    if (c < AMC_CASE_1 || c > AMC_CASE_2B) return h->fail(AMC_E_INVALID, "amc_wall_case handles the specular cases 1, 2a, 2b");
    if (!h->have_prior) return h->fail(AMC_E_STATE, "call amc_drift first");
    int rc = phase_begin(h);
    if (rc != AMC_OK) return rc;
    if (h->sp.acc && c == AMC_CASE_1) h->surf_steps++; /* the first case of a host-RNG wall phase */
    if (h->n) k_case_specular<<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(h->p, c, h->sp);
    amc_step_stats st;
    rc = phase_end(h, &st);
    if (n_hits) *n_hits = st.wall_hits[c];
    return rc;
}

extern "C" int amc_wall_hits_pending(amc_handle *h, int32_t c, int64_t cap, int64_t *n_hits, int64_t *idx,
                                     double *normal3, double *col_z)
{
    if (!h) return AMC_E_INVALID;
    if (h->cfg.kind != AMC_KIND_TEMP || h->cfg.rng_mode != AMC_RNG_HOST) return h->fail(AMC_E_STATE, "not a host-RNG Temp handle");
    if (c < AMC_CASE_3C || c >= AMC_NUM_CASES) return h->fail(AMC_E_INVALID, "energized cases only");
    if (!h->have_prior) return h->fail(AMC_E_STATE, "call amc_drift first");
    int rc = phase_begin(h);
    if (rc != AMC_OK) return rc;
    CK(cudaMemsetAsync(h->d_pend_count, 0, sizeof(int32_t), h->stream));
    if (h->n)
        k_case_detect<<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(h->p, c, h->d_pend_count, h->pend_cap, h->d_pend_slot,
                                                                                      h->d_pend_id, h->d_pend_nrm, h->d_pend_colz);
    CK(cudaGetLastError());
    int32_t cnt = 0;
    CK(cudaMemcpyAsync(&cnt, h->d_pend_count, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (cnt > h->pend_cap) return h->fail(AMC_E_CAPACITY, "pending-hit list overflow");
    std::vector<int32_t> slot(cnt), id(cnt);
    std::vector<double> nrm((size_t)cnt * 3), colz(cnt);
    if (cnt) {
        CK(cudaMemcpy(slot.data(), h->d_pend_slot, cnt * sizeof(int32_t), cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(id.data(), h->d_pend_id, cnt * sizeof(int32_t), cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(nrm.data(), h->d_pend_nrm, (size_t)cnt * 3 * sizeof(double), cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(colz.data(), h->d_pend_colz, cnt * sizeof(double), cudaMemcpyDeviceToHost));
    }
    std::vector<int32_t> order(cnt);
    for (int k = 0; k < cnt; k++) order[k] = k;
    std::sort(order.begin(), order.end(), [&](int a, int b) { return id[a] < id[b]; }); // ascending particle index
    h->pend_slot.assign(cnt, 0);
    h->pend_id.assign(cnt, 0);
    h->pend_case = c;
    if (n_hits) *n_hits = cnt;
    if (cnt > cap) return h->fail(AMC_E_CAPACITY, "caller buffers too small for the pending hits");
    for (int k = 0; k < cnt; k++) {
        int o = order[k];
        h->pend_slot[k] = slot[o];
        h->pend_id[k] = id[o];
        if (idx) idx[k] = id[o];
        if (normal3) { normal3[3 * k] = nrm[3 * o]; normal3[3 * k + 1] = nrm[3 * o + 1]; normal3[3 * k + 2] = nrm[3 * o + 2]; }
        if (col_z) col_z[k] = colz[o];
    }
    return AMC_OK;
}

extern "C" int amc_wall_apply_directions(amc_handle *h, int32_t c, int64_t n_hits, const int64_t *idx, const double *dir3,
                                         const double *surf_e, double *dpz, double *de, int64_t *errors)
{
    if (!h) return AMC_E_INVALID;
    if (h->pend_case != c || (int64_t)h->pend_id.size() != n_hits) return h->fail(AMC_E_STATE, "apply does not match the last amc_wall_hits_pending call");
    for (int64_t k = 0; k < n_hits; k++)
        if (idx && idx[k] != h->pend_id[k]) return h->fail(AMC_E_STATE, "hit indices differ from the pending list");
    if (c == AMC_CASE_4 && n_hits && !surf_e) return h->fail(AMC_E_INVALID, "case 4 needs per-hit surface energies");
    int rc = phase_begin(h);
    if (rc != AMC_OK) return rc;
    h->pend_case = -1;
    if (n_hits) {
        CK(cudaMemcpyAsync(h->d_pend_slot, h->pend_slot.data(), n_hits * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(h->d_pend_dirs, dir3, (size_t)n_hits * 3 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        if (surf_e) CK(cudaMemcpyAsync(h->d_pend_se, surf_e, n_hits * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        k_case_apply<<<grid_for(n_hits, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(h->p, c, (int32_t)n_hits, h->d_pend_slot, h->d_pend_dirs,
                                                                                        h->d_pend_se, h->d_pend_dpz, h->d_pend_de, h->sp);
        if (dpz) CK(cudaMemcpyAsync(dpz, h->d_pend_dpz, n_hits * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        if (de) CK(cudaMemcpyAsync(de, h->d_pend_de, n_hits * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    }
    amc_step_stats st;
    rc = phase_end(h, &st);
    if (errors) *errors = st.errors;
    return rc;
}

// ---- outputs and taps ---------------------------------------------------------------------------
extern "C" int amc_get_histograms(amc_handle *h, uint64_t *counts, uint64_t *n_paths, double *sums4)
{
    if (!h) return AMC_E_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    if (counts) CK(cudaMemcpy(counts, h->p.hist, 4 * AMC_NUM_BINS * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    if (n_paths) CK(cudaMemcpy(n_paths, h->p.path_count, sizeof(uint64_t), cudaMemcpyDeviceToHost));
    if (sums4) {
        unsigned long long limbs[8];
        CK(cudaMemcpy(limbs, h->p.path_sums, sizeof(limbs), cudaMemcpyDeviceToHost));
        for (int k = 0; k < 4; k++)
            sums4[k] = ldexp((double)(long long)limbs[2 * k], -49) + ldexp((double)(long long)limbs[2 * k + 1], -89);
    }
    return AMC_OK;
}

extern "C" int amc_get_pair_list(amc_handle *h, int64_t cap, int64_t *n, int64_t *hi, int64_t *lo, int32_t *group, int32_t *cell)
{
    if (!h) return AMC_E_INVALID;
    if (!h->p.pair_count) return h->fail(AMC_E_STATE, "AMC_TAP_PAIRS not enabled");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    unsigned long long cnt = 0;
    CK(cudaMemcpy(&cnt, h->p.pair_count, sizeof(cnt), cudaMemcpyDeviceToHost));
    if (n) *n = (int64_t)cnt;
    if ((int64_t)cnt > h->p.pair_cap) return h->fail(AMC_E_CAPACITY, "pair tap overflow (raise pair_capacity)");
    if ((int64_t)cnt > cap) return h->fail(AMC_E_CAPACITY, "caller buffers too small for the pair list");
    if (cnt) {
        if (hi) CK(cudaMemcpy(hi, h->p.pair_hi, cnt * sizeof(int64_t), cudaMemcpyDeviceToHost));
        if (lo) CK(cudaMemcpy(lo, h->p.pair_lo, cnt * sizeof(int64_t), cudaMemcpyDeviceToHost));
        if (group) CK(cudaMemcpy(group, h->p.pair_group, cnt * sizeof(int32_t), cudaMemcpyDeviceToHost));
        if (cell) CK(cudaMemcpy(cell, h->p.pair_cell, cnt * sizeof(int32_t), cudaMemcpyDeviceToHost));
    }
    return AMC_OK;
}

extern "C" int amc_get_wall_bits(amc_handle *h, uint16_t *bits)
{
    if (!h) return AMC_E_INVALID;
    if (!h->p.wall_bits) return h->fail(AMC_E_STATE, "AMC_TAP_WALL_BITS not enabled");
    if (h->slab) return h->fail(AMC_E_STATE, "the wall-bits tap is indexed by particle id and not available on slab handles");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(bits, h->p.wall_bits, h->n * sizeof(uint16_t), cudaMemcpyDeviceToHost));
    return AMC_OK;
}

extern "C" int amc_get_completed_paths(amc_handle *h, int64_t cap, int64_t *n, double *total, double *cx, double *cy, double *cz)
{
    if (!h) return AMC_E_INVALID;
    if (!h->p.tap_path_count) return h->fail(AMC_E_STATE, "AMC_TAP_PATHS not enabled");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    unsigned long long cnt = 0;
    CK(cudaMemcpy(&cnt, h->p.tap_path_count, sizeof(cnt), cudaMemcpyDeviceToHost));
    if (n) *n = (int64_t)cnt;
    if ((int64_t)cnt > h->p.path_cap) return h->fail(AMC_E_CAPACITY, "path tap overflow (raise path_capacity)");
    if ((int64_t)cnt > cap) return h->fail(AMC_E_CAPACITY, "caller buffers too small for the path list");
    double *dst[4] = {total, cx, cy, cz};
    for (int k = 0; k < 4; k++)
        if (dst[k] && cnt) CK(cudaMemcpy(dst[k], h->p.tap_paths[k], cnt * sizeof(double), cudaMemcpyDeviceToHost));
    return AMC_OK;
}

extern "C" int amc_clear_taps(amc_handle *h)
{
    if (!h) return AMC_E_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    if (h->p.pair_count) CK(cudaMemset(h->p.pair_count, 0, sizeof(unsigned long long)));
    if (h->p.tap_path_count) CK(cudaMemset(h->p.tap_path_count, 0, sizeof(unsigned long long)));
    if (h->p.wall_bits) CK(cudaMemset(h->p.wall_bits, 0, h->cap * sizeof(uint16_t)));
    return AMC_OK;
}

extern "C" int amc_get_outputs_raw(amc_handle *h, uint64_t *counts, uint64_t *n_paths, uint64_t *limbs8)
{
    if (!h) return AMC_E_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    if (counts) CK(cudaMemcpy(counts, h->p.hist, 4 * AMC_NUM_BINS * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    if (n_paths) CK(cudaMemcpy(n_paths, h->p.path_count, sizeof(uint64_t), cudaMemcpyDeviceToHost));
    if (limbs8) CK(cudaMemcpy(limbs8, h->p.path_sums, 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return AMC_OK;
}

extern "C" int amc_set_outputs_raw(amc_handle *h, const uint64_t *counts, uint64_t n_paths, const uint64_t *limbs8)
{
    if (!h || !counts || !limbs8) return AMC_E_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(h->p.hist, counts, 4 * AMC_NUM_BINS * sizeof(uint64_t), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->p.path_count, &n_paths, sizeof(uint64_t), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->p.path_sums, limbs8, 8 * sizeof(uint64_t), cudaMemcpyHostToDevice));
    return AMC_OK;
}

extern "C" int64_t amc_get_step_index(const amc_handle *h) { return h ? h->step_index : -1; }

extern "C" int amc_set_step_index(amc_handle *h, int64_t step)
{
    if (!h) return AMC_E_INVALID;
    h->step_index = step;
    CK(cudaSetDevice(h->device));
    CK(cudaMemsetAsync(h->p.touch_mark, 0, h->cap * sizeof(int32_t), h->stream)); /* the per-slot step tags of touch_slot */
    return AMC_OK;
}

extern "C" int amc_last_timing(amc_handle *h, double ms[5], int64_t *launches)
{
    if (!h) return AMC_E_INVALID;
    if (ms) memcpy(ms, h->last_ms, sizeof(h->last_ms));
    if (launches) *launches = h->last_launches;
    return AMC_OK;
}

extern "C" int amc_last_detect_ms(amc_handle *h, double *ms)
{
    if (!h || !ms) return AMC_E_INVALID;
    *ms = h->last_detect_ms;
    return AMC_OK;
}

extern "C" int amc_last_scatter_ms(amc_handle *h, double *ms)
{
    if (!h || !ms) return AMC_E_INVALID;
    *ms = h->last_scatter_ms;
    return AMC_OK;
}

// ---- slab decomposition (multi-GPU) ---------------------------------------------------------------
extern "C" int amc_set_stream(amc_handle *h, void *cuda_stream)
{
    if (!h) return AMC_E_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    if (h->own_stream) CK(cudaStreamDestroy(h->stream));
    h->stream = (cudaStream_t)cuda_stream;
    h->own_stream = false;
    return AMC_OK;
}

extern "C" int amc_set_ids(amc_handle *h, const int64_t *ids)
{
    if (!h || !ids) return AMC_E_INVALID;
    if (h->d_flux) return h->fail(AMC_E_STATE, "flux recording indexes its snapshot by particle id: disable it before amc_set_ids");
    CK(cudaSetDevice(h->device));
    std::vector<int32_t> v((size_t)h->n);
    for (int64_t i = 0; i < h->n; i++) {
        if (ids[i] < 0 || ids[i] > 0x7fffffffLL) return h->fail(AMC_E_INVALID, "particle id out of range");
        v[(size_t)i] = (int32_t)ids[i];
    }
    int32_t *stage = h->p.key; /* scratch until the next sort */
    CK(cudaMemcpyAsync(stage, v.data(), h->n * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    if (h->n) k_set_ids<<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(h->p, stage);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(h->stream));
    return AMC_OK;
}

extern "C" int amc_slab_enable(amc_handle *h, const amc_slab_config *c)
{
    if (!h || !c) return AMC_E_INVALID;
    if (h->cfg.pp_mode != AMC_PP_GROUPS) return h->fail(AMC_E_INVALID, "slabs need the colour-group schedule");
    if (c->nranks < 1 || c->rank < 0 || c->rank >= c->nranks || !c->cuts || !c->gz_edge || !c->gz_lo) return h->fail(AMC_E_INVALID, "bad slab config");
    if (c->cuts[c->rank + 1] - c->cuts[c->rank] != h->cfg.nc[2]) return h->fail(AMC_E_INVALID, "handle z grid does not match its slab");
    if (h->p.wall_bits) return h->fail(AMC_E_INVALID, "AMC_TAP_WALL_BITS is indexed by particle id (global on a slab handle): not available with slabs");
    if (h->d_sample) return h->fail(AMC_E_STATE, "enable sampling after amc_slab_enable (a slab handle samples the global grid)");
    if (h->d_surf) return h->fail(AMC_E_STATE, "enable surface recording after amc_slab_enable (a slab handle bins on the global grid)");
    if (h->d_flux) return h->fail(AMC_E_STATE, "flux recording needs a single-domain handle: disable it first (amc_flux_disable)");
    CK(cudaSetDevice(h->device));
    P &p = h->p;
    p.slab = 1; p.srank = c->rank; p.nranks = c->nranks; p.zoff = c->cuts[c->rank]; p.gncz = c->gncz;
    int32_t *dc = nullptr; double *de = nullptr;
    ALLOC(dc, c->nranks + 1); ALLOC(de, c->gncz + 1);
    CK(cudaMemcpy(dc, c->cuts, (c->nranks + 1) * sizeof(int32_t), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(de, c->gz_edge, (c->gncz + 1) * sizeof(double), cudaMemcpyHostToDevice));
    p.cuts = dc; p.gz_edge = de;
    p.g_e0z = c->gz_edge[0];
    p.g_inv_dz = (double)c->gncz / (c->gz_edge[c->gncz] - c->gz_edge[0]);
    p.up_thr = c->rank + 1 < c->nranks ? c->gz_lo[c->cuts[c->rank + 1]] : INFINITY;
    p.down_thr = c->rank > 0 ? c->gz_edge[c->cuts[c->rank]] : -INFINITY;
    p.down_band = c->rank > 0 ? c->gz_lo[c->cuts[c->rank]] : INFINITY;
    p.xf_cap = std::max(c->xfer_capacity, c->xfer_capacity_far); p.bnd_cap = c->bnd_capacity;
    p.xf_cap_nb = c->xfer_capacity; p.xf_cap_far = c->xfer_capacity_far;
    {
        std::vector<int32_t> off(c->nranks), capv(c->nranks);
        int32_t o = 0;
        for (int d = 0; d < c->nranks; d++) {
            capv[d] = std::abs(d - c->rank) == 1 ? c->xfer_capacity : c->xfer_capacity_far;
            off[d] = o;
            o += capv[d] + 1;
        }
        int32_t *doff = nullptr, *dcap = nullptr;
        ALLOC(doff, c->nranks); ALLOC(dcap, c->nranks);
        CK(cudaMemcpy(doff, off.data(), c->nranks * sizeof(int32_t), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(dcap, capv.data(), c->nranks * sizeof(int32_t), cudaMemcpyHostToDevice));
        p.xf_off = doff; p.xf_capv = dcap;
        h->xf_total = o;
    }
    p.xf_send = (double *)c->xfer_send; p.xf_recv = (const double *)c->xfer_recv; /* may be null: amc_slab_p2p_setup allocates */
    p.bnd_send[0] = (double *)c->bnd_send_up; p.bnd_send[1] = (double *)c->bnd_send_down;
    p.bnd_recv[0] = (const double *)c->bnd_recv_up; p.bnd_recv[1] = (const double *)c->bnd_recv_down;
    {
        // the table only ever holds the particles next to a cut (ghost copies, particles a neighbour holds a copy of,
        // hand-overs): a few times the per-step transfer volume, not a fraction of all particles -- it is cleared every step
        int64_t want = std::min<int64_t>(std::max<int64_t>(8 * (2 * (int64_t)c->xfer_capacity + 16 * (int64_t)c->bnd_capacity), 1 << 16), 1 << 25);
        int32_t pow2 = 1 << 16;
        while (pow2 < want) pow2 <<= 1;
        p.rel_cap = pow2;
    }
    p.foreign_cap = std::max(c->bnd_capacity * 16, 4096);
    ALLOC(h->d_counters, c->nranks + 12);
    CK(cudaMemset(h->d_counters, 0, (c->nranks + 12) * sizeof(int32_t)));
    p.applied = reinterpret_cast<uint32_t *>(h->d_counters + c->nranks + 6); p.pg_done = h->d_counters + c->nranks + 8;
    p.xf_count = h->d_counters; p.n_in = h->d_counters + c->nranks; p.bnd_n = h->d_counters + c->nranks + 1;
    p.rel_count = h->d_counters + c->nranks + 3; p.n_foreign = h->d_counters + c->nranks + 4;
    ALLOC(p.bnd_dirty[0], p.bnd_cap); ALLOC(p.bnd_dirty[1], p.bnd_cap);
    ALLOC(p.xf_pack, h->xf_total);
    ALLOC(p.rel_id, p.rel_cap); ALLOC(p.rel_slot, p.rel_cap); ALLOC(p.aux, h->cap);
    ALLOC(h->d_slab_overflow, 4);
    CK(cudaMemset(h->d_slab_overflow, 0, 4 * sizeof(unsigned long long)));
    p.slab_overflow = h->d_slab_overflow;
    p.group_done = -1;
    h->slab = true;
    CK(cudaDeviceSynchronize());
    return AMC_OK;
}

static int slab_overflow_error(amc_handle *h, const unsigned long long ovf[4])
{
    if (!(ovf[0] | ovf[1] | ovf[2] | ovf[3])) return AMC_OK;
    char msg[256];
    snprintf(msg, sizeof(msg), "slab exchange overflow (the particle state of this handle is invalid from here on): %llu transfer records beyond "
             "xfer_capacity=%d or max_particles, %llu relation-table entries, %llu boundary records beyond bnd_capacity=%d, %llu foreign copies",
             ovf[0], h->p.xf_cap, ovf[1], ovf[2], h->p.bnd_cap, ovf[3]);
    return h->fail(AMC_E_CAPACITY, msg);
}

static int slab_check(amc_handle *h)
{
    if (!h) return AMC_E_INVALID;
    if (!h->slab) return h->fail(AMC_E_STATE, "amc_slab_enable has not been called");
    CK(cudaSetDevice(h->device));
    return AMC_OK;
}

extern "C" int amc_slab_advect(amc_handle *h)
{
    int rc = slab_check(h);
    if (rc != AMC_OK) return rc;
    P &p = h->p;
    p.stats = h->d_stats;
    p.step = h->step_index++;
    CK(cudaMemsetAsync(h->d_stats, 0, sizeof(StatsDev), h->stream));
    CK(cudaMemsetAsync(h->d_counters, 0, (p.nranks + 12) * sizeof(int32_t), h->stream));
    CK(cudaMemsetAsync(p.rel_id, 0xff, (size_t)p.rel_cap * sizeof(int32_t), h->stream));
    CK(cudaMemsetAsync(p.band_count, 0, (h->n_buckets + 2) * sizeof(int32_t), h->stream));
    CK(cudaMemsetAsync(p.rest_count, 0, (h->n_buckets + 1) * sizeof(int32_t), h->stream));
    h->slab_phase = PH_DRIFT | PH_WALLS | (p.kind != AMC_KIND_CUBE ? PH_RECAP : 0);
    if (h->sp.acc) h->surf_steps++;
    if (h->n) {
        k_keys<true><<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(p, h->slab_phase);
        if (p.nranks > 1) k_slab_pack<<<dim3(grid_for(p.xf_cap, ADVECT_THREADS), p.nranks), ADVECT_THREADS, 0, h->stream>>>(p, h->slab_phase);
    }
    k_xfer_headers<<<1, 32, 0, h->stream>>>(p);
    h->last_launches += (h->n ? 2 : 0) + 1; /* slab handles: cumulative (amc_last_timing) */
    CK(cudaGetLastError());
    return AMC_OK;
}

extern "C" int amc_slab_sort(amc_handle *h, int64_t *n_resident)
{
    int rc = slab_check(h);
    if (rc != AMC_OK) return rc;
    P &p = h->p;
    int64_t bound = h->n + (int64_t)h->xf_total;
    if (bound > h->cap) bound = h->cap;
    dim3 ug(grid_for(p.xf_cap, ADVECT_THREADS), p.nranks);
    k_xfer_unpack<<<ug, ADVECT_THREADS, 0, h->stream>>>(p);
    int m = h->n_buckets;
    int ntiles = (m + SCAN_TILE - 1) / SCAN_TILE;
    k_scan_tiles<<<ntiles, SCAN_THREADS, 0, h->stream>>>(p.band_count, p.rest_count, p.cell_start, h->d_tile_sums, m);
    k_scan_sums<<<1, SCAN_THREADS, 0, h->stream>>>(h->d_tile_sums, ntiles);
    k_scan_add<<<ntiles, SCAN_THREADS, 0, h->stream>>>(p.cell_start, h->d_tile_sums, m, 0);
    if (bound && h->sp.acc) k_scatter_advect_surf<true><<<grid_for(bound, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(p, h->slab_phase, h->sp);
    else if (bound) k_scatter_advect<true><<<grid_for(bound, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(p, h->slab_phase);
    h->last_launches += 4 + (bound ? 1 : 0);
    CK(cudaGetLastError());
    std::swap(p.a, p.b);
    int32_t counts[2] = {0, 0}; // resident = start of the GONE bucket; n_in for the capacity check
    CK(cudaMemcpyAsync(&counts[0], p.cell_start + (p.ncell_pad + 1), sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(&counts[1], p.n_in, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    unsigned long long ovf[4] = {0, 0, 0, 0};
    CK(cudaMemcpyAsync(ovf, h->d_slab_overflow, sizeof(ovf), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if ((rc = slab_overflow_error(h, ovf)) != AMC_OK) return rc;
    if (h->n + counts[1] > h->cap) return h->fail(AMC_E_CAPACITY, "max_particles too small for the immigrants of this step");
    h->n = counts[0];
    p.n = h->n;
    if (n_resident) *n_resident = h->n;
    return AMC_OK;
}

extern "C" int amc_slab_pairs_begin(amc_handle *h, int32_t pre_round)
{
    int rc = slab_check(h);
    if (rc != AMC_OK) return rc;
    P &p = h->p;
    p.group_done = -1;
    if ((rc = prepare_pairs(h, h->stream)) != AMC_OK) return rc;
    if ((rc = ensure_events(h, h->det_events, 2)) != AMC_OK) return rc;
    CK(cudaEventRecord(h->det_events[0], h->stream));
    if (h->n) launch_detect(h);
    CK(cudaEventRecord(h->det_events[1], h->stream));
    h->slab_det_pending = true;
    if (pre_round) k_bnd_pack<<<2, ADVECT_THREADS, 0, h->stream>>>(p); // immigrants that landed in the top band; else they travel after group 0
    h->last_launches += 2 + (h->n ? 1 : 0) + (pre_round ? 1 : 0);
    CK(cudaGetLastError());
    return AMC_OK;
}

extern "C" int amc_slab_group(amc_handle *h, int32_t g)
{
    int rc = slab_check(h);
    if (rc != AMC_OK) return rc;
    if (g < 0 || g > 7) return h->fail(AMC_E_INVALID, "group out of range");
    P &p = h->p;
    int ncell = p.nc[0] * p.nc[1] * p.nc[2];
    unsigned grid = (unsigned)std::min<int64_t>((int64_t)h->pair_grid, std::max<int64_t>(ncell / 8, 1));
    if (h->n) k_pairs_group<false><<<grid, PAIR_THREADS, 0, h->stream>>>(p, g);
    k_bnd_pack<<<2, ADVECT_THREADS, 0, h->stream>>>(p);
    h->last_launches += (h->n ? 1 : 0) + 1;
    CK(cudaGetLastError());
    return AMC_OK;
}

extern "C" int amc_slab_apply(amc_handle *h, int32_t group_done)
{
    int rc = slab_check(h);
    if (rc != AMC_OK) return rc;
    P &p = h->p;
    p.group_done = group_done;
    if (p.nranks > 1) { k_bnd_apply<false><<<dim3(48, 2), 128, 0, h->stream>>>(p); h->last_launches += 1; }
    CK(cudaGetLastError());
    return AMC_OK;
}

extern "C" int amc_slab_finish(amc_handle *h, amc_step_stats *stats)
{
    int rc = slab_check(h);
    if (rc != AMC_OK) return rc;
    P &p = h->p;
    int32_t nf = 0;
    CK(cudaMemcpyAsync(&nf, p.n_foreign, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    if (h->n && p.kind != AMC_KIND_CUBE) { k_recapture_list<<<148, ADVECT_THREADS, 0, h->stream>>>(p); h->last_launches += 1; }
    unsigned long long ovf[4] = {0, 0, 0, 0};
    CK(cudaMemcpyAsync(ovf, h->d_slab_overflow, sizeof(ovf), cudaMemcpyDeviceToHost, h->stream));
    rc = phase_end(h, stats);
    if (rc != AMC_OK) return rc;
    if (h->slab_det_pending) { /* slab mode: the detection time accumulates over steps (callers take differences) */
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, h->det_events[0], h->det_events[1]));
        h->last_detect_ms += ms;
        h->slab_det_pending = false;
    }
    if ((rc = slab_overflow_error(h, ovf)) != AMC_OK) return rc;
    if (h->n + nf > h->cap) return h->fail(AMC_E_CAPACITY, "max_particles too small for the foreign copies of this step (state invalid)");
    h->n += nf; // foreign copies appended behind the sorted particles; dropped by the next amc_slab_advect
    p.n = h->n;
    return AMC_OK;
}

extern "C" int amc_slab_get_owned(amc_handle *h, int64_t cap, int64_t *n, int64_t *ids, double *x, double *y, double *z,
                                  double *vx, double *vy, double *vz, double *dist, double *dist_x, double *dist_y,
                                  double *dist_z, uint8_t *flag)
{
    int rc = slab_check(h);
    if (rc != AMC_OK) return rc;
    P &p = h->p;
    int32_t *cnt = h->d_counters + p.nranks + 5;
    CK(cudaMemsetAsync(cnt, 0, sizeof(int32_t), h->stream));
    if (h->n) k_compact_owned<<<grid_for(h->n, ADVECT_THREADS), ADVECT_THREADS, 0, h->stream>>>(p, cnt);
    int32_t c = 0;
    CK(cudaMemcpyAsync(&c, cnt, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (n) *n = c;
    if (c > cap) return h->fail(AMC_E_CAPACITY, "caller buffers too small for the owned particles");
    Arrays &b = p.b;
    const SoaView v = soa_view(b.pos, h->cap); /* k_compact_owned wrote positions, ids and flags as separate arrays */
    double *dst[10] = {x, y, z, vx, vy, vz, dist, dist_x, dist_y, dist_z};
    const double *src[10] = {v.x, v.y, v.z, b.vx, b.vy, b.vz, b.d, b.dx, b.dy, b.dz};
    for (int k = 0; k < 10; k++)
        if (dst[k] && c) CK(cudaMemcpyAsync(dst[k], src[k], c * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (flag && c) CK(cudaMemcpyAsync(flag, v.flag, c, cudaMemcpyDeviceToHost, h->stream));
    std::vector<int32_t> tmp((size_t)c);
    if (ids && c) CK(cudaMemcpyAsync(tmp.data(), v.id, c * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (ids) for (int32_t k = 0; k < c; k++) ids[k] = tmp[(size_t)k];
    return AMC_OK;
}

// ---- device-resident multi-GPU stepping ---------------------------------------------------------------
extern "C" int amc_slab_p2p_setup(amc_handle *h, amc_slab_p2p_desc *out)
{
    int rc = slab_check(h);
    if (rc != AMC_OK) return rc;
    if (!out) return h->fail(AMC_E_INVALID, "null descriptor");
    P &p = h->p;
    if (!h->p2p_base) {
        const size_t flag_bytes = ((size_t)(p.nranks + 2) * sizeof(uint32_t) + 255) / 256 * 256;
        const size_t xf_half = (size_t)h->xf_total * AMC_REC, bnd_half = (size_t)(p.bnd_cap + 1) * AMC_REC; /* doubles */
        const size_t bytes = flag_bytes + (2 * xf_half + 4 * bnd_half) * sizeof(double);
        ALLOC(h->p2p_base, bytes);
        CK(cudaMemset(h->p2p_base, 0, bytes));
        amc_slab_p2p_desc &d = h->p2p_desc;
        memset(&d, 0, sizeof(d));
        d.pid = (int64_t)getpid(); d.device = h->device; d.rank = p.srank; d.base = (uint64_t)(uintptr_t)h->p2p_base;
        d.off_flags = 0; d.off_xfer = (int64_t)flag_bytes;
        d.off_bnd_up = d.off_xfer + (int64_t)(2 * xf_half * sizeof(double));
        d.off_bnd_down = d.off_bnd_up + (int64_t)(2 * bnd_half * sizeof(double));
        d.xfer_stride = (int64_t)xf_half; d.bnd_stride = (int64_t)bnd_half;
        cudaIpcMemHandle_t ipc;
        CK(cudaIpcGetMemHandle(&ipc, h->p2p_base));
        static_assert(sizeof(ipc) <= sizeof(d.ipc), "ipc handle size");
        memcpy(d.ipc, &ipc, sizeof(ipc));
        if (!p.xf_send) { double *snd = nullptr; ALLOC(snd, (size_t)h->xf_total * AMC_REC); p.xf_send = snd; }
        ALLOC(h->d_n, 2);
    }
    *out = h->p2p_desc;
    return AMC_OK;
}

extern "C" int amc_slab_p2p_connect(amc_handle *h, const amc_slab_p2p_desc *all)
{
    int rc = slab_check(h);
    if (rc != AMC_OK) return rc;
    if (!all || !h->p2p_base) return h->fail(AMC_E_STATE, "amc_slab_p2p_setup first");
    P &p = h->p;
    std::vector<double *> xf(p.nranks);
    std::vector<uint32_t *> fl(p.nranks);
    std::vector<char *> base(p.nranks, nullptr);
    std::vector<int64_t> strides(p.nranks, 0);
    for (int r = 0; r < p.nranks; r++) {
        const amc_slab_p2p_desc &d = all[r];
        if (d.rank != r) return h->fail(AMC_E_INVALID, "descriptors must be ordered by rank");
        if (d.bnd_stride != h->p2p_desc.bnd_stride) return h->fail(AMC_E_INVALID, "ranks disagree on bnd_capacity");
        strides[r] = d.xfer_stride;
        if (r == p.srank) base[r] = h->p2p_base;
        else if (d.pid == (int64_t)getpid()) { /* same process: the address is valid here, the devices need peer access */
            base[r] = (char *)(uintptr_t)d.base;
            if (d.device != h->device) {
                cudaError_t e = cudaDeviceEnablePeerAccess(d.device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return h->fail(AMC_E_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
                cudaGetLastError();
            }
        } else {
            cudaIpcMemHandle_t ipc;
            memcpy(&ipc, d.ipc, sizeof(ipc));
            void *q = nullptr;
            CK(cudaIpcOpenMemHandle(&q, ipc, cudaIpcMemLazyEnablePeerAccess));
            h->p2p_opened.push_back(q);
            base[r] = (char *)q;
        }
        xf[r] = (double *)(base[r] + d.off_xfer);
        fl[r] = (uint32_t *)(base[r] + d.off_flags);
    }
    double **dxf = nullptr; uint32_t **dfl = nullptr;
    ALLOC(dxf, p.nranks); ALLOC(dfl, p.nranks);
    CK(cudaMemcpy(dxf, xf.data(), p.nranks * sizeof(double *), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dfl, fl.data(), p.nranks * sizeof(uint32_t *), cudaMemcpyHostToDevice));
    p.peer_xf = dxf; p.peer_flag = dfl;
    {
        int64_t *dst = nullptr, *dof = nullptr;
        ALLOC(dst, p.nranks); ALLOC(dof, p.nranks);
        CK(cudaMemcpy(dst, strides.data(), p.nranks * sizeof(int64_t), cudaMemcpyHostToDevice));
        p.peer_xf_stride = dst;
        // where rank d keeps the block of this rank: its blocks are ordered by source rank and sized by |source - d|
        std::vector<int64_t> offs(p.nranks, 0);
        for (int d = 0; d < p.nranks; d++)
            for (int e = 0; e < p.srank; e++) offs[d] += (std::abs(e - d) == 1 ? p.xf_cap_nb : p.xf_cap_far) + 1;
        CK(cudaMemcpy(dof, offs.data(), p.nranks * sizeof(int64_t), cudaMemcpyHostToDevice));
        p.peer_xf_off = dof;
    }
    const amc_slab_p2p_desc &me = h->p2p_desc;
    p.flags = (const uint32_t *)(h->p2p_base + me.off_flags);
    p.xf_recv = (const double *)(h->p2p_base + me.off_xfer);
    p.bnd_recv[0] = (const double *)(h->p2p_base + me.off_bnd_up);
    p.bnd_recv[1] = (const double *)(h->p2p_base + me.off_bnd_down);
    p.peer_bnd[0] = p.srank + 1 < p.nranks ? (double *)(base[p.srank + 1] + all[p.srank + 1].off_bnd_down) : nullptr;
    p.peer_bnd[1] = p.srank > 0 ? (double *)(base[p.srank - 1] + all[p.srank - 1].off_bnd_up) : nullptr;
    p.xf_stride = (int32_t)me.xfer_stride; p.bnd_stride = (int32_t)me.bnd_stride;
    h->p2p = true;
    CK(cudaDeviceSynchronize());
    return AMC_OK;
}

extern "C" int amc_slab_step(amc_handle *h, int32_t n_steps, int32_t pre_round, amc_step_stats *stats)
{
    int rc = slab_check(h);
    if (rc != AMC_OK) return rc;
    if (!h->p2p) return h->fail(AMC_E_STATE, "amc_slab_p2p_connect first");
    if (n_steps < 0) return h->fail(AMC_E_INVALID, "n_steps < 0");
    P &p = h->p;
    const int ncell = p.nc[0] * p.nc[1] * p.nc[2];
    const unsigned pgrid = (unsigned)std::min<int64_t>((int64_t)std::min(h->pair_grid, h->pair_grid_fused), std::max<int64_t>(ncell / 8, 1));
    const int phase = PH_DRIFT | PH_WALLS | (p.kind != AMC_KIND_CUBE ? PH_RECAP : 0);
    memset(h->last_ms, 0, sizeof(h->last_ms));
    sample_reset_timing(h);
    int32_t n32 = (int32_t)h->n;
    CK(cudaMemcpyAsync(h->d_n, &n32, sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    p.n_dev = h->d_n;
    int done = 0;
    while (done < n_steps) {
        const int chunk = std::min(n_steps - done, std::min(h->stats_cap, 64));
        // the count changes by a few hundred per step (migration); the launches of this chunk cover a generous bound
        p.n_hint = std::min<int64_t>(h->cap, h->n + h->n / 32 + 2 * (int64_t)h->xf_total + 4 * (int64_t)p.foreign_cap);
        const unsigned full = grid_for(p.n_hint, ADVECT_THREADS);
        if ((rc = ensure_events(h, h->events, (size_t)chunk * 4 + 1)) != AMC_OK) { p.n_dev = nullptr; return rc; }
        if ((rc = ensure_events(h, h->det_events, (size_t)chunk * 2)) != AMC_OK) { p.n_dev = nullptr; return rc; }
        CK(cudaMemsetAsync(h->d_stats, 0, chunk * sizeof(StatsDev), h->stream));
        CK(cudaEventRecord(h->events[0], h->stream));
        for (int s = 0; s < chunk; s++) {
            p.stats = h->d_stats + s;
            p.step = h->step_index++;
            if (h->sp.acc) h->surf_steps++;
            p.xf_seq = ++h->xf_seq;
            p.parity = (int32_t)(p.xf_seq & 1u);
            // ---- advect (dry run) + packing, all-to-all, unpack, sort
            CK(cudaMemsetAsync(h->d_counters, 0, (p.nranks + 12) * sizeof(int32_t), h->stream));
            CK(cudaMemsetAsync(p.rel_id, 0xff, (size_t)p.rel_cap * sizeof(int32_t), h->stream));
            CK(cudaMemsetAsync(p.band_count, 0, (h->n_buckets + 2) * sizeof(int32_t), h->stream));
            CK(cudaMemsetAsync(p.rest_count, 0, (h->n_buckets + 1) * sizeof(int32_t), h->stream));
            k_keys<true><<<full, ADVECT_THREADS, 0, h->stream>>>(p, phase);
            CK(cudaEventRecord(h->events[4 * s + 1], h->stream));
            if (p.nranks > 1) {
                k_slab_pack<<<dim3(grid_for(p.xf_cap, ADVECT_THREADS), p.nranks), ADVECT_THREADS, 0, h->stream>>>(p, phase);
                k_xfer_push<<<p.nranks, 32, 0, h->stream>>>(p);
                k_xfer_unpack<<<dim3(grid_for(p.xf_cap, ADVECT_THREADS), p.nranks), ADVECT_THREADS, 0, h->stream>>>(p);
            }
            int m = h->n_buckets, ntiles = (m + SCAN_TILE - 1) / SCAN_TILE;
            k_scan_tiles<<<ntiles, SCAN_THREADS, 0, h->stream>>>(p.band_count, p.rest_count, p.cell_start, h->d_tile_sums, m);
            k_scan_sums<<<1, SCAN_THREADS, 0, h->stream>>>(h->d_tile_sums, ntiles);
            k_scan_add<<<ntiles, SCAN_THREADS, 0, h->stream>>>(p.cell_start, h->d_tile_sums, m, 0);
            if (h->sp.acc) k_scatter_advect_surf<true><<<full, ADVECT_THREADS, 0, h->stream>>>(p, phase, h->sp);
            else k_scatter_advect<true><<<full, ADVECT_THREADS, 0, h->stream>>>(p, phase);
            std::swap(p.a, p.b);
            k_slab_set_n<<<1, 32, 0, h->stream>>>(p, 1);
            CK(cudaEventRecord(h->events[4 * s + 2], h->stream));
            // ---- pair pass: detection once, then the colour groups with a hand-over after each
            p.group_done = -1;
            if ((rc = prepare_pairs(h, h->stream)) != AMC_OK) { p.n_dev = nullptr; return rc; }
            CK(cudaEventRecord(h->det_events[2 * s], h->stream));
            launch_detect(h);
            CK(cudaEventRecord(h->det_events[2 * s + 1], h->stream));
            h->last_launches += 12;
            if (p.nranks > 1 && pgrid >= 2 * BND_HEAD_CTAS) {
                // the hand-over rides inside the group launches (k_pairs_group, fused): records of group g are sent by the
                // last CTA of launch g and applied at the head of launch g + 1 while the cells away from the cuts run
                uint32_t prev = 0;
                if (pre_round) { /* immigrants that landed in the band below an even cut travel before the first group */
                    p.bnd_seq = ++h->bnd_seq;
                    k_bnd_apply<true><<<dim3(48, 2), 128, 0, h->stream>>>(p);
                    h->last_launches += 1;
                }
                const bool trace = getenv("AMC_SLAB_TRACE") && s == chunk - 1;
                if (trace && (rc = ensure_events(h, h->grp_events, 10)) != AMC_OK) { p.n_dev = nullptr; return rc; }
                for (int g = 0; g < 8; g++) {
                    p.bnd_seq_apply = prev;
                    p.bnd_seq = ++h->bnd_seq;
                    p.group_done = g - 1;
                    if (trace) CK(cudaEventRecord(h->grp_events[g], h->stream));
                    k_pairs_group<true><<<pgrid, PAIR_THREADS, 0, h->stream>>>(p, g);
                    prev = p.bnd_seq;
                }
                p.group_done = 7;                      /* the records of the last group: wait and apply */
                if (trace) CK(cudaEventRecord(h->grp_events[8], h->stream));
                k_bnd_apply<false><<<dim3(48, 2), 128, 0, h->stream>>>(p);
                if (trace) CK(cudaEventRecord(h->grp_events[9], h->stream));
                h->last_launches += 9;
            } else
            for (int g = pre_round ? -1 : 0; g < 8; g++) {
                if (g >= 0) { k_pairs_group<false><<<pgrid, PAIR_THREADS, 0, h->stream>>>(p, g); h->last_launches += 1; }
                p.bnd_seq = ++h->bnd_seq;
                p.group_done = g;
                if (p.nranks > 1) k_bnd_apply<true><<<dim3(48, 2), 128, 0, h->stream>>>(p); /* sends, then waits for and applies the neighbours' records */
                else k_bnd_pack<<<2, ADVECT_THREADS, 0, h->stream>>>(p);
                h->last_launches += 1;
            }
            CK(cudaEventRecord(h->events[4 * s + 3], h->stream));
            if (p.kind != AMC_KIND_CUBE) { k_recapture_list<<<148, ADVECT_THREADS, 0, h->stream>>>(p); h->last_launches += 1; }
            if (sample_due(h, p.step) && (rc = launch_sample(h, p.n_hint, &h->last_launches)) != AMC_OK) { p.n_dev = nullptr; return rc; } /* count: cur_n */
            k_slab_set_n<<<1, 32, 0, h->stream>>>(p, 0);
            CK(cudaEventRecord(h->events[4 * s + 4], h->stream));
            CK(cudaGetLastError());
        }
        unsigned long long ovf[4] = {0, 0, 0, 0};
        CK(cudaMemcpyAsync(h->h_stats, h->d_stats, chunk * sizeof(StatsDev), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(ovf, h->d_slab_overflow, sizeof(ovf), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(&n32, h->d_n, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
        cudaError_t e = cudaStreamSynchronize(h->stream);
        p.n_dev = nullptr;
        if (e != cudaSuccess) return h->fail(AMC_E_CUDA, std::string("amc_slab_step: ") + cudaGetErrorString(e));
        if ((rc = sample_collect_timing(h)) != AMC_OK) return rc;
        {
            unsigned int timeouts = 0;
            CK(cudaMemcpyFromSymbol(&timeouts, g_flag_timeouts, sizeof(timeouts)));
            if (timeouts) return h->fail(AMC_E_STATE, "a neighbouring rank did not deliver its records within 20 s (peer-to-peer exchange timed out); the state of this handle is undefined");
        }
        h->n = n32; p.n = n32;
        p.n_dev = h->d_n;
        for (int s = 0; s < chunk; s++) {
            float ms;
            for (int k = 0; k < 4; k++) {
                CK(cudaEventElapsedTime(&ms, h->events[4 * s + k], h->events[4 * s + k + 1]));
                h->last_ms[k] += ms;
            }
            CK(cudaEventElapsedTime(&ms, h->det_events[2 * s], h->det_events[2 * s + 1]));
            h->last_detect_ms += ms;
        }
        if (getenv("AMC_SLAB_TRACE") && h->grp_events.size() >= 10 && p.nranks > 1) {
            for (int g = 0; g < 9; g++) {
                float ms = 0;
                if (cudaEventElapsedTime(&ms, h->grp_events[g], h->grp_events[g + 1]) == cudaSuccess) h->group_ms[g] += ms;
            }
            h->group_ms[9] += 1;
        }
        if ((rc = slab_overflow_error(h, ovf)) != AMC_OK) { p.n_dev = nullptr; return rc; }
        for (int s = 0; s < chunk; s++) {
            if ((rc = check_overflow(h, h->h_stats[s])) != AMC_OK) { p.n_dev = nullptr; return rc; }
            if (stats) stats_to_host(h, h->h_stats[s], stats + done + s);
        }
        done += chunk;
    }
    h->last_ms[4] = h->last_ms[0] + h->last_ms[1] + h->last_ms[2] + h->last_ms[3];
    p.n_dev = nullptr;
    p.stats = h->d_stats;
    return AMC_OK;
}

#ifdef AMC_SLAB_PROBE
// debug build: read (and reset) the wall-clock marks of the fused group launches (see g_probe)
extern "C" int amc_debug_probe(unsigned long long out[64], int reset)
{
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out, g_probe, 64 * sizeof(unsigned long long));
    if (reset) {
        unsigned long long z[8][8];
        for (int g = 0; g < 8; g++) for (int k = 0; k < 8; k++) z[g][k] = k == 0 ? ~0ull : 0ull;
        cudaMemcpyToSymbol(g_probe, z, sizeof(z));
    }
    return 0;
}
#endif

// debug (AMC_SLAB_TRACE=1): device time of the colour-group launches of amc_slab_step, summed over the traced steps
extern "C" int amc_debug_group_ms(amc_handle *h, double out[10])
{
    if (!h || !out) return AMC_E_INVALID;
    memcpy(out, h->group_ms, sizeof(h->group_ms));
    return AMC_OK;
}

extern "C" int amc_state_digest(amc_handle *h, uint64_t out[3])
{
    if (!h || !out) return AMC_E_INVALID;
    CK(cudaSetDevice(h->device));
    unsigned long long *d = reinterpret_cast<unsigned long long *>(h->p.path_sums) + 8; /* three spare words behind the path sums */
    CK(cudaMemsetAsync(d, 0, 3 * sizeof(unsigned long long), h->stream));
    if (h->n) k_state_digest<<<148 * 4, ADVECT_THREADS, 0, h->stream>>>(h->p, d);
    CK(cudaGetLastError());
    unsigned long long v[3];
    CK(cudaMemcpyAsync(v, d, sizeof(v), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    out[0] = v[0]; out[1] = v[1]; out[2] = v[2];
    return AMC_OK;
}

#ifdef AMC_PHASE_CLOCK
extern "C" int amc_debug_phase_clocks(unsigned long long out[16], int reset)
{
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out, g_phase_clk, 16 * sizeof(unsigned long long));
    if (reset) { unsigned long long z[16] = {0}; cudaMemcpyToSymbol(g_phase_clk, z, sizeof(z)); }
    return 0;
}
#endif
