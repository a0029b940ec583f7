// amc_kernels.cuh -- the kernels of libamc.so.
//   k_keys            dry run of the timestep -> owner cell + in-cell rank of every particle     (issue / latency)
//   k_scan_*          exclusive scan of the owner-cell histogram                                 (tiny)
//   k_scatter_advect  the timestep itself on the way to the sorted slot                         (HBM streaming)
//   k_build_worklist  reference cells with >= 2 candidates -> detection list                    (tiny)
//   k_detect_tma      neighbour search over every reference cell, all colour groups at once; candidates staged by
//                     cp.async.bulk + mbarrier; <true>: overlap-free seeding                     (issue; 33 B/particle)
//   k_pairs_group     ordered resolution of the flagged / activated cells of one colour group   (latency)
//   k_recapture_list  closing recapture over the slots a collision touched                      (tiny)
//   k_advect, k_scatter, k_recapture_post   the same step as separate in-place passes: phase-level parity entry points
//   k_sweep_detect, k_sweep_events   the serial lexicographic cell sweep of the cube stage, event-driven  (latency)
//   k_cube_sweep      the same sweep as a plain walk over every cell (fall-back when a column list overflows)  (latency)
//   k_pack_pos, k_unpack_pos   the C ABI's separate arrays <-> the 32-byte position records
//   k_case_*          per-case wall kernels for the host-RNG parity mode
//   k_init_synthetic  synthetic Maxwellian initial state
//   k_xfer_*, k_bnd_* slab decomposition: migration / ghost copies, per-group hand-over
//   k_flux            plane flux recording: net crossings of the z planes since the last record point
#pragma once
#include "amc_device.cuh"

#define ADVECT_THREADS 256
#define PAIR_THREADS 128
#define AMC_MV_CAP 32 /* particles one cell visit can move (reference scale: 2-6) */
#define WALK_K 3 /* chains a thread of cell_process walks side by side */
#define PAIR_K 3 /* candidates a thread of k_pairs_group has in flight during the gather */
#define PAIR_OCC 6 /* resident CTAs per SM of k_pairs_group: a colour-group launch lasts one visit if the group's worklist fits the grid, two if not */
#define SWEEP_THREADS 512

// Programmatic dependent launch (griddepcontrol; SASS PREEXIT / ACQBULK): a kernel launched with
// cudaLaunchAttributeProgrammaticStreamSerialization may become resident while the kernel before it in the stream still
// runs.  pdl_trigger() lets the next launch start becoming resident, pdl_wait() returns when the previous kernel has
// completed and its memory operations are visible; nothing that depends on the previous kernel may be touched before it.
// Both are no-ops in a launch without the attribute.  Used where launches follow one another without anything in
// between (launch_pdl in amc_api.cu): colour group g + 1 behind group g, k_scan_sums / k_scan_add behind k_scan_tiles --
// about 2 us per kernel boundary (measured on B200: 12.5 M particles 1.0005 -> 0.9813 ms per step, 557,649 particles
// 0.2556 -> 0.2381 ms).  The same attribute on k_scan_tiles behind k_keys, on k_scatter_advect behind the scan and on group 0
// behind the detection pass (each with a timing event recorded in between, and a predecessor that fills every SM until
// it ends) changed nothing and is not used.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// the whole particle: the position record with one 256-bit load, the seven other values from their arrays; returns the id
__device__ __forceinline__ int32_t load_part(const Arrays &a, int64_t s, Part &q)
{
    const PosRec r = a.pos[s];
    q.x = r.x; q.y = r.y; q.z = r.z; q.flag = r.flag;
    q.vx = a.vx[s]; q.vy = a.vy[s]; q.vz = a.vz[s];
    q.d = a.d[s]; q.dx = a.dx[s]; q.dy = a.dy[s]; q.dz = a.dz[s];
    return r.id;
}
// the same back, in place (the record keeps its id: one 128-bit store for x and y, z and the flag word beside it)
__device__ __forceinline__ void store_part(const Arrays &a, int64_t s, const Part &q)
{
    PosRec *r = a.pos + s;
    *reinterpret_cast<double2 *>(r) = make_double2(q.x, q.y);
    r->z = q.z; r->flag = q.flag & 0xffu;
    a.vx[s] = q.vx; a.vy[s] = q.vy; a.vz[s] = q.vz;
    a.d[s] = q.d; a.dx[s] = q.dx; a.dy[s] = q.dy; a.dz[s] = q.dz;
}
// to another slot: the full record (one 256-bit store)
__device__ __forceinline__ void store_part_id(const Arrays &a, int64_t s, const Part &q, const int32_t id)
{
    st_pos(a.pos + s, q.x, q.y, q.z, id, q.flag & 0xffu);
    a.vx[s] = q.vx; a.vy[s] = q.vy; a.vz[s] = q.vz;
    a.d[s] = q.d; a.dx[s] = q.dx; a.dy[s] = q.dy; a.dz[s] = q.dz;
}

// rank of this lane among all particles incrementing `counter` (identified by `tag` within the warp):
// the lanes with equal tag elect a leader that adds their number once
__device__ __forceinline__ int warp_rank(int32_t *counter, int tag)
{
    unsigned active = __activemask();
    unsigned peers = __match_any_sync(active, tag);
    int leader = __ffs(peers) - 1, lane = threadIdx.x & 31;
    int base = 0;
    if (lane == leader) base = atomicAdd(counter, __popc(peers));
    base = __shfl_sync(peers, base, leader);
    return base + __popc(peers & ((1u << lane) - 1));
}

// ------------------------------------------------------------------------------------------------
// K1 + K4.  One thread per particle slot; `phase` selects the parts of the step to run so the same
// code serves the fused step and the phase-level parity entry points.
//   drift         Pore:427-437 / Temp:673-683 / Cube:180-187
//   walls         Pore:442-485 / Temp:693-753 (device RNG) / Cube:192-226
//   recapture     Pore:354-375 / Temp:560-616
//   keys          owner cell of the final position + rank inside that cell (counting sort, pass 1)
// k_advect_surf: the same with the wall interactions recorded (amc_surface_*), launched only while recording is on
template <bool SURF>
__device__ __forceinline__ void advect_body(const P &p, const int phase, const SurfP *sp)
{
    int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= p.n) return;
    Part q;
    const int32_t id = load_part(p.a, s, q);
    if (p.slab && (q.flag & AMC_FLAG_GHOST)) { // last step's copy of a neighbour's particle: drop it
        if (phase & PH_KEYS) { p.key[s] = p.ncell_pad + 1; p.rank[s] = ~atomicAdd(&p.rest_count[p.ncell_pad + 1], 1); }
        return;
    }
    q.flag &= AMC_FLAG_PATH;
    if (phase & PH_RECAP_POST) { // recapture that closes the previous step's pair pass (Pore:550 / Temp:843-845)
        int cnt = p.kind == AMC_KIND_TEMP ? temp_oob(p.g, q) : 0;
        int moved = p.kind == AMC_KIND_TEMP ? temp_recapture(p.g, q) : pore_recapture(p.g, q);
        if (p.kind != AMC_KIND_TEMP) cnt = moved;
        if (cnt) atomicAdd(&p.stats_prev->oob_pp, (unsigned long long)cnt);
        if (p.kind == AMC_KIND_TEMP && moved) {
            int after = temp_oob(p.g, q);
            if (after) atomicAdd(&p.stats_prev->oob_pp_after, (unsigned long long)after);
        }
    }
    if (phase & PH_DRIFT) {
        q.px = q.x; q.py = q.y; q.pz = q.z;
        double ax = p.dt * q.vx, ay = p.dt * q.vy, az = p.dt * q.vz;
        q.x += ax; q.y += ay; q.z += az;
        q.d += fabs(sqrt((ax * ax + ay * ay) + az * az));
        q.dx += fabs(ax); q.dy += fabs(ay); q.dz += fabs(az);
        if (phase & PH_SAVE_PRIOR) { p.px[s] = q.px; p.py[s] = q.py; p.pz[s] = q.pz; }
    } else if (phase & PH_LOAD_PRIOR) {
        q.px = p.px[s]; q.py = p.py[s]; q.pz = p.pz[s];
    }
    if (phase & PH_WALLS) {
        uint32_t bits = p.kind == AMC_KIND_PORE ? pore_walls<AMC_LIVE, SURF>(p, q, sp)
                                                : (p.kind == AMC_KIND_TEMP ? temp_walls_device<AMC_LIVE, SURF>(p, q, id, sp) : cube_walls<AMC_LIVE, SURF>(p, q, sp));
        if (bits) {
            for (uint32_t b = bits; b; b &= b - 1) atomicAdd(&p.stats->wall_hits[__ffs(b) - 1], 1ull);
        }
        if (p.wall_bits) p.wall_bits[id] = (uint16_t)bits;
    }
    if (phase & PH_RECAP) {
        if (p.kind == AMC_KIND_PORE) {
            int cnt = pore_recapture(p.g, q);
            if (cnt) atomicAdd(&p.stats->oob_walls, (unsigned long long)cnt);
        } else if (p.kind == AMC_KIND_TEMP) {
            int cnt = temp_oob(p.g, q);
            if (cnt) atomicAdd(&p.stats->oob_walls, (unsigned long long)cnt);
            if (temp_recapture(p.g, q)) {
                int after = temp_oob(p.g, q);
                if (after) atomicAdd(&p.stats->oob_walls_after, (unsigned long long)after);
            }
        }
    }
    if ((phase & PH_KEYS) && p.slab) {
        // slab decomposition: the rank that owns the particle's global z layer keeps it; everything
        // else is packed for that rank.  A kept particle inside the overlap band below the upper cut is
        // also sent up as a ghost copy (the cells of the rank above read it as a band member).
        int gz = owner_axis(p.gz_edge, p.gncz, p.g_e0z, p.g_inv_dz, q.z);
        int layer = gz < 0 ? 0 : (gz >= p.gncz ? p.gncz - 1 : gz);
        int dest = 0;
        while (dest + 1 < p.nranks && layer >= p.cuts[dest + 1]) dest++;
        bool ghost_up = dest == p.srank && p.srank + 1 < p.nranks && q.z > p.up_thr;
        // a particle that just crossed the lower cut lands inside the band this rank's bottom cells
        // read: hand ownership down but keep the local copy as the ghost (no round trip needed)
        bool stay_as_ghost = dest == p.srank - 1 && q.z > p.down_band;
        if (ghost_up) q.flag |= AMC_FLAG_REL_UP;
        if (dest != p.srank || ghost_up) {
            int to = dest != p.srank ? dest : p.srank + 1;
            int j = atomicAdd(&p.xf_count[to], 1);
            if (j < p.xf_capv[to]) {
                double *r = p.xf_send + ((size_t)p.xf_off[to] + 1 + j) * AMC_REC;
                r[0] = q.x; r[1] = q.y; r[2] = q.z; r[3] = q.vx; r[4] = q.vy; r[5] = q.vz;
                r[6] = q.d; r[7] = q.dx; r[8] = q.dy; r[9] = q.dz; r[10] = (double)id;
                unsigned rf = q.flag & AMC_FLAG_PATH;
                if (dest == p.srank) rf |= AMC_FLAG_GHOST | AMC_FLAG_REL_DOWN; /* ghost copy for the rank above */
                else if (stay_as_ghost) rf |= AMC_FLAG_REL_UP;                 /* new owner: the rank above keeps a copy */
                r[11] = (double)rf;
            } else atomicAdd(p.slab_overflow + 0, 1ull);
        }
        if (dest != p.srank && !stay_as_ghost) { // emigrant: leaves this rank's arrays at the coming sort
            store_part(p.a, s, q);
            p.key[s] = p.ncell_pad + 1;
            p.rank[s] = ~atomicAdd(&p.rest_count[p.ncell_pad + 1], 1);
            return;
        }
        if (stay_as_ghost) q.flag = (q.flag & AMC_FLAG_PATH) | AMC_FLAG_GHOST | AMC_FLAG_REL_DOWN;
    }
    if (phase & (PH_DRIFT | PH_WALLS | PH_RECAP | PH_RECAP_POST)) store_part(p.a, s, q);
    if (phase & PH_KEYS) {
        int o[3];
        int32_t k = owner_key(p, q.x, q.y, q.z, o);
        p.key[s] = k;
        // band particles go to the front of their owner cell's segment so that neighbouring reference
        // cells only have to read that prefix; rank >= 0: band, rank < 0: ~rank among the others.
        // The state is nearly sorted, so the lanes of a warp share one or two counters: one atomic per
        // distinct counter and warp instead of one per particle.
        bool band = k != p.ncell_pad && any_band(p, q.x, q.y, q.z, o);
        int r = warp_rank(band ? &p.band_count[k] : &p.rest_count[k], (k << 1) | (int)band);
        p.rank[s] = band ? r : ~r;
    }
}
__global__ void __launch_bounds__(ADVECT_THREADS, 4) k_advect(const __grid_constant__ P p, const int phase) { advect_body<false>(p, phase, nullptr); }
__global__ void __launch_bounds__(ADVECT_THREADS, 4) k_advect_surf(const __grid_constant__ P p, const int phase, const __grid_constant__ SurfP sp)
{
    advect_body<true>(p, phase, &sp);
}

// ------------------------------------------------------------------------------------------------
// The fused timestep streams the state ONCE through the SM instead of twice: a light first pass finds out
// where every particle will be after the step (k_keys: 52 B read, 8 B written), and the counting-sort
// scatter then carries out the step itself on the way to the particle's new slot (k_scatter_advect:
// 93 B read, 85 B written) -- 238 B per particle and step instead of the 352 B of k_advect + k_scatter.
// advance_particle is the per-particle part of a timestep before the pair pass (closing recapture of
// the previous step, drift, wall cases, recapture; same references as k_advect).  MODE = AMC_DRY is a
// dry run: same arithmetic and therefore bit-identical positions, but no counters, no completed paths,
// no path-length bookkeeping -- none of which feeds back into the position.  SURF: the live run records the wall
// interactions (amc_surface_*).
template <int MODE, bool SURF = false>
__device__ __forceinline__ void advance_particle(const P &p, Part &q, const int32_t id, const int phase, const SurfP *sp = nullptr)
{
    // Calm particles (energized pore, ~95 % of the gas): both the position before the drift and the one after it
    // lie in one of three regions in which every wall mask (Temp:693-753), every recapture condition (Temp:594-616)
    // and every out-of-bounds count (Temp:560-592) is false whatever the other coordinates are -- the interior of the
    // bottom end cap (below every z threshold, inside the open-air radius), of the top end cap (above every z
    // threshold) and the core of the pore (inside every radius, between the end plates); the bounds are the min / max
    // of the geometry's thresholds, computed in amc_api.cu.  For them the whole step is the drift.
    if (p.calm_ok && (phase & (PH_DRIFT | PH_WALLS | PH_RECAP)) == (PH_DRIFT | PH_WALLS | PH_RECAP)) {
        const double ax = p.dt * q.vx, ay = p.dt * q.vy, az = p.dt * q.vz;
        const double nx = q.x + ax, ny = q.y + ay, nz = q.z + az;
        const double rmax = fmax(q.x * q.x + q.y * q.y, nx * nx + ny * ny), zmin = fmin(q.z, nz), zmax = fmax(q.z, nz);
        const bool calm = (rmax <= p.calm_rA && ((zmin >= 0.0 && zmax < p.calm_zA) || (zmin > p.calm_zB && zmax <= p.g.H))) ||
                          (rmax < p.calm_rC && zmin >= 0.0 && zmax <= p.g.H);
        if (calm) {
            q.px = q.x; q.py = q.y; q.pz = q.z;
            q.x = nx; q.y = ny; q.z = nz;
            if (MODE != AMC_DRY) {
                q.d += fabs(sqrt((ax * ax + ay * ay) + az * az));
                q.dx += fabs(ax); q.dy += fabs(ay); q.dz += fabs(az);
            }
            if (MODE == AMC_LIVE && p.wall_bits) p.wall_bits[id] = 0;
            return;
        }
    }
    if (phase & PH_RECAP_POST) { // recapture that closes the previous step's pair pass (Pore:550 / Temp:843-845)
        int cnt = p.kind == AMC_KIND_TEMP ? temp_oob(p.g, q) : 0;
        int moved = p.kind == AMC_KIND_TEMP ? temp_recapture(p.g, q) : pore_recapture(p.g, q);
        if (p.kind != AMC_KIND_TEMP) cnt = moved;
        if (MODE == AMC_LIVE && cnt) atomicAdd(&p.stats_prev->oob_pp, (unsigned long long)cnt);
        if (MODE == AMC_LIVE && p.kind == AMC_KIND_TEMP && moved) {
            int after = temp_oob(p.g, q);
            if (after) atomicAdd(&p.stats_prev->oob_pp_after, (unsigned long long)after);
        }
    }
    if (phase & PH_DRIFT) {
        q.px = q.x; q.py = q.y; q.pz = q.z;
        double ax = p.dt * q.vx, ay = p.dt * q.vy, az = p.dt * q.vz;
        q.x += ax; q.y += ay; q.z += az;
        if (MODE != AMC_DRY) {
            q.d += fabs(sqrt((ax * ax + ay * ay) + az * az));
            q.dx += fabs(ax); q.dy += fabs(ay); q.dz += fabs(az);
        }
    }
    if (phase & PH_WALLS) {
        uint32_t bits = p.kind == AMC_KIND_PORE ? pore_walls<MODE, SURF>(p, q, sp)
                                                : (p.kind == AMC_KIND_TEMP ? temp_walls_device<MODE, SURF>(p, q, id, sp) : cube_walls<MODE, SURF>(p, q, sp));
        if (MODE == AMC_LIVE) {
            for (uint32_t b = bits; b; b &= b - 1) atomicAdd(&p.stats->wall_hits[__ffs(b) - 1], 1ull);
            if (p.wall_bits) p.wall_bits[id] = (uint16_t)bits;
        }
    }
    if (phase & PH_RECAP) {
        if (p.kind == AMC_KIND_PORE) {
            int cnt = pore_recapture(p.g, q);
            if (MODE == AMC_LIVE && cnt) atomicAdd(&p.stats->oob_walls, (unsigned long long)cnt);
        } else if (p.kind == AMC_KIND_TEMP) {
            int cnt = temp_oob(p.g, q);
            if (MODE == AMC_LIVE && cnt) atomicAdd(&p.stats->oob_walls, (unsigned long long)cnt);
            if (temp_recapture(p.g, q) && MODE == AMC_LIVE) {
                int after = temp_oob(p.g, q);
                if (after) atomicAdd(&p.stats->oob_walls_after, (unsigned long long)after);
            }
        }
    }
}

// slab decomposition: the full post-step record of a particle that leaves for / is copied to another rank.
// Rare (the particles next to a cut), so it has its own register budget; QUIET because the live run of
// the same particle in k_scatter_advect does the recording.
__device__ __forceinline__ void slab_note(const P &p, const int64_t s, const int to, const unsigned extra)
{
    int j = atomicAdd(&p.xf_count[to], 1);
    if (j >= p.xf_capv[to]) { atomicAdd(p.slab_overflow + 0, 1ull); return; }
    p.xf_pack[p.xf_off[to] + 1 + j] = make_int2((int)s, (int)extra);
}
__device__ __forceinline__ void slab_pack(const P &p, const int64_t s, const int32_t id, const int phase, const int to, const int j, const unsigned extra)
{
    Part q;
    load_part(p.a, s, q);
    q.flag &= AMC_FLAG_PATH;
    advance_particle<AMC_QUIET>(p, q, id, phase);
    // peer-to-peer mode: the record goes straight into the receiver's buffer over NVLink (stores from all SMs side
    // by side); k_xfer_push only adds the count and the sequence number
    double *r = p.peer_xf ? p.peer_xf[to] + (size_t)p.parity * (size_t)p.peer_xf_stride[to] + ((size_t)p.peer_xf_off[to] + 1 + j) * AMC_REC
                          : p.xf_send + ((size_t)p.xf_off[to] + 1 + j) * AMC_REC;
    r[0] = q.x; r[1] = q.y; r[2] = q.z; r[3] = q.vx; r[4] = q.vy; r[5] = q.vz;
    r[6] = q.d; r[7] = q.dx; r[8] = q.dy; r[9] = q.dz; r[10] = (double)id;
    r[11] = (double)((q.flag & AMC_FLAG_PATH) | extra);
}

// the records of the particles k_keys<SLAB> noted for travel (~1 % of a slab: the particles next to a cut): kept out
// of k_keys so that the streaming pass carries neither the call nor its registers
__global__ void __launch_bounds__(ADVECT_THREADS) k_slab_pack(const __grid_constant__ P p, const int phase)
{
    const int to = blockIdx.y;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (to == p.srank || j >= min(p.xf_count[to], p.xf_capv[to])) return;
    const int2 e = p.xf_pack[p.xf_off[to] + 1 + j];
    slab_pack(p, e.x, p.a.pos[e.x].id, phase, to, j, (unsigned)e.y);
}

// pass 1 of the fused step: owner cell of the position each particle will have after the step, and its
// rank inside that cell (band particles first, see k_advect).  Slab mode: also decides which rank owns
// the particle after the step and packs the records that travel (see k_advect for the protocol).
#ifndef KEYS_OCC
#define KEYS_OCC 6           /* resident CTAs per SM of k_keys: latency-bound by the rank atomic, 40 registers (7 and 8 measured: see profiles/r2/summary.md) */
#endif
#ifndef KEYS_OCC_SLAB
#define KEYS_OCC_SLAB 6      /* resident CTAs per SM of the slab variant of k_keys (5 at 48 registers and 4 at 64 measured slower: latency-bound) */
#endif
#define AUX_GHOST_UP 1u      /* kept, and copied to the rank above */
#define AUX_STAY_AS_GHOST 2u /* owned by the rank below from now on, the local copy stays as its ghost */
template <bool SLAB>
__global__ void __launch_bounds__(ADVECT_THREADS, SLAB ? KEYS_OCC_SLAB : KEYS_OCC) k_keys(const __grid_constant__ P p, const int phase)
{
    int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= (SLAB ? p.cap : p.n)) return;
    // slab mode: the particle count lives on the device; its load travels together with the particle's own loads
    // (slots behind the count are allocated, their contents are ignored)
    Part q;
    const PosRec r0 = p.a.pos[s]; /* position, id and flag word: one 256-bit load */
    q.x = r0.x; q.y = r0.y; q.z = r0.z; q.vx = p.a.vx[s]; q.vy = p.a.vy[s]; q.vz = p.a.vz[s];
    q.d = q.dx = q.dy = q.dz = 0.0; q.flag = 0;
    const int32_t id = r0.id; /* keys the device RNG of the energized walls */
    if (SLAB) {
        const unsigned fl0 = r0.flag;
        if (s >= cur_n(p)) return;
        if (fl0 & AMC_FLAG_GHOST) { // last step's copy of a neighbour's particle: drop it
            p.key[s] = p.ncell_pad + 1; p.rank[s] = ~atomicAdd(&p.rest_count[p.ncell_pad + 1], 1);
            return;
        }
    }
    advance_particle<AMC_DRY>(p, q, id, phase);
    int o[3];
    const int32_t k = owner_key(p, q.x, q.y, q.z, o);
    if (SLAB) {
        // the local z tables are a window of the global ones: only a particle outside the window (below the first
        // local edge or not below the last) needs the global look-up to find its new rank
        int dest = p.srank;
        if (o[2] < 0 || o[2] >= p.nc[2]) {
            int gz = owner_axis(p.gz_edge, p.gncz, p.g_e0z, p.g_inv_dz, q.z);
            int layer = gz < 0 ? 0 : (gz >= p.gncz ? p.gncz - 1 : gz);
            dest = 0;
            while (dest + 1 < p.nranks && layer >= p.cuts[dest + 1]) dest++;
        }
        const bool ghost_up = dest == p.srank && p.srank + 1 < p.nranks && q.z > p.up_thr;
        const bool stay_as_ghost = dest == p.srank - 1 && q.z > p.down_band;
        if (dest != p.srank) slab_note(p, s, dest, stay_as_ghost ? AMC_FLAG_REL_UP : 0u);
        else if (ghost_up) slab_note(p, s, p.srank + 1, AMC_FLAG_GHOST | AMC_FLAG_REL_DOWN);
        p.aux[s] = (uint8_t)((ghost_up ? AUX_GHOST_UP : 0u) | (stay_as_ghost ? AUX_STAY_AS_GHOST : 0u));
        if (dest != p.srank && !stay_as_ghost) { // emigrant: leaves this rank's arrays at the coming sort
            p.key[s] = p.ncell_pad + 1; p.rank[s] = ~atomicAdd(&p.rest_count[p.ncell_pad + 1], 1);
            return;
        }
    }
    p.key[s] = k;
    bool band = k != p.ncell_pad && any_band(p, q.x, q.y, q.z, o);
    int r = warp_rank(band ? &p.band_count[k] : &p.rest_count[k], (k << 1) | (int)band);
    p.rank[s] = band ? r : ~r;
}

// pass 2: the timestep proper, written straight to the particle's slot in owner-cell order.  Slab mode: the
// particles unpacked behind the resident ones (slots n .. n + n_in) arrive already advanced; ghosts of the last
// step and emigrants go to the bucket behind the last cell and are dropped.  k_scatter_advect_surf: the same with the wall
// interactions recorded (see k_advect).
template <bool SLAB, bool SURF>
__device__ __forceinline__ void scatter_advect_body(const P &p, const int phase, const SurfP *sp)
{
    int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= (SLAB ? p.cap : p.n)) return;
    Part q;
    const int32_t id = load_part(p.a, s, q);
    const int32_t k = p.key[s], r = p.rank[s];
    const int64_t n0 = SLAB ? cur_n(p) : p.n; /* slab mode: on the device, loaded together with the record */
    if (SLAB && s >= n0 + *p.n_in) return;
    if (s < n0 && !(SLAB && (q.flag & AMC_FLAG_GHOST))) {
        q.flag &= AMC_FLAG_PATH;
        advance_particle<AMC_LIVE, SURF>(p, q, id, phase, sp);
        if (SLAB) {
            const unsigned aux = p.aux[s];
            if (aux & AUX_GHOST_UP) q.flag |= AMC_FLAG_REL_UP;
            if (aux & AUX_STAY_AS_GHOST) q.flag = (q.flag & AMC_FLAG_PATH) | AMC_FLAG_GHOST | AMC_FLAG_REL_DOWN;
        }
    }
    const int64_t t = (int64_t)p.cell_start[k] + (r >= 0 ? r : p.band_count[k] + ~r);
    const unsigned fl = q.flag;
    q.flag = fl & (SLAB ? AMC_FLAG_KEEP : AMC_FLAG_PATH);
    store_part_id(p.b, t, q, id);
    if ((phase & PH_RECAP) && k <= p.ncell_pad) { // still out of bounds after this step's recapture: the closing one must see it
        Part c = q;
        bool again = p.kind == AMC_KIND_TEMP ? (temp_oob(p.g, c) != 0) | (temp_recapture(p.g, c) != 0) : (p.kind == AMC_KIND_PORE && pore_recapture(p.g, c) != 0);
        if (again) touch_slot(p, (int32_t)t);
    }
    if (SLAB) {
        if (k <= p.ncell_pad && (fl & (AMC_FLAG_GHOST | AMC_FLAG_REL_UP | AMC_FLAG_REL_DOWN))) rel_insert(p, id, (int32_t)t);
        if (k <= p.ncell_pad && (fl & AMC_FLAG_LATE_UP)) {
            int j = atomicAdd(&p.bnd_n[0], 1);
            if (j < p.bnd_cap) p.bnd_dirty[0][j] = (int32_t)t; else atomicAdd(p.slab_overflow + 2, 1ull);
        }
    }
}
template <bool SLAB>
__global__ void __launch_bounds__(ADVECT_THREADS, 3) k_scatter_advect(const __grid_constant__ P p, const int phase)
{
    scatter_advect_body<SLAB, false>(p, phase, nullptr);
}
template <bool SLAB>
__global__ void __launch_bounds__(ADVECT_THREADS, 3) k_scatter_advect_surf(const __grid_constant__ P p, const int phase, const __grid_constant__ SurfP sp)
{
    scatter_advect_body<SLAB, true>(p, phase, &sp);
}

// ------------------------------------------------------------------------------------------------
// exclusive scan of cell_count[0..m) -> cell_start[0..m], three small kernels (m <= a few million)
#define SCAN_THREADS 1024
#define SCAN_ITEMS 4
#define SCAN_TILE (SCAN_THREADS * SCAN_ITEMS)

__device__ __forceinline__ int block_exclusive_scan(int v, int *total)
{
    __shared__ int warp_sums[32];
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
    if (lane == 31) warp_sums[w] = inc;
    __syncthreads();
    if (w == 0) {
        int ws = warp_sums[lane], wi = ws;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= o) wi += t; }
        warp_sums[lane] = wi - ws;
        if (lane == 31) *total = wi;
    }
    __syncthreads();
    int r = warp_sums[w] + inc - v;
    __syncthreads();
    return r;
}

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_tiles(const int32_t *in, const int32_t *in2, int32_t *out, int32_t *tile_sums, int m)
{
    __shared__ int total;
    int base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
    int v[SCAN_ITEMS], sum = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) { v[k] = base + k < m ? in[base + k] + in2[base + k] : 0; sum += v[k]; }
    pdl_trigger();
    int ex = block_exclusive_scan(sum, &total);
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) { if (base + k < m) out[base + k] = ex; ex += v[k]; }
    if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_sums(int32_t *tile_sums, int ntiles)
{
    __shared__ int total;
    __shared__ int carry;
    pdl_trigger();
    if (threadIdx.x == 0) carry = 0;
    pdl_wait(); /* the tile sums of k_scan_tiles */
    __syncthreads();
    for (int base = 0; base < ntiles; base += SCAN_THREADS) {
        int i = base + threadIdx.x;
        int v = i < ntiles ? tile_sums[i] : 0;
        int ex = block_exclusive_scan(v, &total);
        if (i < ntiles) tile_sums[i] = ex + carry;
        __syncthreads();
        if (threadIdx.x == 0) carry += total;
        __syncthreads();
    }
}
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_add(int32_t *out, const int32_t *tile_sums, int m, int32_t n_total)
{
    int base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
    pdl_wait(); /* the scanned tile sums of k_scan_sums (and, before it, the tiles of k_scan_tiles) */
    int add = tile_sums[blockIdx.x];
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) if (base + k < m) out[base + k] += add;
    if (blockIdx.x == 0 && threadIdx.x == 0) out[m] = n_total;
}

// counting-sort scatter: slot s of the old layout moves to cell_start[key] + rank
__global__ void __launch_bounds__(ADVECT_THREADS) k_scatter(const __grid_constant__ P p)
{
    int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= p.n + (p.slab ? *p.n_in : 0) || s >= p.cap) return;
    int32_t k = p.key[s], r = p.rank[s];
    int64_t t = (int64_t)p.cell_start[k] + (r >= 0 ? r : p.band_count[k] + ~r);
    const PosRec rec = p.a.pos[s];
    const unsigned fl = rec.flag;
    const int32_t id = rec.id;
    st_pos(p.b.pos + t, rec.x, rec.y, rec.z, id, fl & (p.slab ? AMC_FLAG_KEEP : AMC_FLAG_PATH));
    p.b.vx[t] = p.a.vx[s]; p.b.vy[t] = p.a.vy[s]; p.b.vz[t] = p.a.vz[s];
    p.b.d[t] = p.a.d[s]; p.b.dx[t] = p.a.dx[s]; p.b.dy[t] = p.a.dy[s]; p.b.dz[t] = p.a.dz[s];
    if (p.slab) {
        if (k <= p.ncell_pad && (fl & (AMC_FLAG_GHOST | AMC_FLAG_REL_UP | AMC_FLAG_REL_DOWN))) {
            rel_insert(p, id, (int32_t)t);
        }
        if (k <= p.ncell_pad && (fl & AMC_FLAG_LATE_UP)) {
            int j = atomicAdd(&p.bnd_n[0], 1);
            if (j < p.bnd_cap) p.bnd_dirty[0][j] = (int32_t)t; else atomicAdd(p.slab_overflow + 2, 1ull);
        }
    }
}

// back to original index order (amc_get_state): first the inverse permutation (4-byte scatter), then a
// gather with coalesced writes -- random 8-byte reads cost far less than random 8-byte writes
__global__ void __launch_bounds__(ADVECT_THREADS) k_inverse_perm(const __grid_constant__ P p)
{
    int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s < p.n) p.key[p.a.pos[s].id] = (int32_t)s;
}
__global__ void __launch_bounds__(ADVECT_THREADS) k_unsort(const __grid_constant__ P p)
{
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.n) return;
    int64_t s = p.key[t];
    const PosRec r = p.a.pos[s];
    st_pos(p.b.pos + t, r.x, r.y, r.z, (int32_t)t, r.flag & AMC_FLAG_PATH);
    p.b.vx[t] = p.a.vx[s]; p.b.vy[t] = p.a.vy[s]; p.b.vz[t] = p.a.vz[s];
    p.b.d[t] = p.a.d[s]; p.b.dx[t] = p.a.dx[s]; p.b.dy[t] = p.a.dy[s]; p.b.dz[t] = p.a.dz[s];
}

// start of a pair pass: forget the escaped-particle list of the previous pass (single block, so
// every thread reads the old count before it is cleared; unused entries always hold -1)
__global__ void k_pp_begin(const __grid_constant__ P p)
{
    int n = *p.esc_count;
    if (n > p.esc_cap) n = p.esc_cap;
    for (int i = threadIdx.x; i < n * 8; i += blockDim.x) p.esc_cell[i] = -1;
    __syncthreads();
    if (threadIdx.x == 0) *p.esc_count = 0;
}

// recapture that closes a pair pass (Pore:550 / Temp:843-845): positions only
__global__ void __launch_bounds__(ADVECT_THREADS) k_recapture_post(const __grid_constant__ P p)
{
    int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= p.n) return;
    if (p.slab && (p.a.pos[s].flag & AMC_FLAG_GHOST)) return; /* the owning rank recaptures it */
    Part q;
    q.x = p.a.pos[s].x; q.y = p.a.pos[s].y; q.z = p.a.pos[s].z;
    double x0 = q.x, y0 = q.y, z0 = q.z;
    int cnt = p.kind == AMC_KIND_TEMP ? temp_oob(p.g, q) : 0;
    int moved = p.kind == AMC_KIND_TEMP ? temp_recapture(p.g, q) : pore_recapture(p.g, q);
    if (p.kind != AMC_KIND_TEMP) cnt = moved;
    if (cnt) atomicAdd(&p.stats->oob_pp, (unsigned long long)cnt);
    if (p.kind == AMC_KIND_TEMP && moved) {
        int after = temp_oob(p.g, q);
        if (after) atomicAdd(&p.stats->oob_pp_after, (unsigned long long)after);
    }
    if (q.x != x0) p.a.pos[s].x = q.x;
    if (q.y != y0) p.a.pos[s].y = q.y;
    if (q.z != z0) p.a.pos[s].z = q.z;
}

// Only a particle that a collision moved (or that the walls + recapture of this step left out of bounds) can be
// touched by the recapture that closes the pair pass, so the step keeps a list of those slots and the closing
// recapture visits just them: same result as k_recapture_post over everything, a few microseconds instead of a
// pass over all positions.  The list is de-duplicated through a per-slot step tag; an overflowing list makes the
// kernel fall back to the full pass.
__device__ __forceinline__ void recapture_slot(const P &p, const int64_t s)
{
    if (p.slab && (p.a.pos[s].flag & AMC_FLAG_GHOST)) return; /* the owning rank recaptures it */
    Part q;
    q.x = p.a.pos[s].x; q.y = p.a.pos[s].y; q.z = p.a.pos[s].z;
    double x0 = q.x, y0 = q.y, z0 = q.z;
    int cnt = p.kind == AMC_KIND_TEMP ? temp_oob(p.g, q) : 0;
    int moved = p.kind == AMC_KIND_TEMP ? temp_recapture(p.g, q) : pore_recapture(p.g, q);
    if (p.kind != AMC_KIND_TEMP) cnt = moved;
    if (cnt) atomicAdd(&p.stats->oob_pp, (unsigned long long)cnt);
    if (p.kind == AMC_KIND_TEMP && moved) {
        int after = temp_oob(p.g, q);
        if (after) atomicAdd(&p.stats->oob_pp_after, (unsigned long long)after);
    }
    if (q.x != x0) p.a.pos[s].x = q.x;
    if (q.y != y0) p.a.pos[s].y = q.y;
    if (q.z != z0) p.a.pos[s].z = q.z;
}
__global__ void __launch_bounds__(ADVECT_THREADS) k_recapture_list(const __grid_constant__ P p)
{
    const int nt = *p.touched_n;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x, first = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (nt > p.touched_cap) { /* list overflowed: everything */
        for (int64_t s = first, n = cur_n(p); s < n; s += stride) recapture_slot(p, s);
    } else {
        const int32_t tag = 1 + (int32_t)(p.step & 0x3fffffff); /* per-slot marker: handled in this step already */
        for (int64_t i = first; i < nt; i += stride) {
            const int32_t s = p.touched[i];
            if (atomicExch(&p.touch_mark[s], tag) != tag) recapture_slot(p, s);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K2 + K3: one reference cell (ordered resolution; the cells get here through k_detect / esc_link).
//
// The reference visits the members of a cell in ascending global index and tests (i, j<i) against
// the live cell-local arrays, so a collision is visible to every later pair of the same cell
// (Pore:168-241).  "Earlier/later" is the lexicographic order of (larger id, smaller id), so the
// members need not be sorted: the CTA (1) tests all unordered member pairs in parallel and keeps
// the overlapping ones as candidates, (2) repeatedly resolves the candidate with the smallest key
// above a cursor, drops every candidate that involves one of the two moved particles and re-tests
// those two against all members for keys above the cursor.  That reproduces the sequential sweep
// exactly: pairs below the cursor were already passed, pairs not involving a moved particle keep
// their first-scan verdict.
#ifdef AMC_PHASE_CLOCK
// debug build only (tools/phase_clocks.py): cycles spent by thread 0 between the phase boundaries of a cell visit
__device__ unsigned long long g_phase_clk[16];
#define PHASE_MARK(k) do { if (threadIdx.x == 0) { long long now_ = clock64(); atomicAdd(&g_phase_clk[k], (unsigned long long)(now_ - S.t_last)); S.t_last = now_; } } while (0)
#else
#define PHASE_MARK(k) do { } while (0)
#endif

struct CellShared {
    double x[AMC_MAX_MEMBERS], y[AMC_MAX_MEMBERS], z[AMC_MAX_MEMBERS];
    int32_t id[AMC_MAX_MEMBERS], slot[AMC_MAX_MEMBERS], src[AMC_MAX_MEMBERS];
    unsigned long long cand_key[AMC_MAX_CAND];
    int32_t cand_ab[AMC_MAX_CAND]; /* a | b << 16 */
    int n, ncand, sel, done;
    int cand_lost;               /* the candidate list overflowed in this visit: every pick re-scans all pairs (slow, exact) */
    unsigned long long best_key; /* scan mode: smallest pair key above the cursor that overlaps */
    unsigned long long cursor;
    int moved_a, moved_b;
    int kx, ky, kz; /* 0-based cell indices of this visit (colour-group mode) */
    long long t_last;
    double org[3];               /* low corner of the cell: origin of the fp32 coordinates below */
    double hi[3];                /* upper bounds of the cell (membership: org < v < hi, Pore:527-529) */
    /* neighbour search: members chained per slab along x (>= 1.05 filter radii wide) */
    int head[AMC_XBINS + 2];     /* last member hashed into the slab (index + 1), 0 = empty; zero on entry of cell_process */
    uint16_t nxt[AMC_MAX_MEMBERS];    /* chain links of the search; afterwards (activate_moved) the list of the moved members */
    uint16_t mv[AMC_MAX_MEMBERS];     /* 0, or 1 + index of the member's pre-visit position in ox/oy/oz (beyond AMC_MV_CAP: in P::mv_spill) */
    double ox[AMC_MV_CAP], oy[AMC_MV_CAP], oz[AMC_MV_CAP];
    int nmv, nold;
    int hits[AMC_HIT_REC];       /* this work item's record of wl_hit */
    int hm[2 * AMC_MAX_HITS];    /* member index of each listed slot, -1 = not (or no longer) a member */
    int use_hits;                /* the listed pairs are all there is to test (set after the gather) */
    float inv_w;                 /* slabs per unit length */
    int nb;                      /* slabs of this cell, 1..AMC_XBINS */
    unsigned int nexec;          /* distance tests executed by this CTA since the last flush */
    unsigned long long nref;      /* reference-equivalent tests, thread 0 only */
    int rbeg[8], rcum[9];         /* the 8 candidate owner-cell ranges of this visit */
};

__device__ __forceinline__ unsigned long long pair_key(int32_t ia, int32_t ib)
{
    uint32_t hi = ia > ib ? ia : ib, lo = ia > ib ? ib : ia;
    return ((unsigned long long)hi << 32) | lo;
}
__device__ __forceinline__ bool overlap(const P &p, double xa, double ya, double za, double xb, double yb, double zb)
{
    double ddx = xb - xa, ddy = yb - ya, ddz = zb - za;
    return (ddx * ddx + ddy * ddy) + ddz * ddz < p.overlap_sq; /* == sqrt(...) < collision_range, Pore:173-174 */
}
__device__ __forceinline__ void push_cand(CellShared &S, const P &p, int a, int b)
{
    int k = atomicAdd(&S.ncand, 1);
    if (k < AMC_MAX_CAND) { S.cand_key[k] = pair_key(S.id[a], S.id[b]); S.cand_ab[k] = a | (b << 16); }
    else S.cand_lost = 1; /* more overlapping pairs at once than the list holds: the visit switches to scan mode */
    // the resolution will read the velocity / path records of both particles: start them on their way from HBM
    for (int w = 0; w < 2; w++) {
        int s = S.slot[w ? b : a];
        const double *rec[7] = {p.a.vx + s, p.a.vy + s, p.a.vz + s, p.a.d + s, p.a.dx + s, p.a.dy + s, p.a.dz + s};
#pragma unroll
        for (int r = 0; r < 7; r++) asm volatile("prefetch.global.L2 [%0];" ::"l"(rec[r]));
    }
}

// Make sure colour group g2 (which has not started yet) visits cell cc.  cell_active[g2][cc] is 0 while the cell
// is not on the group's worklist, 1 when it is, and e + 2 when it is and escaped-list entry e heads the list of
// the particles that can no longer be found through the sorted layout but are members of that cell (older
// entries follow through esc_next).  e < 0: just activate.  An entry is linked at most once per group.
__device__ __forceinline__ void esc_link(const P &p, int g2, int32_t cc, int cx, int cy, int cz, int e)
{
    if (e >= 0) p.esc_cell[e * 8 + g2] = cc;
    if (cc < 0) return;
#pragma unroll
    for (int nb = 0; nb < 8; nb++) { /* what write_work_item will read if the cell turns out to be new on the list */
        const int oc = ((cx + 1 - (nb >> 2)) * p.pnc[1] + (cy + 1 - ((nb >> 1) & 1))) * p.pnc[2] + (cz + 1 - (nb & 1));
        asm volatile("prefetch.global.L1 [%0];" ::"l"(p.cell_start + oc));
        asm volatile("prefetch.global.L1 [%0];" ::"l"(p.band_count + oc));
    }
    int32_t *slot = &p.cell_active[(size_t)g2 * p.wl_stride + cc];
    int old;
    if (e >= 0) { old = atomicExch(slot, e + 2); p.esc_next[e * 8 + g2] = old; }
    else old = atomicCAS(slot, 0, 1);
    if (old == 0) { /* new on the worklist: the resolution has to search it */
        const size_t w = (size_t)g2 * p.wl_stride + atomicAdd(&p.wl_count[g2], 1);
        write_work_item(p, p.wl + w * AMC_WI, cc, cx, cy, cz);
        p.wl_hit[w * AMC_HIT_REC] = -1;
    } else atomicOr(&p.cell_n[(size_t)g2 * p.wl_stride + cc], AMC_CELL_DIRTY); /* already listed by k_detect: its pair list is stale */
}

// elastic exchange of one overlapping pair (Pore:176-241), executed by all 32 lanes of warp 0.
// m1 = member with the smaller global index (the reference's particle "1" = j), m2 the larger.
// The arithmetic is evaluated redundantly (and identically) on every lane; what follows it is a set of
// independent global-memory round trips -- state stores, histogram updates of the completed paths,
// per-(particle, later colour group) cell activation -- which the lanes issue side by side instead of
// one thread walking through them: the latency of a collision is what a launch of k_pairs_group waits for.
__device__ __forceinline__ void resolve_pair(const P &p, CellShared &S, int m1, int m2, int group, int cell)
{
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, w = lane & 1; /* even lanes hold particle 1's record, odd lanes particle 2's */
    const Arrays &A = p.a;
    const int s1 = S.slot[m1], s2 = S.slot[m2];
    const int so = w ? s2 : s1, mo = w ? m2 : m1;
    // The tail of this function walks through small tables with dependent loads (owner cell of the new position,
    // member cells of the later groups, histogram edges).  The collision moves a particle by a fraction of the
    // collision range, so the entries it will need are the ones around the OLD position: touch them now, while
    // the velocity records are on their way, and the dependent loads become L1 hits.
    if (lane < 12) {
        const int ax = (lane >> 1) % 3, tbl = lane / 6;
        const double v = ax == 0 ? S.x[mo] : (ax == 1 ? S.y[mo] : S.z[mo]);
        const int nc = p.nc[ax];
        int o = (int)((v - p.e0[ax]) * p.inv_d[ax]);
        o = max(0, min(nc - 1, o));
        const double *t0 = (tbl ? p.lo[ax] : p.edge[ax]) + max(0, o - 1), *t1 = (tbl ? p.lo[ax] : p.edge[ax]) + min(nc - 1, o + 2);
        asm volatile("prefetch.global.L1 [%0];" ::"l"(t0));
        asm volatile("prefetch.global.L1 [%0];" ::"l"(t1));
    } else if (lane < 25) {
        asm volatile("prefetch.global.L1 [%0];" ::"l"(p.hist_edges + min(16 * (lane - 12), AMC_NUM_BINS)));
    } else if (lane < 27 && p.pp_mode == AMC_PP_GROUPS) {
        const int e = S.src[lane == 25 ? m1 : m2];
        if (e < 0) {
            const int nb = -1 - e;
            const int oc = ((S.kx + 1 - (nb >> 2)) * p.pnc[1] + (S.ky + 1 - ((nb >> 1) & 1))) * p.pnc[2] + (S.kz + 1 - (nb & 1));
            asm volatile("prefetch.global.L1 [%0];" ::"l"(p.cell_start + oc));
            asm volatile("prefetch.global.L1 [%0];" ::"l"(p.band_count + oc));
        }
    }
    const double ovx = __ldcg(A.vx + so), ovy = __ldcg(A.vy + so), ovz = __ldcg(A.vz + so), od = __ldcg(A.d + so), odx = __ldcg(A.dx + so),
                 ody = __ldcg(A.dy + so), odz = __ldcg(A.dz + so);
    uint32_t of = __ldcg(&A.pos[so].flag);
    const double qvx = __shfl_xor_sync(FULL, ovx, 1), qvy = __shfl_xor_sync(FULL, ovy, 1), qvz = __shfl_xor_sync(FULL, ovz, 1);
    double x1 = S.x[m1], y1 = S.y[m1], z1 = S.z[m1], x2 = S.x[m2], y2 = S.y[m2], z2 = S.z[m2];
    const double vx1 = w ? qvx : ovx, vy1 = w ? qvy : ovy, vz1 = w ? qvz : ovz;
    const double vx2 = w ? ovx : qvx, vy2 = w ? ovy : qvy, vz2 = w ? ovz : qvz;
    const double oldx = w ? x2 : x1, oldy = w ? y2 : y1, oldz = w ? z2 : z1; /* the own particle before the collision */
    double ddx = x2 - x1, ddy = y2 - y1, ddz = z2 - z1;
    double rx = -vx2 + vx1, ry = -vy2 + vy1, rz = -vz2 + vz1;
    double a = (rx * rx + ry * ry) + rz * rz;
    double b = 2 * ((ddx * rx + ddy * ry) + ddz * rz);
    double c = ((ddx * ddx + ddy * ddy) + ddz * ddz) - p.cr * p.cr;
    double disc = b * b - (4 * a) * c;
    if (!(disc >= 0.0) || a == 0.0) { if (lane == 0) atomicAdd(&p.stats->errors, 1ull); return; }
    double root = sqrt(disc);
    double t1 = (-b + root) / (2 * a), t2 = (-b - root) / (2 * a);
    double t = t1 > t2 ? t1 : t2;
    // completed free paths (Pore:186-199): lanes 0-3 the four values of particle 1, lanes 4-7 of particle 2
    {
        const uint32_t qf = __shfl_xor_sync(FULL, of, 1);
        const uint32_t f1 = w ? qf : of, f2 = w ? of : qf;
        const int done1 = (f1 & AMC_FLAG_PATH) != 0, done2 = (f2 & AMC_FLAG_PATH) != 0;
        // value `which` of the own particle, then routed to the lane that records it
        double mine[4];
        mine[0] = fabs(od - fabs(sqrt((ovx * ovx + ovy * ovy) + ovz * ovz) * t));
        mine[1] = fabs(odx - fabs(ovx * t)); mine[2] = fabs(ody - fabs(ovy * t)); mine[3] = fabs(odz - fabs(ovz * t));
        double val = 0.0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            double v = __shfl_sync(FULL, mine[k], (lane >> 2) & 1); /* lane 0 holds particle 1, lane 1 particle 2 */
            if ((lane & 3) == k) val = v;
        }
        unsigned long long base = 0;
        if (p.tap_path_count && lane == 0 && done1 + done2) base = atomicAdd(p.tap_path_count, (unsigned long long)(done1 + done2));
        base = __shfl_sync(FULL, base, 0);
        if (lane < 8) {
            const int pw = lane >> 2, which = lane & 3;
            if (pw ? done2 : done1) {
                hist_add(p, which, val);
                acc_add(p.path_sums + 2 * which, val, SC_L1, SC_L1I, SC_L2);
                if (which == 0) { atomicAdd(p.path_count, 1ull); atomicAdd(&p.stats->paths, 1ull); }
                if (p.tap_path_count) {
                    unsigned long long k = base + (pw ? (unsigned long long)done1 : 0ull);
                    if ((int64_t)k < p.path_cap) p.tap_paths[which][k] = val;
                }
            }
        }
        of |= AMC_FLAG_PATH;
    }
    double nx1 = x1 - vx1 * t, ny1 = y1 - vy1 * t, nz1 = z1 - vz1 * t;
    double nx2 = x2 - vx2 * t, ny2 = y2 - vy2 * t, nz2 = z2 - vz2 * t;
    double n0 = (nx2 - nx1) / p.cr, n1 = (ny2 - ny1) / p.cr, n2 = (nz2 - nz1) / p.cr;
    double pp = (((vx1 * n0 + vy1 * n1) + vz1 * n2) - ((vx2 * n0 + vy2 * n1) + vz2 * n2)) / p.mass;
    double pm = pp * p.mass;
    double wx1 = vx1 - pm * n0, wy1 = vy1 - pm * n1, wz1 = vz1 - pm * n2;
    double wx2 = vx2 + pm * n0, wy2 = vy2 + pm * n1, wz2 = vz2 + pm * n2;
    x1 = nx1 + wx1 * t; y1 = ny1 + wy1 * t; z1 = nz1 + wz1 * t;
    x2 = nx2 + wx2 * t; y2 = ny2 + wy2 * t; z2 = nz2 + wz2 * t;
    const double x = w ? x2 : x1, y = w ? y2 : y1, z = w ? z2 : z1; /* the own particle after the collision */
    if (lane < 2) {
        const double wx = w ? wx2 : wx1, wy = w ? wy2 : wy1, wz = w ? wz2 : wz1;
        S.x[mo] = x; S.y[mo] = y; S.z[mo] = z;
        A.pos[so].x = x; A.pos[so].y = y; A.pos[so].z = z;
        A.vx[so] = wx; A.vy[so] = wy; A.vz[so] = wz;
        A.d[so] = fabs(sqrt((wx * wx + wy * wy) + wz * wz) * t);
        A.dx[so] = fabs(wx * t); A.dy[so] = fabs(wy * t); A.dz[so] = fabs(wz * t);
    }
    if (lane == 0) {
        atomicAdd(&p.stats->pp, 1ull);
        if (p.pair_count) {
            unsigned long long k = atomicAdd(p.pair_count, 1ull);
            if ((int64_t)k < p.pair_cap) { p.pair_hi[k] = S.id[m2]; p.pair_lo[k] = S.id[m1]; p.pair_group[k] = group; p.pair_cell[k] = cell; }
        }
    }
    if (p.slab && lane < 2) {
        // slab decomposition: a moved particle that a neighbouring rank holds a copy of (or now
        // needs, because it entered the band at a cut / crossed it) is queued for the boundary
        // exchange that follows this colour group
        uint32_t &f = of;
        bool up = (f & AMC_FLAG_REL_UP) || z > p.up_thr, down = (f & AMC_FLAG_REL_DOWN) || z < p.down_thr;
        if ((up && !(f & AMC_FLAG_REL_UP)) || (down && !(f & AMC_FLAG_REL_DOWN))) {
            if (!(f & (AMC_FLAG_REL_UP | AMC_FLAG_REL_DOWN | AMC_FLAG_GHOST))) rel_insert(p, S.id[mo], so);
            f |= (up ? AMC_FLAG_REL_UP : 0u) | (down ? AMC_FLAG_REL_DOWN : 0u);
        }
        for (int dir = 0; dir < 2; dir++) {
            unsigned bit = dir == 0 ? AMC_FLAG_DIRTY_UP : AMC_FLAG_DIRTY_DOWN;
            if ((dir == 0 ? up : down) && !(f & bit)) { /* once per group and direction */
                f |= bit;
                int j = atomicAdd(&p.bnd_n[dir], 1);
                if (j < p.bnd_cap) p.bnd_dirty[dir][j] = so; else atomicAdd(p.slab_overflow + 2, 1ull);
            }
        }
    }
    if (lane < 2 && S.mv[mo] == 0) { /* the later colour groups learn about the move when the visit is over (activate_moved) */
        int i = atomicAdd(&S.nold, 1);
        if (i < AMC_MV_CAP) { S.ox[i] = oldx; S.oy[i] = oldy; S.oz[i] = oldz; }
        else { double *sp = p.mv_spill + ((size_t)blockIdx.x * AMC_MAX_MEMBERS + i) * 3; sp[0] = oldx; sp[1] = oldy; sp[2] = oldz; }
        S.mv[mo] = (uint16_t)(i + 1);
    }
    if (lane < 2) A.pos[so].flag = (uint8_t)of;
    __syncwarp();
}

// End of a cell visit in colour-group mode: every cell of a LATER colour group that contains a particle moved in
// this visit has to be visited too (k_detect only listed the cells that held an overlapping pair before the
// pass).  A moved particle whose owner cell changed can, in addition, no longer be found through the sorted
// layout: its member cell for every later group is published in the escaped list (esc_link).  Done once per
// moved particle with its final position, all warps side by side: two particles per warp and round, lane
// 8 * particle + g2 takes care of colour group g2.
__device__ __forceinline__ void activate_moved(const P &p, CellShared &S, const int group)
{
    const unsigned FULL = 0xffffffffu;
    const int tid = threadIdx.x, nthreads = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = nthreads >> 5;
    const int n = S.n;
    for (int k = tid; k < n; k += nthreads)
        if (S.mv[k]) S.nxt[atomicAdd(&S.nmv, 1)] = (uint16_t)k;
    __syncthreads();
    const int nmv = S.nmv;
    const Arrays &A = p.a;
    // the closing recapture has to look at every moved slot (touch_slot: two dependent global atomics): the last warp
    // does that beside the activation work of the first ones instead of in front of it
    if (warp == nwarps - 1)
        for (int i = lane; i < nmv; i += 32) touch_slot(p, S.slot[S.nxt[i]]);
    for (int base = 2 * warp; base < nmv; base += 2 * nwarps) {
        const int pw = (lane >> 3) & 1, g2 = lane & 7;
        int o[3] = {0, 0, 0}, q[3] = {0, 0, 0}, e = -1, e_old = -1, findable = 0, ok = 0;
        double x = 0, y = 0, z = 0, ux = 0, uy = 0, uz = 0;
        if (base + pw < nmv) {
            const int m = S.nxt[base + pw];
            x = S.x[m]; y = S.y[m]; z = S.z[m];
            const int io = S.mv[m] - 1;
            if (io < AMC_MV_CAP) { ux = S.ox[io]; uy = S.oy[io]; uz = S.oz[io]; }
            else { const double *sp = p.mv_spill + ((size_t)blockIdx.x * AMC_MAX_MEMBERS + io) * 3; ux = sp[0]; uy = sp[1]; uz = sp[2]; }
            if ((lane & 7) == 0 && lane < 16) { /* lanes 0 and 8: one per particle */
                const int so = S.slot[m];
                e_old = S.src[m];
                // Nine moved particles out of ten never leave the plain interior of the visited cell: read from the cell's
                // own owner segment (src == -1), inside that owner cell and outside every low-side band before and after
                // the visit.  Such a particle is a member of no other reference cell (member_axis: cell k only, parity of
                // the current group), nothing gains or loses it, and its sorted slot still finds it: nothing to do.
                bool fast = e_old == -1 && p.det_own_is_member;
                if (fast) {
                    const int kk[3] = {S.kx, S.ky, S.kz};
                    const double nv[3] = {x, y, z}, ov[3] = {ux, uy, uz};
#pragma unroll
                    for (int a = 0; a < 3; a++) {
                        const bool last = kk[a] + 1 >= p.nc[a];
                        const double clo = p.edge[a][kk[a]], blo = last ? 0.0 : p.lo[a][kk[a] + 1], hi = S.hi[a];
                        fast = fast && clo <= nv[a] && nv[a] < hi && (last || nv[a] <= blo) && clo <= ov[a] && ov[a] < hi && (last || ov[a] <= blo);
                    }
                }
                if (!fast) {
                int32_t k = owner_key(p, x, y, z, o);
                owner_key(p, ux, uy, uz, q);
                ok = 1;
                if (e_old < 0) { /* found through the sorted layout: src = -1 - (low-side neighbour code) */
                    int nb = -1 - e_old;
                    int oc = ((S.kx + 1 - (nb >> 2)) * p.pnc[1] + (S.ky + 1 - ((nb >> 1) & 1))) * p.pnc[2] + (S.kz + 1 - (nb & 1));
                    /* still findable through the sorted layout: same owner cell, and either it sits in the
                       band prefix of that cell or it is (still) outside every band */
                    findable = k == oc && (so < p.cell_start[oc] + p.band_count[oc] || !any_band(p, x, y, z, o));
                }
                if (!findable) { /* entries are never re-linked: a particle that moves again in a later visit gets a fresh one */
                    e = atomicAdd(p.esc_count, 1);
                    if (e >= p.esc_cap) { atomicAdd(&p.stats->esc_overflow, 1ull); ok = 0; }
                    else { p.esc_slot[e] = so; atomicOr(&A.pos[so].flag, AMC_FLAG_ESC); }
                }
                }
            }
        }
        const int src = pw * 8;
        const int o0 = __shfl_sync(FULL, o[0], src), o1 = __shfl_sync(FULL, o[1], src), o2 = __shfl_sync(FULL, o[2], src);
        const int q0 = __shfl_sync(FULL, q[0], src), q1 = __shfl_sync(FULL, q[1], src), q2 = __shfl_sync(FULL, q[2], src);
        const int ee = __shfl_sync(FULL, e, src), eo = __shfl_sync(FULL, e_old, src);
        const int fnd = __shfl_sync(FULL, findable, src), okk = __shfl_sync(FULL, ok, src);
        if (lane < 16 && g2 > group && okk) {
            int cx = member_axis(p.edge[0], p.lo[0], p.nc[0], o0, (g2 >> 2) & 1, x);
            int cy = member_axis(p.edge[1], p.lo[1], p.nc[1], o1, (g2 >> 1) & 1, y);
            int cz = member_axis(p.edge[2], p.lo[2], p.nc[2], o2, (g2 ^ p.zoff) & 1, z);
            int32_t cc = (cx < 0 || cy < 0 || cz < 0) ? -1 : ((cx >> 1) * p.nh[1] + (cy >> 1)) * p.nh[2] + (cz >> 1);
            if (eo >= 0) p.esc_cell[eo * 8 + g2] = -1; /* retire the entry the particle came in through */
            esc_link(p, g2, cc, cx, cy, cz, fnd ? -1 : ee);
            // the cell the particle was a member of before the visit loses it: its member count changed, so the
            // reference-equivalent test counter needs the visit even though no new overlap can arise there
            int dx = member_axis(p.edge[0], p.lo[0], p.nc[0], q0, (g2 >> 2) & 1, ux);
            int dy = member_axis(p.edge[1], p.lo[1], p.nc[1], q1, (g2 >> 1) & 1, uy);
            int dz = member_axis(p.edge[2], p.lo[2], p.nc[2], q2, (g2 ^ p.zoff) & 1, uz);
            int32_t dc = (dx < 0 || dy < 0 || dz < 0) ? -1 : ((dx >> 1) * p.nh[1] + (dy >> 1)) * p.nh[2] + (dz >> 1);
            if (dc >= 0 && dc != cc) esc_link(p, g2, dc, dx, dy, dz, -1);
        }
    }
}

// smallest pair key above `cur` among the overlapping pairs whose higher-index member this thread owns
__device__ __forceinline__ unsigned long long scan_min_key(const P &p, const CellShared &S, const int n, const unsigned long long cur)
{
    unsigned long long mine = ~0ull;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double xi = S.x[i], yi = S.y[i], zi = S.z[i];
        const int32_t idi = S.id[i];
        for (int j = 0; j < n; j++) {
            if (S.id[j] >= idi) continue; /* each unordered pair once, from its higher-index member */
            const unsigned long long key = pair_key(idi, S.id[j]);
            if (key > cur && key < mine && overlap(p, xi, yi, zi, S.x[j], S.y[j], S.z[j])) mine = key;
        }
    }
    return mine;
}

// Scan mode of cell_process: more pairs overlapped at once than the candidate list holds (a cell far denser than the gas
// this code is tuned for).  From here to the end of the visit every pick is a search over all member pairs for the
// smallest key above the cursor that overlaps right now -- the reference's own sweep order, at O(n^2 / threads) per
// collision.  Kept out of line: rare, and it must not weigh on the register budget of the normal visit.
__device__ __noinline__ void scan_mode_resolve(const P &p, CellShared &S, const int n, const int group, const int cell)
{
    const int tid = threadIdx.x, nthreads = blockDim.x, lane = tid & 31, warp = tid >> 5;
    while (true) {
        if (tid == 0) S.best_key = ~0ull;
        __syncthreads();
        const unsigned long long mine = scan_min_key(p, S, n, S.cursor);
        if (tid == 0) atomicAdd(&S.nexec, (unsigned int)min((long long)n * (n - 1) / 2, 0x7fffffffLL));
        if (mine != ~0ull) atomicMin(&S.best_key, mine);
        __syncthreads();
        const unsigned long long bk = S.best_key;
        if (bk == ~0ull) break;
        for (int k = tid; k < n; k += nthreads) {
            if ((uint32_t)S.id[k] == (uint32_t)(bk >> 32)) S.moved_b = k;      /* higher index: the reference's particle 2 */
            if ((uint32_t)S.id[k] == (uint32_t)(bk & 0xffffffffull)) S.moved_a = k;
        }
        __syncthreads();
        if (warp == 0) {
            resolve_pair(p, S, S.moved_a, S.moved_b, group, cell);
            if (lane == 0) S.cursor = bk;
        }
        __syncthreads();
    }
}

// members are in S.{x,y,z,id,slot,src}[0..S.n); all threads of the block call this
__device__ __forceinline__ void cell_process(const P &p, CellShared &S, int group, int cell)
{
    const int n = S.n, tid = threadIdx.x, nthreads = blockDim.x;
    const int lane = tid & 31, warp = tid >> 5;
    if (tid == 0) S.nref += (unsigned long long)n * (n - 1) / 2;
    // A cell that is here only because k_detect found overlapping-looking pairs in it, and that no particle has
    // entered or left since, needs no search: the listed pairs (slots -> member indices) are all there is to test.
    bool listed = false;
    if (S.use_hits) { /* block-uniform */
        const int nh2 = 2 * S.hits[0];
        for (int k = tid; k < n; k += nthreads) {
            S.mv[k] = 0;
            const int sl = S.slot[k];
            for (int h = 0; h < nh2; h++)
                if (S.hits[1 + h] == sl) S.hm[h] = k;
        }
        if (tid == 0) { S.nmv = 0; S.nold = 0; }
        __syncthreads();
        listed = true;
        for (int h = 0; h < nh2; h++) listed = listed && S.hm[h] >= 0; /* all found (always, unless the state is inconsistent) */
        if (listed) {
            if (2 * tid < nh2) {
                const int ma = S.hm[2 * tid], mb = S.hm[2 * tid + 1];
                if (overlap(p, S.x[ma], S.y[ma], S.z[ma], S.x[mb], S.y[mb], S.z[mb])) push_cand(S, p, ma, mb);
            }
            if (tid == 0) atomicAdd(&S.nexec, (unsigned int)(nh2 >> 1));
            __syncthreads();
        }
    }
    if (!listed) {
    // Only cells that the detection pass flagged (or that received a moved particle) get here, so what counts is
        // the latency of one visit.  Members are chained per slab along x (one shared-memory exchange each, no scan,
        // no reordering); after one barrier every member walks the older entries of its own slab and the whole next
        // slab.  A pair goes through the fp32 filter of k_detect first (cell-relative coordinates, threshold det_thr)
        // and only the few that pass are decided by the exact test (Pore:173-174).
        {
            // the fp32 cell-relative coordinates of the filter are formed from the fp64 members where they are needed (a
            // copy of them would cost 6 KB of the CTA's shared memory, i.e. resident CTAs)
            const float inv_w = S.inv_w, thr = p.det_thr;
            const double org0 = S.org[0], org1 = S.org[1], org2 = S.org[2];
            const int nb1 = S.nb - 1;
            for (int k = tid; k < n; k += nthreads) {
                float fx = (float)(S.x[k] - org0);
                int b = min(nb1, max(0, (int)(fx * inv_w)));
                S.nxt[k] = (uint16_t)atomicExch(&S.head[b], k + 1);
                S.mv[k] = 0;
            }
            if (tid == 0) { S.nmv = 0; S.nold = 0; }
            PHASE_MARK(9); /* chain: own work */
            __syncthreads();
            PHASE_MARK(2); /* chain: barrier */
            unsigned int mine = 0;
            for (int k0 = tid; k0 < n; k0 += WALK_K * nthreads) {
                // WALK_K members per thread walk their chains side by side: every round is one hop for each of them
                float ax[WALK_K], ay[WALK_K], az[WALK_K];
                int e[WALK_K], more[WALK_K];
#pragma unroll
                for (int u = 0; u < WALK_K; u++) {
                    const int k = k0 + u * nthreads;
                    e[u] = 0; more[u] = 0; ax[u] = ay[u] = az[u] = 0.f;
                    if (k < n) {
                        ax[u] = (float)(S.x[k] - org0); ay[u] = (float)(S.y[k] - org1); az[u] = (float)(S.z[k] - org2);
                        const int b = min(nb1, max(0, (int)(ax[u] * inv_w)));
                        e[u] = S.nxt[k]; more[u] = S.head[b + 1];
                    }
                }
                while (true) {
                    int live = 0;
#pragma unroll
                    for (int u = 0; u < WALK_K; u++) {
                        if (e[u] == 0) { e[u] = more[u]; more[u] = 0; }
                        live |= e[u];
                    }
                    if (live == 0) break;
#pragma unroll
                    for (int u = 0; u < WALK_K; u++) {
                        const int q = max(e[u] - 1, 0); /* entry 0 stands in for a finished chain; its result is masked */
                        const float ex = (float)(S.x[q] - org0) - ax[u], ey = (float)(S.y[q] - org1) - ay[u], ez = (float)(S.z[q] - org2) - az[u];
                        const int nx = S.nxt[q];
                        const float d2 = fmaf(ez, ez, fmaf(ey, ey, ex * ex));
                        if (e[u] != 0 && d2 < thr) { /* rare */
                            const int k = k0 + u * nthreads;
                            if (overlap(p, S.x[k], S.y[k], S.z[k], S.x[q], S.y[q], S.z[q])) push_cand(S, p, k, q);
                        }
                        mine += e[u] != 0;
                        e[u] = e[u] != 0 ? nx : 0;
                    }
                }
            }
            PHASE_MARK(10); /* walk: own work */
            mine = __reduce_add_sync(0xffffffffu, mine);
            if (lane == 0 && mine) atomicAdd(&S.nexec, mine);
        }
        __syncthreads();
        for (int c = tid; c < AMC_XBINS + 2; c += nthreads) S.head[c] = 0; /* every walk is done; the barriers of the caller order this before the next cell */
    }
    PHASE_MARK(5); /* search */
    if (S.ncand == 0) return;
    if (tid == 0) { S.cursor = 0; S.done = 0; if (S.ncand > AMC_MAX_CAND) S.ncand = AMC_MAX_CAND; }
    __syncthreads();
    while (true) {
        if (S.cand_lost) { scan_mode_resolve(p, S, n, group, cell); break; } /* block-uniform; rare */
        if (warp == 0) { /* warp-uniform: every lane scans the (few) candidates itself */
            int best = -1;
            unsigned long long bk = ~0ull;
            for (int k = 0; k < S.ncand; k++)
                if (S.cand_key[k] < bk) { bk = S.cand_key[k]; best = k; } /* all stored keys are above the cursor */
            if (best < 0) { if (lane == 0) S.done = 1; }
            else {
                int a = S.cand_ab[best] & 0xffff, b = S.cand_ab[best] >> 16;
                int m1 = S.id[a] < S.id[b] ? a : b, m2 = S.id[a] < S.id[b] ? b : a;
                PHASE_MARK(6); /* pick */
                resolve_pair(p, S, m1, m2, group, cell);
                PHASE_MARK(8); /* resolve_pair */
                if (lane == 0) {
                    S.cursor = bk; S.moved_a = a; S.moved_b = b;
                    int w = 0;
                    for (int k = 0; k < S.ncand; k++) {
                        int ka = S.cand_ab[k] & 0xffff, kb = S.cand_ab[k] >> 16;
                        if (ka == a || ka == b || kb == a || kb == b) continue;
                        S.cand_key[w] = S.cand_key[k]; S.cand_ab[w] = S.cand_ab[k]; w++;
                    }
                    S.ncand = w;
                }
            }
        }
        __syncthreads();
        if (S.done) break;
        {
            int a = S.moved_a, b = S.moved_b;
            unsigned long long cur = S.cursor;
            double xa = S.x[a], ya = S.y[a], za = S.z[a], xb = S.x[b], yb = S.y[b], zb = S.z[b];
            for (int k = tid; k < n; k += nthreads) {
                if (k == a || k == b) continue;
                double xk = S.x[k], yk = S.y[k], zk = S.z[k];
                if (pair_key(S.id[a], S.id[k]) > cur && overlap(p, xa, ya, za, xk, yk, zk)) push_cand(S, p, a, k);
                if (pair_key(S.id[b], S.id[k]) > cur && overlap(p, xb, yb, zb, xk, yk, zk)) push_cand(S, p, b, k);
            }
            if (tid == 0) atomicAdd(&S.nexec, (unsigned int)(2 * (n - 2)));
        }
        __syncthreads();
        if (tid == 0 && S.ncand > AMC_MAX_CAND) S.ncand = AMC_MAX_CAND;
        __syncthreads();
    }
    if (p.pp_mode == AMC_PP_GROUPS) activate_moved(p, S, group);
}

// Detection list of one pair pass: every reference cell whose 8 candidate owner cells hold at least two
// particles (all colour groups together).  k_detect turns it into the per-group worklists of the cells
// that can hold a collision; cells that later receive a moved particle are appended by resolve_pair /
// k_bnd_apply.  One thread per reference cell.
__global__ void __launch_bounds__(ADVECT_THREADS) k_build_worklist(const __grid_constant__ P p)
{
    __shared__ int s_cnt, s_base;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    int cid = blockIdx.x * blockDim.x + threadIdx.x; /* linear over (kx, ky, kz), z fastest */
    int ncell = p.nc[0] * p.nc[1] * p.nc[2];
    int kz = 0, ky = 0, kx = 0, total = 0; /* upper bound of the member count: own owner cell + band prefixes of the 7 lower neighbours */
    if (cid < ncell) {
        kz = cid % p.nc[2]; ky = (cid / p.nc[2]) % p.nc[1]; kx = cid / (p.nc[2] * p.nc[1]);
#pragma unroll
        for (int nb = 0; nb < 8; nb++) {
            int oc = ((kx + 1 - (nb >> 2)) * p.pnc[1] + (ky + 1 - ((nb >> 1) & 1))) * p.pnc[2] + (kz + 1 - (nb & 1));
            total += nb == 0 ? p.cell_start[oc + 1] - p.cell_start[oc] : p.band_count[oc];
        }
    }
    // one global atomic per block: the list counter is a single address
    const bool active = total >= 2;
    const unsigned bal = __ballot_sync(0xffffffffu, active);
    const int lane = threadIdx.x & 31;
    int mine = 0;
    if (lane == 0 && bal) mine = atomicAdd(&s_cnt, __popc(bal));
    mine = __shfl_sync(0xffffffffu, mine, 0) + __popc(bal & ((1u << lane) - 1));
    __syncthreads();
    if (threadIdx.x == 0 && s_cnt) s_base = atomicAdd(p.dl_count, s_cnt);
    __syncthreads();
    if (active) {
        int cell = ((kx >> 1) * p.nh[1] + (ky >> 1)) * p.nh[2] + (kz >> 1);
        write_work_item(p, p.dl + (size_t)(s_base + mine) * AMC_WI, cell, kx, ky, kz);
    }
}

// ------------------------------------------------------------------------------------------------
// Detection pass (the neighbour search proper): ONE launch over every reference cell of all 8 colour
// groups, on the positions as they are before the first group runs.  A cell visit of the reference
// (Pore:160-255) changes nothing unless two of its members overlap, and the members of a cell only
// change when a collision moves one of them -- so the ordered resolution (k_pairs_group) has to visit
//   (a) the cells in which this pass finds an overlapping pair, and
//   (b) the cells of later groups that contain a particle moved by a collision (activated there).
// Everything here is a conservative filter: cell membership is decided exactly (fp64, Pore:527-529),
// distances are tested in fp32 on cell-relative coordinates against a threshold widened by the
// rounding bound (det_thr, amc_api.cu), and anything unusual (more candidates than the CTA holds, a
// full slab) flags the cell.  False positives cost one exact visit; misses are impossible.
//
// Per cell: the candidates are 8 runs of consecutive position records (the owner cell, the band prefixes of its 7
// low-side neighbours), so the header warp hands each run to cp.async.bulk (one 1-D bulk copy per run, SASS UBLKCP) and
// the records land in shared memory while the CTA searches the previous cell; an mbarrier with a transaction count tells
// the CTA when all of them are there.  No thread computes a candidate's slot (det_slot) or issues a global load for it,
// and nothing of the next cell lives in registers during the search.  Members are hashed into a 2-D table of bins over
// (x, y), >= 1.05 filter radii wide along x and twice that along y: at gas density a bin holds about 0.14 particles,
// so a member only looks at its own bin and the four forward neighbours and almost never finds anything to test.
// Table entries carry the visit number in their upper half, so the table is never cleared.  Two barriers per cell.
// 128 threads x 3 candidates at 64 registers and 27.9 KB of shared memory: 8 CTAs per SM.
#define DET_THREADS 128
#define DET_K 3     /* candidates per thread: cells with more than DET_K * DET_THREADS candidates are flagged */
#define DET_CAND (DET_K * DET_THREADS)
#define DET_NB 64   /* bins along x, at most */
#define DET_OCC 8   /* resident CTAs per SM the kernel is compiled for */

struct DetShared {
    static constexpr int NBX = DET_NB, NBY = 32;           /* bins along x / y, at most */
    static constexpr float YF = 2.0f;                       /* width of a y bin in units of the minimal bin width */
    static constexpr int ROW = NBY + 2, TAB = (NBX + 1) * ROW; /* one empty bin on either side of a row, one empty row behind the last */
    unsigned int head[TAB];          /* (visit tag << 16) | (candidate index + 1) of the last member hashed into the bin */
    float4 tile[DET_CAND];           /* by candidate index: cell-relative fp32 position; .w = older member of the same bin (index + 1 as integer bits), 0 = none */
    __align__(128) PosRec raw[DET_CAND]; /* records of the cell about to be searched: written by the bulk copies only */
    __align__(16) int hdr[2][AMC_WI];
    int rbeg[2][8], rcum[2][9];
    float inv_wx[2], inv_wy[2];
    int nbx[2], nby[2];
    int nmem[2];
    int nhit[2];
    unsigned int hit[2][AMC_MAX_HITS]; /* candidate indices of the pairs that passed the filter: (self << 16) | other */
    __align__(8) unsigned long long bar; /* mbarrier: one arrival (the header warp's expect_tx) + the bytes of the copies */
};

// header warp: make the work item `v` (one int per lane) the header in buffer `buf`
__device__ __forceinline__ void det_publish(const P &p, DetShared &S, int buf, int v, int lane)
{
    S.hdr[buf][lane] = v;
    __syncwarp();
    if (lane < 8) {
        S.rbeg[buf][lane] = S.hdr[buf][4 + lane];
        int inc = S.hdr[buf][12 + lane];
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) { int t = __shfl_up_sync(0xffu, inc, o); if (lane >= o) inc += t; }
        S.rcum[buf][lane + 1] = inc;
        if (lane < 2) { /* lane 0: bins along x, lane 1: along y */
            const double *d = reinterpret_cast<const double *>(&S.hdr[buf][20]);
            float wd = (float)(d[2 * lane + 1] - d[2 * lane]);
            int nb = lane == 0 ? (int)fminf((float)DetShared::NBX, floorf(wd / p.det_w)) : (int)fminf((float)DetShared::NBY, floorf(wd / (DetShared::YF * p.det_w)));
            if (nb < 1) nb = 1;
            if (lane == 0) { S.nbx[buf] = nb; S.inv_wx[buf] = (float)nb / wd; S.rcum[buf][0] = 0; }
            else { S.nby[buf] = nb; S.inv_wy[buf] = (float)nb / wd; }
        }
    }
}

// slot of candidate t of the work item in buffer `buf`: the owner cell's own particles first, then the
// band prefixes of the 7 low-side neighbours
__device__ __forceinline__ int det_slot(const DetShared &S, int buf, int t)
{
    if (t < S.rcum[buf][1]) return S.rbeg[buf][0] + t;
    int nb = 1;
#pragma unroll
    for (int r = 2; r < 8; r++) nb += t >= S.rcum[buf][r];
    return S.rbeg[buf][nb] + (t - S.rcum[buf][nb]);
}

// Overlap-free seeding (amc_seed_relax), both out of line: the detection pass of a timestep never gets here.
// A pair that passed the fp32 filter: exact test (Pore:173-174); the particle with the higher index is marked.
__device__ __noinline__ void det_seed_mark(const P &p, const int sa, const int sb)
{
    const Arrays &A = p.a;
    if (overlap(p, A.pos[sa].x, A.pos[sa].y, A.pos[sa].z, A.pos[sb].x, A.pos[sb].y, A.pos[sb].z))
        if (atomicExch(&p.rank[A.pos[sa].id > A.pos[sb].id ? sa : sb], 1) == 0) atomicAdd(&p.stats->pp, 1ull);
}
// A cell with more candidates than the tile holds is not copied; seeding searches it pair by pair on the fp64 positions
// (one-time work at initialisation; the timestep leaves such cells to the ordered resolution).
__device__ __noinline__ void det_seed_big_cell(const P &p, const DetShared &S, const int cur, const int total)
{
    const Arrays &A = p.a;
    const double *bd = reinterpret_cast<const double *>(&S.hdr[cur][20]);
    for (int i = threadIdx.x; i < total; i += DET_THREADS) {
        const int si = det_slot(S, cur, i);
        const double xi = A.pos[si].x, yi = A.pos[si].y, zi = A.pos[si].z;
        if (!(bd[0] < xi && xi < bd[1] && bd[2] < yi && yi < bd[3] && bd[4] < zi && zi < bd[5])) continue;
        for (int j = 0; j < i; j++) {
            const int sj = det_slot(S, cur, j);
            const double xj = A.pos[sj].x, yj = A.pos[sj].y, zj = A.pos[sj].z;
            if (!(bd[0] < xj && xj < bd[1] && bd[2] < yj && yj < bd[3] && bd[4] < zj && zj < bd[5])) continue;
            if (overlap(p, xi, yi, zi, xj, yj, zj))
                if (atomicExch(&p.rank[A.pos[si].id > A.pos[sj].id ? si : sj], 1) == 0) atomicAdd(&p.stats->pp, 1ull);
        }
    }
}

__device__ __forceinline__ uint32_t smem_u32(const void *q) { return (uint32_t)__cvta_generic_to_shared(q); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, const int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, const uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, const uint32_t bytes, unsigned long long *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(__cvta_generic_to_global(src)), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// false when the phase did not complete within ~1 s (a byte count that does not match the copies): the caller reports it
__device__ __forceinline__ bool mbar_wait(unsigned long long *bar, const uint32_t parity)
{
    for (unsigned int spins = 0; spins < (1u << 22); spins++) {
        uint32_t ok;
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok)
                     : "r"(smem_u32(bar)), "r"(parity)
                     : "memory");
        if (ok) return true;
    }
    return false;
}

// header warp: start the bulk copies of the candidates of the work item in header buffer `buf` (published and
// barrier-separated from here).  A cell with more candidates than the tile holds is not copied: it is flagged unseen.
__device__ __forceinline__ void det_fetch(const P &p, DetShared &S, const int buf, const int lane)
{
    const int total = S.rcum[buf][8];
    const bool fits = total <= DET_CAND;
    if (lane == 0) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); /* the threads' reads of S.raw (behind a barrier) before the engine's writes */
        mbar_expect_tx(&S.bar, fits ? (uint32_t)total * (uint32_t)sizeof(PosRec) : 0u);
    }
    __syncwarp();
    if (fits && lane < 8) {
        const int beg = S.rcum[buf][lane], len = S.rcum[buf][lane + 1] - beg;
        if (len > 0) bulk_g2s(&S.raw[beg], p.a.pos + S.rbeg[buf][lane], (uint32_t)len * (uint32_t)sizeof(PosRec), &S.bar);
    }
}

template <bool SEED> /* SEED: the marking variant of amc_seed_relax; the detection pass of a timestep is k_detect_tma<false> */
__global__ void __launch_bounds__(DET_THREADS, DET_OCC) k_detect_tma(const __grid_constant__ P p)
{
    __shared__ DetShared S;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nwork = *p.dl_count;
    const int stride = gridDim.x;
    int w = blockIdx.x;
    if (w >= nwork) return;
    for (int c = tid; c < DetShared::TAB; c += DET_THREADS) S.head[c] = 0;
    if (tid < 2) { S.nmem[tid] = 0; S.nhit[tid] = 0; }
    if (tid == 0) mbar_init(&S.bar, 1);
    const bool hw = warp == DET_THREADS / 32 - 1; /* header warp: the tail of the candidate list, least to do */
    int hn = 0;
    if (hw) {
        det_publish(p, S, 0, p.dl[(size_t)w * AMC_WI + lane], lane);
        if (w + stride < nwork) hn = p.dl[(size_t)(w + stride) * AMC_WI + lane];
    }
    __syncthreads();
    if (hw) det_fetch(p, S, 0, lane);
    unsigned int tests = 0;
    unsigned long long nref = 0; /* header warp, lane 0 */
    const float thr = p.det_thr;
    unsigned int tagw = 0;
    uint32_t phase = 0;
    bool stuck = false;
    for (int it = 0; w < nwork; it++, w += stride) {
        const int cur = it & 1, nxt = cur ^ 1;
        tagw += 0x10000u;
        if (tagw == 0) { /* visit tags exhausted: start over with a clean table */
            __syncthreads();
            for (int c = tid; c < DetShared::TAB; c += DET_THREADS) S.head[c] = 0;
            tagw = 0x10000u;
            __syncthreads();
        }
        const int total = S.rcum[cur][8];
        const bool big = total > DET_CAND;
        bool hit = big;
        if (SEED && big) det_seed_big_cell(p, S, cur, total);
        if (!mbar_wait(&S.bar, phase)) stuck = true; /* the records of this cell are in S.raw */
        phase ^= 1u;
        // ---- hash the members of the current cell
        float fx[DET_K], fy[DET_K], fz[DET_K];
        int bin[DET_K], older[DET_K];
        {
            const double *bd = reinterpret_cast<const double *>(&S.hdr[cur][20]);
            const double lox = bd[0], hix = bd[1], loy = bd[2], hiy = bd[3], loz = bd[4], hiz = bd[5];
            const float inv_wx = S.inv_wx[cur], inv_wy = S.inv_wy[cur];
            const int nbx1 = S.nbx[cur] - 1, nby1 = S.nby[cur] - 1;
            const int own = p.det_own_is_member ? S.rcum[cur][1] : 0; /* the owner cell's particles are members by construction */
            int nm = 0;
#pragma unroll
            for (int k = 0; k < DET_K; k++) {
                const int t = tid + k * DET_THREADS;
                bin[k] = -1;
                if (t < total && !big) {
                    const double2 xy = *reinterpret_cast<const double2 *>(&S.raw[t]);
                    const double x = xy.x, y = xy.y, z = S.raw[t].z;
                    if (t < own || (lox < x && x < hix && loy < y && y < hiy && loz < z && z < hiz)) { /* Pore:527-530 */
                        fx[k] = (float)(x - lox); fy[k] = (float)(y - loy); fz[k] = (float)(z - loz);
                        int b = min(nbx1, (int)(fx[k] * inv_wx)) * DetShared::ROW + min(nby1, (int)(fy[k] * inv_wy)) + 1;
                        unsigned int prev = atomicExch(&S.head[b], tagw | (unsigned int)(t + 1)) ^ tagw;
                        prev = prev < 0x10000u ? prev : 0u;
                        S.tile[t] = make_float4(fx[k], fy[k], fz[k], __uint_as_float(prev));
                        bin[k] = b; older[k] = (int)prev;
                        nm++;
                    }
                }
            }
            nm = __reduce_add_sync(0xffffffffu, nm);
            if (lane == 0 && nm) atomicAdd(&S.nmem[cur], nm);
        }
        const int wn = w + stride;
        if (hw && wn < nwork) {
            det_publish(p, S, nxt, hn, lane);
            if (wn + stride < nwork) hn = p.dl[(size_t)(wn + stride) * AMC_WI + lane];
        }
        __syncthreads();
        // ---- every thread is done with S.raw: the next cell's records start their trip from HBM now
        if (hw && wn < nwork) det_fetch(p, S, nxt, lane);
        // ---- search: the older members of the own bin and everything in the four forward neighbour bins
#pragma unroll
        for (int k = 0; k < DET_K; k++) {
            if (bin[k] < 0) continue;
            const int b = bin[k];
            unsigned int c[5];
            c[0] = (unsigned int)older[k];
            c[1] = S.head[b + 1] ^ tagw; c[2] = S.head[b + DetShared::ROW - 1] ^ tagw;
            c[3] = S.head[b + DetShared::ROW] ^ tagw; c[4] = S.head[b + DetShared::ROW + 1] ^ tagw;
            if (c[0] == 0 && min(min(c[1], c[2]), min(c[3], c[4])) >= 0x10000u) continue;
            unsigned long long pend = c[0];
            int sh = c[0] ? 9 : 0;
#pragma unroll
            for (int n = 1; n < 5; n++)
                if (c[n] < 0x10000u) { pend |= (unsigned long long)c[n] << sh; sh += 9; }
            const unsigned long long all = pend;
            const float ax = fx[k], ay = fy[k], az = fz[k];
            float dmin = 3.0e38f;
            for (unsigned int e = 0;;) {
                if (e == 0) {
                    if (pend == 0) break;
                    e = (unsigned int)pend & 511u;
                    pend >>= 9;
                }
                float4 q = S.tile[e - 1];
                float ex = q.x - ax, ey = q.y - ay, ez = q.z - az;
                dmin = fminf(dmin, fmaf(ez, ez, fmaf(ey, ey, ex * ex)));
                tests++;
                e = __float_as_uint(q.w);
            }
            if (dmin < thr) { /* rare: walk the chains once more and remember the pairs for the ordered resolution */
                hit = true;
                pend = all;
                for (unsigned int e = 0;;) {
                    if (e == 0) {
                        if (pend == 0) break;
                        e = (unsigned int)pend & 511u;
                        pend >>= 9;
                    }
                    float4 q = S.tile[e - 1];
                    float ex = q.x - ax, ey = q.y - ay, ez = q.z - az;
                    if (fmaf(ez, ez, fmaf(ey, ey, ex * ex)) < thr) {
                        const int hh = atomicAdd(&S.nhit[cur], 1);
                        if (hh < AMC_MAX_HITS) S.hit[cur][hh] = ((unsigned int)(tid + k * DET_THREADS) << 16) | (e - 1);
                        if (SEED) det_seed_mark(p, det_slot(S, cur, tid + k * DET_THREADS), det_slot(S, cur, (int)e - 1));
                    }
                    e = __float_as_uint(q.w);
                }
            }
        }
        if (tid == DET_THREADS - 1) { S.nmem[nxt] = 0; S.nhit[nxt] = 0; }
        const int any = __syncthreads_or(hit);
        if (hw) {
            const int *h = S.hdr[cur];
            const int cell = h[0], kx = h[1], ky = h[2], kz = h[3];
            const int g = ((kx & 1) << 2) | ((ky & 1) << 1) | ((kz + p.zoff) & 1);
            const size_t ci = (size_t)g * p.wl_stride + cell;
            if (any) {
                int idx = 0;
                if (lane == 0) { p.cell_active[ci] = 1; idx = atomicAdd(&p.wl_count[g], 1); }
                idx = __shfl_sync(0xffffffffu, idx, 0);
                p.wl[((size_t)g * p.wl_stride + idx) * AMC_WI + lane] = h[lane];
                const int nh = S.nhit[cur];
                const bool listed = !big && nh >= 1 && nh <= AMC_MAX_HITS;
                int32_t *wh = p.wl_hit + ((size_t)g * p.wl_stride + idx) * AMC_HIT_REC;
                if (lane == 0) wh[0] = listed ? nh : -1;
                if (listed && lane < 2 * nh) {
                    const unsigned int hv = S.hit[cur][lane >> 1];
                    wh[1 + lane] = det_slot(S, cur, (lane & 1) ? (int)(hv & 0xffffu) : (int)(hv >> 16));
                }
            } else if (lane == 0) {
                const int nm = S.nmem[cur];
                p.cell_n[ci] = nm;
                nref += (unsigned long long)nm * (nm - 1) / 2;
            }
        }
    }
    tests = __reduce_add_sync(0xffffffffu, tests);
    if (lane == 0 && tests) atomicAdd(&p.stats->checks_exec, (unsigned long long)tests);
    if (hw && lane == 0 && nref) atomicAdd(&p.stats->checks_ref, nref);
    if (stuck) atomicAdd(&p.stats->cand_overflow, 1ull); /* reported by check_overflow: the results of this pass are not to be trusted */
}

// members of one reference cell of a colour group -> S.{x,y,z,id,slot,src}[0..S.n): its own register budget
__device__ __forceinline__ void gather_members(const P &p, CellShared &S, const int group, const int cell)
{
    const int tid = threadIdx.x;
    const Arrays &A = p.a;
    const double lox = S.org[0], hix = S.hi[0], loy = S.org[1], hiy = S.hi[1], loz = S.org[2], hiz = S.hi[2];
    {
            // membership is decided on the live position (Pore:527-530); the 8 ranges are walked as one
            // flat index space so every thread has independent loads in flight
            const int total = S.rcum[8];
            // particles that left their sorted owner cell earlier in this pass and are members of this cell now hang
            // on the cell's own list (head in cell_active, see esc_link): one load for nearly every cell
            int esc_head = 0;
            if (tid == PAIR_THREADS - 1) esc_head = __ldcg(p.cell_active + (size_t)group * p.wl_stride + cell);
            for (int tb = 0; tb < total; tb += PAIR_K * PAIR_THREADS) { /* PAIR_K candidates per thread in flight: one round trip for most cells */
                unsigned fl[PAIR_K]; double x[PAIR_K], y[PAIR_K], z[PAIR_K]; int id[PAIR_K];
#pragma unroll
                for (int k = 0; k < PAIR_K; k++) {
                    int t = tb + tid + k * PAIR_THREADS;
                    if (t < total) {
                        int nb = 0;
#pragma unroll
                        for (int r = 1; r < 8; r++) nb += t >= S.rcum[r];
                        int s = S.rbeg[nb] + (t - S.rcum[nb]);
                        /* past L1: with the fused hand-over another CTA of this launch may have updated the record */
                        const PosRec r = ldcg_pos(A.pos + s); /* the whole record: two 128-bit loads */
                        fl[k] = r.flag; x[k] = r.x; y[k] = r.y; z[k] = r.z; id[k] = r.id;
                    }
                }
                PHASE_MARK(11); /* gather: loads issued */
#pragma unroll
                for (int k = 0; k < PAIR_K; k++) {
                    int t = tb + tid + k * PAIR_THREADS;
                    bool mem = t < total && !(fl[k] & AMC_FLAG_ESC) && lox < x[k] && x[k] < hix && loy < y[k] && y[k] < hiy && loz < z[k] && z[k] < hiz;
                    unsigned bal = __ballot_sync(0xffffffffu, mem); /* one shared atomic per warp, not per member */
                    int base = 0;
                    if ((tid & 31) == 0 && bal) base = atomicAdd(&S.n, __popc(bal));
                    base = __shfl_sync(0xffffffffu, base, 0);
                    if (mem) {
                        int m = base + __popc(bal & ((1u << (tid & 31)) - 1));
                        if (m < AMC_MAX_MEMBERS) {
                            int nb = 0;
#pragma unroll
                            for (int r = 1; r < 8; r++) nb += t >= S.rcum[r];
                            S.x[m] = x[k]; S.y[m] = y[k]; S.z[m] = z[k]; S.id[m] = id[k];
                            S.slot[m] = S.rbeg[nb] + (t - S.rcum[nb]); S.src[m] = -1 - nb;
                        }
                    }
                }
            }
            PHASE_MARK(12); /* gather: members stored */
            for (int v = esc_head; v >= 2;) { /* thread PAIR_THREADS - 1 only */
                const int e = v - 2;
                v = __ldcg(p.esc_next + e * 8 + group);
                if (__ldcg(p.esc_cell + e * 8 + group) != cell) continue; /* the particle moved on since it was linked here */
                int s = __ldcg(p.esc_slot + e);
                int k = atomicAdd(&S.n, 1);
                if (k < AMC_MAX_MEMBERS) { const PosRec r = ldcg_pos(A.pos + s); S.x[k] = r.x; S.y[k] = r.y; S.z[k] = r.z; S.id[k] = r.id; S.slot[k] = s; S.src[k] = e; }
            }
        }
}

// one colour group (Pore:522-549): persistent CTAs walk the group's worklist
#define BND_HEAD_CTAS 8 /* CTAs per direction that apply the neighbours' records at the head of a fused k_pairs_group launch */
#ifdef AMC_SLAB_PROBE
// debug build (tools/gpu_trace.sh): wall-clock marks of a fused launch per colour group, ns since the first CTA started:
// [g][0] first CTA in, [1]/[2] hand-over from above / below applied, [3] last cut-adjacent visit done, [4] last visit done,
// [5] records sent, [6] hand-over records applied (count), [7] cut-adjacent visits (count)
__device__ unsigned long long g_probe[8][8];
__device__ __forceinline__ unsigned long long gtime() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define PROBE_MIN(g, k) do { if (threadIdx.x == 0) atomicMin(&g_probe[g][k], gtime()); } while (0)
#define PROBE_MAX(g, k) do { if (threadIdx.x == 0) atomicMax(&g_probe[g][k], gtime()); } while (0)
#define PROBE_ADD(g, k, v) do { if (threadIdx.x == 0) atomicAdd(&g_probe[g][k], (unsigned long long)(v)); } while (0)
#else
#define PROBE_MIN(g, k) do { } while (0)
#define PROBE_MAX(g, k) do { } while (0)
#define PROBE_ADD(g, k, v) do { } while (0)
#endif
__device__ __forceinline__ void bnd_pack_dir(const P &p, const int dir);                                                       /* slab section below */
__device__ __forceinline__ void bnd_apply_dir(const P &p, const int dir, const uint32_t seq, const int first, const int step);
__device__ __forceinline__ void bnd_pack_warp(const P &p, const int dir, const int lane);

// `fused` (peer-to-peer slab stepping): the hand-over with the neighbouring ranks rides inside this launch.  The first
// 2 x BND_HEAD_CTAS CTAs first apply the records the rank above / below sent after the previous group (waiting for them if need be) and then
// publish p.applied[dir]; the visits of cells in the two layers next to a cut wait for that, all other cells are
// processed meanwhile; the worklist may grow while the records are applied, so a CTA only leaves once both directions
// are applied and no ticket is left; the last CTA to finish packs this group's records straight into the neighbours'
// buffers and publishes p.bnd_seq there.
template <bool fused>
__global__ void __launch_bounds__(PAIR_THREADS, PAIR_OCC) k_pairs_group(const __grid_constant__ P p, const int group)
{
    __shared__ CellShared S;
    const int tid = threadIdx.x;
    if (fused) PROBE_MIN(group, 0);
    if (fused && blockIdx.x < 2 * BND_HEAD_CTAS) { /* BND_HEAD_CTAS CTAs per direction share the records; the last one done publishes */
        const int dir = blockIdx.x & 1;
        if (p.bnd_seq_apply) bnd_apply_dir(p, dir, p.bnd_seq_apply, blockIdx.x >> 1, BND_HEAD_CTAS);
        __syncthreads();
        if (tid == 0) {
            __threadfence();
            if (atomicAdd(p.pg_done + 1 + dir, 1) == BND_HEAD_CTAS - 1) {
                p.pg_done[1 + dir] = 0;
                __threadfence();
                asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p.applied + dir), "r"(p.bnd_seq) : "memory");
                PROBE_MAX(group, 1 + dir);
            }
        }
    }
    // single-domain launches of consecutive groups are programmatically dependent (run_pairs): the CTAs of group g + 1
    // become resident and clear their shared memory while the visits of group g still run, and go on when group g is complete
    if (!fused) pdl_trigger();
    __shared__ __align__(16) int s_hdr[AMC_WI];
    if (tid == 0) { S.nexec = 0; S.nref = 0; }
    for (int c = tid; c < AMC_XBINS + 2; c += PAIR_THREADS) S.head[c] = 0;
    if (!fused) pdl_wait(); /* nothing of the previous launch was read or written up to here */
    int nwork = fused ? __ldcg(p.wl_count + group) : p.wl_count[group];
    bool list_final = !fused;
    const int32_t *wl = p.wl + (size_t)group * p.wl_stride * AMC_WI;
    // warp 0 fetches a work item with one coalesced 128-byte load and already has the next one in flight
    // while the CTA works on the current cell
    // Work items are handed out dynamically (one atomic per cell on a per-group ticket) so a CTA that
    // drew cheap cells simply takes more of them; the ticket for the NEXT cell is drawn before the
    // current one is processed, which keeps its header load in flight.
    __shared__ int s_w;
    int next_hdr = 0, next_w = nwork;
    if (tid < AMC_WI) { /* the first item is the CTA's own index; further ones are drawn from the ticket counter */
        next_w = blockIdx.x;
        next_hdr = wl[(size_t)next_w * AMC_WI + tid]; /* unconditional (the slot exists): in flight together with the count */
        if (tid == 0) s_w = next_w;
    }
    __syncthreads();
    while (true) {
        if (s_w >= nwork) {
            if (list_final) break;
            // out of tickets while the hand-over may still add cells: wait until both directions are applied, then the list is final
            if (tid == 0) { flag_wait(p.applied + 0, p.bnd_seq); flag_wait(p.applied + 1, p.bnd_seq); }
            __syncthreads();
            list_final = true;
            nwork = __ldcg(p.wl_count + group);
            if (s_w >= nwork) break;
            if (tid < AMC_WI) next_hdr = __ldcg(wl + (size_t)s_w * AMC_WI + tid); /* this ticket was beyond the list when it was drawn */
        }
        __syncthreads(); /* previous cell fully processed before S is reused; everyone has read s_w */
#ifdef AMC_PHASE_CLOCK
        if (tid == 0) { S.t_last = clock64(); atomicAdd(&g_phase_clk[15], 1ull); }
#endif
        if (tid < AMC_WI) {
            s_hdr[tid] = next_hdr;
            if (fused || nwork > (int)gridDim.x) { /* more items than CTAs (or a list that can still grow): draw the next one */
                if (tid == 0) next_w = (int)gridDim.x + atomicAdd(&p.wl_next[group], 1);
                next_w = __shfl_sync(0xffffffffu, next_w, 0);
                if (next_w < nwork) next_hdr = wl[(size_t)next_w * AMC_WI + tid];
            } else next_w = nwork;
            __syncwarp();
            if (tid < 8) {
                S.rbeg[tid] = s_hdr[4 + tid];
                int inc = s_hdr[12 + tid];
#pragma unroll
                for (int o = 1; o < 8; o <<= 1) { int t = __shfl_up_sync(0xffu, inc, o); if (tid >= o) inc += t; }
                S.rcum[tid + 1] = inc;
            }
            if (tid < 3) {
                const double *d = reinterpret_cast<const double *>(s_hdr + 20);
                double lo = d[2 * tid], hi = d[2 * tid + 1];
                S.org[tid] = lo; S.hi[tid] = hi;
                if (tid == 0) { /* slabs along x, at least 1.05 filter radii wide */
                    float wd = (float)(hi - lo);
                    int nb = (int)fminf((float)AMC_XBINS, floorf(wd / p.det_w));
                    if (nb < 1) nb = 1;
                    S.nb = nb; S.inv_w = (float)nb / wd;
                    S.rcum[0] = 0; S.n = 0; S.ncand = 0; S.cand_lost = 0; S.kx = s_hdr[1]; S.ky = s_hdr[2]; S.kz = s_hdr[3];
                }
            }
        }
        __syncthreads();
        PHASE_MARK(0); /* header */
        const int cell = s_hdr[0];
        if (fused && !list_final) { /* a cell in the two layers next to a cut: its particles may be part of the hand-over being applied */
            const bool below = s_hdr[3] <= 1 && p.srank > 0, above = s_hdr[3] >= p.nc[2] - 2 && p.srank + 1 < p.nranks;
            if (below || above) {
                if (tid == 0) { if (below) flag_wait(p.applied + 1, p.bnd_seq); if (above) flag_wait(p.applied + 0, p.bnd_seq); }
                __syncthreads();
            }
        }
        if (tid >= PAIR_THREADS - 32 && (tid & 31) < AMC_HIT_REC) /* last warp: this item's pair list from k_detect */
            S.hits[tid & 31] = __ldcg(p.wl_hit + ((size_t)group * p.wl_stride + s_w) * AMC_HIT_REC + (tid & 31));
        if (tid < 2 * AMC_MAX_HITS) S.hm[tid] = -1;
        gather_members(p, S, group, cell);
        __syncthreads();
        PHASE_MARK(1); /* gather */
        if (S.n > AMC_MAX_MEMBERS) {
            __syncthreads();
            if (tid == 0) { atomicAdd(&p.stats->cell_overflow, 1ull); S.n = AMC_MAX_MEMBERS; }
            __syncthreads();
        }
        if (tid == 0) { /* the detection pass already counted this cell if it saw it without an overlapping pair */
            const int raw = __ldcg(p.cell_n + (size_t)group * p.wl_stride + cell);
            const int nA = raw & ~AMC_CELL_DIRTY;
            S.nref -= (unsigned long long)nA * (nA - 1) / 2;
            S.use_hits = S.hits[0] >= 0 && !(raw & AMC_CELL_DIRTY);
        }
        __syncthreads();
        if (S.n >= 2) cell_process(p, S, group, cell);
        PHASE_MARK(7); /* resolution loop (cells with candidates) */
#ifdef AMC_SLAB_PROBE
        if (fused) {
            const bool nearcut = (s_hdr[3] <= 1 && p.srank > 0) || (s_hdr[3] >= p.nc[2] - 2 && p.srank + 1 < p.nranks);
            if (nearcut) { PROBE_MAX(group, 3); PROBE_ADD(group, 7, 1); }
            PROBE_MAX(group, 4);
        }
#endif
        __syncthreads();
        if (tid == 0) s_w = next_w;
        __syncthreads();
    }
    __syncthreads();
    if (tid == 0) { /* one pair of global atomics per CTA instead of per cell */
        if (S.nref) atomicAdd(&p.stats->checks_ref, S.nref);
        if (S.nexec) atomicAdd(&p.stats->checks_exec, (unsigned long long)S.nexec);
    }
    if (fused) { /* the last CTA of the launch sends this group's records to the neighbours */
        __shared__ int s_last;
        if (tid == 0) { __threadfence(); s_last = atomicAdd(p.pg_done, 1) == (int)gridDim.x - 1; }
        __syncthreads();
        if (s_last) {
            __threadfence();
            if (tid < 64) bnd_pack_warp(p, tid >> 5, tid & 31); /* warp 0: up, warp 1: down */
            if (tid == 0) *p.pg_done = 0;
            __syncthreads();
            PROBE_MAX(group, 5);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Cube stage: serial sweep x -> y -> z over the cells with write-back after every cell; the x-layer
// membership is taken once per x layer, the y-layer membership once per column and the z-layer
// membership per cell, each from the positions live at that moment (Cube:232-238, 326-336).
// One CTA walks the cells in reference order; the particle state stays in original index order.
__global__ void __launch_bounds__(SWEEP_THREADS) k_cube_sweep(const __grid_constant__ P p)
{
    __shared__ CellShared S;
    __shared__ int nx, nxy;
    const int tid = threadIdx.x;
    const Arrays &A = p.a;
    int32_t *lx = p.key, *lxy = p.rank;
    if (!p.sw_state[0]) return; /* the event-driven sweep (k_sweep_detect / k_sweep_events) did this pass */
    if (tid == 0) { S.nexec = 0; S.nref = 0; }
    for (int c = tid; c < AMC_XBINS + 2; c += SWEEP_THREADS) S.head[c] = 0;
    for (int xl = 0; xl < p.nc[0]; xl++) {
        if (tid == 0) nx = 0;
        __syncthreads();
        {
            double lo = p.lo[0][xl], hi = p.edge[0][xl + 1];
            for (int i = tid; i < p.n; i += SWEEP_THREADS) {
                double v = A.pos[i].x;
                if (lo < v && v < hi) lx[atomicAdd(&nx, 1)] = i;
            }
        }
        __syncthreads();
        for (int yl = 0; yl < p.nc[1]; yl++) {
            if (tid == 0) nxy = 0;
            __syncthreads();
            {
                double lo = p.lo[1][yl], hi = p.edge[1][yl + 1];
                for (int k = tid; k < nx; k += SWEEP_THREADS) {
                    int i = lx[k];
                    double v = A.pos[i].y;
                    if (lo < v && v < hi) lxy[atomicAdd(&nxy, 1)] = i;
                }
            }
            __syncthreads();
            for (int zl = 0; zl < p.nc[2]; zl++) {
                if (tid == 0) {
                    S.n = 0; S.ncand = 0; S.cand_lost = 0; S.use_hits = 0; S.org[0] = p.lo[0][xl]; S.org[1] = p.lo[1][yl]; S.org[2] = p.lo[2][zl];
                    float wd = (float)(p.edge[0][xl + 1] - p.lo[0][xl]);
                    int nb = (int)fminf((float)AMC_XBINS, floorf(wd / p.det_w));
                    if (nb < 1) nb = 1;
                    S.nb = nb; S.inv_w = (float)nb / wd;
                }
                __syncthreads();
                {
                    double lo = p.lo[2][zl], hi = p.edge[2][zl + 1];
                    for (int k = tid; k < nxy; k += SWEEP_THREADS) {
                        int i = lxy[k];
                        double v = A.pos[i].z;
                        if (lo < v && v < hi) {
                            int m = atomicAdd(&S.n, 1);
                            if (m < AMC_MAX_MEMBERS) { S.x[m] = A.pos[i].x; S.y[m] = A.pos[i].y; S.z[m] = v; S.id[m] = i; S.slot[m] = i; S.src[m] = -1; }
                        }
                    }
                }
                __syncthreads();
                if (S.n > AMC_MAX_MEMBERS) {
                    if (tid == 0) { atomicAdd(&p.stats->cell_overflow, 1ull); S.n = AMC_MAX_MEMBERS; }
                    __syncthreads();
                }
                if (S.n >= 2) cell_process(p, S, 0, (xl * p.nc[1] + yl) * p.nc[2] + zl);
                __syncthreads();
            }
        }
    }
    if (tid == 0) {
        if (S.nref) atomicAdd(&p.stats->checks_ref, S.nref);
        if (S.nexec) atomicAdd(&p.stats->checks_exec, (unsigned long long)S.nexec);
    }
}

// ------------------------------------------------------------------------------------------------
// Event-driven form of the same serial sweep.  A cell visit changes nothing unless two members overlap, and a
// cell's members only change when a collision moves one of them, so of the 3,375 visits per timestep of the
// shipped cube ~60 matter.  Pass 1 (k_sweep_detect, one CTA per (x layer, y layer) column, all columns side by
// side) takes the positions as they are before the sweep: per column the particles inside the x and y masks, per
// cell the member count n0 and whether two members overlap (exact test) -> bitmap of flagged cells.  Pass 2
// (k_sweep_events, one CTA) walks the flagged cells in sweep order with cell_process; every particle a visit moved
// flags the LATER cells that hold it now or held it before the visit (their member set changed: a new overlap can
// arise and the reference-equivalent test counter needs the new count).  A skipped cell has, when the reference
// visits it, exactly the members pass 1 saw and no overlapping pair.
//
// The reference takes the x mask once per x layer, the y mask once per column and the z mask per cell, each from
// the positions live at that moment (Cube:233,235,237), so a particle moved inside a layer is still seen at its old
// x by the rest of that layer.  Moved particles (sw_tag == sw_pass, listed in sw_ml) therefore carry snapshots:
// sw_xs = the x the current layer's mask saw, sw_ys = the y the current column's mask saw, refreshed from the live
// position when the walk enters a new layer / column.  Everything else has not moved: live == what the masks saw.
// tests/cube_events_model.py is the Python restatement, checked against the oracle's serial sweep on the CPU.
#define SWD_THREADS 256
#define SWE_THREADS 256

// cells k of axis a with lo[k] < v < edge[k+1]: the owner cell and, inside its low-side band, the next one
__device__ __forceinline__ int axis_cells(const P &p, const int a, const double v, int out[2])
{
    const int nc = p.nc[a];
    const int o = owner_axis(p.edge[a], nc, p.e0[a], p.inv_d[a], v); /* -1 below edge[0], nc at / above edge[nc] or NaN */
    if (o >= nc) return 0;
    int cnt = 0;
    if (o >= 0 && p.lo[a][o] < v) out[cnt++] = o;
    if (o + 1 < nc && p.lo[a][o + 1] < v) out[cnt++] = o + 1;
    return cnt;
}

__global__ void __launch_bounds__(SWD_THREADS) k_sweep_detect(const __grid_constant__ P p)
{
    __shared__ double sx[AMC_MAX_MEMBERS], sy[AMC_MAX_MEMBERS], sz[AMC_MAX_MEMBERS];
    __shared__ int s_n, s_m;
    const int tid = threadIdx.x;
    const Arrays &A = p.a;
    const int col = blockIdx.x, xl = col / p.nc[1], yl = col % p.nc[1];
    int32_t *list = p.sw_col + (size_t)col * p.sw_colcap;
    if (tid == 0) s_n = 0;
    __syncthreads();
    {
        const double lox = p.lo[0][xl], hix = p.edge[0][xl + 1], loy = p.lo[1][yl], hiy = p.edge[1][yl + 1];
        for (int64_t i0 = tid; i0 < p.n; i0 += 4 * SWD_THREADS) { /* four particles per thread and round: their loads travel together */
            double x[4], y[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int64_t i = i0 + u * SWD_THREADS;
                x[u] = i < p.n ? A.pos[i].x : hix; y[u] = i < p.n ? A.pos[i].y : hiy;
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
                if (!(lox < x[u] && x[u] < hix && loy < y[u] && y[u] < hiy)) continue;
                const int k = atomicAdd(&s_n, 1);
                if (k < p.sw_colcap) list[k] = (int32_t)(i0 + u * SWD_THREADS);
            }
        }
    }
    __syncthreads();
    int ncol = s_n;
    if (ncol > p.sw_colcap) { /* more than the list holds: this pass is left to the plain sweep */
        if (tid == 0) atomicExch(&p.sw_state[0], 1ull);
        ncol = p.sw_colcap;
    }
    if (tid == 0) p.sw_col_n[col] = ncol;
    unsigned long long nref = 0; /* thread 0 */
    for (int zl = 0; zl < p.nc[2]; zl++) {
        if (tid == 0) s_m = 0;
        __syncthreads();
        const double loz = p.lo[2][zl], hiz = p.edge[2][zl + 1];
        for (int k = tid; k < ncol; k += SWD_THREADS) {
            const int i = list[k];
            const double z = A.pos[i].z;
            if (loz < z && z < hiz) {
                const int m = atomicAdd(&s_m, 1);
                if (m < AMC_MAX_MEMBERS) { sx[m] = A.pos[i].x; sy[m] = A.pos[i].y; sz[m] = z; }
            }
        }
        __syncthreads();
        const int nm = s_m;
        const int cell = (xl * p.nc[1] + yl) * p.nc[2] + zl;
        int hit = nm > AMC_MAX_MEMBERS; /* the visit reports the overflow */
        if (!hit)
            for (int a = tid; a < nm; a += SWD_THREADS)
                for (int b = 0; b < a; b++)
                    if (overlap(p, sx[a], sy[a], sz[a], sx[b], sy[b], sz[b])) hit = 1;
        hit = __syncthreads_or(hit);
        if (tid == 0) {
            p.cell_n[cell] = nm;
            nref += (unsigned long long)nm * (nm - 1) / 2;
            if (hit) atomicOr(reinterpret_cast<unsigned int *>(p.cell_active) + (cell >> 5), 1u << (cell & 31));
        }
    }
    if (tid == 0 && nref) atomicAdd(&p.sw_state[1], nref);
}

__global__ void __launch_bounds__(SWE_THREADS) k_sweep_events(const __grid_constant__ P p)
{
    __shared__ CellShared S;
    __shared__ int s_c, s_nml;
    const int tid = threadIdx.x, lane = tid & 31;
    const Arrays &A = p.a;
    if (p.sw_state[0]) return; /* a column list overflowed: k_cube_sweep does this pass */
    unsigned int *bits = reinterpret_cast<unsigned int *>(p.cell_active);
    const int ncell = p.nc[0] * p.nc[1] * p.nc[2], nwords = (ncell + 31) >> 5;
    if (tid == 0) { S.nexec = 0; S.nref = 0; s_nml = 0; s_c = 0; }
    for (int c = tid; c < AMC_XBINS + 2; c += SWE_THREADS) S.head[c] = 0;
    int cur_xl = -1, cur_col = -1;
    __syncthreads();
    while (true) {
        // ---- the next flagged cell at or behind the cursor (warp 0: 32 bitmap words per round)
        if (tid < 32) {
            const int c0 = s_c;
            int found = -1;
            for (int w0 = c0 >> 5; w0 < nwords && found < 0; w0 += 32) {
                const int w = w0 + lane;
                unsigned int v = w < nwords ? __ldcg(bits + w) : 0u; /* atomics land in L2 */
                if (w == (c0 >> 5)) v &= ~0u << (c0 & 31);
                const unsigned int bal = __ballot_sync(0xffffffffu, v != 0u);
                if (bal) {
                    const int src = __ffs(bal) - 1;
                    const unsigned int vv = __shfl_sync(0xffffffffu, v, src);
                    found = ((w0 + src) << 5) + __ffs(vv) - 1;
                }
            }
            if (lane == 0) s_c = found >= 0 && found < ncell ? found : -1;
        }
        __syncthreads();
        const int cell = s_c;
        if (cell < 0) break;
        const int zl = cell % p.nc[2], yl = (cell / p.nc[2]) % p.nc[1], xl = cell / (p.nc[2] * p.nc[1]);
        const int col = xl * p.nc[1] + yl;
        // ---- a new layer / column takes its mask from the live positions (Cube:233,235)
        if (xl != cur_xl || col != cur_col) {
            const int nml = s_nml;
            for (int k = tid; k < nml; k += SWE_THREADS) {
                const int i = p.sw_ml[k];
                if (xl != cur_xl) p.sw_xs[i] = A.pos[i].x;
                p.sw_ys[i] = A.pos[i].y;
            }
            cur_xl = xl; cur_col = col;
        }
        if (tid == 0) {
            S.n = 0; S.ncand = 0; S.cand_lost = 0; S.use_hits = 0; S.nold = 0; S.nmv = 0;
            S.org[0] = p.lo[0][xl]; S.org[1] = p.lo[1][yl]; S.org[2] = p.lo[2][zl];
            float wd = (float)(p.edge[0][xl + 1] - p.lo[0][xl]);
            int nb = (int)fminf((float)AMC_XBINS, floorf(wd / p.det_w));
            if (nb < 1) nb = 1;
            S.nb = nb; S.inv_w = (float)nb / wd;
        }
        __syncthreads();
        // ---- members: the column's particles that have not moved, and the moved ones through their snapshots
        {
            const double lox = p.lo[0][xl], hix = p.edge[0][xl + 1], loy = p.lo[1][yl], hiy = p.edge[1][yl + 1];
            const double loz = p.lo[2][zl], hiz = p.edge[2][zl + 1];
            const int ncol = p.sw_col_n[col], nml = s_nml;
            const int32_t *list = p.sw_col + (size_t)col * p.sw_colcap;
            for (int k = tid; k < ncol + nml; k += SWE_THREADS) {
                const int i = k < ncol ? list[k] : p.sw_ml[k - ncol];
                const int tag = p.sw_tag[i];                                /* one round trip for all four */
                const double z = A.pos[i].z, x = A.pos[i].x, y = A.pos[i].y;
                const bool tagged = tag == p.sw_pass;
                if (k < ncol && tagged) continue; /* comes through the moved list */
                if (!(loz < z && z < hiz)) continue;
                const double mx = tagged ? p.sw_xs[i] : x, my = tagged ? p.sw_ys[i] : y;
                if (!(lox < mx && mx < hix && loy < my && my < hiy)) continue;
                const int m = atomicAdd(&S.n, 1);
                if (m < AMC_MAX_MEMBERS) { S.x[m] = x; S.y[m] = y; S.z[m] = z; S.id[m] = i; S.slot[m] = i; S.src[m] = -1; }
            }
        }
        __syncthreads();
        if (S.n > AMC_MAX_MEMBERS) {
            if (tid == 0) { atomicAdd(&p.stats->cell_overflow, 1ull); S.n = AMC_MAX_MEMBERS; }
            __syncthreads();
        }
        if (tid == 0) { /* pass 1 counted this cell with the members it saw */
            const unsigned long long n0 = (unsigned long long)p.cell_n[cell];
            S.nref -= n0 * (n0 - 1) / 2;
        }
        const int n = S.n;
        if (n >= 2) {
            cell_process(p, S, 0, cell);
            __syncthreads();
            // ---- every moved member: snapshot at its first move of the pass, and the later cells that hold it now or
            // held it before this visit
            if (S.nold > 0) {
                for (int k = tid; k < n; k += SWE_THREADS) {
                    const int io = (int)S.mv[k] - 1;
                    if (io < 0) continue;
                    double t[2][3];
                    if (io < AMC_MV_CAP) { t[0][0] = S.ox[io]; t[0][1] = S.oy[io]; t[0][2] = S.oz[io]; }
                    else { const double *sp = p.mv_spill + ((size_t)blockIdx.x * AMC_MAX_MEMBERS + io) * 3; t[0][0] = sp[0]; t[0][1] = sp[1]; t[0][2] = sp[2]; }
                    t[1][0] = S.x[k]; t[1][1] = S.y[k]; t[1][2] = S.z[k];
                    const int i = S.id[k];
                    if (p.sw_tag[i] != p.sw_pass) {
                        p.sw_tag[i] = p.sw_pass;
                        p.sw_xs[i] = t[0][0]; p.sw_ys[i] = t[0][1];
                        p.sw_ml[atomicAdd(&s_nml, 1)] = i;
                    }
                    for (int w = 0; w < 2; w++) {
                        int cx[2], cy[2], cz[2];
                        const int nx = axis_cells(p, 0, t[w][0], cx), ny = axis_cells(p, 1, t[w][1], cy), nz = axis_cells(p, 2, t[w][2], cz);
                        for (int c = 0; c < nz; c++) /* same column (x and y masks are this visit's), later cell */
                            if (cz[c] > zl) { const int cc = col * p.nc[2] + cz[c]; atomicOr(bits + (cc >> 5), 1u << (cc & 31)); }
                        for (int b = 0; b < ny; b++) /* same layer, later column */
                            if (cy[b] > yl)
                                for (int c = 0; c < nz; c++) { const int cc = (xl * p.nc[1] + cy[b]) * p.nc[2] + cz[c]; atomicOr(bits + (cc >> 5), 1u << (cc & 31)); }
                        for (int a = 0; a < nx; a++) /* later layer */
                            if (cx[a] > xl)
                                for (int b = 0; b < ny; b++)
                                    for (int c = 0; c < nz; c++) { const int cc = (cx[a] * p.nc[1] + cy[b]) * p.nc[2] + cz[c]; atomicOr(bits + (cc >> 5), 1u << (cc & 31)); }
                    }
                }
            }
        }
        __syncthreads();
        if (tid == 0) s_c = cell + 1;
        __syncthreads();
    }
    if (tid == 0) {
        const unsigned long long nref = S.nref + p.sw_state[1];
        if (nref) atomicAdd(&p.stats->checks_ref, nref);
        if (S.nexec) atomicAdd(&p.stats->checks_exec, (unsigned long long)S.nexec);
    }
}

// ------------------------------------------------------------------------------------------------
// host-RNG parity mode (AMC_KIND_TEMP): one wall case at a time (Temp:693-753)
// specular cases 1, 2a, 2b applied directly; returns the hit count in stats->wall_hits[c].  sp.acc != null: record the
// hits (amc_surface_*), here and in k_case_apply
__global__ void __launch_bounds__(ADVECT_THREADS) k_case_specular(const __grid_constant__ P p, const int c, const __grid_constant__ SurfP sp)
{
    int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= p.n) return;
    Part q;
    load_part(p.a, s, q);
    q.px = p.px[s]; q.py = p.py[s]; q.pz = p.pz[s];
    if (!temp_mask(p, c, q)) return;
    atomicAdd(&p.stats->wall_hits[c], 1ull);
    if (p.wall_bits) p.wall_bits[p.a.pos[s].id] |= (uint16_t)(1u << c);
    if (sp.acc) temp_specular<AMC_LIVE, true>(p, c, q, &sp);
    else temp_specular(p, c, q);
    store_part(p.a, s, q);
}
// energized cases: list the hits (slot, id, normal, contact height); order fixed up on the host
__global__ void __launch_bounds__(ADVECT_THREADS) k_case_detect(const __grid_constant__ P p, const int c, int32_t *count,
                                                                int32_t cap, int32_t *out_slot, int32_t *out_id,
                                                                double *out_nrm, double *out_colz)
{
    int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= p.n) return;
    Part q;
    load_part(p.a, s, q);
    q.px = p.px[s]; q.py = p.py[s]; q.pz = p.pz[s];
    if (!temp_mask(p, c, q)) return;
    int k = atomicAdd(count, 1);
    if (k >= cap) return;
    double t, col[3], nrm[3];
    if (!temp_contact(p.g, c, q, t, col, nrm)) { nrm[0] = nrm[1] = nrm[2] = col[2] = __longlong_as_double(0x7ff8000000000000ll); }
    out_slot[k] = (int32_t)s; out_id[k] = p.a.pos[s].id;
    out_nrm[3 * k] = nrm[0]; out_nrm[3 * k + 1] = nrm[1]; out_nrm[3 * k + 2] = nrm[2];
    out_colz[k] = col[2];
}
__global__ void __launch_bounds__(ADVECT_THREADS) k_case_apply(const __grid_constant__ P p, const int c, int32_t nh,
                                                               const int32_t *slots, const double *dirs,
                                                               const double *surf_e, double *out_dpz, double *out_de,
                                                               const __grid_constant__ SurfP sp)
{
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nh) return;
    int64_t s = slots[k];
    Part q;
    load_part(p.a, s, q);
    q.px = p.px[s]; q.py = p.py[s]; q.pz = p.pz[s];
    out_dpz[k] = 0.0; out_de[k] = 0.0;
    atomicAdd(&p.stats->wall_hits[c], 1ull);
    if (p.wall_bits) p.wall_bits[p.a.pos[s].id] |= (uint16_t)(1u << c);
    double t, col[3], nrm[3], dpz, dE;
    if (!temp_contact(p.g, c, q, t, col, nrm)) {
        atomicAdd(&p.stats->errors, 1ull);
        if (sp.acc) surf_outside(sp, c);
        return;
    }
    double dir[3] = {dirs[3 * k], dirs[3 * k + 1], dirs[3 * k + 2]};
    double Es = c == AMC_CASE_4 ? surf_e[k] : (temp_is_cold(c) ? p.g.E_cold : p.g.E_hot);
    double alpha = c == AMC_CASE_4 ? p.g.alpha_g : p.g.alpha_c;
    const double vx = q.vx, vy = q.vy, vz = q.vz;
    temp_energized(p, q, t, col, dir, Es, alpha, dpz, dE);
    if (sp.acc) surf_record(p, sp, c, col[0], col[1], col[2], q.vx - vx, q.vy - vy, q.vz - vz, dE);
    out_dpz[k] = dpz; out_de[k] = c == AMC_CASE_4 ? 0.0 : dE;
    store_part(p.a, s, q);
}
// operator-level entry point (amc_wall_operator): one wall operator of the reference applied to the particles an
// N-long boolean mask selects, exactly as the reference functions take it (Pore:257-348, Temp:311-347)
__global__ void __launch_bounds__(ADVECT_THREADS) k_wall_operator(const __grid_constant__ P p, const int op, const uint8_t *mask, const double param)
{
    int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= p.n) return;
    if (!mask[p.a.pos[s].id]) return;
    Part q;
    load_part(p.a, s, q);
    q.px = q.x; q.py = q.y; q.pz = q.z;
    switch (op) {
    case AMC_OP_PLANE_MFP: pore_plane_wall<AMC_LIVE>(p, q, param); break;  /* hit_vertical_wall, Pore:257-292 */
    case AMC_OP_SIDE_MFP: pore_side_wall<AMC_LIVE>(p, q, param); break;    /* hit_cylinder_side_wall, Pore:294-348 */
    case AMC_OP_PLANE_SPECULAR: {                                          /* hit_vertical_specular_wall, Temp:311-315 */
        double t = (q.z - param) / q.vz;
        q.vz = -q.vz;
        q.z = param + t * q.vz;
        break;
    }
    case AMC_OP_SIDE_SPECULAR: {                                           /* hit_cylinder_specular_side_wall, Temp:317-347 */
        double t;
        if (!side_quadratic(q.x, q.y, q.vx, q.vy, param, t)) { atomicAdd(&p.stats->errors, 1ull); return; }
        reflect_xy(q, param, t);
        break;
    }
    }
    atomicAdd(&p.stats->wall_hits[0], 1ull);
    store_part(p.a, s, q);
}

// synthetic Maxwellian state (amc_init_synthetic): one thread per global particle index, grid-stride
// position of synthetic particle i: region by cumulative weight, uniform inside it.  attempt 0 = the draw of
// amc_init_synthetic; amc_seed_relax re-draws overlapping particles with attempt 1, 2, ...
__device__ __forceinline__ void synthetic_position(const amc_init_spec &sp, const int64_t i, const uint32_t attempt, const double u[4],
                                                   double &x, double &y, double &z)
{
    int reg = 0;
    while (reg + 1 < sp.n_regions && u[0] >= sp.cum_weight[reg]) reg++;
    if (sp.shape == 0) {
        double rr = sp.radius[reg] * sqrt(u[1]), s, c;
        sincos(6.283185307179586 * u[2], &s, &c);
        x = rr * c; y = rr * s;
    } else {
        x = sp.bx[reg] * u[1]; y = sp.by[reg] * u[2];
    }
    z = sp.z_lo[reg] + (sp.z_hi[reg] - sp.z_lo[reg]) * u[3];
}
__device__ __forceinline__ void synthetic_uniforms(const amc_init_spec &sp, const int64_t i, const uint32_t attempt, const int c0, const int nc, double *u)
{
    const uint32_t k0 = (uint32_t)sp.seed, k1 = (uint32_t)(sp.seed >> 32);
    for (int c = 0; c < nc; c++) {
        uint32_t r[4] = {(uint32_t)i, (uint32_t)((uint64_t)i >> 32), 0x1417u + (attempt << 16), (uint32_t)(c0 + c)};
        philox4x32_10(r, k0, k1);
        u[2 * c] = u53(r[0], r[1]); u[2 * c + 1] = u53(r[2], r[3]);
    }
}
// amc_seed_relax: new positions for the particles the detection pass marked (rank[slot] = 1)
__global__ void __launch_bounds__(ADVECT_THREADS) k_seed_redraw(const __grid_constant__ P p, const __grid_constant__ amc_init_spec sp, const uint32_t attempt)
{
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= p.n || p.rank[s] != 1) return;
    double u[4], x, y, z;
    synthetic_uniforms(sp, p.a.pos[s].id, attempt, 0, 2, u);
    synthetic_position(sp, p.a.pos[s].id, attempt, u, x, y, z);
    p.a.pos[s].x = x; p.a.pos[s].y = y; p.a.pos[s].z = z;
}

__global__ void __launch_bounds__(ADVECT_THREADS) k_init_synthetic(const __grid_constant__ P p, const __grid_constant__ amc_init_spec sp,
                                                                   const int keep_all, int32_t *count, const int64_t cap)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < sp.n_total; i += stride) {
        double u[8];
        synthetic_uniforms(sp, i, 0u, 0, 4, u);
        double x, y, z;
        synthetic_position(sp, i, 0u, u, x, y, z);
        if (!keep_all && !(z >= sp.keep_z_lo && z < sp.keep_z_hi)) continue;
        double s1, c1, s2, c2;
        const double r1 = sp.sigma * sqrt(-2.0 * log(1.0 - u[4])), r2 = sp.sigma * sqrt(-2.0 * log(1.0 - u[6]));
        sincos(6.283185307179586 * u[5], &s1, &c1);
        sincos(6.283185307179586 * u[7], &s2, &c2);
        int64_t t = i;
        if (!keep_all) {
            t = atomicAdd(count, 1);
            if (t >= cap) continue; /* reported by the host from the final count */
        }
        st_pos(p.a.pos + t, x, y, z, (int32_t)i, 0u);
        p.a.vx[t] = r1 * c1; p.a.vy[t] = r1 * s1; p.a.vz[t] = r2 * c2;
        p.a.d[t] = 0.0; p.a.dx[t] = 0.0; p.a.dy[t] = 0.0; p.a.dz[t] = 0.0;
    }
}

// The C ABI hands positions, ids and flags over as separate arrays (the reference's module globals); on the device they
// live in the position records.  amc_set_state copies the host arrays into the SoaView laid over the idle b record
// array and packs them; amc_get_state unpacks the other way before its copies.
__global__ void __launch_bounds__(ADVECT_THREADS) k_pack_pos(const __grid_constant__ P p, const int with_ids)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    const SoaView v = soa_view(p.b.pos, p.cap);
    st_pos(p.a.pos + i, v.x[i], v.y[i], v.z[i], with_ids ? v.id[i] : (int32_t)i, v.flag[i]); /* slot == particle index unless ids are given */
}
__global__ void __launch_bounds__(ADVECT_THREADS) k_unpack_pos(const __grid_constant__ P p)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    const SoaView v = soa_view(p.b.pos, p.cap);
    const PosRec r = p.a.pos[i];
    v.x[i] = r.x; v.y[i] = r.y; v.z[i] = r.z; v.id[i] = r.id; v.flag[i] = (uint8_t)r.flag;
}
__global__ void __launch_bounds__(ADVECT_THREADS) k_set_ids(const __grid_constant__ P p, const int32_t *ids)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < p.n) p.a.pos[i].id = ids[i];
}

// ================================================================================================
// Slab decomposition along z (multi-GPU).  Records are AMC_REC doubles: 10 state values, the global
// particle id and flag bits; every buffer starts with one header record whose first double is the
// record count.  Buffers are exchanged by the host side (NCCL through torch.distributed, or plain
// device copies when several ranks share one GPU in the tests).

// write the per-destination counts into the header records of the transfer buffer
__global__ void k_xfer_headers(const __grid_constant__ P p)
{
    int d = threadIdx.x;
    if (d < p.nranks) {
        int c = p.xf_count[d];
        p.xf_send[(size_t)p.xf_off[d] * AMC_REC] = (double)(c < p.xf_capv[d] ? c : p.xf_capv[d]);
    }
}

// peer-to-peer all-to-all: block d writes the number of records this rank has for rank d into rank d's xfer_recv
// and then publishes the step's sequence number in rank d's flag word for this rank
__global__ void __launch_bounds__(32) k_xfer_push(const __grid_constant__ P p)
{
    const int d = blockIdx.x;
    if (d == p.srank) return;
    if (threadIdx.x != 0) return;
    // the records were written by k_keys (slab_pack); a kernel boundary lies between those stores and this release
    const int c = min(p.xf_count[d], p.xf_capv[d]);
    double *dst = p.peer_xf[d] + (size_t)p.parity * (size_t)p.peer_xf_stride[d] + (size_t)p.peer_xf_off[d] * AMC_REC;
    dst[0] = (double)c;
    flag_publish(p.peer_flag[d] + p.srank, p.xf_seq);
}

// unpack immigrants and ghost copies received from every rank behind the current particles
// (slots n .. n + n_in) and give them owner keys / ranks like k_advect does
__global__ void __launch_bounds__(ADVECT_THREADS) k_xfer_unpack(const __grid_constant__ P p)
{
    int src = blockIdx.y;
    if (p.peer_xf) { /* peer-to-peer mode: rank `src` wrote the block itself; wait for its sequence number */
        if (src == p.srank) return;
        if (threadIdx.x == 0) flag_wait(p.flags + src, p.xf_seq);
        __syncthreads();
    }
    const double *blk = p.xf_recv + (p.peer_xf ? (size_t)p.parity * p.xf_stride : 0) + (size_t)p.xf_off[src] * AMC_REC;
    int cnt = (int)__ldcg(blk);
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= cnt) return;
    const double *r = blk + (size_t)(1 + j) * AMC_REC;
    int64_t s = cur_n(p) + atomicAdd(p.n_in, 1);
    if (s >= p.cap) { atomicAdd(p.slab_overflow + 0, 1ull); return; } /* reported by amc_slab_sort; the state is invalid afterwards */
    Part q;
    q.x = __ldcg(r + 0); q.y = __ldcg(r + 1); q.z = __ldcg(r + 2); q.vx = __ldcg(r + 3); q.vy = __ldcg(r + 4); q.vz = __ldcg(r + 5);
    q.d = __ldcg(r + 6); q.dx = __ldcg(r + 7); q.dy = __ldcg(r + 8); q.dz = __ldcg(r + 9);
    q.flag = (uint32_t)__ldcg(r + 11);
    int o[3];
    int32_t k = owner_key(p, q.x, q.y, q.z, o);
    if (!(q.flag & (AMC_FLAG_GHOST | AMC_FLAG_REL_UP)) && p.srank + 1 < p.nranks && q.z > p.up_thr && k != p.ncell_pad)
        q.flag |= AMC_FLAG_REL_UP | AMC_FLAG_LATE_UP; /* immigrant inside the band below the upper cut */
    store_part_id(p.a, s, q, (int32_t)__ldcg(r + 10));
    p.key[s] = k;
    if (k != p.ncell_pad && any_band(p, q.x, q.y, q.z, o)) p.rank[s] = atomicAdd(&p.band_count[k], 1);
    else p.rank[s] = ~atomicAdd(&p.rest_count[k], 1);
}

// after a colour group: turn the dirty slots into update records, one block per direction (up, down);
// the block clears its queue counter when it is done
__device__ __forceinline__ void bnd_pack_dir(const P &p, const int dir)
{
    const int cnt = min(__ldcg(p.bnd_n + dir), p.bnd_cap);
    const bool peer = p.peer_xf != nullptr;
    const bool has_nb = dir == 0 ? p.srank + 1 < p.nranks : p.srank > 0;
    // peer-to-peer mode: the records go straight into the neighbour's receive buffer (half = parity of the round)
    double *buf = peer ? (has_nb ? p.peer_bnd[dir] + (size_t)(p.bnd_seq & 1u) * p.bnd_stride : nullptr) : p.bnd_send[dir];
    const Arrays &A = p.a;
    if (buf == nullptr) { if (threadIdx.x == 0) p.bnd_n[dir] = 0; return; }
    if (threadIdx.x == 0) buf[0] = (double)cnt;
    for (int j = threadIdx.x; j < cnt; j += blockDim.x) {
        int s = __ldcg(p.bnd_dirty[dir] + j);
        double *r = buf + (size_t)(1 + j) * AMC_REC;
        const PosRec pr = ldcg_pos(A.pos + s);
        r[0] = pr.x; r[1] = pr.y; r[2] = pr.z; r[3] = __ldcg(A.vx + s); r[4] = __ldcg(A.vy + s); r[5] = __ldcg(A.vz + s);
        r[6] = __ldcg(A.d + s); r[7] = __ldcg(A.dx + s); r[8] = __ldcg(A.dy + s); r[9] = __ldcg(A.dz + s); r[10] = (double)pr.id;
        r[11] = (double)(pr.flag & AMC_FLAG_PATH);
        // clear this direction's "queued" bit (32-bit atomic on the word that holds the flag byte)
        unsigned bit = dir == 0 ? AMC_FLAG_DIRTY_UP : AMC_FLAG_DIRTY_DOWN;
        atomicAnd(&A.pos[s].flag, ~bit);
    }
    if (peer) __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        p.bnd_n[dir] = 0;
        if (peer) flag_publish(p.peer_flag[dir == 0 ? p.srank + 1 : p.srank - 1] + p.nranks + (dir == 0 ? 1 : 0), p.bnd_seq); /* I am "below" for the rank above */
    }
}
__global__ void __launch_bounds__(ADVECT_THREADS) k_bnd_pack(const __grid_constant__ P p) { bnd_pack_dir(p, blockIdx.x); }
// the same by ONE WARP (peer-to-peer mode only): the tail of a fused k_pairs_group launch sends both directions side by
// side, and only one thread per direction pays for the system-scope fence (the records are few; what costs is the fence)
__device__ __forceinline__ void bnd_pack_warp(const P &p, const int dir, const int lane)
{
    const int cnt = min(__ldcg(p.bnd_n + dir), p.bnd_cap);
    const bool has_nb = dir == 0 ? p.srank + 1 < p.nranks : p.srank > 0;
    const Arrays &A = p.a;
    if (!has_nb) { if (lane == 0) p.bnd_n[dir] = 0; return; }
    double *buf = p.peer_bnd[dir] + (size_t)(p.bnd_seq & 1u) * p.bnd_stride;
    if (lane == 0) buf[0] = (double)cnt;
    for (int j = lane; j < cnt; j += 32) {
        int s = __ldcg(p.bnd_dirty[dir] + j);
        double *r = buf + (size_t)(1 + j) * AMC_REC;
        const PosRec pr = ldcg_pos(A.pos + s);
        r[0] = pr.x; r[1] = pr.y; r[2] = pr.z; r[3] = __ldcg(A.vx + s); r[4] = __ldcg(A.vy + s); r[5] = __ldcg(A.vz + s);
        r[6] = __ldcg(A.d + s); r[7] = __ldcg(A.dx + s); r[8] = __ldcg(A.dy + s); r[9] = __ldcg(A.dz + s); r[10] = (double)pr.id;
        r[11] = (double)(pr.flag & AMC_FLAG_PATH);
        unsigned bit = dir == 0 ? AMC_FLAG_DIRTY_UP : AMC_FLAG_DIRTY_DOWN;
        atomicAnd(&A.pos[s].flag, ~bit);
    }
    __syncwarp();
    if (lane == 0) {
        p.bnd_n[dir] = 0;
        flag_publish(p.peer_flag[dir == 0 ? p.srank + 1 : p.srank - 1] + p.nranks + (dir == 0 ? 1 : 0), p.bnd_seq);
    }
}

// apply the update records received from one neighbour (dir 0: from the rank above, 1: from below).
// One CTA per record: find the particle by id among the related particles, or append it as a new
// foreign copy; then make sure the later colour groups of this pass can find it (escaped list).
// the records of hand-over round `seq` from one neighbour (dir 0: the rank above, 1: below), records first, first + step, ...
// by this CTA (128 threads)
__device__ __forceinline__ void bnd_apply_dir(const P &p, const int dir, const uint32_t seq, const int first, const int step)
{
    __shared__ int s_slot, s_esc;
    if (dir == 0 ? p.srank + 1 >= p.nranks : p.srank == 0) return; /* no neighbour on that side */
    const double *buf = p.bnd_recv[dir];
    if (p.peer_xf) { /* peer-to-peer mode: the neighbour wrote the records itself; wait for this round's sequence number */
        buf += (size_t)(seq & 1u) * p.bnd_stride;
        if (threadIdx.x == 0) flag_wait(p.flags + p.nranks + dir, seq);
        __syncthreads();
    }
    int cnt = (int)__ldcg(buf);
#ifdef AMC_SLAB_PROBE
    if (first == 0 && p.group_done >= -1 && p.group_done < 7) PROBE_ADD(p.group_done + 1, 6, cnt);
#endif
    const int64_t n_base = cur_n(p);
    for (int j = first; j < cnt; j += step) {
    __syncthreads();
    const double *r = buf + (size_t)(1 + j) * AMC_REC;
    const int32_t id = (int32_t)__ldcg(r + 10);
    const int tid = threadIdx.x;
    if (tid == 0) { s_slot = -1; s_esc = -1; }
    __syncthreads();
    if (tid == 0) s_slot = rel_find(p, id);
    __syncthreads();
    const Arrays &A = p.a;
    if (tid == 0 && s_slot < 0) { // unknown here: a particle the neighbour moved into this rank's reach
        int f = atomicAdd(p.n_foreign, 1);
        if (f >= p.foreign_cap || n_base + f >= p.cap) { atomicAdd(p.slab_overflow + 3, 1ull); s_slot = -2; }
        else {
            int s = (int)n_base + f;
            s_slot = s;
            A.pos[s].id = id;
            A.pos[s].flag = (uint8_t)(AMC_FLAG_GHOST | (dir == 0 ? AMC_FLAG_REL_UP : AMC_FLAG_REL_DOWN));
            rel_insert(p, id, s);
        }
    }
    __syncthreads();
    const int s = s_slot;
    if (s < 0) continue;
    const unsigned fl = A.pos[s].flag;
    if (fl & AMC_FLAG_ESC) { // already on the escaped list: find its (latest) entry
        int ne = min(*p.esc_count, p.esc_cap);
        for (int e = tid; e < ne; e += blockDim.x)
            if (p.esc_slot[e] == s) atomicMax(&s_esc, e);
    }
    __syncthreads();
    if (tid >= 32) continue; /* warp 0: lane 0 places the record, lanes 0-7 take one colour group each */
    const double x = __ldcg(r + 0), y = __ldcg(r + 1), z = __ldcg(r + 2);
    unsigned nf = (fl & ~AMC_FLAG_PATH) | ((unsigned)__ldcg(r + 11) & AMC_FLAG_PATH);
    int o[3] = {0, 0, 0};
    const int e_old = s_esc;
    int e = -1, findable = 0, ok = 1;
    int q[3] = {0, 0, 0};
    double ux = x, uy = y, uz = z; /* where this rank had the particle so far (new foreign copy: nowhere else) */
    if (tid == 0) {
        // slots below the count of the sort hold sorted particles; the ones behind it are foreign copies appended by
        // earlier hand-overs of this pass (always on the escaped list): both have a previous position here
        const bool sorted = s < n_base;
        if (sorted || (fl & AMC_FLAG_ESC)) { ux = A.pos[s].x; uy = A.pos[s].y; uz = A.pos[s].z; }
        // a sorted particle that has not escaped still sits in the owner cell it was sorted into
        const int32_t sk = owner_key(p, ux, uy, uz, q);
        A.pos[s].x = x; A.pos[s].y = y; A.pos[s].z = z; A.vx[s] = __ldcg(r + 3); A.vy[s] = __ldcg(r + 4); A.vz[s] = __ldcg(r + 5);
        A.d[s] = __ldcg(r + 6); A.dx[s] = __ldcg(r + 7); A.dy[s] = __ldcg(r + 8); A.dz[s] = __ldcg(r + 9);
        int32_t k = owner_key(p, x, y, z, o);
        if (e_old < 0)
            findable = sorted && k == sk && (s < p.cell_start[sk] + p.band_count[sk] || !any_band(p, x, y, z, o));
        if (!findable) {
            e = atomicAdd(p.esc_count, 1);
            if (e >= p.esc_cap) { atomicAdd(&p.stats->esc_overflow, 1ull); ok = 0; }
            else { p.esc_slot[e] = s; nf |= AMC_FLAG_ESC; }
        }
        A.pos[s].flag = (uint8_t)nf;
        touch_slot(p, s);
    }
    const unsigned FULL = 0xffffffffu;
    const int o0 = __shfl_sync(FULL, o[0], 0), o1 = __shfl_sync(FULL, o[1], 0), o2 = __shfl_sync(FULL, o[2], 0);
    e = __shfl_sync(FULL, e, 0); findable = __shfl_sync(FULL, findable, 0); ok = __shfl_sync(FULL, ok, 0);
    const int q0 = __shfl_sync(FULL, q[0], 0), q1 = __shfl_sync(FULL, q[1], 0), q2 = __shfl_sync(FULL, q[2], 0);
    const double vx_ = __shfl_sync(FULL, ux, 0), vy_ = __shfl_sync(FULL, uy, 0), vz_ = __shfl_sync(FULL, uz, 0);
    // the cells of the remaining groups that hold this particle must be visited (k_detect did not see this position)
    const int g2 = tid;
    if (ok && g2 < 8 && g2 > p.group_done) {
        int cx = member_axis(p.edge[0], p.lo[0], p.nc[0], o0, (g2 >> 2) & 1, x);
        int cy = member_axis(p.edge[1], p.lo[1], p.nc[1], o1, (g2 >> 1) & 1, y);
        int cz = member_axis(p.edge[2], p.lo[2], p.nc[2], o2, (g2 ^ p.zoff) & 1, z);
        int32_t cc = (cx < 0 || cy < 0 || cz < 0) ? -1 : ((cx >> 1) * p.nh[1] + (cy >> 1)) * p.nh[2] + (cz >> 1);
        if (e_old >= 0) p.esc_cell[e_old * 8 + g2] = -1;
        esc_link(p, g2, cc, cx, cy, cz, findable ? -1 : e);
        // the cell that held the copy so far loses it (see activate_moved)
        int dx = member_axis(p.edge[0], p.lo[0], p.nc[0], q0, (g2 >> 2) & 1, vx_);
        int dy = member_axis(p.edge[1], p.lo[1], p.nc[1], q1, (g2 >> 1) & 1, vy_);
        int dz = member_axis(p.edge[2], p.lo[2], p.nc[2], q2, (g2 ^ p.zoff) & 1, vz_);
        int32_t dc = (dx < 0 || dy < 0 || dz < 0) ? -1 : ((dx >> 1) * p.nh[1] + (dy >> 1)) * p.nh[2] + (dz >> 1);
        if (dc >= 0 && dc != cc) esc_link(p, g2, dc, dx, dy, dz, -1);
    }
    }
}
template <bool PACK>
__global__ void __launch_bounds__(128) k_bnd_apply(const __grid_constant__ P p)
{
    const int dir = blockIdx.y;
    // peer-to-peer mode: the same launch first sends this rank's own records (block 0 of each direction) -- nothing
    // below depends on them: a particle is moved by exactly one rank per colour group
    if (PACK && blockIdx.x == 0) { bnd_pack_dir(p, dir); __syncthreads(); }
    bnd_apply_dir(p, dir, p.bnd_seq, blockIdx.x, gridDim.x);
}

// device-resident stepping: the particle count after the sort (start of the bucket of the dropped particles) and,
// at the end of the step, the foreign copies appended by the hand-overs
__global__ void k_slab_set_n(const __grid_constant__ P p, const int after_sort)
{
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    if (after_sort) {
        if ((int64_t)p.n_dev[0] + *p.n_in > p.n_hint) atomicAdd(p.slab_overflow + 0, 1ull); /* the grids of this call were too small */
        p.n_dev[0] = p.cell_start[p.ncell_pad + 1];
    } else p.n_dev[0] += min(*p.n_foreign, p.foreign_cap);
}

// compact the particles this rank owns (everything that is not a ghost copy) into the b arrays
__global__ void __launch_bounds__(ADVECT_THREADS) k_compact_owned(const __grid_constant__ P p, int32_t *count)
{
    int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= p.n) return;
    unsigned fl = p.a.pos[s].flag;
    if (fl & AMC_FLAG_GHOST) return;
    int t = atomicAdd(count, 1);
    // positions, ids and flags leave as separate arrays laid over the b record array (SoaView, amc_api.cu)
    const PosRec r = p.a.pos[s];
    const SoaView v = soa_view(p.b.pos, p.cap);
    v.x[t] = r.x; v.y[t] = r.y; v.z[t] = r.z; v.id[t] = r.id; v.flag[t] = (uint8_t)(fl & AMC_FLAG_PATH);
    p.b.vx[t] = p.a.vx[s]; p.b.vy[t] = p.a.vy[s]; p.b.vz[t] = p.a.vz[s];
    p.b.d[t] = p.a.d[s]; p.b.dx[t] = p.a.dx[s]; p.b.dy[t] = p.a.dy[s]; p.b.dz[t] = p.a.dz[s];
}

// Order-independent 128-bit checksum of the particles this handle owns (ghost copies excluded): for every
// particle and field f, a = mix64(bits(value) ^ mix64(16 * id + f)); out[0] += a, out[1] += mix64(a + C), out[2] += 1
// per particle (all mod 2^64).  Sums commute, so the value does not depend on the slot order or on how the
// particles are spread over ranks: a 1-GPU run and an N-rank slab run of the same job agree iff their id-ordered
// states agree bit for bit (amc.digest_of_arrays is the NumPy restatement).
__device__ __forceinline__ unsigned long long mix64(unsigned long long z)
{
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__global__ void __launch_bounds__(ADVECT_THREADS) k_state_digest(const __grid_constant__ P p, unsigned long long *out)
{
    __shared__ unsigned long long sh[3];
    if (threadIdx.x < 3) sh[threadIdx.x] = 0;
    __syncthreads();
    unsigned long long a0 = 0, a1 = 0, cnt = 0;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < p.n; s += stride) {
        const unsigned fl = p.a.pos[s].flag;
        if (fl & AMC_FLAG_GHOST) continue;
        const unsigned long long id = (unsigned long long)(uint32_t)p.a.pos[s].id;
        const double v[10] = {p.a.pos[s].x, p.a.pos[s].y, p.a.pos[s].z, p.a.vx[s], p.a.vy[s], p.a.vz[s], p.a.d[s], p.a.dx[s], p.a.dy[s], p.a.dz[s]};
#pragma unroll
        for (int f = 0; f < 11; f++) {
            const unsigned long long bits = f < 10 ? (unsigned long long)__double_as_longlong(v[f < 10 ? f : 0]) : (unsigned long long)(fl & AMC_FLAG_PATH);
            const unsigned long long a = mix64(bits ^ mix64(16ull * id + (unsigned long long)f));
            a0 += a; a1 += mix64(a + 0xD6E8FEB86659FD93ull);
        }
        cnt++;
    }
    for (int o = 16; o; o >>= 1) {
        a0 += __shfl_xor_sync(0xffffffffu, a0, o); a1 += __shfl_xor_sync(0xffffffffu, a1, o); cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    }
    if ((threadIdx.x & 31) == 0) { atomicAdd(&sh[0], a0); atomicAdd(&sh[1], a1); atomicAdd(&sh[2], cnt); }
    __syncthreads();
    if (threadIdx.x < 3 && sh[threadIdx.x]) atomicAdd(&out[threadIdx.x], sh[threadIdx.x]);
}

// ---------------------------------------------------------------- field sampling (amc_sample_*)
// Per-cell moments of the state at the end of a timestep (include/amc.h): count, and sum v, sum v^2 per axis as
// two fixed-point limbs each.  The particles sit sorted by owner cell, so the lanes of a warp hold two or three
// runs of one cell: the lanes of each cell (__match_any_sync) add their words with __reduce_add_sync and one lane
// issues one set of 13 atomics per cell and warp.  __reduce_add_sync adds 32-bit values: a word is split into its
// low 21 bits (unsigned) and the rest (signed), whose sums over 32 lanes cannot overflow while every word of the
// warp is below 2^40 in magnitude (|v| < 2^17 m/s); a warp with a larger word falls back to per-particle atomics.
// Plain 32-byte record + 3 velocities per particle: 56 bytes read, nothing written but the atomics.
#define SAMPLE_THREADS 256
struct SampleArgs {
    unsigned long long *acc;     /* [cells][AMC_SAMPLE_WORDS] */
    unsigned long long *outside; /* [1] */
    const double *zedge;         /* z edges of the sampling grid (a slab handle: the global ones) */
    int32_t ncz;
    double ze0, zinv;
};
__device__ __forceinline__ void sample_limbs(const double v, const double s1, const double s1inv, const double s2, long long &i1, long long &i2)
{
    i1 = __double2ll_rn(v * s1);
    const double rem = v - (double)i1 * s1inv;
    i2 = __double2ll_rn(rem * s2);
}

// velocity distribution (amc_vdf_*): per z layer of the sampling grid, histograms of vx, vy, vz over [-v_max, v_max]
// and of the speed over [0, v_max], AMC_VDF_HISTS x (n_bins + 2) words [under, bins, over] (include/amc.h).  A kernel
// parameter of its own, so that P and every other kernel stay as they are.
struct VdfArgs {
    unsigned long long *acc; /* [ncz][AMC_VDF_HISTS][n_bins + 2] */
    const double *edges;     /* [2][n_bins + 1]: np.linspace of the component range, then of the speed range */
    double lo[2], hi[2];     /* [0]: components (-v_max, v_max), [1]: speed (0, v_max) */
    int32_t n_bins;
};
// word of x in a histogram of range h: 0 under (x < lo), 1 + the bin of np.histogram(x, n_bins, (lo, hi)) with the edge
// corrections of hist_add, n_bins + 1 over (x > hi or NaN)
__device__ __forceinline__ int vdf_word(const VdfArgs &va, const int h, const double x)
{
    const double lo = va.lo[h], hi = va.hi[h];
    const int nb = va.n_bins;
    if (x < lo) return 0;
    if (!(x <= hi)) return nb + 1;
    const double *e = va.edges + h * (nb + 1);
    long long idx = (long long)(((x - lo) / (hi - lo)) * (double)nb);
    if (idx == nb) idx--;
    if (x < e[idx]) idx--;
    else if (x >= e[idx + 1] && idx != nb - 1) idx++;
    return (int)idx + 1;
}
// one count per histogram of a sampled particle (layer >= 0), straight to global memory.  A per-CTA copy of the
// histograms in shared memory was slower (DESIGN section 14): at ~18 particles per cell a CTA sees few particles of a
// layer, so the flush issues about as many atomics as it saves.
__device__ __forceinline__ void vdf_add(const VdfArgs &va, const int layer, const double v[3])
{
    static_assert(AMC_VDF_HISTS == 4, "histograms of vdf_add");
    const int hw = va.n_bins + 2;
    unsigned long long *a = va.acc + (size_t)layer * AMC_VDF_HISTS * hw;
    const double speed = sqrt((v[0] * v[0] + v[1] * v[1]) + v[2] * v[2]);
    atomicAdd(a + vdf_word(va, 0, v[0]), 1ull);
    atomicAdd(a + hw + vdf_word(va, 0, v[1]), 1ull);
    atomicAdd(a + 2 * hw + vdf_word(va, 0, v[2]), 1ull);
    atomicAdd(a + 3 * hw + vdf_word(va, 1, speed), 1ull);
}

// VDF: also bin the velocity distribution of the sampled particles (vdf_add), in the same pass over the state
template <bool VDF>
__global__ void __launch_bounds__(SAMPLE_THREADS) k_sample(const __grid_constant__ P p, const SampleArgs sa, const __grid_constant__ VdfArgs va)
{
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned lane = threadIdx.x & 31u;
    int cell = -1; /* -1: no particle of this rank in the slot, -2: outside the grid */
    long long w[12];
#pragma unroll
    for (int k = 0; k < 12; k++) w[k] = 0;
    if (s < cur_n(p)) {
        const PosRec r = p.a.pos[s];
        if (!(r.flag & AMC_FLAG_GHOST)) { /* the owning rank samples it (same predicate as k_state_digest) */
            const int ox = owner_axis(p.edge[0], p.nc[0], p.e0[0], p.inv_d[0], r.x);
            const int oy = owner_axis(p.edge[1], p.nc[1], p.e0[1], p.inv_d[1], r.y);
            const int oz = owner_axis(sa.zedge, sa.ncz, sa.ze0, sa.zinv, r.z);
            if (ox < 0 || ox >= p.nc[0] || oy < 0 || oy >= p.nc[1] || oz < 0 || oz >= sa.ncz) cell = -2;
            else {
                cell = (ox * p.nc[1] + oy) * sa.ncz + oz;
                const double v[3] = {p.a.vx[s], p.a.vy[s], p.a.vz[s]};
#pragma unroll
                for (int a = 0; a < 3; a++) {
                    sample_limbs(v[a], 0x1p19, 0x1p-19, 0x1p49, w[2 * a], w[2 * a + 1]);
                    sample_limbs(v[a] * v[a], 0x1p6, 0x1p-6, 0x1p36, w[6 + 2 * a], w[6 + 2 * a + 1]);
                }
                if constexpr (VDF) vdf_add(va, oz, v);
            }
        }
    }
    static_assert(AMC_SAMPLE_V1 == 19 && AMC_SAMPLE_V2 == 49 && AMC_SAMPLE_Q1 == 6 && AMC_SAMPLE_Q2 == 36, "scales of k_sample");
    const unsigned outside = __ballot_sync(0xffffffffu, cell == -2);
    if (lane == 0 && outside) atomicAdd(sa.outside, (unsigned long long)__popc(outside));
    bool narrow = true;
#pragma unroll
    for (int k = 0; k < 12; k++) narrow &= (unsigned long long)(w[k] + (1ll << 40)) < (1ull << 41);
    if (__any_sync(0xffffffffu, !narrow)) { /* a word beyond 2^40: one set of atomics per particle */
        if (cell >= 0) {
            unsigned long long *a = sa.acc + (size_t)cell * AMC_SAMPLE_WORDS;
            atomicAdd(a, 1ull);
#pragma unroll
            for (int k = 0; k < 12; k++) if (w[k]) atomicAdd(a + 1 + k, (unsigned long long)w[k]);
        }
        return;
    }
    const unsigned peers = __match_any_sync(0xffffffffu, cell);
    unsigned todo = __ballot_sync(0xffffffffu, cell >= 0);
    while (todo) { /* one cell of the warp at a time: every lane of `grp` executes the reductions with the same mask */
        const int first = __ffs(todo) - 1;
        const unsigned grp = __shfl_sync(0xffffffffu, peers, first);
        todo &= ~grp;
        if (grp & (1u << lane)) {
            long long tot[12];
#pragma unroll
            for (int k = 0; k < 12; k++) {
                const unsigned lo = __reduce_add_sync(grp, (unsigned)(w[k] & 0x1FFFFF));
                const int hi = __reduce_add_sync(grp, (int)(w[k] >> 21));
                tot[k] = (long long)hi * (1ll << 21) + (long long)lo;
            }
            if ((int)lane == first) {
                unsigned long long *a = sa.acc + (size_t)cell * AMC_SAMPLE_WORDS;
                atomicAdd(a, (unsigned long long)__popc(grp));
#pragma unroll
                for (int k = 0; k < 12; k++) if (tot[k]) atomicAdd(a + 1 + k, (unsigned long long)tot[k]);
            }
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------- plane flux recording (amc_flux_*)
// Net crossings of the z planes of the sampling grid between consecutive record points (include/amc.h).  One thread
// per slot: the 32-byte record gives z and the id, and the plane count of z is compared with the snapshot snap[id].
// Only a particle that crossed a plane -- a fraction of a percent per step at the pore's timestep -- loads its
// velocity and adds its words with 64-bit atomics: a few hundred thousand atomics per step at 12.5 M particles,
// spread over the planes, so a warp-level reduction of them would not pay for itself.  A kernel parameter of its own,
// so that P and every other kernel stay as they are.
#define FLUX_THREADS 256
struct FluxArgs {
    unsigned long long *acc; /* [ncz + 1][AMC_FLUX_WORDS] */
    int32_t *snap;           /* [max_particles] plane count of every particle id at the last record point */
    unsigned long long *bad; /* [1] k_flux_snap: ids outside 0 .. n-1 or met twice */
};
// cnt(z): the number of planes edge[k] <= z, k = 0 .. nc (np.searchsorted(edge, z, side='right'); NaN: nc + 1).  The
// guess from the uniform spacing is corrected against the uploaded edges, so the answer is NumPy's for every z.
__device__ __forceinline__ int flux_count(const double *edge, const int nc, const double e0, const double inv_d, const double z)
{
    if (z != z) return nc + 1;
    const double t = (z - e0) * inv_d;
    int c = !(t >= 0.0) ? 0 : (t >= (double)nc ? nc + 1 : (int)t + 1);
    while (c > 0 && z < edge[c - 1]) c--;
    while (c <= nc && edge[c] <= z) c++;
    return c;
}
// the snapshot of the current state (snap[0 .. n-1] preset to -1): every id must be met once, in 0 .. n-1
__global__ void __launch_bounds__(FLUX_THREADS) k_flux_snap(const __grid_constant__ P p, const FluxArgs fa)
{
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= p.n) return;
    const PosRec r = p.a.pos[s];
    if ((uint32_t)r.id >= (uint32_t)p.n) { atomicAdd(fa.bad, 1ull); return; }
    const int c = flux_count(p.edge[2], p.nc[2], p.e0[2], p.inv_d[2], r.z);
    if (atomicExch(fa.snap + r.id, c) != -1) atomicAdd(fa.bad, 1ull);
}
// one record point: 32 bytes of record + a 4-byte snapshot read per particle; a crossing adds one full contribution
// to every plane it passed and writes the snapshot back
__global__ void __launch_bounds__(FLUX_THREADS) k_flux(const __grid_constant__ P p, const FluxArgs fa)
{
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= p.n) return;
    const PosRec r = p.a.pos[s];
    const int c1 = flux_count(p.edge[2], p.nc[2], p.e0[2], p.inv_d[2], r.z);
    const int c0 = fa.snap[r.id];
    if (c1 == c0) return;
    fa.snap[r.id] = c1;
    const double v[3] = {p.a.vx[s], p.a.vy[s], p.a.vz[s]};
    const double sg = c1 > c0 ? 1.0 : -1.0;
    static_assert(AMC_FLUX_WORDS == 10 && AMC_FLUX_V1 == 16 && AMC_FLUX_V2 == 46 && AMC_FLUX_Q1 == 2 && AMC_FLUX_Q2 == 32, "words of k_flux");
    long long w[8];
#pragma unroll
    for (int a = 0; a < 3; a++) sample_limbs(sg * v[a], 0x1p16, 0x1p-16, 0x1p46, w[2 * a], w[2 * a + 1]);
    sample_limbs(sg * ((v[0] * v[0] + v[1] * v[1]) + v[2] * v[2]), 0x1p2, 0x1p-2, 0x1p32, w[6], w[7]);
    for (int k = min(c0, c1); k < max(c0, c1); k++) {
        unsigned long long *a = fa.acc + (size_t)k * AMC_FLUX_WORDS;
        atomicAdd(a + (c1 > c0 ? 0 : 1), 1ull);
#pragma unroll
        for (int j = 0; j < 8; j++) if (w[j]) atomicAdd(a + 2 + j, (unsigned long long)w[j]);
    }
}
