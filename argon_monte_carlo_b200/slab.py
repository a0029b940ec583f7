"""Slab decomposition of one simulation along the pore axis z over several GPUs (BASELINE.json
north_star: 1/2/4/8 B200 with halo exchange and particle migration every step).

The reference has nothing like this (its only parallelism is a process pool over the cells of a
colour group, Open_Air_Pore_MC.py:522-549); the requirement is that the decomposed run leaves the
same results as the single-domain run.  Each rank owns the reference cells of a contiguous range of
global z layers, cut on cell boundaries and balanced by particle count (62 % of the pore's particles
sit in the two end caps).  Per timestep:

  1. advect + walls on the owned particles; emigrants and ghost copies (particles inside the overlap
     band below the upper cut) are packed per destination rank           amc_slab_advect
  2. one all-to-all moves them                                             transport.alltoall
  3. unpack + counting sort of owned + ghost particles                     amc_slab_sort
  4. for each of the 8 colour groups (plus one round before the first): the pair kernel, then the few
     particles moved by a collision that the neighbour also holds (or now needs) are exchanged with
     the ranks above / below and applied                                   amc_slab_group / neighbors / amc_slab_apply
  5. recapture, counters                                                   amc_slab_finish

Every reference cell is processed by exactly one rank, in the same colour-group order, with members
ordered by global particle index, and a particle touched on both sides of a cut is handed over after
each group, so the N-rank run is bit-identical to the 1-rank run (tests/test_gpu_slab.py).

Transports: `LocalTransport` (all ranks in this process, device copies; used by the single-GPU tests)
and `DistTransport` (one rank per process over torch.distributed: NCCL on GPUs, gloo for the CPU
test of the host logic).
"""
from __future__ import annotations

import ctypes as C
from types import SimpleNamespace

import numpy as np

from . import amc

REC = 12  # doubles per exchanged record


class AmcSlabConfig(C.Structure):
    _fields_ = [("rank", C.c_int32), ("nranks", C.c_int32), ("cuts", C.POINTER(C.c_int32)), ("gncz", C.c_int32),
                ("gz_edge", amc.c_double_p), ("gz_lo", amc.c_double_p), ("xfer_capacity", C.c_int32),
                ("xfer_capacity_far", C.c_int32), ("bnd_capacity", C.c_int32), ("xfer_send", C.c_void_p), ("xfer_recv", C.c_void_p),
                ("bnd_send_up", C.c_void_p), ("bnd_send_down", C.c_void_p), ("bnd_recv_up", C.c_void_p),
                ("bnd_recv_down", C.c_void_p)]


class AmcSlabP2PDesc(C.Structure):
    """struct amc_slab_p2p_desc (include/amc.h): where a rank's exchange buffers live, for its peers to map."""
    _fields_ = [("pid", C.c_int64), ("device", C.c_int32), ("rank", C.c_int32), ("base", C.c_uint64), ("ipc", C.c_uint8 * 64),
                ("off_flags", C.c_int64), ("off_xfer", C.c_int64), ("off_bnd_up", C.c_int64), ("off_bnd_down", C.c_int64),
                ("xfer_stride", C.c_int64), ("bnd_stride", C.c_int64)]


def owner_layer(z, edges):
    """Global z layer of each particle, clamped into [0, ncz-1] like the device does for routing."""
    k = np.searchsorted(edges, z, side="right") - 1
    return np.clip(k, 0, len(edges) - 2)


def _feasible_cuts(cum, nranks, limit, min_layers, odd_only):
    """Cuts with at least min_layers layers and at most `limit` particles per slab, or None.  Dynamic programme over
    (slab, end layer): slab r can end at layer k if slab r-1 can end at some j in [first j with cum[k]-cum[j] <= limit,
    k - min_layers]; `last[k]` = largest reachable end <= k keeps the range test O(1).  odd_only: interior cuts on odd
    layers."""
    ncz = len(cum) - 1
    ks = np.arange(ncz + 1)
    jmin = np.searchsorted(cum, cum - limit, side="left")           # smallest j with cum[j] >= cum[k] - limit
    reach = np.zeros(ncz + 1, dtype=bool)
    reach[0] = True
    prev = []
    for r in range(1, nranks + 1):
        last = np.where(reach, ks, -1)
        last = np.maximum.accumulate(last)                          # largest reachable end <= k
        hi = ks - min_layers
        cand = np.where(hi >= 0, last[np.maximum(hi, 0)], -1)       # best predecessor end for a slab ending at k
        ok = cand >= jmin
        if r < nranks:
            if odd_only:
                ok &= (ks % 2 == 1)
            ok[ncz] = False
        prev.append(np.where(ok, cand, -1))
        reach = ok
    if not reach[ncz]:
        return None
    cuts = [ncz]
    for r in range(nranks - 1, -1, -1):
        cuts.append(int(prev[r][cuts[-1]]))
    return cuts[::-1]


def balanced_cuts(z, edges, nranks, min_layers=2, prefer_odd=True, odd_tolerance=0.03):
    """Cut indices (nranks+1) on z-cell boundaries that minimise the particle count of the fullest slab (bisection on
    that count with a dynamic-programming feasibility test).  Odd cuts are preferred -- the cells just above an odd cut belong to
    the odd z colour groups, so a ghost that has to be exported late (an immigrant that lands in the band below the
    cut) is only needed from group 1 on and travels with the hand-over after group 0, no extra round before it --
    unless they make the fullest slab more than odd_tolerance fuller than the unconstrained optimum."""
    ncz = len(edges) - 1
    if nranks * min_layers > ncz:
        raise ValueError("too many ranks for %d z layers" % ncz)
    hist = np.bincount(owner_layer(np.asarray(z), np.asarray(edges)), minlength=ncz).astype(np.float64)
    cum = np.concatenate([[0.0], np.cumsum(hist)])

    def best(odd_only):
        lo, hi = cum[-1] / nranks, cum[-1]
        if _feasible_cuts(cum, nranks, hi, min_layers, odd_only) is None:
            return None, np.inf
        for _ in range(60):
            mid = 0.5 * (lo + hi)
            if _feasible_cuts(cum, nranks, mid, min_layers, odd_only) is None:
                lo = mid
            else:
                hi = mid
        cuts = _feasible_cuts(cum, nranks, hi, min_layers, odd_only)
        return cuts, max(cum[b] - cum[a] for a, b in zip(cuts, cuts[1:]))

    free, load_free = best(False)
    if prefer_odd and nranks > 1:
        odd, load_odd = best(True)
        if odd is not None and load_odd <= load_free * (1.0 + odd_tolerance):
            return np.array(odd, dtype=np.int32)
    return np.array(free, dtype=np.int32)


def local_grid(grid, z0, z1):
    """The part of the global cell grid a rank owns: all of x and y, z layers [z0, z1)."""
    return SimpleNamespace(nc=(grid.nc[0], grid.nc[1], int(z1 - z0)), c0=(grid.c0[0], grid.c0[1], grid.c0[2] + int(z0)),
                           edge=[grid.edge[0], grid.edge[1], np.ascontiguousarray(grid.edge[2][z0:z1 + 1])],
                           lo=[grid.lo[0], grid.lo[1], np.ascontiguousarray(grid.lo[2][z0:z1])])


class SlabRank:
    """One rank: a libamc handle restricted to its z layers plus its exchange buffers (torch tensors)."""

    def __init__(self, cfg, rank, cuts, device, xfer_capacity, bnd_capacity, max_particles, seed=None, kind=None,
                 taps=0, cheb=None, xfer_capacity_far=512, grid=None, p2p=False):
        self.rank, self.nranks, self.cuts = rank, len(cuts) - 1, cuts
        self.device = device
        g = grid or cfg.grid
        self.sim = amc.Simulation(cfg, kind=kind, pp_mode=amc.PP_GROUPS, device=device, seed=seed,
                                  grid=local_grid(g, cuts[rank], cuts[rank + 1]), max_particles=max_particles, taps=taps,
                                  cheb=cheb)
        self.sim.sample_grid = g    # sampling covers the global grid: a particle is binned where it is, whoever owns it
        self.p2p = p2p
        if p2p:
            # device-resident stepping (amc_slab_step): the handle owns the exchange buffers and runs on its own stream
            c = self._slab_config(g, cuts, rank, xfer_capacity, xfer_capacity_far, bnd_capacity)
            self.sim._check(self.sim.lib.amc_slab_enable(self.sim.h, C.byref(c)), "amc_slab_enable")
            self.desc = AmcSlabP2PDesc()
            self.sim._check(self.sim.lib.amc_slab_p2p_setup(self.sim.h, C.byref(self.desc)), "amc_slab_p2p_setup")
            return
        import torch
        dev = torch.device("cuda", device)
        with torch.cuda.device(dev):
            z = lambda *s: torch.zeros(*s, dtype=torch.float64, device=dev)
            # one block per peer: large for the two neighbours (migrants + ghost copies), small for the rest
            caps = [xfer_capacity if abs(d - rank) == 1 else xfer_capacity_far for d in range(self.nranks)]
            self.xfer_splits = [(c + 1) * REC for c in caps]
            self.xfer_offsets = np.concatenate([[0], np.cumsum(self.xfer_splits)]).astype(np.int64)
            self.xfer_send, self.xfer_recv = z(int(self.xfer_offsets[-1])), z(int(self.xfer_offsets[-1]))
            # boundary buffers live inside one [nranks, ...] tensor per direction of travel so that the
            # hand-over can also be done with a single all_to_all_single (block r = traffic with rank r)
            self.bnd_send_all, self.bnd_recv_all = z(self.nranks, bnd_capacity + 1, REC), z(self.nranks, bnd_capacity + 1, REC)
            spare = lambda: z(bnd_capacity + 1, REC)
            up, down = rank + 1 < self.nranks, rank > 0
            self.bnd_send_up = self.bnd_send_all[rank + 1] if up else spare()
            self.bnd_recv_up = self.bnd_recv_all[rank + 1] if up else spare()
            self.bnd_send_down = self.bnd_send_all[rank - 1] if down else spare()
            self.bnd_recv_down = self.bnd_recv_all[rank - 1] if down else spare()
            stream = torch.cuda.current_stream(dev).cuda_stream
        c = self._slab_config(g, cuts, rank, xfer_capacity, xfer_capacity_far, bnd_capacity)
        c.xfer_send, c.xfer_recv = self.xfer_send.data_ptr(), self.xfer_recv.data_ptr()
        c.bnd_send_up, c.bnd_send_down = self.bnd_send_up.data_ptr(), self.bnd_send_down.data_ptr()
        c.bnd_recv_up, c.bnd_recv_down = self.bnd_recv_up.data_ptr(), self.bnd_recv_down.data_ptr()
        lib, h = self.sim.lib, self.sim.h
        self.sim._check(lib.amc_set_stream(h, C.c_void_p(stream)), "amc_set_stream")
        self.sim._check(lib.amc_slab_enable(h, C.byref(c)), "amc_slab_enable")

    def _slab_config(self, g, cuts, rank, xfer_capacity, xfer_capacity_far, bnd_capacity):
        c = AmcSlabConfig()
        c.rank, c.nranks = rank, self.nranks
        self._cuts = np.ascontiguousarray(cuts, dtype=np.int32)
        self._edge = np.ascontiguousarray(g.edge[2], dtype=np.float64)
        self._lo = np.ascontiguousarray(g.lo[2], dtype=np.float64)
        c.cuts = self._cuts.ctypes.data_as(C.POINTER(C.c_int32))
        c.gncz, c.gz_edge, c.gz_lo = g.nc[2], amc._dp(self._edge), amc._dp(self._lo)
        c.xfer_capacity, c.xfer_capacity_far, c.bnd_capacity = xfer_capacity, xfer_capacity_far, bnd_capacity
        return c

    def connect(self, descs):
        """descs: the AmcSlabP2PDesc of every rank, ordered by rank."""
        arr = (AmcSlabP2PDesc * len(descs))(*descs)
        self.sim._check(self.sim.lib.amc_slab_p2p_connect(self.sim.h, arr), "amc_slab_p2p_connect")

    def call(self, name, *args):
        self.sim._check(getattr(self.sim.lib, name)(self.sim.h, *args), name)

    def xfer_block(self, buf, peer):
        return buf[int(self.xfer_offsets[peer]):int(self.xfer_offsets[peer + 1])]


class LocalTransport:
    """All ranks live in this process (possibly on one GPU): exchanges are device copies."""

    def alltoall(self, ranks):
        for dst in ranks:
            for src in ranks:
                dst.xfer_block(dst.xfer_recv, src.rank).copy_(src.xfer_block(src.xfer_send, dst.rank), non_blocking=True)

    def neighbors(self, ranks):
        by_rank = {r.rank: r for r in ranks}
        for r in ranks:
            if r.rank + 1 in by_rank:
                by_rank[r.rank + 1].bnd_recv_down.copy_(r.bnd_send_up, non_blocking=True)
            if r.rank - 1 in by_rank:
                by_rank[r.rank - 1].bnd_recv_up.copy_(r.bnd_send_down, non_blocking=True)

    def allreduce_sum(self, value):
        return value

    def allreduce_u64(self, values):
        return values if isinstance(values, np.ndarray) else tuple(values)


class DistTransport:
    """One rank per process over torch.distributed (NCCL over NVLink on the GPU box; gloo on CPU tensors
    in the host-logic test).  Fixed-size buffers, so no size negotiation and no host synchronisation."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist, self.group = dist, group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        import os
        # neighbour hand-over: batched send/recv with the two neighbours (default; couples only adjacent
        # ranks) or, with AMC_SLAB_A2A=1, one all_to_all_single (half the launch latency, but a global
        # synchronisation point per round; measured slightly slower at 8 GPUs)
        self.nbr_a2a = dist.get_backend(group) == "nccl" and os.environ.get("AMC_SLAB_A2A", "0") == "1"
        self.native_a2a = dist.get_backend(group) == "nccl"

    def alltoall(self, ranks):
        (r,) = ranks
        if self.native_a2a:   # block sizes are symmetric (|src - dst| decides), so send and receive splits coincide
            self.dist.all_to_all_single(r.xfer_recv, r.xfer_send, output_split_sizes=r.xfer_splits,
                                        input_split_sizes=r.xfer_splits, group=self.group)
            return
        ops = []
        for peer in range(self.world):
            if peer == self.rank:
                r.xfer_block(r.xfer_recv, peer).copy_(r.xfer_block(r.xfer_send, peer))
                continue
            ops.append(self.dist.P2POp(self.dist.isend, r.xfer_block(r.xfer_send, peer), peer, self.group))
            ops.append(self.dist.P2POp(self.dist.irecv, r.xfer_block(r.xfer_recv, peer), peer, self.group))
        for req in (self.dist.batch_isend_irecv(ops) if ops else []):
            req.wait()

    def neighbors(self, ranks):
        (r,) = ranks
        if self.nbr_a2a:
            self.dist.all_to_all_single(r.bnd_recv_all, r.bnd_send_all, group=self.group)
            return
        ops = getattr(r, "_nbr_ops", None)
        if ops is None:     # the buffers are fixed: build the P2P descriptors once
            ops = []
            if self.rank + 1 < self.world:
                ops.append(self.dist.P2POp(self.dist.isend, r.bnd_send_up, self.rank + 1, self.group))
                ops.append(self.dist.P2POp(self.dist.irecv, r.bnd_recv_up, self.rank + 1, self.group))
            if self.rank > 0:
                ops.append(self.dist.P2POp(self.dist.isend, r.bnd_send_down, self.rank - 1, self.group))
                ops.append(self.dist.P2POp(self.dist.irecv, r.bnd_recv_down, self.rank - 1, self.group))
            r._nbr_ops = ops
        for req in (self.dist.batch_isend_irecv(ops) if ops else []):
            req.wait()

    def allreduce_sum(self, value):
        import torch
        t = torch.as_tensor(np.asarray(value, dtype=np.float64))
        if self.dist.get_backend(self.group) == "nccl":
            t = t.cuda()
        self.dist.all_reduce(t, group=self.group)
        return t.cpu().numpy()


    def allgather_bytes(self, blob):
        """The byte strings of all ranks, ordered by rank (used once, to exchange the peer-to-peer descriptors)."""
        out = [None] * self.world
        self.dist.all_gather_object(out, bytes(blob), group=self.group)
        return out

    def allreduce_u64(self, values):
        """Component-wise sum mod 2^64 over all ranks (int64 adds wrap like uint64 ones).  A uint64 ndarray comes back
        as an ndarray of the same shape, anything else as a tuple of ints."""
        import torch
        arr = np.array(values, dtype=np.uint64)
        t = torch.as_tensor(arr.view(np.int64).copy())
        if self.dist.get_backend(self.group) == "nccl":
            t = t.cuda()
        self.dist.all_reduce(t, group=self.group)
        out = t.cpu().numpy().view(np.uint64).reshape(arr.shape)
        return out if isinstance(values, np.ndarray) else tuple(int(v) for v in out)


SUM_KEYS = ("wall_collisions", "pp_collisions", "pair_checks_ref", "pair_checks_exec", "oob_after_walls", "oob_after_pp",
            "oob_after_walls_recapture", "oob_after_pp_recapture", "errors", "completed_paths", "dpz", "e_cold", "e_hot",
            "collisions")


class SlabSimulation:
    """A simulation decomposed into `nranks` z slabs.  `local_ranks`: the ranks this process drives
    (all of them with LocalTransport, exactly one with DistTransport)."""

    def __init__(self, cfg, nranks, z_for_cuts, transport=None, local_ranks=None, devices=None, xfer_capacity=None,
                 bnd_capacity=2048, slack=1.35, seed=None, kind=None, taps=0, cuts=None, n_total=None, grid=None, p2p=False):
        """grid: cell grid to decompose (default cfg.grid); the cube stage passes a colour-group grid here
        because its own serial sweep cannot be sharded (BASELINE config 4)."""
        self.cfg, self.nranks = cfg, nranks
        self.grid = grid or cfg.grid
        self.transport = transport or LocalTransport()
        self.local_ranks = list(range(nranks)) if local_ranks is None else list(local_ranks)
        g = self.grid
        self.cuts = balanced_cuts(z_for_cuts, g.edge[2], nranks) if cuts is None else np.asarray(cuts, dtype=np.int32)
        layer = owner_layer(np.asarray(z_for_cuts), g.edge[2])
        # z_for_cuts may be a sample of a larger state of n_total particles
        sample_scale = 1.0 if n_total is None else max(1.0, float(n_total) / max(len(layer), 1))
        per_rank = np.array([np.count_nonzero((layer >= self.cuts[r]) & (layer < self.cuts[r + 1])) for r in range(nranks)])
        per_rank = (per_rank * sample_scale).astype(np.int64)
        if xfer_capacity is None:
            # per step and cut: ghosts = the particles of the layer below the cut that lie within one
            # collision range of it, plus the migrants (about a fifth of that at dt = tau/1000)
            hist = np.bincount(layer, minlength=g.nc[2])
            band = float(cfg.collision_range) / float(g.edge[2][1] - g.edge[2][0])
            xfer_capacity = int(max(4096, 4 * hist.max() * band * sample_scale + 2048))
        cheb = None
        if cfg.kind == "temp":
            from .config import gap_energy_chebyshev
            cheb = gap_energy_chebyshev(cfg, 16)
        devices = devices or [0] * len(self.local_ranks)
        self.ranks = [SlabRank(cfg, r, self.cuts, devices[i], xfer_capacity, bnd_capacity,
                               int(per_rank[r] * slack) + 2 * xfer_capacity + nranks * 512 + 16 * bnd_capacity + 4096,
                               seed=seed, kind=kind, taps=taps, cheb=cheb, grid=g, p2p=p2p)
                      for i, r in enumerate(self.local_ranks)]
        self.p2p = p2p
        if p2p:
            # one rank per GPU and process: exchange the buffer descriptors once, map the peers' buffers (NVLink)
            if len(self.ranks) != 1 or isinstance(self.transport, LocalTransport):
                if nranks != 1:
                    raise ValueError("p2p stepping needs one rank per process and GPU (DistTransport)")
                self.ranks[0].connect([self.ranks[0].desc])
            else:
                blobs = self.transport.allgather_bytes(bytes(self.ranks[0].desc))
                self.ranks[0].connect([AmcSlabP2PDesc.from_buffer_copy(b) for b in blobs])
        self.n_global = 0
        # the hand-over round before the first colour group is only needed if some cut is even
        self.pre_round = any(int(c) % 2 == 0 for c in self.cuts[1:-1])
        self.phase_ms = None        # set by step(timing=True): [advect, exchange+sort, pair groups+hand-over, finish]
        self.debug_counts = False   # True: tally exchanged records per step (host sync; tests only)
        self.exchanged = {"xfer": 0, "boundary": 0}

    def _tally(self, kind):
        if self.debug_counts:
            for r in self.ranks:
                if kind == "xfer":
                    self.exchanged["xfer"] += int(sum(r.xfer_send[int(o)].item() for o in r.xfer_offsets[:-1]))
                else:
                    self.exchanged["boundary"] += int(r.bnd_send_up[0, 0].item()) + int(r.bnd_send_down[0, 0].item())

    def set_state(self, x, y, z, vx, vy, vz, dist=None, dist_x=None, dist_y=None, dist_z=None, flag=None):
        """Global arrays in original particle index order; each local rank takes the particles whose z
        layer it owns (ids = global indices)."""
        n = len(x)
        self.n_global = n
        layer = owner_layer(np.asarray(z), self.grid.edge[2])
        opt = lambda a, m: None if a is None else np.asarray(a)[m]
        for r in self.ranks:
            m = (layer >= self.cuts[r.rank]) & (layer < self.cuts[r.rank + 1])
            ids = np.nonzero(m)[0].astype(np.int64)
            r.sim.set_state(np.asarray(x)[m], np.asarray(y)[m], np.asarray(z)[m], np.asarray(vx)[m], np.asarray(vy)[m],
                            np.asarray(vz)[m], opt(dist, m), opt(dist_x, m), opt(dist_y, m), opt(dist_z, m), opt(flag, m))
            r.call("amc_set_ids", ids.ctypes.data_as(amc.c_int64_p))

    def init_synthetic(self, make_spec):
        """Generate the state on the devices (amc_init_synthetic): make_spec(keep_z) returns the AmcInitSpec of the
        whole job restricted to a z range, e.g. lambda kz: init_state.pore_spec(cfg, 17, keep_z=kz).  Every local rank
        keeps the particles of its own layers; particle i is the same whatever the number of ranks."""
        edges = self.grid.edge[2]
        n_global = 0
        for r in self.ranks:
            lo = -np.inf if r.rank == 0 else float(edges[self.cuts[r.rank]])
            hi = np.inf if r.rank == len(self.cuts) - 2 else float(edges[self.cuts[r.rank + 1]])
            spec = make_spec((lo, hi))
            r.sim.init_synthetic(spec)
            n_global = int(spec.n_total)
        self.n_global = n_global

    def set_local_state(self, ids, x, y, z, vx, vy, vz, dist=None, dist_x=None, dist_y=None, dist_z=None, flag=None,
                        n_global=None):
        """Distributed use: this process's single rank receives exactly the particles it owns."""
        (r,) = self.ranks
        r.sim.set_state(x, y, z, vx, vy, vz, dist, dist_x, dist_y, dist_z, flag)
        ids = np.ascontiguousarray(ids, dtype=np.int64)
        r.call("amc_set_ids", ids.ctypes.data_as(amc.c_int64_p))
        self.n_global = n_global if n_global is not None else self.n_global

    def step_fused(self, n_steps=1, reduce=True):
        """n_steps timesteps through amc_slab_step: everything -- migration, ghost copies, the hand-over after every
        colour group -- is enqueued by the library and moves peer to peer; one host synchronisation per call.  Returns
        the per-step counter dicts (summed over all ranks if reduce) ; self.phase_ms = device time of
        [advect, exchange + sort, pair groups + hand-over, finish] summed over the steps."""
        (r,) = self.ranks
        st = (amc.AmcStepStats * n_steps)()
        r.call("amc_slab_step", C.c_int32(n_steps), C.c_int32(int(self.pre_round)), st)
        ms, _ = r.sim.last_timing()
        self.phase_ms = np.array(ms[:4])
        out = [s.as_dict() for s in st]
        if reduce and not isinstance(self.transport, LocalTransport):
            mat = np.array([np.concatenate([[float(d[k]) for k in SUM_KEYS], d["wall_hits"].astype(np.float64)]) for d in out])
            mat = self.transport.allreduce_sum(mat)
            for d, vec in zip(out, mat):
                for i, k in enumerate(SUM_KEYS):
                    d[k] = type(d[k])(vec[i]) if not isinstance(d[k], float) else float(vec[i])
                d["wall_hits"] = vec[len(SUM_KEYS):].astype(np.int64)
        return out

    def step(self, n_steps=1, reduce=True, timing=False):
        """n_steps timesteps; returns per-step counter dicts summed over this process's ranks (and over
        all processes when the transport is distributed and reduce=True).  timing=True additionally
        brackets the phases with CUDA events on the current stream (self.phase_ms, summed over steps)."""
        out = []
        T, R = self.transport, self.ranks
        marks = []
        if timing:
            import torch

            def mark():
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                marks.append(e)
        else:
            def mark():
                pass
        for _ in range(n_steps):
            mark()
            for r in R:
                r.call("amc_slab_advect")
            mark()
            self._tally("xfer")
            T.alltoall(R)
            for r in R:
                r.call("amc_slab_sort", None)
            mark()
            for r in R:
                r.call("amc_slab_pairs_begin", C.c_int32(int(self.pre_round)))
            if self.pre_round:
                self._tally("boundary")
                T.neighbors(R)
                for r in R:
                    r.call("amc_slab_apply", C.c_int32(-1))
            for g in range(8):
                for r in R:
                    r.call("amc_slab_group", C.c_int32(g))
                self._tally("boundary")
                T.neighbors(R)
                for r in R:
                    r.call("amc_slab_apply", C.c_int32(g))
            mark()
            tot = None
            for r in R:
                st = amc.AmcStepStats()
                r.call("amc_slab_finish", C.byref(st))
                if r.sim.sample_due(amc.load_library().amc_get_step_index(r.sim.h) - 1):
                    r.sim.sample_now()
                d = st.as_dict()
                if tot is None:
                    tot = d
                else:
                    for k in SUM_KEYS:
                        tot[k] = tot[k] + d[k]
                    tot["wall_hits"] = tot["wall_hits"] + d["wall_hits"]
            if reduce and not isinstance(T, LocalTransport):
                vec = np.concatenate([[float(tot[k]) for k in SUM_KEYS], tot["wall_hits"].astype(np.float64)])
                vec = T.allreduce_sum(vec)
                for i, k in enumerate(SUM_KEYS):
                    tot[k] = type(tot[k])(vec[i]) if not isinstance(tot[k], float) else float(vec[i])
                tot["wall_hits"] = vec[len(SUM_KEYS):].astype(np.int64)
            mark()
            out.append(tot)
        if timing:
            import torch
            torch.cuda.synchronize()
            ms = np.zeros(4)
            for k in range(n_steps):
                for j in range(4):
                    ms[j] += marks[5 * k + j].elapsed_time(marks[5 * k + j + 1])
            self.phase_ms = ms
        return out

    def owned(self, out=None):
        """Per local rank: (ids, dict of state arrays) of the particles it currently owns.
        out: optional list (one per local rank) of dicts with preallocated -- e.g. pinned -- arrays
        'ids' (int64), the ten float64 state arrays and 'flag' (uint8)."""
        res = []
        keys = ("x", "y", "z", "vx", "vy", "vz", "dist", "dist_x", "dist_y", "dist_z")
        for i, r in enumerate(self.ranks):
            if out is not None:
                buf = out[i]
                cap = len(buf["ids"])
            else:
                cap = max(int(amc.load_library().amc_num_particles(r.sim.h)), 1)
                buf = {k: np.empty(cap) for k in keys}
                buf["ids"] = np.empty(cap, dtype=np.int64)
                buf["flag"] = np.empty(cap, dtype=np.uint8)
            n = C.c_int64(0)
            r.call("amc_slab_get_owned", C.c_int64(cap), C.byref(n), buf["ids"].ctypes.data_as(amc.c_int64_p),
                   *[amc._dp(buf[k]) for k in keys], buf["flag"].ctypes.data_as(amc.c_uint8_p))
            k = int(n.value)
            d = {key: buf[key][:k] for key in keys}
            d["flag"] = buf["flag"][:k]
            res.append((buf["ids"][:k], d))
        return res

    def get_state(self):
        """Global arrays in original index order assembled from the local ranks (all ranks local)."""
        keys = ("x", "y", "z", "vx", "vy", "vz", "dist", "dist_x", "dist_y", "dist_z")
        out = {k: np.full(self.n_global, np.nan) for k in keys}
        out["flag"] = np.zeros(self.n_global, dtype=np.uint8)
        seen = 0
        for ids, d in self.owned():
            for k in keys + ("flag",):
                out[k][ids] = d[k]
            seen += len(ids)
        out["_owned_total"] = seen
        return out

    def state_digest(self, reduce=True):
        """(sum0, sum1, count) of amc_state_digest over the owned particles of all ranks: equal to the digest of
        the single-domain run of the same job iff the id-ordered states agree bit for bit."""
        d = amc.combine_digests([r.sim.state_digest() for r in self.ranks])
        return self.transport.allreduce_u64(d) if reduce else d

    # ------------------------------------------------------------------ field sampling
    def sample_enable(self, every=0, first_step=0):
        """Field sampling on every local rank (Simulation.sample_enable); each rank bins its own particles on the
        global grid, so the merged accumulators equal those of the single-domain run bit for bit."""
        for r in self.ranks:
            r.sim.sample_enable(every, first_step)

    def sample_disable(self):
        for r in self.ranks:
            r.sim.sample_disable()

    def sample_now(self):
        for r in self.ranks:
            r.sim.sample_now()

    def sample_raw(self, reduce=True):
        """(acc, samples taken, particles outside the grid) summed over the local ranks and, with a distributed
        transport and reduce=True, over all processes (element-wise uint64 sums)."""
        acc, ns, no = amc.merge_sample_ranks([r.sim.sample_raw() for r in self.ranks])
        if reduce and not isinstance(self.transport, LocalTransport):
            acc = self.transport.allreduce_u64(acc)
            (no,) = self.transport.allreduce_u64((no,))
        return acc, ns, no

    def last_sample_ms(self):
        return [r.sim.last_sample_ms() for r in self.ranks]

    def vdf_enable(self, n_bins, v_max):
        """Velocity distribution on every local rank (Simulation.vdf_enable; after sample_enable): each rank bins its
        own particles by the global z layers, so the merged histograms equal those of the single-domain run."""
        for r in self.ranks:
            r.sim.vdf_enable(n_bins, v_max)

    def vdf_disable(self):
        for r in self.ranks:
            r.sim.vdf_disable()

    def vdf_raw(self, reduce=True):
        """VDF words summed over the local ranks and, with a distributed transport and reduce=True, over all processes
        (element-wise uint64 sums)."""
        acc = None
        with np.errstate(over="ignore"):
            for r in self.ranks:
                a = r.sim.vdf_raw()
                acc = a if acc is None else acc + a
        if reduce and not isinstance(self.transport, LocalTransport):
            acc = self.transport.allreduce_u64(acc)
        return acc

    # ------------------------------------------------------------------ surface recording
    def surface_enable(self):
        """Surface recording on every local rank (Simulation.surface_enable); a hit is recorded by the rank that owns
        the particle, on the global grid, so the merged accumulators equal those of the single-domain run bit for bit."""
        for r in self.ranks:
            r.sim.surface_enable()

    def surface_disable(self):
        for r in self.ranks:
            r.sim.surface_disable()

    def surface_raw(self, reduce=True):
        """(acc, wall phases recorded, outside) summed over the local ranks and, with a distributed transport and
        reduce=True, over all processes (element-wise uint64 sums)."""
        acc, ns, out = amc.merge_surface_ranks([r.sim.surface_raw() for r in self.ranks])
        if reduce and not isinstance(self.transport, LocalTransport):
            acc = self.transport.allreduce_u64(acc)
            out = self.transport.allreduce_u64(out)
        return acc, ns, out

    def histograms(self):
        counts, n, sums = None, 0, None
        for r in self.ranks:
            c, k, s = r.sim.histograms()
            counts = c if counts is None else counts + c
            n += k
            sums = s if sums is None else sums + s
        return counts, n, sums

    def pair_list(self):
        parts = [r.sim.pair_list() for r in self.ranks]
        return tuple(np.concatenate([p[i] for p in parts]) for i in range(4))

    def particles_per_rank(self):
        return [int(amc.load_library().amc_num_particles(r.sim.h)) for r in self.ranks]

    def close(self):
        for r in self.ranks:
            r.sim.close()
