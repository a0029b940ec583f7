#!/usr/bin/env python
"""Benchmark of the per-timestep hard-sphere collision loop (BASELINE.json metric:
collision-resolved particle-steps/s at 1/2/4/8 B200 + fraction of the HBM roofline).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                  [--workload temp_pore|cube] [--particles-per-gpu M] [--dump-outputs DIR]

One "step" = one whole timestep (drift, walls, recapture, cell sort, pair detection, the ordered
8-colour-group resolution, recapture, MFP / momentum bookkeeping) over all particles of the job.

Workload (config.workload): a synthetic Maxwellian argon gas in the energized thruster-pore
geometry of Temperature_Pore_MC.py, every length scaled so that each GPU holds
--particles-per-gpu particles (default 12.5 M; at 8 GPUs that is BASELINE.json's 100 M-particle
config 5).  The state (1 GB per GPU at fp64) is far larger than the 126 MB L2, so consecutive
steps never re-read a warm cache.  `also` carries the same measurement for config 2
(Open_Air_Pore_MC.py at the reference particle count, L2 flushed between timed steps).

--impl reference: the reference's CPU implementation of the path, timed on the host cores: the
unmodified Temperature_Pore_MC.py (staged into the git-ignored baseline/_ref by __graft_entry__.build(),
baseline/stage.py; one timestep of its 557,649-particle configuration, ~1.5 minutes, times taken from
the script's own prints).  The C port of its algorithm (oracle/amc_oracle.c, OpenMP over the cells of
a colour group, thread count pinned to os.cpu_count()) is timed beside it as `cpu_baseline_port` and
stands in when the staged copy is missing.

Out of band (never inside a timed region): N = 1 replays two steps of the workload through the CPU
oracle and compares the states bit for bit (`verify`); N > 1 replays the whole job as one domain on
rank 0's GPU and compares the order-independent state checksum (`verify.identical_to_single_gpu`).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (it may be read-only)

B_STEP = 162.0      # algorithmic bytes per particle-step, fp64 state read + written once (SURVEY 8d)
B_PAIR = 32.0       # algorithmic bytes per particle for the pair kernel: 3 x f64 position + cell header
DUMP_SAMPLE = 1 << 19   # particles in the --dump-outputs sample: 11 state arrays + the indices, x 8 B x 2^19 = 50 MB


def dump_outputs(path, sim, last):
    """--dump-outputs: what the timed path hands its caller after its last step, as float64 .npy files in `path`:
    the particle state (get_state, particle-index order) of a fixed, seeded sample of the particles, the sample's
    particle indices, and the counters of that step.  The inputs are seeded too, so the files of two builds run with
    the same arguments can be compared one by one."""
    os.makedirs(path, exist_ok=True)
    state = sim.get_state()
    n = len(state["x"])
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_SAMPLE), replace=False))
    np.save(os.path.join(path, "particle_index.npy"), idx.astype(np.float64))
    for k, v in state.items():
        np.save(os.path.join(path, k + ".npy"), v[idx].astype(np.float64))
    for k, v in last.items():
        if k != "pair_checks_exec":     # the pair tests the kernels executed: a measure of their work, not a result
            np.save(os.path.join(path, "step_" + k + ".npy"), np.atleast_1d(np.asarray(v, dtype=np.float64)))


def ncu_traffic(kernel, particles):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of `kernel` from the committed ncu --set full
    capture (profiles/ncu_traffic.json, written by tools/ncu_traffic.py from the capture's raw page); None unless
    the capture was taken on this workload (same particle count)."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            for rec in json.load(f)["kernels"]:
                if kernel == rec["kernel"] and abs(rec["particles"] - particles) <= 1e-3 * particles:
                    return {"bytes": rec["dram_bytes"], "source": rec["source"]}
    except Exception:
        pass
    return None


def detect_kernel():
    """name of the detection kernel libamc.so launches: candidates staged by cp.async.bulk (default) or loaded by the
    threads (AMC_DETECT=ldg), see launch_detect in csrc/amc_api.cu"""
    return "k_detect" if os.environ.get("AMC_DETECT") == "ldg" else "k_detect_tma"


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region.  nvidia-smi needs up to a second to start
    (longer with eight busy GPUs) while a timed region lasts tens of milliseconds, so the sampler is launched early
    (launch()) and the rows are selected afterwards by their timestamps: mark_start() / stop() bracket the timed region;
    when fewer than three rows fall inside it, the rows of the warm-up steps just before it (same kernels, same load)
    are added and `window` says so."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index
        self.t_launch = self.t_start = self.t_warm = None

    def launch(self):
        if self.proc is not None:
            return
        import datetime
        self.t_launch = datetime.datetime.now()
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "10"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def mark_warmup(self):
        import datetime
        self.t_warm = datetime.datetime.now()

    def start(self):
        """Beginning of the timed region."""
        import datetime
        self.launch()
        self.t_start = datetime.datetime.now()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        import datetime
        t_end = datetime.datetime.now()
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        parsed = []
        for r in self.rows:
            try:
                ts = datetime.datetime.strptime(r[0], "%Y/%m/%d %H:%M:%S.%f")
                parsed.append((ts, float(r[1]), float(r[2]), [nm for k, nm in enumerate(names) if r[4 + k].lower().startswith("active")]))
            except Exception:
                pass
        slack = datetime.timedelta(milliseconds=15)       # nvidia-smi stamps a row when it prints it
        pick = [q for q in parsed if self.t_start <= q[0] <= t_end + slack]
        window = "timed region"
        if len(pick) < 3 and self.t_warm is not None:
            pick = [q for q in parsed if self.t_warm <= q[0] <= t_end + slack]
            window = "warm-up steps + timed region"
        sm, mx = [q[1] for q in pick], [q[2] for q in pick]
        reasons = sorted({nm for q in pick for nm in q[3]})
        out = {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
               "samples": len(sm), "window": window, "reasons": reasons}
        if not sm:   # say why: nothing printed, nothing parsed, or nothing inside the window
            out["rows_printed"], out["rows_parsed"] = len(self.rows), len(parsed)
            out["first_row"] = ",".join(self.rows[0]) if self.rows else None
            out["window_start"] = str(self.t_warm or self.t_start)
        return out


def scaled_temp_config(total_particles):
    from argon_monte_carlo_b200 import config
    base = 557649
    scale = (total_particles / base) ** (1.0 / 3.0)
    cfg = config.pore_config(True, scale=scale)
    return cfg, scale


def run_cube(args, world, rank, local, dev, barrier, max_over_ranks, sum_over_ranks):
    """BASELINE config 4: --cube-particles (default 10 M) Maxwellian argon atoms in a cube with specular walls
    at the reference density, colour-group pair schedule with ~21.4 nm cells, slab-decomposed along z
    over the GPUs (strong scaling: the total is fixed)."""
    import torch
    import torch.distributed as dist
    from argon_monte_carlo_b200 import amc, config, init_state, slab
    n = args.cube_particles
    base = config.cube_config()
    scale = (n / base.num_molecules) ** (1.0 / 3.0)
    n_sub = 2 * max(1, int(round(base.cube_x * scale / 21.43e-9 / 2)))
    cfg = config.cube_config(scale=scale, n_sub=n_sub)
    cfg.dt = cfg.tau / 1000                                           # SURVEY 8d: dt = tau/1000 for the synthetic configs
    grid = config.Grid(nc=(n_sub,) * 3, c0=(0, 0, 0), d=(cfg.dx, cfg.dy, cfg.dz), band=(cfg.collision_range,) * 3)
    state = init_state.synthetic_cube_state(cfg, n, seed=127)
    if world == 1:
        sim = amc.Simulation(cfg, kind=amc.KIND_CUBE, pp_mode=amc.PP_GROUPS, grid=grid, max_particles=n, device=local)
        sim.set_state(*state)
        sim.step_quiet(args.warmup)
        barrier()
        sim.step_quiet(args.steps)
        ms = sim.last_timing()[0]
        dev_ms, phases = ms[4], {"keys": ms[0] / args.steps, "scan_scatter_advect": ms[1] / args.steps, "pairs": ms[2] / args.steps,
                                 "pair_detect": sim.last_detect_ms() / args.steps}
        sim.close()
    else:
        cuts = slab.balanced_cuts(state[2], grid.edge[2], world)
        layer = slab.owner_layer(state[2], grid.edge[2])
        m = (layer >= cuts[rank]) & (layer < cuts[rank + 1])
        fused = os.environ.get("AMC_SLAB_MODE", "p2p") == "p2p"
        sim = slab.SlabSimulation(cfg, world, state[2], transport=slab.DistTransport(), local_ranks=[rank], devices=[local],
                                  cuts=cuts, kind=amc.KIND_CUBE, grid=grid, seed=127, p2p=fused)
        sim.set_local_state(np.nonzero(m)[0], *[a[m] for a in state], n_global=n)
        step = (lambda k, timing=False: sim.step_fused(k, reduce=False)) if fused else (lambda k, timing=False: sim.step(k, reduce=False, timing=timing))
        step(args.warmup)
        barrier()
        step(args.steps, timing=True)
        ms = sim.phase_ms
        barrier()
        digest = sim.state_digest()
        dev_ms = max_over_ranks(float(ms.sum()))
        phases = {"advect_walls": ms[0] / args.steps, "exchange_sort": ms[1] / args.steps,
                  "pairs_and_handover": ms[2] / args.steps, "finish": ms[3] / args.steps}
        sim.close()
        verify = {"digest": ["%016x" % d for d in digest[:2]], "particles_counted": digest[2], "steps": args.warmup + args.steps}
        if rank == 0 and not args.no_verify:     # out of band: the same job as one domain on rank 0's GPU
            one = amc.Simulation(cfg, kind=amc.KIND_CUBE, pp_mode=amc.PP_GROUPS, grid=grid, max_particles=n, device=local)
            one.set_state(*state)
            one.step_quiet(args.warmup + args.steps)
            d1 = one.state_digest()
            one.close()
            verify.update(digest_single_gpu=["%016x" % d for d in d1[:2]], identical_to_single_gpu=tuple(d1) == tuple(digest))
        barrier()
    out = {"metric": "collision-resolved particle-steps/s", "value": n * args.steps / (dev_ms * 1e-3), "unit": "particle-steps/s",
           "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": "cube_%dM: Maxwellian argon in a %.0f nm cube, specular walls, colour-group pair schedule, "
                                  "%d^3 cells, z slabs over %d GPU(s)" % (n // 1000000, cfg.cube_x * 1e9, n_sub, world),
                      "particles_total": n, "l2": "inputs larger than L2"},
           "phases_ms_per_step": phases}
    if world > 1:
        out["verify"] = verify
    if rank == 0:
        emit(out)
    if world > 1:
        dist.destroy_process_group()


def run_ours(args):
    import torch
    import torch.distributed as dist
    from argon_monte_carlo_b200 import amc, config, init_state

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    hbm_peak, peak_src = measured_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    if args.workload == "cube":
        return run_cube(args, world, rank, local, dev, barrier, max_over_ranks, sum_over_ranks)
    if world > 1:
        return run_slabs(args, world, rank, local, dev, hbm_peak, peak_src, barrier, max_over_ranks, sum_over_ranks)

    # ---------------------------------------------------------------- main workload
    clocks = ClockSampler(local)
    clocks.launch()                             # nvidia-smi needs up to a second to start: long before the timed region
    m = args.particles_per_gpu
    cfg, scale = scaled_temp_config(m)          # each rank: one domain of m particles (weak scaling)
    if args.device_init:   # the same synthetic gas, generated by the device-side initialiser (amc_init_synthetic)
        n = cfg.num_molecules
        sim = amc.Simulation(cfg, seed=17 + rank, device=local, max_particles=n)
        sim.init_synthetic(init_state.pore_spec(cfg, seed=17 + rank))
    else:
        state = init_state.synthetic_pore_state(cfg, seed=17 + rank)
        n = len(state[0])
        sim = amc.Simulation(cfg, seed=17 + rank, device=local, max_particles=n)
        sim.set_state(*state)
    sim.step_quiet(1)                       # (one extra untimed step: kernels loaded, allocations touched)
    torch.cuda.synchronize()
    clocks.mark_warmup()
    for _ in range(args.warmup):
        sim.step_quiet(1)
    barrier()
    clocks.start()
    t0 = time.perf_counter()
    stats = sim.step(args.steps)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    ms, launches = sim.last_timing()
    barrier()
    clk = clocks.stop()
    digest = sim.state_digest()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, sim, stats[-1])
    dev_ms = max_over_ranks(ms[4])
    total_particles = sum_over_ranks(float(n))
    value = total_particles * args.steps / (dev_ms * 1e-3)
    pair_ms = ms[2] / args.steps
    det_ms = sim.last_detect_ms() / args.steps
    checks_ref = float(np.mean([s["pair_checks_ref"] for s in stats]))
    checks_exec = float(np.mean([s["pair_checks_exec"] for s in stats]))
    collisions = float(np.mean([s["collisions"] for s in stats]))
    # dominant pair kernel: k_detect, ONE launch per step over every reference cell (the neighbour search; the
    # ordered resolution that follows only visits the ~0.05 % of cells it flags).  Per launch: algorithmic bytes =
    # 32 B x particles (SURVEY 8d: 3 x f64 position + cell header), duration = CUDA events around the launch on the
    # handle's stream; traffic = dram read + write of one launch from the ncu --set full capture of this workload
    # (profiles/ncu_traffic.json; null when no capture of this workload is committed)
    traffic = ncu_traffic(detect_kernel(), n)
    roofline = {"bound": "hbm", "kernel": detect_kernel() + " (pair detection, 1 launch per step)",
                "achieved": B_PAIR * n / (det_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                "peak_source": peak_src, "algorithmic_bytes_per_launch": B_PAIR * n,
                "avg_launch_ms": det_ms,
                "traffic": traffic["bytes"] if traffic else None, "traffic_source": traffic["source"] if traffic else None}
    roofline["frac"] = roofline["achieved"] / hbm_peak
    # the longest kernel of the step, for the record: k_scatter_advect streams the whole state once (93 B read + 85 B
    # written per particle: the 162 B of state plus sort key, rank and particle id)
    sc_ms = sim.last_scatter_ms() / args.steps
    sc_traffic = ncu_traffic("k_scatter_advect", n)
    roofline_scatter = {"bound": "hbm", "kernel": "k_scatter_advect (the timestep on the way to the sorted slot, 1 launch per step)",
                        "achieved": 178.0 * n / (sc_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s", "algorithmic_bytes_per_launch": 178.0 * n,
                        "avg_launch_ms": sc_ms, "traffic": sc_traffic["bytes"] if sc_traffic else None}
    roofline_scatter["frac"] = roofline_scatter["achieved"] / hbm_peak
    whole = {"achieved": B_STEP * n * args.steps / (ms[4] * 1e-3) / 1e9, "unit": "GB/s"}
    whole["frac"] = whole["achieved"] / hbm_peak

    # ---------------------------------------------------------------- e2e: host buffers in and out every step
    keys = ("x", "y", "z", "vx", "vy", "vz", "dist", "dist_x", "dist_y", "dist_z")
    pinned = {k: torch.empty(n, dtype=torch.float64).pin_memory() for k in keys}
    pinned["flag"] = torch.empty(n, dtype=torch.uint8).pin_memory()
    host = {k: v.numpy() for k, v in pinned.items()}
    sim.get_state(host)
    e2e_steps = max(1, min(args.steps, 5))
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        sim.set_state(*[host[k] for k in keys], flag=host["flag"])
        sim.step_quiet(1)
        sim.get_state(host)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    bytes_io = n * 81
    e2e = {"value": total_particles * e2e_steps / e2e_s, "unit": "particle-steps/s", "steps": e2e_steps,
           "h2d_bytes_per_step": bytes_io, "d2h_bytes_per_step": bytes_io}
    # for information: the same host buffers, but the way the drop-in drivers call the library -- state in once,
    # amc_step(K) with the per-step counters / momentum / energy rows coming back to the host, state out once
    try:
        kk = max(1, min(args.steps, 20))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sim.set_state(*[host[k] for k in keys], flag=host["flag"])
        rows = sim.step(kk)
        sim.get_state(host)
        torch.cuda.synchronize()
        dtc = time.perf_counter() - t0
        e2e["state_resident_between_steps"] = {"value": n * kk / dtc, "unit": "particle-steps/s", "steps_per_call": kk,
                                               "h2d_bytes_per_call": bytes_io, "d2h_bytes_per_call": bytes_io + 200 * len(rows)}
    except Exception as exc:   # never lose the benchmark line over the extra figure
        e2e["state_resident_between_steps"] = {"error": str(exc)}
    sim.close()

    out = {
        "metric": "collision-resolved particle-steps/s", "value": value, "unit": "particle-steps/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "temp_pore_scaled: energized thruster pore (Temperature_Pore_MC geometry x %.3f), "
                               "%d particles per GPU, device RNG; state %.2f GB per GPU > L2" % (scale, n, n * 85 / 1e9),
                   "particles_total": int(total_particles), "cells": list(cfg.grid.nc),
                   "parallelism": "1 domain per GPU" if world == 1 else "%d independent domains (replicas)" % world,
                   "l2": "inputs larger than L2"},
        "clocks": clk, "e2e": e2e, "gpu_launches": launches,
        "roofline": roofline, "roofline_longest_kernel": roofline_scatter, "roofline_whole_step": whole,
        "phases_ms_per_step": {"keys": ms[0] / args.steps, "scan_scatter_advect": ms[1] / args.steps,
                               "pair_detect": det_ms, "pair_resolve": pair_ms - det_ms, "recapture": ms[3] / args.steps},
        "collision_checks_per_s": {"reference_equivalent": checks_ref * world / (dev_ms / args.steps * 1e-3),
                                   "executed": checks_exec * world / (dev_ms / args.steps * 1e-3)},
        "collisions_per_step": collisions, "wall_s": wall,
        "state_digest": {"digest": ["%016x" % d for d in digest[:2]], "particles_counted": digest[2], "steps": 1 + args.warmup + args.steps},
    }

    # ---------------------------------------------------------------- config 2 beside it (rank 0, N = 1 only)
    if rank == 0 and world == 1 and not args.no_also:
        out["also"] = bench_pore_ref(args, hbm_peak)
        out["also_configs"] = bench_other_configs(args)
    if rank == 0 and world == 1 and not args.no_verify:
        out["verify"] = verify_against_oracle(cfg, state if not args.device_init else None, local)
    if rank == 0 and world == 1 and not args.no_cpu:
        out["cpu_baseline"] = cpu_baseline(steps=8, warmup=2)
        if not args.no_ref:
            out["cpu_baseline_reference"] = reference_baseline(1)
    if rank == 0:
        emit(out)
    if world > 1:
        dist.destroy_process_group()


def run_slabs(args, world, rank, local, dev, hbm_peak, peak_src, barrier, max_over_ranks, sum_over_ranks):
    """N > 1: ONE energized pore of N x particles-per-gpu particles, slab-decomposed along z over the N
    GPUs (NCCL all-to-all for migration + ghost copies, neighbour send/recv after every colour group)."""
    import torch
    import torch.distributed as dist
    from argon_monte_carlo_b200 import init_state, slab
    clocks = ClockSampler(local)
    clocks.launch()                          # nvidia-smi takes seconds to start with eight busy GPUs: long before the timed region
    cfg, scale = scaled_temp_config(args.particles_per_gpu * world)
    edges = cfg.grid.edge[2]
    _, _, _, zs, _, _, _ = init_state.synthetic_pore_chunk(cfg, 17, 0, 1 << 22)   # representative sample: regions are drawn at random
    cuts = slab.balanced_cuts(zs, edges, world)

    from argon_monte_carlo_b200 import amc
    fused = os.environ.get("AMC_SLAB_MODE", "p2p") == "p2p"     # p2p: amc_slab_step; nccl: step-wise entry points over NCCL
    sim = slab.SlabSimulation(cfg, world, zs, transport=slab.DistTransport(), local_ranks=[rank], devices=[local],
                              cuts=cuts, n_total=cfg.num_molecules, seed=17, p2p=fused)
    step = (lambda k, timing=False: sim.step_fused(k, reduce=False)) if fused else (lambda k, timing=False: sim.step(k, reduce=False, timing=timing))
    # the gas is generated on the devices (amc_init_synthetic): particle i depends only on (seed, i), so every rank
    # makes exactly its own slab and the 1-GPU replay below makes the very same job
    sim.init_synthetic(lambda kz: init_state.pore_spec(cfg, 17, keep_z=kz))
    n = sim.particles_per_rank()[0]
    step(1)                                 # (one extra untimed step: kernels loaded, peers mapped, allocations touched)
    launches0 = sim.ranks[0].sim.last_timing()[1]
    barrier()
    clocks.mark_warmup()
    step(args.warmup)
    barrier()
    clocks.start()
    det0 = sim.ranks[0].sim.last_detect_ms()
    t0 = time.perf_counter()
    stats = step(args.steps, timing=True)
    wall = time.perf_counter() - t0
    ms = sim.phase_ms
    barrier()
    clk = clocks.stop()
    if os.environ.get("AMC_SLAB_TRACE"):
        import ctypes as C
        gm = (C.c_double * 10)()
        sim.ranks[0].sim.lib.amc_debug_group_ms(sim.ranks[0].sim.h, gm)
        sys.stderr.write("rank %d group launch ms (traced steps %d): %s\n" % (rank, int(gm[9]), " ".join("%.4f" % (v / max(gm[9], 1)) for v in gm[:9])))
    launches = sim.ranks[0].sim.last_timing()[1] - launches0       # counted by the library: kernels this rank launched
    launches_timed = launches * args.steps // (args.steps + args.warmup)
    digest = sim.state_digest()                                    # id-ordered state of all ranks after warmup + steps
    dev_ms = max_over_ranks(float(ms.sum()))
    per_rank = torch.zeros(world, 5, dtype=torch.float64, device=dev)
    per_rank[rank, :4] = torch.as_tensor(ms / args.steps, dtype=torch.float64)
    per_rank[rank, 4] = float(n)
    dist.all_reduce(per_rank)
    total_particles = float(cfg.num_molecules)
    n_now = sum_over_ranks(float(sim.particles_per_rank()[0]))
    value = total_particles * args.steps / (dev_ms * 1e-3)
    pair_ms = ms[2] / args.steps
    checks_ref = sum_over_ranks(float(np.mean([s["pair_checks_ref"] for s in stats])))
    collisions = sum_over_ranks(float(np.mean([s["collisions"] for s in stats])))
    n_max = max_over_ranks(float(n))
    det_ms = max_over_ranks((sim.ranks[0].sim.last_detect_ms() - det0) / args.steps)
    roofline = {"bound": "hbm", "kernel": detect_kernel() + " (pair detection, 1 launch per step and rank; slowest rank)",
                "achieved": B_PAIR * n_max / (det_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                "peak_source": peak_src, "avg_launch_ms": det_ms, "traffic": None}
    roofline["frac"] = roofline["achieved"] / hbm_peak
    # e2e: host buffers in and out every step
    keys = ("x", "y", "z", "vx", "vy", "vz", "dist", "dist_x", "dist_y", "dist_z")
    e2e_steps = max(1, min(args.steps, 3))
    cap = int(n * 1.1) + 65536
    pinned = {k: torch.empty(cap, dtype=torch.float64).pin_memory().numpy() for k in keys}
    pinned["ids"] = torch.empty(cap, dtype=torch.int64).pin_memory().numpy()
    pinned["flag"] = torch.empty(cap, dtype=torch.uint8).pin_memory().numpy()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        (oid, od), = sim.owned(out=[pinned])
        sim.set_local_state(oid, *[od[k] for k in keys], flag=od["flag"])
        step(1)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    e2e = {"value": total_particles * e2e_steps / e2e_s, "unit": "particle-steps/s", "steps": e2e_steps,
           "h2d_bytes_per_step": int(n * 89), "d2h_bytes_per_step": int(n * 89)}
    sim.close()
    # out of band: rank 0 repeats the whole job as ONE domain on its own GPU; the N-rank run must have left the
    # same id-ordered state (order-independent checksum over all particles, amc_state_digest)
    verify = {"skipped": "--no-verify"}
    if not args.no_verify:
        verify = {"digest": ["%016x" % d for d in digest[:2]], "particles_counted": digest[2],
                  "steps": 1 + args.warmup + args.steps}
        if rank == 0:
            try:
                torch.cuda.empty_cache()
                one = amc.Simulation(cfg, seed=17, device=local, max_particles=cfg.num_molecules)
                one.init_synthetic(init_state.pore_spec(cfg, 17))
                one.step_quiet(1 + args.warmup + args.steps)
                d1 = one.state_digest()
                one.close()
                verify.update(digest_single_gpu=["%016x" % d for d in d1[:2]], identical_to_single_gpu=tuple(d1) == tuple(digest))
            except Exception as exc:
                verify["single_gpu_replay_failed"] = str(exc)[-200:]
        barrier()
    out = {
        "metric": "collision-resolved particle-steps/s", "value": value, "unit": "particle-steps/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "verify": verify,
        "config": {"workload": "temp_pore_scaled: ONE energized thruster pore (Temperature_Pore_MC geometry x %.3f), "
                               "%d particles = %d per GPU, device RNG, slab-decomposed along z over %d GPUs"
                               % (scale, cfg.num_molecules, args.particles_per_gpu, world),
                   "particles_total": int(total_particles), "cells": list(cfg.grid.nc), "cuts": [int(c) for c in cuts],
                   "particles_max_per_gpu": int(n_max),
                   "parallelism": "z slabs; migration, ghost copies and the hand-over after every colour group written peer to peer "
                                  "over NVLink by kernels (amc_slab_step), torch.distributed/NCCL for set-up and reductions only" if fused
                                  else "z slabs, NCCL all-to-all + neighbour send/recv (step-wise entry points)",
                   "l2": "inputs larger than L2"},
        "clocks": clk, "e2e": e2e, "gpu_launches": int(launches_timed),
        "roofline": roofline,
        "phases_ms_per_step": {"advect_walls": ms[0] / args.steps, "exchange_sort": ms[1] / args.steps,
                               "pairs_and_handover": ms[2] / args.steps, "pair_detect_slowest_rank": det_ms,
                               "finish": ms[3] / args.steps},
        "collision_checks_per_s": {"reference_equivalent": checks_ref / (dev_ms / args.steps * 1e-3)},
        "collisions_per_step": collisions, "wall_s": wall, "resident_particles": int(n_now),
        "per_rank": {"columns": ["advect_walls_ms", "exchange_sort_ms", "pairs_and_handover_ms", "finish_ms", "particles"],
                     "rows": [[round(float(v), 4) for v in row] for row in per_rank.cpu().tolist()]},
    }
    if rank == 0:
        emit(out)
    dist.destroy_process_group()


def bench_pore_ref(args, hbm_peak):
    """BASELINE.json config 2: Open_Air_Pore_MC.py, reference particle count, reference seeds."""
    import torch
    from argon_monte_carlo_b200 import amc, config, init_state
    cfg = config.pore_config(False)
    state = init_state.pore_initial_state(cfg)
    sim = amc.Simulation(cfg)
    sim.set_state(*state)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    for _ in range(max(args.warmup, 3)):
        sim.step_quiet(1)
    tot = np.zeros(5)
    k = max(args.steps, 10)
    for _ in range(k):
        flush.fill_(1)                      # write 512 MB > 126 MB L2 between timed steps
        torch.cuda.synchronize()
        sim.step_quiet(1)
        ms, launches = sim.last_timing()
        tot += np.array(ms)
    n = len(state[0])
    sim.close()
    return {"workload": "pore_ref: Open_Air_Pore_MC.py, N=%d, seeds 17, L2 flushed between timed steps" % n,
            "value": n * k / (tot[4] * 1e-3), "unit": "particle-steps/s", "ms_per_step": tot[4] / k,
            "phases_ms_per_step": {"keys": tot[0] / k, "scan_scatter_advect": tot[1] / k, "pairs": tot[2] / k,
                                   "recapture": tot[3] / k},
            "launches_per_step": launches, "steps": k}


def verify_against_oracle(cfg, state, device, steps=2):
    """Outside every timed region: `steps` timesteps of the benchmarked workload from its initial state on the GPU
    and through the CPU oracle; the id-ordered states must agree bit for bit (tests/test_gpu_bench_workload.py is
    the same check under pytest, pair set included)."""
    from oracle import oracle as O, steps as S
    from argon_monte_carlo_b200 import amc, config, init_state
    if state is None:
        return {"skipped": "device-initialised state"}
    O.set_ref_mode(False)
    O.set_num_threads(os.cpu_count())
    cheb = config.gap_energy_chebyshev(cfg, 16)
    sim = amc.Simulation(cfg, seed=17, cheb=cheb, device=device, max_particles=len(state[0]))
    sim.set_state(*state)
    st = O.ParticleState(*state)
    g = sim.step(steps)
    got, dig = sim.get_state(), sim.state_digest()
    sim.close()
    t0 = time.perf_counter()
    r = [S.temp_step_philox(st, cfg, 17, k, cheb) for k in range(steps)]
    ok = all(np.array_equal(got[k], getattr(st, k)) for k in O.STATE_KEYS) and np.array_equal(got["flag"].astype(bool), st.flag.astype(bool))
    ok_counts = all(a["collisions"] == b["collisions"] and a["pair_checks_ref"] == b["checks"] for a, b in zip(g, r))
    return {"against": "oracle/amc_oracle.c (CPU restatement of the reference algorithm)", "steps": steps, "particles": st.n,
            "state_bit_identical": bool(ok), "counters_identical": bool(ok_counts),
            "digest_matches": dig == amc.digest_of_arrays(np.arange(st.n), st.arrays()),
            "collisions_per_step": [int(a["collisions"]) for a in g], "oracle_s": time.perf_counter() - t0}


def reference_baseline(steps, kind="temp"):
    """SURVEY 8(d): the unmodified upstream script on the host cores (baseline/stage.py; the staged copy lives in
    the git-ignored baseline/_ref, which travels to the GPU box)."""
    try:
        sys.path.insert(0, os.path.join(ROOT, "baseline"))
        import stage
        if not stage.staged():
            return {"unavailable": "baseline/_ref not staged (python baseline/stage.py stage in the build container)"}
        return stage.run(kind, steps, timeout=1500)
    except Exception as exc:
        return {"unavailable": str(exc)[-300:]}


def bench_other_configs(args):
    """The remaining single-GPU configurations of BASELINE.json beside the headline one, each a short measurement
    (device time per step from CUDA events, L2 flushed between timed steps where the state fits into it):
    cfg 1 Open_Air_Cube_MC.py as shipped (serial sweep), cfg 3 Temperature_Pore_MC.py (device RNG), cfg 4 the
    10 M-particle cube with the colour-group schedule on one GPU."""
    import torch
    from argon_monte_carlo_b200 import amc, config, init_state
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    res = []

    def timed(sim, k, do_flush):
        sim.step_quiet(3)
        tot = np.zeros(5)
        for _ in range(k):
            if do_flush:
                flush.fill_(1)
                torch.cuda.synchronize()
            sim.step_quiet(1)
            tot += np.array(sim.last_timing()[0])
        return tot / k
    try:
        cfg = config.cube_config()
        st = init_state.cube_initial_state(cfg)
        sim = amc.Simulation(cfg)
        sim.set_state(*st)
        ms = timed(sim, 10, True)
        sim.close()
        res.append({"workload": "cfg1: Open_Air_Cube_MC.py as shipped, N=%d, serial cell sweep (reference order, event-driven: k_sweep_detect + k_sweep_events)" % len(st[0]), "ms_per_step": ms[4],
                    "value": len(st[0]) / (ms[4] * 1e-3), "unit": "particle-steps/s"})
        cfg = config.pore_config(True)
        st = init_state.pore_initial_state(cfg)
        sim = amc.Simulation(cfg, seed=17)
        sim.set_state(*st)
        ms = timed(sim, 20, True)
        sim.close()
        res.append({"workload": "cfg3: Temperature_Pore_MC.py, N=%d, energized walls, device RNG" % len(st[0]), "ms_per_step": ms[4],
                    "value": len(st[0]) / (ms[4] * 1e-3), "unit": "particle-steps/s"})
        n = 10_000_000
        base = config.cube_config()
        scale = (n / base.num_molecules) ** (1.0 / 3.0)
        n_sub = 2 * max(1, int(round(base.cube_x * scale / 21.43e-9 / 2)))
        cfg = config.cube_config(scale=scale, n_sub=n_sub)
        cfg.dt = cfg.tau / 1000
        grid = config.Grid(nc=(n_sub,) * 3, c0=(0, 0, 0), d=(cfg.dx, cfg.dy, cfg.dz), band=(cfg.collision_range,) * 3)
        sim = amc.Simulation(cfg, kind=amc.KIND_CUBE, pp_mode=amc.PP_GROUPS, grid=grid, max_particles=n)
        sim.init_synthetic(init_state.cube_spec(cfg, n, 127))
        ms = timed(sim, 10, False)
        sim.close()
        res.append({"workload": "cfg4: 10 M-particle Maxwellian cube, colour-group schedule, one GPU (2/4/8 GPUs: bench.py --workload cube --gpus N)",
                    "ms_per_step": ms[4], "value": n / (ms[4] * 1e-3), "unit": "particle-steps/s"})
    except Exception as exc:      # never lose the benchmark line over the side measurements
        res.append({"error": str(exc)[-200:]})
    return res


def cpu_baseline(steps, warmup, particles=None):
    """The oracle port on the host cores, on a bounded sample of the workload: the energized pore at
    the reference particle count (same density, cell size and step as the GPU run).  The OpenMP team is pinned
    to os.cpu_count() threads so that `cores` is the same whatever OMP_NUM_THREADS the launcher exported
    (torchrun sets it to 1)."""
    from oracle import oracle as O, steps as S
    from argon_monte_carlo_b200 import config, init_state
    O.set_ref_mode(False)
    O.set_num_threads(os.cpu_count())
    cfg = config.pore_config(True)
    cheb = config.gap_energy_chebyshev(cfg, 16)
    st = O.ParticleState(*init_state.synthetic_pore_state(cfg, seed=17))
    for k in range(warmup):
        S.temp_step_philox(st, cfg, 17, k, cheb)
    t0 = time.perf_counter()
    for k in range(steps):
        S.temp_step_philox(st, cfg, 17, warmup + k, cheb)
    dt = time.perf_counter() - t0
    return {"value": st.n * steps / dt, "unit": "particle-steps/s", "cores": O.num_threads(), "kind": "port",
            "sample": "C port of the reference algorithm (oracle/amc_oracle.c, OpenMP over cells), energized pore at "
                      "%d particles, %d steps; the unmodified Python reference measured 6.4-7.1e3 particle-steps/s "
                      "on 8 cores (BASELINE.md)" % (st.n, steps), "ms_per_step": dt / steps * 1e3}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    steps = max(1, min(args.steps, 20))
    port = cpu_baseline(steps=steps, warmup=min(args.warmup, 3))
    # the reference's own implementation of the path: the unmodified Temperature_Pore_MC.py (multiprocessing over
    # cpu_count()+1 workers), one timestep of ~1.5 min; the C port of its algorithm is reported beside it and stands
    # in when the staged copy is missing
    ref = {"unavailable": "--port-only"} if args.port_only else reference_baseline(1)
    cb = ref if "value" in ref else port
    out = {"impl": "reference", "metric": "collision-resolved particle-steps/s", "value": cb["value"],
           "unit": "particle-steps/s", "n_gpus": world, "steps": 1 if cb is ref else steps, "warmup": 0 if cb is ref else min(args.warmup, 3),
           "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f64", "data": "synthetic" if cb is port else "reference initial state (seeds 17)",
           "config": {"workload": "temp_pore_scaled (bounded sample: the same energized pore at the reference size, "
                                  "557,649 particles; throughput per particle is size-independent at fixed density)"},
           "cpu_baseline": cb, "cpu_baseline_port": port,
           "e2e": {"value": cb["value"], "unit": "particle-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if cb is port:
        out["reference_script"] = ref
    emit(out)


_REAL_STDOUT = None


def protect_stdout():
    """Libraries (NCCL prints its version banner) write to fd 1; the contract is ONE JSON line on stdout.
    Point fd 1 at stderr for the whole run and keep the real stdout for the result line."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(obj):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(obj) + "\n")
    out.flush()


def main():
    protect_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--particles-per-gpu", type=int, default=12_500_000)
    ap.add_argument("--workload", default="temp_pore", choices=["temp_pore", "cube"],
                    help="temp_pore (default, the headline workload) or cube (BASELINE config 4, secondary)")
    ap.add_argument("--cube-particles", type=int, default=10_000_000)
    ap.add_argument("--device-init", action="store_true", help="1 GPU: generate the synthetic state on the device instead of on the host")
    ap.add_argument("--no-also", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-ref", action="store_true", help="skip the 1.5-minute run of the unmodified upstream script (cpu_baseline_reference)")
    ap.add_argument("--no-verify", action="store_true", help="skip the out-of-band check against the oracle / the 1-GPU replay")
    ap.add_argument("--port-only", action="store_true", help="--impl reference: time only the C port of the reference algorithm")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="single-GPU temp_pore: after the timed steps, write the state of a seeded particle sample and the "
                         "last step's counters to DIR/<name>.npy (float64, about 50 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "temp_pore" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs is available for the single-GPU temp_pore workload of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
