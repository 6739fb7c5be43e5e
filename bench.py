#!/usr/bin/env python
"""bench.py — MD steps/s of the non-bonded + VelocityVerlet hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c3] [--dump-outputs DIR]

A "step" is one VelocityVerlet MD step (kick, drift, neighbour policy, pairwise forces, kick, CM removal)
of the workload; at N=1 the workload is BASELINE config[1]: the 256 000-atom argon LJ fluid, cubic PBC,
rc 1.2 nm, Float32 (SURVEY.md §8d C2-(ii): FCC + jitter, 90 K, dt 2 fs).

  value   device-resident: K steps inside one mb_simulate_vv call on device arrays, CUDA-event timed.
  e2e     the same metric through the reference-facing C-ABI call with HOST (pinned) buffers: every call
          uploads coords+velocities, runs `md_steps_per_call` steps and downloads them (what
          simulate!(sys, sim, n) costs a Molly user whose System lives in host memory).
  roofline  dominant kernel = brick_force_kernel; algorithmic bytes 36 B/atom/launch (SURVEY.md §8d:
          read x 12 + params 12 + write F 12) / mean launch time measured with CUDA events by the
          library's stage timers; peak = MEASURED_PEAKS.json hbm_gbs. The FP32-ALU fraction that actually
          binds this kernel is reported beside it (`fp32`).
  cpu_baseline  the oracle's restatement of Molly's multithreaded CPU algorithm (threaded cell list every 10 steps with
          the GPU arm's list radius, threaded pair loop with per-thread force copies) on the same workload, bounded sample.
  workloads  (default run only) the other configurations BASELINE.json names, shorter runs, same fields: c3 = 6mrr
          (replicas when N > 1: its box does not shard), c4 = 1M-atom LJ fluid (decomposed like c2 when N > 1).
  --dump-outputs DIR  after the timed steps of each workload <w>, the coordinates and velocities a caller of simulate()
          holds (float32, every atom) are written to DIR/<w>_coords.npy and DIR/<w>_velocities.npy. The inputs are seeded,
          so two builds run with the same arguments can be compared output for output (c2 and c4 repeat bit for bit on a B200;
          c3 does not: two runs of the default line differed by up to 3.4e-4 nm after its 40 + 400 steps).
  N > 1   spatial decomposition of ONE system (strong scaling); roofline / fp32 use the per-rank share of bytes and pairs
          and the slowest rank's kernel time.

--impl reference times that CPU restatement alone (Julia is not installed, so Molly.jl itself cannot run;
kind = "port").
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
for p in (os.path.join(ROOT, "tests"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import mbhelpers as H  # noqa: E402

METRIC = "md_steps_per_sec"
UNIT = "steps/s"


def workload(name: str, dtype):
    """Returns (system description, mollyb200 interactions factory, oracle interactions, dt, r_cut, label)."""
    import mollyb200 as mb
    from oracle import oracle as o
    if name == "c2":
        sd = H.lj_fluid(40, seed=42, dtype=dtype)  # 256 000 atoms, L = 22.977 nm
        rc = 1.2
        inters = (mb.LennardJones(cutoff=mb.DistanceCutoff(rc), use_neighbors=True),)
        ointers = [o.Inter(o.LJ, o.CUT_DISTANCE, rc, use_neighbors=True)]
        return sd, inters, ointers, 0.002, rc, "256k-atom LJ fluid, cubic PBC, 1.2nm cutoff, Float32"
    if name == "c4":
        sd = H.lj_fluid(63, seed=42, dtype=dtype)  # 1 000 188 atoms
        rc = 1.2
        inters = (mb.LennardJones(cutoff=mb.DistanceCutoff(rc), use_neighbors=True),)
        ointers = [o.Inter(o.LJ, o.CUT_DISTANCE, rc, use_neighbors=True)]
        return sd, inters, ointers, 0.002, rc, "1M-atom LJ fluid, cubic PBC, 1.2nm cutoff, Float32"
    if name == "c3":
        g = dict(np.load(os.path.join(ROOT, "tests", "golden", "6mrr.npz")))
        sd = H.sixmrr_description(g)
        sd = dict(sd, coords=sd["coords"].astype(dtype), velocities=sd["velocities"].astype(dtype), golden=g)
        w_lj, w_c = float(g["lj14scale"]), float(g["coulomb14scale"])
        inters = (mb.LennardJones(cutoff=mb.DistanceCutoff(1.0), use_neighbors=True, weight_special=w_lj),
                  mb.CoulombReactionField(dist_cutoff=1.0, use_neighbors=True, weight_special=w_c))
        ointers = [o.Inter(o.LJ, o.CUT_DISTANCE, 1.0, weight_special=w_lj, use_neighbors=True),
                   o.Inter(o.CRF, o.CUT_DISTANCE, 1.0, weight_special=w_c, use_neighbors=True)]
        return sd, inters, ointers, 0.0005, 1.0, ("6mrr solvated protein (15 954 atoms), AMBER ff99SBildn + TIP3P, LJ + "
                                                  "CoulombReactionField + bonds/angles/torsions, VelocityVerlet + Andersen, Float32")
    raise SystemExit(f"unknown workload {name}")


# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [t.strip() for t in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                smax.append(float(f[1]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def default_r_list(wl, rc):
    """List radius = cutoff + skin. The skins are tuned on B200 (profiles/r02_experiments.md section 8): 0.08 nm for C2 (a rebuild every
    ~36 steps), 0.10 nm for C4 (its rebuild costs 4x as much), 0.12 nm for 6mrr at 300 K / 0.5 fs. Both arms use the same radius."""
    return rc + {"c2": 0.08, "c3": 0.12, "c4": 0.10}.get(wl, 0.10)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(workload_name: str):
    """DRAM bytes per launch of the force kernel from the committed ncu capture, if any."""
    p = os.path.join(ROOT, "profiles", f"force_kernel_{workload_name}.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("dram_bytes_per_launch")
        except Exception:
            return None
    return None


# ----------------------------------------------------------------------------------------------------
def run_cpu(sd, ointers, dt, rc, steps, warmup, dtype=np.float32, r_list=None):
    """Molly-algorithm CPU restatement (oracle): threaded cell list every 10 steps (the reference's find_neighbors policy,
    src/neighbors.jl:671) with the GPU arm's list radius, threaded pair loop, all host threads."""
    if r_list is None:
        r_list = rc + (0.12 if "golden" in sd else 0.10)
    from oracle import oracle as o
    if "golden" in sd:  # 6mrr: pairwise in C (threaded), bonded terms in numpy, f64
        try:
            import psutil
            o.DEFAULT_THREADS = max(o.max_threads(), psutil.cpu_count(logical=False) or 1)  # not OMP_NUM_THREADS=1 of a launcher
        except Exception:
            pass
        t0 = time.perf_counter()
        H.oracle_vv_with_bonded(sd["golden"], sd["coords"].astype(np.float64), sd["velocities"].astype(np.float64), dt, steps,
                                r_list=r_list, nl_every=10)
        t = time.perf_counter() - t0
        return steps / t, o.max_threads(), t
    orc = H.make_oracle(sd, ointers, dtype=dtype)
    # "all the host threads it can use": one thread per logical CPU is often slower than one per physical core for this
    # memory-bound loop, so both are timed on the same sample and the faster one is reported
    cands = {o.max_threads()}
    try:
        import psutil
        phys, logical = psutil.cpu_count(logical=False), psutil.cpu_count(logical=True)
        cands |= {c for c in (phys, logical) if c}
    except Exception:
        pass
    best = None
    x0, v0 = sd["coords"].astype(dtype), sd["velocities"].astype(dtype)
    for nt in sorted(cands):
        x, v = x0, v0
        if warmup > 0:
            x, v, _ = orc.simulate_vv(x, v, dt, warmup, remove_cm_every=1, r_list=r_list, nl_every=10, n_threads=nt)
        t0 = time.perf_counter()
        orc.simulate_vv(x, v, dt, steps, remove_cm_every=1, r_list=r_list, nl_every=10, n_threads=nt)
        t = time.perf_counter() - t0
        if best is None or steps / t > best[0]:
            best = (steps / t, nt, t)
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=["c2", "c3", "c4"])
    ap.add_argument("--r-list", type=float, default=None)
    ap.add_argument("--rebuild-every", type=int, default=0, help="0 = displacement-triggered (exact)")
    ap.add_argument("--brick", type=int, nargs=3, default=(0, 0, 0))
    ap.add_argument("--lanes", type=int, default=0)
    ap.add_argument("--md-steps-per-call", type=int, default=100)
    ap.add_argument("--cpu-steps", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cm", action="store_true", help="diagnostic: remove_CM_motion=false")
    ap.add_argument("--replicas", action="store_true", help="N>1: independent replicas instead of the spatial decomposition")
    ap.add_argument("--no-extra", action="store_true", help="only the primary workload (no `workloads` object)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write each workload's coordinates and velocities after its timed steps to DIR/<workload>_<name>.npy")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n_gpus = args.gpus
    wl = args.workload or "c2"
    dtype = np.float32

    # ------------------------------------------------------------------ reference arm (CPU restatement)
    if args.impl == "reference":
        if rank != 0:
            return
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes the GPU arm's outputs; the reference arm keeps no state to dump")
        sd, inters, ointers, dt, rc, label = workload(wl, dtype)
        steps = args.steps if args.steps is not None else (10 if wl != "c3" else 100)
        steps = min(steps, 20 if wl == "c2" else (10 if wl == "c4" else 60))  # bounded sample ...
        steps = 10 * max(1, steps // 10)  # ... of whole neighbour-list periods (Molly's default: find_neighbors every 10 steps)
        warm = min(args.warmup if args.warmup is not None else 1, 2)
        r_list = args.r_list if args.r_list is not None else default_r_list(wl, rc)
        sps, nt, t = run_cpu(sd, ointers, dt, rc, steps, warm, r_list=r_list)
        out = {"impl": "reference", "metric": METRIC, "value": sps, "unit": UNIT, "n_gpus": n_gpus, "steps": steps,
               "warmup": warm, "ms_per_step": 1e3 / sps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
               "dtype": "f32", "data": "synthetic",
               "config": {"workload": label, "n_atoms": int(sd["n"]), "dt_ps": dt, "r_cut_nm": rc, "r_list_nm": r_list},
               "cpu_baseline": {"value": sps, "unit": UNIT, "cores": nt, "kind": "port",
                                "sample": cpu_sample_text(steps, t, r_list) + "; Julia is not installed"},
               "e2e": {"value": sps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
               "ns_per_day": sps * dt * 1e3 * 0.0864}
        print(json.dumps(out))
        return

    # ------------------------------------------------------------------ our arm
    import torch
    import mollyb200 as mb
    if not torch.cuda.is_available() or mb.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = dict(rank=rank, world=world, local_rank=local_rank, dist=dist, n_gpus=n_gpus)
    steps = args.steps if args.steps is not None else (1000 if wl != "c4" else 300)
    warmup = max(args.warmup if args.warmup is not None else 100, 3)
    out = run_ours(wl, args, ctx, steps, warmup, with_cpu=not args.no_cpu_baseline, with_e2e=not args.no_e2e)
    # The other configurations BASELINE.json names ride in the same line (shorter runs): C3 = 6mrr (one GPU: the 5.7 nm box
    # does not shard, extra GPUs run replicas), C4 = 1M-atom LJ fluid (spatially decomposed like C2 when N > 1).
    if args.workload is None and not args.no_extra:
        extra = {}
        for w2, st2, wu2 in (("c3", min(steps, 400), min(warmup, 40)), ("c4", min(steps, 120), min(warmup, 20))):
            try:
                extra[w2] = run_ours(w2, args, ctx, max(st2, 5), max(wu2, 3), with_cpu=False, with_e2e=not args.no_e2e, brief=True)
            except Exception as e:  # the primary line must survive an extra workload's failure
                extra[w2] = {"error": f"{type(e).__name__}: {e}"[:300]}
        if rank == 0:
            out["workloads"] = extra
    if rank == 0:
        print(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()


def run_ours(wl, args, ctx, steps, warmup, with_cpu, with_e2e, brief=False):
    """One workload on this arm; returns the JSON fields (rank 0) or None (other ranks)."""
    import torch
    import mollyb200 as mb
    rank, world, local_rank, dist, n_gpus = ctx["rank"], ctx["world"], ctx["local_rank"], ctx["dist"], ctx["n_gpus"]
    dtype = np.float32
    sd, inters, ointers, dt, rc, label = workload(wl, dtype)
    n = int(sd["n"])
    r_list = args.r_list if args.r_list is not None else default_r_list(wl, rc)

    atoms = mb.atoms_from_arrays(sd["mass"], sd["charge"], sd["sigma"], sd["eps"], dtype)
    nf = mb.GPUNeighborFinder(dist_cutoff=r_list, excluded_pairs=sd.get("excluded", np.zeros((0, 2), np.int32)) + 1,
                              special_pairs=sd.get("special", np.zeros((0, 2), np.int32)) + 1, n_steps=args.rebuild_every)
    dev = torch.device("cuda", local_rank)
    xs = torch.from_numpy(sd["coords"].astype(dtype)).to(dev).contiguous()
    vs = torch.from_numpy(sd["velocities"].astype(dtype)).to(dev).contiguous()
    specific = H.sixmrr_specific_lists(sd["golden"]) if "golden" in sd else ()
    sysm = mb.System(atoms=atoms, coords=xs, boundary=mb.CubicBoundary(*sd["box"]), velocities=vs, pairwise_inters=inters,
                     neighbor_finder=nf, dtype=dtype, device=local_rank, specific_inter_lists=specific)
    sysm.engine()
    if any(args.brick) or args.lanes:
        sysm.set_launch_config(tuple(args.brick), args.lanes)
    # C3's 5.7 nm box is smaller than 2.5 r_list per slab for any N > 1: replicas only (DESIGN.md section 5)
    decomposed = world > 1 and not args.replicas and wl != "c3"
    if decomposed:
        # spatial decomposition: z-slabs, halo exchange inside the library; torch.distributed only ships the id
        uid = [mb.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        mb.comm_init(sysm, uid[0], rank, world)
    coupling = mb.AndersenThermostat(300.0, 1.0) if wl == "c3" else None  # config 3: VelocityVerlet + Andersen
    sim = mb.VelocityVerlet(dt=dt, coupling=coupling, remove_CM_motion=0 if args.no_cm else 1)
    rng = np.random.default_rng(1234 + rank)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        tt = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    # warm-up (also builds the neighbour structure and derives capacities)
    mb.simulate(sysm, sim, warmup, rng=rng)
    st0 = sysm.stats()
    # ---- timed device-resident region: exactly `steps` MD steps
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    mb.simulate(sysm, sim, steps, init_step=warmup, rng=rng)
    ev1.record()
    barrier()
    t_ms = max_over_ranks(ev0.elapsed_time(ev1))
    clocks = sampler.stop() if rank == 0 else None
    st1 = sysm.stats()
    if args.dump_outputs and rank == 0:  # before the profiled run below advances the state
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in (("coords", xs), ("velocities", vs)):
            np.save(os.path.join(args.dump_outputs, f"{wl}_{name}.npy"), t.cpu().numpy())
    # decomposed: all ranks advance ONE system; replicas: every rank advances its own copy
    mult = 1 if decomposed or world == 1 else world
    value = mult * steps / (t_ms * 1e-3)
    launches = st1["kernel_launches"] - st0["kernel_launches"]

    # ---- stage timers (separate short run so the event records do not perturb the number above)
    prof_steps = min(200, steps)
    sysm.set_profiling(True)
    barrier()  # decomposed runs: a late rank would show up as waiting time inside its neighbours' kernels
    mb.simulate(sysm, sim, prof_steps, init_step=warmup + steps, rng=rng)
    stp = sysm.stats()
    sysm.set_profiling(False)
    force_us = max_over_ranks(1e3 * stp["force_ms"] / max(stp["force_launches"], 1))  # slowest rank's kernel
    vv_us = max_over_ranks(1e3 * stp["vv_ms"] / max(stp["vv_launches"], 1))
    rebuilds_prof = stp["n_rebuilds"] - st1["n_rebuilds"]
    # stream mode enqueues the gated rebuild pipeline every step (2-3 us no-op kernels unless the flag is set), so this
    # total is an upper bound of the real rebuild cost; profiles/r02_launches_*.md has the per-kernel numbers
    rebuild_total_ms = stp["rebuild_ms"]

    # ---- e2e through the C ABI with host (pinned) buffers
    e2e = None
    if with_e2e:
        spc = min(args.md_steps_per_call, max(steps, 5))
        hx = torch.empty((n, 3), dtype=torch.float32).pin_memory()
        hv = torch.empty((n, 3), dtype=torch.float32).pin_memory()
        hx.copy_(xs.cpu())
        hv.copy_(vs.cpu())
        hsys = mb.System(atoms=atoms, coords=hx.numpy(), boundary=mb.CubicBoundary(*sd["box"]), velocities=hv.numpy(),
                         pairwise_inters=inters, neighbor_finder=nf, dtype=dtype, device=local_rank,
                         specific_inter_lists=specific)
        hsys.engine()
        if any(args.brick) or args.lanes:
            hsys.set_launch_config(tuple(args.brick), args.lanes)
        if decomposed:
            uid = [mb.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            mb.comm_init(hsys, uid[0], rank, world)
        ncalls = max(3, steps // spc)
        mb.simulate(hsys, sim, spc, rng=rng)  # warm-up calls (first build)
        mb.simulate(hsys, sim, spc, init_step=spc, rng=rng)
        mb.simulate(hsys, sim, spc, init_step=2 * spc, rng=rng)
        barrier()
        t0 = time.perf_counter()
        for c in range(ncalls):
            mb.simulate(hsys, sim, spc, init_step=(3 + c) * spc, rng=rng)  # H2D + spc steps + D2H, synchronous
        torch.cuda.synchronize()
        t_e2e = max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": mult * ncalls * spc / t_e2e, "unit": UNIT, "h2d_bytes_per_step": 2 * n * 3 * 4,
               "d2h_bytes_per_step": 2 * n * 3 * 4, "md_steps_per_call": spc, "calls": ncalls,
               "note": "one 'step' of the e2e region = one simulate!-style call of md_steps_per_call MD steps with host "
                       "coords+velocities uploaded and downloaded inside the timed region"}
        hsys.close()

    # ---- CPU baseline on rank 0 (bounded sample), same r_list as the GPU arm
    cpu = None
    if rank == 0 and n_gpus == 1 and with_cpu:
        cs = args.cpu_steps or (10 if wl == "c2" else (3 if wl == "c4" else 40))
        sps, nt, t = run_cpu(sd, ointers, dt, rc, cs, 1, r_list=r_list)
        cpu = {"value": sps, "unit": UNIT, "cores": nt, "kind": "port", "sample": cpu_sample_text(cs, t, r_list)}

    out = None
    if rank == 0:
        peak, peak_src = measured_peaks()
        share = world if decomposed else 1          # a decomposed rank's kernel covers 1/world of the atoms and pairs
        alg_bytes = 36.0 * n / share                # SURVEY.md section 8d: force-only call, f32, per launch of the timed kernel
        step_bytes = 140.0 * n / share              # whole step: K1 64 + force 36 + K2 40 B/atom
        achieved = alg_bytes / (force_us * 1e-6) / 1e9 if force_us > 0 else None
        step_gbs = step_bytes / (t_ms / steps * 1e-3) / 1e9
        pairs_in_cut = {"c2": 1.955e7, "c4": 7.64e7, "c3": 2.63e6}[wl]
        flop_per_pair = 42.0 if wl != "c3" else 50.0
        fp32_peak = 148 * 128 * 2 * (clocks["sm_mhz"] or 1965.0) * 1e6 / 1e12 if clocks else None
        fp32_ach = (pairs_in_cut / share) * flop_per_pair / (force_us * 1e-6) / 1e12 if force_us > 0 else None
        par = ("single GPU" if world == 1 else (
            f"spatial decomposition: {world} z-slabs; per step: "
            + ("halo positions stored into the neighbours' extended arrays over NVLink peer memory by the drift kernel, "
               "24-byte all-to-all of sum(m v) by the kick kernel" if st1.get("peer_transport")
               else "NCCL send/recv halo exchange + 24-byte all-reduce")
            + f"; rebuild interval {st1.get('reserved_', 0)} steps (adapted from displacements)"
            if decomposed else f"{world} independent replicas (one per GPU)"))
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": steps, "warmup": warmup,
            "ms_per_step": t_ms / steps, "higher_is_better": True,
            # fixed-size systems: more GPUs share the same atoms (strong); replicas multiply the work (weak)
            "scaling": "weak" if (world > 1 and not decomposed) else "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": label, "n_atoms": n, "dt_ps": dt, "r_cut_nm": rc, "r_list_nm": r_list,
                       "rebuild_policy": "displacement-triggered" if args.rebuild_every == 0 else f"every {args.rebuild_every}",
                       "parallelism": par,
                       "brick_dims": st1["brick_dims"], "list_stride": st1["list_stride"], "n_bricks": st1["n_bricks"],
                       "l2": "not flushed between steps: step k+1 consumes the state step k wrote; per-step working set = "
                             f"{(st1['n_list_entries'] * 2 + n * 100) / 1e6:.0f} MB (neighbour list + state) vs 126 MB L2"},
            "ns_per_day": value * dt * 1e3 * 0.0864,
            "gpu_launches": int(launches),
            "rebuilds_in_timed_region": int(st1["n_rebuilds"] - st0["n_rebuilds"]),
            "violations": int(st1["violations"]),
            "clocks": clocks,
            "e2e": e2e,
            "roofline": {"bound": "hbm", "kernel": "brick_force_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak) if achieved else None, "traffic": ncu_traffic(wl), "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg_bytes, "launch_us": force_us,
                         "per_rank_share": f"1/{share} of the atoms per launch (slowest rank's kernel time)",
                         "whole_step": {"algorithmic_bytes": step_bytes, "achieved": step_gbs, "frac": step_gbs / peak}},
            "fp32": {"achieved_tflops": fp32_ach, "peak_tflops": fp32_peak,
                     "frac": (fp32_ach / fp32_peak) if (fp32_ach and fp32_peak) else None,
                     "convention": f"{flop_per_pair:.0f} flop per in-cutoff pair x {pairs_in_cut / share:.3g} pairs per rank (SURVEY.md §8d)",
                     "pair_interactions_per_s": pairs_in_cut * value / mult},
            "stage_us": {"force": force_us, "vv_kernels_mean": vv_us,
                         "rebuild_pipeline_total_ms_stream_mode": rebuild_total_ms,
                         "rebuilds_during_profile": int(rebuilds_prof), "profile_steps": prof_steps},
            "cpu_baseline": cpu,
        }
        if brief:
            for k in ("higher_is_better", "vs_baseline", "data", "cpu_baseline", "warmup"):
                out.pop(k, None)
    sysm.close()
    return out


def cpu_sample_text(steps, seconds, r_list):
    return (f"{steps} MD steps of the same workload in {seconds:.1f} s (oracle restatement of Molly's threaded CPU path: threaded "
            f"cell-list build every 10 steps like CellListMap's parallel map_pairwise!, threaded pair loop with per-thread force "
            f"copies; r_list = {r_list:.2f} nm as on the GPU arm)")


if __name__ == "__main__":
    main()
