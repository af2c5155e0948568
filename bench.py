#!/usr/bin/env python
"""Headline benchmark: column*wavelength*layer flux updates per second of the fused RCE step.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (default)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU code on the host cores
    python bench.py --gpus N --steps K --dump-outputs DIR    # default workload: also write rank 0's outputs as DIR/*.npy

Workload (BASELINE.json configs[3]): 65,536-column synthetic perturbed-profile ensemble PER GPU,
repwvl-100 table (100 wavelengths x 20 layers x 30 angles), one "step" = one full reference loop
iteration (main.cpp:531-583) for every column.  Columns shard over the ranks with no data-path
collective (weak scaling); the only inter-GPU traffic is the per-step allreduce of four scalars.
Prints ONE JSON line on rank 0.  See DESIGN.md "Measurement" for the roofline definitions.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")

NLAY = 20
METRIC = "column*wavelength*layer flux updates/s (repwvl-100 RCE step)"
UNIT = "updates/s"

# FP64-pipe work per unit (one column x wavelength x layer through one step), counted on the REFERENCE's
# expression tree (SURVEY.md section 8(d), Appendix A): 31 exp, 33 divides, ~520 add/mul/fma.
ALG_EXP, ALG_DIV, ALG_FMA = 31, 33, 520
# FP64-pipe instructions this repo's kernels really execute per unit, and DRAM bytes per column-step, come from the
# ncu capture recorded in profiles/roofline_capture.json (written by tools/update_roofline_capture.py from the raw
# ncu CSVs) together with the sha256 of the kernel sources the capture was taken on: when the sources move without a
# new capture the line says "stale": true (and tests/test_host.py fails).
CAPTURE_JSON = os.path.join(ROOT, "profiles", "roofline_capture.json")
KERNEL_SOURCES = ["rcm_kernels.cuh", "rcm_device_math.cuh", "rcm_step_kernel.cuh", "rcm_split_kernels.cuh",
                  "rcm_split_unit_loop.inc", "rcm_lbl_kernels.cuh"]


def kernel_sources_sha():
    import hashlib
    h = hashlib.sha256()
    for f in KERNEL_SOURCES:
        with open(os.path.join(ROOT, "our_first_climate_model_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def load_capture():
    with open(CAPTURE_JSON) as f:
        cap = json.load(f)
    cap["current_sha"] = kernel_sources_sha()
    cap["stale"] = cap["current_sha"] != cap.get("sources_sha256")
    return cap


def _env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def build_ensemble(rcm, ncol, seed):
    atm = rcm.read_atm(os.path.join(GOLDEN, "column21.atm"))
    pl = atm[:, 1].copy()
    Tlev, vlev = rcm.make_ensemble(ncol, seed, pl, atm[:, 2].copy(), atm[:, 4:9].T.copy())
    st = rcm.init_columns(pl, Tlev, vlev)
    st["plevel"] = pl
    st["Tsurf"] = np.full(ncol, 288.2)  # main.cpp:357
    return st


class ClockSampler:
    """ONE nvidia-smi process (on rank 0) samples clocks / throttle reasons of the first `ngpu` GPUs every 20 ms.  It is
    started well before the timed region (nvidia-smi needs a while to deliver its first row, longer with 8 GPUs);
    window() marks the timed region, stop() evaluates the rows that arrived inside it."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, ngpu):
        self.ngpu, self.rows, self.proc, self.t0, self.t1 = ngpu, [], None, None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def wait_first(self, timeout=10.0):
        t = time.time()
        while self.proc is not None and not self.rows and time.time() - t < timeout:
            time.sleep(0.02)

    def window(self, t0, t1):
        self.t0, self.t1 = t0, t1

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        per = {}
        mx, reasons, n_in = None, set(), 0
        # rows of the timed region (one sampling period of slack on both sides: a row describes the 20 ms before it)
        for ts, r in self.rows:
            try:
                idx, sm, mxr = int(r[0]), float(r[1]), float(r[2])
            except (ValueError, IndexError):
                continue
            if idx >= self.ngpu or (self.t0 is not None and not (self.t0 - 0.01 <= ts <= self.t1 + 0.06)):
                continue
            n_in += 1
            mx = mxr
            per.setdefault(idx, []).append(sm)
            for nm, v in zip(names, r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        med = {i: statistics.median([x for x in v if mx and x > 0.5 * mx] or v) for i, v in per.items()}
        allv = [x for v in per.values() for x in v]
        busy = [x for x in allv if mx and x > 0.5 * mx] or allv
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": n_in, "per_gpu_sm_mhz": {"min": min(med.values()), "max": max(med.values())} if med else None,
                "gpus_sampled": len(per)}


# ------------------------------------------------------------------------------------------------------
# CPU reference arm / baseline: the reference's own code (oracle/_ref, built from /root/reference) on all
# host cores, one process per core (BASELINE.md section 3), or the plain-C port when _ref is not there.
# ------------------------------------------------------------------------------------------------------
def _cpu_worker(args):
    kind, table, seed, ncol, nsteps = args[:5]
    os.environ["RCM_SHIM_REREAD"] = "1" if len(args) > 5 and args[5] else "0"  # literal flavour: table file re-read every step
    import our_first_climate_model_b200 as rcm
    st = build_ensemble(rcm, ncol, seed)
    solar = rcm.solar_setup()["solar_irr"]
    t0 = time.perf_counter()
    if kind == "reference":
        from oracle import refcpu as R
        R.advance(table, st["plevel"], st["rel_hum"], solar, st["Tlayer"], st["Tsurf"], st["vmr9"], nsteps)
    else:
        from oracle import port as P
        P.advance(P.load_rcmtab(table), st["plevel"], st["rel_hum"], solar, st["Tlayer"], st["Tsurf"], st["vmr9"],
                  nsteps)
    return time.perf_counter() - t0


def cpu_throughput(nwvl, cols_per_core, nsteps, repeats=1, reread=False):
    """-> (units/s over all cores, cores, kind, per-repeat wall times).  reread: the literal flavour of BASELINE.md 3.4(b) -
    read_tau opens and reads the table file at every step as main.cpp:564-566 does (reference build only)."""
    import multiprocessing as mp
    from oracle import refcpu as R
    kind = "reference" if R.available() else "port"
    if kind == "port":
        from oracle import port as P
        P.build()
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    table = os.path.join(GOLDEN, f"Reduced{nwvl}Forcing.rcmtab")
    walls = []
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        pool.map(_cpu_worker, [(kind, table, 1, 2, 1)] * cores)  # load libraries, page in the table
        for rep in range(repeats):
            t0 = time.perf_counter()
            pool.map(_cpu_worker, [(kind, table, 1000 + i, cols_per_core, nsteps, reread) for i in range(cores)])
            walls.append(time.perf_counter() - t0)
    units = cores * cols_per_core * nsteps * nwvl * NLAY
    return units / statistics.median(walls), cores, kind, walls


def workload_config(ncol, nwvl, world):
    """`config` of the JSON line - the same for this repo's arm and the reference arm."""
    return {"workload": f"{ncol}-column synthetic perturbed-profile ensemble per GPU, repwvl-{nwvl} "
                        "RCE step (BASELINE configs[3])", "columns_per_gpu": ncol, "nwvl": nwvl,
            "nlayer": NLAY, "nangle": 30, "parallelism": f"columns sharded over {world} GPU(s)",
            "l2": "no flush: per-step working set (state + fluxes, ~130 MB at 65,536 columns) exceeds the "
                  "126 MB L2 and the kernel is FP64-pipe bound (DRAM < 1% of peak)"}


def run_reference(args, rank, world):
    if rank != 0:
        return 0
    cols = args.cpu_cols
    # every "step" is one bounded sample: cols columns x 1 reference iteration per core, all cores busy
    vals = []
    cores = kind = None
    for i in range(args.warmup + args.steps):
        v, cores, kind, walls = cpu_throughput(args.nwvl, cols, 1)
        if i >= args.warmup:
            vals.append((v, walls[0]))
    value = statistics.median(v for v, _ in vals)
    ms = 1e3 * statistics.median(w for _, w in vals)
    sample = f"{cols} columns x 1 step per core on {cores} cores per bench step, table cached in RAM"
    # the literal flavour (BASELINE.md 3.4(b)): the same sample with the table file re-opened and re-read at every
    # read_tau call, i.e. once per column-step, as the reference driver does (main.cpp:564-566); reported beside, not instead
    literal = None
    if kind == "reference":
        lv, _, _, lw = cpu_throughput(args.nwvl, cols, 1, reread=True)
        literal = {"value": lv, "unit": UNIT, "sample": f"{cols} columns x 1 step per core, table file re-read by every "
                   f"read_tau (page cache warm), {lw[0]:.1f} s wall"}
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            # the same `config` as this repo's arm; what a bench step of this arm is: see cpu_baseline.sample
            "config": workload_config(args.ncol, args.nwvl, args.gpus),
            "sample": f"each bench step = {cols} columns x 1 reference iteration (main.cpp:531-583) per host core, a bounded "
                      f"sample of that workload",
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample, "literal_reread": literal},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------------
def bind_to_gpu_numa(torch, local_rank):
    """Best effort: run this rank (and first-touch its pinned buffers) on the NUMA node its GPU hangs off."""
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        nodes = [d for d in os.listdir("/sys/devices/system/node") if re.fullmatch(r"node\d+", d)]
        if node < 0 or len(nodes) < 2:
            return {"node": node, "nodes": len(nodes), "bound": False}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"node": node, "nodes": len(nodes), "bound": bool(cpus)}
    except Exception as e:  # noqa: BLE001 - purely advisory
        return {"bound": False, "why": str(e)[:80]}


def gather_floats(rdist, torch, x, world):
    """One float per rank -> list over ranks (device all_gather; world == 1: [x])."""
    if world == 1:
        return [float(x)]
    import torch.distributed as dist
    t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
    out = torch.zeros(world, dtype=torch.float64, device="cuda")
    dist.all_gather_into_tensor(out, t)
    return [float(v) for v in out.cpu()]


def timed_loop(torch, rdist, stream, world, steps, one_step, finish):
    """EXACTLY `steps` calls of one_step(), bracketed by barrier + synchronize, CUDA events on the launching stream;
    `finish()` (the read of the last collective) is inside the timed region.  -> (ms max over ranks, finish() value)"""
    if world > 1:
        rdist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        one_step()
    res = finish()
    e1.record(stream)
    if world > 1:
        rdist.barrier()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    return (rdist.max_over_ranks(ms) if world > 1 else ms), res


DUMP_LIMIT_BYTES = 64 * 10**6 - (1 << 16)  # 64 MB in all, .npy headers included


def dump_outputs(out_dir, state, scalars, seed=2024):
    """Writes the solver state after the last timed step (per-column arrays, as rcm_get_state returns them) and that step's
    ensemble scalars as <out_dir>/<name>.npy, so that two builds run with the same arguments can be compared array for
    array.  Above DUMP_LIMIT_BYTES a fixed, seeded sample of the columns is written; columns.npy names the ones kept."""
    ncol = next(iter(state.values())).shape[0]
    per_col = sum(a.nbytes for a in state.values()) // ncol + 8  # + the float64 column index
    keep = max(1, (DUMP_LIMIT_BYTES - scalars.nbytes) // per_col)
    cols = np.arange(ncol) if ncol <= keep else np.sort(np.random.default_rng(seed).choice(ncol, size=keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in state.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a[cols])
    np.save(os.path.join(out_dir, "columns.npy"), cols.astype(np.float64))
    np.save(os.path.join(out_dir, "step_scalars.npy"), scalars.astype(np.float64))


def oracle_parity(rcm, st, solver, nsteps, nwvl, n_check=64, seed=2024):
    """Ties the timed run to the oracle: n_check seeded members of THIS run's ensemble are taken through the same
    `nsteps` iterations by the reference (oracle/_ref, else the C port) from the initial state and compared with
    the solver's state after the timed region."""
    from oracle import refcpu as R
    rng = np.random.default_rng(seed)
    idx = np.sort(rng.choice(st["Tlayer"].shape[0], size=min(n_check, st["Tlayer"].shape[0]), replace=False))
    out = solver.get_state()
    solar = rcm.solar_setup()["solar_irr"]
    table = os.path.join(GOLDEN, f"Reduced{nwvl}Forcing.rcmtab")
    args = (st["plevel"], st["rel_hum"][idx], solar, st["Tlayer"][idx], st["Tsurf"][idx], st["vmr9"][idx], nsteps)
    if R.available():
        ref, kind = R.advance(table, *args), "reference"
    else:
        from oracle import port as P
        ref, kind = P.advance(P.load_rcmtab(table), *args), "port"
    scale = np.abs(ref["E_up"]).max(axis=1, keepdims=True)
    rel = max(float(np.max(np.abs(out[k][idx] - ref[k]) / scale)) for k in ("E_up", "E_down"))
    rel_dE = float(np.max(np.abs(out["dE"][idx] - ref["dE"]) / scale))
    dT = float(np.max(np.abs(out["Tlayer"][idx] - ref["Tlayer"])))
    return {"oracle": kind, "n_checked": int(idx.size), "steps": int(nsteps), "max_rel_flux": rel, "max_rel_dE": rel_dE,
            "max_abs_dT": dT, "tolerance": 1e-9, "ok": bool(rel < 1e-9 and rel_dE < 1e-9 and dT < 1e-6)}


def run_b200(args, rank, world, local_rank):
    import torch
    import our_first_climate_model_b200 as rcm
    from our_first_climate_model_b200 import distributed as rdist

    if not torch.cuda.is_available() or rcm.device_count() == 0:
        raise SystemExit("bench.py: no CUDA device - the solver has no CPU fallback")
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa(torch, local_rank)
    if world > 1:
        rdist.init("nccl")
    ncol = args.ncol
    st = build_ensemble(rcm, ncol, 12345 + rank)
    solver = rcm.Solver(local_rank)
    stream = torch.cuda.Stream()  # the solver launches on this torch stream: events and NCCL see its work
    torch.cuda.set_stream(stream)
    solver.set_stream(stream.cuda_stream)
    solver.set_repwvl_table_from(rcm.Table(os.path.join(GOLDEN, f"Reduced{args.nwvl}Forcing.rcmtab")))
    solver.set_columns(st["plevel"], st["Tlayer"], st["Tsurf"], st["vmr9"], st["rel_hum"])
    nwvl = solver.nwvl
    units_per_step = ncol * nwvl * NLAY

    sampler = None
    if rank == 0:  # one nvidia-smi for all the GPUs of the job, started long before the timed region
        sampler = ClockSampler(world)
        sampler.start()
    peaks = {}
    if rank == 0:
        for i, nm in enumerate(("dfma", "exp", "div", "exp_solver")):
            peaks[nm] = solver.fp64_microbench(i)  # 1e9 ops/s

    exch = rdist.StepScalarExchange(torch.device("cuda", local_rank), ring=args.ring, solver=solver)

    def one_step():
        ptr = solver.advance_async(1)  # K5 + unit kernel + K5 + scalar reduction, all on `stream`
        # the per-step collective: one asynchronous 32-byte all_gather per step (no stall, see StepScalarExchange)
        exch.submit(rdist.device_view(ptr, 4))

    for _ in range(args.warmup):
        one_step()
    exch.latest()  # also loads the handful of torch kernels the read-out uses before the clock starts
    torch.cuda.synchronize()
    if sampler is not None:
        sampler.wait_first()
    solver.kernel_time_ms(reset=True)
    l0 = solver.launch_count()
    t_w0 = time.time()
    ms_total, scal = timed_loop(torch, rdist, stream, world, args.steps, one_step, exch.latest)
    toa_mean = float(scal[0]) / (world * ncol)
    clocks = None
    if sampler is not None:
        sampler.window(t_w0, time.time())
        clocks = sampler.stop()
    launches = solver.launch_count() - l0
    k_ms, k_n = solver.kernel_time_ms(reset=True)
    value = world * units_per_step * args.steps / (ms_total * 1e-3)
    k_ms_ranks = gather_floats(rdist, torch, k_ms, world)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, solver.get_state(), scal.cpu().numpy())

    # ---- parity of THIS run against the oracle (rank 0, 64 seeded members, all the steps done so far) ------------
    parity = oracle_parity(rcm, st, solver, args.warmup + args.steps, nwvl) if rank == 0 and not args.no_parity else None

    # ---- e2e: host buffers in and out through rcm_step_host, copies inside the timed region ------------
    # Per step the caller hands over what changed - T and Tsurf - and reads back fluxes, heating rates and the new
    # temperatures.  The VMR rows are uploaded once (first call): four species are constant and H2O follows the
    # feedback on the device, as in the reference loop.
    nact = solver.nactive
    pin = lambda *shape: torch.empty(*shape, dtype=torch.float64).pin_memory()
    T_in, Ts_in, v_in = pin(ncol, NLAY), pin(ncol), pin(ncol, nact, NLAY)
    Ed, Eu, dE, T_out, Ts_out = pin(ncol, 21), pin(ncol, 21), pin(ncol, NLAY), pin(ncol, NLAY), pin(ncol)
    T_in.copy_(torch.from_numpy(st["Tlayer"]))
    Ts_in.copy_(torch.from_numpy(st["Tsurf"]))
    active = [k for k in range(9) if solver.params.species_mask >> k & 1]
    v_in.copy_(torch.from_numpy(np.ascontiguousarray(st["vmr9"][:, active, :])))
    first = [t.data_ptr() for t in (T_in, Ts_in, v_in, Ed, Eu, dE, T_out, Ts_out)]
    ptrs = list(first)
    ptrs[2] = 0  # NULL: the VMRs stay on the device
    h2d = (T_in.numel() + Ts_in.numel()) * 8
    d2h = (Ed.numel() + Eu.numel() + dE.numel() + T_out.numel() + Ts_out.numel()) * 8
    solver.step_host_ptrs(*first)
    for _ in range(max(1, args.warmup // 2)):
        solver.step_host_ptrs(*ptrs)
    if world > 1:
        rdist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        solver.step_host_ptrs(*ptrs)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    e2e_ranks = gather_floats(rdist, torch, e2e_s, world)
    e2e_s = max(e2e_ranks)
    e2e_value = world * units_per_step * args.steps / e2e_s
    olr_check = float(Eu[0, 0])
    graph_stats = dict(zip(("captures", "replays"), solver.host_graph_stats()))

    # ---- strong scaling (BASELINE configs[3] as north_star states it): ONE 65,536-column ensemble over the ranks ----
    strong = None
    total = args.strong_total
    if not args.no_strong:
        import hashlib
        lo, hi = rdist.shard_range(total, rank, world)
        sl = slice(lo, hi)
        # rank 0's weak ensemble is the global one (seed 12345); other ranks rebuild it to cut their shard
        g = st if rank == 0 and total == ncol else build_ensemble(rcm, total, 12345)
        solver.set_columns(g["plevel"], g["Tlayer"][sl], g["Tsurf"][sl], g["vmr9"][sl], g["rel_hum"][sl])
        exs = rdist.StepScalarExchange(torch.device("cuda", local_rank), ring=args.ring, solver=solver)

        def s_step():
            exs.submit(rdist.device_view(solver.advance_async(1), 4))

        for _ in range(args.warmup):
            s_step()
        exs.latest()
        solver.kernel_time_ms(reset=True)
        ms_s, _ = timed_loop(torch, rdist, stream, world, args.steps, s_step, exs.latest)
        ks_ms, _ = solver.kernel_time_ms(reset=True)
        chk = hashlib.sha256(solver.get_state(("Tlayer",))["Tlayer"][:64].tobytes()).hexdigest()[:16] if rank == 0 else None
        # the RCE driver's form: blocks of fused steps, one allreduce per block
        blk = max(args.steps, 10)

        def s_block():
            rdist.allreduce_step_scalars(rdist.device_view(solver.advance_async(blk), 4 * blk))

        s_block()
        ms_b, _ = timed_loop(torch, rdist, stream, world, 2, s_block, lambda: None)
        ks_ranks = gather_floats(rdist, torch, ks_ms, world)
        strong = {"columns_total": total, "columns_per_gpu": hi - lo, "value": total * nwvl * NLAY * args.steps / (ms_s * 1e-3),
                  "unit": UNIT, "ms_per_step": ms_s / args.steps, "scaling": "strong",
                  "kernel_ms_per_rank": {"min": min(ks_ranks), "max": max(ks_ranks)},
                  "driver_blocks": {"steps_per_block": blk, "ms_per_step": ms_b / (2 * blk),
                                    "value": total * nwvl * NLAY * 2 * blk / (ms_b * 1e-3)},
                  # Tlayer of the ensemble's first 64 columns after check_steps iterations: the same bytes for every N
                  # (per-column results do not depend on the sharding - split path)
                  "check_T_sha_first64": chk, "check_steps": args.warmup + args.steps + 3 * blk}
    lbl = None
    if not args.no_lbl:
        solver.close()
        lbl = lbl_block(args, rank, world, local_rank, torch, rcm, rdist, stream, min(args.steps, args.lbl_steps))

    if rank != 0:
        return 0
    # ---- roofline of the dominant kernel: FP64 pipe -------------------------------------------------------
    cap = load_capture()
    exec_per_unit = cap["step"]["exec_fp64_per_unit"]
    dram_per_colstep = cap["step"]["dram_bytes_per_column_step"]
    r_fma, r_exp, r_div = peaks["dfma"], peaks["exp"], peaks["div"]
    alg_per_unit = ALG_FMA + ALG_EXP * (r_fma / r_exp) + ALG_DIV * (r_fma / r_div)
    k_units_per_s = units_per_step / (k_ms * 1e-3) if k_ms > 0 else 0.0
    achieved = k_units_per_s * exec_per_unit / 1e9  # FP64-pipe instructions really executed per second
    roofline = {"bound": "fp64", "achieved": achieved, "peak": r_fma, "unit": "G FP64-pipe instr/s",
                "frac": achieved / r_fma if r_fma else None,
                "traffic": dram_per_colstep * ncol if dram_per_colstep else None,
                "kernel": cap["step"]["kernel"], "kernel_ms": k_ms, "kernel_launches": k_n,
                "kernel_ms_per_rank": {"min": min(k_ms_ranks), "max": max(k_ms_ranks)},
                "algorithmic_fp64_instr_per_unit": alg_per_unit,
                "executed_fp64_instr_per_unit": exec_per_unit,
                "reference_tree_frac": (k_units_per_s * alg_per_unit / 1e9 / r_fma) if r_fma else None,
                "capture": cap["step"].get("capture"), "capture_sha": cap.get("sources_sha256"), "stale": cap["stale"],
                "peak_source": "measured in this run: DFMA, exp(), divide microbenchmarks "
                               f"({r_fma:.0f}/{r_exp:.0f}/{r_div:.0f} Gop/s); MEASURED_PEAKS.json has no FP64 figure",
                "hbm_GBps": (dram_per_colstep * ncol / (k_ms * 1e-3) / 1e9) if k_ms > 0 else None}
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        v, cores, kind, walls = cpu_throughput(nwvl, args.cpu_cols, args.cpu_steps)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
               "sample": f"{args.cpu_cols} columns x {args.cpu_steps} steps per core, one process per core, "
                         f"table cached in RAM ({walls[0]:.1f} s wall)"}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": workload_config(ncol, nwvl, world),
            "roofline": roofline, "cpu_baseline": cpu, "parity": parity,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": 1e3 * e2e_s / args.steps,
                    "ms_per_step_per_rank": {"min": 1e3 * min(e2e_ranks) / args.steps, "max": 1e3 * max(e2e_ranks) / args.steps},
                    "api": "rcm_step_host (pinned host buffers; T and Tsurf up, E_down/E_up/dE/T/Tsurf down every step; the "
                           "VMR rows went up once - H2O follows the feedback on the device; columns travel in 10 chunks (eight, the first and the last split again) through "
                           "3 streams, copies overlap the step; from the second call on the pipeline is one CUDA graph launch)",
                    "host_graph": graph_stats, "numa": numa, "check_olr_col0": olr_check},
            "strong": strong, "lbl": lbl,
            "gpu_launches": launches, "clocks": clocks, "fp64_peaks_Gops": peaks,
            "ensemble": {"toa_net_mean_Wm2": toa_mean, "collective": f"1 async all_gather of 4 doubles per step, ring of {args.ring}"
                         if world > 1 else "none (1 rank)"}}
    print(json.dumps(line), flush=True)
    if parity is not None and not parity["ok"]:
        print(f"bench.py: PARITY FAILURE against the oracle: {parity}", file=sys.stderr)
        return 3
    return 0


# ------------------------------------------------------------------------------------------------------
# Second workload: BASELINE configs[4], a 4,096-column line-by-line ensemble with 2xCO2 forcing, columns sharded
# over the ranks (total fixed: strong scaling).  The reference's LBL tables are not distributed: synthetic tables in
# its format (rcm_make_lbl_tables), --lbl-nwvl wavelengths.  Appended to the default line as "lbl"; --workload lbl
# prints it as a line of its own.
# ------------------------------------------------------------------------------------------------------
def build_lbl_case(rcm, ncol, nwvl, seed):
    atm = rcm.read_atm(os.path.join(GOLDEN, "column21.lbl.atm"))
    full = rcm.read_atm(os.path.join(GOLDEN, "column21.atm"))
    pl = atm[:, 1].copy()
    Tlev, vlev = rcm.make_ensemble(ncol, seed, pl, atm[:, 2].copy(), full[:, 4:9].T.copy())
    st = rcm.init_columns(pl, Tlev, vlev, 1.0)  # 2xCO2 enters through co2_factor of the LBL tables
    base = rcm.init_columns(pl, atm[None, :, 2].copy(), full[None, :, 4:9].transpose(0, 2, 1).copy(), 1.0)
    h2o_ref, o3_ref = base["vmr9"][0, 0].copy(), base["vmr9"][0, 2].copy()
    wvl, tau5 = rcm.make_lbl_tables(nwvl, 777, pl, h2o_ref, o3_ref)
    return dict(pl=pl, st=st, Tsurf=Tlev[:, 20].copy(), wvl=wvl, tau5=tau5, h2o_ref=h2o_ref, o3_ref=o3_ref)


def _lbl_cpu_worker(args):
    seed, ncol, nwvl = args
    import our_first_climate_model_b200 as rcm
    from oracle import port as P
    c = build_lbl_case(rcm, ncol, nwvl, seed)
    solar = rcm.solar_setup()["solar_irr"]
    t0 = time.perf_counter()
    P.lbl_advance(c["wvl"], c["tau5"], c["pl"], c["st"]["rel_hum"], c["h2o_ref"], c["st"]["vmr9"][:, 2] / c["o3_ref"], 2.0,
                  solar, c["st"]["Tlayer"], c["Tsurf"], c["st"]["vmr9"][:, 0], 1)
    return time.perf_counter() - t0


def lbl_block(args, rank, world, local_rank, torch, rcm, rdist, stream, steps):
    total, nwvl = args.lbl_ncol, args.lbl_nwvl
    lo, hi = rdist.shard_range(total, rank, world)
    ncol = hi - lo
    c = build_lbl_case(rcm, total, nwvl, 4242)
    sl = slice(lo, hi)
    solver = rcm.Solver(local_rank)
    solver.set_stream(stream.cuda_stream)
    solver.set_lbl_tables(c["wvl"], c["tau5"], c["h2o_ref"], c["o3_ref"], 2.0)
    solver.set_columns(c["pl"], c["st"]["Tlayer"][sl], c["Tsurf"][sl], c["st"]["vmr9"][sl], c["st"]["rel_hum"][sl])
    exch = rdist.StepScalarExchange(torch.device("cuda", local_rank), ring=args.ring, solver=solver)
    peak = solver.fp64_microbench(0) if rank == 0 else 0.0

    def one_step():
        exch.submit(rdist.device_view(solver.advance_async(1), 4))

    for _ in range(args.warmup):
        one_step()
    exch.latest()
    torch.cuda.synchronize()
    l0 = solver.launch_count()
    solver.kernel_time_ms(reset=True)
    ms_total, scal = timed_loop(torch, rdist, stream, world, steps, one_step, exch.latest)
    launches = solver.launch_count() - l0
    k_ms, k_n = solver.kernel_time_ms(reset=True)
    k_ranks = gather_floats(rdist, torch, k_ms, world)
    units_per_step = total * nwvl * NLAY
    value = units_per_step * steps / (ms_total * 1e-3)
    # parity of this run: 4 seeded members through the oracle's LBL composition (rank 0)
    parity = None
    if rank == 0 and not args.no_parity:
        from oracle import port as P
        idx = np.sort(np.random.default_rng(7).choice(ncol, size=min(4, ncol), replace=False))
        out = solver.get_state()
        g = lambda a: a[sl][idx]
        ref = P.lbl_advance(c["wvl"], c["tau5"], c["pl"], g(c["st"]["rel_hum"]), c["h2o_ref"], g(c["st"]["vmr9"])[:, 2] / c["o3_ref"],
                            2.0, rcm.solar_setup()["solar_irr"], g(c["st"]["Tlayer"]), g(c["Tsurf"]), g(c["st"]["vmr9"])[:, 0],
                            args.warmup + steps)
        scale = np.abs(ref["E_up"]).max(axis=1, keepdims=True)
        rel = max(float(np.max(np.abs(out[k][idx] - ref[k]) / scale)) for k in ("E_up", "E_down"))
        dT = float(np.max(np.abs(out["Tlayer"][idx] - ref["Tlayer"])))
        parity = {"oracle": "port (builder's LBL composition; components pinned by the reference)", "n_checked": int(idx.size),
                  "steps": args.warmup + steps, "max_rel_flux": rel, "max_abs_dT": dT, "tolerance": 1e-9,
                  "ok": bool(rel < 1e-9 and dT < 1e-6)}
    # e2e: host buffers through rcm_step_host (T, Tsurf up; fluxes, heating rates, T down; VMRs went up once)
    nact = solver.nactive
    pin = lambda *shape: torch.empty(*shape, dtype=torch.float64).pin_memory()
    T_in, Ts_in, v_in = pin(ncol, NLAY), pin(ncol), pin(ncol, nact, NLAY)
    Ed, Eu, dE, T_out, Ts_out = pin(ncol, 21), pin(ncol, 21), pin(ncol, NLAY), pin(ncol, NLAY), pin(ncol)
    T_in.copy_(torch.from_numpy(c["st"]["Tlayer"][sl]))
    Ts_in.copy_(torch.from_numpy(c["Tsurf"][sl]))
    active = [k for k in range(9) if solver.params.species_mask >> k & 1]
    v_in.copy_(torch.from_numpy(np.ascontiguousarray(c["st"]["vmr9"][sl][:, active, :])))
    first = [t.data_ptr() for t in (T_in, Ts_in, v_in, Ed, Eu, dE, T_out, Ts_out)]
    ptrs = list(first)
    ptrs[2] = 0
    h2d = (T_in.numel() + Ts_in.numel()) * 8
    d2h = (Ed.numel() + Eu.numel() + dE.numel() + T_out.numel() + Ts_out.numel()) * 8
    solver.step_host_ptrs(*first)
    if world > 1:
        rdist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        solver.step_host_ptrs(*ptrs)
    torch.cuda.synchronize()
    e2e_s = max(gather_floats(rdist, torch, time.perf_counter() - t0, world))
    solver.close()
    if rank != 0:
        return None
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        import multiprocessing as mp
        cores = len(os.sched_getaffinity(0))
        cols = args.lbl_cpu_cols
        with mp.get_context("fork").Pool(cores) as pool:
            pool.map(_lbl_cpu_worker, [(1, 1, 200)] * cores)
            t0 = time.perf_counter()
            pool.map(_lbl_cpu_worker, [(100 + i, cols, nwvl) for i in range(cores)])
            wall = time.perf_counter() - t0
        cpu = {"value": cores * cols * nwvl * NLAY / wall, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{cols} columns x 1 step per core of the oracle's LBL composition (the reference has no LBL driver), "
                         f"{wall:.1f} s wall"}
    cap = load_capture()
    exec_per_unit = cap["lbl"]["exec_fp64_per_unit"]
    k_units = (ncol * nwvl * NLAY) / (k_ms * 1e-3) if k_ms > 0 else 0.0
    achieved = k_units * exec_per_unit / 1e9
    return {"metric": "column*wavelength*layer flux updates/s (line-by-line RCE step)", "value": value, "unit": UNIT,
            "n_gpus": world, "steps": steps, "warmup": args.warmup, "ms_per_step": ms_total / steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{total}-column line-by-line ensemble, 2xCO2, {nwvl} synthetic wavelengths "
                                   "(BASELINE configs[4]); columns sharded over the ranks", "columns_total": total,
                       "nwvl": nwvl, "nlayer": NLAY, "nangle": 30, "parallelism": f"{world} GPU(s)",
                       "l2": "tables (5 x nwvl x 20 doubles = 16 MB at 20,000 wavelengths) are re-read by every tile: L2-resident"},
            "roofline": {"bound": "fp64", "achieved": achieved, "peak": peak, "unit": "G FP64-pipe instr/s",
                         "frac": achieved / peak if peak else None, "traffic": None, "kernel": cap["lbl"]["kernel"],
                         "kernel_ms": k_ms, "kernel_launches": k_n, "kernel_ms_per_rank": {"min": min(k_ranks), "max": max(k_ranks)},
                         "executed_fp64_instr_per_unit": exec_per_unit, "capture": cap["lbl"].get("capture"),
                         "capture_sha": cap.get("sources_sha256"), "stale": cap["stale"]},
            "cpu_baseline": cpu, "parity": parity,
            "e2e": {"value": units_per_step * steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": 1e3 * e2e_s / steps, "api": "rcm_step_host"},
            "gpu_launches": launches,
            "ensemble": {"toa_net_mean_Wm2": float(scal[0]) / total}}


def run_b200_lbl(args, rank, world, local_rank):
    import torch
    import our_first_climate_model_b200 as rcm
    from our_first_climate_model_b200 import distributed as rdist
    if not torch.cuda.is_available() or rcm.device_count() == 0:
        raise SystemExit("bench.py: no CUDA device - the solver has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        rdist.init("nccl")
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    sampler = ClockSampler(world)
    if rank == 0:
        sampler.start()
    line = lbl_block(args, rank, world, local_rank, torch, rcm, rdist, stream, args.steps)
    if rank != 0:
        return 0
    line["clocks"] = sampler.stop()  # the whole block (no window): warm-up, timed steps, e2e leg
    print(json.dumps(line), flush=True)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ncol", type=int, default=65536, help="columns per GPU")
    ap.add_argument("--nwvl", type=int, default=100, choices=[10, 20, 100])
    ap.add_argument("--cpu-cols", type=int, default=None, help="columns per core in a CPU sample")
    ap.add_argument("--cpu-steps", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="repwvl", choices=["repwvl", "lbl"],
                    help="repwvl = the headline metric (BASELINE configs[3]); lbl = configs[4], optional")
    ap.add_argument("--lbl-ncol", type=int, default=4096, help="columns of the LBL ensemble (all ranks together)")
    ap.add_argument("--lbl-nwvl", type=int, default=20000)
    ap.add_argument("--lbl-steps", type=int, default=10, help="timed LBL steps of the block appended to the default line")
    ap.add_argument("--lbl-cpu-cols", type=int, default=8)
    ap.add_argument("--no-lbl", action="store_true", help="skip the LBL block of the default line")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check of the timed run")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling block (one ensemble over the ranks)")
    ap.add_argument("--strong-total", type=int, default=65536, help="columns of the strong-scaling ensemble (N > 1)")
    ap.add_argument("--ring", type=int, default=32, help="slots of the asynchronous scalar exchange")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write rank 0's state and last-step scalars as DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.workload != "repwvl"):
        ap.error("--dump-outputs writes the outputs of the default workload (--impl b200 --workload repwvl)")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    rank, world, local_rank = _env_int("RANK", 0), _env_int("WORLD_SIZE", 1), _env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        if args.cpu_cols is None:
            args.cpu_cols = 256
        return run_reference(args, rank, world)
    if args.cpu_cols is None:
        args.cpu_cols = 512
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29531", os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    if args.workload == "lbl":
        return run_b200_lbl(args, rank, world, local_rank)
    return run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    sys.exit(main())
