#!/usr/bin/env python
"""bench.py -- Wilson-Dslash GFLOPS / HBM GB/s on a 32^4 local volume (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            our arm (libquda_b200.so on B200)
  python bench.py ... --dump-outputs DIR                   also save what the last of the K timed steps computed (DIR/out.npy)
  python bench.py --impl reference ...                     the reference's CPU dslash (oracle/_ref) on host cores
  python bench.py --sweep                                  (dev) launch-geometry sweep, writes gpurun_out/sweep.json

A "step" is ONE application of the single-parity Wilson Dslash (out_p = D in_{1-p}) to a 32^4 local lattice,
fp32 storage/compute, 12-parameter gauge reconstruction (BASELINE.json configs[1]).  `value` = GFLOP/s with the
reference's flop model (1320 flop per output site, include/dslash.h:475-528), whole job over all ranks, fields
resident in HBM.  `e2e` = same metric through the C ABI with HOST (pinned) spinor buffers: H2D of the input
spinor, Dslash, D2H of the result every step; the gauge field stays resident, as it does after loadGaugeQuda.
Per-step working set = 302 MB (> 126 MB L2): inputs larger than L2, no explicit flush.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# The CPU arm (reference Dslash on the host cores) is an OpenMP code: pin its threads to cores, one per place, before any
# OpenMP runtime is loaded -- unpinned it swung 5x between otherwise identical boxes (VERDICT r1).
# ONLY in a process that runs the CPU arm: under torchrun (N > 1) every rank is its own process with OMP_NUM_THREADS=1, and
# a bound single thread lands on place 0 -- all ranks' host threads would share ONE core and the launch rate collapses
# (measured: 2-GPU steps went from 56 to 110 us with the binding on; profiles/r02_scale2_pinned_ranks.json).
_CPU_ARM = ("--impl" in sys.argv and "reference" in sys.argv) or int(os.environ.get("WORLD_SIZE", "1")) == 1
if _CPU_ARM and int(os.environ.get("RANK", "0")) == 0:
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "threads")

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

PREC_BYTES = {"double": 8, "single": 4, "half": 2}
DTYPE = {"double": "f64", "single": "f32", "half": "i16-blockfloat"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--prec", default="single", choices=list(PREC_BYTES))
    ap.add_argument("--recon", type=int, default=12, choices=[18, 12, 8])
    ap.add_argument("--dim", type=int, nargs=4, default=[32, 32, 32, 32])
    ap.add_argument("--tile", type=int, nargs=4, default=None)
    ap.add_argument("--op", default="wilson", choices=["wilson", "clover_pc", "cg"],
                    help="clover_pc: ApplyWilsonCloverPreconditioned (BASELINE config 3), compressed clover, dynamic inverse")
    ap.add_argument("--global-dim", type=int, nargs=4, default=[48, 48, 48, 96], help="--op cg: global lattice (config 5)")
    ap.add_argument("--tol", type=float, default=1e-10, help="--op cg: relative residual target")
    ap.add_argument("--kappa", type=float, default=0.12195)
    ap.add_argument("--nsrc", type=int, default=1, help="sources per call (multi-RHS batch sharing the gauge field); at N > 1 with one batched halo exchange per call")
    ap.add_argument("--no-mrhs", action="store_true", help="skip the extra multi-RHS measurement of the default line")
    ap.add_argument("--sweep", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the fp64 / half / clover-pc sub-lines of the default run")
    ap.add_argument("--breakdown", action="store_true", help="(N>1) also time pack / interior / exterior separately")
    ap.add_argument("--grid", type=int, nargs=4, default=None,
                    help="(N>1) process grid (x y z t), product = N; default splits t, then z, then y.  BASELINE config 4's "
                         "2x1x1x1 is --grid 2 1 1 1 (the strided x face)")
    ap.add_argument("--no-halo-check", action="store_true", help="(N>1) skip the partitioned-vs-global-oracle parity check")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the output spinor(s) of the last one to DIR/<name>.npy (see dump_outputs)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "b200" or a.op == "cg" or a.sweep):
        ap.error("--dump-outputs applies to the timed Dslash of --impl b200 (--op wilson or clover_pc)")
    return a


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.rows, self.stop_flag, self.index = [], False, index
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop_flag:
            try:
                o = subprocess.check_output(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                             "-i", str(self.index)], timeout=5).decode().strip()
                self.rows.append([c.strip() for c in o.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop_flag = True
        self.t.join(timeout=6)

    def summary(self):
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(float(self.rows[0][1])), "reasons": reasons,
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ reference arm
def cpu_reference(X, prec, budget_s=20.0, min_reps=2):
    """Time the reference's own host Dslash (oracle/_ref, kind 'reference'; our restatement 'port' otherwise)
    on all host cores.  Returns (gflops, info dict)."""
    cores = os.cpu_count() or 1
    # torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm is meant to use all host cores: set the variable
    # before the OpenMP runtime is loaded and, in case it already is, tell the runtime directly
    os.environ["OMP_NUM_THREADS"] = str(cores)
    import ctypes
    import numpy as np
    import oracle
    try:
        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(cores)
    except OSError:
        pass
    hp = 8 if prec == "double" else 4
    g = oracle.random_gauge(X, hp, seed=137)
    s = oracle.random_spinor(X, hp, seed=137)
    Vh = oracle.volume(X) // 2
    if oracle.have_ref():
        R = oracle.Reference(X)
        fn, kind = (lambda: R.wil_dslash(g, s, 0, 0)), "reference"
    else:
        fn, kind = (lambda: oracle.wil_dslash(g, s, X, 0, 0)), "port"
    fn()
    t0 = time.perf_counter()
    reps = 0
    while reps < min_reps or (time.perf_counter() - t0 < budget_s and reps < 1000):
        fn()
        reps += 1
    dt = (time.perf_counter() - t0) / reps
    gf = 1320.0 * Vh / dt * 1e-9
    return gf, {"value": gf, "unit": "GFLOP/s", "cores": cores, "kind": kind, "ms_per_call": dt * 1e3,
                "pinning": {"OMP_PROC_BIND": os.environ.get("OMP_PROC_BIND"), "OMP_PLACES": os.environ.get("OMP_PLACES"),
                            "numa": numa_layout()},
                "sample": f"{reps} applications of the single-parity Wilson Dslash on {'x'.join(map(str, X))} "
                          f"({'fp64' if hp == 8 else 'fp32'} host fields), OpenMP over {cores} threads"}


def numa_layout():
    """sockets / NUMA nodes / threads per core of the host (lscpu), for the CPU arm's record"""
    try:
        o = subprocess.check_output(["lscpu"], timeout=5).decode()
        keep = {}
        for line in o.splitlines():
            k, _, v = line.partition(":")
            if k.strip() in ("Socket(s)", "NUMA node(s)", "Thread(s) per core", "Core(s) per socket", "Model name"):
                keep[k.strip()] = v.strip()
        return keep
    except Exception:  # noqa: BLE001
        return None


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    X = a.dim
    per = []
    info = None
    for i in range(a.warmup + a.steps):
        gf, info = cpu_reference(X, a.prec, budget_s=max(1.0, 60.0 / max(1, a.warmup + a.steps)), min_reps=1)
        if i >= a.warmup:
            per.append(info["ms_per_call"])
    ms = sum(per) / len(per)
    Vh = X[0] * X[1] * X[2] * X[3] // 2
    val = 1320.0 * Vh / (ms * 1e-3) * 1e-9
    info["value"] = val
    out = {"impl": "reference", "metric": "wilson_dslash_gflops", "value": val, "unit": "GFLOP/s", "n_gpus": a.gpus,
           "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": DTYPE[a.prec], "data": "synthetic",
           "config": workload(a), "cpu_baseline": info,
           "e2e": {"value": val, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def workload(a):
    return {"workload": f"Wilson Dslash (single parity, no xpay), {'x'.join(map(str, a.dim))} local lattice, "
                        f"{a.prec} recon-{a.recon}, interior kernel" + (" + halo" if a.gpus > 1 else ""),
            "l2": "per-step working set 8G+2S per site > 126 MB L2 at 32^4, and the steps rotate through 4 (input, output) "
                  "spinor pairs so that outputs are written back to HBM; no explicit flush",
            "grid": list(a.grid) if a.grid else process_grid(a.gpus)}


def halo_parity_check(grid, dist, prec, recon, Xl=(16, 16, 16, 16)):
    """N > 1: before anything is timed, apply the partitioned operator (the very call the timed loop makes: pack, NVLink
    remote writes, interior, boundary -- one fused launch per Dslash) to seeded oracle-order fields and compare every
    rank's block with the oracle on the GLOBAL lattice (the reference's dslash_ctest criterion, tests/dslash_ctest.cpp:
    107-122).  Returns (max deviation over ranks, tolerance).  The oracle is the checker here, never what is measured."""
    import numpy as np
    import torch
    import oracle
    from common import CudaMem
    from quda_b200 import comm, dirac as DR, dslash as D, fields as F
    Xl = [int(v) for v in Xl]
    Xg = [Xl[d] * grid.dims[d] for d in range(4)]
    hp = 8 if prec == 8 else 4
    gauge = oracle.random_gauge(Xg, hp, seed=137)  # the same global fields on every rank (same seeds)
    parity, kappa = 1, 0.12195
    s = oracle.random_spinor(Xg, hp, seed=5)
    xs = oracle.random_spinor(Xg, hp, seed=6)
    gl = comm.local_slice(gauge, Xg, Xl, grid.coords, "gauge")
    ghost_from = []
    for d in range(4):
        c = list(grid.coords)
        c[d] = (c[d] - 1) % grid.dims[d]
        ghost_from.append(comm.local_slice(gauge, Xg, Xl, c, "gauge") if grid.dims[d] > 1 else None)
    gbuf, gmeta = F.gauge_to_native(gl, Xl, prec, recon, ghost_from=ghost_from)
    U = D.GaugeField(CudaMem.put(gbuf), Xl, prec, recon, gmeta, t_boundary=-1, first_time_slice=grid.first_time_slice(),
                     last_time_slice=grid.last_time_slice())
    sl = comm.local_slice(s, Xg, Xl, grid.coords, ("spinor1", 1 - parity))
    xl = comm.local_slice(xs, Xg, Xl, grid.coords, ("spinor1", parity))
    din = D.ColorSpinorField(CudaMem.put(F.spinor_to_native(sl, prec)), Xl, prec)
    dx = D.ColorSpinorField(CudaMem.put(F.spinor_to_native(xl, prec)), Xl, prec)
    out = D.ColorSpinorField(CudaMem.empty(F.spinor_bytes(Xl, prec)), Xl, prec)
    ex = comm.HaloExchange(grid, Xl, prec, mode="p2p", dist=dist)
    cs = ex.comm_struct()
    op = DR.Dirac("wilson", U, 0.0, comm=cs, stream=torch.cuda.current_stream().cuda_stream)
    dev = 0.0
    for dagger in (0, 1):
        for _ in range(3):  # repeated applications exercise the double-buffered ghost zones
            op.DslashXpay(out, din, parity, dx, -kappa, dagger=bool(dagger))
        torch.cuda.synchronize()
        ref = xs.astype(np.float64) - kappa * oracle.wil_dslash(gauge, s, Xg, parity, dagger).astype(np.float64)
        got = F.spinor_from_native(CudaMem.get(out.buf), F.volume_cb(Xl), prec)
        want = comm.local_slice(ref, Xg, Xl, grid.coords, ("spinor1", parity))
        dev = max(dev, float(oracle.compare_spinor(want, got)[1]))
    import ctypes as C
    from quda_b200 import lib as L_
    L_.check(L_.load().b200_comm_check(C.byref(cs), None))
    t = torch.tensor([dev], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    del op
    return float(t.item()), float(oracle.tolerance(PREC_NAME_BY_BYTES[prec], recon))


PREC_NAME_BY_BYTES = {8: "double", 4: "single", 2: "half"}


def process_grid(n):
    # split t first, then z, then y (x keeps the contiguous rows local): 2 -> (1,1,1,2) ... 8 -> (1,2,2,2)
    g = [1, 1, 1, 1]
    d = 3
    while n > 1:
        g[d] *= 2
        n //= 2
        d = d - 1 if d > 0 else 3
    return g


# ------------------------------------------------------------------------------------------------ our arm
def run_b200(a):
    import numpy as np
    import torch
    import oracle
    from common import CudaMem, Problem
    from quda_b200 import dslash as D
    from quda_b200 import fields as F
    from quda_b200 import lib as L

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        if not os.environ.get("NCCL_DEBUG"):
            os.environ["NCCL_DEBUG"] = "WARN"  # keep stdout to the one JSON line (an empty value makes NCCL print its banner)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = L.load()
    X = a.dim
    prec = PREC_BYTES[a.prec]
    Vh = F.volume_cb(X)

    # synthetic fields: random SU(3) links (unitary, so all recon modes are exact) and uniform spinors, built
    # directly in native order on the device to keep set-up time bounded
    torch.manual_seed(1234 + rank)
    grid = ex = None
    if world > 1:
        from quda_b200 import comm
        dims = list(a.grid) if a.grid else comm.ProcessGrid.default_dims(world)
        assert dims[0] * dims[1] * dims[2] * dims[3] == world, f"--grid {dims} does not have {world} ranks"
        grid = comm.ProcessGrid(dims, rank)
    P = make_device_problem(X, prec, a.recon, grid)
    src, dst = P["in"], P["out"]
    stream = torch.cuda.current_stream().cuda_stream
    halo_mode = None
    if world > 1:
        # fused pack + NVLink peer-write halo; NCCL send/recv only if CUDA IPC is unavailable on this box
        try:
            ex = comm.HaloExchange(grid, X, prec, mode="p2p", dist=dist)
            halo_mode = "p2p-remote-write"
        except Exception as e:  # noqa: BLE001
            if rank == 0:
                print(f"[bench] CUDA-IPC halo unavailable ({e}); falling back to NCCL send/recv", file=sys.stderr)
            ex = comm.HaloExchange(grid, X, prec, mode="nccl", dist=dist)
            halo_mode = "nccl-sendrecv"

    halo_parity = None
    if ex is not None and halo_mode.startswith("p2p") and not a.no_halo_check:
        dev, tol = halo_parity_check(grid, dist, prec, a.recon)
        halo_parity = {"parity_dev": dev, "tolerance": tol, "local_lattice": "16x16x16x16", "reference": "CPU oracle on the global lattice",
                       "ok": bool(dev <= tol)}
        if dev > tol:
            if rank == 0:
                print(json.dumps({"error": "partitioned Dslash differs from the global oracle", "halo": halo_parity}))
            dist.destroy_process_group()
            sys.exit(3)

    dirac = None
    if ex is not None and halo_mode.startswith("p2p"):
        # drive the partitioned Dslash through the C++ operator layer (one native call per step: pack on the side
        # stream, interior tiles, boundary tiles) -- the Python-level schedule costs more host time than the GPU needs
        from quda_b200 import dirac as DR
        comm_cs = ex.comm_struct()
        dirac = DR.Dirac("wilson", P["U"], 0.0, comm=comm_cs, stream=stream)

    clover_bytes = 0
    if a.op == "clover_pc":
        assert world == 1, "--op clover_pc is a single-GPU measurement"
        P["A"] = make_device_clover(X, prec)
        clover_bytes = 56 * prec

    # rotate through NROT (input, output) pairs so that no step finds its output (or input) lines still dirty / resident
    # in the 126 MB L2 from the previous step: every byte of B_min really crosses HBM (VERDICT r1: traffic 266 < 302 MB)
    NROT = 4
    pairs = [(src, dst)] + [(new_spinor(P, seed=501 + i), new_spinor(P, seed=None)) for i in range(NROT - 1)]
    rot = [0]

    nsrc = max(1, a.nsrc)
    ex_batch = None
    if nsrc > 1:
        srcs = [src] + [new_spinor(P, seed=77 + i) for i in range(nsrc - 1)]
        dsts = [dst] + [new_spinor(P, seed=None) for i in range(nsrc - 1)]
        if world > 1:
            # a multi-RHS batch on the partitioned lattice: ONE batched exchange per step (one pack launch and one arrival
            # signal per face for all sources, b200_pack_ghost_multi), batched interior tiles, per-source boundary tiles
            assert a.op == "wilson" and halo_mode.startswith("p2p"), "--nsrc at N > 1: Wilson over the NVLink peer-write halo"
            ex_batch = comm.HaloExchange(grid, X, prec, mode="p2p", dist=dist, n_src=nsrc)

    def step(tile=None):
        src, dst = pairs[rot[0] % NROT]
        rot[0] += 1
        if ex_batch is not None:
            comm.apply_wilson_distributed(ex_batch, dsts, srcs, P["U"], 0.0, None, 0, 0, stream=stream, tile=tile or a.tile)
        elif nsrc > 1:
            fn = D.ApplyWilsonCloverPreconditioned if a.op == "clover_pc" else D.ApplyWilson
            extra = (P["A"],) if a.op == "clover_pc" else ()
            fn(dsts, srcs, P["U"], *extra, 0.0, None, 0, 0, tile=tile or a.tile, stream=stream)
        elif a.op == "clover_pc":
            D.ApplyWilsonCloverPreconditioned(dst, src, P["U"], P["A"], 0.0, None, 0, 0, tile=tile or a.tile, stream=stream)
        elif ex is None:
            D.ApplyWilson(dst, src, P["U"], 0.0, None, 0, 0, tile=tile or a.tile, stream=stream)
        elif dirac is not None:
            dirac.Dslash(dst, src, 0)
        else:
            comm.apply_wilson_distributed(ex, dst, src, P["U"], 0.0, None, 0, 0, stream=stream, tile=tile or a.tile)

    if a.sweep:
        return sweep(a, P, lib)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    es0, es1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as cs:
        for _ in range(max(3, a.warmup)):
            step()
        barrier()
        lib.b200_reset_launch_count()
        ev0.record()
        for _ in range(a.steps):
            step()
        ev1.record()
        barrier()
        launches = lib.b200_launch_count()
        if a.dump_outputs:
            # copied now: the loops below write to the same buffers (the multi-RHS line with another kernel)
            last = [d.buf.clone() for d in (dsts if nsrc > 1 else [pairs[(rot[0] - 1) % NROT][1]])]
        # the timed region above lasts only K x ~55 us, far below nvidia-smi's sampling period: keep the identical
        # kernel running for ~1.5 s more so that the clock / throttle record covers this very workload, and report
        # its (power-capped) steady-state step time next to the K-step figure
        # (the number of extra steps is derived from the timed region, NOT from each rank's wall clock: on a partitioned
        # lattice every rank must make exactly the same number of Dslash calls or its neighbours wait for faces forever)
        ms_probe = ev0.elapsed_time(ev1) / a.steps
        if world > 1:
            tp = torch.tensor([ms_probe], device="cuda")
            dist.all_reduce(tp, op=dist.ReduceOp.MAX)
            ms_probe = float(tp.item())
        n_s = max(100, int(1500.0 / max(ms_probe, 1e-3)) // 100 * 100)
        es0.record()
        for _ in range(n_s // 100):
            for _ in range(100):
                step()
            torch.cuda.synchronize()
        es1.record()
        barrier()
    sustained_ms = es0.elapsed_time(es1) / max(1, n_s)
    ms_total = ev0.elapsed_time(ev1)
    if world > 1:
        t = torch.tensor([ms_total], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms = ms_total / a.steps
    flops = D.flops_per_site(L.OP_CLOVER_PC if a.op == "clover_pc" else L.OP_WILSON) * Vh * world * nsrc
    gflops = flops / (ms * 1e-3) * 1e-9
    bmin = D.min_bytes_per_site(prec, a.recon, clover_bytes=clover_bytes)
    if nsrc > 1:  # compulsory traffic of one call: the link (and clover) stream once, the spinors once per source
        S1 = 24 * prec + (4 if prec == 2 else 0)
        bmin = (8 * a.recon * prec + clover_bytes) + nsrc * 2 * S1
    S = 24 * prec + (4 if prec == 2 else 0)
    bquda = 8 * a.recon * prec + 8 * S
    peak, peak_src = measured_peaks()
    ach = bmin * Vh / (ms * 1e-3) * 1e-9  # per GPU: per-rank bytes / per-step time
    out = {"metric": "wilson_dslash_gflops", "value": gflops, "unit": "GFLOP/s", "n_gpus": world, "steps": a.steps,
           "warmup": max(3, a.warmup), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": DTYPE[a.prec], "data": "synthetic", "config": workload(a),
           "hbm_gbs_effective": ach, "gbytes_quda_model": bquda * Vh / (ms * 1e-3) * 1e-9,
           "gpu_launches": int(launches),
           "sustained": {"ms_per_step": sustained_ms, "steps": n_s, "value": flops / (sustained_ms * 1e-3) * 1e-9,
                         "note": "same kernel looped for ~1.5 s after the timed steps (power-capped steady state)"},
           "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                        "traffic": ncu_traffic(a) if world == 1 else None,
                        "traffic_source": "committed ncu capture of this kernel at N=1 (profiles/traffic.json), MB per launch" if world == 1 else None,
                        "peak_source": peak_src,
                        "kernel": "dslash_interior_kernel", "algorithmic_bytes_per_launch": bmin * Vh},
           "clocks": cs.summary()}
    if world > 1:
        # where the step time goes: the same GPU running the unpartitioned kernel on its local lattice (what N = 1 times),
        # and the pack role alone (face gather + NVLink remote writes + flag protocol)
        def timed(fn, n=50):
            for _ in range(5):
                fn()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                fn()
            e1.record()
            barrier()
            t = torch.tensor([e0.elapsed_time(e1) / n * 1e3], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        out["breakdown_us"] = {
            "step": ms * 1e3,
            "unpartitioned_kernel_same_gpus": timed(lambda: D.ApplyWilson(pairs[0][1], pairs[0][0], P["U"], 0.0, None, 0, 0, stream=stream, tile=a.tile)),
            "pack_and_send_alone": timed(lambda: ex.start(pairs[0][0], 1, 0, stream=stream)) if halo_mode.startswith("p2p") else None,
        }
    if world > 1:
        out["halo"] = {"mode": halo_mode, "grid": grid.dims, "bytes_per_step_per_gpu": int(sum(
            2 * ex.face_bytes[d] for d in range(4) if ex.comm_dim[d])), "timed_out": bool(ex.timed_out()) if halo_mode.startswith("p2p") else False}
        out["halo"]["gbs_per_gpu"] = out["halo"]["bytes_per_step_per_gpu"] / (ms * 1e-3) * 1e-9
        out["halo"]["schedule"] = "one fused launch per Dslash: pack CTAs (NVLink remote write + arrival flags) | interior CTAs | boundary CTAs"
        if halo_parity is not None:
            out["halo"].update(halo_parity)
        if ex_batch is not None:
            out["halo"]["schedule"] = "multi-RHS batch: one batched pack (one arrival signal per face for all sources) + boundary tiles per source " \
                                      "on the side stream, batched interior tiles on the main stream"
            out["halo"]["bytes_per_step_per_gpu"] *= nsrc
            out["halo"]["gbs_per_gpu"] *= nsrc
            out["halo"]["timed_out"] = bool(ex_batch.timed_out())

    if nsrc > 1:
        out["config"]["workload"] += f", {nsrc} sources per call (multi-RHS)"
        out["roofline"]["kernel"] = "dslash_mrhs_kernel" if mrhs_flavour(prec, a.recon) == "thread" else "dslash_mrhs_cta_kernel"
        out["roofline"]["traffic"] = None
        out["ms_per_rhs"] = ms / nsrc
    elif world == 1 and a.op == "wilson" and not a.no_mrhs:
        try:
            out["multi_rhs"] = multi_rhs_line(a, P, D, L, stream, prec, Vh, peak)
        except Exception as e:  # noqa: BLE001  -- the single-source line above stands on its own
            out["multi_rhs"] = {"error": str(e)}
    if world == 1 and a.op == "wilson" and nsrc == 1 and not a.no_extra and a.prec == "single" and a.recon == 12:
        # the other precisions / BASELINE config 3 on the same box, so that they are driver-visible numbers too
        out["other_configs"] = []
        for pname, rc, opname in (("double", 18, "wilson"), ("half", 12, "wilson"), ("half", 8, "clover_pc"), ("half", 8, "clover_pc_static")):
            try:
                out["other_configs"].append(sub_line(a, pname, rc, opname, stream, peak))
            except Exception as e:  # noqa: BLE001
                out["other_configs"].append({"prec": pname, "recon": rc, "op": opname, "error": str(e)})
    if a.op != "wilson":
        out["metric"] = "wilson_clover_pc_dslash_gflops"
        out["config"]["workload"] = out["config"]["workload"].replace("Wilson Dslash", "Wilson-clover preconditioned Dslash (A^-1 D, compressed clover, per-site Cholesky)")
    if not a.no_e2e and a.op == "wilson" and (world == 1 or dirac is not None):
        # N > 1: every rank runs the pipeline on its own block through the partitioned operator (halo exchange inside,
        # all ranks' PCIe copies in flight together); the time is the max over ranks
        mk = None
        if world > 1:
            from quda_b200 import dirac as DR2
            mk = lambda st: DR2.Dirac("wilson", P["U"], 0.0, comm=comm_cs, stream=st)  # noqa: E731
        res = e2e(a, P, lib, Vh, prec, world, make_dirac=mk, dist=dist if world > 1 else None)
        if rank == 0:
            out["e2e"] = res
    if rank == 0 and not a.no_cpu_baseline:
        try:
            _, info = cpu_reference(X, a.prec, budget_s=15.0)
            out["cpu_baseline"] = info
        except Exception as e:  # the checker is optional for the measurement itself
            out["cpu_baseline"] = {"value": None, "error": str(e)}
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, "out" if world == 1 else f"out_rank{rank}", last, prec, Vh, DUMP_BYTES // world)
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def sub_line(a, pname, recon, opname, stream, peak, steps=100):
    """one more (precision, reconstruct, operator) on the same lattice: device-timed steps over 3 rotating (in, out) pairs"""
    import torch
    from quda_b200 import dslash as D
    from quda_b200 import fields as F
    from quda_b200 import lib as L
    prec = PREC_BYTES[pname]
    X = a.dim
    Vh = F.volume_cb(X)
    P = make_device_problem(X, prec, recon)
    # clover_pc: compressed clover (56 reals / site) with the per-site Cholesky solve in the kernel (QUDA_DYNAMIC_CLOVER);
    # clover_pc_static: the reference's default build -- A^-1 stored uncompressed (72 reals / site), applied by a 6x6 mat-vec
    A = None
    if opname == "clover_pc":
        A = make_device_clover(X, prec)
    elif opname == "clover_pc_static":
        A = make_device_clover(X, prec, static_inverse=True)
    pairs = [(P["in"], P["out"])] + [(new_spinor(P, seed=601 + i), new_spinor(P, seed=None)) for i in range(2)]

    def step(i):
        src, dst = pairs[i % 3]
        if A is not None:
            D.ApplyWilsonCloverPreconditioned(dst, src, P["U"], A, 0.0, None, 0, 0, stream=stream)
        else:
            D.ApplyWilson(dst, src, P["U"], 0.0, None, 0, 0, stream=stream)

    for i in range(6):
        step(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step(i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    cb = (72 if opname == "clover_pc_static" else 56) * prec if A is not None else 0
    bmin = D.min_bytes_per_site(prec, recon, clover_bytes=cb)
    flops = D.flops_per_site(L.OP_CLOVER_PC if A is not None else L.OP_WILSON) * Vh
    ach = bmin * Vh / (ms * 1e-3) * 1e-9
    return {"prec": pname, "recon": recon, "op": opname, "ms_per_step": ms, "value": flops / (ms * 1e-3) * 1e-9, "unit": "GFLOP/s",
            "algorithmic_bytes_per_launch": bmin * Vh, "hbm_gbs_effective": ach, "frac": ach / peak, "steps": steps}


def mrhs_flavour(prec, recon):
    """launch.h::mrhs_mode: which multi-RHS kernel b200_dslash_apply_multi picks (unless B200_MRHS_MODE overrides)"""
    env = os.environ.get("B200_MRHS_MODE")
    if env in ("thread", "cta"):
        return env
    return "cta" if (prec == 8 or (prec == 4 and recon == 12)) else "thread"


def new_spinor(P, seed=None):
    """another native spinor of P's shape: uniform random (seed given) or zero"""
    import torch
    from quda_b200 import dslash as D
    ref = P["in"]
    if seed is None:
        buf = torch.zeros_like(ref.buf)
    else:
        g = torch.Generator(device="cuda").manual_seed(seed)
        if ref.prec == 2:
            buf = ref.buf.clone()  # block-float layout: reuse the (valid) source image
        else:
            dt = torch.float64 if ref.prec == 8 else torch.float32
            buf = torch.rand(ref.buf.numel() * ref.buf.element_size() // ref.prec, dtype=dt, device="cuda", generator=g).view(torch.uint8)
    return D.ColorSpinorField(buf, ref.X, ref.prec, ref.n_parity)


DUMP_BYTES = 64 << 20


def dump_outputs(path, name, bufs, prec, Vh, budget):
    """--dump-outputs: native single-parity spinor buffers -> path/<name>.npy, shape [len(bufs),] Vh x 4 x 3 x 2 in the
    precision's real type (float64 for double, float32 otherwise), spin and colour as stored (no basis rotation).  Above
    `budget` bytes: a fixed sample of sites (seed 0) from all buffers together, shape n x 4 x 3 x 2, the same at every run."""
    import numpy as np
    from quda_b200 import fields as F
    arr = np.stack([F.spinor_from_native(b.cpu().numpy(), Vh, prec, rotate=False).astype(F.real_dtype(prec)) for b in bufs])
    sites = arr.reshape(-1, 4, 3, 2)
    keep = budget // sites[0].nbytes
    if len(sites) > keep:
        arr = sites[np.sort(np.random.default_rng(0).choice(len(sites), keep, replace=False))]
    elif len(bufs) == 1:
        arr = arr[0]
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, name + ".npy"), arr)


def multi_rhs_line(a, P, D, L, stream, prec, Vh, peak, nsrc=8, steps=50):
    """Batched Dslash (the reference's cvector_ref form, SURVEY 8f row 4): nsrc sources sharing the gauge field in one
    call; per-source time and the fraction of the (amortised) compulsory traffic 8G/batch + 2S per source."""
    import torch
    srcs = [P["in"]] + [new_spinor(P, seed=77 + i) for i in range(nsrc - 1)]
    dsts = [P["out"]] + [new_spinor(P, seed=None) for i in range(nsrc - 1)]
    call = lambda: D.ApplyWilson(dsts, srcs, P["U"], 0.0, None, 0, 0, tile=a.tile, stream=stream)  # noqa: E731
    for _ in range(5):
        call()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        call()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    S1 = 24 * prec + (4 if prec == 2 else 0)
    bytes_call = (8 * a.recon * prec + nsrc * 2 * S1) * Vh  # B_min = 8G/n + 2S per site and source (SURVEY 8f row 4)
    ach = bytes_call / (ms * 1e-3) * 1e-9
    return {"n_src": nsrc, "flavour": mrhs_flavour(prec, a.recon), "ms_per_call": ms, "us_per_rhs": ms / nsrc * 1e3,
            "value": 1320 * Vh * nsrc / (ms * 1e-3) * 1e-9, "unit": "GFLOP/s",
            "algorithmic_bytes_per_call": bytes_call, "hbm_gbs_effective": ach, "frac": ach / peak, "steps": steps}


def random_su3_device(X):
    """random SU(3) links [4][V][3][3][2] fp64 on the device, built like the reference's tests do
    (tests/utils/host_utils.cpp:1022-1098): two random rows, Gram-Schmidt, third row = conjugate cross product"""
    import torch
    V = X[0] * X[1] * X[2] * X[3]
    r1 = torch.randn(4 * V, 3, dtype=torch.complex128, device="cuda")
    r2 = torch.randn(4 * V, 3, dtype=torch.complex128, device="cuda")
    r1 = r1 / torch.linalg.vector_norm(r1, dim=1, keepdim=True)
    r2 = r2 - (r1.conj() * r2).sum(dim=1, keepdim=True) * r1
    r2 = r2 / torch.linalg.vector_norm(r2, dim=1, keepdim=True)
    r0 = torch.stack([r1[:, 1] * r2[:, 2] - r1[:, 2] * r2[:, 1], r1[:, 2] * r2[:, 0] - r1[:, 0] * r2[:, 2],
                      r1[:, 0] * r2[:, 1] - r1[:, 1] * r2[:, 0]], dim=1).conj()
    q = torch.stack([r0, r1, r2], dim=1)
    return torch.view_as_real(q).reshape(4, V, 3, 3, 2).contiguous()


def boundary_links_from_neighbours(u, X, grid):
    """per partitioned dimension: the backward neighbour's x[d] = X[d]-1 links of direction d, in face order (NCCL)"""
    import torch
    import torch.distributed as dist
    from quda_b200 import fields as F
    Vh = F.volume_cb(X)
    faces = [None] * 4
    for d in range(4):
        if grid is None or grid.dims[d] == 1:
            continue
        g6 = u.reshape(4, 2, Vh, 3, 3, 2)
        mine = torch.stack([g6[d, p][torch.from_numpy(F.face_sites(X, d, X[d] - 1, p)).cuda()] for p in range(2)]).contiguous()
        theirs = torch.empty_like(mine)
        ops = [dist.P2POp(dist.isend, mine, grid.neighbor(d, +1)), dist.P2POp(dist.irecv, theirs, grid.neighbor(d, -1))]
        for w in dist.batch_isend_irecv(ops):
            w.wait()
        torch.cuda.synchronize()
        faces[d] = theirs
    return faces


def device_clover(X, prec, seed=5):
    """Synthetic clover term built on the device (1 + Hermitian noise of norm 0.01 with the symmetry the compressed format
    assumes, as tests/utils/host_utils.cpp:1162-1188) and marshaled by b200_copy_clover into the native compressed layout."""
    import ctypes as C
    import torch
    from quda_b200 import dslash as D
    from quda_b200 import fields as F
    from quda_b200 import lib as L
    Vh = F.volume_cb(X)
    V = 2 * Vh
    g = torch.Generator(device="cuda").manual_seed(seed)
    c = torch.rand((V, 2, 36), dtype=torch.float64, device="cuda", generator=g) * 0.02 - 0.01
    for dst, src in zip((3, 4, 5, 30, 31, 32, 33, 34, 35), (0, 1, 2, 6, 7, 8, 9, 16, 17)):
        c[:, :, dst] = -c[:, :, src]
    c[:, :, :6] += 1.0
    blk = c.reshape(-1, 36)
    diagonal = float((0.25 * (blk[:, 0:3] + blk[:, 3:6])).mean())
    half = 0.5 * blk
    mx = float(torch.maximum((half[:, 0:3] - diagonal).abs().max(), half[:, 6:30].abs().max()))
    nbytes = 2 * 2 * 28 * Vh * prec
    buf = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
    meta = dict(parity_stride_bytes=nbytes // 2, diagonal=diagonal, max_element=2.0 * mx, compressed=1)
    A = D.CloverField(buf, X, prec, meta, dynamic=True)
    d = A.desc()
    Xc = (C.c_int * 4)(*[int(v) for v in X])
    L.check(L.load().b200_copy_clover(C.byref(d), prec, Xc, c.data_ptr(), 8, None))
    torch.cuda.synchronize()
    return A


def run_cg(a):
    """BASELINE config 5: Wilson-clover, even-odd preconditioned (symmetric, even-even), CG on the normal equations to
    `--tol`, double precision with single-precision sloppy operator + reliable updates (lib/inv_cg_quda.cpp), on a FIXED
    global lattice (default 48^3 x 96) split over the ranks -- strong scaling.  Reports iterations, time to solution and
    the solver's sustained GFLOP/s (the reference's own accounting, tests/invert_test.cpp:335-338)."""
    import torch
    from quda_b200 import comm, dirac as DR, dslash as D, fields as F, lib as L

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        if not os.environ.get("NCCL_DEBUG"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = L.load()
    dims = comm.ProcessGrid.default_dims(world)
    grid = comm.ProcessGrid(dims, rank) if world > 1 else None
    Xg = a.global_dim
    X = [Xg[d] // dims[d] for d in range(4)]
    assert all(X[d] * dims[d] == Xg[d] and X[d] % 2 == 0 for d in range(4)), f"global lattice {Xg} does not split over {dims}"
    Vh = F.volume_cb(X)
    torch.manual_seed(4321 + rank)
    u = random_su3_device(X)
    faces = boundary_links_from_neighbours(u, X, grid)
    ops, keep = {}, []
    stream = torch.cuda.current_stream().cuda_stream
    for prec, recon in ((8, 18), (4, 12)):
        gbuf, gmeta = F.gauge_to_native_torch(u, X, prec, recon, ghost_faces=faces)
        U = D.GaugeField(gbuf, X, prec, recon, gmeta, anisotropy=1.0, t_boundary=-1,
                         first_time_slice=grid.first_time_slice() if grid else True,
                         last_time_slice=grid.last_time_slice() if grid else True)
        A = device_clover(X, prec)
        cs = None
        if world > 1:
            ex = comm.HaloExchange(grid, X, prec, mode="p2p", dist=dist)
            cs = ex.comm_struct()
            keep += [ex, cs]
        ops[prec] = DR.Dirac("cloverpc", U, a.kappa, clover=A, comm=cs, stream=stream)
        keep += [U, A]
    del u
    pc = ops[8]
    pb = F.spinor_bytes(X, 8)
    g = torch.Generator(device="cuda").manual_seed(99 + rank)
    b = torch.rand(2 * pb // 8, dtype=torch.float64, device="cuda", generator=g).view(torch.uint8)
    bdev = D.ColorSpinorField(b, X, 8, 2)
    xdev = D.ColorSpinorField(torch.zeros(2 * pb, dtype=torch.uint8, device="cuda"), X, 8, 2)
    rhs = D.ColorSpinorField(torch.zeros(pb, dtype=torch.uint8, device="cuda"), X, 8)

    def solve():
        xdev.buf.zero_()
        src_p, sol_p = pc.prepare(xdev, bdev)
        src = D.ColorSpinorField(xdev.buf[src_p * pb:(src_p + 1) * pb], X, 8)
        sol = D.ColorSpinorField(xdev.buf[sol_p * pb:(sol_p + 1) * pb], X, 8)
        pc.Mdag(rhs, src)
        sol.buf.zero_()
        res = DR.invert_cg(pc, ops[4], sol, rhs, tol=a.tol, maxiter=20000)
        pc.reconstruct(xdev, bdev)
        return res

    with ClockSampler(local_rank) as cs_clk:
        for _ in range(1 if a.warmup > 0 else 0):
            solve()  # one untimed solve: first-use allocations, clocks
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        lib.b200_reset_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = solve()
        e1.record()
        torch.cuda.synchronize()
        launches = lib.b200_launch_count()
    secs = e0.elapsed_time(e1) * 1e-3
    if world > 1:
        t = torch.tensor([secs, res.secs], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        secs, solver_secs = float(t[0]), float(t[1])
    else:
        solver_secs = res.secs
    # full-system true residual |b - M x| / |b| recomputed with the UNpreconditioned double-precision operator
    full = DR.Dirac("clover", ops[8].U, a.kappa, clover=ops[8].clover, comm=ops[8].comm, stream=stream)
    Mx = D.ColorSpinorField(torch.zeros(2 * pb, dtype=torch.uint8, device="cuda"), X, 8, 2)
    full.M(Mx, xdev)
    torch.cuda.synchronize()
    # plain sums over the native buffers are layout independent
    d2 = (Mx.buf.view(torch.float64) - bdev.buf.view(torch.float64)).pow(2).sum()
    b2 = bdev.buf.view(torch.float64).pow(2).sum()
    nrm = torch.stack([d2, b2])
    if world > 1:
        dist.all_reduce(nrm)
    true_res = float((nrm[0] / nrm[1]).sqrt())
    gflops = res.gflops * res.secs / solver_secs * world  # per-rank flop count is identical on every rank
    out = {"metric": "wilson_clover_cg_gflops", "value": gflops, "unit": "GFLOP/s", "n_gpus": world, "steps": 1,
           "warmup": 1 if a.warmup > 0 else 0, "ms_per_step": secs * 1e3, "higher_is_better": True, "scaling": "strong",
           "vs_baseline": None, "dtype": "f64/f32 mixed", "data": "synthetic",
           "config": {"workload": f"Wilson-clover CG (MdagM of the symmetric even-even preconditioned operator, prepare + "
                                  f"reconstruct included), global {'x'.join(map(str, Xg))}, local {'x'.join(map(str, X))}, "
                                  f"double recon-18 / single recon-12 sloppy with reliable updates, tol {a.tol:g}, kappa {a.kappa}",
                      "grid": dims},
           "cg": {"iterations": res.iter, "reliable_updates": res.reliable_updates, "time_to_solution_s": secs,
                  "solver_secs": solver_secs, "solver_true_res_normal_eq": res.true_res, "true_res_full_system": true_res,
                  "flop_accounting": "blas flops + 1320 per Dslash site application (clover flops not counted), as the reference"},
           "gpu_launches": int(launches), "clocks": cs_clk.summary()}
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def ncu_traffic(a):
    """dram bytes per launch of the interior kernel from the committed ncu capture (profiles/), if any."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get(f"{a.prec}-r{a.recon}")
    return None


def make_device_problem(X, prec, recon, grid=None):
    """Native-order synthetic fields (random unitary links via QR on the device, uniform spinors).  With a process grid
    the pad of every partitioned dimension is filled with the backward neighbour's boundary links (NCCL exchange)."""
    import numpy as np
    import torch
    from quda_b200 import dslash as D
    from quda_b200 import fields as F

    Vh = F.volume_cb(X)
    V = 2 * Vh
    # random SU(3) the way the reference's tests build it (tests/utils/host_utils.cpp:1022-1098): two random rows,
    # Gram-Schmidt, third row = conjugate cross product -- all element-wise torch ops on the device
    r1 = torch.randn(4 * V, 3, dtype=torch.complex128, device="cuda")
    r2 = torch.randn(4 * V, 3, dtype=torch.complex128, device="cuda")
    r1 = r1 / torch.linalg.vector_norm(r1, dim=1, keepdim=True)
    r2 = r2 - (r1.conj() * r2).sum(dim=1, keepdim=True) * r1
    r2 = r2 / torch.linalg.vector_norm(r2, dim=1, keepdim=True)
    r0 = torch.stack([r1[:, 1] * r2[:, 2] - r1[:, 2] * r2[:, 1], r1[:, 2] * r2[:, 0] - r1[:, 0] * r2[:, 2],
                      r1[:, 0] * r2[:, 1] - r1[:, 1] * r2[:, 0]], dim=1).conj()
    q = torch.stack([r0, r1, r2], dim=1)
    u = torch.view_as_real(q).reshape(4, V, 3, 3, 2).contiguous()
    del r0, r1, r2, q
    ghost_faces = None
    if grid is not None:
        import torch.distributed as dist
        ghost_faces = [None] * 4
        for d in range(4):
            if grid.dims[d] == 1:
                continue
            g6 = u.reshape(4, 2, Vh, 3, 3, 2)
            mine = torch.stack([g6[d, p][torch.from_numpy(F.face_sites(X, d, X[d] - 1, p)).cuda()] for p in range(2)]).contiguous()
            theirs = torch.empty_like(mine)
            ops = [dist.P2POp(dist.isend, mine, grid.neighbor(d, +1)), dist.P2POp(dist.irecv, theirs, grid.neighbor(d, -1))]
            for w in dist.batch_isend_irecv(ops):
                w.wait()
            torch.cuda.synchronize()
            ghost_faces[d] = theirs
    gbuf, gmeta = F.gauge_to_native_torch(u, X, prec, recon, ghost_faces=ghost_faces)
    del u
    U = D.GaugeField(gbuf, X, prec, recon, gmeta, anisotropy=1.0, t_boundary=1,
                     first_time_slice=grid.first_time_slice() if grid else True,
                     last_time_slice=grid.last_time_slice() if grid else True)
    rng = np.random.default_rng(7)
    s = rng.random((Vh, 4, 3, 2))
    sbuf = F.spinor_to_native(s, prec, rotate=False)
    inp = D.ColorSpinorField(torch.from_numpy(sbuf).cuda(), X, prec, 1)
    out = D.ColorSpinorField(torch.zeros(len(sbuf), dtype=torch.uint8, device="cuda"), X, prec, 1)
    return {"U": U, "in": inp, "out": out, "host_in": sbuf}


def make_device_clover(X, prec, static_inverse=False):
    """Synthetic clover term in the native compressed layout: 1 + small Hermitian noise with the symmetry the 28-real
    format assumes (the construction of tests/utils/host_utils.cpp:1162-1188 with numpy's generator).
    static_inverse: an uncompressed field applied as a stored A^-1 (synthetic values: timing only)."""
    import numpy as np
    import torch
    from quda_b200 import dslash as D
    from quda_b200 import fields as F
    V = 2 * F.volume_cb(X)
    rng = np.random.default_rng(5)
    c = (rng.random((V, 2, 36)) * 0.02 - 0.01)
    for dst, src in zip((3, 4, 5, 30, 31, 32, 33, 34, 35), (0, 1, 2, 6, 7, 8, 9, 16, 17)):
        c[:, :, dst] = -c[:, :, src]
    c[:, :, :6] += 1.0
    buf, meta = F.clover_to_native(c, X, prec, compressed=not static_inverse)
    return D.CloverField(torch.from_numpy(buf).cuda(), X, prec, meta, dynamic=not static_inverse)


def e2e(a, P, lib, Vh, prec, world, make_dirac=None, dist=None):
    """Same metric through the public calls with HOST spinor buffers (pinned, host interface order): every step copies
    its input spinor host->device, converts it to the native order (b200_copy_spinor), applies the Dslash, converts the
    result back and copies it device->host -- the dslashQuda flow (lib/interface_quda.cpp:1709-1783).  Steps are software-pipelined over three
    streams with double-buffered device fields (copy-in of step i+1 and copy-out of step i-1 overlap the kernel of
    step i), the way a multi-source workload drives dslashQuda; every step still moves all of its bytes."""
    import numpy as np
    import torch
    from quda_b200 import dslash as D
    X = P["in"].X
    nat_bytes = len(P["host_in"])
    # host interface order: [site][spin][colour][re,im] fp32, DeGrand-Rossi basis (what dslashQuda is handed)
    h_in = torch.from_numpy(np.random.default_rng(11).random((Vh, 4, 3, 2), dtype=np.float32)).pin_memory()
    nbytes = h_in.numel() * 4
    h_out = [torch.empty((Vh, 4, 3, 2), dtype=torch.float32).pin_memory() for _ in range(2)]
    s_hin = [torch.empty((Vh, 4, 3, 2), dtype=torch.float32, device="cuda") for _ in range(2)]
    s_hout = [torch.empty((Vh, 4, 3, 2), dtype=torch.float32, device="cuda") for _ in range(2)]
    d_in = [D.ColorSpinorField(torch.empty(nat_bytes, dtype=torch.uint8, device="cuda"), X, prec) for _ in range(2)]
    d_out = [D.ColorSpinorField(torch.empty(nat_bytes, dtype=torch.uint8, device="cuda"), X, prec) for _ in range(2)]
    s_in, s_k, s_out = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
    op = make_dirac(s_k.cuda_stream) if make_dirac is not None else None  # partitioned operator bound to the kernel stream
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_k = [torch.cuda.Event() for _ in range(2)]
    ev_out = [torch.cuda.Event() for _ in range(2)]

    def run(n):
        for i in range(n):
            b = i & 1
            with torch.cuda.stream(s_in):
                s_in.wait_event(ev_k[b])       # staging buffer b free once the kernels two steps back have read it
                s_hin[b].copy_(h_in, non_blocking=True)
                ev_in[b].record(s_in)
            with torch.cuda.stream(s_k):
                s_k.wait_event(ev_in[b])
                s_k.wait_event(ev_out[b])      # s_hout[b] free once its previous content went to the host
                D.copy_spinor(d_in[b], s_hin[b], True, stream=s_k.cuda_stream)      # host order -> native (UKQCD)
                if op is not None:
                    op.Dslash(d_out[b], d_in[b], 0)
                else:
                    D.ApplyWilson(d_out[b], d_in[b], P["U"], 0.0, None, 0, 0, tile=a.tile, stream=s_k.cuda_stream)
                D.copy_spinor(d_out[b], s_hout[b], False, stream=s_k.cuda_stream)   # native -> host order
                ev_k[b].record(s_k)
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_k[b])
                h_out[b].copy_(s_hout[b], non_blocking=True)
                ev_out[b].record(s_out)

    run(4)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    n = max(6, min(a.steps, 60))
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(s_in)
    run(n)
    s_out.synchronize()
    ev1.record(s_out)
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / n
    if dist is not None:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return {"value": D.flops_per_site() * Vh * world / (ms * 1e-3) * 1e-9, "unit": "GFLOP/s", "ms_per_step": ms,
            "h2d_bytes_per_step": nbytes * world, "d2h_bytes_per_step": nbytes * world, "steps": n,
            "ranks_measured": world,
            "note": "host spinor in/out in the interface order (fp32 [site][spin][colour][2], DeGrand-Rossi, pinned); per "
                    "step: H2D, reorder+basis rotation kernel, Dslash, reorder kernel, D2H; 3-stream pipeline; gauge "
                    "resident as after loadGaugeQuda"}


def sweep(a, P, lib):
    """Dev tool: time the interior kernel for a list of tilings; results -> gpurun_out/sweep.json."""
    import torch
    from quda_b200 import dslash as D
    from quda_b200 import fields as F
    X = a.dim
    prec = PREC_BYTES[a.prec]
    Vh = F.volume_cb(X)
    tiles = []
    for t0 in (2, 4, 8, 16):
        for t1 in (1, 2, 4, 8, 16, 32):
            for t2 in (1, 2, 4, 8):
                for t3 in (1, 2, 4, 8):
                    v = t0 * t1 * t2 * t3
                    if v in (64, 128, 256, 512) and t0 <= X[0] // 2 and t1 <= X[1] and t2 <= X[2] and t3 <= X[3]:
                        tiles.append((t0, t1, t2, t3))
    stream = torch.cuda.current_stream().cuda_stream
    res = []
    bmin = D.min_bytes_per_site(prec, a.recon)
    for t in tiles:
        for _ in range(3):
            D.ApplyWilson(P["out"], P["in"], P["U"], 0.0, None, 0, 0, tile=t, stream=stream)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        n = 20
        for _ in range(n):
            D.ApplyWilson(P["out"], P["in"], P["U"], 0.0, None, 0, 0, tile=t, stream=stream)
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) / n * 1e3
        res.append({"tile": t, "us": us, "gbs": bmin * Vh / us * 1e-3})
    res.sort(key=lambda r: r["us"])
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    name = f"sweep_{a.prec}_r{a.recon}.json"
    json.dump(res, open(os.path.join(ROOT, "gpurun_out", name), "w"), indent=0)
    for r in res[:8]:
        print("sweep", a.prec, a.recon, r)
    print("sweep worst", res[-1])


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    elif args.op == "cg":
        run_cg(args)
    else:
        run_b200(args)
