#!/usr/bin/env python3
"""Benchmark of the batched SOCP interior-point hot path (BASELINE.json metric: SOCP solves/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload mpc02|mpc02pct5|mpc02pim|socmpc|lp25fv47] [--batch B] [--scaling strong|weak]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch: updateData (per-instance h, b) + solve for
every instance of the batch.  Workload at N=1: BASELINE.json configs[2] - the reference's MPC data
set x65536 with perturbed h/b.  The checkout lacks data_MPC01.hpp / test/MPC/MPC01.h (SURVEY.md F3),
so the reference's own sibling fixture MPC02 (test/MPC/MPC02.h) stands in; `--workload socmpc` runs a
builder-defined SOC-bearing MPC instead.  One process per GPU (torchrun), the batch is sharded by
instance, no data-path collective; --scaling strong (default) = --batch instances IN TOTAL (the metric's
configuration: 65536 over 1/2/4/8 GPUs), weak = per GPU.

JSON line (rank 0): value = whole-job solves/s with inputs resident in HBM (device-timed, max over
ranks); e2e = the same through the C ABI with HOST buffers (H2D of h,b and D2H of x + exit flags in
the timed region); roofline = the dominant kernel (eicos_solve_kkt: triangular solves + refinement
residual) against the measured HBM peak; cpu_baseline = the CPU oracle on this box's host cores.
--dump-outputs DIR writes what the last timed device-resident step returned (rank 0's instances) as
DIR/<name>.npy; the inputs are seeded, so two builds run with the same arguments can be compared
output for output.
`--impl reference` times the reference path on the host cores: the reference itself needs Eigen,
which is absent (oracle/Makefile), so it is the oracle port, one solver per core, updateData +
solve per instance exactly as BASELINE.md section 3 prescribes.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="mpc02", choices=["mpc02", "mpc02pct5", "mpc02pim", "socmpc", "lp25fv47"])
    ap.add_argument("--batch", type=int, default=65536, help="instances in total (strong, the metric's configuration) or per GPU (weak)")
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"])
    ap.add_argument("--workers", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-handles", type=int, default=0,
                    help="end-to-end arm: handles (one stream and one host thread each) on the device behind eicos_multi_solve; "
                         "copies of one slice overlap the kernels of the others (1 = eicos_batch_solve on the device arm's handle; "
                         "0 = choose: one handle per 16384 instances of this GPU's share, at most 4)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float64, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, x, exits, iters):
    """What the caller of the device-resident path receives: exit.npy and iter.npy of every instance, and x.npy, the
    solutions of every instance or, where they would not fit DUMP_BYTES, of a fixed seeded sample of the instances
    (x_instances.npy lists them, in order)."""
    import torch
    batch, n = x.shape
    rows = min(batch, (DUMP_BYTES - 4 * 128 - 16 * batch) // (8 * (n + 1)))  # 128: an .npy header
    idx = np.arange(batch) if rows == batch else np.sort(np.random.default_rng(0).choice(batch, rows, replace=False))
    xs = torch.index_select(x, 0, torch.from_numpy(idx).to(x.device)).cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("x", xs), ("x_instances", idx), ("exit", exits), ("iter", iters)):
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def make_problem(workload):
    """Problem data + a function producing the per-instance stacks for `batch` instances."""
    from eicos_b200.workloads import MPC_REL, perturbed, perturbed_matrices, soc_mpc, soc_mpc_batch
    if workload == "mpc02pim":  # SURVEY.md 8f row 1: every instance brings its own G / A values (linearised dynamics)
        d = np.load(os.path.join(ROOT, "tests", "golden", "fixtures", "MPC02.npz"))
        P = {k: d[k] for k in d.files}
        for k in ("n", "m", "p", "l", "ncones"):
            P[k] = int(P[k])
        name = ("MPC02 (reference test/MPC/MPC02.h) x{B}, per-instance G*(1+-0.1%) A*(1+-0.1%) values on the shared "
                "pattern plus h*(1+-0.2%) b*(1+-2%), via updateData(Gpr, Apr, c, h, b); equilibration per instance on the device")

        def gen(batch, seed):
            W = perturbed(P, batch, rel=MPC_REL, seed=seed)
            M = perturbed_matrices(P, batch, rel=0.001, seed=seed + 50000)
            W["Gs"], W["As"] = M["Gs"], M["As"]
            return W
        return P, name, gen
    if workload == "mpc02pct5":  # SURVEY.md 8d config 3 as written: h and b perturbed by +-5 % (most instances turn infeasible)
        d = np.load(os.path.join(ROOT, "tests", "golden", "fixtures", "MPC02.npz"))
        P = {k: d[k] for k in d.files}
        for k in ("n", "m", "p", "l", "ncones"):
            P[k] = int(P[k])
        name = ("MPC02 (reference test/MPC/MPC02.h) x{B}, h*(1+-5%) b*(1+-5%) per instance via updateData "
                "(the survey's recipe: a mix of optimal and primal-infeasible instances), G/A/c shared")
        return P, name, lambda batch, seed: perturbed(P, batch, rel=0.05, seed=seed)
    if workload == "mpc02":
        d = np.load(os.path.join(ROOT, "tests", "golden", "fixtures", "MPC02.npz"))
        P = {k: d[k] for k in d.files}
        for k in ("n", "m", "p", "l", "ncones"):
            P[k] = int(P[k])
        name = ("MPC02 (reference test/MPC/MPC02.h; stands in for the missing MPC01) x{B}, "
                "h*(1+-0.2%) b*(1+-2%) per instance via updateData, G/A/c shared")
        return P, name, lambda batch, seed: perturbed(P, batch, rel=MPC_REL, seed=seed)
    if workload == "lp25fv47":  # BASELINE.json configs[4]: c and b perturbed by 1 % (SURVEY.md 8d)
        d = np.load(os.path.join(ROOT, "tests", "golden", "fixtures", "lp_25fv47.npz"))
        P = {k: d[k] for k in d.files}
        for k in ("n", "m", "p", "l", "ncones"):
            P[k] = int(P[k])
        name = "lp_25fv47 (reference test/LPnetlib/lp_25fv47.h) x{B}, c*(1+-1%) b*(1+-1%) per instance, G/A/h shared"
        return P, name, lambda batch, seed: perturbed(P, batch, rel=0.01, seed=seed, vary=("c", "b"))
    P = soc_mpc(T=40)
    name = "builder-defined SOC MPC (2-D double integrator, T=40, 80 cones of dim 3/5) x{B}, x0/ref per instance"
    return P, name, lambda batch, seed: soc_mpc_batch(P, batch, seed=seed)


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_baseline(P, gen, cores, seconds_target=15.0):
    """CPU oracle, one solver per core, updateData+solve per instance, on a bounded sample."""
    import oracle
    probe_n = max(2 * cores, 8)
    W = gen(probe_n, 991)
    t = oracle.batch_run(P, probe_n, Gs=W.get("Gs"), As=W.get("As"), hs=W["hs"], bs=W["bs"], cs=W.get("cs"), nthreads=cores, want_solution=False)["seconds"]
    per = max(t / probe_n, 1e-6)
    sample = int(min(8192, max(probe_n, seconds_target / per)))
    W = gen(sample, 992)
    r = oracle.batch_run(P, sample, Gs=W.get("Gs"), As=W.get("As"), hs=W["hs"], bs=W["bs"], cs=W.get("cs"), nthreads=cores, want_solution=False)
    return {"value": sample / r["seconds"], "unit": "solves/s", "cores": cores, "kind": "port",
            "exit_flags": {int(k): int(v) for k, v in zip(*np.unique(r["exit"], return_counts=True))},
            "iterations_mean": float(r["iter"].mean()),
            "sample": f"{sample} instances of the same workload, {cores} threads, one solver per thread, "
                      f"updateData+solve per instance (includes re-equilibration and the per-solve AMD ordering), "
                      f"{r['seconds']:.1f} s; exit flags {dict(zip(*[a.tolist() for a in np.unique(r['exit'], return_counts=True)]))}, "
                      f"mean iterations {float(r['iter'].mean()):.1f}"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path (oracle port) on the host cores, rank 0 only."""
    if rank != 0:
        return
    P, name, gen = make_problem(args.workload)
    import oracle
    cores = host_cores()
    probe = gen(max(2 * cores, 8), 990)
    nprobe = max(2 * cores, 8)
    t = oracle.batch_run(P, nprobe, Gs=probe.get("Gs"), As=probe.get("As"), cs=probe.get("cs"), hs=probe["hs"], bs=probe["bs"], nthreads=cores, want_solution=False)["seconds"]
    per = max(t / nprobe, 1e-6)
    total_steps = args.steps + args.warmup
    sample = int(min(4096, max(cores, (120.0 / total_steps) / per)))  # whole run within a few minutes
    W = gen(sample, 1234)
    for _ in range(args.warmup):
        oracle.batch_run(P, sample, Gs=W.get("Gs"), As=W.get("As"), cs=W.get("cs"), hs=W["hs"], bs=W["bs"], nthreads=cores, want_solution=False)
    secs, exits = 0.0, None
    for _ in range(args.steps):
        r = oracle.batch_run(P, sample, Gs=W.get("Gs"), As=W.get("As"), cs=W.get("cs"), hs=W["hs"], bs=W["bs"], nthreads=cores, want_solution=False)
        secs += r["seconds"]
        exits = r["exit"]
    value = args.steps * sample / secs
    desc = (f"{sample} instances per step ({args.steps} steps), {cores} threads, one solver per thread, "
            f"updateData+solve per instance; optimal: {int((exits == 0).sum())}/{sample}")
    line = {"impl": "reference", "metric": "SOCP solves/sec", "value": value, "unit": "solves/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": name.format(B=args.batch * (args.gpus if args.scaling == "weak" else 1)), "reference_impl": "CPU oracle port of EiCOS (Eigen absent: the reference itself cannot be built)"},
            "cpu_baseline": {"value": value, "unit": "solves/s", "cores": cores, "kind": "port", "sample": desc},
            "e2e": {"value": value, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import eicos_b200
    from eicos_b200.sharding import shard_range

    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    P, name, gen = make_problem(args.workload)
    if args.scaling == "weak":
        batch = args.batch
        seed = 1234 + rank
    else:
        lo, hi = shard_range(args.batch, rank, world)
        batch = hi - lo
        seed = 1234 + rank
    n, m, p = P["n"], P["m"], P["p"]
    W = gen(batch, seed)
    # per-instance stacks (pinned host copies); a vector the workload does not vary stays shared (None)
    host = {k: (torch.from_numpy(np.ascontiguousarray(W[k])).pin_memory() if W.get(k) is not None else None)
            for k in ("cs", "hs", "bs", "Gs", "As")}
    pim = host["Gs"] is not None or host["As"] is not None
    x_h = torch.empty((batch, n), dtype=torch.float64).pin_memory()
    exit_h = torch.empty((batch,), dtype=torch.int32).pin_memory()

    solver = eicos_b200.BatchSolver(P, device=local, capacity=batch, workers=args.workers, instance_matrices=pim)
    dims = solver.dims()
    stream = torch.cuda.ExternalStream(solver.stream(), device=dev)

    devb = {k: (v.to(dev) if v is not None else None) for k, v in host.items()}
    dptr = {k: (v.data_ptr() if v is not None else 0) for k, v in devb.items()}
    x_d = torch.empty((batch, n), dtype=torch.float64, device=dev)
    exit_d = torch.empty((batch,), dtype=torch.int32, device=dev)
    iter_d = torch.empty((batch,), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()

    def step_device():
        solver.solve_device(batch, d_Gs=dptr["Gs"], d_As=dptr["As"], d_cs=dptr["cs"], d_hs=dptr["hs"], d_bs=dptr["bs"], d_x=x_d.data_ptr(),
                            d_exit=exit_d.data_ptr(), d_iter=iter_d.data_ptr())

    lib = solver.lib
    # (slices below ~16k instances run at the per-tile latency floor: splitting further only adds launches)
    e2e_handles = args.e2e_handles if args.e2e_handles > 0 else max(1, min(4, batch // 16384))
    multi = []  # the end-to-end arm's handle (built after the device arm has released its workspace)

    def step_host():
        L = lib.L
        import ctypes as C
        dp = C.POINTER(C.c_double)
        hp = {k: (C.cast(v.data_ptr(), dp) if v is not None else None) for k, v in host.items()}
        if multi:
            lib.check(L.eicos_multi_solve(
                multi[0].h, batch, hp["Gs"], hp["As"], hp["cs"], hp["hs"], hp["bs"],
                C.cast(x_h.data_ptr(), dp), None, None, None,
                C.cast(exit_h.data_ptr(), C.POINTER(C.c_int)), None))
            return
        lib.check(L.eicos_batch_solve_matrices(
            solver.h, batch, hp["Gs"], hp["As"], hp["cs"], hp["hs"], hp["bs"],
            C.cast(x_h.data_ptr(), dp), None, None, None,
            C.cast(exit_h.data_ptr(), C.POINTER(C.c_int)), None))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, collect=None, ev_stream=None):
        # events on the stream the kernels are launched on (device arm), or - for the synchronous host-buffer calls,
        # which return when their streams have drained - on torch's current stream
        ev_stream = ev_stream or stream
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(ev_stream)
        for _ in range(steps):
            fn()
            if collect is not None:
                collect(solver.stats())
        e1.record(ev_stream)
        barrier()
        ms = e0.elapsed_time(e1)
        timed.local_ms = ms
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    # ---- device-resident arm
    solver.set_timing(True)
    for _ in range(args.warmup):
        step_device()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    stats = []
    ms = timed(step_device, args.steps, stats.append)
    local_ms = timed.local_ms
    clocks = sampler.stop() if rank == 0 else None
    solver.set_timing(False)
    total_batch = batch * world if args.scaling == "weak" else args.batch
    value = total_batch * args.steps / (ms * 1e-3)
    exits = exit_d.cpu().numpy()
    iters = iter_d.cpu().numpy()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, x_d, exits, iters)

    # ---- end to end through the C ABI with host buffers
    e2e = None
    if not args.no_e2e:
        ev_stream = None
        if e2e_handles > 1:
            # several handles on THIS device behind one eicos_multi handle: contiguous slices, one stream and one host
            # thread each, so the H2D / D2H copies of one slice overlap the kernels of the others
            solver.close()
            del devb, x_d, exit_d, iter_d
            torch.cuda.empty_cache()
            multi.append(eicos_b200.MultiBatchSolver(P, devices=[local] * e2e_handles, capacity=-(-batch // e2e_handles),
                                                     workers=args.workers, lib=lib, instance_matrices=pim))
            ev_stream = torch.cuda.current_stream()
        for _ in range(max(1, min(args.warmup, 3))):
            step_host()
        ms_e = timed(step_host, args.steps, ev_stream=ev_stream)
        what = "pinned host " + ",".join(k[:-1] for k in ("Gs", "As", "cs", "hs", "bs") if host[k] is not None) + " in"
        e2e = {"value": total_batch * args.steps / (ms_e * 1e-3), "unit": "solves/s",
               "h2d_bytes_per_step": int(sum(v.numel() * 8 for v in host.values() if v is not None)),
               "d2h_bytes_per_step": int(batch * (n * 8 + 4)),
               "ms_per_step": ms_e / args.steps,
               "handles_on_device": e2e_handles,
               "api": ("eicos_multi_solve (include/eicos_b200.h) over %d handles on the device: %s; x and exit flags out" % (e2e_handles, what)
                       if e2e_handles > 1 else
                       ("eicos_batch_solve_matrices" if pim else "eicos_batch_solve") + " (include/eicos_b200.h): " + what + "; x and exit flags out")}
        assert np.array_equal(exit_h.numpy(), exits)

    # per-rank step time and iteration counts (the slowest rank sets the job's time: its slowest instance runs the
    # most interior-point iterations, and every one of them is at least a latency floor long)
    per_rank = None
    if world > 1:
        mine = torch.tensor([0.0, float(iters.max()), float(iters.mean()), float(batch)], dtype=torch.float64, device=dev)
        mine[0] = local_ms / args.steps
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = [{"rank": r, "ms_per_step": float(t[0]), "iterations_max": int(t[1]), "iterations_mean": float(t[2]),
                     "instances": int(t[3])} for r, t in enumerate(allr)]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel, from CUDA events inside the timed region (rank 0)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    N, nnzL, tile = dims["dim_K"], dims["nnzL"], dims["tile_width"]
    nnzV = dims["nnzV"]
    ms_solve = sum(s["ms_solve"] for s in stats)
    ms_factor = sum(s["ms_factor"] for s in stats)
    ms_other = sum(s["ms_other"] for s in stats)
    ms_kernels = ms_solve + ms_factor + ms_other
    rounds = sum(s["ir_rounds"] for s in stats)
    lane_rounds = sum(s["lane_rounds"] for s in stats)
    ms_resid = sum(s["ms_resid"] for s in stats)
    ms_vector = sum(s["ms_vector"] for s in stats)
    resid_tiles = sum(s["resid_launch_tiles"] for s in stats)
    vector_tiles = sum(s["vector_launch_tiles"] for s in stats)
    mt = m  # rows of a z-shaped vector (+ 2 per cone, none in the LP workloads)
    solve_launches = sum(s["solve_launches"] for s in stats)
    factor_launches = sum(s["factor_launches"] for s in stats)
    factor_tiles = sum(s["factor_launch_tiles"] for s in stats)
    # algorithmic bytes (SURVEY.md 8d, shared-A/G variant): one solve round = triangular solves
    # 8(2 nnzL + 3N) + refinement residual 8*4N per instance; a launch processes tile-rounds x 32 lanes
    # (per-instance matrices: the residual also reads every G / A value once, the factorisation too)
    nnzGA = (int(np.asarray(P["Gpr"]).size) + int(np.asarray(P["Apr"]).size)) if pim else 0
    bytes_round = 8.0 * (2 * nnzL + 7 * N + nnzGA) * tile
    solve_gbs = rounds * bytes_round / (ms_solve * 1e-3) / 1e9 if ms_solve > 0 else 0.0
    bytes_factor = 8.0 * (nnzV + nnzL + N + nnzGA) * tile
    factor_gbs = factor_tiles * bytes_factor / (ms_factor * 1e-3) / 1e9 if ms_factor > 0 else 0.0
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath))
        if traffic.get("_workload") != args.workload or traffic.get("_batch_per_gpu") != batch:
            traffic = None  # the ncu capture is of another configuration
    roofline = {"bound": "hbm", "kernel": "eicos_solve_kkt", "achieved": solve_gbs, "peak": peak, "unit": "GB/s",
                "frac": solve_gbs / peak, "peak_source": peak_src,
                "traffic": (traffic or {}).get("eicos_solve_kkt"),
                "algorithmic_bytes_per_launch": rounds * bytes_round / max(solve_launches, 1),
                "avg_launch_ms": ms_solve / max(solve_launches, 1),
                "share_of_step": ms_solve / ms_kernels if ms_kernels else None,
                "units": "tile-rounds x %d lanes: one unit = one solve round (forward + backward sweep + refinement residual) of one "
                         "instance, 8 (2 nnzL + 7 N) bytes (SURVEY.md 8d: B_sol + B_res, shared-A/G variant); finished lanes of a live "
                         "tile count (frac_lane_rounds counts only the rounds each instance needed itself)" % tile,
                "frac_lane_rounds": (lane_rounds * bytes_round / tile / (ms_solve * 1e-3) / 1e9 / peak) if ms_solve > 0 else None,
                "ldl_factor": {"kernel": "eicos_ldl_factor", "achieved": factor_gbs, "frac": factor_gbs / peak,
                               "algorithmic_bytes_per_launch": factor_tiles * bytes_factor / max(factor_launches, 1),
                               "avg_launch_ms": ms_factor / max(factor_launches, 1),
                               "share_of_step": ms_factor / ms_kernels if ms_kernels else None,
                               "traffic": (traffic or {}).get("eicos_ldl_factor")},
                # computeResiduals: [c|b|h], [x|y|z], s in, r out (+ the instance's G / A values); the three vector
                # kernels of an iteration: about 22 N-row passes together (DESIGN.md section 2)
                "residuals": {"kernel": "eicos_residuals",
                              "achieved": (resid_tiles * 8.0 * (3 * N + mt + nnzGA) * tile / (ms_resid * 1e-3) / 1e9) if ms_resid > 0 else 0.0,
                              "avg_launch_ms": ms_resid / max(sum(s["resid_launches"] for s in stats), 1),
                              "share_of_step": ms_resid / ms_kernels if ms_kernels else None},
                "vector_kernels": {"kernel": "eicos_iter_head + eicos_iter_mid + eicos_iter_tail",
                                   "achieved": (vector_tiles * 8.0 * (22.0 / 3.0) * N * tile / (ms_vector * 1e-3) / 1e9) if ms_vector > 0 else 0.0,
                                   "avg_launch_ms": ms_vector / max(sum(s["vector_launches"] for s in stats), 1),
                                   "share_of_step": ms_vector / ms_kernels if ms_kernels else None}}
    for k in ("residuals", "vector_kernels"):
        roofline[k]["frac"] = roofline[k]["achieved"] / peak

    # where the tiles spend their time inside eicos_solve_kkt (clock64 per phase, summed over tiles)
    pc = np.sum([s["kkt_phase_cycles"] for s in stats], axis=0).astype(float)
    phase_share = dict(zip(("rhs_norm", "forward", "backward", "residual", "bookkeeping"),
                           (pc / max(pc.sum(), 1.0)).round(4).tolist()))

    cpu = None
    if not args.no_cpu_baseline:
        cpu = cpu_baseline(P, gen, host_cores())

    ex_u, ex_c = np.unique(exits, return_counts=True)
    line = {"metric": "SOCP solves/sec", "value": value, "unit": "solves/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": name.format(B=total_batch), "batch_per_gpu": batch, "total_batch": total_batch,
                       "n": n, "m": m, "p": p, "dim_K": N, "nnzK": dims["nnzK"], "nnzL": nnzL,
                       "etree_height": dims["etree_height"], "workers_per_tile": dims["workers"],
                       "l2": "inputs and workspace (%.1f GB) are far larger than L2" % (dims["workspace_bytes"] / 1e9),
                       "exit_flags": dict(zip(ex_u.tolist(), ex_c.tolist())),
                       "iterations_mean": float(iters.mean()), "iterations_max": int(iters.max()),
                       "parallelism": f"batch sharded by instance over {world} GPU(s), no collective"},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
            "gpu_launches": int(sum(s["launches"] for s in stats)),
            "kernel_ms": {"solve_kkt": ms_solve, "ldl_factor": ms_factor, "other": ms_other, "residuals": ms_resid, "vector": ms_vector},
            "kkt_phase_share": phase_share,
            "per_rank": per_rank,
            "clocks": clocks}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
