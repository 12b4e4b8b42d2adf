"""Cost of the forward-mode tangent at the bench batch: MPC02 x 65 536 (bench.py's seeded h / b), device-resident, on
one GPU.

Times, in one process and after warm-up, with CUDA events around whole synchronised calls:
  - one forward step (eicos_batch_solve_device);
  - one tangent step with a direction in c, h and b only (eicos_batch_tangent_device, all four outputs);
  - one tangent step with directions in G and A as well (reads the 5 GB of direction stacks);
  - one adjoint step (eicos_batch_adjoint_device, all five gradients).
The gap between the two tangent steps is the cost of reading the G / A stacks.  Prints one JSON object with the status
counts and the GPU's name and power limit, read in the same run.
    python tools/tangent_bench.py [--batch 65536] [--steps 3] [--warmup 1] [--out FILE]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from adjoint_bench import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out")
    args = ap.parse_args()

    import torch
    import eicos_b200
    import oracle
    from eicos_b200.workloads import MPC_REL, perturbed

    P = oracle.load_fixture("MPC02")
    B = args.batch
    W = perturbed(P, B, rel=MPC_REL, seed=1234)  # bench.py's default workload and seed on rank 0
    dev = torch.device("cuda", 0)
    f64 = dict(dtype=torch.float64, device=dev)
    hs = torch.from_numpy(np.ascontiguousarray(W["hs"])).to(dev)
    bs = torch.from_numpy(np.ascontiguousarray(W["bs"])).to(dev)
    solver = eicos_b200.BatchSolver(P, device=0, capacity=B)
    n, m, p = solver.n, solver.m, solver.p
    x, y, z, s = (torch.empty((B, k), **f64) for k in (n, p, m, m))
    ex = torch.empty((B,), dtype=torch.int32, device=dev)
    gen = torch.Generator(dev).manual_seed(1)
    v = {k: torch.randn((B, c), generator=gen, **f64) for k, c in (("c", n), ("h", m), ("b", p), ("G", solver.nnzG), ("A", solver.nnzA))}
    g = [torch.randn((B, k), generator=gen, **f64) for k in (n, p, m)]
    o = {k: torch.empty((B, c), **f64) for k, c in (("x", n), ("y", p), ("z", m), ("s", m))}
    d = {k: torch.empty((B, c), **f64) for k, c in (("c", n), ("h", m), ("b", p), ("G", solver.nnzG), ("A", solver.nnzA))}
    st_chb, st_all, st_adj = (torch.empty((B,), dtype=torch.int32, device=dev) for _ in range(3))

    def forward():
        solver.solve_device(B, d_hs=hs.data_ptr(), d_bs=bs.data_ptr(), d_x=x.data_ptr(), d_y=y.data_ptr(),
                            d_z=z.data_ptr(), d_s=s.data_ptr(), d_exit=ex.data_ptr())

    def tangent(with_matrices, status):
        solver.tangent_device(B, d_x=x.data_ptr(), d_y=y.data_ptr(), d_z=z.data_ptr(), d_s=s.data_ptr(),
                              d_exit=ex.data_ptr(), d_dc=v["c"].data_ptr(), d_dh=v["h"].data_ptr(), d_db=v["b"].data_ptr(),
                              d_dG=v["G"].data_ptr() if with_matrices else 0, d_dA=v["A"].data_ptr() if with_matrices else 0,
                              d_ox=o["x"].data_ptr(), d_oy=o["y"].data_ptr(), d_oz=o["z"].data_ptr(), d_os=o["s"].data_ptr(),
                              d_status=status.data_ptr())

    def adjoint():
        solver.adjoint_device(B, d_x=x.data_ptr(), d_y=y.data_ptr(), d_z=z.data_ptr(), d_s=s.data_ptr(),
                              d_exit=ex.data_ptr(), d_gx=g[0].data_ptr(), d_gy=g[1].data_ptr(), d_gz=g[2].data_ptr(),
                              d_dc=d["c"].data_ptr(), d_dh=d["h"].data_ptr(), d_db=d["b"].data_ptr(),
                              d_dG=d["G"].data_ptr(), d_dA=d["A"].data_ptr(), d_status=st_adj.data_ptr())

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(args.steps):
            fn()
        t1.record()
        torch.cuda.synchronize()
        return t0.elapsed_time(t1) / args.steps

    gpu = gpu_info()
    ms_fwd = timed(forward)
    ms_chb = timed(lambda: tangent(False, st_chb))
    finite_chb = bool(all(torch.isfinite(a).all() for a in o.values()))
    ms_all = timed(lambda: tangent(True, st_all))
    finite_all = bool(all(torch.isfinite(a).all() for a in o.values()))
    ms_adj = timed(adjoint)
    exits = ex.cpu().numpy()
    opt = (exits == 0) | (exits == 10)

    def hist(t):
        a = t.cpu().numpy()
        return {str(int(k)): int(c) for k, c in zip(*np.unique(a, return_counts=True))}, int((a[opt] == 0).sum())

    (h_chb, ok_chb), (h_all, ok_all), (h_adj, ok_adj) = hist(st_chb), hist(st_all), hist(st_adj)
    stack_gb = B * (solver.nnzG + solver.nnzA) * 8 / 1e9
    result = {"workload": f"MPC02 x{B}, h*(1+-0.2%) b*(1+-2%), seed 1234, device-resident", "gpu": gpu,
              "steps": args.steps, "warmup": args.warmup,
              "ms_forward": ms_fwd, "ms_tangent_chb": ms_chb, "ms_tangent_chbGA": ms_all, "ms_adjoint": ms_adj,
              "ms_read_GA_stacks": ms_all - ms_chb, "GA_stack_GB": stack_gb,
              "GA_stack_GBps": stack_gb / ((ms_all - ms_chb) / 1e3) if ms_all > ms_chb else None,
              "optimal": int(opt.sum()), "status_0_of_optimal": {"tangent_chb": ok_chb, "tangent_chbGA": ok_all, "adjoint": ok_adj},
              "status_histogram": {"tangent_chb": h_chb, "tangent_chbGA": h_all, "adjoint": h_adj},
              "tangents_finite": finite_chb and finite_all, "gpu_after": gpu_info()}
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
