"""Cost of the backward pass at the bench batch: MPC02 x 65 536 (bench.py's seeded h / b), device-resident, on one GPU.

Times one forward step (eicos_batch_solve_device) and one backward step (eicos_batch_adjoint_device, all five
gradients) with CUDA events around whole calls, after warm-up, and counts the status-0 instances.  Prints one JSON
object with the GPU's name and power limit, read in the same run.
    python tools/adjoint_bench.py [--batch 65536] [--steps 3] [--warmup 1] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


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
    g = [torch.randn((B, k), generator=gen, **f64) for k in (n, p, m)]
    d = {k: torch.empty((B, c), **f64) for k, c in (("c", n), ("h", m), ("b", p), ("G", solver.nnzG), ("A", solver.nnzA))}
    st = torch.empty((B,), dtype=torch.int32, device=dev)

    def forward():
        solver.solve_device(B, d_hs=hs.data_ptr(), d_bs=bs.data_ptr(), d_x=x.data_ptr(), d_y=y.data_ptr(),
                            d_z=z.data_ptr(), d_s=s.data_ptr(), d_exit=ex.data_ptr())

    def backward():
        solver.adjoint_device(B, d_x=x.data_ptr(), d_y=y.data_ptr(), d_z=z.data_ptr(), d_s=s.data_ptr(),
                              d_exit=ex.data_ptr(), d_gx=g[0].data_ptr(), d_gy=g[1].data_ptr(), d_gz=g[2].data_ptr(),
                              d_dc=d["c"].data_ptr(), d_dh=d["h"].data_ptr(), d_db=d["b"].data_ptr(),
                              d_dG=d["G"].data_ptr(), d_dA=d["A"].data_ptr(), d_status=st.data_ptr())

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
    ms_bwd = timed(backward)
    exits, status = ex.cpu().numpy(), st.cpu().numpy()
    result = {"workload": f"MPC02 x{B}, h*(1+-0.2%) b*(1+-2%), seed 1234, device-resident", "gpu": gpu,
              "steps": args.steps, "warmup": args.warmup,
              "ms_forward": ms_fwd, "ms_backward": ms_bwd, "backward_over_forward": ms_bwd / ms_fwd,
              "optimal": int(((exits == 0) | (exits == 10)).sum()), "status_0": int((status == 0).sum()),
              "status_histogram": {str(int(k)): int(v) for k, v in zip(*np.unique(status, return_counts=True))},
              "gradients_finite": bool(all(torch.isfinite(v).all() for v in d.values())),
              "gpu_after": gpu_info()}
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
