"""What looser tolerances buy: the bench batch (MPC02 x 65 536, bench.py's seeded h / b, device-resident) solved at
the default settings and at looser ones (tolerances 1e-6, reduced tolerances 1e-3), on one GPU.

Prints one JSON object: per settings, solves/s over the timed steps (CUDA events around whole solves), mean and
maximum iteration count, the exit-flag histogram; and the GPU's name and power limit, read in the same run.
    python tools/settings_bench.py [--batch 65536] [--steps 3] [--warmup 1] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SETTINGS = {
    "default": {},
    "loose": dict(feastol=1e-6, abstol=1e-6, reltol=1e-6, feastol_inacc=1e-3, abstol_inacc=1e-3, reltol_inacc=1e-3),
}


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
    hs = torch.from_numpy(np.ascontiguousarray(W["hs"])).to(dev)
    bs = torch.from_numpy(np.ascontiguousarray(W["bs"])).to(dev)
    x = torch.empty((B, P["n"]), dtype=torch.float64, device=dev)
    ex = torch.empty((B,), dtype=torch.int32, device=dev)
    it = torch.empty((B,), dtype=torch.int32, device=dev)
    solver = eicos_b200.BatchSolver(P, device=0, capacity=B)
    result = {"workload": f"MPC02 x{B}, h*(1+-0.2%) b*(1+-2%), seed 1234, device-resident", "gpu": gpu_info(),
              "steps": args.steps, "warmup": args.warmup, "runs": {}}
    for name, st in SETTINGS.items():
        solver.set_settings(**dict(eicos_b200.default_settings(), **st))

        def step():
            solver.solve_device(B, d_hs=hs.data_ptr(), d_bs=bs.data_ptr(), d_x=x.data_ptr(), d_exit=ex.data_ptr(),
                                d_iter=it.data_ptr())

        for _ in range(args.warmup):
            step()
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(args.steps):
            step()
        t1.record()
        torch.cuda.synchronize()
        ms = t0.elapsed_time(t1) / args.steps
        iters, exits = it.cpu().numpy(), ex.cpu().numpy()
        flags, counts = np.unique(exits, return_counts=True)
        result["runs"][name] = {"settings": solver.settings(), "ms_per_solve": ms, "solves_per_s": B / (ms * 1e-3),
                                "iter_mean": float(iters.mean()), "iter_max": int(iters.max()),
                                "exit_histogram": {str(int(f)): int(c) for f, c in zip(flags, counts)}}
    d, l = result["runs"]["default"], result["runs"]["loose"]
    result["loose_over_default"] = {"solves_per_s": l["solves_per_s"] / d["solves_per_s"],
                                    "iter_mean": l["iter_mean"] / d["iter_mean"]}
    result["gpu_after"] = gpu_info()
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
