#!/usr/bin/env python
"""Cost of sh_get_atom_stress on the benchmark's one-GPU workload (bench.make_workload at N=1: the relaxed 96,000-particle
packing, l_max 30, 48x96 quadrature).

  python tools/time_atom_stress.py [--steps 2000] [--every 100] [--rounds 2] [--out DIR]

1. ms/step of sh_run over --steps steps, without and with one sh_get_atom_stress call every --every steps, alternated
   --rounds times on two engines built from the same workload (device time of sh_run plus the host wall time of the
   whole block, which includes the calls).
2. Wall time of one call (kernels, the collective return path when decomposed, and the copy of the four outputs to the
   host), median of 20.
3. Device time of the new kernels from torch.profiler with CUDA activities, in a separate traced section.
Prints one JSON line with the card name and power limit; --out also writes it to DIR/time_atom_stress.json.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402
import shpkg  # noqa: E402

KERNELS = ("atom_stress_entry_pair_kernel", "atom_stress_row_kernel", "atom_stress_add_returned_kernel")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--every", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_atom_stress.py: no CUDA device")
    pkg = shpkg.load()
    wargs = argparse.Namespace(particles=96000, workload="relaxed", lmax=30, ntheta=48, nphi=96, flow=15.0, vel_sigma=0.02)
    cfg = bench.make_workload(wargs, pkg)
    sims = []
    for _ in range(2):
        g = pkg.ShGpu()
        pkg.workloads.apply(g, cfg)
        g.compute_forces()
        g.run(5)
        g.get_atom_stress(0)      # first call allocates
        sims.append(g)
    res = {"off": [], "on": []}
    for _ in range(a.rounds):
        for key, g in (("off", sims[0]), ("on", sims[1])):
            dev = 0.0
            g.synchronize()
            t0 = time.perf_counter()
            for _ in range(a.steps // a.every):
                g.run(a.every)
                dev += g.get_run_time()["last"]
                if key == "on":
                    g.get_atom_stress(0)
            g.synchronize()
            wall = time.perf_counter() - t0
            res[key].append(dict(ms_step_device=1e3 * dev / a.steps, ms_step_wall=1e3 * wall / a.steps))
    g = sims[1]
    npairs = len(g.get_pairs()["V"])
    calls = []
    for mode in (0, 1, 0, 1) * 5:
        g.synchronize()
        t0 = time.perf_counter()
        g.get_atom_stress(mode)
        calls.append(time.perf_counter() - t0)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for mode in (0, 1) * 5:
            g.get_atom_stress(mode)
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.key_averages():
        for k in KERNELS:
            if k in ev.key:
                t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
                kern[k] = dict(us_per_call=t / max(ev.count, 1), calls=ev.count)
    line = dict(card=card(), particles=len(cfg["x"]), pairs=npairs, steps=a.steps, every=a.every,
                off=res["off"], on=res["on"], call_wall_ms_median=1e3 * float(np.median(calls)), kernels=kern)
    print(json.dumps(line), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "time_atom_stress.json"), "w") as f:
            json.dump(line, f, indent=1)
    for s in sims:
        s.close()


if __name__ == "__main__":
    main()
