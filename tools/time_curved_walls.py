#!/usr/bin/env python
"""Cost of the curved container walls on a silo cut from the benchmark's packing: the relaxed 128,000-particle tiling
(l_max 30, 48x96 quadrature, bench.make_workload without the bulk flow), kept inside the z-cylinder inscribed in the box,
periodic in z only (about 100k particles).

  python tools/time_curved_walls.py [--steps 1000] [--rounds 2] [--out DIR]

1. ms/step of sh_run with and without the cylinder, alternated --rounds times on two engines built from the same atoms
   (device time of sh_run).
2. Device time per call of curved_wall_kernel (torch.profiler, CUDA activities, separate traced section).
3. Device time per call of the plane wall_kernel on the uncut tiling in a box of four plane walls (x and y), periodic in z.
Atoms "in reach" are those the kernel does not cull (distance to the wall < rmax).  Prints one JSON line with the card name
and power limit; --out also writes it to DIR/time_curved_walls.json.
"""
import argparse
import json
import os
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402
import shpkg  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def kernel_us(g, torch, names, calls=20):
    """Device time per launch of each named kernel over `calls` force evaluations."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            g.compute_forces()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        for k in names:
            if ev.key.split("(")[0].split("::")[-1].strip() == k:
                t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
                out[k] = dict(us_per_call=t / max(ev.count, 1), calls=ev.count)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_curved_walls.py: no CUDA device")
    pkg = shpkg.load()
    wargs = argparse.Namespace(particles=128000, workload="relaxed", lmax=30, ntheta=48, nphi=96, flow=0.0, vel_sigma=0.02)
    full = bench.make_workload(wargs, pkg)
    lo, hi, _ = full["box"]
    lo, hi = np.asarray(lo, float), np.asarray(hi, float)
    mid, R = 0.5 * (lo + hi), 0.5 * min(hi[0] - lo[0], hi[1] - lo[1])
    rho = np.hypot(full["x"][:, 0] - mid[0], full["x"][:, 1] - mid[1])
    keep = rho < R - 0.3
    silo = dict(full)
    for key in ("shape_id", "x", "v", "quat", "angmom"):
        silo[key] = np.asarray(full[key])[keep]
    silo["box"] = (lo, hi, (0, 0, 1))
    k, m = full["coeff"]
    walled = dict(silo, curved_walls=[("cylinder", (mid[0], mid[1], 0.0), (0, 0, 1.0), R, k, m)])
    sims = {}
    for key, cfg in (("without", silo), ("with", walled)):
        g = pkg.ShGpu()
        pkg.workloads.apply(g, cfg)
        g.compute_forces()
        g.run(20)
        sims[key] = g
    rmax = np.array([sims["with"].shape_props(s)["rmax"] for s in range(len(full["shapes"]))])
    in_reach = int((rho[keep] + rmax[silo["shape_id"]] >= R).sum())
    res = {"without": [], "with": []}
    for _ in range(a.rounds):
        for key in ("without", "with"):
            g = sims[key]
            g.synchronize()
            g.run(a.steps)
            res[key].append(1e3 * g.get_run_time()["last"] / a.steps)
    curved = kernel_us(sims["with"], torch, ("curved_wall_kernel",))
    for g in sims.values():
        g.close()
    # plane walls: the uncut tiling in a box of four planes at its x and y faces, periodic in z
    box = dict(full, box=(lo, hi, (0, 0, 1)))
    box["walls"] = [(lo, (1.0, 0, 0), k, m), (hi, (-1.0, 0, 0), k, m), (lo, (0, 1.0, 0), k, m), (hi, (0, -1.0, 0), k, m)]
    x = np.asarray(full["x"])
    h = np.minimum(np.minimum(x[:, 0] - lo[0], hi[0] - x[:, 0]), np.minimum(x[:, 1] - lo[1], hi[1] - x[:, 1]))
    plane_reach = int((h < rmax[full["shape_id"]]).sum())
    g = pkg.ShGpu()
    pkg.workloads.apply(g, box)
    g.compute_forces()
    g.run(20)
    plane = kernel_us(g, torch, ("wall_kernel",))
    g.close()
    line = dict(card=card(), silo_particles=int(keep.sum()), cylinder_radius=R, atoms_in_reach_of_cylinder=in_reach,
                ms_step_without_cylinder=res["without"], ms_step_with_cylinder=res["with"], steps=a.steps,
                curved_wall_kernel=curved.get("curved_wall_kernel"),
                plane_box_particles=len(x), atoms_in_reach_of_planes=plane_reach, wall_kernel=plane.get("wall_kernel"))
    print(json.dumps(line), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "time_curved_walls.json"), "w") as f:
            json.dump(line, f, indent=1)


if __name__ == "__main__":
    main()
