#!/usr/bin/env python
"""Write the shape / data files the example input scripts in examples/ read (deterministic)."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import shpkg

W = shpkg.load().workloads


def write_shape(fn, lmax, a, b):
    with open(fn, "w") as f:
        f.write("# l m a_lm b_lm  (real orthonormal SH, no Condon-Shortley phase)\n")
        for l in range(lmax + 1):
            for m in range(l + 1):
                k = l * (l + 1) // 2 + m
                f.write("%d %d %.17g %.17g\n" % (l, m, a[k], b[k]))


def write_data(fn, cfg, box):
    n = len(cfg["x"])
    with open(fn, "w") as f:
        f.write("LAMMPS-style data file for atom_style spherharm (id type x y z qw qx qy qz)\n\n")
        f.write("%d atoms\n%d atom types\n\n" % (n, len(cfg["shapes"])))
        for d, nm in enumerate("xyz"):
            f.write("%.17g %.17g %slo %shi\n" % (box[0][d], box[1][d], nm, nm))
        f.write("\nAtoms\n\n")
        for i in range(n):
            f.write("%d %d %s %s\n" % (i + 1, cfg["shape_id"][i] + 1, " ".join("%.17g" % v for v in cfg["x"][i]),
                                     " ".join("%.17g" % v for v in cfg["quat"][i])))
        f.write("\nVelocities\n\n")
        for i in range(n):
            f.write("%d %s\n" % (i + 1, " ".join("%.17g" % v for v in cfg["v"][i])))


def main(outdir=os.path.join(ROOT, "examples")):
    os.makedirs(outdir, exist_ok=True)
    a, b = W.ellipsoid_shape(20)
    write_shape(os.path.join(outdir, "ellipsoid_l20.sh"), 20, a, b)
    cfg = W.config2_wall(10)
    lo = cfg["x"].min(0) - 3.0
    hi = cfg["x"].max(0) + 3.0
    lo[2] = 0.0
    write_data(os.path.join(outdir, "data.wall_1000"), cfg, (lo, hi))
    # BASELINE configs[3] at example size: periodic mono-shape packing sheared by Lees-Edwards images (in.shear_box)
    cfg = W.shear_box(W.packing((5, 4, 4), 20, (32, 64), nshapes=1, seed=33, periodic=True, vel_sigma=0.3), 0.6)
    write_data(os.path.join(outdir, "data.shear_320"), cfg, (cfg["box"][0], cfg["box"][1]))
    # silo filling (in.silo): particles inside a z-cylinder of radius 6 above a floor plane at z = 0
    cfg = W.config_silo()
    write_data(os.path.join(outdir, "data.silo_256"), cfg, ((-7.0, -7.0, 0.0), (7.0, 7.0, cfg["x"][:, 2].max() + 3.0)))


if __name__ == "__main__":
    main(*sys.argv[1:])
