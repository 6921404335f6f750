"""CPU tests of per-atom stress / energy / contact counts (sh_get_atom_stress; shlmp compute stress/atom, pe/atom,
contact/atom and dump custom columns).

- shlmp -check accepts the compute and dump custom syntax and rejects malformed forms with LAMMPS-style messages.
- The numpy per-atom reference that tests/test_gpu_atom_stress.py compares the library against is checked on the CPU
  oracle: built from per-pair records alone, summed over atoms it must give orc_get_stress's virial in both modes
  (centre-to-centre halves and contact branch vectors), with the minimum image and with the Lees-Edwards image.
"""
import os
import subprocess

import numpy as np
import pytest

import oracle_py as O
import shpkg

pkg = shpkg.load()
W = pkg.workloads
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EX = os.path.join(ROOT, "examples")


# ---- numpy reference ---------------------------------------------------------------------------------------------------
def separation(xi, xj, box, shear_offset=None):
    """x_i - x_j with the periodic minimum image; with shear_offset (rate * Ly * t) the Lees-Edwards image: the cell n_y
    boxes up is displaced by n_y * offset along x."""
    lo, hi, per = box
    L = np.asarray(hi, float) - np.asarray(lo, float)
    d = np.array(xi, float) - np.asarray(xj, float)
    if shear_offset is not None:
        ny = np.rint(d[:, 1] / L[1])
        d[:, 1] -= ny * L[1]
        d[:, 0] -= ny * shear_offset
        d[:, 0] -= L[0] * np.rint(d[:, 0] / L[0])
        if per[2]:
            d[:, 2] -= L[2] * np.rint(d[:, 2] / L[2])
        return d
    for k in range(3):
        if per[k]:
            d[:, k] -= L[k] * np.rint(d[:, k] / L[k])
    return d


def atom_stress_reference(pairs, x, tags, box, mode, E=None, shear_offset=None):
    """Per-atom virial (n,3,3), energy (n,) and contact count (n,) of the atoms `tags` (positions x) from per-pair records
    (get_pairs: tag_i, tag_j, V, F = force on i, centroid in the frame of i).  Only pairs with V > 0 count.
    mode 0: each atom gets 1/2 (x_i - x_j) (x) F; mode 1: atom a gets (x_a - x_c) (x) F_a.  E: per-pair energies."""
    idx = {int(t): k for k, t in enumerate(tags)}
    m = pairs["V"] > 0
    i = np.array([idx[int(t)] for t in pairs["tag_i"][m]], dtype=np.int64)
    j = np.array([idx[int(t)] for t in pairs["tag_j"][m]], dtype=np.int64)
    F, xc = pairs["F"][m], pairs["centroid"][m]
    d = separation(x[i], x[j], box, shear_offset)
    if mode == 0:
        Wi = Wj = 0.5 * d[:, :, None] * F[:, None, :]
    else:
        Wi = (x[i] - xc)[:, :, None] * F[:, None, :]
        Wj = (x[i] - d - xc)[:, :, None] * (-F)[:, None, :]
    n = len(tags)
    vir = np.zeros((n, 3, 3))
    np.add.at(vir, i, Wi)
    np.add.at(vir, j, Wj)
    en = np.zeros(n)
    if E is not None:
        np.add.at(en, i, 0.5 * E[m])
        np.add.at(en, j, 0.5 * E[m])
    cnt = np.zeros(n, dtype=np.int64)
    np.add.at(cnt, i, 1)
    np.add.at(cnt, j, 1)
    return vir, en, cnt


def dense_cfg(seed=21, nshapes=3, shapes=None):
    cfg = W.packing((4, 4, 4), 12, (16, 32), nshapes=nshapes, seed=seed, periodic=True, name="as", skin=0.05,
                    vel_sigma=0.5, dt=4e-4, nn_frac=1.75)
    if shapes is not None:
        cfg["shapes"] = shapes
        cfg["shape_id"] = (np.arange(len(cfg["x"])) % len(shapes)).astype(np.int32)
    return cfg


@pytest.mark.parametrize("shear", [0.0, 0.6])
def test_reference_sums_to_oracle_virial(shear):
    cfg = dense_cfg()
    cfg["dissipation"] = (3.0, 2.0, 0.4)
    if shear:
        cfg = W.shear_box(cfg, shear)
        cfg["v"] = cfg["v"] + np.array([0.0, 8.0, 0.0])     # atoms cross the sheared boundary
    o = O.Oracle(threads=8)
    W.apply(o, cfg)
    nsteps = 30 if shear else 5
    o.run(nsteps)
    at, pr = o.get_atoms(), o.get_pairs()
    assert (pr["V"] > 0).sum() >= 50
    off = shear * (cfg["box"][1][1] - cfg["box"][0][1]) * nsteps * cfg["dt"] if shear else None
    if shear:   # the oracle never wraps: some pairs must straddle the sheared boundary for the image to matter
        d = at["x"][pr["tag_i"] - 1] - at["x"][pr["tag_j"] - 1]
        assert np.any(np.abs(d[pr["V"] > 0, 1]) > 0.5 * (cfg["box"][1][1] - cfg["box"][0][1]))
    ref = o.get_stress()["virial"]
    tags = np.arange(1, len(cfg["x"]) + 1)
    for mode in (0, 1):
        vir, _, cnt = atom_stress_reference(pr, at["x"], tags, cfg["box"], mode, shear_offset=off)
        err = np.abs(vir.sum(0) - ref).max() / np.linalg.norm(ref)
        assert err <= 1e-12, (mode, err)
        assert cnt.sum() == 2 * (pr["V"] > 0).sum()
    # the two modes differ per atom (the branch vectors are not the centre-to-centre halves) but not in total
    v0 = atom_stress_reference(pr, at["x"], tags, cfg["box"], 0, shear_offset=off)[0]
    v1 = atom_stress_reference(pr, at["x"], tags, cfg["box"], 1, shear_offset=off)[0]
    assert np.abs(v0 - v1).max() > 1e-3 * np.abs(v0).max()
    o.close()


# ---- shlmp -check -------------------------------------------------------------------------------------------------------
def shlmp_check(text, extra=()):
    from lammps_spherharm_b200 import build as b
    return subprocess.run([b.build_host(), "-check"] + list(extra), input=text, cwd=EX, capture_output=True, text=True,
                          timeout=120)


HEAD = ("atom_style spherharm 20 32 64 ellipsoid_l20.sh\nregion box block -5 5 -5 5 -5 5\ncreate_box 1 box\n"
        "pair_style spherharm\npair_coeff 1 1 1000 1\ncreate_atoms 1 single 0 0 0\n")
COMPUTES = ("compute 1 all stress/atom NULL\ncompute 2 all pe/atom\ncompute 3 all contact/atom\n"
            "compute 4 all stress/atom NULL ke\ncompute 5 all stress/atom NULL pair branch centroid\n"
            "compute 6 all stress/atom NULL virial ke branch center\n")
DUMP = ("dump 1 all custom 10 dump.as id type x y z vx vy vz qw qx qy qz fx fy fz tqx tqy tqz angmomx angmomy angmomz "
        "c_1[1] c_1[2] c_1[3] c_1[4] c_1[5] c_1[6] c_2 c_3 c_4[1] c_5[6] c_6[3]\n")


@pytest.mark.parametrize("gpus", [None, "4"])
def test_check_accepts_computes_and_dump_columns(gpus):
    res = shlmp_check(HEAD + COMPUTES + DUMP + "run 20\n", extra=("-gpus", gpus) if gpus else ())
    assert res.returncode == 0, res.stderr
    assert "run 20 with 1 atoms" in res.stdout


@pytest.mark.parametrize("text,msg", [
    ("compute 1 all centro/atom\n", "Unknown compute style centro/atom"),
    ("compute 1 mobile pe/atom\n", "Could not find compute group ID mobile"),
    ("compute 1 all stress/atom\n", "Illegal compute stress/atom command"),
    ("compute 1 all stress/atom mytemp\n", "Could not find compute stress/atom temperature ID mytemp"),
    ("compute 1 all stress/atom NULL bond\n", "Illegal compute stress/atom command"),
    ("compute 1 all stress/atom NULL branch middle\n", "Illegal compute stress/atom command"),
    ("compute 1 all pe/atom\ncompute 1 all contact/atom\n", "Reuse of compute ID 1"),
    ("dump 1 all custom 10 d.out id type mass\n", "Invalid attribute mass in dump custom command"),
    ("dump 1 all custom 10 d.out id c_9\n", "Could not find dump custom compute ID: 9"),
    ("compute 1 all stress/atom NULL\ndump 1 all custom 10 d.out id c_1[7]\n", "Dump custom compute 1 vector is accessed out-of-range"),
    ("compute 1 all stress/atom NULL\ndump 1 all custom 10 d.out id c_1[0]\n", "Dump custom compute 1 vector is accessed out-of-range"),
    ("compute 1 all stress/atom NULL\ndump 1 all custom 10 d.out id c_1\n", "Dump custom compute 1 does not calculate per-atom vector"),
    ("compute 2 all pe/atom\ndump 1 all custom 10 d.out id c_2[1]\n", "Dump custom compute 2 does not calculate per-atom array"),
    ("compute 3 all contact/atom\ndump 1 all custom 10 d.out c_3[2]\n", "Dump custom compute 3 does not calculate per-atom array"),
    ("dump 1 mobile custom 10 d.out id\n", "Could not find dump group ID mobile"),
])
def test_check_rejects_malformed_computes_and_dumps(text, msg):
    res = shlmp_check(HEAD + text + "run 1\n")
    assert res.returncode == 1
    assert "ERROR: " + msg in res.stderr, res.stderr
