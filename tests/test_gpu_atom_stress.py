"""GPU tests of per-atom stress / energy / contact counts (sh_get_atom_stress, ShGpu.get_atom_stress) and of the shlmp
computes and dump custom columns built on it.

The numpy reference (test_atom_stress_cpu.py, checked there against the oracle's virial) is fed with the library's own
pair records (sh_get_pairs) and with the oracle's.  Shapes include the off-centre egg, on which the centre-to-centre
halves (mode 0) and the contact branch vectors (mode 1) differ per atom.  Each test prints its worst error ("worst ...").
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_py as O
import shpkg
from test_atom_stress_cpu import atom_stress_reference
from test_shape_frame_cpu import egg_shape

pkg = shpkg.load()
W = pkg.workloads
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu
PIPELINES = [0, 1, 4, 16]


def report(name, err, tol):
    print("worst %-40s %.2e  (tolerance %.0e)" % (name, err, tol))


def shapes_cfg(dissip, ncell=(4, 4, 4), seed=21):
    cfg = W.packing(ncell, 20, (32, 64), nshapes=3, seed=seed, periodic=True, name="as", skin=0.05, vel_sigma=0.5,
                    dt=4e-4, nn_frac=1.75)
    cfg["shapes"] = [egg_shape(20), W.perturbed_shape(20, 3), W.ellipsoid_shape(20)]
    cfg["shape_id"] = (np.arange(len(cfg["x"])) % 3).astype(np.int32)
    if dissip:
        cfg["dissipation"] = (3.0, 2.0, 0.4)
        cfg["angmom"] = np.random.default_rng(5).normal(0, 0.5, size=cfg["angmom"].shape)
    return cfg


def owned_by_tag(g):
    """Atoms, tags and per-atom values of the owned atoms, sorted by tag (plain or decomposed engine)."""
    nl = g.dd_info()["nlocal"] if g.dd else g.n
    tag = g.get_tags()[:nl]
    o = np.argsort(tag)
    at = {k: v[:nl][o] for k, v in g.get_atoms().items()}
    s = {m: {k: v[o] for k, v in g.get_atom_stress(m).items()} for m in (0, 1)}
    return tag[o], at, s


def kinetic_reference(g, cfg, v):
    m = np.array([cfg["density"] * g.shape_props(s)["volume"] for s in range(len(cfg["shapes"]))])[cfg["shape_id"]]
    return m[:, None, None] * v[:, :, None] * v[:, None, :]


_oracle_pairs = {}


def oracle_state(cfg, dissip):
    if dissip not in _oracle_pairs:
        o = O.Oracle(threads=8)
        W.apply(o, cfg)
        o.compute_forces()
        _oracle_pairs[dissip] = (o.get_pairs(), o.get_atoms())
        o.close()
    return _oracle_pairs[dissip]


@pytest.mark.parametrize("dissip", [False, True])
@pytest.mark.parametrize("variant", PIPELINES)
def test_per_atom_values_vs_reference(variant, dissip):
    cfg = shapes_cfg(dissip)
    k, ex = cfg["coeff"]
    g = pkg.ShGpu(); W.apply(g, cfg); g.set_pair_tuning(0, 0, variant)
    g.compute_forces()
    # oracle pairs on the same state: mode 0 (the centroid of a grazing contact is ill-conditioned, DESIGN §6)
    po, ao = oracle_state(cfg, dissip)
    tags = np.arange(1, len(cfg["x"]) + 1)
    v0 = g.get_atom_stress(0)["virial"]
    ro = atom_stress_reference(po, ao["x"], tags, cfg["box"], 0)[0]
    e = np.abs(v0 - ro).max() / np.abs(ro).max()
    report("oracle pairs mode 0 (pipeline %d, dissip %d)" % (variant, dissip), e, 1e-9)
    assert e <= 1e-9
    # the library's own pairs, after a few steps
    g.run(20)
    at, pr = g.get_atoms(), g.get_pairs()
    assert (pr["V"] > 0).sum() >= 100
    E = k * pr["V"] ** ex
    out = {}
    for mode in (0, 1):
        s = g.get_atom_stress(mode)
        vir, en, cnt = atom_stress_reference(pr, at["x"], tags, cfg["box"], mode, E=E)
        sc = np.abs(vir).max()
        ev = np.abs(s["virial"] - vir).max() / sc
        ee = np.abs(s["energy"] - en).max() / np.abs(en).max()
        report("own pairs mode %d virial (pipeline %d, dissip %d)" % (mode, variant, dissip), ev, 1e-12)
        report("own pairs mode %d energy (pipeline %d, dissip %d)" % (mode, variant, dissip), ee, 1e-12)
        assert ev <= 1e-12 and ee <= 1e-12
        assert np.array_equal(s["contacts"], cnt)
        K = kinetic_reference(g, cfg, at["v"])
        assert np.abs(s["kinetic"] - K).max() <= 1e-13 * np.abs(K).max()
        out[mode] = s["virial"]
    # on the egg the branch vectors are not the centre-to-centre halves
    assert np.abs(out[0] - out[1]).max() > 1e-3 * np.abs(out[0]).max()
    g.close()


@pytest.mark.parametrize("variant", [0, 16])
def test_sums_equal_global_stress(variant):
    cfg = shapes_cfg(True)
    g = pkg.ShGpu(); W.apply(g, cfg); g.set_pair_tuning(0, 0, variant)
    g.run(30)
    st = g.get_stress()
    for mode in (0, 1):
        s = g.get_atom_stress(mode)
        e = np.abs(s["virial"].sum(0) - st["virial"]).max() / np.linalg.norm(st["virial"])
        report("sum of virial = sh_get_stress (mode %d)" % mode, e, 1e-12)
        assert e <= 1e-12
        assert np.abs(s["kinetic"].sum(0) - st["kinetic"]).max() <= 1e-12 * np.linalg.norm(st["kinetic"])
        assert abs(s["energy"].sum() - g.get_energy()["e_contact"]) <= 1e-12 * g.get_energy()["e_contact"]
    g.close()


def wall_cfg():
    cfg = W.config2_wall(n_side=4, exponent=1.5)
    cfg["shapes"] = [egg_shape(20), W.perturbed_shape(20, 3)]
    cfg["shape_id"] = (np.arange(len(cfg["x"])) % 2).astype(np.int32)
    cfg["x"] = cfg["x"] * np.array([1, 1, 0.9]) - np.array([0, 0, 1.0])   # the bottom layer starts pressed into the wall
    k = cfg["coeff"][0]
    cfg["walls"] = [((0, 0, 0), (0, 0, 1.0), k, 1.5), ((0.6, 0, 0), (1.0, 0.15, 0.35), k, 1.5)]
    return cfg


def test_wall_energy_counts_and_walls_add_no_virial():
    cfg = wall_cfg()
    g = pkg.ShGpu(); W.apply(g, cfg)
    g.run(300)
    s = g.get_atom_stress(0)
    ec = g.get_energy()["e_contact"]
    assert (s["contacts"] > 0).sum() >= 5
    e = abs(s["energy"].sum() - ec) / ec
    report("sum of energy = e_contact with walls", e, 1e-12)
    assert e <= 1e-12
    at = g.get_atoms()
    # the same state with and without walls: identical pair phase, so the virial is bitwise equal
    res = []
    for walls in (cfg["walls"], []):
        c2 = dict(cfg, x=at["x"], v=at["v"], quat=at["quat"], angmom=at["angmom"], walls=walls)
        h = pkg.ShGpu(); W.apply(h, c2); h.compute_forces()
        res.append((h.get_atom_stress(0), h.get_atom_stress(1), h.get_energy()["e_contact"]))
        h.close()
    (a0, a1, ea), (b0, b1, eb) = res
    assert np.array_equal(a0["virial"], b0["virial"]) and np.array_equal(a1["virial"], b1["virial"])
    assert np.array_equal(a0["contacts"], b0["contacts"])
    assert ea - eb > 1e-3 * ea and (a0["energy"] > b0["energy"]).any()      # the wall energy is part of the sum
    g.close()


def dd_cfg():
    cfg = shapes_cfg(False, ncell=(6, 4, 4))
    cfg["skin"] = 0.03
    cfg["v"] = cfg["v"] + np.array([8.0, 1.0, 0.0])      # a drift: atoms cross the box, migration and rebuilds
    return cfg


@pytest.mark.parametrize("self_ghosts", [0, 1])
def test_bitwise_repeatable_and_trajectory_untouched(self_ghosts):
    cfg = dd_cfg()

    def engine():
        g = pkg.ShGpu()
        if self_ghosts:
            g.set_tuning("dd_self_ghosts", 1); g.dd_init(0, 1)
        W.apply(g, cfg)
        g.compute_forces()
        return g

    a, b = engine(), engine()
    for mode in (0, 1):
        s1, s2 = a.get_atom_stress(mode), a.get_atom_stress(mode)
        for key in s1:
            assert np.array_equal(s1[key], s2[key]), key
    for _ in range(20):       # the same 10-step runs, with and without a call after each
        a.run(10)
        a.get_atom_stress(1)
        b.run(10)
    ra, rb = a.get_atoms(), b.get_atoms()
    for key in ra:
        assert np.array_equal(ra[key], rb[key]), key
    if self_ghosts:
        assert a.dd_info()["border_builds"] >= 3
    a.close(); b.close()


@pytest.mark.parametrize("newton", [1, 0])
def test_self_ghost_decomposition_equals_periodic_engine(newton):
    cfg = dd_cfg()
    ref = pkg.ShGpu(); W.apply(ref, cfg); ref.set_tuning("sync_rebuild", 1)
    dd = pkg.ShGpu(); dd.set_tuning("dd_self_ghosts", 1); dd.set_tuning("newton", newton); dd.dd_init(0, 1)
    W.apply(dd, cfg)
    ref.compute_forces(); dd.compute_forces()
    assert dd.dd_info()["nghost"] > 0
    tr, _, sr = owned_by_tag(ref)
    td, _, sd = owned_by_tag(dd)
    assert np.array_equal(tr, td)
    for mode in (0, 1):
        ev = np.abs(sd[mode]["virial"] - sr[mode]["virial"]).max() / np.abs(sr[mode]["virial"]).max()
        ee = np.abs(sd[mode]["energy"] - sr[mode]["energy"]).max() / np.abs(sr[mode]["energy"]).max()
        report("self ghosts newton %d mode %d virial" % (newton, mode), ev, 1e-11)
        assert ev <= 1e-11 and ee <= 1e-12
        assert np.array_equal(sd[mode]["contacts"], sr[mode]["contacts"])
        assert np.array_equal(sd[mode]["kinetic"], sr[mode]["kinetic"])
    ref.close(); dd.close()


def test_lees_edwards_shear_box():
    rate = 0.6
    cfg = W.shear_box(shapes_cfg(True, ncell=(5, 4, 4), seed=33), rate)
    cfg["v"] = cfg["v"] + np.array([0.0, 8.0, 0.0])      # atoms cross the sheared boundary
    g = pkg.ShGpu(); W.apply(g, cfg)
    nsteps = 150
    g.run(nsteps)
    tag, at, s = owned_by_tag(g)
    pr = g.get_pairs()
    lo, hi, _ = cfg["box"]
    off = rate * (hi[1] - lo[1]) * nsteps * cfg["dt"]
    d = at["x"][np.searchsorted(tag, pr["tag_i"])] - at["x"][np.searchsorted(tag, pr["tag_j"])]
    assert np.any(np.abs(d[pr["V"] > 0, 1]) > 0.5 * (hi[1] - lo[1]))    # contacts across the sheared boundary
    k, ex = cfg["coeff"]
    st = g.get_stress()
    for mode in (0, 1):
        vir, en, cnt = atom_stress_reference(pr, at["x"], tag, cfg["box"], mode, E=k * pr["V"] ** ex, shear_offset=off)
        ev = np.abs(s[mode]["virial"] - vir).max() / np.abs(vir).max()
        report("Lees-Edwards mode %d virial" % mode, ev, 1e-12)
        assert ev <= 1e-12
        assert np.abs(s[mode]["energy"] - en).max() <= 1e-12 * np.abs(en).max()
        assert np.array_equal(s[mode]["contacts"], cnt)
        assert np.abs(s[mode]["virial"].sum(0) - st["virial"]).max() <= 1e-12 * np.linalg.norm(st["virial"])
    g.close()


# ---- shlmp ------------------------------------------------------------------------------------------------------------------
SCRIPT_COMPUTES = ("compute 1 all stress/atom NULL\ncompute 2 all pe/atom\ncompute 3 all contact/atom\n"
                   "compute 4 all stress/atom NULL pair branch centroid\n")
SCRIPT_DUMP = ("dump 1 all custom 100 dump.stress id type x y z fx fy fz c_1[1] c_1[2] c_1[3] c_1[4] c_1[5] c_1[6] c_2 c_3 "
               "c_4[1] c_4[4] c_4[6]\n")


def stress_script():
    txt = open(os.path.join(ROOT, "examples", "in.shear_box")).read()
    lines = [l for l in txt.splitlines() if not l.startswith("dump")]
    i = next(k for k, l in enumerate(lines) if l.startswith("run"))
    return "\n".join(lines[:i]) + "\n" + SCRIPT_COMPUTES + SCRIPT_DUMP + "\n".join(lines[i:]) + "\n"


def run_script(d, ngpus):
    from lammps_spherharm_b200 import build as b
    ex = os.path.join(ROOT, "examples")
    for f in os.listdir(ex):
        if not f.startswith("dump."):
            os.symlink(os.path.join(ex, f), d / f)
    (d / "in.stress").write_text(stress_script())
    res = subprocess.run([b.build_host(), "-in", "in.stress", "-gpus", str(ngpus)], cwd=d, capture_output=True, text=True,
                         timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    lines = (d / "dump.stress").read_text().splitlines()
    h = max(i for i, l in enumerate(lines) if l.startswith("ITEM: ATOMS"))
    assert lines[h] == "ITEM: ATOMS " + SCRIPT_DUMP.split(None, 6)[6].strip()
    rows = np.array([[float(v) for v in l.split()] for l in lines[h + 1:]])
    return rows[np.argsort(rows[:, 0])]


def test_shlmp_computes_match_capi(tmp_path):
    rows = run_script(tmp_path, 1)
    cfg = W.shear_box(W.packing((5, 4, 4), 20, (32, 64), nshapes=1, seed=33, periodic=True, vel_sigma=0.3), 0.6)
    cfg["skin"], cfg["dt"] = 0.04, 4e-4
    g = pkg.ShGpu(); W.apply(g, cfg); g.run(300)
    tag, at, s = owned_by_tag(g)
    assert len(rows) == len(tag) == 320 and np.array_equal(rows[:, 0], tag)
    comp = [(0, 0), (1, 1), (2, 2), (0, 1), (0, 2), (1, 2)]
    s1 = -np.stack([s[0]["kinetic"][:, a, b] + s[0]["virial"][:, a, b] for a, b in comp], axis=1)
    s4 = -np.stack([s[1]["virial"][:, a, b] for a, b in (comp[0], comp[3], comp[5])], axis=1)
    for name, got, want in (("f", rows[:, 5:8], at["f"]), ("c_1", rows[:, 8:14], s1), ("c_2", rows[:, 14], s[0]["energy"]),
                            ("c_4", rows[:, 16:19], s4)):
        e = np.abs(got - want).max() / np.abs(want).max()
        report("shlmp %s vs ctypes" % name, e, 1e-9)
        assert e <= 1e-9, name
    assert np.array_equal(rows[:, 15].astype(np.int64), s[0]["contacts"])
    assert (s[0]["contacts"] > 0).sum() > 10
    g.close()


def test_shlmp_two_gpus_computes_match_one_gpu(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    a = tmp_path / "g1"; a.mkdir()
    b = tmp_path / "g2"; b.mkdir()
    r1, r2 = run_script(a, 1), run_script(b, 2)
    assert r1.shape == r2.shape
    for lo, hi in ((2, 5), (5, 8), (8, 14), (14, 15), (16, 19)):
        assert np.abs(r1[:, lo:hi] - r2[:, lo:hi]).max() <= 1e-8 * np.abs(r1[:, lo:hi]).max(), (lo, hi)
    assert np.array_equal(r1[:, 15], r2[:, 15])


WORKER = r'''
import os, sys
import numpy as np
import torch, torch.distributed as dist
ROOT = sys.argv[1]; out = sys.argv[2]
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import shpkg
from test_gpu_atom_stress import dd_cfg
pkg = shpkg.load(); D = pkg.load_decomp()
local = int(os.environ["LOCAL_RANK"]); torch.cuda.set_device(local)
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
cfg = dd_cfg()
sim = D.native_engine(pkg, cfg, local)
sim.compute_forces()
nl = sim.dd_info()["nlocal"]
mine = {"tag": sim.get_tags()[:nl]}
for m in (0, 1):
    for k, v in sim.get_atom_stress(m).items():
        mine["%s%d" % (k, m)] = v
parts = [None] * world
dist.all_gather_object(parts, mine)
if rank == 0:
    tag = np.concatenate([p["tag"] for p in parts]); o = np.argsort(tag)
    got = {k: np.concatenate([p[k] for p in parts])[o] for k in mine}
    g = pkg.ShGpu(device=local); pkg.workloads.apply(g, cfg); g.compute_forces()
    assert np.array_equal(got["tag"], np.arange(1, len(cfg["x"]) + 1))
    for m in (0, 1):
        r = g.get_atom_stress(m)
        assert np.abs(got["virial%d" % m] - r["virial"]).max() <= 1e-11 * np.abs(r["virial"]).max(), m
        assert np.abs(got["energy%d" % m] - r["energy"]).max() <= 1e-12 * np.abs(r["energy"]).max(), m
        assert np.array_equal(got["contacts%d" % m], r["contacts"]), m
        assert np.array_equal(got["kinetic%d" % m], r["kinetic"]), m
    g.close()
    open(out, "w").write("ok")
sim.close()
dist.destroy_process_group()
'''


def test_two_gpu_native_decomposition_matches_one_gpu(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    w = tmp_path / "worker.py"
    w.write_text(WORKER)
    out = tmp_path / "ok.txt"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29653", str(w), ROOT, str(out)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert out.read_text() == "ok"
