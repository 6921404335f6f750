"""GPU tests of the curved container walls (sh_add_cylinder_wall, sh_add_sphere_wall; curved_wall_kernel) against the
numpy node-table reference and closed forms of test_curved_walls_cpu.py, central differences of the contact energy, the
CPU oracle (single atoms and a silo trajectory), the plane walls and pair forces they add to, the self-ghost
decomposition, the per-atom energies and the shlmp front-end.  Each test prints its worst error next to its tolerance.
"""
import os

import numpy as np
import pytest

import oracle_py as O
import shpkg
from test_curved_walls_cpu import (CONTAINERS, CURVED_SHAPES, CurvedOracle, container_atoms, container_errors, curved_sum,
                                   oracle_tables, perpendicular, place_in_container)
from test_gpu_shlmp import read_last_dump, run_shlmp
from test_gpu_walls_integrator import PIPELINES, build, fd_check, report, tables, wall_pair_cfg, wall_sum
from test_shape_frame_cpu import SHAPES

pkg = shpkg.load()
W = pkg.workloads
pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def add_curved(sim, wall, k, m):
    if wall[0] == "cylinder":
        sim.add_cylinder_wall(wall[1], wall[2], wall[3], k, m)
    else:
        sim.add_sphere_wall(wall[1], wall[2], k, m)


# ==== 1: kernel against the numpy reference and the oracle =============================================================
@pytest.mark.parametrize("container", sorted(CONTAINERS))
@pytest.mark.parametrize("exponent", [1.0, 1.5, 2.0])
def test_curved_wall_single_atoms_vs_reference(exponent, container):
    """Egg, perturbed, ellipsoid and sphere at three depths (grazing, medium, SH origin past the wall) in random poses,
    plus one atom far from the wall: f and torque to 1e-12 |F|, e_contact to 1e-12, the oracle to 1e-10."""
    grid, wall = (48, 96), CONTAINERS[container]
    rng = np.random.default_rng(int(exponent * 10) + 100 * sorted(CONTAINERS).index(container))
    shapes = [SHAPES[s]() for s in CURVED_SHAPES]
    s0 = O.Oracle()
    tab = oracle_tables(s0, grid, shapes)
    s0.close()
    x, q, sid = container_atoms(tab, wall, rng)
    if wall[-1] < 3:
        x, q, sid = x[:3], q[:3], sid[:3]
    far = np.asarray(wall[1], float) - (6.0 * np.asarray(wall[2], float) / np.linalg.norm(wall[2]) if wall[0] == "cylinder" else 0.0)
    x, q, sid = np.vstack([x, far]), np.vstack([q, W.random_quaternions(rng, 1)]), np.append(sid, 0)
    g, o = pkg.ShGpu(), CurvedOracle(threads=8)
    for s in (g, o):
        build(s, shapes, grid, x, q, shape_id=sid, k=0.0)
        add_curved(s, wall, 80.0, exponent)
        s.compute_forces()
    fr, tr, Er, nt = curved_sum(tab, x, q, sid, [wall + (80.0, exponent)])
    ag, ao = g.get_atoms(), o.get_atoms()
    assert nt[-1] == 0 and nt.sum() >= len(x) - 1 - len(shapes)
    assert np.all(ag["f"][nt == 0] == 0) and np.all(ag["torque"][nt == 0] == 0)
    fs = np.maximum(np.linalg.norm(fr, axis=1), 1e-300)[:, None]
    on = nt > 0
    ef = np.max(np.abs(ag["f"] - fr)[on] / fs[on])
    et = np.max(np.abs(ag["torque"] - tr)[on] / fs[on])
    eE = abs(g.get_energy()["e_contact"] - Er) / Er
    eo = max(np.max(np.abs(ag["f"] - ao["f"])[on] / fs[on]), np.max(np.abs(ag["torque"] - ao["torque"])[on] / fs[on]))
    report("1 curved f / |F| m=%g %s" % (exponent, container), ef, 1e-12)
    report("1 curved torque / |F| m=%g %s" % (exponent, container), et, 1e-12)
    report("1 curved e_contact m=%g %s" % (exponent, container), eE, 1e-12)
    report("1 curved vs oracle m=%g %s" % (exponent, container), eo, 1e-10)
    assert ef <= 1e-12 and et <= 1e-12 and eE <= 1e-12 and eo <= 1e-10
    g.close(); o.close()


# ==== 2: closed forms on the device ===================================================================================
def device_evaluate(grid, tab, x, q, wall, k):
    g = pkg.ShGpu()
    build(g, [(0, *W.sphere_shape(0, 1.0))], grid, x, q, k=0.0)
    add_curved(g, wall, k, 1.0)
    g.compute_forces()
    a, e = g.get_atoms(), g.get_atom_stress()["energy"]
    g.close()
    return a["f"], a["torque"], e


@pytest.mark.parametrize("wall_kind", ["sphere", "cylinder"])
def test_curved_wall_closed_forms_on_device(wall_kind):
    e48 = container_errors((48, 96), wall_kind, device_evaluate)
    e80 = container_errors((80, 160), wall_kind, device_evaluate)
    for key in ("V", "F"):
        report("2 %s %s 48x96 -> 80x160" % (wall_kind, key), e80[key], e48[key])
        assert e80[key] < e48[key] and e48[key] < 0.03, (key, e48[key], e80[key])
    for e in (e48, e80):
        assert e["tau"] <= 1e-12, e


# ==== 3: forces and torques are minus the energy gradient ==============================================================
@pytest.mark.parametrize("exponent", [1.0, 1.5])
@pytest.mark.parametrize("container", ["tilted_cylinder", "sphere"])
def test_curved_wall_forces_are_minus_energy_gradient(container, exponent):
    grid, wall = (64, 128), CONTAINERS[container]
    rng = np.random.default_rng(int(exponent * 4) + len(container))
    shapes = [SHAPES["egg20"]()]
    worst = 0.0
    for trial in range(3):
        q = W.random_quaternions(rng, 1)
        g = pkg.ShGpu()
        build(g, shapes, grid, np.zeros((1, 3)), q, k=0.0)
        props, p, n = tables(g, 0, grid)
        d = rng.normal(size=3)
        if wall[0] == "cylinder":
            u = np.asarray(wall[2], float) / np.linalg.norm(wall[2])
            d -= (d @ u) * u
        d /= np.linalg.norm(d)
        x = place_in_container(p, props, q[0], wall, d, 1.0, "medium")[None, :]
        add_curved(g, wall, 200.0, exponent)
        w, fmin = fd_check(g, x, q, [0])
        assert fmin > 1.0, "no contact"
        worst = max(worst, w)
        g.close()
    report("3 -grad E egg-%s m=%g" % (container, exponent), worst, 0.08)
    assert worst <= 0.08


# ==== 4, 8: curved walls, plane walls and pairs together; per-atom energies ===========================================
def mixed_cfg():
    cfg = wall_pair_cfg()
    x = cfg["x"]
    mid = 0.5 * (x.min(0) + x.max(0))
    rad = np.hypot(x[:, 0] - mid[0], x[:, 1] - mid[1]).max()
    cfg["curved_walls"] = [("cylinder", (mid[0], mid[1], 0.0), (0, 0, 2.0), rad + 0.3, 500.0, 1.5),
                           ("sphere", mid, np.linalg.norm(x - mid, axis=1).max() + 0.45, 300.0, 1.0)]
    return cfg


def curved_of(cfg):
    return [(w[0], np.asarray(w[1], float)) + tuple(w[2:]) for w in cfg["curved_walls"]]


@pytest.mark.parametrize("variant", PIPELINES)
def test_curved_and_plane_walls_add_to_pair_forces(variant):
    """Per-atom force = its pair forces (get_pairs) + the plane walls' reference + the curved walls' reference."""
    cfg = mixed_cfg()
    g = pkg.ShGpu(); W.apply(g, cfg); g.set_pair_tuning(0, 0, variant); g.compute_forces()
    pr, a = g.get_pairs(), g.get_atoms()
    assert (pr["V"] > 0).sum() >= 10
    n = len(cfg["x"])
    fsum, tsum = np.zeros((n, 3)), np.zeros((n, 3))
    for k in range(len(pr["V"])):
        i, j = int(pr["tag_i"][k]) - 1, int(pr["tag_j"][k]) - 1
        fsum[i] += pr["F"][k]; fsum[j] -= pr["F"][k]
        tsum[i] += pr["tau_i"][k]; tsum[j] += pr["tau_j"][k]
    tab = [tables(g, s, cfg["grid"]) for s in range(2)]
    walls = [(np.asarray(p, float), nrm, k, m) for (p, nrm, k, m) in cfg["walls"]]
    fp, tp, Ep, ntp = wall_sum(tab, cfg["x"], cfg["quat"], cfg["shape_id"], walls)
    fc, tc, Ec, ntc = curved_sum(tab, cfg["x"], cfg["quat"], cfg["shape_id"], curved_of(cfg))
    assert (ntc > 0).sum() >= 4 and ((ntc > 0) & (ntp > 0)).sum() >= 1, (ntc, ntp)
    fs = np.abs(a["f"]).max()
    err = max(np.abs(a["f"] - fsum - fp - fc).max(), np.abs(a["torque"] - tsum - tp - tc).max()) / fs
    report("4 curved + plane + pairs (pipeline %d)" % variant, err, 1e-12)
    assert err <= 1e-12
    g.close()


def test_atom_stress_energies_sum_to_e_contact_with_curved_walls():
    cfg = mixed_cfg()
    g = pkg.ShGpu(); W.apply(g, cfg); g.compute_forces()
    e = g.get_atom_stress()["energy"]
    ec = g.get_energy()["e_contact"]
    tab = [tables(g, s, cfg["grid"]) for s in range(2)]
    walls = [(np.asarray(p, float), nrm, k, m) for (p, nrm, k, m) in cfg["walls"]]
    _, _, Ep, _ = wall_sum(tab, cfg["x"], cfg["quat"], cfg["shape_id"], walls)
    _, _, Ec, ntc = curved_sum(tab, cfg["x"], cfg["quat"], cfg["shape_id"], curved_of(cfg))
    assert Ec > 0 and (ntc > 0).sum() >= 4
    report("8 sum pe/atom vs e_contact", abs(e.sum() - ec) / ec, 1e-12)
    assert abs(e.sum() - ec) <= 1e-12 * ec
    # the same state without walls: e_contact differs by the walls' reference energy, the virial not at all
    g2 = pkg.ShGpu(); W.apply(g2, dict(cfg, walls=[], curved_walls=[])); g2.compute_forces()
    e2 = g2.get_energy()["e_contact"]
    report("8 e_contact - pair energy vs wall reference", abs(ec - e2 - Ep - Ec) / ec, 1e-12)
    assert abs(ec - e2 - Ep - Ec) <= 1e-12 * ec
    assert np.array_equal(g.get_stress()["virial"], g2.get_stress()["virial"])
    g.close(); g2.close()


# ==== 5: eight curved walls =============================================================================================
def test_eight_curved_walls_accepted_ninth_refused():
    grid = (48, 96)
    shapes = [SHAPES["egg20"]()]
    q = W.random_quaternions(np.random.default_rng(8), 1)
    x = np.array([[0.2, -0.1, 0.3]])
    k = np.arange(8) + 0.5
    th, ph = np.arccos(1 - 2 * k / 8), np.pi * (1 + 5 ** 0.5) * k
    dirs = np.stack([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th)], 1)
    walls = []
    for i, d in enumerate(dirs):     # containers shifted by 0.3 along d: each cuts the egg on the far side
        if i % 2:
            walls.append(("sphere", x[0] - 0.3 * d, 0.95, 50.0 + i, 1.0 + 0.1 * i))
        else:
            walls.append(("cylinder", x[0] - 0.3 * d, perpendicular(d) * (1.0 + 0.2 * i), 0.9, 50.0 + i, 1.0 + 0.1 * i))
    g = pkg.ShGpu()
    build(g, shapes, grid, x, q, k=0.0)
    for w in walls:
        add_curved(g, w[:-2], w[-2], w[-1])
    g.compute_forces()
    tab = [tables(g, 0, grid)]
    fr, tr, Er, nt = curved_sum(tab, x, q, [0], walls)
    a = g.get_atoms()
    sc = max(np.linalg.norm(fr[0]), np.linalg.norm(tr[0]), 1.0)
    err = max(np.abs(a["f"][0] - fr[0]).max(), np.abs(a["torque"][0] - tr[0]).max()) / sc
    report("5 eight curved walls", err, 1e-12)
    assert err <= 1e-12 and abs(g.get_energy()["e_contact"] - Er) <= 1e-12 * Er
    assert nt[0] == 8, nt                       # every wall slot contributes
    with pytest.raises(pkg.ShGpuError, match="too many curved walls"):
        g.add_sphere_wall((0, 0, 0), 5.0, 1.0, 1.0)
    for bad in (lambda: g.add_cylinder_wall((0, 0, 0), (0, 0, 0), 5.0, 1.0, 1.0),
                lambda: g.add_cylinder_wall((0, 0, 0), (0, 0, 1), 0.0, 1.0, 1.0),
                lambda: g.add_sphere_wall((0, 0, 0), -1.0, 1.0, 1.0),
                lambda: g.add_sphere_wall((0, 0, 0), 1.0, -1.0, 1.0),
                lambda: g.add_sphere_wall((0, 0, 0), 1.0, 1.0, 0.9)):
        with pytest.raises(pkg.ShGpuError):
            bad()
    g.close()


# ==== 6: silo trajectory against the oracle ============================================================================
def silo_cfg():
    cfg = W.config_silo(n_layers=4, radius=6.0, exponent=1.5)
    cfg["x"] = cfg["x"] * np.array([1, 1, 0.9]) - np.array([0, 0, 0.7])
    k = cfg["coeff"][0]
    cfg["curved_walls"] = [("cylinder", (0, 0, 0), (0, 0, 1), 5.45, k, 1.5)]
    return cfg


@pytest.mark.parametrize("variant", PIPELINES)
def test_silo_trajectory_vs_oracle(variant):
    cfg = silo_cfg()
    g = pkg.ShGpu(); W.apply(g, cfg); g.set_pair_tuning(0, 0, variant); g.set_damping(0.5, 0.2)
    o = CurvedOracle(threads=8); W.apply(o, cfg); o.set_damping(0.5, 0.2)
    g.compute_forces()
    tab = [tables(g, 0, cfg["grid"])]
    _, _, _, ntc = curved_sum(tab, cfg["x"], cfg["quat"], cfg["shape_id"], curved_of(cfg))
    assert (ntc > 0).sum() >= 4, ntc                # the cylinder acts from the start
    g.run(500); o.run(500)
    ag, ao = g.get_atoms(), o.get_atoms()
    assert (o.get_pairs()["V"] > 0).sum() >= 5
    worst = 0.0
    for k, tol in (("x", 1e-9), ("v", 1e-8), ("quat", 1e-9), ("angmom", 1e-8)):
        e = np.abs(ag[k] - ao[k]).max() / max(1.0, np.abs(ao[k]).max())
        worst = max(worst, e / tol)
        assert e <= tol, (k, e)
    eg, eo = g.get_energy()["e_contact"], o.get_energy()["e_contact"]
    assert eo > 0 and abs(eg - eo) <= 1e-8 * eo
    report("6 silo trajectory (pipeline %d) err/tol" % variant, worst, 1.0)
    g.close(); o.close()


# ==== 7: z-cylinder with the in-library decomposition, periodic z =======================================================
@pytest.mark.parametrize("newton", [1, 0])
def test_zcylinder_with_self_ghost_decomposition(newton):
    cfg = W.packing((4, 4, 3), 20, (32, 64), nshapes=4, seed=21, periodic=True, name="ddc", skin=0.03, vel_sigma=0.5, dt=4e-4)
    cfg["v"] = cfg["v"] + np.array([0.0, 1.0, 8.0])
    cfg["box"] = (cfg["box"][0], cfg["box"][1], (0, 0, 1))
    x = cfg["x"]
    mid = 0.5 * (x.min(0) + x.max(0))
    rad = np.hypot(x[:, 0] - mid[0], x[:, 1] - mid[1]).max()
    cfg["curved_walls"] = [("cylinder", (mid[0], mid[1], 0.0), (0, 0, 1.0), rad + 0.25, 2e3, 1.0)]
    ref = pkg.ShGpu(); W.apply(ref, cfg); ref.set_tuning("sync_rebuild", 1)
    dd = pkg.ShGpu(); dd.set_tuning("dd_self_ghosts", 1); dd.set_tuning("newton", newton); dd.dd_init(0, 1)
    W.apply(dd, cfg)
    ref.compute_forces(); dd.compute_forces()
    r0 = ref.get_atoms()
    info = dd.dd_info()
    nl = info["nlocal"]
    order = np.argsort(dd.get_tags()[:nl])
    d0 = {k: v[:nl][order] for k, v in dd.get_atoms().items()}
    assert nl == len(cfg["x"]) and info["nghost"] > 0
    fs = np.abs(r0["f"]).max()
    tab = [tables(ref, s, cfg["grid"]) for s in range(4)]
    _, _, _, ntc = curved_sum(tab, cfg["x"], cfg["quat"], cfg["shape_id"], curved_of(cfg))
    assert (ntc > 0).sum() >= 4, ntc             # the cylinder pushes (ghosts must never receive its force)
    ef = max(np.abs(d0["f"] - r0["f"]).max(), np.abs(d0["torque"] - r0["torque"]).max()) / fs
    report("7 forces, newton %d" % newton, ef, 1e-11)
    assert ef <= 1e-11
    ref.run(200); dd.run(200)
    r1 = ref.get_atoms()
    info = dd.dd_info()
    nl = info["nlocal"]
    order = np.argsort(dd.get_tags()[:nl])
    d1 = {k: v[:nl][order] for k, v in dd.get_atoms().items()}
    L = np.asarray(cfg["box"][1]) - np.asarray(cfg["box"][0])
    dx = d1["x"] - r1["x"]; dx[:, 2] -= L[2] * np.rint(dx[:, 2] / L[2])
    report("7 trajectory x, newton %d" % newton, np.abs(dx).max(), 1e-9)
    assert np.abs(dx).max() <= 1e-9
    for k, tol in (("v", 1e-8), ("quat", 1e-9), ("angmom", 1e-8)):
        assert np.abs(d1[k] - r1[k]).max() <= tol * max(1.0, np.abs(r1[k]).max()), k
    assert info["border_builds"] >= 2, info
    ref.close(); dd.close()


# ==== 9: shlmp in.silo ================================================================================================
def test_silo_script_matches_capi(tmp_path):
    out = run_shlmp("in.silo", tmp_path)
    assert "Loop time" in out
    rows = read_last_dump(tmp_path / "dump.silo")
    assert len(rows) == 256
    assert np.hypot(rows[:, 2], rows[:, 3]).max() < 6.0 and rows[:, 4].min() > 0.0     # nobody left the silo
    cfg = W.config_silo()
    cfg["box"] = (np.array([-7.0, -7.0, 0.0]), np.array([7.0, 7.0, cfg["x"][:, 2].max() + 3.0]), (0, 0, 0))
    g = pkg.ShGpu(); W.apply(g, cfg); g.set_damping(0.5, 0.5); g.run(5000)
    at = g.get_atoms()
    assert np.abs(at["x"][:, 2] - cfg["x"][:, 2]).max() > 1.0                       # the particles did fall
    assert np.abs(rows[:, 2:5] - at["x"]).max() < 1e-9
    assert np.abs(rows[:, 5:9] - at["quat"]).max() < 1e-9
    assert np.abs(rows[:, 9:12] - at["v"]).max() < 1e-8
    g.close()


def test_silo_script_two_gpus_reproduces_one_gpu(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    script = open(os.path.join(ROOT, "examples", "in.silo")).read()
    dumps = []
    for ng in (1, 2):
        d = tmp_path / ("silo_%d" % ng); d.mkdir()
        (d / "in.case").write_text(script)
        out = run_shlmp("in.case", d, extra=("-gpus", str(ng)))
        assert ("on %d GPU" % ng) in out
        dumps.append(read_last_dump(d / "dump.silo"))
    a, b = dumps
    assert a.shape == b.shape == (256, a.shape[1])
    assert np.abs(a[:, 2:5] - b[:, 2:5]).max() < 1e-9
    assert np.abs(a[:, 5:9] - b[:, 5:9]).max() < 1e-9
    assert np.abs(a[:, 9:12] - b[:, 9:12]).max() < 1e-8
