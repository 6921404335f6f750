"""GPU tests of the plane-wall kernel, gravity, viscous damping and the rigid-body step against references that do not
share the library's conventions: numpy from the node table (test_shape_frame_cpu.py), closed forms, finite differences
of the contact energy and an ODE solver.  The parity suite compares the CUDA path with the CPU oracle only, which was
written with the same operation sequence; a convention both share passes every parity test but none of these.

Shapes: the off-centre egg (|com| ~ 0.19, tilted principal axes) beside perturbed ellipsoids (l_max 20 and 30), the
axis-aligned ellipsoid and the sphere, so that the lever arm c - x and the principal-frame rotation Rp do not cancel.
Each test prints its worst observed error next to its tolerance ("worst ...").
"""
import numpy as np
import pytest
from scipy.integrate import solve_ivp

import oracle_py as O
import shpkg
from test_shape_frame_cpu import (SHAPES, axis_quat, check_frame, egg_shape, frame_reference, in_plane, place_at_depth,
                                  pose, quat_mat, quat_mul, rotation_angle, wall_reference)

pkg = shpkg.load()
W = pkg.workloads
pytestmark = pytest.mark.gpu
PIPELINES = [0, 16]


def report(name, err, tol):
    print("worst %-34s %.2e  (tolerance %.0e)" % (name, err, tol))


def build(sim, shapes, grid, x, quat, v=None, angmom=None, shape_id=None, k=1e3, exponent=1.0, dt=1e-4, skin=0.3):
    """Shapes given as (lmax, a, b); every pair of shapes gets (k, exponent)."""
    sim.set_quadrature(*grid)
    ids = [sim.add_shape(lmax, a, b, 1.0) for (lmax, a, b) in shapes]
    n = len(x)
    sim.set_atoms(np.zeros(n, np.int32) if shape_id is None else np.asarray(shape_id, np.int32), np.asarray(x, float),
                  np.zeros((n, 3)) if v is None else v, quat, np.zeros((n, 3)) if angmom is None else angmom)
    for i in ids:
        for j in ids:
            if j >= i:
                sim.pair_coeff(i, j, k, exponent)
    sim.set_neighbor(skin, 1, 1)
    sim.set_timestep(dt)
    return ids


def tables(sim, sid, grid):
    props = sim.shape_props(sid)
    p, n = sim.nodes(sid, grid[0] * grid[1])
    return props, p, n


# ==== A: the device library's shape frame ==============================================================================
@pytest.mark.parametrize("name", sorted(SHAPES))
def test_device_shape_frame_vs_divergence_theorem(name):
    lmax, a, b = SHAPES[name]()
    g = pkg.ShGpu()
    g.set_quadrature(48, 96)
    sid = g.add_shape(lmax, a, b, 1.3)
    props, p, n = tables(g, sid, (48, 96))
    check_frame(props, p, n, 1.3, np.linalg.norm(p, axis=1).max())
    g.close()


# ==== B: wall kernel against the numpy reference =======================================================================
NORMALS = {"+z": (0, 0, 1.0), "-z": (0, 0, -1.0), "tilted": (0.3, -0.5, 0.81), "tilted_len3": (-1.2, 0.9, 2.4)}
WALL_SHAPES = ("egg20", "egg30", "perturbed20", "perturbed30", "ellipsoid20", "sphere")


def wall_sum(tab, x, q, sid, walls):
    """Reference f, torque per atom and total energy over all walls; also the number of walls each atom touches."""
    n = len(x)
    f, t, nt, E = np.zeros((n, 3)), np.zeros((n, 3)), np.zeros(n, int), 0.0
    for i in range(n):
        props, p, nn = tab[sid[i]]
        for (pt, nrm, k, m) in walls:
            F, tau, e, nsub = wall_reference(p, nn, props, x[i], q[i], np.asarray(pt, float), nrm, k, m)
            f[i] += F; t[i] += tau; E += e
            nt[i] += e > 0
    return f, t, E, nt


def run_walls(sims, shapes, grid, x, q, sid, walls):
    tabs = None
    for s in sims:
        build(s, shapes, grid, x, q, shape_id=sid)
        for (pt, nrm, k, m) in walls:
            s.add_wall(pt, nrm, k, m)
        s.compute_forces()
        if tabs is None:
            tabs = [tables(s, i, grid) for i in range(len(shapes))]
    return tabs


@pytest.mark.parametrize("normal", sorted(NORMALS))
@pytest.mark.parametrize("exponent", [1.0, 1.5, 2.0])
def test_wall_single_atoms_vs_reference(exponent, normal):
    """Six shapes x three depths (grazing: 6 nodes under the plane; medium; the SH origin under the plane), random
    poses, one wall; per-atom f and torque to 1e-12 |F|, e_contact to 1e-12, and the oracle to 1e-10."""
    grid, nrm = (48, 96), NORMALS[normal]
    shapes = [SHAPES[s]() for s in WALL_SHAPES]
    rng = np.random.default_rng(int(10 * exponent) + 100 * sorted(NORMALS).index(normal))
    point = np.array([0.5, -0.3, 0.2])
    g, o = pkg.ShGpu(), O.Oracle(threads=8)
    # the node tables (and so the placement) do not depend on the atoms: take them from a scratch context
    s0 = O.Oracle()
    s0.set_quadrature(*grid)
    tab = [None] * len(shapes)
    for i, (lmax, a, b) in enumerate(shapes):
        s0.add_shape(lmax, a, b, 1.0)
        tab[i] = tables(s0, i, grid)
    s0.close()
    t1, t2 = in_plane(nrm)
    x, q, sid = [], [], []
    for i in range(len(shapes)):
        for j, depth in enumerate(("grazing", "medium", "deep")):
            qq = W.random_quaternions(rng, 1)[0]
            x.append(place_at_depth(tab[i][1], tab[i][0], qq, point + 4.0 * i * t1 + 4.0 * j * t2, nrm, depth))
            q.append(qq); sid.append(i)
    x, q, sid = np.array(x), np.array(q), np.array(sid)
    walls = [(point, nrm, 80.0, exponent)]
    run_walls((g, o), shapes, grid, x, q, sid, walls)
    fr, tr, Er, nt = wall_sum(tab, x, q, sid, walls)
    ag, ao = g.get_atoms(), o.get_atoms()
    # a grazing cap of a few nodes can have a discrete volume <= 0: then the contact is skipped, by both sides
    assert nt.sum() >= len(x) - len(shapes)
    assert np.all(ag["f"][nt == 0] == 0) and np.all(ag["torque"][nt == 0] == 0)
    fs = np.maximum(np.linalg.norm(fr, axis=1), 1e-300)[:, None]
    ef = np.max(np.abs(ag["f"] - fr) / fs)
    et = np.max(np.abs(ag["torque"] - tr) / fs)
    eE = abs(g.get_energy()["e_contact"] - Er) / Er
    eo = max(np.max(np.abs(ag["f"] - ao["f"]) / fs), np.max(np.abs(ag["torque"] - ao["torque"]) / fs))
    report("B wall f / |F| m=%g %s" % (exponent, normal), ef, 1e-12)
    report("B wall torque / |F| m=%g %s" % (exponent, normal), et, 1e-12)
    report("B wall e_contact m=%g %s" % (exponent, normal), eE, 1e-12)
    report("B wall vs oracle m=%g %s" % (exponent, normal), eo, 1e-10)
    assert ef <= 1e-12 and et <= 1e-12 and eE <= 1e-12 and eo <= 1e-10
    # the lever arm matters: (c - x) x F, the torque term that the off-centre shapes add, is far above the tolerance
    lever = [np.cross(x[i] - pose(tab[sid[i]][0], q[i], x[i])[1], fr[i]) for i in range(len(x))]
    assert np.abs(lever).max() > 0.05 * np.abs(fr).max()
    g.close(); o.close()


def test_six_wall_box_corners_and_out_of_reach_atoms():
    """216 atoms in random poses inside a box of six walls (normals pointing inwards): face atoms touch one wall, edge
    atoms two, corner atoms three; atoms out of reach get exactly zero force and torque."""
    grid = (32, 64)
    shapes = [SHAPES["egg20"](), SHAPES["perturbed20"]()]
    rng = np.random.default_rng(12)
    gx = np.arange(6) * 3.0
    x = np.stack(np.meshgrid(gx, gx, gx, indexing="ij"), -1).reshape(-1, 3) + rng.uniform(-0.15, 0.15, (216, 3))
    q = W.random_quaternions(rng, 216)
    sid = rng.integers(0, 2, 216)
    lo, hi = -0.45, 15.45
    walls = []
    for d in range(3):
        e = np.eye(3)[d]
        walls.append((lo * e, e, 300.0, 1.5))
        walls.append((hi * e, -e, 300.0, 1.5))
    g, o = pkg.ShGpu(), O.Oracle(threads=8)
    tab = run_walls((g, o), shapes, grid, x, q, sid, walls)
    fr, tr, Er, nt = wall_sum(tab, x, q, sid, walls)
    assert (nt == 3).sum() >= 4 and (nt == 2).sum() >= 12 and (nt == 0).sum() >= 64, np.bincount(nt)
    assert np.all(g.get_pairs()["V"] == 0)           # no pair contacts: the forces are the walls' only
    ag, ao = g.get_atoms(), o.get_atoms()
    out = nt == 0
    assert np.all(ag["f"][out] == 0) and np.all(ag["torque"][out] == 0)
    fs = np.linalg.norm(fr[~out], axis=1)[:, None]
    ef = max(np.max(np.abs(ag["f"][~out] - fr[~out]) / fs), np.max(np.abs(ag["torque"][~out] - tr[~out]) / fs))
    eE = abs(g.get_energy()["e_contact"] - Er) / Er
    report("B six-wall box f, torque / |F|", ef, 1e-12)
    report("B six-wall box e_contact", eE, 1e-12)
    assert ef <= 1e-12 and eE <= 1e-12
    assert np.abs(ag["f"] - ao["f"]).max() <= 1e-10 * np.abs(ao["f"]).max()
    g.close(); o.close()


def test_sixteen_walls_accepted_seventeenth_refused():
    """Sixteen tilted planes all cutting one egg: every wall slot contributes; a 17th wall is refused."""
    grid = (48, 96)
    shapes = [SHAPES["egg20"]()]
    q = W.random_quaternions(np.random.default_rng(16), 1)
    k = np.arange(16) + 0.5
    th, ph = np.arccos(1 - 2 * k / 16), np.pi * (1 + 5 ** 0.5) * k
    dirs = np.stack([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th)], 1)
    x = np.array([[0.2, -0.1, 0.3]])
    # plane with inward normal -d through the point 0.75 from x along d: cuts the egg's outer part in direction d
    walls = [(x[0] + 0.75 * d, -d * (1.0 + 0.1 * i), 50.0 + i, 1.0 + 0.07 * i) for i, d in enumerate(dirs)]
    g = pkg.ShGpu()
    tab = run_walls((g,), shapes, grid, x, q, [0], walls)
    fr, tr, Er, nt = wall_sum(tab, x, q, [0], walls)
    assert nt[0] >= 12, nt
    a = g.get_atoms()
    sc = max(np.linalg.norm(fr[0]), np.linalg.norm(tr[0]), 1.0)
    err = max(np.abs(a["f"][0] - fr[0]).max(), np.abs(a["torque"][0] - tr[0]).max()) / sc
    report("B sixteen walls", err, 1e-12)
    assert err <= 1e-12
    assert abs(g.get_energy()["e_contact"] - Er) <= 1e-12 * Er
    with pytest.raises(pkg.ShGpuError):
        g.add_wall((0, 0, 0), (0, 0, 1.0), 1.0, 1.0)
    g.close()


def wall_pair_cfg():
    cfg = W.packing((2, 2, 2), 20, (32, 64), nshapes=2, seed=5, periodic=False, nn_frac=1.75, name="wallpair")
    cfg["shapes"] = [egg_shape(20), W.perturbed_shape(20, 3)]
    x = cfg["x"]
    lo = x.min(0)
    cfg["walls"] = [((0, 0, lo[2] - 0.35), (0, 0, 1.0), 400.0, 1.5), (lo + np.array([-0.4, 0, 0]), (1.0, 0.2, 0.3), 600.0, 1.0)]
    return cfg


@pytest.mark.parametrize("variant", PIPELINES)
def test_wall_forces_add_to_pair_forces(variant):
    """With pair contacts present the per-atom force is the sum of that atom's pair forces (get_pairs) plus the walls'
    reference: the gather adds the wall slots after the pair slots, and nothing else."""
    cfg = wall_pair_cfg()
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
    fr, tr, Er, nt = wall_sum(tab, cfg["x"], cfg["quat"], cfg["shape_id"], walls)
    assert (nt > 0).sum() >= 4
    fs = np.abs(a["f"]).max()
    err = max(np.abs(a["f"] - fsum - fr).max(), np.abs(a["torque"] - tsum - tr).max()) / fs
    report("B walls + pairs (pipeline %d)" % variant, err, 1e-12)
    assert err <= 1e-12
    g.close()


# ==== C: analytic caps ================================================================================================
def cap_errors(grid):
    """Spheres (R = 1, random orientations) and axis-aligned ellipsoids (semi-axes 1, 0.8 in the plane, 0.6 along the
    normal) cut by the wall z = 0 at four depths each.  Returns, per shape, the error of the summed cap volume and the
    RMS over the atoms of |f - F_exact z| / F_exact, and the largest |torque| / |F|."""
    k, out = 5.0, {}
    rng = np.random.default_rng(31)
    for name, lmax, (a, b), ds in (("sphere", 0, W.sphere_shape(0, 1.0), (0.3, 0.45, 0.6, 0.75)),
                                   ("ellipsoid", 20, W.ellipsoid_shape(20, 1.0, 0.8, 0.6), (0.15, 0.25, 0.35, 0.45))):
        x = np.array([[5.0 * i, 0, d] for i, d in enumerate(ds)])
        g = pkg.ShGpu()
        build(g, [(lmax, a, b)], grid, x, W.random_quaternions(rng, len(ds)))
        if name == "ellipsoid":       # q = quat_principal: Rs = R(q) Rp^T = 1, the ellipsoid's axes are the space axes
            g.put_state(quat=np.tile(g.shape_props(0)["quat_principal"], (len(ds), 1)))
        g.add_wall((0, 0, 0), (0, 0, 1.0), k, 1.0)
        g.compute_forces()
        at = g.get_atoms()
        A, B, Cc = (1.0, 1.0, 1.0) if name == "sphere" else (1.0, 0.8, 0.6)
        h = Cc - np.array(ds)
        V = np.pi * A * B * h * h * (3 * Cc - h) / (3 * Cc * Cc)          # sphere: pi h^2 (3R - h) / 3
        F = k * np.pi * A * B * (1 - (np.array(ds) / Cc) ** 2)             # sphere: k pi a^2, a^2 = R^2 - d^2
        out["V " + name] = abs(g.get_energy()["e_contact"] / k - V.sum()) / V.sum()
        ferr = np.linalg.norm(at["f"] - F[:, None] * np.array([0, 0, 1.0]), axis=1) / F
        out["F " + name] = np.sqrt(np.mean(ferr ** 2))
        out["tau " + name] = np.max(np.linalg.norm(at["torque"], axis=1) / F)
        g.close()
    return out


def test_wall_caps_closed_forms():
    e48, e80 = cap_errors((48, 96)), cap_errors((80, 160))
    for key in ("V sphere", "F sphere", "V ellipsoid", "F ellipsoid"):
        report("C cap %s 48x96 -> 80x160" % key, e80[key], e48[key])
        assert e80[key] < e48[key] and e48[key] < 0.03, (key, e48[key], e80[key])
    for e in (e48, e80):
        for key in ("tau sphere", "tau ellipsoid"):
            assert e[key] <= 1e-12, (key, e[key])       # symmetric caps: no torque about the centre


# ==== D: energy consistency ===========================================================================================
def fd_check(g, x, q, atoms, h=0.02):
    """Central differences of e_contact: -dE/dx_i against f_i and -dE/dtheta_i (space-frame rotation about x_i,
    q' = q(dtheta) (x) q) against torque_i.  Returns the worst error / |f_i| and |f_i|."""
    g.put_state(x=x, quat=q); g.compute_forces()
    a = g.get_atoms()
    worst, fmin = 0.0, np.inf
    for i in atoms:
        fn = np.linalg.norm(a["f"][i])
        fmin = min(fmin, fn)
        for d in range(3):
            e = []
            for s in (1, -1):
                xx = x.copy(); xx[i, d] += s * h
                g.put_state(x=xx, quat=q); g.compute_forces(); e.append(g.get_energy()["e_contact"])
            worst = max(worst, abs(-(e[0] - e[1]) / (2 * h) - a["f"][i, d]) / fn)
            e = []
            for s in (1, -1):
                qq = q.copy(); qq[i] = quat_mul(axis_quat(s * h * np.eye(3)[d]), q[i])
                g.put_state(x=x, quat=qq); g.compute_forces(); e.append(g.get_energy()["e_contact"])
            worst = max(worst, abs(-(e[0] - e[1]) / (2 * h) - a["torque"][i, d]) / fn)
    g.put_state(x=x, quat=q)
    return worst, fmin


@pytest.mark.parametrize("exponent", [1.0, 1.5])
@pytest.mark.parametrize("case", ["egg-egg", "egg-perturbed", "egg-wall"])
def test_forces_are_minus_energy_gradient(case, exponent):
    grid = (64, 128)
    rng = np.random.default_rng(int(exponent * 4) + 7 * len(case))
    shapes = [SHAPES["egg20"](), SHAPES["perturbed20"]() if case == "egg-perturbed" else SHAPES["egg20"]()]
    worst = 0.0
    for trial in range(3):
        q = W.random_quaternions(rng, 2)
        g = pkg.ShGpu()
        if case == "egg-wall":
            x = np.array([[0, 0, 0.0], [30.0, 0, 0]])
            build(g, shapes, grid, x, q, shape_id=[0, 1], k=200.0, exponent=exponent)
            props, p, n = tables(g, 0, grid)
            nrm = np.array([0.3, -0.5, 0.81])
            x[0] = place_at_depth(p, props, q[0], np.zeros(3), nrm, "medium")
            g.add_wall((0, 0, 0), nrm, 200.0, exponent)
            atoms = [0]
        else:
            dirv = rng.normal(size=3); dirv /= np.linalg.norm(dirv)
            x = np.array([np.zeros(3), 1.45 * dirv])
            build(g, shapes, grid, x, q, shape_id=[0, 1], k=200.0, exponent=exponent)
            atoms = [0, 1]
        w, fmin = fd_check(g, x, q, atoms)
        assert fmin > 1.0, "no contact"
        worst = max(worst, w)
        g.close()
    report("D -grad E %s m=%g" % (case, exponent), worst, 0.08)
    assert worst <= 0.08


def test_angular_momentum_balance_of_a_pair():
    """sum_i (x_i x F_i + tau_i) of egg-perturbed pairs in six poses: below 1e-2 |F| Rmax, and its mean over the poses
    shrinks with the quadrature."""
    shapes = [SHAPES["egg20"](), SHAPES["perturbed20"]()]
    res = {}
    for grid in ((48, 96), (96, 192)):
        rng = np.random.default_rng(8)
        res[grid] = []
        for trial in range(6):
            q = W.random_quaternions(rng, 2)
            d = rng.normal(size=3); d /= np.linalg.norm(d)
            x = np.array([[0.1, 0, 0], [0.1, 0, 0] + 1.45 * d])
            g = pkg.ShGpu()
            build(g, shapes, grid, x, q, shape_id=[0, 1])
            g.compute_forces()
            a = g.get_atoms()
            rmax = max(g.shape_props(0)["rmax"], g.shape_props(1)["rmax"])
            Ltot = np.cross(x, a["f"]).sum(0) + a["torque"].sum(0)
            res[grid].append(np.linalg.norm(Ltot) / (np.linalg.norm(a["f"][0]) * rmax))
            g.close()
    r48, r96 = np.array(res[(48, 96)]), np.array(res[(96, 192)])
    report("D angular momentum max 48x96", r48.max(), 1e-2)
    report("D angular momentum mean 96x192", r96.mean(), r48.mean())
    assert r48.max() < 1e-2 and r96.max() < 1e-2 and r96.mean() < r48.mean(), (r48, r96)


# ==== E: integrator against closed forms ==============================================================================
def free_atoms(rng, n=8):
    """Atoms 10 apart (no contacts), random velocities and spins, egg and perturbed shapes."""
    x = np.stack(np.meshgrid(*[np.arange(2) * 10.0] * 3, indexing="ij"), -1).reshape(-1, 3)[:n]
    return x, rng.normal(0, 1, (n, 3)), W.random_quaternions(rng, n), rng.normal(0, 0.5, (n, 3)), np.arange(n) % 2


def test_gravity_closed_form():
    rng = np.random.default_rng(1)
    x0, v0, q0, L0, sid = free_atoms(rng)
    g = pkg.ShGpu()
    build(g, [SHAPES["egg20"](), SHAPES["perturbed20"]()], (16, 32), x0, q0, v=v0, angmom=L0, shape_id=sid, dt=1e-3)
    grav = np.array([0.4, -1.3, -9.81])
    g.set_gravity(grav)
    g.run(1000)
    a = g.get_atoms()
    t = 1.0
    xr, vr = x0 + v0 * t + 0.5 * grav * t * t, v0 + grav * t
    ex = np.abs(a["x"] - xr).max() / np.abs(xr).max()
    ev = np.abs(a["v"] - vr).max() / np.abs(vr).max()
    report("E gravity x, v (1000 steps)", max(ex, ev), 1e-11)
    assert ex <= 1e-11 and ev <= 1e-11
    assert np.all(a["f"] == 0)
    g.close()


@pytest.mark.parametrize("with_gravity", [False, True])
def test_damping_recurrence(with_gravity):
    """Viscous damping: v and L are multiplied by 1 - dt gamma / 2 in both half steps (after the kick)."""
    rng = np.random.default_rng(2)
    x, v, q0, L0, sid = free_atoms(rng)
    L = L0
    dt, gl, gr, nsteps = 1e-3, 0.5, 0.2, 1000
    grav = np.array([0.4, -1.3, -9.81]) if with_gravity else np.zeros(3)
    g = pkg.ShGpu()
    build(g, [SHAPES["egg20"](), SHAPES["perturbed20"]()], (16, 32), x, q0, v=v, angmom=L, shape_id=sid, dt=dt)
    g.set_gravity(grav)
    g.set_damping(gl, gr)
    g.run(nsteps)
    a = g.get_atoms()
    dv, dL, dth = 1.0 - 0.5 * dt * gl, 1.0 - 0.5 * dt * gr, 0.5 * dt
    x, v, L = x.copy(), v.copy(), L.copy()
    for _ in range(nsteps):
        v = (v + dth * (0.0 + grav)) * dv
        x = x + dt * v
        L = (L + dth * 0.0) * dL
        v = (v + dth * (0.0 + grav)) * dv
        L = (L + dth * 0.0) * dL
    err = max(np.abs(a[k] - r).max() / np.abs(r).max() for k, r in (("x", x), ("v", v), ("angmom", L)))
    report("E damping (gravity %s)" % with_gravity, err, 1e-13)
    assert err <= 1e-13
    assert np.abs(a["angmom"] - L0).max() > 0.1 * np.abs(L0).max()       # the spins were damped
    g.close()


def free_rotation(dt, T, grid=(32, 64)):
    """One egg spinning freely near its intermediate axis; returns the library state, the reference rotation of the
    shape frame from solve_ivp, and the energies at the start and the end."""
    lmax, a, b = SHAPES["egg20"]()
    g = pkg.ShGpu()
    q0 = W.random_quaternions(np.random.default_rng(9), 1)
    build(g, [(lmax, a, b)], grid, np.zeros((1, 3)), q0, dt=dt)
    props, p, n = tables(g, 0, grid)
    Ic = frame_reference(p, n, 1.0)["Ic"]               # shape-frame inertia tensor from the node table
    ev, U = np.linalg.eigh(Ic)                          # U[:, 1]: intermediate axis, shape frame
    Rs0 = quat_mat(q0[0]) @ quat_mat(props["quat_principal"]).T
    L = Rs0 @ (ev[1] * 2.0 * (U[:, 1] + 0.02 * U[:, 0] + 0.01 * U[:, 2]))
    g.put_state(angmom=L[None, :].copy())
    e0 = g.get_energy()
    g.run(int(round(T / dt)))
    st, e1 = g.get_atoms(), g.get_energy()
    Ici = np.linalg.inv(Ic)

    def rhs(t, y):                                      # y = quaternion of Rs; q' = 1/2 (0, w) (x) q
        Rs = quat_mat(y)
        w = Rs @ Ici @ Rs.T @ L
        return 0.5 * quat_mul(np.concatenate([[0.0], w]), y)

    qs0 = np.array(quat_from_mat(Rs0))
    sol = solve_ivp(rhs, (0, T), qs0, method="DOP853", rtol=1e-12, atol=1e-14)
    Rref = quat_mat(sol.y[:, -1])
    Rg = quat_mat(st["quat"][0]) @ quat_mat(props["quat_principal"]).T
    g.close()
    return st, L, rotation_angle(Rg.T @ Rref), e0, e1, 0.5 * L @ Rs0 @ Ici @ Rs0.T @ L


def quat_from_mat(R):
    w = np.sqrt(max(0.0, 1.0 + np.trace(R))) / 2.0
    return np.array([w, (R[2, 1] - R[1, 2]) / (4 * w), (R[0, 2] - R[2, 0]) / (4 * w), (R[1, 0] - R[0, 1]) / (4 * w)])


def test_free_rotation_of_the_egg():
    T = 3.0
    st1, L, err1, e0, e1, ke_ref = free_rotation(2e-3, T)
    st2, _, err2, _, e2, _ = free_rotation(1e-3, T)
    assert np.array_equal(st1["angmom"][0], L) and np.array_equal(st2["angmom"][0], L)     # no torque: L bit for bit
    for st in (st1, st2):
        assert abs(np.linalg.norm(st["quat"][0]) - 1.0) <= 1e-14
    assert abs(e0["ke_rot"] - ke_ref) <= 1e-12 * ke_ref          # omega = I_space^-1 L with the node-table tensor
    dke = max(abs(e1["ke_rot"] - e0["ke_rot"]), abs(e2["ke_rot"] - e0["ke_rot"])) / e0["ke_rot"]
    report("E free rotation angle dt", err1, 2e-5)
    report("E free rotation angle dt/2", err2, err1 / 3)
    report("E free rotation KE_rot drift", dke, 1e-10)
    assert err1 <= 2e-5 and err2 * 3 <= err1
    assert dke <= 1e-10


# ==== F: trajectories with walls, gravity and damping against the oracle ================================================
def wall_settle_cfg():
    cfg = W.config2_wall(n_side=4, exponent=1.5)
    cfg["shapes"] = [egg_shape(20), W.perturbed_shape(20, 3)]
    cfg["shape_id"] = (np.arange(len(cfg["x"])) % 2).astype(np.int32)
    cfg["x"] = cfg["x"] * np.array([1, 1, 0.9]) - np.array([0, 0, 0.7])
    k = cfg["coeff"][0]
    cfg["walls"] = [((0, 0, 0), (0, 0, 1.0), k, 1.5), ((0.6, 0, 0), (1.0, 0.15, 0.35), k, 1.5)]
    return cfg


@pytest.mark.parametrize("variant", PIPELINES)
def test_trajectory_walls_gravity_damping_vs_oracle(variant):
    cfg = wall_settle_cfg()
    g = pkg.ShGpu(); W.apply(g, cfg); g.set_pair_tuning(0, 0, variant); g.set_damping(0.5, 0.2)
    o = O.Oracle(threads=8); W.apply(o, cfg); o.set_damping(0.5, 0.2)
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
    report("F trajectory (pipeline %d) err/tol" % variant, worst, 1.0)
    g.close(); o.close()


# ==== G: walls with the in-library decomposition =======================================================================
@pytest.mark.parametrize("newton", [1, 0])
def test_walls_with_self_ghost_decomposition(newton):
    """Periodic in x and y, walls in z: ghosts must never receive wall forces (only owned atoms get the wall slots)."""
    cfg = W.packing((4, 4, 3), 20, (32, 64), nshapes=4, seed=21, periodic=True, name="ddw", skin=0.03, vel_sigma=0.5, dt=4e-4)
    cfg["v"] = cfg["v"] + np.array([8.0, 1.0, 0.0])
    cfg["box"] = (cfg["box"][0], cfg["box"][1], (1, 1, 0))
    zlo, zhi = cfg["x"][:, 2].min(), cfg["x"][:, 2].max()
    cfg["walls"] = [((0, 0, zlo - 0.25), (0, 0, 1.0), 2e3, 1.0), ((0, 0, zhi + 0.25), (0, 0, -1.0), 2e3, 1.5)]
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
    assert np.linalg.norm(r0["f"].sum(0)) > 0.1 * fs          # the walls push (pair forces alone sum to zero)
    ef = max(np.abs(d0["f"] - r0["f"]).max(), np.abs(d0["torque"] - r0["torque"]).max()) / fs
    report("G forces, newton %d" % newton, ef, 1e-11)
    assert ef <= 1e-11
    ref.run(200); dd.run(200)
    r1 = ref.get_atoms()
    info = dd.dd_info()
    nl = info["nlocal"]
    order = np.argsort(dd.get_tags()[:nl])
    d1 = {k: v[:nl][order] for k, v in dd.get_atoms().items()}
    L = np.asarray(cfg["box"][1]) - np.asarray(cfg["box"][0])
    dx = d1["x"] - r1["x"]; dx[:, :2] -= L[:2] * np.rint(dx[:, :2] / L[:2])
    report("G trajectory x, newton %d" % newton, np.abs(dx).max(), 1e-9)
    assert np.abs(dx).max() <= 1e-9
    for k, tol in (("v", 1e-8), ("quat", 1e-9), ("angmom", 1e-8)):
        assert np.abs(d1[k] - r1[k]).max() <= tol * max(1.0, np.abs(r1[k]).max()), k
    assert info["border_builds"] >= 2, info
    ref.close(); dd.close()
