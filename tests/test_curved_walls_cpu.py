"""CPU tests of the curved container walls (cylinder and sphere, particles inside): a numpy reference built from the node
table alone against closed forms and against the oracle, and the shlmp syntax of fix wall/spherharm zcylinder / sphere.

The submerged volume is the flux of a field phi with div phi = 1 that vanishes on the wall, summed over the nodes past
the wall:  cylinder phi = (|rho|^2 - R^2) / (2 |rho|^2) rho  (rho: the part of P - a normal to the axis),
sphere phi = (|r|^3 - R^3) / (3 |r|^3) r  (r = P - centre).  Force and torque are the plane wall's: F = -p sum N,
tau = -p sum (P - x) x N, p = m k V^(m-1).  The GPU tests (test_gpu_curved_walls.py) use the helpers below.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest
from scipy import integrate

import oracle_py as O
import shpkg
from test_shape_frame_cpu import SHAPES, pose
from test_shlmp_check_cpu import HEAD, shlmp

W = shpkg.load().workloads
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_CW_LIB = None


# ---- the oracle with curved walls (tests/curved_wall_oracle.c: the unchanged oracle plus the curved-wall loop) ---------
def curved_oracle_lib():
    global _CW_LIB
    if _CW_LIB is None:
        out = os.path.join(tempfile.mkdtemp(prefix="curved_oracle_"), "libcurvedoracle.so")
        gcc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
        subprocess.check_call([gcc, "-O2", "-std=c11", "-fPIC", "-mfma", "-mavx2", "-ffp-contract=off", "-fopenmp", "-shared",
                               "-o", out, os.path.join(ROOT, "tests", "curved_wall_oracle.c"), "-lm"])
        lib = C.CDLL(out)
        lib.cw_create.restype = C.c_void_p
        lib.cw_oracle.restype = C.c_void_p
        lib.cw_oracle.argtypes = [C.c_void_p]
        lib.cw_destroy.argtypes = [C.c_void_p]
        lib.orc_last_error.restype = C.c_char_p
        lib.orc_last_error.argtypes = [C.c_void_p]
        _CW_LIB = lib
    return _CW_LIB


class CurvedOracle(O.Oracle):
    """The CPU oracle's call surface plus add_cylinder_wall / add_sphere_wall; compute_forces and run include the curved
    walls after the planes, in insertion order, with curved_wall_kernel's operation sequence."""

    def __init__(self, threads=1):
        self.L = curved_oracle_lib()
        self.cw = C.c_void_p(self.L.cw_create())
        self.h = C.c_void_p(self.L.cw_oracle(self.cw))
        self.L.orc_set_threads(self.h, int(threads))
        self.n = 0

    def close(self):
        if getattr(self, "cw", None):
            self.L.cw_destroy(self.cw)
            self.cw, self.h = None, None

    def add_cylinder_wall(self, point, axis, radius, k, exponent):
        p, u = O._d(point), O._d(axis)
        self._ck(self.L.cw_add_cylinder_wall(self.cw, O._p(p), O._p(u), C.c_double(radius), C.c_double(k), C.c_double(exponent)))

    def add_sphere_wall(self, center, radius, k, exponent):
        c = O._d(center)
        self._ck(self.L.cw_add_sphere_wall(self.cw, O._p(c), C.c_double(radius), C.c_double(k), C.c_double(exponent)))

    def compute_forces(self):
        self._ck(self.L.cw_compute_forces(self.cw))

    def run(self, nsteps):
        self._ck(self.L.cw_run(self.cw, C.c_int64(nsteps)))


# ---- reference ------------------------------------------------------------------------------------------------------
def radial(P, wall):
    """Vector from the wall's axis (cylinder, perpendicular to it) or centre (sphere) to each point P."""
    if wall[0] == "cylinder":
        _, a, u, _R = wall
        u = np.asarray(u, float) / np.linalg.norm(u)
        r = P - np.asarray(a, float)
        return r - np.outer(r @ u, u)
    return P - np.asarray(wall[1], float)


def curved_wall_reference(p, n, props, x, q, wall, k, m):
    """One curved wall on one atom, space frame.  wall = ("cylinder", point, axis, R) or ("sphere", centre, R).
    Returns (F, torque about x, E, V, number of nodes past the wall)."""
    R = wall[-1]
    Rs, c = pose(props, q, x)
    P = c + p @ Rs.T
    N = n @ Rs.T
    r = radial(P, wall)
    r2 = (r * r).sum(1)
    out = r2 > R * R
    if not out.any():
        return np.zeros(3), np.zeros(3), 0.0, 0.0, 0
    ro, q2 = r[out], r2[out]
    if wall[0] == "cylinder":
        g = (q2 - R * R) / (2 * q2)
    else:
        q3 = q2 * np.sqrt(q2)
        g = (q3 - R ** 3) / (3 * q3)
    V = (g * (ro * N[out]).sum(1)).sum()
    if not V > 0:
        return np.zeros(3), np.zeros(3), 0.0, V, int(out.sum())
    pr = m * k * V ** (m - 1.0)
    F = -pr * N[out].sum(0)
    tau = -pr * np.cross(P[out] - x, N[out]).sum(0)
    return F, tau, k * V ** m, V, int(out.sum())


def curved_sum(tab, x, q, sid, walls):
    """Reference f, torque per atom and total energy over all curved walls (("cylinder", point, axis, R, k, m) or
    ("sphere", centre, R, k, m)), and the number of walls each atom touches."""
    n = len(x)
    f, t, nt, E = np.zeros((n, 3)), np.zeros((n, 3)), np.zeros(n, int), 0.0
    for i in range(n):
        props, p, nn = tab[sid[i]]
        for w in walls:
            F, tau, e, _, _ = curved_wall_reference(p, nn, props, x[i], q[i], w[:-2], w[-2], w[-1])
            f[i] += F; t[i] += tau; E += e
            nt[i] += e > 0
    return f, t, E, nt


def perpendicular(u):
    u = np.asarray(u, float) / np.linalg.norm(u)
    t = np.cross(u, [1.0, 0, 0] if abs(u[0]) < 0.9 else [0, 1.0, 0])
    return t / np.linalg.norm(t)


def place_in_container(p, props, q, wall, e, along, depth):
    """COM of an atom in orientation q pushed along the unit direction e (perpendicular to the axis for a cylinder)
    against the wall, `along` further along the axis (cylinder): depth = "grazing" (about 6 nodes past the wall),
    "medium" (0.35 of the shape's extent along e past it) or "deep" (the SH origin 0.1 past the wall)."""
    R = wall[-1]
    Rs, c = pose(props, q, np.zeros(3))
    h = np.sort((c + p @ Rs.T) @ e)          # node heights along e relative to the COM
    if depth == "grazing":
        s = R - 0.5 * (h[-6] + h[-7])
    elif depth == "medium":
        s = R - (h[-1] - 0.35 * (h[-1] - h[0]))
    else:
        s = R + 0.1 - c @ e
    base = np.asarray(wall[1], float)
    if wall[0] == "cylinder":
        u = np.asarray(wall[2], float) / np.linalg.norm(wall[2])
        base = base + along * u
    return base + s * e


def oracle_tables(sim, grid, shapes):
    sim.set_quadrature(*grid)
    tab = []
    for (lmax, a, b) in shapes:
        sid = sim.add_shape(lmax, a, b, 1.0)
        tab.append((sim.shape_props(sid), *sim.nodes(sid, grid[0] * grid[1])))
    return tab


# ---- closed forms ---------------------------------------------------------------------------------------------------
def lens_volume(a, R, D):
    """Volume of the intersection of balls of radii a and R with centres D apart (|R - a| < D < R + a)."""
    return np.pi * (R + a - D) ** 2 * (D * D + 2 * D * a - 3 * a * a + 2 * D * R + 6 * a * R - 3 * R * R) / (12 * D)


def ball_outside_cylinder(a, R, D):
    """V and sum N (radial component, pointing away from the axis) of a ball of radius a, centre D from the axis of a
    cylinder of radius R, outside the cylinder: 1-D integrals over the height z."""
    def seg(z):                                # area of the slice disc (radius s, centre D) outside the circle R
        s = np.sqrt(max(a * a - z * z, 0.0))
        if s == 0 or D + s <= R:
            return 0.0
        if D >= R + s:
            return np.pi * s * s
        c1 = np.arccos((D * D + s * s - R * R) / (2 * D * s))
        c2 = np.arccos((D * D + R * R - s * s) / (2 * D * R))
        inter = s * s * c1 + R * R * c2 - 0.5 * np.sqrt((-D + s + R) * (D + s - R) * (D - s + R) * (D + s + R))
        return np.pi * s * s - inter

    def g(z):                                  # 2 sin(theta0(z)): the cut face's flux per unit height / R
        c = (R * R + D * D + z * z - a * a) / (2 * R * D)
        return 2.0 * np.sqrt(1 - c * c) if abs(c) <= 1 else 0.0
    zmax = np.sqrt(max(a * a - (R - D) ** 2, 0.0))
    V = integrate.quad(seg, -a, a, points=[-zmax, zmax], limit=400, epsabs=1e-14, epsrel=1e-13)[0]
    S = R * integrate.quad(g, -zmax, zmax, limit=400, epsabs=1e-14, epsrel=1e-13)[0]
    return V, S


def container_errors(grid, wall_kind, evaluate):
    """A radius-1 sphere against a container of radius 5 at four depths, random orientations and directions.
    `evaluate(grid, tab, x, q, wall, k)` returns per-atom forces (n, 3), torques (n, 3) and energies (n,).  Returns the RMS
    over the atoms of |V - V_exact| / V_exact and of |f - F_exact| / |F_exact|, and the largest |torque| / |F|.  (Errors
    of single atoms are quadrature clipping and do not fall monotonically at one depth; their RMS does.)"""
    k, a, R = 5.0, 1.0, 5.0
    rng = np.random.default_rng(41 if wall_kind == "sphere" else 43)
    o = O.Oracle()
    tab = oracle_tables(o, grid, [(0, *W.sphere_shape(0, a))])
    o.close()
    ds = np.array([4.3, 4.45, 4.6, 4.75])
    q = W.random_quaternions(rng, len(ds))
    if wall_kind == "sphere":
        wall = ("sphere", np.array([0.3, -0.2, 0.1]), R)
        dirs = np.eye(3)[[0, 1, 2, 0]] * np.array([[1], [1], [1], [-1.0]])
        x = wall[1] + ds[:, None] * dirs
        Vx = 4 / 3 * np.pi * a ** 3 - lens_volume(a, R, ds)
        Sx = np.pi * (R * R - ((ds * ds + R * R - a * a) / (2 * ds)) ** 2)
    else:
        u = np.array([0.2, -0.4, 1.0])
        wall = ("cylinder", np.array([0.3, -0.2, 0.1]), u, R)
        e1 = perpendicular(u); e2 = np.cross(u / np.linalg.norm(u), e1)
        dirs = np.array([e1, e2, -e1, (e1 + e2) / np.sqrt(2)])
        x = wall[1] + ds[:, None] * dirs + (4.0 * np.arange(4))[:, None] * u / np.linalg.norm(u)
        Vx, Sx = np.array([ball_outside_cylinder(a, R, d) for d in ds]).T
    f, t, e = evaluate(grid, tab, x, q, wall, k)
    Fx = k * Sx[:, None] * -dirs                  # towards the axis / centre, m = 1
    ferr = np.linalg.norm(f - Fx, axis=1) / np.linalg.norm(Fx, axis=1)
    return dict(V=np.sqrt(np.mean(((e / k - Vx) / Vx) ** 2)), F=np.sqrt(np.mean(ferr ** 2)),
                tau=np.max(np.linalg.norm(t, axis=1) / np.linalg.norm(Fx, axis=1)))


def numpy_evaluate(grid, tab, x, q, wall, k):
    props, p, n = tab[0]
    res = [curved_wall_reference(p, n, props, x[i], q[i], wall, k, 1.0) for i in range(len(x))]
    return np.array([r[0] for r in res]), np.array([r[1] for r in res]), np.array([r[2] for r in res])


@pytest.mark.parametrize("wall_kind", ["sphere", "cylinder"])
def test_reference_closed_forms(wall_kind):
    e48 = container_errors((48, 96), wall_kind, numpy_evaluate)
    e80 = container_errors((80, 160), wall_kind, numpy_evaluate)
    for key in ("V", "F"):
        print("%s %s: 48x96 %.2e  80x160 %.2e" % (wall_kind, key, e48[key], e80[key]))
        assert e80[key] < e48[key] and e48[key] < 0.03, (key, e48[key], e80[key])
    for e in (e48, e80):
        assert e["tau"] <= 1e-12, e


# ---- numpy reference against the oracle -----------------------------------------------------------------------------
CURVED_SHAPES = ("egg20", "perturbed20", "ellipsoid20", "sphere")
CONTAINERS = {
    "zcylinder": ("cylinder", (0.0, 0.0, 0.0), (0.0, 0.0, 1.0), 5.0),
    "tilted_cylinder": ("cylinder", (0.4, -0.3, 0.2), (0.3, -0.5, 0.81), 4.0),
    "unnormalised_cylinder": ("cylinder", (-0.5, 0.2, 0.7), (-1.2, 0.9, 2.4), 3.5),
    "sphere": ("sphere", (0.4, -0.3, 0.2), 5.0),
    "small_sphere": ("sphere", (-0.2, 0.1, 0.3), 2.5),
}
DEPTHS = ("grazing", "medium", "deep")


def container_atoms(tab, wall, rng):
    """One atom per shape and depth, each pushed against the wall in its own direction (random poses)."""
    x, q, sid = [], [], []
    if wall[0] == "cylinder":
        u = np.asarray(wall[2], float) / np.linalg.norm(wall[2])
        e1 = perpendicular(u); e2 = np.cross(u, e1)
    for i in range(len(tab)):
        for j, depth in enumerate(DEPTHS):
            qq = W.random_quaternions(rng, 1)[0]
            if wall[0] == "cylinder":
                ang = 2 * np.pi * j / len(DEPTHS)
                e, along = np.cos(ang) * e1 + np.sin(ang) * e2, 4.0 * i
            else:                                  # spread over the sphere: a Fibonacci point per atom
                kk = i * len(DEPTHS) + j + 0.5
                th, ph = np.arccos(1 - 2 * kk / (len(tab) * len(DEPTHS))), np.pi * (1 + 5 ** 0.5) * kk
                e, along = np.array([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th)]), 0.0
            x.append(place_in_container(tab[i][1], tab[i][0], qq, wall, e, along, depth))
            q.append(qq); sid.append(i)
    return np.array(x), np.array(q), np.array(sid)


@pytest.mark.parametrize("container", sorted(CONTAINERS))
@pytest.mark.parametrize("exponent", [1.0, 1.5, 2.0])
def test_reference_matches_oracle(exponent, container):
    grid = (32, 64)
    rng = np.random.default_rng(int(exponent * 10) + 100 * sorted(CONTAINERS).index(container))
    wall = CONTAINERS[container]
    o = CurvedOracle()
    tab = oracle_tables(o, grid, [SHAPES[s]() for s in CURVED_SHAPES])
    x, q, sid = container_atoms(tab, wall, rng)
    if wall[-1] < 3:                               # the small sphere holds one shape at a time: check the first only
        x, q, sid = x[:3], q[:3], sid[:3]
    o.set_atoms(sid.astype(np.int32), x, quat=q)
    for i in range(len(tab)):
        for j in range(i, len(tab)):
            o.pair_coeff(i, j, 0.0, 1.0)         # no pair forces: only the wall acts
    walls = [wall + (70.0, exponent)]
    if wall[0] == "cylinder":
        o.add_cylinder_wall(wall[1], wall[2], wall[3], 70.0, exponent)
    else:
        o.add_sphere_wall(wall[1], wall[2], 70.0, exponent)
    o.compute_forces()
    at = o.get_atoms()
    f, t, E, nt = curved_sum(tab, x, q, sid, walls)
    assert nt.sum() >= len(x) - len(tab), nt
    fs = np.maximum(np.linalg.norm(f, axis=1), 1e-300)[:, None]
    assert np.all(at["f"][nt == 0] == 0)
    assert np.max(np.abs(at["f"] - f) / fs) <= 1e-12
    assert np.max(np.abs(at["torque"] - t) / fs) <= 1e-12
    assert abs(o.get_energy()["e_contact"] - E) <= 1e-12 * E
    o.close()


def test_oracle_refuses_bad_curved_walls():
    o = CurvedOracle()
    for call in (lambda: o.add_cylinder_wall((0, 0, 0), (0, 0, 0), 1.0, 1.0, 1.0),
                 lambda: o.add_cylinder_wall((0, 0, 0), (0, 0, 1), 0.0, 1.0, 1.0),
                 lambda: o.add_sphere_wall((0, 0, 0), -1.0, 1.0, 1.0),
                 lambda: o.add_sphere_wall((0, 0, 0), 1.0, -1.0, 1.0),
                 lambda: o.add_sphere_wall((0, 0, 0), 1.0, 1.0, 0.5)):
        with pytest.raises(RuntimeError):
            call()
    for i in range(8):
        o.add_sphere_wall((0, 0, 0), 5.0 + i, 1.0, 1.0)
    with pytest.raises(RuntimeError, match="too many curved walls"):
        o.add_cylinder_wall((0, 0, 0), (0, 0, 1), 5.0, 1.0, 1.0)
    o.close()


# ---- shlmp syntax ---------------------------------------------------------------------------------------------------
def test_silo_example_parses():
    res = shlmp(script_file="in.silo")
    assert res.returncode == 0, res.stderr
    assert "run 5000 with 256 atoms, 1 shape(s), 2 wall(s) OK" in res.stdout


def test_curved_wall_syntax_is_accepted():
    text = HEAD + ("pair_style spherharm\npair_coeff 1 1 1000 1\ncreate_atoms 1 single 0 0 0\n"
                   "fix 1 all wall/spherharm zcylinder 4.5 1000 1.5\nfix 2 all wall/spherharm sphere 0 0 0.5 4.8 1000 1\n"
                   "fix 3 all wall/spherharm zplane -4 1000 1\nrun 1\n")
    res = shlmp(script_text=text)
    assert res.returncode == 0, res.stderr
    assert "run 1 with 1 atoms, 1 shape(s), 3 wall(s) OK" in res.stdout


ILLEGAL = "Illegal fix wall/spherharm command"


@pytest.mark.parametrize("fix,msg", [
    ("fix 1 all wall/spherharm zcylinder 4.5 1000", ILLEGAL),
    ("fix 1 all wall/spherharm zcylinder 4.5 1000 1 hi", ILLEGAL),
    ("fix 1 all wall/spherharm sphere 0 0 4.5 1000 1", ILLEGAL),
    ("fix 1 all wall/spherharm zcylinder 0 1000 1", ILLEGAL),
    ("fix 1 all wall/spherharm zcylinder -2 1000 1", ILLEGAL),
    ("fix 1 all wall/spherharm sphere 0 0 0 0 1000 1", ILLEGAL),
    ("fix 1 all wall/spherharm zcylinder 4 -1 1", ILLEGAL),
    ("fix 1 all wall/spherharm sphere 0 0 0 4 1000 0.5", ILLEGAL),
    ("fix 1 all wall/spherharm ycylinder 4.5 1000 1", ILLEGAL),
    ("fix 1 all wall/spherharm cone 0 0 0 4.5 1000 1", ILLEGAL),
    ("\n".join("fix %d all wall/spherharm zcylinder %d 1000 1" % (i, 4 + i) for i in range(9)),
     ILLEGAL + ": at most 8 zcylinder / sphere walls"),
])
def test_malformed_curved_walls_are_rejected(fix, msg):
    res = shlmp(script_text=HEAD + "pair_style spherharm\n" + fix + "\nrun 1\n")
    assert res.returncode == 1
    assert "ERROR: " + msg in res.stderr, res.stderr
