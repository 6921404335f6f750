"""CPU tests of the rigid-body frame of a shape and of the plane-wall contact, against references built here from the node
table alone (no library value enters them except the node points and area elements).

Frame (csrc/shape_tables.cpp, oracle/sh_oracle.c): `inertia` holds the principal moments about the centre of mass and
Rp = R(quat_principal) has the principal axes as its COLUMNS, i.e. Rp maps principal-frame coordinates to shape-frame
coordinates and Rp^T Ic Rp = diag(inertia).  An atom's quaternion q is the orientation of its principal frame, so the
shape -> space rotation is Rs = R(q) Rp^T and the SH origin sits at c = x - Rs com (DESIGN §3.2).

The shapes include an off-centre "egg" (|com| ~ 0.19, principal axes far from the shape axes): for the centred,
axis-aligned ellipsoid com = 0 and Rp = 1, where a lever-arm or frame error cancels.  Both host-side table builders
are tested, the oracle's and the product's (compiled into tests/shape_tables_harness.cpp); the GPU tests
(test_gpu_walls_integrator.py) check the device library's copy and use the helpers below.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle_py as O
import shpkg

W = shpkg.load().workloads
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- shapes ---------------------------------------------------------------------------------------------------------
def egg_shape(lmax):
    """Sphere of radius 0.8 plus l = 1 and l = 2 terms: centre of mass ~ (0.08, 0.00, 0.17) off the SH origin and
    principal axes far from the shape axes."""
    a, b = W.sphere_shape(lmax, 0.8)
    a[W.lm_index(1, 0)] += 0.35
    a[W.lm_index(1, 1)] += 0.2
    a[W.lm_index(2, 1)] += 0.15
    b[W.lm_index(2, 2)] += 0.1
    return a, b


SHAPES = {
    "egg20": lambda: (20, *egg_shape(20)),
    "egg30": lambda: (30, *egg_shape(30)),
    "perturbed20": lambda: (20, *W.perturbed_shape(20, 3)),
    "perturbed30": lambda: (30, *W.perturbed_shape(30, 4)),
    "ellipsoid20": lambda: (20, *W.ellipsoid_shape(20)),
    "sphere": lambda: (4, *W.sphere_shape(4, 0.9)),
}


# ---- rotations (w, x, y, z) -------------------------------------------------------------------------------------------
def quat_mat(q):
    w, x, y, z = np.asarray(q, float) / np.linalg.norm(q)
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def quat_mul(a, b):
    a0, av, b0, bv = a[0], np.asarray(a[1:]), b[0], np.asarray(b[1:])
    return np.concatenate([[a0 * b0 - av @ bv], a0 * bv + b0 * av + np.cross(av, bv)])


def axis_quat(axis_angle):
    """Quaternion of the rotation by |v| about v."""
    v = np.asarray(axis_angle, float)
    t = np.linalg.norm(v)
    if t == 0:
        return np.array([1.0, 0, 0, 0])
    return np.concatenate([[np.cos(0.5 * t)], np.sin(0.5 * t) * v / t])


def rotation_angle(R):
    return np.arccos(np.clip(0.5 * (np.trace(R) - 1.0), -1.0, 1.0))


# ---- references -----------------------------------------------------------------------------------------------------
def frame_reference(p, n, density):
    """Volume, centre of mass and inertia tensor about the COM (shape frame) of the closed surface given by node points
    p and area elements n = n dS, by the divergence theorem:  V = 1/3 sum p.n,  V com = 1/4 sum p (p.n),
    M_ij = int x_i x_j dV = 1/5 sum p_i p_j (p.n);  I = density (tr(Mc) 1 - Mc) with Mc = M - V com com^T."""
    pn = np.einsum("kd,kd->k", p, n)
    V = pn.sum() / 3.0
    com = (p * pn[:, None]).sum(0) / 4.0 / V
    M = np.einsum("ki,kj,k->ij", p, p, pn) / 5.0
    Mc = M - V * np.outer(com, com)
    Ic = density * (np.trace(Mc) * np.eye(3) - Mc)
    return dict(volume=V, com=com, Ic=Ic, mass=density * V)


def pose(props, q, x):
    """Rs = R(q) Rp^T (shape -> space), c = x - Rs com."""
    Rs = quat_mat(q) @ quat_mat(props["quat_principal"]).T
    return Rs, np.asarray(x, float) - Rs @ props["com"]


def wall_reference(p, n, props, x, q, point, normal, k, m):
    """Plane wall on one atom: submerged nodes (c + Rs p - point).n < 0, V = 1/3 sum (P - foot).N with foot the point of
    the plane nearest c, pressure m k V^(m-1), E = k V^m, F = -pressure sum N, torque about x = -pressure sum (P - x) x N.
    Returns (F, torque, E, number of submerged nodes)."""
    nh = np.asarray(normal, float) / np.linalg.norm(normal)
    Rs, c = pose(props, q, x)
    P = c + p @ Rs.T
    N = n @ Rs.T
    sub = (P - point) @ nh < 0
    if not sub.any():
        return np.zeros(3), np.zeros(3), 0.0, 0
    foot = c - ((c - point) @ nh) * nh
    V = ((P[sub] - foot) * N[sub]).sum() / 3.0
    if not V > 0:
        return np.zeros(3), np.zeros(3), 0.0, int(sub.sum())
    pr = m * k * V ** (m - 1.0)
    F = -pr * N[sub].sum(0)
    tau = -pr * np.cross(P[sub] - x, N[sub]).sum(0)
    return F, tau, k * V ** m, int(sub.sum())


def node_heights(p, props, x, q, normal):
    """Signed heights (P - x).n of every node of an atom at x, q above a plane through x with the given normal."""
    nh = np.asarray(normal, float) / np.linalg.norm(normal)
    Rs, c = pose(props, q, x)
    return (c + p @ Rs.T - x) @ nh


def in_plane(normal):
    """Two unit vectors spanning the plane with this normal."""
    nh = np.asarray(normal, float) / np.linalg.norm(normal)
    t1 = np.cross(nh, [1.0, 0, 0] if abs(nh[0]) < 0.9 else [0, 1.0, 0])
    t1 /= np.linalg.norm(t1)
    return t1, np.cross(nh, t1)


def place_at_depth(p, props, q, point, normal, depth):
    """Atom position (COM) whose shape, in orientation q, crosses the plane through `point`: depth = "grazing" (6 nodes
    submerged, the plane half-way between the 6th and 7th lowest node), "medium" (0.35 of the shape's extent along the
    normal under the plane) or "deep" (the SH origin itself under the plane)."""
    nh = np.asarray(normal, float) / np.linalg.norm(normal)
    g = np.sort(node_heights(p, props, np.zeros(3), q, nh))
    if depth == "grazing":
        assert g[6] - g[5] > 1e-9
        s = -0.5 * (g[5] + g[6])
    elif depth == "medium":
        s = -(g[0] + 0.35 * (g[-1] - g[0]))
    else:
        Rs, c = pose(props, q, np.zeros(3))
        s = -(c @ nh) - 0.1          # c.n = -0.1 above the plane: the origin is under it
    return np.asarray(point, float) + s * nh


# ---- the product's host-side table builder, through the test harness -------------------------------------------------
@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    out = tmp_path_factory.mktemp("sthf") / "libshtables_frame.so"
    gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.check_call([gxx, "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-pthread", "-o", str(out),
                           os.path.join(ROOT, "tests", "shape_tables_harness.cpp"),
                           os.path.join(ROOT, "lammps-spherharm_b200", "csrc", "shape_tables.cpp")])
    lib = C.CDLL(str(out))
    lib.sth_build.restype = C.c_void_p
    lib.sth_build.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_int]
    lib.sth_free.argtypes = [C.c_void_p]
    lib.sth_frame.argtypes = [C.c_void_p, C.c_void_p]
    lib.sth_nodes.argtypes = [C.c_void_p] * 3
    return lib


def product_tables(lib, lmax, a, b, density, grid):
    a, b = np.ascontiguousarray(a, float), np.ascontiguousarray(b, float)
    err = C.create_string_buffer(256)
    t = lib.sth_build(lmax, a.ctypes.data, b.ctypes.data, density, grid[0], grid[1], 16, err, 256)
    assert t, err.value
    nq = grid[0] * grid[1]
    out, p, n = np.zeros(11), np.zeros((nq, 3)), np.zeros((nq, 3))
    lib.sth_frame(t, out.ctypes.data)
    lib.sth_nodes(t, p.ctypes.data, n.ctypes.data)
    lib.sth_free(t)
    return dict(volume=out[0], com=out[1:4], inertia=out[4:7], quat_principal=out[7:11]), p, n


def oracle_tables(lmax, a, b, density, grid):
    o = O.Oracle()
    o.set_quadrature(*grid)
    sid = o.add_shape(lmax, a, b, density)
    props, (p, n) = o.shape_props(sid), o.nodes(sid, grid[0] * grid[1])
    o.close()
    return props, p, n


def check_frame(props, p, n, density, rscale):
    """The assertions of the frame test; shared with the GPU test of the device library's tables."""
    ref = frame_reference(p, n, density)
    assert abs(props["volume"] - ref["volume"]) <= 1e-12 * ref["volume"]
    assert np.abs(props["com"] - ref["com"]).max() <= 1e-12 * rscale
    Ic, Imax = ref["Ic"], np.abs(ref["Ic"]).max()
    assert np.abs(np.sort(props["inertia"]) - np.linalg.eigvalsh(Ic)).max() <= 1e-10 * Imax
    qp = np.asarray(props["quat_principal"])
    assert abs(np.linalg.norm(qp) - 1.0) <= 1e-14
    Rp = quat_mat(qp)
    assert abs(np.linalg.det(Rp) - 1.0) <= 1e-13
    D = Rp.T @ Ic @ Rp          # principal -> shape frame: the tensor is diagonal in the order of `inertia`
    assert np.abs(D - np.diag(props["inertia"])).max() <= 1e-10 * Imax, D
    return ref


@pytest.mark.parametrize("lib", ["oracle", "product"])
@pytest.mark.parametrize("name", sorted(SHAPES))
def test_shape_frame_vs_divergence_theorem(name, lib, harness):
    lmax, a, b = SHAPES[name]()
    density, grid = 1.3, (48, 96)
    props, p, n = oracle_tables(lmax, a, b, density, grid) if lib == "oracle" else \
        product_tables(harness, lmax, a, b, density, grid)
    rscale = np.linalg.norm(p, axis=1).max()
    ref = check_frame(props, p, n, density, rscale)
    if name.startswith("egg"):
        # the frame really is off-centre and tilted (a test on it is not a test on the centred ellipsoid)
        assert np.linalg.norm(ref["com"]) > 0.15
        assert abs(abs(props["quat_principal"][0]) - 1.0) > 0.1


def test_both_table_builders_agree(harness):
    lmax, a, b = SHAPES["egg20"]()
    po, p1, n1 = oracle_tables(lmax, a, b, 1.3, (32, 64))
    pp, p2, n2 = product_tables(harness, lmax, a, b, 1.3, (32, 64))
    assert np.array_equal(p1, p2) and np.array_equal(n1, n2)
    for k in ("volume", "com", "inertia", "quat_principal"):
        assert np.array_equal(np.asarray(po[k]), np.asarray(pp[k])), k


@pytest.mark.parametrize("exponent", [1.0, 1.5, 2.0])
def test_wall_reference_matches_oracle(exponent):
    """The numpy wall reference (space frame, nodes moved one by one) against the oracle's shape-frame evaluation, on the
    egg and a perturbed shape, tilted normals given at length != 1, three depths and random poses."""
    grid = (32, 64)
    rng = np.random.default_rng(int(exponent * 10))
    normals = [(0, 0, 1.0), (0.3, -0.5, 2.0), (-0.2, 0.7, -0.6)]
    for sname in ("egg20", "perturbed20"):
        lmax, a, b = SHAPES[sname]()
        for nrm in normals:
            o = O.Oracle()
            o.set_quadrature(*grid)
            sid = o.add_shape(lmax, a, b, 1.0)
            props, (p, n) = o.shape_props(sid), o.nodes(sid, grid[0] * grid[1])
            point = np.array([0.3, -0.2, 0.1])
            xs, qs = [], []
            t1, _ = in_plane(nrm)
            for i, depth in enumerate(("grazing", "medium", "deep")):
                q = W.random_quaternions(rng, 1)[0]
                xs.append(place_at_depth(p, props, q, point + 4.0 * i * t1, nrm, depth))
                qs.append(q)
            o.set_atoms(np.zeros(3, np.int32), np.array(xs), quat=np.array(qs))
            o.add_wall(point, nrm, 70.0, exponent)
            o.compute_forces()
            at, E = o.get_atoms(), 0.0
            for i in range(3):
                F, tau, e, nsub = wall_reference(p, n, props, xs[i], qs[i], point, nrm, 70.0, exponent)
                assert nsub > 0
                fs = np.linalg.norm(F)
                assert np.abs(at["f"][i] - F).max() <= 1e-12 * fs
                assert np.abs(at["torque"][i] - tau).max() <= 1e-12 * fs
                E += e
            assert abs(o.get_energy()["e_contact"] - E) <= 1e-12 * E
            o.close()
