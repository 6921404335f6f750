"""Synthetic SPHERHARM workloads (BASELINE.json configs, SURVEY §8d) — host-side numpy only.

Everything here is input generation (shape coefficients, packings, the LAMMPS-style parameter
set); no force or neighbor computation happens in Python.  `apply(sim, cfg)` drives any object
with the sh_* call surface (lammps_spherharm_b200.ShGpu, or the CPU oracle in tests/bench).
"""
import numpy as np


# ---------------------------------------------------------------------------------------------
# spherical-harmonic helpers (real orthonormal, no Condon-Shortley phase; SURVEY A.1/A.2)
# ---------------------------------------------------------------------------------------------
def legendre_norm(lmax, x):
    """P[l, m, :] fully normalised associated Legendre at x (array)."""
    x = np.atleast_1d(np.asarray(x, dtype=np.float64))
    s = np.sqrt((1.0 - x) * (1.0 + x))
    P = np.zeros((lmax + 1, lmax + 1, x.size))
    pmm = np.full_like(x, np.sqrt(1.0 / (4.0 * np.pi)))
    for m in range(lmax + 1):
        if m > 0:
            pmm = np.sqrt((2.0 * m + 1.0) / (2.0 * m)) * s * pmm
        P[m, m] = pmm
        if m < lmax:
            P[m + 1, m] = np.sqrt(2.0 * m + 3.0) * x * pmm
        for l in range(m + 2, lmax + 1):
            A = np.sqrt((4.0 * l * l - 1.0) / (l * l - m * m))
            B = np.sqrt(((l - 1.0) ** 2 - m * m) / (4.0 * (l - 1.0) ** 2 - 1.0))
            P[l, m] = A * (x * P[l - 1, m] - B * P[l - 2, m])
    return P


def lm_index(l, m):
    return l * (l + 1) // 2 + m


def project(lmax, rfunc, n_theta=128, n_phi=256):
    """Project r(theta, phi) onto (a_lm, b_lm), index l(l+1)/2+m."""
    gx, gw = np.polynomial.legendre.leggauss(n_theta)
    phi = (np.arange(n_phi) + 0.5) * 2.0 * np.pi / n_phi
    theta = np.arccos(gx)
    r = rfunc(theta[:, None], phi[None, :])                       # (nt, np)
    P = legendre_norm(lmax, gx)                                   # (L+1, L+1, nt)
    T = (lmax + 1) * (lmax + 2) // 2
    a, b = np.zeros(T), np.zeros(T)
    dphi = 2.0 * np.pi / n_phi
    for m in range(lmax + 1):
        cm = (r * np.cos(m * phi)[None, :]).sum(1) * dphi          # (nt,)
        sm = (r * np.sin(m * phi)[None, :]).sum(1) * dphi
        fm = 1.0 if m == 0 else 2.0
        for l in range(m, lmax + 1):
            a[lm_index(l, m)] = fm * np.sum(gw * P[l, m] * cm)
            b[lm_index(l, m)] = fm * np.sum(gw * P[l, m] * sm)
    return a, b


def evaluate(lmax, a, b, theta, phi):
    theta, phi = np.broadcast_arrays(np.asarray(theta, float), np.asarray(phi, float))
    P = legendre_norm(lmax, np.cos(theta).ravel())
    ph = phi.ravel()
    r = np.zeros(ph.size)
    for l in range(lmax + 1):
        for m in range(l + 1):
            k = lm_index(l, m)
            r += P[l, m] * (a[k] * np.cos(m * ph) + b[k] * np.sin(m * ph))
    return r.reshape(theta.shape)


def ellipsoid_radius(ax, by, cz):
    def r(theta, phi):
        st, ct = np.sin(theta), np.cos(theta)
        return 1.0 / np.sqrt((st * np.cos(phi) / ax) ** 2 + (st * np.sin(phi) / by) ** 2 + (ct / cz) ** 2)
    return r


def ellipsoid_shape(lmax, ax=1.0, by=0.8, cz=0.6):
    return project(lmax, ellipsoid_radius(ax, by, cz))


def sphere_shape(lmax, radius=1.0):
    T = (lmax + 1) * (lmax + 2) // 2
    a = np.zeros(T)
    a[0] = radius * np.sqrt(4.0 * np.pi)
    return a, np.zeros(T)


def perturbed_shape(lmax, seed, axis_range=(0.6, 1.0), amp=0.05):
    """Ellipsoid base (axes ~ U[axis_range]) + random l>=2 perturbation ~ N(0, (amp l^-2)^2);
    re-drawn until star-shaped with r > 0.3 (SURVEY §8d, config 3)."""
    rng = np.random.default_rng(seed)
    for _ in range(100):
        axes = rng.uniform(axis_range[0], axis_range[1], size=3)
        axes[0] = axis_range[1]
        a, b = project(lmax, ellipsoid_radius(*axes))
        for l in range(2, lmax + 1):
            sig = amp / (l * l)
            for m in range(l + 1):
                a[lm_index(l, m)] += rng.normal(0, sig)
                if m > 0:
                    b[lm_index(l, m)] += rng.normal(0, sig)
        th = np.linspace(0.01, np.pi - 0.01, 90)[:, None]
        ph = np.linspace(0, 2 * np.pi, 180, endpoint=False)[None, :]
        if evaluate(lmax, a, b, th, ph).min() > 0.3:
            return a, b
    raise RuntimeError("could not draw a star-shaped perturbed shape")


def random_quaternions(rng, n):
    q = rng.normal(size=(n, 4))
    return q / np.linalg.norm(q, axis=1)[:, None]


# ---------------------------------------------------------------------------------------------
# packings
# ---------------------------------------------------------------------------------------------
def fcc_positions(ncell, nn_dist):
    """FCC lattice, ncell=(nx,ny,nz) cubic cells, nearest-neighbour distance nn_dist."""
    a = nn_dist * np.sqrt(2.0)
    basis = np.array([[0, 0, 0], [0.5, 0.5, 0], [0.5, 0, 0.5], [0, 0.5, 0.5]])
    gx, gy, gz = np.meshgrid(np.arange(ncell[0]), np.arange(ncell[1]), np.arange(ncell[2]), indexing="ij")
    cells = np.stack([gx.ravel(), gy.ravel(), gz.ravel()], axis=1).astype(float)
    pos = (cells[:, None, :] + basis[None, :, :]).reshape(-1, 3) * a
    return pos, np.array(ncell, dtype=float) * a


def cubic_positions(ncell, spacing):
    gx, gy, gz = np.meshgrid(np.arange(ncell[0]), np.arange(ncell[1]), np.arange(ncell[2]), indexing="ij")
    pos = np.stack([gx.ravel(), gy.ravel(), gz.ravel()], axis=1).astype(float) * spacing
    return pos, np.array(ncell, dtype=float) * spacing


# ---------------------------------------------------------------------------------------------
# BASELINE.json configs
# ---------------------------------------------------------------------------------------------
def config1_two_particle(lmax=20, grid=(32, 64), seed=1, random_orient=True, exponent=1.0, k=1e3):
    """configs[0]: two identical SH ellipsoid-like particles, head-on collision."""
    a, b = ellipsoid_shape(lmax)
    rng = np.random.default_rng(seed)
    quat = random_quaternions(rng, 2) if random_orient else np.tile([1.0, 0, 0, 0], (2, 1))
    return dict(name="cfg1_two_particle", lmax=lmax, grid=grid, shapes=[(a, b)], density=1.0,
                shape_id=np.zeros(2, np.int32), x=np.array([[-1.2, 0, 0], [1.2, 0, 0.0]]),
                v=np.array([[1.0, 0, 0], [-1.0, 0, 0]]), quat=quat, angmom=np.zeros((2, 3)),
                box=None, coeff=(k, exponent), walls=[], gravity=(0, 0, 0), skin=0.1, dt=1e-4)


def config2_wall(n_side=10, lmax=20, grid=(32, 64), seed=2, k=1e4, exponent=1.0):
    """configs[1]: n_side^3 mono-shape SH particles settling under gravity onto a wall."""
    a, b = ellipsoid_shape(lmax)
    rng = np.random.default_rng(seed)
    pos, _ = cubic_positions((n_side,) * 3, 2.2)
    pos += np.array([1.1, 1.1, 1.2])
    n = len(pos)
    return dict(name="cfg2_wall_%d" % n, lmax=lmax, grid=grid, shapes=[(a, b)], density=1.0,
                shape_id=np.zeros(n, np.int32), x=pos, v=np.zeros((n, 3)), quat=random_quaternions(rng, n),
                angmom=np.zeros((n, 3)), box=None, coeff=(k, exponent),
                walls=[((0, 0, 0), (0, 0, 1), k, exponent)], gravity=(0, 0, -9.81), skin=0.2, dt=2e-4)


def config_silo(n_layers=16, radius=6.0, lmax=20, grid=(32, 64), seed=4, k=1e4, exponent=1.0):
    """Silo filling: mono-shape SH ellipsoids (semi-axes 1, 0.8, 0.6) on a square lattice of spacing 2.2 inside an
    infinite z-cylinder of the given radius about x = y = 0, settling under gravity onto the floor plane z = 0."""
    a, b = ellipsoid_shape(lmax)
    rng = np.random.default_rng(seed)
    g = np.arange(-radius, radius + 1e-9, 2.2)
    gx, gy = np.meshgrid(g - g.mean(), g - g.mean(), indexing="ij")
    disc = np.stack([gx.ravel(), gy.ravel()], 1)
    disc = disc[np.hypot(disc[:, 0], disc[:, 1]) <= radius - 1.3]
    pos = np.concatenate([np.column_stack([disc, np.full(len(disc), 1.2 + 2.2 * l)]) for l in range(n_layers)])
    n = len(pos)
    return dict(name="silo_%d" % n, lmax=lmax, grid=grid, shapes=[(a, b)], density=1.0,
                shape_id=np.zeros(n, np.int32), x=pos, v=np.zeros((n, 3)), quat=random_quaternions(rng, n),
                angmom=np.zeros((n, 3)), box=None, coeff=(k, exponent), walls=[((0, 0, 0), (0, 0, 1), k, exponent)],
                curved_walls=[("cylinder", (0, 0, 0), (0, 0, 1), radius, k, exponent)], gravity=(0, 0, -9.81),
                skin=0.2, dt=2e-4)


def packing(ncell, lmax, grid, nshapes=8, seed=30, nn_frac=1.9, periodic=True, k=1e3, exponent=1.0,
            vel_sigma=0.05, name="packing", skin=0.05, dt=1e-4):
    """Dense synthetic packing: FCC sites at nn distance nn_frac*Rmax-scale with random orientations and
    polydisperse-shape SH particles (8 perturbed-ellipsoid shapes by default; configs[2..4])."""
    shapes = [perturbed_shape(lmax, seed + s) for s in range(nshapes)] if nshapes > 1 else [ellipsoid_shape(lmax)]
    rng = np.random.default_rng(seed + 1000)
    pos, box = fcc_positions(ncell, nn_frac)
    n = len(pos)
    pos = pos + 0.25 * nn_frac + rng.uniform(-0.03, 0.03, size=pos.shape)
    return dict(name=name, lmax=lmax, grid=grid, shapes=shapes, density=1.0,
                shape_id=rng.integers(0, len(shapes), size=n).astype(np.int32), x=pos,
                v=rng.normal(0, vel_sigma, size=(n, 3)), quat=random_quaternions(rng, n), angmom=np.zeros((n, 3)),
                box=(np.zeros(3), box, (1, 1, 1) if periodic else (0, 0, 0)), coeff=(k, exponent), walls=[],
                gravity=(0, 0, 0), skin=skin, dt=dt)


def shear_box(cfg, rate):
    """configs[3] style: turn a periodic packing into a Lees-Edwards shear box (flow x, gradient y) with the linear
    velocity profile v_x = rate * (y - y_mid) on top of its velocities."""
    cfg = dict(cfg)
    lo, hi, _ = cfg["box"]
    v = np.array(cfg["v"], dtype=float, copy=True)
    v[:, 0] += rate * (np.asarray(cfg["x"])[:, 1] - 0.5 * (lo[1] + hi[1]))
    cfg["v"] = v
    cfg["shear"] = float(rate)
    cfg["name"] = cfg["name"] + "_shear"
    return cfg


def config3_packing(n_target=100000, lmax=30, grid=(48, 96), seed=30):
    """configs[2]: ~100k polydisperse-shape packing, 8 SH shape types, l_max=30."""
    m = max(2, int(round((n_target / 4.0) ** (1.0 / 3.0))))
    return packing((m, m, m), lmax, grid, nshapes=8, seed=seed, name="cfg3_packing_%d_l%d" % (4 * m ** 3, lmax))


def tiled_packing(reps=(3, 3, 3), snapshot=None, vel_sigma=0.02, seed=7, k=1e3, exponent=1.0, skin=0.05, dt=1e-4):
    """Mechanically relaxed dense packing (tools/make_packing.py: compressed under damping with the GPU
    code itself to the jamming density, phi ~ 0.71) replicated periodically reps = (rx, ry, rz) times.
    The committed unit cell holds 4000 particles, 8 SH shape types, l_max = 30, 48x96 quadrature."""
    import os
    if snapshot is None:
        snapshot = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "packing_l30_4000.npz")
    z = np.load(snapshot, allow_pickle=False)
    lmax, grid, nshapes, sseed = int(z["lmax"]), tuple(int(v) for v in z["grid"]), int(z["nshapes"]), int(z["seed"])
    box = np.array(z["box"], dtype=float)
    shapes = [perturbed_shape(lmax, sseed + s) for s in range(nshapes)]
    shifts = np.array([[i, j, k2] for i in range(reps[0]) for j in range(reps[1]) for k2 in range(reps[2])], dtype=float)
    x = (z["x"][None, :, :] + (shifts * box)[:, None, :]).reshape(-1, 3)
    quat = np.tile(z["quat"], (len(shifts), 1))
    sid = np.tile(z["shape_id"], len(shifts)).astype(np.int32)
    n = len(x)
    rng = np.random.default_rng(seed)
    return dict(name="relaxed_packing_%d_l%d" % (n, lmax), lmax=lmax, grid=grid, shapes=shapes, density=1.0,
                shape_id=sid, x=x, v=rng.normal(0, vel_sigma, size=(n, 3)), quat=quat, angmom=np.zeros((n, 3)),
                box=(np.zeros(3), box * np.array(reps, dtype=float), (1, 1, 1)), coeff=(k, exponent), walls=[],
                gravity=(0, 0, 0), skin=skin, dt=dt)


def apply(sim, cfg):
    """Drive a sim object (sh_* call surface) with a config dict."""
    if cfg["box"] is not None:
        sim.set_box(*cfg["box"])
    if cfg.get("shear"):
        sim.set_shear(cfg["shear"])          # Lees-Edwards: flow x, gradient y (before the atoms are created)
    sim.set_quadrature(*cfg["grid"])
    ids = [sim.add_shape(cfg["lmax"], a, b, cfg["density"]) for (a, b) in cfg["shapes"]]
    sim.set_atoms(cfg["shape_id"], cfg["x"], cfg["v"], cfg["quat"], cfg["angmom"])
    k, e = cfg["coeff"]
    for i in ids:
        for j in ids:
            if j >= i:
                sim.pair_coeff(i, j, k, e)
    if cfg.get("dissipation"):
        gn, gt, mu = cfg["dissipation"]
        for i in ids:
            for j in ids:
                if j >= i:
                    sim.pair_dissipation(i, j, gn, gt, mu)
    for (pt, nrm, kw, ew) in cfg["walls"]:
        sim.add_wall(pt, nrm, kw, ew)
    # optional: ("cylinder", point, axis, radius, k, exponent) or ("sphere", centre, radius, k, exponent), in order
    for wall in cfg.get("curved_walls", ()):
        if wall[0] == "cylinder":
            sim.add_cylinder_wall(*wall[1:])
        elif wall[0] == "sphere":
            sim.add_sphere_wall(*wall[1:])
        else:
            raise ValueError("unknown curved wall %r" % (wall[0],))
    sim.set_gravity(cfg["gravity"])
    sim.set_neighbor(cfg["skin"], 1, 1)
    sim.set_timestep(cfg["dt"])
    return ids
