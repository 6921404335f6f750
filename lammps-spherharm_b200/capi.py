"""ctypes binding of libshgpu.so (include/shgpu.h).  Plain pointers and sizes only.

The class mirrors the LAMMPS input-script surface of the SPHERHARM path (SURVEY §8b):
set_box / set_quadrature+add_shape (atom_style spherharm) / set_atoms (create_atoms, set quat) /
pair_coeff (pair_style spherharm) / add_wall / add_cylinder_wall / add_sphere_wall / set_gravity / set_neighbor / set_timestep / run.
No CPU fallback exists: if the CUDA extension is missing or no device is present, this raises.
"""
import ctypes as C
import os
import re

import numpy as np

from . import build as _build

_LIB = None
c_dp = C.POINTER(C.c_double)
c_ip = C.POINTER(C.c_int)
c_lp = C.POINTER(C.c_int64)


class ShGpuError(RuntimeError):
    pass


def header_path():
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "include", "shgpu.h")


def exported_symbols():
    """Names of every function include/shgpu.h declares."""
    txt = open(header_path()).read()
    return sorted(set(re.findall(r"\b(sh_[a-z0-9_]+)\s*\(", txt)) - {"sh_ctx"})


def load_library(build_if_needed=True):
    global _LIB
    if _LIB is None:
        so = _build.build() if build_if_needed else _build.SO
        if not os.path.exists(so):
            raise ShGpuError("libshgpu.so is not built (run __graft_entry__.build()); there is no fallback")
        _LIB = C.CDLL(so)
        _LIB.sh_last_error.restype = C.c_char_p
        _LIB.sh_last_error.argtypes = [C.c_void_p]
    return _LIB


def _d(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


def _p(a, t=c_dp):
    return None if a is None else a.ctypes.data_as(t)


class ShGpu:
    def __init__(self, device=0):
        self.L = load_library()
        self.h = C.c_void_p()
        rc = self.L.sh_create(C.byref(self.h), int(device))
        if rc != 0:
            self.h = None
            raise ShGpuError("sh_create failed (rc=%d): no usable CUDA device; libshgpu has no CPU fallback" % rc)
        self.n = 0
        self.dd = False

    def close(self):
        if getattr(self, "h", None):
            self.L.sh_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise ShGpuError("shgpu: " + self.L.sh_last_error(self.h).decode())

    # ---- configuration ---------------------------------------------------------------------
    def set_box(self, lo, hi, periodic):
        lo, hi = _d(lo), _d(hi)
        per = np.ascontiguousarray(periodic, dtype=np.int32)
        self._ck(self.L.sh_set_box(self.h, _p(lo), _p(hi), _p(per, c_ip)))

    def set_quadrature(self, n_theta, n_phi):
        self._ck(self.L.sh_set_quadrature(self.h, int(n_theta), int(n_phi)))

    def add_shape(self, lmax, a_lm, b_lm, density=1.0):
        a, b = _d(a_lm), _d(b_lm)
        sid = C.c_int(-1)
        self._ck(self.L.sh_add_shape(self.h, int(lmax), _p(a), _p(b), C.c_double(density), C.byref(sid)))
        return sid.value

    def shape_props(self, shape):
        vol, rmax, rmin = C.c_double(), C.c_double(), C.c_double()
        com, inertia, qp = np.zeros(3), np.zeros(3), np.zeros(4)
        rc = self.L.sh_get_shape_props(self.h, int(shape), C.byref(vol), _p(com), _p(inertia), _p(qp),
                                       C.byref(rmax), C.byref(rmin))
        if rc != 0:
            raise ShGpuError("shape id out of range")
        return dict(volume=vol.value, com=com, inertia=inertia, quat_principal=qp, rmax=rmax.value, rmin=rmin.value)

    def nodes(self, shape, nq):
        p, nds = np.zeros((nq, 3)), np.zeros((nq, 3))
        if self.L.sh_get_nodes(self.h, int(shape), _p(p), _p(nds)) != 0:
            raise ShGpuError("shape id out of range")
        return p, nds

    def set_atoms(self, shape, x, v=None, quat=None, angmom=None, tag=None):
        shape = np.ascontiguousarray(shape, dtype=np.int32)
        n = len(shape)
        x, v, quat, angmom = _d(x), _d(v), _d(quat), _d(angmom)
        tag = None if tag is None else np.ascontiguousarray(tag, dtype=np.int64)
        self._ck(self.L.sh_set_atoms(self.h, C.c_int64(n), _p(tag, c_lp), _p(shape, c_ip), _p(x), _p(v), _p(quat),
                                     _p(angmom)))
        self.n = self.refresh_n() if self.dd else n

    def pair_coeff(self, si, sj, k, exponent):
        self._ck(self.L.sh_pair_coeff(self.h, int(si), int(sj), C.c_double(k), C.c_double(exponent)))

    def pair_dissipation(self, si, sj, gamma_n, gamma_t, mu):
        self._ck(self.L.sh_pair_dissipation(self.h, int(si), int(sj), C.c_double(gamma_n), C.c_double(gamma_t), C.c_double(mu)))

    def get_stress(self):
        w, k = np.zeros(9), np.zeros(9)
        self._ck(self.L.sh_get_stress(self.h, _p(w), _p(k)))
        return dict(virial=w.reshape(3, 3), kinetic=k.reshape(3, 3))

    def get_atom_stress(self, mode=0):
        """Per-atom virial (n,3,3), kinetic (n,3,3), energy (n,) and contacts (n,) of the owned atoms (include/shgpu.h
        sh_get_atom_stress).  mode 0: centre-to-centre halves (LAMMPS compute stress/atom); 1: contact branch vectors.
        Collective in a decomposed run: every rank calls it; n = nlocal."""
        n = self.dd_info()["nlocal"] if self.dd else self.n
        w, k, e, c = np.zeros((n, 3, 3)), np.zeros((n, 3, 3)), np.zeros(n), np.zeros(n, dtype=np.int32)
        self._ck(self.L.sh_get_atom_stress(self.h, C.c_int64(n), int(mode), _p(w), _p(k), _p(e), _p(c, c_ip)))
        return dict(virial=w, kinetic=k, energy=e, contacts=c)

    def add_wall(self, point, normal, k, exponent):
        p, nn = _d(point), _d(normal)
        self._ck(self.L.sh_add_wall(self.h, _p(p), _p(nn), C.c_double(k), C.c_double(exponent)))

    def add_cylinder_wall(self, point, axis, radius, k, exponent):
        """Infinite cylindrical container (particles inside): axis through `point` along `axis`, radius `radius`."""
        p, u = _d(point), _d(axis)
        self._ck(self.L.sh_add_cylinder_wall(self.h, _p(p), _p(u), C.c_double(radius), C.c_double(k), C.c_double(exponent)))

    def add_sphere_wall(self, center, radius, k, exponent):
        """Spherical container (particles inside) of centre `center` and radius `radius`."""
        c = _d(center)
        self._ck(self.L.sh_add_sphere_wall(self.h, _p(c), C.c_double(radius), C.c_double(k), C.c_double(exponent)))

    def set_gravity(self, g):
        g = _d(g)
        self._ck(self.L.sh_set_gravity(self.h, _p(g)))

    def set_neighbor(self, skin, every=1, check=1):
        self._ck(self.L.sh_set_neighbor(self.h, C.c_double(skin), int(every), int(check)))

    def set_damping(self, gamma_lin, gamma_rot):
        self._ck(self.L.sh_set_damping(self.h, C.c_double(gamma_lin), C.c_double(gamma_rot)))

    def set_timestep(self, dt):
        self._ck(self.L.sh_set_timestep(self.h, C.c_double(dt)))

    def set_pair_tuning(self, threads_per_cta=0, ctas_per_sm=0, variant=0):
        self._ck(self.L.sh_set_pair_tuning(self.h, int(threads_per_cta), int(ctas_per_sm), int(variant)))

    # ---- execution ---------------------------------------------------------------------------
    def compute_forces(self):
        self._ck(self.L.sh_compute_forces(self.h))

    def run(self, nsteps):
        self._ck(self.L.sh_run(self.h, C.c_int64(nsteps)))

    def put_state(self, x=None, v=None, quat=None, angmom=None):
        """x/v/quat/angmom: C-contiguous float64 (n x 3 / n x 4) host arrays or raw int pointers."""
        def ptr(a):
            if a is None:
                return None
            if isinstance(a, int):
                return C.cast(a, c_dp)
            assert a.dtype == np.float64 and a.flags.c_contiguous
            return a.ctypes.data_as(c_dp)
        self._ck(self.L.sh_put_state(self.h, C.c_int64(self.n), ptr(x), ptr(v), ptr(quat), ptr(angmom)))

    def get_forces(self, f, torque):
        def ptr(a):
            return C.cast(a, c_dp) if isinstance(a, int) else a.ctypes.data_as(c_dp)
        self._ck(self.L.sh_get_forces(self.h, C.c_int64(self.n), ptr(f), ptr(torque)))

    # ---- in-library domain decomposition (NCCL inside libshgpu) -------------------------------------
    @staticmethod
    def dd_unique_id():
        L = load_library()
        buf = C.create_string_buffer(128)
        rc = L.sh_dd_unique_id(buf, 128)
        if rc != 0:
            raise ShGpuError("sh_dd_unique_id failed (rc=%d): NCCL not available" % rc)
        return buf.raw

    def dd_init(self, rank, nranks, uid=None, pgrid=None):
        pg = None if pgrid is None else np.ascontiguousarray(pgrid, dtype=np.int32)
        self._ck(self.L.sh_dd_init(self.h, int(rank), int(nranks), uid, _p(pg, c_ip)))
        self.dd = True

    def dd_info(self):
        pg, br = np.zeros(3, np.int32), np.zeros(3, np.int32)
        v = [C.c_int64() for _ in range(4)]
        self._ck(self.L.sh_dd_get_info(self.h, _p(pg, c_ip), _p(br, c_ip), *[C.byref(t) for t in v]))
        return dict(pgrid=tuple(int(a) for a in pg), brick=tuple(int(a) for a in br), nlocal=v[0].value, nghost=v[1].value,
                    migrated=v[2].value, border_builds=v[3].value)

    def get_tags(self):
        self.refresh_n()
        t = np.zeros(self.n, dtype=np.int64)
        self._ck(self.L.sh_get_tags(self.h, C.c_int64(self.n), _p(t, c_lp)))
        return t

    def get_step_trace(self):
        n = C.c_int64(0)
        self._ck(self.L.sh_get_step_trace(self.h, C.c_int64(0), C.byref(n), None, None))
        ms, fl = np.zeros(n.value), np.zeros(n.value, dtype=np.int32)
        self._ck(self.L.sh_get_step_trace(self.h, C.c_int64(n.value), C.byref(n), _p(ms), _p(fl, c_ip)))
        return ms, fl

    def set_shear(self, rate):
        self._ck(self.L.sh_set_shear(self.h, C.c_double(rate)))
        self.dd = True

    def refresh_n(self):
        """owned + ghost atoms of this rank (changes when the decomposition migrates atoms)"""
        n = C.c_int64(0)
        self.L.sh_get_natoms(self.h, C.byref(n))
        self.n = n.value
        return self.n

    # ---- multi-rank support (decomp.py drives these) ------------------------------------------
    def set_ghost_count(self, nghost):
        self._ck(self.L.sh_set_ghost_count(self.h, C.c_int64(nghost)))

    def step_begin(self):
        flag = C.c_int(0)
        self._ck(self.L.sh_step_begin(self.h, C.byref(flag)))
        return flag.value

    def step_end(self, rebuild):
        self._ck(self.L.sh_step_end(self.h, int(rebuild)))

    def mark_begin(self):
        self._ck(self.L.sh_mark_begin(self.h))

    def mark_end(self):
        s = C.c_double()
        self._ck(self.L.sh_mark_end(self.h, C.byref(s)))
        return s.value

    def synchronize(self):
        self._ck(self.L.sh_synchronize(self.h))

    def pack_atoms(self, m, d_idx_ptr, d_shift_ptr, d_out_ptr):
        """device pointers (ints): gathers x+shift, quat of atoms d_idx[0..m) into d_out (m x 7)."""
        self._ck(self.L.sh_pack_atoms(self.h, C.c_int64(m), C.c_void_p(d_idx_ptr), C.c_void_p(d_shift_ptr),
                                      C.c_void_p(d_out_ptr)))

    def unpack_ghosts(self, first, m, d_in_ptr):
        self._ck(self.L.sh_unpack_ghosts(self.h, C.c_int64(first), C.c_int64(m), C.c_void_p(d_in_ptr)))

    def get_run_time(self):
        a, b = C.c_double(), C.c_double()
        self._ck(self.L.sh_get_run_time(self.h, C.byref(a), C.byref(b)))
        return dict(last=a.value, total=b.value)

    def write_snapshot(self, path, step=0):
        self._ck(self.L.sh_write_snapshot(self.h, str(path).encode(), C.c_int64(step)))

    def read_snapshot(self, path):
        step, n = C.c_int64(0), C.c_int64(0)
        self._ck(self.L.sh_read_snapshot(self.h, str(path).encode(), C.byref(step)))
        self.L.sh_get_natoms(self.h, C.byref(n))
        self.n = n.value
        return step.value

    # ---- read-back ---------------------------------------------------------------------------
    def get_atoms(self, fields=("x", "v", "quat", "angmom", "f", "torque")):
        n = self.refresh_n() if self.dd else self.n
        shapes = dict(x=3, v=3, quat=4, angmom=3, f=3, torque=3)
        out = {k: (np.zeros((n, shapes[k])) if k in fields else None) for k in shapes}
        self._ck(self.L.sh_get_atoms(self.h, C.c_int64(n), _p(out["x"]), _p(out["v"]), _p(out["quat"]),
                                     _p(out["angmom"]), _p(out["f"]), _p(out["torque"])))
        return {k: v for k, v in out.items() if v is not None}

    def get_pairs(self):
        npairs = C.c_int64(0)
        self._ck(self.L.sh_get_pairs(self.h, C.c_int64(0), C.byref(npairs), None, None, None, None, None, None, None))
        m = npairs.value
        ti, tj = np.zeros(m, dtype=np.int64), np.zeros(m, dtype=np.int64)
        V, F, tau_i, tau_j, xc = np.zeros(m), np.zeros((m, 3)), np.zeros((m, 3)), np.zeros((m, 3)), np.zeros((m, 3))
        self._ck(self.L.sh_get_pairs(self.h, C.c_int64(m), C.byref(npairs), _p(ti, c_lp), _p(tj, c_lp), _p(V), _p(F),
                                     _p(tau_i), _p(tau_j), _p(xc)))
        return dict(tag_i=ti, tag_j=tj, V=V, F=F, tau_i=tau_i, tau_j=tau_j, centroid=xc)

    def get_energy(self):
        a, b, c = C.c_double(), C.c_double(), C.c_double()
        self._ck(self.L.sh_get_energy(self.h, C.byref(a), C.byref(b), C.byref(c)))
        return dict(ke_trans=a.value, ke_rot=b.value, e_contact=c.value)

    def get_counters(self):
        v = [C.c_int64() for _ in range(6)]
        self._ck(self.L.sh_get_counters(self.h, *[C.byref(t) for t in v]))
        keys = ("pair_evals", "nodes_transformed", "nodes_evaluated", "nodes_inside", "neighbor_builds",
                "kernel_launches")
        return {k: t.value for k, t in zip(keys, v)}

    def get_ghost_pair_evals(self):
        v = C.c_int64()
        self._ck(self.L.sh_get_ghost_pair_evals(self.h, C.byref(v)))
        return v.value

    def get_timers(self):
        sp, sn, so, nl = C.c_double(), C.c_double(), C.c_double(), C.c_int64()
        self._ck(self.L.sh_get_timers(self.h, C.byref(sp), C.byref(nl), C.byref(sn), C.byref(so)))
        return dict(seconds_pair=sp.value, pair_launches=nl.value, seconds_neigh=sn.value, seconds_other=so.value)

    def get_counter_raw(self, index):
        v = C.c_int64()
        self._ck(self.L.sh_get_counter_raw(self.h, int(index), C.byref(v)))
        return v.value

    def get_split_times(self):
        v = [C.c_double() for _ in range(4)]
        self._ck(self.L.sh_get_split_times(self.h, *[C.byref(t) for t in v]))
        return dict(zip(("cull", "eval", "reduce", "deep"), (t.value for t in v)))

    def get_split_stats(self):
        a, b, c, d, e = C.c_double(), C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64()
        self._ck(self.L.sh_get_split_stats(self.h, C.byref(a), C.byref(b), C.byref(c), C.byref(d), C.byref(e)))
        return dict(seconds_eval=a.value, eval_launches=b.value, deep_pairs=c.value, pool_grows=d.value,
                    cache_builds=e.value)

    def get_cache_stats(self):
        nb, sec, lv, slow, rm = C.c_int64(), C.c_double(), C.c_int(), C.c_int64(), C.c_int64()
        self._ck(self.L.sh_get_cache_stats(self.h, C.byref(nb), C.byref(sec), C.byref(lv), C.byref(slow), C.byref(rm)))
        return dict(cache_builds=nb.value, seconds_cache=sec.value, level=lv.value, slow_pairs=slow.value,
                    cache_remaps=rm.value)

    def set_tuning(self, key, value):
        """Named knobs (include/shgpu.h sh_set_tuning): cull_wpb, eval_pts, cache_level, cube_n."""
        self._ck(self.L.sh_set_tuning(self.h, str(key).encode(), C.c_double(value)))

    def reset_timers(self):
        self._ck(self.L.sh_reset_timers(self.h))

    def measure_fp64_peak(self):
        f, clk = C.c_double(), C.c_double()
        self._ck(self.L.sh_measure_fp64_peak(self.h, C.byref(f), C.byref(clk)))
        return dict(flops_per_s=f.value, sm_clock_mhz_if_64_lanes=clk.value)
