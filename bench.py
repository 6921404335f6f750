#!/usr/bin/env python
"""bench.py — headline benchmark of the SPHERHARM contact hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # CPU arm (oracle; see below)

Workload at N=1: BASELINE.json configs[2] — "~100k polydisperse-shape packing (8 SH shape types, l_max=30) granular
pour": the mechanically relaxed jammed packing (96,000 particles, 48x96 surface quadrature, periodic box) moving as a
dense flow (bulk velocity + thermal noise), so that the timed steps contain neighbor-list rebuilds and candidate-cache
rebuilds (counted in the line).  A "step" is one full timestep of sh_run (integrate, neighbor decide/build, pair phase,
gather, integrate).  After the warm-up, exactly K = --steps steps are timed as one block on the device (CUDA events on the
library's stream; max over ranks); `ms_per_step` / `value` are that block's mean.  The default K keeps the window above
2 s on a B200.  `--dump-outputs DIR` writes what the last timed step computed as .npy files (see dump_outputs).
`value` = contact-pair evaluations per second with the state resident in HBM.  `e2e` = the same metric through the
Pair::compute-style C-ABI offload with HOST buffers: every step pushes x/quat from pinned host memory (sh_put_state),
runs sh_compute_forces and reads f/torque back.

N>1: ONE periodic packing of ~N x 96k particles, spatially decomposed into N bricks with ghost exchange every step and
migration on rebuild steps ("weak" scaling: fixed work per GPU).  The same run also measures the north-star's STRONG
case, the 1,008,000-particle box, on the N GPUs (`strong_1M`; the N=1 run leaves its number in the system's temporary
directory for the efficiency of later N>1 runs on the same machine).

Reference arm: the reference (imaranresearch/LAMMPS-SPHERHARM) mount holds only a README, so there is no reference
binary or package to install or compile; `--impl reference` times this repo's CPU oracle (oracle/, kind="port") with
all host threads on the SAME workload (same particle count, same config dict), each step a full oracle timestep.
PARITY/BASELINE UNPINNED — it is the builder's restatement, not LAMMPS+MPI.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the source tree as it found it (which may be read-only)

import shpkg  # noqa: E402

# dram__bytes_read.sum + dram__bytes_write.sum per record of pair_eval_kernel, ncu --set full capture
# (profiles/r02_eval_kernel_ncu_summary.txt); algorithmic bytes are 33 per record (32 B record in, 1 B flag out)
EVAL_DRAM_BYTES_PER_RECORD = 33.0
METRIC = "contact_pair_evals_per_s"
UNIT = "pair-evals/s"
DUMP_ATOMS = 1 << 17        # --dump-outputs: every owned atom up to this many, a seeded sample of this many beyond
DUMP_PAIR_ATOMS = 1 << 14   # ... and the pair records (as atom i) of a seeded sample of this many atoms
DUMP_MAX_BYTES = 64 << 20


def f_eval(lmax):
    """SURVEY §8(d) model: 7 flops per (l,m) term + 14 per m + 40 per node."""
    T = (lmax + 1) * (lmax + 2) // 2
    return 7 * T + 14 * (lmax + 1) + 40


def f_eval_executed(lmax):
    """FP64 flops the loop in csrc/device_math.cuh actually executes per node: the l = m term is a load, the l = m+1
    term 1 DMUL + 2 DFMA, every further term 1 DMUL + 3 DFMA; per m>0 the rotation (2 DMUL + 2 DFMA) and 2 DFMA; plus
    sqrt / divide / 3 DMUL per node (counted 40 as in the model)."""
    L = lmax
    T = (L + 1) * (L + 2) // 2
    full = T - (L + 1) - L            # terms with l >= m + 2
    return 7 * full + 5 * L + 6 * L + 4 * (L + 1) + 40


def algorithmic_flops(c, lmax):
    """SURVEY §8(d): flops = 24/transformed node + F_eval(L)/evaluated node + 30/inside node + 200/pair."""
    return 24.0 * c["nodes_transformed"] + f_eval(lmax) * c["nodes_evaluated"] + 30.0 * c["nodes_inside"] + \
        200.0 * c["pair_evals"]


class ClockSampler:
    """One streaming `nvidia-smi -lms 50` process for the duration of the timed region."""
    QUERY = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown," \
            "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown," \
            "clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.25)          # let the first samples land before the timed region starts
        except Exception:
            self.proc = None

    def stop(self):
        rows = []
        if self.proc is not None:
            time.sleep(0.06)
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
            except Exception:
                self.proc.kill()
                out = ""
            for line in out.splitlines():
                parts = [p.strip() for p in line.split(",")]
                if len(parts) >= 7:
                    try:
                        float(parts[0])
                        rows.append(parts)
                    except ValueError:
                        pass
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[0]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[3 + k].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][1]),
                "power_w_max": max(float(r[2]) for r in rows), "samples": len(rows), "reasons": reasons}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def tile_reps(n):
    """Replications (a >= b >= c) of the 4000-particle unit cell closest to n particles."""
    t = max(1.0, n / 4000.0)
    r = max(1, int(round(t ** (1.0 / 3.0))))
    return min(((abs(a * b * c - t), (a, b, c)) for a in (r - 1, r, r + 1) for b in (r - 1, r, r + 1)
                for c in (r - 1, r, r + 1) if a >= 1 and b >= 1 and c >= 1 and a >= b >= c), key=lambda u: u[0])[1]


def make_workload(args, pkg, n_particles=None):
    W = pkg.workloads
    n = n_particles or args.particles
    if args.workload == "relaxed" and (args.lmax, args.ntheta, args.nphi) == (30, 48, 96):
        # relaxed jammed unit cell (4000 particles) tiled periodically to ~n particles; dense flow: bulk + thermal velocity
        cfg = W.tiled_packing(tile_reps(n), vel_sigma=args.vel_sigma)
        cfg["v"] = cfg["v"] + np.array([args.flow, 0.0, 0.0])
        return cfg
    cfg = W.config3_packing(n, lmax=args.lmax, grid=(args.ntheta, args.nphi), seed=30)
    cfg["v"] = cfg["v"] + np.array([args.flow, 0.0, 0.0])
    return cfg


def workload_config(args, n):
    """The `config` object — identical in the GPU arm and the reference arm."""
    kind = ("mechanically relaxed jammed packing (phi~0.71, compressed under damping by this code; 4000-particle "
            "periodic unit cell tiled)") if args.workload == "relaxed" else "jittered FCC-seeded packing (phi~0.56)"
    return {"workload": "BASELINE configs[2]: ~100k polydisperse-shape SH packing, 8 shape types, l_max=%d, periodic, granular "
                        "flow (bulk velocity %g + thermal %g, dt 1e-4, skin 0.05: neighbor list and candidate cache are "
                        "rebuilt inside the timed region); %s" % (args.lmax, args.flow, args.vel_sigma, kind),
            "n_particles": int(n), "lmax": args.lmax, "quadrature": "%dx%d" % (args.ntheta, args.nphi),
            "l2_policy": "inputs larger than L2: the per-step working set (atom SoA, pair list, per-pair / per-entry result "
                         "slots, candidate cache, survivor records: > 300 MB at 96k particles) exceeds the 126 MB L2 and "
                         "is rewritten every step; shape tables are L2/shared-memory resident by design"}


def cpu_oracle_run(args, pkg, steps, warmup, n_particles=None):
    """Oracle (CPU port) with all host threads on the bench workload itself."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py as O
    cores = os.cpu_count() or 1
    W = pkg.workloads
    cfg = make_workload(args, pkg, n_particles)
    o = O.Oracle(threads=cores)
    W.apply(o, cfg)
    o.compute_forces()       # setup (neighbor list + first force evaluation), untimed like the GPU arm
    for _ in range(warmup):
        o.run(1)
    c0 = o.get_counters()
    t0 = time.perf_counter()
    o.run(steps)
    dt = time.perf_counter() - t0
    c1 = o.get_counters()
    pairs = c1["pair_evals"] - c0["pair_evals"]
    n = len(cfg["x"])
    o.close()
    return dict(value=pairs / dt, unit=UNIT, cores=cores, kind="port",
                sample="%s: %d particles, %d step(s) of the bench workload, %d pair evals in %.2f s (oracle, OpenMP %d threads); "
                       "builder's CPU restatement, NOT the reference (LAMMPS+MPI unavailable)"
                       % (cfg["name"], n, steps, pairs, dt, cores),
                particle_steps_per_s=n * steps / dt, ms_per_step=1e3 * dt / steps, n_particles=n)


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return 0
    pkg = shpkg.load()
    # same packing, same particle count as the GPU arm; ~5 s per oracle step on 16 cores, so the step count is bounded
    steps = max(1, min(args.steps, 12))
    warm = min(args.warmup, 1)
    n = len(make_workload(args, pkg)["x"])
    res = cpu_oracle_run(args, pkg, steps, warm)
    line = {"impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, n),
            "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "particle_steps_per_s": res["particle_steps_per_s"], "gpu_launches": 0,
            "steps_timed": steps, "warmup_run": warm,
            "note": "oracle steps are ~5 s each on 16 host threads: %d timed step(s) after %d warm-up step(s) of the SAME "
                    "%d-particle workload" % (steps, warm, n)}
    print(json.dumps(line))
    return 0


class Runner:
    """One engine per rank; with more than one rank the decomposition runs inside libshgpu (sh_dd_*, NCCL in the library)."""

    def __init__(self, pkg, cfg, local, world, tuning=None):
        self.pkg, self.world = pkg, world
        pre = {k: v for k, v in (tuning or {}).items() if k == "cube_n"}
        if world > 1:
            D = pkg.load_decomp()
            self.sim = D.native_engine(pkg, cfg, local, tuning=pre)
        else:
            self.sim = pkg.ShGpu(device=local)
            for k, v in pre.items():
                self.sim.set_tuning(k, v)
            pkg.workloads.apply(self.sim, cfg)
        for k, v in (tuning or {}).items():
            if k != "cube_n":
                self.sim.set_tuning(k, v)

    @property
    def n(self):
        return self.sim.dd_info()["nlocal"]

    def setup(self):
        self.sim.compute_forces()

    def block(self, steps):
        """K steps, device-timed on the library's stream (sh_run brackets its steps with CUDA events); returns seconds."""
        self.sim.run(steps)
        return self.sim.get_run_time()["last"]

    def close(self):
        self.sim.close()


def multi_gpu_check(pkg, local, world, rank):
    """N-GPU forces and a short trajectory against ONE GPU on a small snapshot (rank 0 holds both), before any timing."""
    D = pkg.load_decomp()
    W = pkg.workloads
    cfg = W.packing((8, 6, 6), 20, (32, 64), nshapes=4, seed=21, periodic=True, name="mgc", skin=0.03, vel_sigma=0.5, dt=4e-4)
    sim = D.native_engine(pkg, cfg, local)
    sim.compute_forces()
    f0 = D.gather_owned_native(sim, ("f", "torque"))
    sim.run(60)
    x1 = D.gather_owned_native(sim, ("x",))
    info = sim.dd_info()
    sim.close()
    if rank != 0:
        return None
    g = pkg.ShGpu(device=local)
    W.apply(g, cfg)
    g.compute_forces()
    r0 = g.get_atoms(("f", "torque"))
    g.run(60)
    r1 = g.get_atoms(("x",))
    g.close()
    fs = float(np.abs(r0["f"]).max())
    L = np.asarray(cfg["box"][1]) - np.asarray(cfg["box"][0])
    dx = x1["x"] - r1["x"]
    dx -= L * np.rint(dx / L)
    return {"n_particles": len(cfg["x"]), "force_max_rel_err": float(np.abs(f0["f"] - r0["f"]).max() / fs),
            "torque_max_rel_err": float(np.abs(f0["torque"] - r0["torque"]).max() / fs),
            "x_max_abs_err_after_60_steps": float(np.abs(dx).max()), "border_builds": info["border_builds"],
            "what": "forces of the N-rank decomposed run vs one GPU on the same snapshot, then 60 steps with rebuilds + migration"}


def dump_outputs(sim, pkg, rank, world, outdir):
    """What the timed sh_run computed in its last step, as float64 DIR/<name>.npy: the owned atoms' x, v, quat, angmom,
    f and torque sorted by tag (atom_tag), and on one GPU the per-pair records V, F, tau_i, tau_j and centroid of the pairs
    whose atom i is in a fixed, seeded sample of atoms, sorted by tag pair (pair_tags).  Collective over ranks."""
    at = pkg.load_decomp().gather_owned_native(sim)
    pairs = sim.get_pairs() if world == 1 else None   # several ranks: pairs with ghosts exist on both sides
    if rank != 0:
        return
    n = len(at["tag"])
    rows = np.arange(n) if n <= DUMP_ATOMS else np.sort(np.random.default_rng(0).choice(n, DUMP_ATOMS, replace=False))
    out = {k: at[k][rows] for k in ("x", "v", "quat", "angmom", "f", "torque")}
    out["atom_tag"] = at["tag"][rows]
    if pairs is not None:
        sample = np.random.default_rng(1).choice(at["tag"], min(n, DUMP_PAIR_ATOMS), replace=False)
        keep = np.flatnonzero(np.isin(pairs["tag_i"], sample))
        keep = keep[np.lexsort((pairs["tag_j"][keep], pairs["tag_i"][keep]))]
        out["pair_tags"] = np.stack([pairs["tag_i"][keep], pairs["tag_j"][keep]], axis=1)
        for k in ("V", "F", "tau_i", "tau_j", "centroid"):
            out["pair_" + k] = pairs[k][keep]
    out = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in out.items()}
    total = sum(v.nbytes for v in out.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_MAX_BYTES))
    os.makedirs(outdir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(outdir, k + ".npy"), v)


def timed_blocks(run, args, torch, dist, use_dist, min_window, max_blocks):
    """Repeat the K-step block until the measured window is >= min_window; per block the max over ranks."""
    def barrier():
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()
    times = []
    total = 0.0
    while True:
        barrier()
        s = run.block(args.steps)
        t = torch.tensor([s], dtype=torch.float64, device="cuda")
        if use_dist:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        s = float(t.item())
        times.append(s)
        total += s
        if total >= min_window or len(times) >= max_blocks:
            break
    barrier()
    return times


def run_graft(args):
    rank, world, local = dist_env()
    pkg = shpkg.load()
    import torch  # plumbing: device selection, barriers, max-over-ranks
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the SPHERHARM path has no CPU fallback")
    torch.cuda.set_device(local)
    use_dist = world > 1
    dist = None
    if use_dist:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def allsum(vals):
        t = torch.tensor([float(v) for v in vals], dtype=torch.float64, device="cuda")
        if use_dist:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return t.tolist()

    mgc = multi_gpu_check(pkg, local, world, rank) if use_dist else None
    if rank == 0 and mgc is not None:
        assert mgc["force_max_rel_err"] <= 1e-10 and mgc["x_max_abs_err_after_60_steps"] <= 1e-9, mgc

    # ---- main workload (weak scaling across ranks)
    cfg = make_workload(args, pkg, args.particles if args.strong else args.particles * world)
    n_global = len(cfg["x"])
    run = Runner(pkg, cfg, local, world)
    sim = run.sim
    peak = sim.measure_fp64_peak() if rank == 0 else None
    run.setup()
    run.block(max(args.warmup, 3))
    # the first neighbor / cache rebuilds grow buffers (cudaMalloc): keep warming up until two rebuilds have happened
    extra_warm = 0
    while sim.get_counters()["neighbor_builds"] < 3 and extra_warm < 200:
        run.block(10)
        extra_warm += 10
    sim.reset_timers()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()     # before the first barrier: its start-up delay must not sit inside any rank's timed region
    wall0 = time.perf_counter()
    times = timed_blocks(run, args, torch, dist, use_dist, min_window=0.0, max_blocks=1)   # exactly --steps steps
    wall = time.perf_counter() - wall0
    clocks = sampler.stop() if rank == 0 else None
    steps_timed = args.steps
    block_s = times[0]
    if args.dump_outputs:
        dump_outputs(sim, pkg, rank, world, args.dump_outputs)
    cnt = sim.get_counters()
    tim = sim.get_timers()
    st_t, ev_nodes = sim.get_split_times(), sim.get_counter_raw(5)   # per-kernel device times of the timed region
    cache = sim.get_cache_stats()
    spl = sim.get_split_stats()
    dd_info = sim.dd_info()
    # a pair that straddles a brick boundary is evaluated by both ranks: count it once (half on each side)
    pairs_local = cnt["pair_evals"] - 0.5 * sim.get_ghost_pair_evals()
    n_owned = run.n
    pairs_total, psteps_total, nb_total, cb_total = allsum([pairs_local, n_owned * steps_timed, cnt["neighbor_builds"],
                                                            cache["cache_builds"] + cache["cache_remaps"]])
    pairs_per_step = pairs_total / steps_timed

    # ---- e2e: Pair::compute offload through the C-ABI with pinned HOST buffers, copies inside the timed region.
    # The host code owns the atoms in this mode (a LAMMPS pair style calling sh_put_state / sh_compute_forces /
    # sh_get_forces).  Several ranks: the host's own communication layer supplies the ghosts (LAMMPS CommBrick), so every
    # rank drives a plain engine over its owned + ghost atoms (sh_set_ghost_count; forces for the owned atoms only).
    st = sim.get_atoms(("x", "v", "quat", "angmom"))           # owned + ghost atoms of this rank
    nall = len(st["x"])
    if use_dist:
        tags = sim.get_tags()
        info = sim.dd_info()
        lo, hi, per = cfg["box"]
        sub = dict(cfg)
        sub["box"] = (lo, hi, [int(per[d] and info["pgrid"][d] == 1) for d in range(3)])
        sub["shape_id"] = np.asarray(cfg["shape_id"])[tags - 1]
        sub.update(x=st["x"], v=st["v"], quat=st["quat"], angmom=st["angmom"])
        run.close()
        sim = pkg.ShGpu(device=local)
        pkg.workloads.apply(sim, sub)
        sim.set_ghost_count(info["nghost"])
        sim.compute_forces()
        cnt_e2e_base = sim.get_counters()["pair_evals"]
        ghost_e2e_base = sim.get_ghost_pair_evals()
    hx = torch.from_numpy(st["x"]).pin_memory()
    hq = torch.from_numpy(st["quat"]).pin_memory()
    hf = torch.empty((nall, 3), dtype=torch.float64).pin_memory()
    ht = torch.empty((nall, 3), dtype=torch.float64).pin_memory()
    e2e_steps = max(20, args.steps)
    for _ in range(3):
        sim.put_state(x=hx.data_ptr(), quat=hq.data_ptr()); sim.compute_forces(); sim.get_forces(hf.data_ptr(), ht.data_ptr())
    c0 = sim.get_counters()["pair_evals"]
    if use_dist:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        hx[:, 0] += args.flow * 1e-4  # the host code owns and advances the positions between calls (the flow of the workload)
        sim.put_state(x=hx.data_ptr(), quat=hq.data_ptr())
        sim.compute_forces()
        sim.get_forces(hf.data_ptr(), ht.data_ptr())
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if use_dist:   # a pair with a ghost is evaluated by both ranks in this (newton off) mode: count it once
        e2e_pairs = (sim.get_counters()["pair_evals"] - c0) * (1.0 - 0.5 * ghost_e2e_base / max(1.0, float(cnt_e2e_base)))
    else:
        e2e_pairs = (sim.get_counters()["pair_evals"] - c0) * (pairs_local / max(1.0, float(cnt["pair_evals"])))
    et = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if use_dist:
        dist.all_reduce(et, op=dist.ReduceOp.MAX)
    e2e_pairs_total = allsum([e2e_pairs])[0]
    e2e_value = e2e_pairs_total / float(et.item())
    sim.close()

    # ---- the same packing through the coarse (24-cell) bound tables: the FP64-heavy variant, for the roofline discussion
    coarse = None
    if rank == 0 and world == 1 and not args.no_extras:
        r2 = Runner(pkg, cfg, local, 1, tuning={"cube_n": 24})
        r2.setup(); r2.block(5); r2.sim.reset_timers()
        t_coarse = r2.block(args.steps)
        c2, t2, s2 = r2.sim.get_counters(), r2.sim.get_timers(), r2.sim.get_split_times()
        fl2 = algorithmic_flops(c2, args.lmax)
        coarse = {"cube_n": 24, "ms_per_step": 1e3 * t_coarse / args.steps,
                  "evaluated_nodes_per_pair": c2["nodes_evaluated"] / max(1, c2["pair_evals"]),
                  "pair_phase_tflops": fl2 / max(t2["seconds_pair"], 1e-12) / 1e12,
                  "pair_phase_frac": fl2 / max(t2["seconds_pair"], 1e-12) / peak["flops_per_s"],
                  "eval_kernel_frac": f_eval(args.lmax) * float(r2.sim.get_counter_raw(5)) / max(s2["eval"], 1e-12) / peak["flops_per_s"],
                  "note": "same packing, same decisions, 24 instead of 144 direction cells per cube-face edge: ~4x more series "
                          "evaluations, a higher FP64 fraction and a SLOWER step; the default trades FP64 work for table look-ups"}
        r2.close()

    # ---- strong scaling: the 1,008,000-particle box on the N GPUs of this run
    strong = None
    if not args.no_extras and not args.strong and args.workload == "relaxed":
        strong = strong_case(args, pkg, torch, dist, use_dist, local, world, rank, allsum)

    if rank == 0:
        flops = algorithmic_flops(cnt, args.lmax)
        pair_s = tim["seconds_pair"]
        peak_tf = peak["flops_per_s"] / 1e12
        T = (args.lmax + 1) * (args.lmax + 2) // 2
        slots = 12.0 * cnt["nodes_transformed"] + (4 * T + 10 * (args.lmax + 1) + 30) * cnt["nodes_evaluated"] + 15.0 * cnt["nodes_inside"]
        # The pair phase is cull / evaluate / reduce (+ the fused kernel on deep contacts, + cache builds).  The roofline
        # object describes the FP64-bound kernel, pair_eval_kernel: algorithmic flops = F_eval(L) per record it evaluated
        # (SURVEY §8d model; the flops the loop executes are reported beside it), over its own CUDA-event time.
        ev_s = max(st_t["eval"], 1e-12)
        ev_flops, ev_flops_exec = f_eval(args.lmax) * float(ev_nodes), f_eval_executed(args.lmax) * float(ev_nodes)
        achieved = ev_flops / ev_s / 1e12
        launches = max(1, tim["pair_launches"])
        kshare = {k: v / max(pair_s, 1e-12) for k, v in st_t.items()}
        kshare["cache_build"] = cache["seconds_cache"] / max(pair_s, 1e-12)
        phase_tf = flops / max(pair_s, 1e-12) / 1e12
        roofline = {"bound": "fp64", "kernel": "pair_eval_kernel", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                    "frac": achieved / peak_tf,
                    "frac_uses": "SURVEY §8(d) model flops (F_eval = %d per evaluated node at l_max=%d); executed FP64 flops are %d per "
                                 "node -> achieved_executed" % (f_eval(args.lmax), args.lmax, f_eval_executed(args.lmax)),
                    "achieved_executed": ev_flops_exec / ev_s / 1e12, "frac_executed": ev_flops_exec / ev_s / 1e12 / peak_tf,
                    "traffic": EVAL_DRAM_BYTES_PER_RECORD * float(ev_nodes) / launches,
                    "traffic_source": "ncu capture r02 (profiles/), %.1f B/record" % EVAL_DRAM_BYTES_PER_RECORD,
                    "eval_kernel_avg_launch_ms": 1e3 * ev_s / launches,
                    "eval_kernel_flops_per_launch": ev_flops / launches,
                    "peak_source": "K0 DFMA microbenchmark run in this process (MEASURED_PEAKS.json has no FP64 entry); "
                                   "nominal 148 SM x 64 lanes x 2 x 1.965 GHz = 37.2 TFLOP/s",
                    "frac_of_nominal": achieved / 37.2,
                    "pair_phase": {"achieved_tflops": phase_tf, "frac": phase_tf / peak_tf, "ms_per_step": 1e3 * pair_s / steps_timed,
                                   "kernel_ms_per_step": {k: 1e3 * v / steps_timed for k, v in st_t.items()},
                                   "kernel_share_of_phase": kshare,
                                   "pipe_slot_frac": slots * 2.0 / max(pair_s, 1e-12) / peak["flops_per_s"],
                                   "note": "with the proven 144-cell bound tables only ~4 nodes per pair reach the FP64 series "
                                           "(r01: 22), so the phase is no longer FP64-bound: cull and reduce are latency / issue "
                                           "bound FP32 + integer kernels; see coarse_tables for the FP64-heavy variant"},
                    "coarse_tables": coarse,
                    "pair_phase_share_of_step": pair_s / max(sum(times), 1e-12),
                    "evaluated_nodes_per_pair": cnt["nodes_evaluated"] / max(1, cnt["pair_evals"]),
                    "candidate_nodes_per_pair": cnt["nodes_transformed"] / max(1, cnt["pair_evals"]),
                    "inside_nodes_per_pair": cnt["nodes_inside"] / max(1, cnt["pair_evals"])}
        cpu = cpu_oracle_run(args, pkg, 1, 0) if (world == 1 and not args.no_cpu) else None
        line = {"metric": METRIC, "value": pairs_per_step * args.steps / block_s, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "warmup_steps_run": max(args.warmup, 3) + extra_warm, "ms_per_step": 1e3 * block_s / args.steps, "higher_is_better": True,
                "scaling": "strong" if args.strong else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": workload_config(args, n_global),
                "timing": {"steps_timed": steps_timed, "window_s": block_s, "wall_ms_per_step": 1e3 * wall / steps_timed,
                           "rule": "one device-timed block of exactly --steps steps after the warm-up (max over ranks); "
                                   "ms_per_step and value are its mean"},
                "decomposition": "single GPU" if world == 1 else
                                 "%s bricks inside libshgpu (sh_dd_*): NCCL ghost exchange every step, device-side migration + "
                                 "border lists on rebuild steps" % "x".join(str(v) for v in dd_info["pgrid"]),
                "particle_steps_per_s": psteps_total / steps_timed * args.steps / block_s,
                "neighbor_builds": int(nb_total), "cache_builds": int(cb_total),
                "rebuilds": {"neighbor_builds_per_rank": cnt["neighbor_builds"], "neighbor_build_ms_each": 1e3 * tim["seconds_neigh"] / max(1, cnt["neighbor_builds"]),
                             "cache_builds_per_rank": cache["cache_builds"], "cache_remaps_per_rank": cache["cache_remaps"], "cache_build_or_remap_ms_each": 1e3 * cache["seconds_cache"] / max(1, cache["cache_builds"] + cache["cache_remaps"]),
                             "steps_timed": steps_timed, "cache_margin_level": cache["level"], "slow_path_pairs": cache["slow_pairs"],
                             "deep_pairs": spl["deep_pairs"], "pool_grows": spl["pool_grows"]},
                "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(nall * 7 * 8),
                        "d2h_bytes_per_step": int(nall * 6 * 8), "steps": e2e_steps,
                        "path": "sh_put_state(x,quat pinned host) + sh_compute_forces + sh_get_forces(f,torque pinned host)"},
                "gpu_launches": int(cnt["kernel_launches"]),
                "roofline": roofline}
        if strong is not None:
            line["strong_1M"] = strong
        if mgc is not None:
            line["multi_gpu_check"] = mgc
        line["migrated_atoms_per_rank"] = dd_info["migrated"]
        line["comm_ms_per_step"] = 1e3 * tim["seconds_other"] / steps_timed   # rank 0: exchange sections incl. waiting for neighbours
        line["ghosts_per_rank"] = dd_info["nghost"]
        if cpu:
            line["cpu_baseline"] = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
    if use_dist:
        dist.destroy_process_group()
    return line if rank == 0 else None


def strong_case(args, pkg, torch, dist, use_dist, local, world, rank, allsum):
    """BASELINE configs[3] size: 1,008,000 particles (6x6x7 unit cells), fixed TOTAL size on the N GPUs of this run."""
    import copy
    a = copy.copy(args)
    a.flow = 0.0
    cfg = make_workload(a, pkg, 1008000)
    lo, hi, _ = cfg["box"]
    rate = args.shear_velocity / float(hi[1] - lo[1])       # Lees-Edwards: the box top moves at shear_velocity relative to the bottom
    cfg = pkg.workloads.shear_box(cfg, rate)
    run = Runner(pkg, cfg, local, world)
    run.setup()
    run.block(3)
    run.sim.reset_timers()
    a.steps = 10
    times = timed_blocks(run, a, torch, dist, use_dist, min_window=1.0, max_blocks=20)
    cnt = run.sim.get_counters()
    pairs_local = cnt["pair_evals"] - 0.5 * run.sim.get_ghost_pair_evals()
    steps_timed = len(times) * a.steps
    pairs_total, nb = allsum([pairs_local, cnt["neighbor_builds"]])
    med = float(np.median(times)) / a.steps
    info = run.sim.dd_info()
    tim = run.sim.get_timers()
    spl = run.sim.get_split_times()
    run.close()
    if rank != 0:
        return None
    out = {"n_particles": len(cfg["x"]), "n_gpus": world, "ms_per_step": 1e3 * med, "value": pairs_total / steps_timed / med, "unit": UNIT,
           "steps_timed": steps_timed, "neighbor_builds": int(nb), "scaling": "strong",
           "mean_ms_per_step": 1e3 * sum(times) / steps_timed, "pair_ms_per_step": 1e3 * tim["seconds_pair"] / steps_timed,
           "comm_ms_per_step": 1e3 * tim["seconds_other"] / steps_timed, "neigh_ms_per_step": 1e3 * tim["seconds_neigh"] / steps_timed,
           "kernel_ms_per_step": {k: 1e3 * v / steps_timed for k, v in spl.items()},
           "shear_rate": rate, "decomposition": "x".join(str(v) for v in info["pgrid"]), "ghosts_per_rank": info["nghost"],
           "workload": "BASELINE configs[3]: the bench packing tiled 6x6x7 (1,008,000 particles) as a periodic SHEAR box: Lees-Edwards "
                       "images (sh_set_shear; flow x, gradient y, linear velocity profile, box top moving at %g relative to the bottom) "
                       "+ thermal %g; neighbor and cache rebuilds inside the timed region" % (args.shear_velocity, args.vel_sigma)}
    path = os.path.join(tempfile.gettempdir(), "spherharm_bench_strong_1M_n1.json")
    if world == 1:
        try:
            with open(path, "w") as f:
                json.dump(out, f)
        except OSError:
            pass
        out["efficiency_vs_1gpu"] = 1.0
    else:
        try:
            one = json.load(open(path))
            out["one_gpu_ms_per_step"] = one["ms_per_step"]
            out["one_gpu_source"] = "earlier N=1 run on this machine (%s)" % path
        except Exception:
            one = None
            try:
                one = json.load(open(os.path.join(ROOT, "profiles", "r02_strong_1M_1gpu.json")))
                out["one_gpu_ms_per_step"] = one["ms_per_step"]
                out["one_gpu_source"] = "committed one-GPU run profiles/r02_strong_1M_1gpu.json (no N=1 run in this session)"
            except Exception:
                one = None
        out["efficiency_vs_1gpu"] = (one["ms_per_step"] / (world * out["ms_per_step"])) if one else None
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000, help="timed steps (one device-timed block)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="graft", choices=["graft", "reference"])
    ap.add_argument("--particles", type=int, default=100000)
    ap.add_argument("--workload", default="relaxed", choices=["relaxed", "lattice"],
                    help="relaxed: committed jammed unit cell tiled periodically; lattice: jittered FCC sites")
    ap.add_argument("--lmax", type=int, default=30)
    ap.add_argument("--ntheta", type=int, default=48)
    ap.add_argument("--nphi", type=int, default=96)
    ap.add_argument("--flow", type=float, default=15.0, help="bulk flow velocity along x (granular pour)")
    ap.add_argument("--shear-velocity", type=float, default=15.0, help="strong_1M case: velocity of the box top relative to the bottom")
    ap.add_argument("--vel-sigma", type=float, default=0.02, help="thermal velocity on top of the flow")
    ap.add_argument("--strong", action="store_true", help="N>1: keep the TOTAL particle count at --particles (strong scaling)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the coarse-table comparison and the 1M strong-scaling case")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl != "graft":
        ap.error("--dump-outputs applies to the CUDA path (--impl graft)")
    if args.warmup < 3 and args.impl == "graft":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    # stdout carries exactly ONE line, the JSON: anything a library prints on fd 1 meanwhile (NCCL's version banner when the
    # communicator inside libshgpu comes up) goes to stderr
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        line = run_graft(args)
    except BaseException:
        # one rank failing must not leave the others waiting in a collective until the driver's timeout
        import traceback
        traceback.print_exc()
        sys.stderr.flush()
        os._exit(1)
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)
    if line is not None:
        print(json.dumps(line), flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
