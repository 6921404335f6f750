/* shgpu.h — C ABI of the B200-native SPHERHARM contact hot path (libshgpu.so).
 *
 * What each entry point replaces.  The reference is imaranresearch/LAMMPS-SPHERHARM; the mount
 * /root/reference contains only README.md:1-3 (the heading "SPHERHARM Package to simulate complex
 * shaped granular particles"), so no reference file:line exists to cite beyond that.  The
 * interfaces named below are the LAMMPS style interfaces that BASELINE.json:5 (north_star) says the
 * path sits behind ("atom_style spherharm, pair_style/pair_coeff spherharm, fix nve/sh-style
 * quaternion integrator, wall fixes"); see SURVEY.md §8(b) and INTEGRATION.md for the binding a
 * LAMMPS maintainer would add on the reference side.
 *
 * Conventions: every call returns int (0 = OK, <0 = error; text via sh_last_error; -99 = an internal
 * C++ exception such as std::bad_alloc was caught at the boundary).  No C++ exception crosses the boundary.  The handle is opaque, owned by the library and not thread-safe
 * (one host thread drives one handle, bound to one CUDA device).  Host arrays passed in are copied;
 * arrays passed out are filled into caller-owned buffers of the stated length (NULL = skip).
 * Reals are double, indices int32, tags int64.  Per-atom vectors are AoS rows (n x 3, quaternion
 * n x 4 as w,x,y,z).  There is NO CPU fallback: without a usable CUDA device sh_create fails.
 */
#ifndef SHGPU_H
#define SHGPU_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct sh_ctx sh_ctx;

/* lifecycle ------------------------------------------------------------------------------- */
int sh_create(sh_ctx **h, int device_id);           /* LAMMPS::LAMMPS + package init            */
int sh_destroy(sh_ctx *h);
const char *sh_last_error(const sh_ctx *h);         /* Error::all(FLERR,msg) text               */
int sh_version(void);

/* domain (input: boundary / region / create_box) ---------------------------------------------- */
int sh_set_box(sh_ctx *h, const double lo[3], const double hi[3], const int periodic[3]);

/* atom_style spherharm <lmax> <quadrature> <shape files>  (AtomVec::process_args) ------------- */
int sh_set_quadrature(sh_ctx *h, int n_theta, int n_phi);   /* Gauss-Legendre x uniform-phi     */
int sh_add_shape(sh_ctx *h, int lmax, const double *a_lm, const double *b_lm, double density,
                 int *shape_id_out);                /* a/b index l(l+1)/2+m, real orthonormal SH */
int sh_get_shape_props(const sh_ctx *h, int shape, double *volume, double com[3],
                       double inertia[3], double quat_principal[4], double *rmax, double *rmin);
int sh_get_nodes(const sh_ctx *h, int shape, double *p /*nq x 3*/, double *nds /*nq x 3*/);

/* create_atoms / read_data / set quat  (AtomVec::data_atom, create_atom) ---------------------- */
int sh_set_atoms(sh_ctx *h, int64_t n, const int64_t *tag, const int *shape, const double *x,
                 const double *v, const double *quat, const double *angmom);

/* pair_style spherharm / pair_coeff i j k exponent  (Pair::settings, Pair::coeff) -------------- */
int sh_pair_coeff(sh_ctx *h, int shape_i, int shape_j, double k, double exponent);
/* dissipative contact terms (pair_coeff i j k exponent gamma_n gamma_t mu in shlmp; SURVEY §8f-4; the reference's model is
 * unknown — builder's choice, oracle A.5b): viscous normal damping gamma_n (the normal force never turns attractive) and
 * tangential damping gamma_t capped by Coulomb friction mu |F_n|, both from the relative velocity at the overlap centroid,
 * with the matching torques.  All zero (default) = the purely elastic volume contact. */
int sh_pair_dissipation(sh_ctx *h, int shape_i, int shape_j, double gamma_n, double gamma_t, double mu);
/* fix wall for SH particles (Fix::post_force): plane through point, normal into the domain -- */
int sh_add_wall(sh_ctx *h, const double point[3], const double normal[3], double k,
                double exponent);
/* fix gravity --------------------------------------------------------------------------------- */
int sh_set_gravity(sh_ctx *h, const double g[3]);
/* neighbor <skin> bin / neigh_modify every N check yes|no ------------------------------------- */
int sh_set_neighbor(sh_ctx *h, double skin, int every, int check);
/* timestep ------------------------------------------------------------------------------------- */
int sh_set_timestep(sh_ctx *h, double dt);
/* fix viscous-style damping: after each half kick v *= (1 - dt/2 gamma_lin), angmom *= (1 - dt/2 gamma_rot) */
int sh_set_damping(sh_ctx *h, double gamma_lin, double gamma_rot);

/* run N  (Verlet::setup + Verlet::run: fix nve/sh initial_integrate, neighbor decide/build,
 * Pair::compute, wall post_force, final_integrate) -------------------------------------------- */
int sh_run(sh_ctx *h, int64_t nsteps);
/* one Pair::compute + wall post_force on the current state (run 0) ---------------------------- */
int sh_compute_forces(sh_ctx *h);

/* one timestep in two halves (the multi-rank driver exchanges ghosts in between) ---------------- */
int sh_step_begin(sh_ctx *h, int *rebuild_wanted);   /* initial_integrate + neighbor decide (local)  */
int sh_step_end(sh_ctx *h, int rebuild);             /* ghost poses, build, Pair::compute, final_integrate */
int sh_synchronize(sh_ctx *h);
int sh_mark_begin(sh_ctx *h);                        /* CUDA-event stopwatch on the library stream */
int sh_mark_end(sh_ctx *h, double *seconds);

/* multi-rank (Comm::borders / forward_comm of the atom style's pack_comm / unpack_comm): the last
 * nghost atoms passed to sh_set_atoms are ghosts.  d_idx, d_shift, d_out, d_in are DEVICE pointers;
 * a record is 7 doubles: x + shift (3), quat (4). ------------------------------------------------- */
int sh_set_ghost_count(sh_ctx *h, int64_t nghost);
int sh_pack_atoms(sh_ctx *h, int64_t m, const int *d_idx, const double *d_shift, double *d_out);
int sh_unpack_ghosts(sh_ctx *h, int64_t first, int64_t m, const double *d_in);

/* Multi-GPU behind the C ABI (SURVEY §8b; replaces Comm::exchange / Comm::borders / forward_comm of LAMMPS' CommBrick
 * for this atom style).  One handle = one rank = one GPU; ranks are processes (torchrun / MPI) or threads of one process.
 * Rank 0 calls sh_dd_unique_id (an ncclUniqueId, 128 bytes) and the host distributes it (MPI_Bcast, torch.distributed, a
 * shared variable between threads); every rank then calls sh_dd_init BEFORE sh_set_atoms.  From then on sh_set_box takes
 * the GLOBAL box, sh_set_atoms may be handed all atoms on every rank (each keeps the ones inside its brick), and sh_run /
 * sh_compute_forces are collective: ghost exchange every step, atom migration + border lists on neighbor-rebuild steps,
 * all on the device with NCCL point-to-point inside the library.  pgrid = NULL (or zeros) picks the brick grid.
 * Read-back calls see this rank's atoms: owned first, then ghosts (sh_dd_get_info, sh_get_tags). */
int sh_dd_unique_id(char *id, int cap);
int sh_dd_init(sh_ctx *h, int rank, int nranks, const char *id, const int *pgrid);
int sh_dd_get_info(const sh_ctx *h, int pgrid[3], int brick[3], int64_t *nlocal, int64_t *nghost,
                   int64_t *migrated, int64_t *border_builds);
int sh_get_tags(const sh_ctx *h, int64_t n, int64_t *tags);
/* per-step device times (ms) of the last sh_run when the "step_trace" knob is on (at most 4096 steps); flags: bit 0 the
 * step rebuilt the neighbor list, bit 1 rebuilt the candidate cache, bit 2 remapped it, bit 3 had to grow a device buffer */
int sh_get_step_trace(const sh_ctx *h, int64_t cap, int64_t *nsteps, double *ms, int *flags);
/* fix deform xy + remap v (Lees-Edwards shear, BASELINE configs[3]): flow along x, gradient along y, rate = dvx/dy.
 * Before sh_set_atoms; needs a box periodic in x and y; x is never decomposed. */
int sh_set_shear(sh_ctx *h, double rate);

/* Pair::compute-style offload for a host code that owns the atoms (the drop-in a LAMMPS pair style
 * wrapper uses every step): push x / quat (v, angmom optional; NULL = keep), sh_compute_forces,
 * then read f / torque.  The neighbor list is kept across calls and rebuilt when the skin is
 * exhausted.  Host pointers may be pageable or pinned. ------------------------------------------ */
int sh_put_state(sh_ctx *h, int64_t n, const double *x, const double *v, const double *quat,
                 const double *angmom);
int sh_get_forces(const sh_ctx *h, int64_t n, double *f, double *torque);

/* write_restart / read_restart (AtomVec::pack_restart): binary snapshot of the owned atoms (tag, shape, x, v, quat,
 * angmom) and the box.  Shapes / coefficients / fixes are re-issued by the caller before reading, as in LAMMPS. */
int sh_write_snapshot(const sh_ctx *h, const char *path, int64_t step);
int sh_read_snapshot(sh_ctx *h, const char *path, int64_t *step_out);

/* state read-back (dump / thermo / compute) ---------------------------------------------------- */
int sh_get_natoms(const sh_ctx *h, int64_t *n);
int sh_get_atoms(const sh_ctx *h, int64_t n, double *x, double *v, double *quat, double *angmom,
                 double *f, double *torque);         /* in sh_set_atoms order                    */
int sh_get_pairs(const sh_ctx *h, int64_t cap, int64_t *npairs, int64_t *tag_i, int64_t *tag_j,
                 double *V, double *F, double *tau_i, double *tau_j, double *centroid);
int sh_get_energy(const sh_ctx *h, double *ke_trans, double *ke_rot, double *e_contact);
/* compute pressure / stress (row-major 3x3 sums over this rank): kinetic = sum_i m v v over owned atoms, virial =
 * sum_pairs (x_i - x_j) (x) F_i with pairs that involve a ghost counted half; pressure tensor = (kinetic + virial summed
 * over the ranks) / box volume.  Wall forces are not included. */
int sh_get_stress(const sh_ctx *h, double virial[9], double kinetic[9]);
/* compute stress/atom, pe/atom, contact/atom: per-atom quantities of the first n owned atoms (sh_get_atoms order, row i of
 * each output), from the forces of the last sh_compute_forces / sh_run step (the state sh_get_stress reads).  Sums over
 * every pair (i, j) of atom i:
 *   virial   (n x 9, row-major 3a+b)  mode 0 (LAMMPS compute stress/atom): W_i = sum_j 1/2 (x_i - x_j)_a F_ij,b with the
 *            centre-of-mass separation (periodic / Lees-Edwards image) of sh_get_stress and F_ij the force on i;
 *            mode 1 (contact branch vectors, Love-Weber per-particle stress): W_i = sum_j (x_i - x_c)_a F_ij,b with x_c the
 *            pair's overlap centroid (sh_get_pairs), so a contact's moment goes to the particle whose surface carries it;
 *            a pair with V <= 0 contributes nothing.  In both modes the sum over all owned atoms (and ranks) equals
 *            sh_get_stress's virial up to summation order.  Walls contribute no virial.
 *   kinetic  (n x 9)  m v_a v_b; sums to sh_get_stress's kinetic.
 *   energy   (n)      1/2 sum_j E_ij + wall energy of i; sums to sh_get_energy's e_contact.
 *   contacts (n)      pairs of i with V > 0 (wall contacts are not counted).
 * NULL outputs are skipped; n out of [0, owned atoms] or a mode other than 0 / 1 fails.  Without valid forces the pair
 * and wall parts are zero.  Fixed-order sums: two calls on the same state are bitwise equal, and the call leaves the
 * trajectory untouched.  In-library decomposition: collective (every rank calls it); with newton on the halves held by
 * ghost rows are returned to their owners. */
int sh_get_atom_stress(const sh_ctx *h, int64_t n, int mode, double *virial, double *kinetic, double *energy,
                       int *contacts);
int sh_get_counters(const sh_ctx *h, int64_t *pair_evals, int64_t *nodes_transformed,
                    int64_t *nodes_evaluated, int64_t *nodes_inside, int64_t *neighbor_builds,
                    int64_t *kernel_launches);
/* pair evaluations whose second atom is a ghost (each such pair is also evaluated by the owner rank) */
int sh_get_ghost_pair_evals(const sh_ctx *h, int64_t *ghost_pair_evals);
/* device time (CUDA events on the library's stream) accumulated since sh_reset_timers; seconds_other = the decomposition's
 * communication sections (pack + NCCL + unpack of the ghost exchange and the force return, migration + borders), which
 * include the time spent waiting for slower neighbour ranks ---------- */
int sh_get_timers(const sh_ctx *h, double *seconds_pair, int64_t *pair_launches,
                  double *seconds_neigh, double *seconds_other);
int sh_reset_timers(sh_ctx *h);
/* split pair pipeline: device time of the SH-evaluation kernel, its launches, pairs routed to the fused
 * deep-contact kernel, survivor-pool growths, candidate-cache builds */
/* raw device counters: 0 pairs, 1 nodes transformed, 2 evaluated, 3 inside, 4 pairs with a ghost, 5 evaluated by
 * pair_eval_kernel (the rest of [2] comes from the fused deep-contact kernel) */
int sh_get_counter_raw(const sh_ctx *h, int index, int64_t *value);
int sh_get_split_times(const sh_ctx *h, double *seconds_cull, double *seconds_eval, double *seconds_reduce,
                       double *seconds_deep);
int sh_get_split_stats(const sh_ctx *h, double *seconds_eval, int64_t *eval_launches, int64_t *deep_pairs,
                       int64_t *pool_redos, int64_t *cache_builds);
/* candidate cache of the split pipeline: full builds, device time of builds + remaps, margin level in use, pairs that
 * took the window (slow) path, remaps (cache carried over a neighbor rebuild) */
int sh_get_cache_stats(const sh_ctx *h, int64_t *cache_builds, double *seconds_cache, int *level, int64_t *slow_pairs,
                       int64_t *cache_remaps);
/* device time of sh_run (events on the library's stream bracketing all steps of the call) -------- */
int sh_get_run_time(const sh_ctx *h, double *seconds_last_run, double *seconds_total);

/* tuning knobs of the pair phase; 0 = default.  variant bits: 1 CTA-per-pair full-scan kernel, 2 direction-cell
 * bound off, 4 fused warp-per-pair kernel, 8 candidate cache off, 32 no cache remap on neighbor rebuilds, 16 force the split pipeline (systems with fewer
 * than 16384 pairs default to the fused kernel) -------------------------------------------------- */
int sh_set_pair_tuning(sh_ctx *h, int threads_per_cta, int ctas_per_sm, int variant);

/* named knobs (0 = default): "cull_wpb" warps per CTA of the cached cull kernel (1, 2, 4, 8; default 1); "cull_lpp"
 * lanes per pair in that kernel (16, 32; default 16); "eval_pts" points per lane of pair_eval_kernel (2, 4; default 4);
 * "eval_occ" its minimum CTAs per SM at 2 points (3, 4); "eval_mode" 1 = one block per CTA (default), 2 = persistent
 * chunks; "cache_level" margin level of the candidate cache (-1 adaptive (default), 0..2 = 0.5 / 1 / 2 % of rmax);
 * "cube_n" direction cells per cube-face edge of the per-shape bound tables (8..144, default 144; before sh_add_shape);
 * "sync_rebuild" 1 = sh_run decides neighbor rebuilds from the current step's displacement flag (one host round trip per
 * step) instead of the one-step-ahead prediction (default 0: the host never waits for the device inside sh_run);
 * "peer_exchange" (in-library decomposition, more than one rank; default 1) 1 = the per-step ghost exchange and force
 * return go through NVLink peer memory: the pack kernels store straight into the neighbours' inboxes (CUDA IPC between
 * processes, peer access between rank threads) and a one-warp kernel exchanges sequence flags; 0 = NCCL send/recv;
 * "newton" (in-library decomposition; default 1) 1 = a pair that straddles a rank boundary is evaluated by one rank (chosen
 * from the two tags) and the force / torque on the ghost is returned to its owner every step (reverse communication, 48 B
 * per ghost); 0 = both ranks evaluate it and keep their own half (no return trip);
 * "step_trace" 1 = record a CUDA event per step in sh_run (sh_get_step_trace);
 * "dd_self_ghosts" 1 = (testing) with the decomposition on, periodic dimensions are served by ghost images even when they
 * are not divided, so that one GPU exercises migration, border lists and the ghost exchange against itself */
int sh_set_tuning(sh_ctx *h, const char *key, double value);

/* FP64 FMA-pipe peak microbenchmark (K0): returns measured DFMA flop/s of the device ----------- */
int sh_measure_fp64_peak(sh_ctx *h, double *flops_per_s, double *sm_clock_mhz_est);

#ifdef __cplusplus
}
#endif
#endif
