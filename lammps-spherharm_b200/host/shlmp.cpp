// shlmp.cpp — host front-end: runs a LAMMPS input script (the SPHERHARM subset, SURVEY §8b) on
// libshgpu.so.  It mirrors the reference's style interfaces for this path — AtomVec (atom_style
// spherharm), Pair (pair_style spherharm: settings / coeff / init_style / compute), Fix (nve/sh,
// wall/spherharm, gravity, viscous: init / initial_integrate / post_force / final_integrate are all
// executed on the device inside sh_run) — with the same command names, argument meaning and
// "ERROR: ... (file:line)" behaviour.  Reference sources: NOT IN MOUNT (README only).
//
// Supported commands: units dimension newton comm_modify atom_modify log echo (accepted, no effect);
// atom_style spherharm <lmax> <n_theta> <n_phi> <shapefile>... ; boundary ; region <id> block ... ;
// create_box <ntypes> <region> ; create_atoms <type> single x y z ; read_data <file> ; mass/density via
// `set type <t> density <rho>` ; set atom <id> quat a b c theta | quat/random <seed> ; velocity all set
// vx vy vz ; velocity <id> set ... ; pair_style spherharm ; pair_coeff i j k exponent [gamma_n gamma_t mu] ; fix <id> <grp>
// nve/sh | wall/spherharm <xplane|yplane|zplane> <pos> <k> <exponent> [hi] | gravity <g> vector x y z |
// viscous <gamma> ; neighbor <skin> bin ; neigh_modify every N [check yes|no] ; timestep ; thermo N ;
// compute <id> all stress/atom NULL [ke] [pair] [virial] [branch center|centroid] | pe/atom | contact/atom ;
// dump <id> all custom N <file> <columns> (id type x y z vx vy vz qw qx qy qz fx fy fz tqx tqy tqz angmomx angmomy angmomz
// c_ID c_ID[k]) ; run N ; write_restart <file> ; read_restart <file> ; print "..." ;
// fix <id> <grp> deform N xy erate <rate> remap v   (Lees-Edwards shear: flow x, gradient y)
//
// compute stress/atom gives LAMMPS's 6-vector -(K + W) (xx yy zz xy xz yz; K = m v v, W the per-atom pair virial of
// sh_get_atom_stress) in stress x volume units.  `branch centroid` (a shlmp extension) takes W from the contact branch
// vectors (particle centre to overlap centroid, the granular-mechanics per-particle stress) instead of the LAMMPS
// centre-to-centre halves.
//
// shlmp -gpus N: N ranks = N threads of this process, one GPU each, every rank interprets the script (as MPI ranks do in
// LAMMPS); the domain decomposition, ghost exchange and migration run inside libshgpu (sh_dd_*, NCCL); rank 0 prints
// thermo output and writes the dumps from the state gathered over the ranks.
//
// Shape file: text rows `l m a_lm b_lm` (real orthonormal SH, no Condon-Shortley phase; missing rows = 0).
// Data file: LAMMPS-style header (`N atoms`, `T atom types`, `xlo xhi` ...) and an `Atoms` section with
// rows `id type x y z qw qx qy qz` (an optional `Velocities` section: `id vx vy vz`).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <algorithm>
#include <condition_variable>
#include <map>
#include <mutex>
#include <numeric>
#include <random>
#include <thread>
#include <unordered_map>
#include <sstream>
#include <string>
#include <vector>

extern "C" {
#include "../../include/shgpu.h"
}

namespace {

struct Err { std::string msg; };
[[noreturn]] void error_all(const std::string &file, int line, const std::string &m) {
  std::ostringstream o; o << "ERROR: " << m << " (" << file << ":" << line << ")";
  throw Err{o.str()};
}
#define FLERR __FILE__, __LINE__

struct Shlmp;

// ---- atom_style spherharm ---------------------------------------------------------------------
struct AtomVecSpherharm {
  int lmax = -1, n_theta = 0, n_phi = 0;
  std::vector<std::string> shape_files;
  std::vector<double> density;
  // per-atom host staging (AoS), flushed to the device by Shlmp::init()
  std::vector<int64_t> tag; std::vector<int> type;
  std::vector<double> x, v, quat, angmom;
  void process_args(const std::vector<std::string> &a) {
    if (a.size() < 5) error_all(FLERR, "Illegal atom_style spherharm command: need lmax n_theta n_phi shapefile(s)");
    lmax = std::stoi(a[1]); n_theta = std::stoi(a[2]); n_phi = std::stoi(a[3]);
    shape_files.assign(a.begin() + 4, a.end());
    density.assign(shape_files.size(), 1.0);
  }
  void create_atom(int itype, const double *xx) {
    tag.push_back((int64_t)tag.size() + 1); type.push_back(itype);
    for (int d = 0; d < 3; d++) { x.push_back(xx[d]); v.push_back(0); angmom.push_back(0); }
    quat.push_back(1); quat.push_back(0); quat.push_back(0); quat.push_back(0);
  }
  size_t nlocal() const { return tag.size(); }
};

void read_shape_file(const std::string &fn, int lmax, std::vector<double> &a, std::vector<double> &b) {
  std::ifstream f(fn);
  if (!f) error_all(FLERR, "Cannot open shape file " + fn);
  const int T = (lmax + 1) * (lmax + 2) / 2;
  a.assign(T, 0.0); b.assign(T, 0.0);
  std::string line;
  while (std::getline(f, line)) {
    auto h = line.find('#'); if (h != std::string::npos) line.erase(h);
    std::istringstream is(line);
    int l, m; double av, bv;
    if (!(is >> l >> m >> av >> bv)) continue;
    if (l < 0 || m < 0 || m > l) error_all(FLERR, "Bad (l,m) in shape file " + fn);
    if (l > lmax) continue;
    a[l * (l + 1) / 2 + m] = av; b[l * (l + 1) / 2 + m] = bv;
  }
}

// per-atom computes (compute stress/atom, pe/atom, contact/atom), all evaluated by sh_get_atom_stress
struct Compute {
  std::string id;
  enum Style { STRESS, PE, CONTACT } style = STRESS;
  bool ke = true, pair = true;
  int mode = 0;                                   // sh_get_atom_stress mode: 0 centre-to-centre, 1 contact centroid
  int ncols() const { return style == STRESS ? 6 : 0; }   // 0 = per-atom scalar
};

// one dump custom column: an atom attribute, or column `col` of compute `ci` (-1 = its scalar)
struct DumpCol {
  enum Kind { ID, TYPE, X, V, Q, F, TQ, L, COMP } kind = ID;
  int comp = 0, ci = -1, col = -1;
};
const char *kDefaultDumpCols = "id type x y z qw qx qy qz vx vy vz";

struct Dump { std::string file, header; int every = 0; std::vector<DumpCol> cols; };

// the ranks of one shlmp job (threads): a reusable barrier and per-rank slots for gathers / reductions
struct Team {
  int n = 1;
  char uid[128] = {0};
  std::mutex m; std::condition_variable cv; int waiting = 0; long generation = 0;
  bool failed = false;
  struct Part { std::vector<int64_t> tag; std::vector<double> x, v, quat, extra; double e[3] = {0, 0, 0}; };
  std::vector<Part> part;
  void barrier() {
    std::unique_lock<std::mutex> lk(m);
    const long g = generation;
    if (++waiting == n) { waiting = 0; generation++; cv.notify_all(); }
    else cv.wait(lk, [&] { return generation != g || failed; });
  }
  void abort() { std::lock_guard<std::mutex> lk(m); failed = true; cv.notify_all(); }
};

struct Shlmp {
  sh_ctx *h = nullptr;
  bool dry = false;     // -check: parse and validate the script (files, arguments, command order) without a device
  AtomVecSpherharm avec;
  bool box_defined = false, initialised = false, pair_defined = false, nve_defined = false;
  double lo[3] = {0, 0, 0}, hi[3] = {1, 1, 1};
  int periodic[3] = {1, 1, 1};
  std::map<std::string, std::vector<double>> regions;
  struct Coeff { int i, j; double k, e, gn, gt, mu; };
  std::vector<Coeff> coeffs;
  struct Wall { double p[3], n[3], k, e; };
  std::vector<Wall> walls;
  double g[3] = {0, 0, 0}, gamma = 0, skin = 0.1, dt = 1e-4;
  int every = 1, check = 1, thermo = 0;
  int64_t step = 0;
  std::vector<Dump> dumps;
  std::vector<Compute> computes;
  std::string restart_file;
  int rank = 0, nranks = 1;
  Team *team = nullptr;
  double shear_rate = 0.0;
  bool decomposed = false;           // the device order of the atoms is the library's, not the script's: go by tag
  std::unordered_map<int64_t, int> type_of_tag;
  // this rank's owned atoms as last pulled from the device
  std::vector<int64_t> ltag; std::vector<double> lx, lv, lq;
  // per-atom values that the dumps of the current step need beyond x / v / quat, in avec order, `nextra` per atom:
  // f (3), torque (3), angmom (3) when wanted, then the columns of every wanted compute (extra_off[ci], -1 = not pulled)
  std::vector<double> extra;
  int nextra = 0;
  std::vector<int> extra_off;
  enum { EX_F = 0, EX_TQ = 1, EX_L = 2 };
  int ex_off[3] = {-1, -1, -1};

  void ck(int rc) { if (rc != 0) error_all(FLERR, sh_last_error(h)); }
  bool master() const { return rank == 0; }

  // Pair::init_style + AtomVec upload + fixes' init
  void init() {
    if (initialised) return;
    if (avec.lmax < 0) error_all(FLERR, "atom_style spherharm is required");
    if (!box_defined) error_all(FLERR, "Box must be defined before run");
    if (dry) {
      if (!pair_defined) error_all(FLERR, "pair_style spherharm is required");
      for (auto &fn : avec.shape_files) { std::vector<double> a, b; read_shape_file(fn, avec.lmax, a, b); }
      for (size_t i = 0; i < avec.nlocal(); i++)
        if (avec.type[i] < 1 || avec.type[i] > (int)avec.shape_files.size()) error_all(FLERR, "Invalid atom type");
      initialised = true;
      return;
    }
    if (!restart_file.empty() && avec.nlocal() > 0) error_all(FLERR, "read_restart cannot be combined with create_atoms / read_data");
    if (!pair_defined) error_all(FLERR, "pair_style spherharm is required");
    if (nranks > 1) { ck(sh_dd_init(h, rank, nranks, team->uid, nullptr)); decomposed = true; }
    ck(sh_set_box(h, lo, hi, periodic));
    if (shear_rate != 0.0) { ck(sh_set_shear(h, shear_rate)); decomposed = true; }
    if (decomposed && !restart_file.empty()) error_all(FLERR, "read_restart is not supported with -gpus > 1 or fix deform");
    ck(sh_set_quadrature(h, avec.n_theta, avec.n_phi));
    for (size_t s = 0; s < avec.shape_files.size(); s++) {
      std::vector<double> a, b;
      read_shape_file(avec.shape_files[s], avec.lmax, a, b);
      int id;
      ck(sh_add_shape(h, avec.lmax, a.data(), b.data(), avec.density[s], &id));
    }
    std::vector<int> shape(avec.nlocal());
    for (size_t i = 0; i < avec.nlocal(); i++) {
      if (avec.type[i] < 1 || avec.type[i] > (int)avec.shape_files.size()) error_all(FLERR, "Invalid atom type");
      shape[i] = avec.type[i] - 1;
    }
    if (restart_file.empty()) {
      ck(sh_set_atoms(h, (int64_t)avec.nlocal(), avec.tag.data(), shape.data(), avec.x.data(), avec.v.data(), avec.quat.data(), avec.angmom.data()));
    } else {   // read_restart: atoms, box and step come from the snapshot
      int64_t st = 0, n = 0;
      ck(sh_read_snapshot(h, restart_file.c_str(), &st));
      step = st;
      ck(sh_get_natoms(h, &n));
      avec.tag.resize(n); avec.type.assign(n, 1); avec.x.resize(3 * n); avec.v.resize(3 * n); avec.quat.resize(4 * n); avec.angmom.resize(3 * n);
      for (int64_t i = 0; i < n; i++) avec.tag[i] = i + 1;
    }
    for (auto &c : coeffs) { ck(sh_pair_coeff(h, c.i - 1, c.j - 1, c.k, c.e)); if (c.gn > 0 || c.gt > 0) ck(sh_pair_dissipation(h, c.i - 1, c.j - 1, c.gn, c.gt, c.mu)); }
    for (auto &w : walls) ck(sh_add_wall(h, w.p, w.n, w.k, w.e));
    ck(sh_set_gravity(h, g));
    ck(sh_set_damping(h, gamma, gamma));
    ck(sh_set_neighbor(h, skin, every, check));
    ck(sh_set_timestep(h, dt));
    for (size_t i = 0; i < avec.nlocal(); i++) type_of_tag[avec.tag[i]] = avec.type[i];
    initialised = true;
  }
  // which per-atom values beyond x / v / quat the given dumps need: fills ex_off / extra_off / nextra
  void plan_extra(const std::vector<const Dump *> &due) {
    bool want[3] = {false, false, false};
    std::vector<bool> wc(computes.size(), false);
    for (auto *d : due)
      for (auto &c : d->cols) {
        if (c.kind == DumpCol::F) want[EX_F] = true;
        else if (c.kind == DumpCol::TQ) want[EX_TQ] = true;
        else if (c.kind == DumpCol::L) want[EX_L] = true;
        else if (c.kind == DumpCol::COMP) wc[c.ci] = true;
      }
    nextra = 0;
    for (int k = 0; k < 3; k++) { ex_off[k] = want[k] ? nextra : -1; nextra += want[k] ? 3 : 0; }
    extra_off.assign(computes.size(), -1);
    for (size_t ci = 0; ci < computes.size(); ci++)
      if (wc[ci]) { extra_off[ci] = nextra; nextra += std::max(1, computes[ci].ncols()); }
  }
  // the planned extra values of this rank's first nl owned atoms (device order), nextra per atom.  sh_get_atom_stress is
  // collective in a decomposed run: every rank gets here with the same plan.
  std::vector<double> local_extra(int64_t nl) {
    std::vector<double> out((size_t)nl * nextra);
    if (nextra == 0) return out;
    std::vector<double> a3[3];
    for (int k = 0; k < 3; k++) if (ex_off[k] >= 0) a3[k].resize(3 * nl);
    if (nl && (ex_off[EX_F] >= 0 || ex_off[EX_TQ] >= 0 || ex_off[EX_L] >= 0))
      ck(sh_get_atoms(h, nl, nullptr, nullptr, nullptr, ex_off[EX_L] >= 0 ? a3[EX_L].data() : nullptr,
                      ex_off[EX_F] >= 0 ? a3[EX_F].data() : nullptr, ex_off[EX_TQ] >= 0 ? a3[EX_TQ].data() : nullptr));
    for (int k = 0; k < 3; k++)
      if (ex_off[k] >= 0) for (int64_t i = 0; i < nl; i++) for (int d = 0; d < 3; d++) out[(size_t)nextra * i + ex_off[k] + d] = a3[k][3 * i + d];
    for (int mode = 0; mode < 2; mode++) {
      bool any = false;
      for (size_t ci = 0; ci < computes.size(); ci++) any = any || (extra_off[ci] >= 0 && computes[ci].mode == mode);
      if (!any) continue;
      std::vector<double> W((size_t)9 * nl), K((size_t)9 * nl), E(nl);
      std::vector<int> C(nl);
      ck(sh_get_atom_stress(h, nl, mode, W.data(), K.data(), E.data(), C.data()));
      for (size_t ci = 0; ci < computes.size(); ci++) {
        const Compute &c = computes[ci];
        if (extra_off[ci] < 0 || c.mode != mode) continue;
        for (int64_t i = 0; i < nl; i++) {
          double *o = &out[(size_t)nextra * i + extra_off[ci]];
          if (c.style == Compute::PE) o[0] = E[i];
          else if (c.style == Compute::CONTACT) o[0] = (double)C[i];
          else {
            static const int comp[6] = {0, 4, 8, 1, 2, 5};   // xx yy zz xy xz yz
            for (int k = 0; k < 6; k++) {
              double s = 0.0;
              if (c.ke) s += K[9 * i + comp[k]];
              if (c.pair) s += W[9 * i + comp[k]];
              o[k] = -s;
            }
          }
        }
      }
    }
    return out;
  }
  // device -> host staging (dump / thermo).  Decomposed runs: every rank pulls its owned atoms, rank 0 merges them by tag
  // into the script-order arrays of avec (and `extra`, as planned by plan_extra).
  void pull_state() {
    if (!decomposed) {
      const int64_t n = (int64_t)avec.nlocal();
      if (n) ck(sh_get_atoms(h, n, avec.x.data(), avec.v.data(), avec.quat.data(), avec.angmom.data(), nullptr, nullptr));
      extra = local_extra(n);
      return;
    }
    int64_t nl = 0, ng = 0;
    ck(sh_dd_get_info(h, nullptr, nullptr, &nl, &ng, nullptr, nullptr));
    const int64_t nall = nl + ng;
    std::vector<int64_t> tg(nall); std::vector<double> x(3 * nall), v(3 * nall), q(4 * nall);
    if (nall) { ck(sh_get_tags(h, nall, tg.data())); ck(sh_get_atoms(h, nall, x.data(), v.data(), q.data(), nullptr, nullptr, nullptr)); }
    Team::Part mine;
    mine.tag.assign(tg.begin(), tg.begin() + nl); mine.x.assign(x.begin(), x.begin() + 3 * nl); mine.v.assign(v.begin(), v.begin() + 3 * nl);
    mine.quat.assign(q.begin(), q.begin() + 4 * nl);
    mine.extra = local_extra(nl);
    if (team) { team->part[rank] = std::move(mine); team->barrier(); }
    if (master()) {
      std::unordered_map<int64_t, size_t> where;
      for (size_t i = 0; i < avec.nlocal(); i++) where[avec.tag[i]] = i;
      extra.assign(avec.nlocal() * nextra, 0.0);
      auto merge = [&](const Team::Part &p) {
        for (size_t k = 0; k < p.tag.size(); k++) {
          const size_t i = where.at(p.tag[k]);
          for (int d = 0; d < 3; d++) { avec.x[3 * i + d] = p.x[3 * k + d]; avec.v[3 * i + d] = p.v[3 * k + d]; }
          for (int d = 0; d < 4; d++) avec.quat[4 * i + d] = p.quat[4 * k + d];
          for (int d = 0; d < nextra; d++) extra[(size_t)nextra * i + d] = p.extra[(size_t)nextra * k + d];
        }
      };
      if (team) for (auto &p : team->part) merge(p); else merge(mine);
    }
    if (team) team->barrier();
  }
  void write_thermo(bool header) {
    double e[3];
    ck(sh_get_energy(h, &e[0], &e[1], &e[2]));
    if (team) {
      for (int d = 0; d < 3; d++) team->part[rank].e[d] = e[d];
      team->barrier();
      if (master()) for (int r = 1; r < nranks; r++) for (int d = 0; d < 3; d++) e[d] += team->part[r].e[d];
      team->barrier();
    }
    if (!master()) return;
    if (header) printf("%10s %16s %16s %16s %16s\n", "Step", "KinEng", "RotKinEng", "E_contact", "TotEng");
    printf("%10lld %16.9g %16.9g %16.9g %16.9g\n", (long long)step, e[0], e[1], e[2], e[0] + e[1] + e[2]);
    fflush(stdout);
  }
  void write_dumps(bool force) {
    std::vector<const Dump *> due;
    for (auto &d : dumps) if (force || (d.every > 0 && step % d.every == 0)) due.push_back(&d);
    if (due.empty()) return;
    plan_extra(due);
    pull_state();
    if (!master()) return;
    std::string line;
    char buf[64];
    for (auto *dp : due) {
      const Dump &d = *dp;
      FILE *f = fopen(d.file.c_str(), step == 0 || force ? (step == 0 ? "w" : "a") : "a");
      if (!f) error_all(FLERR, "Cannot open dump file " + d.file);
      fprintf(f, "ITEM: TIMESTEP\n%lld\nITEM: NUMBER OF ATOMS\n%zu\nITEM: BOX BOUNDS\n", (long long)step, avec.nlocal());
      for (int k = 0; k < 3; k++) fprintf(f, "%.17g %.17g\n", lo[k], hi[k]);
      fprintf(f, "ITEM: ATOMS %s\n", d.header.c_str());
      for (size_t i = 0; i < avec.nlocal(); i++) {
        line.clear();
        for (size_t k = 0; k < d.cols.size(); k++) {
          const DumpCol &c = d.cols[k];
          const double *ex = extra.data() + (size_t)nextra * i;
          switch (c.kind) {
            case DumpCol::ID: snprintf(buf, sizeof buf, "%lld", (long long)avec.tag[i]); break;
            case DumpCol::TYPE: snprintf(buf, sizeof buf, "%d", avec.type[i]); break;
            case DumpCol::X: snprintf(buf, sizeof buf, "%.17g", avec.x[3 * i + c.comp]); break;
            case DumpCol::V: snprintf(buf, sizeof buf, "%.17g", avec.v[3 * i + c.comp]); break;
            case DumpCol::Q: snprintf(buf, sizeof buf, "%.17g", avec.quat[4 * i + c.comp]); break;
            case DumpCol::F: snprintf(buf, sizeof buf, "%.17g", ex[ex_off[EX_F] + c.comp]); break;
            case DumpCol::TQ: snprintf(buf, sizeof buf, "%.17g", ex[ex_off[EX_TQ] + c.comp]); break;
            case DumpCol::L: snprintf(buf, sizeof buf, "%.17g", ex[ex_off[EX_L] + c.comp]); break;
            case DumpCol::COMP: snprintf(buf, sizeof buf, "%.17g", ex[extra_off[c.ci] + std::max(c.col, 0)]); break;
          }
          if (k) line += ' ';
          line += buf;
        }
        line += '\n';
        fputs(line.c_str(), f);
      }
      fclose(f);
    }
  }
  void run(int64_t nsteps) {
    if (dry) { init(); if (shear_rate != 0.0 && !(periodic[0] && periodic[1])) error_all(FLERR, "fix deform xy needs a box periodic in x and y"); printf("check: run %lld with %zu atoms, %zu shape(s), %zu wall(s) OK\n", (long long)nsteps, avec.nlocal(), avec.shape_files.size(), walls.size()); step += nsteps; return; }
    if (!nve_defined && master()) fprintf(stderr, "WARNING: no fix nve/sh defined; atoms are integrated by the device step anyway\n");
    init();
    ck(sh_compute_forces(h));
    write_thermo(true);
    if (step == 0) write_dumps(false);
    int64_t done = 0;
    while (done < nsteps) {
      int64_t chunk = nsteps - done;
      if (thermo > 0) chunk = std::min<int64_t>(chunk, thermo - (step % thermo));
      for (auto &d : dumps) if (d.every > 0) chunk = std::min<int64_t>(chunk, d.every - (step % d.every));
      ck(sh_run(h, chunk));
      done += chunk; step += chunk;
      if (thermo > 0 && step % thermo == 0) write_thermo(false);
      write_dumps(false);
    }
    if (thermo <= 0 || step % thermo) write_thermo(false);
    int64_t pe, nt, ne, ni, nb, kl;
    ck(sh_get_counters(h, &pe, &nt, &ne, &ni, &nb, &kl));
    double sp, sn, so; int64_t pl;
    ck(sh_get_timers(h, &sp, &pl, &sn, &so));
    double rl, rt; ck(sh_get_run_time(h, &rl, &rt));
    if (master()) printf("Loop time of %g on %d GPU%s for %lld steps with %zu atoms\n", rt, nranks, nranks > 1 ? "s" : "", (long long)nsteps, avec.nlocal());
    if (master()) printf("Pair  time (device) %g s in %lld launches | Neigh %g s in %lld builds | pair evals %lld | nodes evaluated %lld inside %lld\n",
           sp, (long long)pl, sn, (long long)nb, (long long)pe, (long long)ne, (long long)ni);
    plan_extra({});
    pull_state();
  }
};

std::vector<std::string> tokenize(const std::string &line) {
  std::vector<std::string> t; std::string cur; bool q = false;
  for (char c : line) {
    if (c == '"') { q = !q; continue; }
    if (!q && c == '#') break;
    if (!q && (c == ' ' || c == '\t' || c == '\r')) { if (!cur.empty()) { t.push_back(cur); cur.clear(); } }
    else cur += c;
  }
  if (!cur.empty()) t.push_back(cur);
  return t;
}

void read_data(Shlmp &S, const std::string &fn) {
  std::ifstream f(fn);
  if (!f) error_all(FLERR, "Cannot open file " + fn);
  std::string line, section;
  long natoms = -1;
  std::getline(f, line);  // title
  while (std::getline(f, line)) {
    auto t = tokenize(line);
    if (t.empty()) continue;
    if (t.size() >= 2 && t[1] == "atoms") { natoms = std::stol(t[0]); continue; }
    if (t.size() >= 3 && t[1] == "atom" && t[2] == "types") continue;
    if (t.size() >= 4 && t[2] == "xlo") { S.lo[0] = std::stod(t[0]); S.hi[0] = std::stod(t[1]); S.box_defined = true; continue; }
    if (t.size() >= 4 && t[2] == "ylo") { S.lo[1] = std::stod(t[0]); S.hi[1] = std::stod(t[1]); continue; }
    if (t.size() >= 4 && t[2] == "zlo") { S.lo[2] = std::stod(t[0]); S.hi[2] = std::stod(t[1]); continue; }
    if (t[0] == "Atoms" || t[0] == "Velocities") { section = t[0]; continue; }
    if (section == "Atoms") {
      if (t.size() < 9) error_all(FLERR, "Incorrect atom format in data file: need id type x y z qw qx qy qz");
      double xx[3] = {std::stod(t[2]), std::stod(t[3]), std::stod(t[4])};
      S.avec.create_atom(std::stoi(t[1]), xx);
      S.avec.tag.back() = std::stoll(t[0]);
      for (int d = 0; d < 4; d++) S.avec.quat[4 * (S.avec.nlocal() - 1) + d] = std::stod(t[5 + d]);
    } else if (section == "Velocities") {
      if (t.size() < 4) error_all(FLERR, "Incorrect velocity format in data file");
      const int64_t id = std::stoll(t[0]);
      for (size_t i = 0; i < S.avec.nlocal(); i++) if (S.avec.tag[i] == id) for (int d = 0; d < 3; d++) S.avec.v[3 * i + d] = std::stod(t[1 + d]);
    }
  }
  if (natoms >= 0 && (long)S.avec.nlocal() != natoms) error_all(FLERR, "Did not assign all atoms correctly");
}

int find_compute(const Shlmp &S, const std::string &id) {
  for (size_t k = 0; k < S.computes.size(); k++) if (S.computes[k].id == id) return (int)k;
  return -1;
}

// compute ID all stress/atom NULL [ke] [pair] [virial] [branch center|centroid] | pe/atom [pair] | contact/atom
void add_compute(Shlmp &S, const std::vector<std::string> &t) {
  if (t.size() < 4) error_all(FLERR, "Illegal compute command");
  if (t[2] != "all") error_all(FLERR, "Could not find compute group ID " + t[2]);
  if (find_compute(S, t[1]) >= 0) error_all(FLERR, "Reuse of compute ID " + t[1]);
  Compute c;
  c.id = t[1];
  const std::string &style = t[3];
  if (style == "stress/atom") {
    if (t.size() < 5) error_all(FLERR, "Illegal compute stress/atom command");
    if (t[4] != "NULL") error_all(FLERR, "Could not find compute stress/atom temperature ID " + t[4]);
    bool which = false, ke = false, pair = false;
    for (size_t k = 5; k < t.size(); k++) {
      if (t[k] == "ke") { ke = true; which = true; }
      else if (t[k] == "pair" || t[k] == "virial") { pair = true; which = true; }
      else if (t[k] == "branch" && k + 1 < t.size() && (t[k + 1] == "center" || t[k + 1] == "centroid")) c.mode = t[++k] == "centroid" ? 1 : 0;
      else error_all(FLERR, "Illegal compute stress/atom command");
    }
    if (which) { c.ke = ke; c.pair = pair; }
    c.style = Compute::STRESS;
  } else if (style == "pe/atom") {
    for (size_t k = 4; k < t.size(); k++) if (t[k] != "pair") error_all(FLERR, "Illegal compute pe/atom command");
    c.style = Compute::PE;
  } else if (style == "contact/atom") {
    if (t.size() > 4) error_all(FLERR, "Illegal compute contact/atom command");
    c.style = Compute::CONTACT;
  } else {
    error_all(FLERR, "Unknown compute style " + style);
  }
  S.computes.push_back(c);
}

// dump ID all custom N file [columns]; without columns the historic default list
void add_dump(Shlmp &S, const std::vector<std::string> &t) {
  if (t.size() < 6) error_all(FLERR, "Illegal dump command");
  if (t[2] != "all") error_all(FLERR, "Could not find dump group ID " + t[2]);
  Dump d;
  d.every = std::stoi(t[4]); d.file = t[5];
  std::vector<std::string> cols(t.begin() + 6, t.end());
  if (cols.empty()) { std::istringstream is(kDefaultDumpCols); for (std::string w; is >> w;) cols.push_back(w); }
  static const std::map<std::string, std::pair<DumpCol::Kind, int>> attrs = {
      {"id", {DumpCol::ID, 0}}, {"type", {DumpCol::TYPE, 0}}, {"x", {DumpCol::X, 0}}, {"y", {DumpCol::X, 1}}, {"z", {DumpCol::X, 2}},
      {"vx", {DumpCol::V, 0}}, {"vy", {DumpCol::V, 1}}, {"vz", {DumpCol::V, 2}}, {"qw", {DumpCol::Q, 0}}, {"qx", {DumpCol::Q, 1}},
      {"qy", {DumpCol::Q, 2}}, {"qz", {DumpCol::Q, 3}}, {"fx", {DumpCol::F, 0}}, {"fy", {DumpCol::F, 1}}, {"fz", {DumpCol::F, 2}},
      {"tqx", {DumpCol::TQ, 0}}, {"tqy", {DumpCol::TQ, 1}}, {"tqz", {DumpCol::TQ, 2}}, {"angmomx", {DumpCol::L, 0}},
      {"angmomy", {DumpCol::L, 1}}, {"angmomz", {DumpCol::L, 2}}};
  for (const std::string &a : cols) {
    DumpCol col;
    auto it = attrs.find(a);
    if (it != attrs.end()) { col.kind = it->second.first; col.comp = it->second.second; }
    else if (a.compare(0, 2, "c_") == 0 && a.size() > 2) {
      std::string name = a.substr(2);
      int idx = -1;
      const size_t br = name.find('[');
      if (br != std::string::npos) {
        if (name.back() != ']' || br + 2 >= name.size()) error_all(FLERR, "Invalid attribute " + a + " in dump custom command");
        const std::string num = name.substr(br + 1, name.size() - br - 2);
        if (num.find_first_not_of("0123456789") != std::string::npos) error_all(FLERR, "Invalid attribute " + a + " in dump custom command");
        idx = std::stoi(num);
        name = name.substr(0, br);
      }
      const int ci = find_compute(S, name);
      if (ci < 0) error_all(FLERR, "Could not find dump custom compute ID: " + name);
      const int nc = S.computes[ci].ncols();
      if (idx < 0 && nc > 0) error_all(FLERR, "Dump custom compute " + name + " does not calculate per-atom vector");
      if (idx >= 0 && nc == 0) error_all(FLERR, "Dump custom compute " + name + " does not calculate per-atom array");
      if (idx >= 0 && (idx < 1 || idx > nc)) error_all(FLERR, "Dump custom compute " + name + " vector is accessed out-of-range");
      col.kind = DumpCol::COMP; col.ci = ci; col.col = idx - 1;
    } else {
      error_all(FLERR, "Invalid attribute " + a + " in dump custom command");
    }
    d.cols.push_back(col);
    d.header += (d.header.empty() ? "" : " ") + a;
  }
  S.dumps.push_back(d);
}

void execute(Shlmp &S, const std::vector<std::string> &t) {
  const std::string &c = t[0];
  auto need = [&](size_t n) { if (t.size() < n) error_all(FLERR, "Illegal " + c + " command"); };
  if (c == "units" || c == "dimension" || c == "comm_modify" || c == "atom_modify" || c == "log" || c == "echo" || c == "thermo_style" ||
      c == "thermo_modify" || c == "processors" || c == "group") return;
  if (c == "newton") { need(2); if (t[1] != "off") fprintf(stderr, "WARNING: newton on requested; this engine always accumulates per owned atom (newton off)\n"); return; }
  if (c == "atom_style") { need(2); if (t[1] != "spherharm") error_all(FLERR, "Unknown atom style " + t[1]); S.avec.process_args(std::vector<std::string>(t.begin() + 1, t.end())); return; }
  if (c == "boundary") { need(4); for (int d = 0; d < 3; d++) S.periodic[d] = (t[1 + d] == "p"); return; }
  if (c == "region") { need(9); if (t[2] != "block") error_all(FLERR, "Only region block is supported"); std::vector<double> v; for (int k = 3; k < 9; k++) v.push_back(std::stod(t[k])); S.regions[t[1]] = v; return; }
  if (c == "create_box") { need(3); auto it = S.regions.find(t[2]); if (it == S.regions.end()) error_all(FLERR, "Create_box region ID does not exist"); for (int d = 0; d < 3; d++) { S.lo[d] = it->second[2 * d]; S.hi[d] = it->second[2 * d + 1]; } S.box_defined = true; return; }
  if (c == "create_atoms") { need(6); if (t[2] != "single") error_all(FLERR, "Only create_atoms <type> single x y z is supported"); double xx[3] = {std::stod(t[3]), std::stod(t[4]), std::stod(t[5])}; S.avec.create_atom(std::stoi(t[1]), xx); return; }
  if (c == "read_data") { need(2); read_data(S, t[1]); return; }
  if (c == "set") {
    need(5);
    if (S.initialised) error_all(FLERR, "set after the first run is not supported");
    if (t[1] == "type" && t[3] == "density") { const int ty = std::stoi(t[2]); if (ty < 1 || ty > (int)S.avec.density.size()) error_all(FLERR, "Invalid type in set command"); S.avec.density[ty - 1] = std::stod(t[4]); return; }
    std::vector<size_t> sel;
    if (t[1] == "atom") { const int64_t id = std::stoll(t[2]); for (size_t i = 0; i < S.avec.nlocal(); i++) if (S.avec.tag[i] == id) sel.push_back(i); }
    else if (t[1] == "group" || t[1] == "type") { for (size_t i = 0; i < S.avec.nlocal(); i++) if (t[1] == "group" || S.avec.type[i] == std::stoi(t[2])) sel.push_back(i); }
    else error_all(FLERR, "Illegal set command");
    if (t[3] == "quat") {
      need(8);
      double ax[3] = {std::stod(t[4]), std::stod(t[5]), std::stod(t[6])}, th = std::stod(t[7]) * M_PI / 180.0;
      const double nn = std::sqrt(ax[0] * ax[0] + ax[1] * ax[1] + ax[2] * ax[2]);
      if (nn == 0) error_all(FLERR, "Invalid rotation axis in set command");
      for (size_t i : sel) { S.avec.quat[4 * i] = std::cos(th / 2); for (int d = 0; d < 3; d++) S.avec.quat[4 * i + 1 + d] = std::sin(th / 2) * ax[d] / nn; }
    } else if (t[3] == "quat/random") {
      std::mt19937_64 rng(std::stoull(t[4])); std::normal_distribution<double> N(0, 1);
      for (size_t i : sel) { double q[4], s2 = 0; for (double &v : q) { v = N(rng); s2 += v * v; } for (int d = 0; d < 4; d++) S.avec.quat[4 * i + d] = q[d] / std::sqrt(s2); }
    } else if (t[3] == "angmom") { need(7); for (size_t i : sel) for (int d = 0; d < 3; d++) S.avec.angmom[3 * i + d] = std::stod(t[4 + d]); }
    else error_all(FLERR, "Illegal set command keyword " + t[3]);
    return;
  }
  if (c == "velocity") {
    need(6);
    if (t[2] != "set") error_all(FLERR, "Only velocity <all|atom-id> set vx vy vz is supported");
    for (size_t i = 0; i < S.avec.nlocal(); i++) if (t[1] == "all" || S.avec.tag[i] == std::stoll(t[1])) for (int d = 0; d < 3; d++) if (t[3 + d] != "NULL") S.avec.v[3 * i + d] = std::stod(t[3 + d]);
    return;
  }
  if (c == "pair_style") { need(2); if (t[1] != "spherharm") error_all(FLERR, "Unknown pair style " + t[1]); S.pair_defined = true; return; }
  if (c == "pair_coeff") {
    need(5);
    if (!S.pair_defined) error_all(FLERR, "Pair_coeff command before pair_style is defined");
    const int nt = (int)S.avec.shape_files.size();
    auto range = [&](const std::string &s, int &a, int &b) { if (s == "*") { a = 1; b = nt; } else { a = b = std::stoi(s); } if (a < 1 || b > nt) error_all(FLERR, "Incorrect args for pair coefficients"); };
    int i0, i1, j0, j1; range(t[1], i0, i1); range(t[2], j0, j1);
    double gn = 0, gt = 0, mu = 0;   // optional: pair_coeff i j k exponent gamma_n gamma_t mu (dissipative contact terms)
    if (t.size() >= 8) { gn = std::stod(t[5]); gt = std::stod(t[6]); mu = std::stod(t[7]); if (gn < 0 || gt < 0 || mu < 0) error_all(FLERR, "Incorrect args for pair coefficients"); }
    else if (t.size() != 5) error_all(FLERR, "Incorrect args for pair coefficients");
    for (int i = i0; i <= i1; i++) for (int j = std::max(i, j0); j <= j1; j++) S.coeffs.push_back({i, j, std::stod(t[3]), std::stod(t[4]), gn, gt, mu});
    return;
  }
  if (c == "fix") {
    need(4);
    const std::string &style = t[3];
    if (style == "nve/sh") { S.nve_defined = true; return; }
    if (style == "wall/spherharm") {
      need(8);
      Shlmp::Wall w{}; const int d = t[4] == "xplane" ? 0 : t[4] == "yplane" ? 1 : t[4] == "zplane" ? 2 : -1;
      if (d < 0) error_all(FLERR, "Illegal fix wall/spherharm command");
      const bool upper = t.size() > 8 && t[8] == "hi";
      w.p[d] = std::stod(t[5]); w.n[d] = upper ? -1.0 : 1.0; w.k = std::stod(t[6]); w.e = std::stod(t[7]);
      S.walls.push_back(w); return;
    }
    if (style == "gravity") { need(9); if (t[5] != "vector") error_all(FLERR, "Only fix gravity <g> vector x y z is supported"); const double gm = std::stod(t[4]); double v[3] = {std::stod(t[6]), std::stod(t[7]), std::stod(t[8])}; const double nn = std::sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]); for (int d = 0; d < 3; d++) S.g[d] = gm * v[d] / nn; return; }
    if (style == "viscous") { need(5); S.gamma = std::stod(t[4]); return; }
    if (style == "deform") {   // fix ID group deform N xy erate R [remap v]: Lees-Edwards shear at engineering rate R
      need(8);
      if (t[5] != "xy" || t[6] != "erate") error_all(FLERR, "Only fix deform N xy erate <rate> remap v is supported");
      if (S.initialised) error_all(FLERR, "fix deform after the first run is not supported");
      S.shear_rate = std::stod(t[7]);
      return;
    }
    error_all(FLERR, "Unknown fix style " + style);
  }
  if (c == "neighbor") { need(2); S.skin = std::stod(t[1]); return; }
  if (c == "neigh_modify") { for (size_t k = 1; k + 1 < t.size(); k += 2) { if (t[k] == "every") S.every = std::stoi(t[k + 1]); else if (t[k] == "check") S.check = t[k + 1] == "yes"; } return; }
  if (c == "timestep") { need(2); S.dt = std::stod(t[1]); if (!(S.dt > 0)) error_all(FLERR, "Illegal timestep command"); if (S.initialised && !S.dry) S.ck(sh_set_timestep(S.h, S.dt)); return; }
  if (c == "thermo") { need(2); S.thermo = std::stoi(t[1]); return; }
  if (c == "compute") { add_compute(S, t); return; }
  if (c == "dump") { add_dump(S, t); return; }
  if (c == "run") { need(2); S.run(std::stoll(t[1])); return; }
  if (c == "write_restart") {
    need(2); S.init();
    if (S.decomposed) error_all(FLERR, "write_restart is not supported with -gpus > 1 or fix deform");
    if (!S.dry) S.ck(sh_write_snapshot(S.h, t[1].c_str(), S.step));
    return;
  }
  if (c == "read_restart") {   // atoms + box from a snapshot; atom_style (shapes) must already be defined
    need(2);
    if (S.avec.lmax < 0) error_all(FLERR, "atom_style spherharm must be defined before read_restart");
    S.restart_file = t[1]; S.box_defined = true;
    return;
  }
  if (c == "print") { need(2); if (S.master()) printf("%s\n", t[1].c_str()); return; }
  error_all(FLERR, "Unknown command: " + c);
}

// one rank: interpret the whole script on its own handle / device
int run_rank(int rank, int nranks, int device, Team *team, const std::vector<std::string> &lines, bool check_only) {
  Shlmp S;
  S.dry = check_only; S.rank = rank; S.nranks = nranks; S.team = team;
  try {
    if (!check_only && sh_create(&S.h, device) != 0) {
      fprintf(stderr, "ERROR: no usable CUDA device %d (libshgpu has no CPU fallback)\n", device);
      if (team) team->abort();
      return 1;
    }
    if (rank == 0) printf("shlmp (SPHERHARM on libshgpu %d)%s\n", sh_version(), nranks > 1 ? ", decomposed over several GPUs" : "");
    std::string acc;
    for (const std::string &line : lines) {
      if (!line.empty() && line.back() == '&') { acc += line.substr(0, line.size() - 1); continue; }
      acc += line;
      auto t = tokenize(acc); acc.clear();
      if (t.empty()) continue;
      execute(S, t);
    }
  } catch (Err &e) {
    fprintf(stderr, "%s\n", e.msg.c_str());
    if (team) team->abort();
    if (S.h) sh_destroy(S.h);
    return 1;
  } catch (std::exception &e) {
    fprintf(stderr, "ERROR: %s\n", e.what());
    if (team) team->abort();
    if (S.h) sh_destroy(S.h);
    return 1;
  }
  if (S.h) sh_destroy(S.h);
  return 0;
}

}  // namespace

int main(int argc, char **argv) {
  std::string infile; int device = 0, ngpus = 1; bool check_only = false;
  for (int k = 1; k < argc; k++) {
    std::string a = argv[k];
    if ((a == "-in" || a == "-i") && k + 1 < argc) infile = argv[++k];
    else if (a == "-device" && k + 1 < argc) device = std::atoi(argv[++k]);
    else if (a == "-gpus" && k + 1 < argc) ngpus = std::atoi(argv[++k]);
    else if (a == "-check") check_only = true;
    else if (a == "-h" || a == "--help") { printf("usage: shlmp -in <input script> [-device N] [-gpus N] [-check]\n"); return 0; }
  }
  if (ngpus < 1 || ngpus > 64) { fprintf(stderr, "ERROR: -gpus must be 1..64\n"); return 1; }
  std::ifstream fin; std::istream *in = &std::cin;
  if (!infile.empty()) { fin.open(infile); if (!fin) { fprintf(stderr, "ERROR: Cannot open input script %s\n", infile.c_str()); return 1; } in = &fin; }
  std::vector<std::string> lines;
  for (std::string line; std::getline(*in, line);) lines.push_back(line);
  if (ngpus == 1 || check_only) return run_rank(0, 1, device, nullptr, lines, check_only);
  Team team;
  team.n = ngpus; team.part.resize(ngpus);
  if (sh_dd_unique_id(team.uid, (int)sizeof team.uid) != 0) { fprintf(stderr, "ERROR: NCCL is not available (libnccl.so.2)\n"); return 1; }
  std::vector<int> rc(ngpus, 0);
  std::vector<std::thread> th;
  for (int r = 0; r < ngpus; r++) th.emplace_back([&, r] { rc[r] = run_rank(r, ngpus, device + r, &team, lines, false); });
  for (auto &t : th) t.join();
  return *std::max_element(rc.begin(), rc.end());
}
