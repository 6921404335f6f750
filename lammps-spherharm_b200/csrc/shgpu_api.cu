// shgpu_api.cu — context, step driver and extern "C" boundary of libshgpu.so (include/shgpu.h).
//
// Host-side step driver = the Verlet::setup / Verlet::run frame of SURVEY §3.1 restricted to the
// SPHERHARM path: integrate_initial -> (neighbor decide/build) -> pair -> wall -> gather ->
// integrate_final, all on one CUDA stream.  There is no CPU compute path: every force, torque,
// neighbor list and integration step is produced by the kernels in this directory.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/shgpu.h"
#include "devbuf.h"
#include "dd_types.h"
#include "neighbor_kernels.cuh"
#include "pair_kernel.cuh"
#include "pair_warp_kernel.cuh"
#include "pair_split_kernels.cuh"
#include "shape_tables.h"
#include "step_kernels.cuh"
#include "atom_stress_kernels.cuh"

using namespace shgpu;

namespace {

struct ShapeDev {
  DevBuf<double> Ap, node;   // node: 6 x nq
  DevBuf<double2> ab, pn;    // pn: packed node records for the pair reduction (DevShape::pn)
  DevBuf<float> row_x, cubew[SH_CACHE_LEVELS];
  DevBuf<float2> cube;       // {ub2, lb2} per direction cell
  DevBuf<float4> pf4;        // FP32 node points
};

}  // namespace

enum { CACHE_INVALID = 0, CACHE_VALID = 1, CACHE_REMAP = 2 };

struct sh_ctx {
  std::string err;
  int device = 0, sm_count = 148;
  cudaStream_t stream = nullptr;
  // domain
  double lo[3] = {-1e30, -1e30, -1e30}, hi[3] = {1e30, 1e30, 1e30};
  int periodic[3] = {0, 0, 0};
  bool box_set = false;
  // shapes
  int n_theta = 32, n_phi = 64;
  std::vector<ShapeTables> shapes;
  std::vector<ShapeDev> shape_dev;
  std::vector<DevShape> shape_host_view;
  DevBuf<DevShape> d_shapes;
  bool shapes_dirty = true;
  int total_terms = 0;
  std::vector<double> pk, pm;  // SH_MAX_SHAPES^2
  std::vector<double> pgn, pgt, pmu;   // dissipation: normal / tangential damping, Coulomb coefficient
  bool dissip = false;
  DevBuf<double> d_pk, d_pm, d_pgn, d_pgt, d_pmu, stress_part;
  bool coeff_dirty = true;
  WallSet walls{};
  double g[3] = {0, 0, 0}, skin = 0.0, dt = 1e-4, gamma_lin = 0.0, gamma_rot = 0.0;
  int neigh_every = 1, neigh_check = 1;
  // atoms
  int64_t n = 0, nghost = 0;   // n = owned + ghost atoms; the last nghost are ghosts (multi-rank)
  int stride = 0;
  DevBuf<double> x, v, q, L, f, tq, c, Rs, c0, wallf, ewall, ke;
  DevBuf<int> shape;
  std::vector<int64_t> tag;          // host mirror of d_tag (owned + ghost order); refreshed lazily
  DevBuf<long long> d_tag;
  bool tags_host_valid = true;
  DevBuf<double> gf;                 // 6 x stride: force / torque accumulated on ghosts (reverse communication)
  double time = 0.0;                 // simulation time (steps x dt), drives the Lees-Edwards offset
  DdCtx dd;                          // in-library domain decomposition (dd_host.cuh)
  // lagged neighbor decision (sh_run): flag of step s-1 = "step s will exceed the skin"
  int *h_lagflag = nullptr;          // pinned: [0..1] prediction ring, [2] skin violations
  cudaEvent_t ev_lag[2] = {nullptr, nullptr};
  int lag_slot = 0; bool lag_pending = false, lag_mode = true, lag_pred_valid = false;
  bool cache_sync_ranks = false;     // candidate-cache rebuilds are decided from the MAX over ranks of the "nearly used up" flag
  int64_t step_index = 0, cache_build_step = -10;
  double cache_time = 0.0;           // simulation time of the last full cache build (Lees-Edwards offset then)
  // optional per-step device timeline of the last sh_run ("step_trace" knob)
  bool step_trace = false;
  std::vector<cudaEvent_t> ev_step;
  std::vector<float> step_ms;
  std::vector<int> step_flags, step_flags_last;   // bit 0 neighbor rebuild, bit 1 cache build, bit 2 cache remap
  // neighbor
  DevBuf<int> cell_of, cell_count, cell_start, cell_fill, cell_atoms, tile_sum, cnt_full, cnt_half, nbr_off, half_off,
      nbr_j, pair_i, pair_j, pair_eij, pair_eji, pair_img, scalars;  // scalars: [0]=scan total [1]=rebuild flag [2]=work counter [3]/[4]=cache exhausted (hard/soft) [8]/[9]=list totals
  DevBuf<double> bbox, slot, pres, stage;
  // split pair pipeline (pair_split_kernels.cuh)
  DevBuf<SurvRec> pool;
  DevBuf<int> pool_kin;
  DevBuf<unsigned char> out_zero;                 // SplitArgs::out_zero; valid only while out_zero_valid
  bool out_zero_valid = false;                     // cleared by a list build and by every pair phase outside run_split_pipeline
  DevBuf<long long> pool_base, pool_cap;
  DevBuf<PdEntry> pd;
  DevBuf<PairHot> cache_hot[2];       // double-buffered: a neighbor rebuild remaps the live cache into the other buffer
  DevBuf<SplitScalars> split_sc;
  DevBuf<EvalPlanDev> eval_plan;
  DevBuf<int> big_list, slow_list, split_flags;   // split_flags: [2]=cache overflow
  DevBuf<int> inpool;                              // node indices proven inside by the cull beyond the inline capacity
  long long h_in_cap = 0;
  std::vector<long long> h_pool_cap;
  unsigned long long *h_pool_count = nullptr;  // pinned scratch for cache builds
  SplitScalars *h_split_sc = nullptr;          // pinned: advisory read-back of the previous pair phase
  int *h_cache_invalid = nullptr;              // pinned
  cudaEvent_t ev_sc = nullptr;                 // recorded after the read-back copies
  bool sc_pending = false;
  int sc_nshape = 0;
  double sec_eval = 0, sec_cull = 0, sec_reduce = 0, sec_deep = 0, sec_cache = 0; int64_t eval_launches = 0;
  std::vector<int> ev2_kind;
  int64_t big_pairs = 0, slow_pairs = 0, pool_grows = 0, cache_builds = 0;
  int cache_level = 0, cache_level_pin = -1;   // margin level of the candidate cache (adaptive unless pinned)
  int64_t cache_age = 0;                       // pair phases since the last cache build
  bool cache_exhausted = false;                // the last invalidation came from the displacement margin
  int cube_n = 0;                              // direction cells per cube-face edge (0 = default)
  int eval_pts = 0, eval_occ = 0, eval_mode = 0;   // pair_eval_kernel: points per lane, min CTAs/SM, 1 = one block per CTA
  long long last_records = 0;                  // records of the previous pair phase (advisory)
  // candidate cache
  DevBuf<unsigned short> cache_pool[2];
  DevBuf<int> old_half_off, old_pair_j, fresh_list;   // pair list before the last rebuild (remap), pairs new to the cache
  int old_nown = 0, cache_cur = 0;
  // cache carry-over across a DECOMPOSED rebuild (atoms are renumbered, ghosts re-created): snapshot of the old atoms
  DevBuf<double> old_c, old_cc0, old_cq0;
  DevBuf<long long> old_tag;
  DevBuf<int> ghost_hash, amap;      // hash of the old ghosts by tag; new atom -> old atom (or -1)
  int old_n = 0, old_stride = 0, ghost_hash_size = 0;
  bool carry = false;
  int64_t cache_remaps = 0, atoms_epoch = 0, cache_epoch = -1;   // epoch: bumped whenever the atom set / order changes
  DevBuf<unsigned long long> cache_count;
  long long cache_cap = 0;
  int cache_state = 0;                 // CACHE_INVALID / CACHE_VALID / CACHE_REMAP
  DevBuf<double> cc0, cq0, drift;
  bool eval_pending = false;
  DevBuf<unsigned long long> counters;
  int npairs = 0, nentries = 0, nrows = 0;   // nrows: atoms with CSR rows (owned; owned + ghost with newton on)
  int slot_stride = 0, pres_stride = 0;
  int *h_pinned = nullptr;  // [0] total/flag scratch
  bool forces_valid = false, list_valid = false;
  int64_t steps_since_build = 0;
  // stats
  int64_t neighbor_builds = 0, kernel_launches = 0;
  std::vector<cudaEvent_t> ev, ev2;  // pairs of (start,stop): whole pair phase / evaluation kernel
  size_t ev_used = 0, ev2_used = 0;
  double sec_pair = 0, sec_neigh = 0, sec_comm = 0, sec_other = 0, sec_run_last = 0, sec_run_total = 0;
  cudaEvent_t run_e0 = nullptr, run_e1 = nullptr;
  int64_t pair_launches = 0;
  // sh_get_atom_stress: per-atom outputs, entry -> pair map, newton-on ghost records (allocated by its first call)
  DevBuf<double> as_vir, as_kin, as_en, as_send, as_recv;
  DevBuf<int> as_cnt, as_epair;
  // tuning
  int tune_threads = 0, tune_ctas_per_sm = 0, tune_variant = 0, tune_cull_wpb = 0, tune_cull_lpp = 0;
};

namespace {

int fail(sh_ctx *h, const std::string &m) { h->err = m; return -1; }
int cuda_fail(sh_ctx *h, const char *where, cudaError_t e) {
  h->err = std::string(where) + ": " + cudaGetErrorString(e);
  return -2;
}
#define CU(call) do { cudaError_t _e = (call); if (_e != cudaSuccess) return cuda_fail(h, #call, _e); } while (0)

inline int cdiv(int64_t a, int b) { return (int)((a + b - 1) / b); }

AtomView view(sh_ctx *h) {
  AtomView A;
  A.x = h->x.p; A.v = h->v.p; A.q = h->q.p; A.L = h->L.p; A.f = h->f.p; A.tq = h->tq.p;
  A.c = h->c.p; A.Rs = h->Rs.p; A.c0 = h->c0.p; A.wallf = h->wallf.p; A.shape = h->shape.p;
  A.cc0 = h->cc0.p; A.cq0 = h->cq0.p;
  A.n = (int)(h->n - h->nghost); A.stride = h->stride;   // kernels over OWNED atoms
  return A;
}
AtomView view_all(sh_ctx *h) { AtomView A = view(h); A.n = (int)h->n; return A; }

int upload_shapes(sh_ctx *h) {
  if (!h->shapes_dirty) return 0;
  const int ns = (int)h->shapes.size();
  h->shape_dev.resize(ns);
  h->shape_host_view.resize(ns);
  try {
    for (int s = 0; s < ns; s++) {
      const ShapeTables &t = h->shapes[s];
      ShapeDev &d = h->shape_dev[s];
      if (d.Ap.p) continue;  // already uploaded
      const int tpad = (t.nterms + 3) / 4 * 4 + 4;   // zero records pad the software-pipelined loop
      d.Ap.ensure(tpad); d.ab.ensure(tpad); d.node.ensure((size_t)6 * t.nq); d.row_x.ensure(t.n_theta);
      CU(cudaMemset(d.Ap.p, 0, tpad * sizeof(double))); CU(cudaMemset(d.ab.p, 0, tpad * sizeof(double2)));
      {
        std::vector<float> rx(t.row_x.begin(), t.row_x.end());
        CU(cudaMemcpy(d.row_x.p, rx.data(), rx.size() * sizeof(float), cudaMemcpyHostToDevice));
        std::vector<float4> pf((size_t)t.nq);
        for (int k = 0; k < t.nq; k++) pf[k] = make_float4((float)t.node_p[0][k], (float)t.node_p[1][k], (float)t.node_p[2][k], 0.0f);
        d.pf4.ensure(pf.size());
        CU(cudaMemcpy(d.pf4.p, pf.data(), pf.size() * sizeof(float4), cudaMemcpyHostToDevice));
        for (int lv = 0; lv < SH_CACHE_LEVELS; lv++) {
          d.cubew[lv].ensure(t.cube_wide2[lv].size());
          CU(cudaMemcpy(d.cubew[lv].p, t.cube_wide2[lv].data(), t.cube_wide2[lv].size() * sizeof(float), cudaMemcpyHostToDevice));
        }
        std::vector<float2> ul(t.cube_ub2.size());
        for (size_t c = 0; c < ul.size(); c++) ul[c] = make_float2(t.cube_ub2[c], t.cube_lb2[c]);
        d.cube.ensure(ul.size());
        CU(cudaMemcpy(d.cube.p, ul.data(), ul.size() * sizeof(float2), cudaMemcpyHostToDevice));
      }
      std::vector<double2> ab(t.nterms);
      for (int k = 0; k < t.nterms; k++) ab[k] = make_double2(t.ah[k], t.bh[k]);
      CU(cudaMemcpy(d.Ap.p, t.Ap.data(), t.nterms * sizeof(double), cudaMemcpyHostToDevice));
      CU(cudaMemcpy(d.ab.p, ab.data(), t.nterms * sizeof(double2), cudaMemcpyHostToDevice));
      for (int e = 0; e < 3; e++) {
        CU(cudaMemcpy(d.node.p + (size_t)e * t.nq, t.node_p[e].data(), t.nq * sizeof(double), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(d.node.p + (size_t)(3 + e) * t.nq, t.node_n[e].data(), t.nq * sizeof(double), cudaMemcpyHostToDevice));
      }
      {
        std::vector<double2> pn((size_t)4 * t.nq);
        for (int k = 0; k < t.nq; k++) {
          pn[4 * (size_t)k] = make_double2(t.node_p[0][k], t.node_p[1][k]);
          pn[4 * (size_t)k + 1] = make_double2(t.node_p[2][k], t.node_n[0][k]);
          pn[4 * (size_t)k + 2] = make_double2(t.node_n[1][k], t.node_n[2][k]);
          pn[4 * (size_t)k + 3] = make_double2(0.0, 0.0);
        }
        d.pn.ensure(pn.size());
        CU(cudaMemcpy(d.pn.p, pn.data(), pn.size() * sizeof(double2), cudaMemcpyHostToDevice));
      }
      DevShape &v = h->shape_host_view[s];
      v.lmax = t.lmax; v.nterms = t.nterms; v.nq = t.nq; v.nchunks = (t.nq + 31) / 32;
      v.rmax = t.rmax; v.rmin = t.rmin; v.rmax2 = t.rmax * t.rmax; v.rmin2 = t.rmin * t.rmin;
      v.mass = t.mass; v.inv_mass = 1.0 / t.mass;
      for (int e = 0; e < 3; e++) { v.inertia[e] = t.inertia[e]; v.com[e] = t.com[e]; }
      for (int r = 0; r < 3; r++) for (int cidx = 0; cidx < 3; cidx++) v.Rp[3 * r + cidx] = t.Rp[r][cidx];
      v.Ap = d.Ap.p; v.ab = d.ab.p;
      v.px = d.node.p; v.py = d.node.p + t.nq; v.pz = d.node.p + 2 * (size_t)t.nq;
      v.nx = d.node.p + 3 * (size_t)t.nq; v.ny = d.node.p + 4 * (size_t)t.nq; v.nz = d.node.p + 5 * (size_t)t.nq;
      v.pn = d.pn.p;
      v.n_theta = t.n_theta; v.n_phi = t.n_phi; v.nterms4 = (t.nterms + 3) / 4 * 4; v.row_x = d.row_x.p; v.cube_ul = d.cube.p; v.cube_n = t.cube_n; v.pad2_ = 0; v.pf4 = d.pf4.p;
      for (int lv = 0; lv < SH_CACHE_LEVELS; lv++) { v.cube_w2[lv] = d.cubew[lv].p; v.cache_delta[lv] = t.cache_delta[lv]; }
    }
    int off = 0;
    for (int s = 0; s < ns; s++) { h->shape_host_view[s].tab_off = off; off += h->shape_host_view[s].nterms4 + 4; }
    h->total_terms = off;
    h->d_shapes.ensure(std::max(ns, 1));
  } catch (std::string &e) { return fail(h, e); }
  if (ns) CU(cudaMemcpy(h->d_shapes.p, h->shape_host_view.data(), ns * sizeof(DevShape), cudaMemcpyHostToDevice));
  h->shapes_dirty = false;
  return 0;
}

int upload_coeffs(sh_ctx *h) {
  if (!h->coeff_dirty) return 0;
  const size_t nn = SH_MAX_SHAPES * SH_MAX_SHAPES;
  try { h->d_pk.ensure(nn); h->d_pm.ensure(nn); h->d_pgn.ensure(nn); h->d_pgt.ensure(nn); h->d_pmu.ensure(nn); }
  catch (std::string &e) { return fail(h, e); }
  CU(cudaMemcpy(h->d_pk.p, h->pk.data(), nn * sizeof(double), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(h->d_pm.p, h->pm.data(), nn * sizeof(double), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(h->d_pgn.p, h->pgn.data(), nn * sizeof(double), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(h->d_pgt.p, h->pgt.data(), nn * sizeof(double), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(h->d_pmu.p, h->pmu.data(), nn * sizeof(double), cudaMemcpyHostToDevice));
  h->coeff_dirty = false;
  return 0;
}

// exclusive scan of in[0..n) into out[0..n], out[n] = total (also left in *d_total on the device)
int exclusive_scan(sh_ctx *h, const int *in, int *out, int n, int *d_total) {
  const int ntiles = std::max(1, cdiv(n, SCAN_TILE));
  try { h->tile_sum.ensure(ntiles); } catch (std::string &e) { return fail(h, e); }
  scan_tile_kernel<<<ntiles, SCAN_THREADS, 0, h->stream>>>(in, out, h->tile_sum.p, n);
  scan_sums_kernel<<<1, 1024, 0, h->stream>>>(h->tile_sum.p, ntiles, d_total);
  scan_add_kernel<<<std::max(1, cdiv(n, 256)), 256, 0, h->stream>>>(out, h->tile_sum.p, n, d_total);
  h->kernel_launches += 3;
  return 0;
}

// CUDA-event stopwatch classes on the library stream (rings drained at step boundaries): 0 cull, 1 evaluate, 2 reduce,
// 3 deep contacts, 4 candidate-cache build, 5 neighbor build, 6 ghost exchange
int ev_tick(sh_ctx *h, int kind) {
  if (h->ev2_used + 2 > h->ev2.size()) return 0;
  h->ev2_kind[h->ev2_used / 2] = kind;
  if (cudaEventRecord(h->ev2[h->ev2_used], h->stream) != cudaSuccess) return -2;
  return 0;
}
void ev_tock(sh_ctx *h) {
  if (h->ev2_used + 2 <= h->ev2.size()) { cudaEventRecord(h->ev2[h->ev2_used + 1], h->stream); h->ev2_used += 2; }
}

int build_neighbors(sh_ctx *h) {
  const int n = (int)h->n, st = h->stride, nown = (int)(h->n - h->nghost);
  if (ev_tick(h, 5)) return -2;
  // a live candidate cache over the SAME atoms (single rank, no set_atoms in between) survives the rebuild: keep the
  // old half list so that run_split_pipeline can carry the cache entries over to the new pairs
  const bool keep_cache = h->carry || (h->cache_state == CACHE_VALID && h->list_valid && h->nghost == 0 && h->npairs > 0 && h->atoms_epoch == h->cache_epoch);
  if (keep_cache && !h->carry) {
    try { h->old_half_off.ensure((size_t)nown + 2); h->old_pair_j.ensure((size_t)h->npairs + 1); } catch (std::string &e) { return fail(h, e); }
    CU(cudaMemcpyAsync(h->old_half_off.p, h->half_off.p, ((size_t)nown + 1) * sizeof(int), cudaMemcpyDeviceToDevice, h->stream));
    CU(cudaMemcpyAsync(h->old_pair_j.p, h->pair_j.p, (size_t)h->npairs * sizeof(int), cudaMemcpyDeviceToDevice, h->stream));
    h->old_nown = nown;
  }
  CU(cudaMemsetAsync(h->scalars.p + 1, 0, sizeof(int), h->stream));  // displacement flag
  double rmaxg = 0;
  for (auto &s : h->shapes) rmaxg = std::max(rmaxg, s.rmax);
  const double cut = 2.0 * rmaxg + h->skin;
  BinGrid G;
  G.skin = h->skin;
  bool need_bbox = false;
  for (int d = 0; d < 3; d++) {
    G.periodic[d] = h->periodic[d];
    G.boxlen[d] = h->hi[d] - h->lo[d];
    if (h->periodic[d]) {
      if (G.boxlen[d] < 2.0 * cut) return fail(h, "periodic box shorter than 2x cutoff");
    } else need_bbox = true;
  }
  double bmin[3] = {0, 0, 0}, bmax[3] = {0, 0, 0};
  if (need_bbox && n > 0) {
    auto enc = [](double v) { long long b; std::memcpy(&b, &v, 8); return b >= 0 ? b : (b ^ 0x7fffffffffffffffLL); };
    auto dec = [](long long b) { long long u = b >= 0 ? b : (b ^ 0x7fffffffffffffffLL); double v; std::memcpy(&v, &u, 8); return v; };
    long long init[6];
    for (int d = 0; d < 3; d++) { init[d] = enc(1e300); init[3 + d] = enc(-1e300); }
    CU(cudaMemcpyAsync(h->bbox.p, init, sizeof init, cudaMemcpyHostToDevice, h->stream));
    bbox_kernel<<<std::min(1024, cdiv(n, 256)), 256, 0, h->stream>>>(h->c.p, n, st, h->bbox.p);
    h->kernel_launches++;
    long long out[6];
    CU(cudaMemcpyAsync(out, h->bbox.p, sizeof out, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    for (int d = 0; d < 3; d++) { bmin[d] = dec(out[d]); bmax[d] = dec(out[3 + d]); }
    for (int d = 0; d < 3; d++) if (!std::isfinite(bmin[d]) || !std::isfinite(bmax[d])) return fail(h, "non-finite atom coordinates");
  }
  int64_t ncell = 1;
  for (int d = 0; d < 3; d++) {
    if (h->periodic[d]) { G.lo[d] = h->lo[d]; G.len[d] = G.boxlen[d]; }
    else { G.lo[d] = bmin[d]; G.len[d] = (bmax[d] - bmin[d]) * (1.0 + 1e-9) + 1e-9; }
    int nc = (int)std::floor(G.len[d] / cut);
    nc = std::max(1, std::min(nc, 1024));
    if (h->periodic[d] && nc < 3) nc = 1;
    G.nc[d] = nc;
    ncell *= nc;
  }
  // limit the grid to a few cells per atom (sparse, spread-out systems)
  while (ncell > std::max<int64_t>(4096, 8 * (int64_t)n)) {
    int dmax = 0;
    for (int d = 1; d < 3; d++) if (G.nc[d] > G.nc[dmax]) dmax = d;
    ncell /= G.nc[dmax];
    G.nc[dmax] = std::max(1, G.nc[dmax] / 2);
    if (h->periodic[dmax] && G.nc[dmax] < 3) G.nc[dmax] = 1;
    ncell *= G.nc[dmax];
  }
  try {
    h->cell_of.ensure(n + 1); h->cell_count.ensure(ncell + 1); h->cell_start.ensure(ncell + 2); h->cell_fill.ensure(ncell + 1);
    h->cell_atoms.ensure(n + 1); h->cnt_full.ensure(n + 1); h->cnt_half.ensure(n + 1); h->nbr_off.ensure(n + 2); h->half_off.ensure(n + 2);
  } catch (std::string &e) { return fail(h, e); }
  const int nb = std::max(1, cdiv(n, 256));
  CU(cudaMemsetAsync(h->cell_count.p, 0, (ncell + 1) * sizeof(int), h->stream));
  CU(cudaMemsetAsync(h->cell_fill.p, 0, (ncell + 1) * sizeof(int), h->stream));
  bin_count_kernel<<<nb, 256, 0, h->stream>>>(h->c.p, n, st, G, h->cell_of.p, h->cell_count.p);
  if (exclusive_scan(h, h->cell_count.p, h->cell_start.p, (int)ncell, h->scalars.p)) return -1;
  bin_fill_kernel<<<nb, 256, 0, h->stream>>>(n, h->cell_of.p, h->cell_start.p, h->cell_fill.p, h->cell_atoms.p);
  bin_sort_kernel<<<cdiv(ncell, 256), 256, 0, h->stream>>>((int)ncell, h->cell_start.p, h->cell_atoms.p);
  // newton on (in-library decomposition): ghosts get rows too (they collect the reactions that go back to their owners)
  const bool newton = h->dd.on && h->dd.newton && h->nghost > 0;
  const int nrows = newton ? n : nown;
  const long long *ntags = newton ? h->d_tag.p : nullptr;
  h->nrows = nrows;
  const int nbo = std::max(1, cdiv(nrows, 256));
  nbr_count_kernel<<<nbo, 256, 0, h->stream>>>(h->c.p, h->shape.p, h->d_shapes.p, nrows, nown, ntags, st, G, h->cell_of.p, h->cell_start.p,
                                              h->cell_atoms.p, h->cnt_full.p, h->cnt_half.p);
  h->kernel_launches += 4;
  int nentries = 0, npairs = 0;
  if (exclusive_scan(h, h->cnt_full.p, h->nbr_off.p, nrows, h->scalars.p + 8)) return -1;
  if (exclusive_scan(h, h->cnt_half.p, h->half_off.p, nrows, h->scalars.p + 9)) return -1;
  CU(cudaMemcpyAsync(h->h_pinned, h->scalars.p + 8, 2 * sizeof(int), cudaMemcpyDeviceToHost, h->stream));   // the one host
  CU(cudaStreamSynchronize(h->stream));                                                                     // sync of a rebuild
  nentries = h->h_pinned[0]; npairs = h->h_pinned[1];
  try {
    h->nbr_j.ensure(nentries + 1); h->pair_i.ensure(npairs + 1); h->pair_j.ensure(npairs + 1);
    h->pair_eij.ensure(npairs + 1); h->pair_eji.ensure(npairs + 1); h->pair_img.ensure(npairs + 1);
    if ((size_t)nentries + 1 > (size_t)h->slot_stride) { h->slot_stride = (int)((nentries + 1) * 1.25) + 64; h->slot.release(); h->slot.ensure((size_t)6 * h->slot_stride); }
    if ((size_t)npairs + 1 > (size_t)h->pres_stride) { h->pres_stride = (int)((npairs + 1) * 1.25) + 64; h->pres.release(); h->pres.ensure((size_t)14 * h->pres_stride); }
  } catch (std::string &e) { return fail(h, e); }
  nbr_fill_kernel<<<nbo, 256, 0, h->stream>>>(h->c.p, h->shape.p, h->d_shapes.p, nrows, nown, ntags, st, G, h->cell_of.p, h->cell_start.p,
                                             h->cell_atoms.p, h->nbr_off.p, h->half_off.p, h->nbr_j.p, h->pair_i.p,
                                             h->pair_j.p, h->pair_eij.p, h->pair_img.p);
  pair_reverse_kernel<<<std::max(1, cdiv(npairs, 256)), 256, 0, h->stream>>>(npairs, nrows, h->pair_i.p, h->pair_j.p, h->nbr_off.p,
                                                                             h->nbr_j.p, h->pair_eji.p);
  copy_origin_kernel<<<nb, 256, 0, h->stream>>>(h->c.p, h->c0.p, n, st);
  h->kernel_launches += 3;
  ev_tock(h);
  CU(cudaGetLastError());
  h->npairs = npairs; h->nentries = nentries;
  h->list_valid = true; h->steps_since_build = 0; h->neighbor_builds++;
  h->out_zero_valid = false;   // new pairs and CSR entries
  // the pair list changed: a live cache over the same atoms is remapped, anything else is rebuilt
  h->cache_state = keep_cache ? CACHE_REMAP : CACHE_INVALID;
  if (!keep_cache) h->carry = false;
  return 0;
}

int drain_events(sh_ctx *h) {
  if (h->ev_used == 0 && h->ev2_used == 0) return 0;
  CU(cudaStreamSynchronize(h->stream));
  for (size_t k = 0; k + 1 < h->ev2_used; k += 2) {
    float ms = 0;
    cudaEventElapsedTime(&ms, h->ev2[k], h->ev2[k + 1]);
    double *dst[8] = {&h->sec_cull, &h->sec_eval, &h->sec_reduce, &h->sec_deep, &h->sec_cache, &h->sec_neigh, &h->sec_comm, &h->sec_other};
    *dst[h->ev2_kind[k / 2] & 7] += ms * 1e-3;
  }
  h->ev2_used = 0;
  for (size_t k = 0; k + 1 < h->ev_used; k += 2) {
    float ms = 0;
    cudaEventElapsedTime(&ms, h->ev[k], h->ev[k + 1]);
    h->sec_pair += ms * 1e-3;
  }
  h->ev_used = 0;
  return 0;
}

}  // namespace
#include "dd_host.cuh"
namespace {

template <int NT>
int launch_pair(sh_ctx *h, const PairArgs &A, int ctas_per_sm, size_t smem) {
  CU(cudaFuncSetAttribute(pair_kernel<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 48 * 1024)));
  int occ = 0;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pair_kernel<NT>, NT, smem));
  if (occ < 1) return fail(h, "pair kernel does not fit on an SM (shared memory)");
  if (ctas_per_sm > 0) occ = std::min(occ, ctas_per_sm);
  const int grid = std::max(1, std::min(A.npairs, occ * h->sm_count));
  pair_kernel<NT><<<grid, NT, smem, h->stream>>>(A);
  return 0;
}

template <int NW, bool SMEM_TABLES>
int launch_pair_warp(sh_ctx *h, const PairArgs &A, int ctas_per_sm, int max_grid = 1 << 30) {
  const size_t smem = pair_warp_smem_bytes(h->total_terms, NW, SMEM_TABLES);
  CU(cudaFuncSetAttribute(pair_warp_kernel<NW, SMEM_TABLES>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 48 * 1024)));
  int occ = 0;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pair_warp_kernel<NW, SMEM_TABLES>, NW * 32, smem));
  if (occ < 1) return fail(h, "pair warp kernel does not fit on an SM");
  if (ctas_per_sm > 0) occ = std::min(occ, ctas_per_sm);
  const int grid = std::max(1, std::min(std::min((A.npairs + NW - 1) / NW, occ * h->sm_count), max_grid));
  pair_warp_kernel<NW, SMEM_TABLES><<<grid, NW * 32, smem, h->stream>>>(A, (int)h->shapes.size(), h->total_terms, (h->tune_variant & 2) ? 0 : 1);
  return 0;
}

int launch_fused(sh_ctx *h, const PairArgs &P, int max_grid = 1 << 30) {
  const bool fits = pair_warp_smem_bytes(h->total_terms, 16, true) <= 200 * 1024;
  const int tw = h->tune_threads ? h->tune_threads : 512;
  const int cps = h->tune_ctas_per_sm;
  if (fits) {
    if (tw == 256) return launch_pair_warp<8, true>(h, P, cps, max_grid);
    if (tw == 128) return launch_pair_warp<4, true>(h, P, cps, max_grid);
    if (tw == 384) return launch_pair_warp<12, true>(h, P, cps, max_grid);
    return launch_pair_warp<16, true>(h, P, cps, max_grid);
  }
  if (tw == 256) return launch_pair_warp<8, false>(h, P, cps, max_grid);
  return launch_pair_warp<16, false>(h, P, cps, max_grid);
}

template <int WPB, int PTS, int MINB>
int launch_eval(sh_ctx *h, const SplitArgs &S, int maxT) {
  const size_t smem = (size_t)maxT * 24 + 32;
  auto kern = pair_eval_kernel<WPB, PTS, MINB>;
  CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 48 * 1024)));
  int occ = 0;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, WPB * 32, smem));
  if (occ < 1) return fail(h, "pair_eval_kernel does not fit on an SM");
  const int rpb = WPB * 32 * PTS;
  eval_plan_kernel<<<1, 32, 0, h->stream>>>(S, (int)h->shapes.size(), rpb, h->eval_plan.p);
  const int chunked = h->eval_mode == 2;
  int grid = occ * h->sm_count;
  if (!chunked) {   // one block per CTA: grid from the previous phase's record count (+ slack), grid-stride covers the rest
    long long est = h->last_records > 0 ? h->last_records + h->last_records / 16 : 0;
    if (est == 0) for (long long c : h->h_pool_cap) est += c;
    grid = (int)std::max<long long>(grid, std::min<long long>(est / rpb + (long long)h->shapes.size() + 1, 1 << 22));
  }
  kern<<<grid, WPB * 32, smem, h->stream>>>(h->d_shapes.p, S, h->eval_plan.p, h->counters.p, chunked);
  h->kernel_launches += 2;
  return 0;
}

// advisory read-back of the previous pair phase (pool fill, deep / slow pairs, cache validity): never needed for the
// correctness of that phase (a full pool sends pairs to the fused kernel), only to size the next one
int absorb_split_feedback(sh_ctx *h) {
  if (!h->sc_pending) return 0;
  CU(cudaEventSynchronize(h->ev_sc));
  h->sc_pending = false;
  const SplitScalars &sc = *h->h_split_sc;
  h->big_pairs += sc.nbig; h->slow_pairs += sc.nslow;
  const int ns = std::min<int>(h->sc_nshape, (int)h->h_pool_cap.size());
  for (int s = 0; s < ns; s++)
    if ((long long)sc.pool_count[s] > h->h_pool_cap[s] * 9 / 10) {
      h->h_pool_cap[s] = (long long)(sc.pool_count[s] * 3 / 2) + 4096;
      h->pool_grows++;
    }
  if ((long long)sc.in_count > h->h_in_cap * 9 / 10) { h->h_in_cap = (long long)(sc.in_count * 3 / 2) + 4096; h->pool_grows++; }
  h->last_records = 0;
  for (int s = 0; s < ns; s++) h->last_records += (long long)std::min<unsigned long long>(sc.pool_count[s], (unsigned long long)h->h_pool_cap[s]);
  // hard flag: that phase already ran on the window path; soft flag: rebuild now, while the cache is still valid
  // (several ranks: the decision comes from the MAX over ranks instead, step_once, so that every rank rebuilds its cache
  // on the same step and nobody waits for a neighbour's build on top of its own)
  if (!h->cache_sync_ranks && (h->h_cache_invalid[0] != 0 || h->h_cache_invalid[1] != 0) && h->cache_state != CACHE_INVALID) { h->cache_state = CACHE_INVALID; h->cache_exhausted = true; }
  return 0;
}

// cached cull (+ window cull on the slow list) -> evaluate -> reduce -> fused kernel on the deep-contact list.
// Nothing in here waits for the device except a candidate-cache (re)build.
int run_split_pipeline(sh_ctx *h, PairArgs &P) {
  const int ns = (int)h->shapes.size(), np = P.npairs;
  constexpr int WPB = 8;
  int rc;
  if ((rc = absorb_split_feedback(h))) return rc;
  try {
    h->pd.ensure((size_t)2 * np + 2); h->big_list.ensure(np + 1); h->slow_list.ensure(np + 1);
    if (h->out_zero.cap < (size_t)np + 1) { h->out_zero.ensure(np + 1); h->out_zero_valid = false; }
    h->pool_base.ensure(SH_MAX_SHAPES); h->pool_cap.ensure(SH_MAX_SHAPES); h->split_sc.ensure(1); h->eval_plan.ensure(1); h->split_flags.ensure(4);
  } catch (std::string &e) { return fail(h, e); }
  if (!h->h_pool_count) {
    CU(cudaMallocHost(&h->h_pool_count, 8 * sizeof(unsigned long long)));
    CU(cudaMallocHost(&h->h_split_sc, sizeof(SplitScalars)));
    CU(cudaMallocHost(&h->h_cache_invalid, 2 * sizeof(int)));
    CU(cudaEventCreateWithFlags(&h->ev_sc, cudaEventDisableTiming));
  }
  if ((int)h->h_pool_cap.size() != ns) {   // first sizing: 24 records per pair, spread over the shapes, x2
    h->h_pool_cap.assign(ns, std::max<long long>(4096, (long long)np * 24 / std::max(1, ns) * 2));
  }
  auto tick = [&](int kind) -> int { return ev_tick(h, kind); };
  auto tock = [&]() { ev_tock(h); };
  const int use_bounds = (h->tune_variant & 2) ? 0 : 1;
  // ---- candidate cache: (re)build when the pair list changed or a particle used up its displacement margin
  CacheArgs C;
  C.enabled = (h->tune_variant & (8 | 2)) ? 0 : 1;   // the cache is built from the direction-cell bounds
  C.invalid = h->scalars.p + 3;
  if (C.enabled) {
    const int cur = h->cache_cur;
    try { h->cache_hot[cur].ensure((size_t)np + 2); h->cache_count.ensure(2); h->fresh_list.ensure((size_t)np + 2); }
    catch (std::string &e) { return fail(h, e); }
    // origin of the moment sums of the displacement fit: the box centre (finite boxes) keeps them well conditioned
    double pc[3];
    for (int d = 0; d < 3; d++) pc[d] = (h->hi[d] < 1e29 && h->lo[d] > -1e29) ? 0.5 * (h->lo[d] + h->hi[d]) : 0.0;
    auto check_validity = [&]() -> int {   // raises the device flag scalars[3] when a particle used up its margin
      double dmin = 1e300;
      for (auto &sh : h->shapes) dmin = std::min(dmin, sh.cache_delta[h->cache_level]);
      double rmaxg = 0;
      for (auto &sh : h->shapes) rmaxg = std::max(rmaxg, sh.rmax);
      const double rpair = 2.0 * rmaxg + 2.0 * h->skin;   // no pair of the list is further apart than this
      CU(cudaMemsetAsync(h->drift.p, 0, CACHE_FIT_N * sizeof(double), h->stream));
      cache_drift_kernel<<<cdiv(h->n, 256), 256, 0, h->stream>>>(view_all(h), pc[0], pc[1], pc[2], h->drift.p);
      cache_fit_solve_kernel<<<1, 32, 0, h->stream>>>(h->drift.p, h->drift.p + 32);
      cache_check_kernel<<<cdiv(h->n, 256), 256, 0, h->stream>>>(view_all(h), h->d_shapes.p, h->cache_level, 0.5 * dmin, h->drift.p + 32,
                                                                 pc[0], pc[1], pc[2], rpair, h->scalars.p + 3);
      h->kernel_launches += 3;
      return 0;
    };
    if (h->cache_state == CACHE_REMAP && h->cache_level + 1 < SH_CACHE_LEVELS && !(h->tune_variant & 32)) {
      // the pair list was rebuilt over the same atoms: pairs that were in the old list keep their candidates, the new
      // ones are built with the next larger margin.  No host synchronisation.
      const int nxt = 1 - cur;
      try { h->cache_hot[nxt].ensure((size_t)np + 2); h->cache_pool[nxt].ensure((size_t)h->cache_cap + 64); }
      catch (std::string &e) { return fail(h, e); }
      const int *amap = nullptr;
      if (h->carry) {   // decomposed rebuild: find every new atom among the old ones, carry its cache reference state over
        try { h->amap.ensure((size_t)h->n + 2); } catch (std::string &e) { return fail(h, e); }
        const int nstay = h->dd.last_nstay, nown = (int)(h->n - h->nghost);
        CU(cudaMemsetAsync(h->drift.p + 64, 0, CACHE_FIT_N * sizeof(double), h->stream));
        const double le_doff = h->dd.le_rate * h->dd.glen[1] * (h->time - h->cache_time);
        dd_cache_map_kernel<<<cdiv(h->n, 256), 256, 0, h->stream>>>(view_all(h), h->d_tag.p, nown, nstay, h->dd.order.p, h->old_tag.p, h->old_c.p,
                                                                    h->old_stride, h->old_nown, h->old_n, h->ghost_hash.p, h->ghost_hash_size,
                                                                    0.25 * h->dd.G.rc * h->dd.G.rc, h->old_cc0.p, h->old_cq0.p, h->amap.p, h->dd.glen[1], le_doff,
                                                                    pc[0], pc[1], pc[2], h->drift.p + 64);
        cache_fit_solve_kernel<<<1, 32, 0, h->stream>>>(h->drift.p + 64, h->drift.p + 96);
        dd_cache_new_atoms_kernel<<<cdiv(h->n, 256), 256, 0, h->stream>>>(view_all(h), h->amap.p, h->drift.p + 96, pc[0], pc[1], pc[2]);
        h->kernel_launches += 3;
        amap = h->amap.p;
        h->carry = false; h->cache_epoch = h->atoms_epoch;
      }
      if ((rc = check_validity())) return rc;
      if (tick(4)) return -2;
      CU(cudaMemsetAsync(h->cache_count.p, 0, 2 * sizeof(unsigned long long), h->stream));
      CU(cudaMemsetAsync(h->split_flags.p + 2, 0, 2 * sizeof(int), h->stream));
      C.pool = h->cache_pool[nxt].p; C.hot = h->cache_hot[nxt].p; C.count = h->cache_count.p;
      C.cap = h->cache_cap; C.overflow = h->split_flags.p + 2; C.level = h->cache_level + 1;
      cache_remap_kernel<<<cdiv(np, 256), 256, 0, h->stream>>>(P, h->old_half_off.p, h->old_pair_j.p, h->old_nown, h->cache_hot[cur].p,
                                                                h->cache_pool[cur].p, C, h->fresh_list.p, h->split_flags.p + 3, amap);
      pair_cache_build_kernel<4><<<std::max(1, std::min(cdiv(np, 4), h->sm_count * 8)), 4 * 32, 0, h->stream>>>(P, C, h->fresh_list.p, h->split_flags.p + 3);
      tock();
      h->kernel_launches += 2;
      h->cache_cur = nxt; h->cache_state = CACHE_VALID; h->cache_remaps++;
    } else if (h->cache_state != CACHE_VALID) {
      // margin level: a cache that was used up quickly gets a wider margin, one that lived long a tighter one
      if (h->cache_level_pin >= 0) h->cache_level = h->cache_level_pin;
      else if (h->cache_exhausted) {
        // (level 2 leaves no wider level for the pairs a neighbor rebuild adds, so every rebuild would be a full cache
        // build: the adaptive choice stops at level 1; a full build costs about as much as 5 pair phases)
        if (h->cache_age < 40 && h->cache_level < 1) h->cache_level++;
        else if (h->cache_age > 400 && h->cache_level > 0) h->cache_level--;
      }
      h->cache_exhausted = false;
      if (h->cache_cap < (long long)np * 48) h->cache_cap = (long long)np * 48;
      if (tick(4)) return -2;
      for (int attempt = 0;; attempt++) {
        if (attempt > 6) return fail(h, "candidate cache kept overflowing");
        try { h->cache_pool[cur].ensure((size_t)h->cache_cap + 64); } catch (std::string &e) { return fail(h, e); }
        CU(cudaMemsetAsync(h->cache_count.p, 0, 2 * sizeof(unsigned long long), h->stream));
        CU(cudaMemsetAsync(h->split_flags.p + 2, 0, sizeof(int), h->stream));
        C.pool = h->cache_pool[cur].p; C.hot = h->cache_hot[cur].p; C.count = h->cache_count.p;
        C.cap = h->cache_cap; C.overflow = h->split_flags.p + 2; C.level = h->cache_level;
        pair_cache_build_kernel<4><<<cdiv(np, 4), 4 * 32, 0, h->stream>>>(P, C, nullptr, nullptr);
        h->kernel_launches++;
        CU(cudaMemcpyAsync(h->h_pool_count, h->cache_count.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
        CU(cudaMemcpyAsync(h->h_pool_count + 1, h->split_flags.p + 2, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));
        if (*reinterpret_cast<const int *>(h->h_pool_count + 1) == 0) break;
        h->cache_cap = (long long)(h->h_pool_count[0] * 3 / 2) + 4096;
      }
      cache_origin_kernel<<<cdiv(h->n, 256), 256, 0, h->stream>>>(view_all(h));
      CU(cudaMemsetAsync(h->scalars.p + 3, 0, 2 * sizeof(int), h->stream));
      tock();
      h->kernel_launches++;
      h->cache_state = CACHE_VALID; h->cache_builds++; h->cache_age = 0; h->cache_epoch = h->atoms_epoch; h->cache_build_step = h->step_index;
      h->cache_time = h->time;
    } else {
      if ((rc = check_validity())) return rc;
    }
    h->cache_age++;
  }
  C.pool = h->cache_pool[h->cache_cur].p; C.hot = h->cache_hot[h->cache_cur].p; C.count = h->cache_count.p;
  C.cap = h->cache_cap; C.overflow = h->split_flags.p + 2; C.level = h->cache_level;
  std::vector<long long> base(ns);
  long long tot = 0;
  for (int s2 = 0; s2 < ns; s2++) { base[s2] = tot; tot += h->h_pool_cap[s2]; }
  if (h->h_in_cap < (long long)np * 2 + 4096) h->h_in_cap = (long long)np * 2 + 4096;
  if (h->h_in_cap > 0xfffffff0LL) h->h_in_cap = 0xfffffff0LL;      // 32-bit offsets in the run descriptors
  try { h->pool.ensure((size_t)tot + 64); h->pool_kin.ensure((size_t)tot + 64); h->inpool.ensure((size_t)h->h_in_cap + 64); } catch (std::string &e) { return fail(h, e); }
  CU(cudaMemcpyAsync(h->pool_base.p, base.data(), ns * sizeof(long long), cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(h->pool_cap.p, h->h_pool_cap.data(), ns * sizeof(long long), cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemsetAsync(h->split_sc.p, 0, sizeof(SplitScalars), h->stream));
  SplitArgs S;
  S.pool = h->pool.p; S.pool_kin = h->pool_kin.p; S.pool_base = h->pool_base.p; S.pool_cap = h->pool_cap.p; S.sc = h->split_sc.p;
  S.pd = h->pd.p; S.out_zero = h->out_zero.p; S.big_list = h->big_list.p; S.slow_list = h->slow_list.p; S.inpool = h->inpool.p; S.in_cap = h->h_in_cap;
  // ---- A
  if (tick(0)) return -2;
  if (C.enabled) {
    // one pair per half warp (default) or per warp ("cull_lpp" 32); WPB warps per CTA
    const int cw = h->tune_cull_wpb > 0 ? h->tune_cull_wpb : 1;
    const int ppw = h->tune_cull_lpp == 32 ? 1 : 2;
    const int grid = cdiv(np, cw * ppw);
    ShapeLiteTable T{};
    for (int s2 = 0; s2 < ns && s2 < SH_MAX_SHAPES; s2++) {
      const DevShape &v = h->shape_host_view[s2];
      T.s[s2].pf4 = v.pf4; T.s[s2].cube_ul = v.cube_ul; T.s[s2].px = v.px; T.s[s2].py = v.py; T.s[s2].pz = v.pz;
      T.s[s2].cube_n = v.cube_n; T.s[s2].rmax = v.rmax; T.s[s2].rmax2 = v.rmax2; T.s[s2].rmin2 = v.rmin2;
    }
#define LAUNCH_CULL(W, L) pair_cull_cached_kernel<W, L><<<grid, W * 32, 0, h->stream>>>(P, S, C, use_bounds, T)
    if (ppw == 1) { if (cw == 1) LAUNCH_CULL(1, 32); else if (cw == 2) LAUNCH_CULL(2, 32); else if (cw == 8) LAUNCH_CULL(8, 32); else LAUNCH_CULL(4, 32); }
    else { if (cw == 1) LAUNCH_CULL(1, 16); else if (cw == 2) LAUNCH_CULL(2, 16); else if (cw == 8) LAUNCH_CULL(8, 16); else LAUNCH_CULL(4, 16); }
#undef LAUNCH_CULL
    h->kernel_launches++;
  }
  {
    constexpr int WW = 2;   // persistent; pairs differ a lot in length, small CTAs retire independently
    const int grid = std::max(1, std::min(cdiv(np, WW), h->sm_count * 16));
    pair_cull_window_kernel<WW><<<grid, WW * 32, 0, h->stream>>>(P, S, C, use_bounds);
    h->kernel_launches++;
  }
  tock();
  // ---- B
  int maxT = 1;
  for (int s2 = 0; s2 < ns; s2++) maxT = std::max(maxT, h->shape_host_view[s2].nterms4 + 4);
  if (tick(1)) return -2;
  if (h->eval_pts == 2) rc = h->eval_occ == 3 ? launch_eval<WPB, 2, 3>(h, S, maxT) : launch_eval<WPB, 2, 4>(h, S, maxT);
  else rc = launch_eval<WPB, 4, 2>(h, S, maxT);
  if (rc) return rc;
  tock();
  h->eval_launches++;
  // ---- C
  if (tick(2)) return -2;
  if (!h->out_zero_valid) {   // nothing is known about the outputs' contents
    CU(cudaMemsetAsync(h->out_zero.p, 0, (size_t)np, h->stream));
    h->out_zero_valid = true;
  }
  pair_reduce_kernel<<<cdiv(np, 256), 128, 0, h->stream>>>(P, S);
  tock();
  h->kernel_launches++;
  // ---- deep contacts / pairs that found the pool full: fused kernel over the device-side list
  {
    PairArgs Pb = P;
    Pb.pair_list = h->big_list.p; Pb.npairs = np; Pb.npairs_dev = &h->split_sc.p->nbig; Pb.work_counter = &h->split_sc.p->deep_counter;
    if (tick(3)) return -2;
    rc = launch_fused(h, Pb, h->sm_count);
    if (rc) return rc;
    tock();
    h->kernel_launches++;
  }
  CU(cudaMemcpyAsync(h->h_split_sc, h->split_sc.p, sizeof(SplitScalars), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(h->h_cache_invalid, h->scalars.p + 3, 2 * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaEventRecord(h->ev_sc, h->stream));
  h->sc_pending = true; h->sc_nshape = ns;
  return 0;
}

int compute_forces_device(sh_ctx *h) {
  const int n = (int)(h->n - h->nghost);   // forces are accumulated on owned atoms only
  const bool newton_dd = h->dd.on && h->dd.newton && h->dd.borders_ok && (h->dd.peer.enabled || h->nghost > 0 || h->dd.nsend > 0);
  if (n == 0 && !newton_dd) { h->forces_valid = true; return 0; }
  AtomView A = view(h);
  const int nb = std::max(1, cdiv(n, 256));
  if (h->npairs > 0) {
    PairArgs P;
    P.shapes = h->d_shapes.p; P.c = h->c.p; P.Rs = h->Rs.p; P.x = h->x.p; P.shape = h->shape.p; P.stride = h->stride;
    P.pair_i = h->pair_i.p; P.pair_j = h->pair_j.p; P.pair_eij = h->pair_eij.p; P.pair_eji = h->pair_eji.p; P.pair_img = h->pair_img.p;
    P.npairs = h->npairs; P.slot = h->slot.p; P.slot_stride = h->slot_stride; P.pres = h->pres.p; P.pres_stride = h->pres_stride;
    P.pk = h->d_pk.p; P.pm = h->d_pm.p;
    P.dissip = h->dissip ? 1 : 0; P.v = h->v.p; P.L = h->L.p; P.q = h->q.p; P.pgn = h->d_pgn.p; P.pgt = h->d_pgt.p; P.pmu = h->d_pmu.p;
    if (h->dissip && h->nghost > 0 && !h->dd.on) return fail(h, "dissipative contact terms need ghost velocities: use the in-library decomposition (sh_dd_init)");
    for (int d = 0; d < 3; d++) { P.boxlen[d] = h->hi[d] - h->lo[d]; P.periodic[d] = h->periodic[d]; }
    P.work_counter = h->scalars.p + 2; P.counters = h->counters.p;
    int maxT = 1, maxq = 32;
    for (auto &s : h->shapes) { maxT = std::max(maxT, s.nterms); maxq = std::max(maxq, s.nq); }
    P.max_terms = maxT; P.max_nq = maxq; P.nlocal = n; P.pair_list = nullptr; P.npairs_dev = nullptr;
    CU(cudaMemsetAsync(h->scalars.p + 2, 0, sizeof(int), h->stream));
    const int nt = h->tune_threads ? h->tune_threads : 128;
    // the event rings are drained only here, at a step boundary, before the outer start event (ADVICE r1)
    if (h->ev_used + 2 > h->ev.size() || h->ev2_used + 16 > h->ev2.size()) { if (drain_events(h)) return -2; }
    CU(cudaEventRecord(h->ev[h->ev_used], h->stream));
    int rc;
    if (h->tune_variant & 1) {           // CTA-per-pair kernel (full-table scan)
      h->out_zero_valid = false;
      if (nt == 256) rc = launch_pair<256>(h, P, h->tune_ctas_per_sm, pair_smem_bytes(maxT, maxq, 8));
      else if (nt == 64) rc = launch_pair<64>(h, P, h->tune_ctas_per_sm, pair_smem_bytes(maxT, maxq, 2));
      else rc = launch_pair<128>(h, P, h->tune_ctas_per_sm, pair_smem_bytes(maxT, maxq, 4));
    } else if ((h->tune_variant & 4) || (!(h->tune_variant & 16) && h->npairs < 16384)) {
      // fused warp-per-pair kernel: explicit (bit 4), or small systems where the split pipeline's extra
      // launches and its host sync cost more than they save (bit 16 forces the split pipeline)
      h->out_zero_valid = false;
      rc = launch_fused(h, P);
    } else {                             // split pipeline (default): cull / evaluate / reduce
      rc = run_split_pipeline(h, P);
    }
    if (rc) return rc;
    CU(cudaEventRecord(h->ev[h->ev_used + 1], h->stream));
    h->ev_used += 2;
    h->pair_launches++; h->kernel_launches++;
  }
  if (h->walls.n > 0 && n > 0) {
    wall_kernel<<<cdiv((int64_t)n * 32, 256), 256, 0, h->stream>>>(A, h->d_shapes.p, h->walls, h->ewall.p);
    h->kernel_launches++;
  }
  // newton on: the ghosts have rows too, holding the reactions of the cross-rank pairs evaluated here
  const int nrows = h->list_valid && h->nrows > n ? h->nrows : n;
  if (nrows > 0) {
    AtomView G2 = view_all(h);
    G2.n = nrows;
    gather_kernel<<<cdiv(nrows, 256), 256, 0, h->stream>>>(G2, h->nbr_off.p, h->slot.p, h->slot_stride, h->walls.n > 0 ? n : 0);
    h->kernel_launches++;
  }
  if (newton_dd) { int rc = dd_reverse(h); if (rc) return rc; }
  CU(cudaGetLastError());
  h->forces_valid = true;
  h->carry = false;   // a snapshot that this pair phase did not consume is stale from here on
  return 0;
}

int prepare(sh_ctx *h) {
  if (h->n > 0 && h->shapes.empty()) return fail(h, "no shapes defined");
  int rc;
  if ((rc = upload_shapes(h))) return rc;
  if ((rc = upload_coeffs(h))) return rc;
  return 0;
}

// tags on the host (sh_get_pairs, snapshots, sh_get_tags): refreshed lazily after the device moved atoms around
int sync_tags_host(sh_ctx *h) {
  if (h->tags_host_valid) return 0;
  h->tag.resize(h->n);
  if (h->n > 0) {
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaMemcpy(h->tag.data(), h->d_tag.p, (size_t)h->n * sizeof(long long), cudaMemcpyDeviceToHost));
  }
  h->tags_host_valid = true;
  return 0;
}

// neighbor trigger: half the skin, less the distance the Lees-Edwards images have slid since the last build
double neighbor_trigger(const sh_ctx *h) {
  double t = 0.5 * h->skin;
  if (h->dd.on && h->dd.le_rate != 0.0) t = std::max(0.0, 0.5 * (h->skin - std::fabs(h->dd.le_rate * h->dd.glen[1] * (h->time - h->dd.le_time_build))));
  return t;
}

// all ranks must take the same rebuild decision: MAX over ranks of a device flag
int reduce_flag(sh_ctx *h, int *d_flag) {
  if (h->dd.on && h->dd.nranks > 1) NC(h->dd.nccl->AllReduce(d_flag, d_flag, 1, ncclInt, ncclMax, h->dd.comm, h->stream));
  return 0;
}

int setup_forces(sh_ctx *h) {
  int rc;
  if ((rc = prepare(h))) return rc;
  const bool dd = h->dd.on;
  bool fresh_borders = false;
  if (dd) {
    if (!h->dd.geometry_ok) { if ((rc = dd_setup_geometry(h))) return rc; }
    if (!h->dd.borders_ok) { if ((rc = dd_borders(h))) return rc; fresh_borders = true; }
    else if (h->list_valid) { if ((rc = dd_forward(h))) return rc; }
  }
  if (h->n > 0 || dd) {
    const double trig = neighbor_trigger(h);
    if (h->n > 0) {
      pose_kernel<<<cdiv(h->n, 256), 256, 0, h->stream>>>(view_all(h), h->d_shapes.p, h->list_valid ? trig * trig : -1.0, h->scalars.p + 1, 0, (int)h->n);
      h->kernel_launches++;
    }
    bool rebuild = !h->list_valid;
    if (!rebuild) {
      if ((rc = reduce_flag(h, h->scalars.p + 1))) return rc;
      CU(cudaMemcpyAsync(h->h_pinned + 4, h->scalars.p + 1, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
      CU(cudaStreamSynchronize(h->stream));
      rebuild = h->h_pinned[4] != 0;
    }
    if (rebuild && dd && !fresh_borders) {   // atoms moved since the borders were made: migrate, new ghosts, new poses
      if ((rc = dd_rebuild(h))) return rc;
      if (h->n > 0) {
        pose_kernel<<<cdiv(h->n, 256), 256, 0, h->stream>>>(view_all(h), h->d_shapes.p, -1.0, h->scalars.p + 1, 0, (int)h->n);
        h->kernel_launches++;
      }
    }
    if (rebuild) { if ((rc = build_neighbors(h))) return rc; }
  }
  h->lag_pending = false;
  return compute_forces_device(h);
}

}  // namespace

// =====================================================================================
extern "C" {

int sh_version(void) { return 100; }

int sh_create(sh_ctx **out, int device_id) {
  if (!out) return -1;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return -3;  // no CUDA device: no fallback
  if (device_id < 0 || device_id >= ndev) return -4;
  sh_ctx *h = new sh_ctx();
  h->device = device_id;
  if (cudaSetDevice(device_id) != cudaSuccess) { delete h; return -5; }
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device_id);
  h->sm_count = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) { delete h; return -6; }
  h->pk.assign(SH_MAX_SHAPES * SH_MAX_SHAPES, 1.0);
  h->pm.assign(SH_MAX_SHAPES * SH_MAX_SHAPES, 1.0);
  h->pgn.assign(SH_MAX_SHAPES * SH_MAX_SHAPES, 0.0); h->pgt.assign(SH_MAX_SHAPES * SH_MAX_SHAPES, 0.0); h->pmu.assign(SH_MAX_SHAPES * SH_MAX_SHAPES, 0.0);
  try {
    h->scalars.ensure(16); h->bbox.ensure(8); h->counters.ensure(16); h->drift.ensure(128);
  } catch (std::string &) { delete h; return -7; }
  cudaMemset(h->scalars.p, 0, 16 * sizeof(int));
  cudaMemset(h->counters.p, 0, 16 * sizeof(unsigned long long));
  cudaMallocHost(&h->h_pinned, 64);
  cudaMallocHost(&h->h_lagflag, 16 * sizeof(int));
  std::memset(h->h_lagflag, 0, 16 * sizeof(int));
  cudaMallocHost(&h->dd.h_int, 256 * sizeof(int));
  for (auto &e : h->ev_lag) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
  cudaEventCreate(&h->run_e0); cudaEventCreate(&h->run_e1);
  h->ev.resize(2048); h->ev2.resize(4096); h->ev2_kind.resize(2048);
  for (auto &e : h->ev) cudaEventCreate(&e);
  for (auto &e : h->ev2) cudaEventCreate(&e);
  *out = h;
  return 0;
}

int sh_destroy(sh_ctx *h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  for (auto &d : h->shape_dev) { d.Ap.release(); d.ab.release(); d.node.release(); d.row_x.release(); d.cube.release(); d.pf4.release(); d.pn.release(); for (auto &w : d.cubew) w.release(); }
  h->d_shapes.release(); h->d_pk.release(); h->d_pm.release(); h->d_pgn.release(); h->d_pgt.release(); h->d_pmu.release(); h->stress_part.release();
  DevBuf<double> *db[] = {&h->x, &h->v, &h->q, &h->L, &h->f, &h->tq, &h->c, &h->Rs, &h->c0, &h->wallf, &h->ewall, &h->ke, &h->bbox, &h->slot, &h->pres};
  for (auto *b : db) b->release();
  DevBuf<int> *ib[] = {&h->shape, &h->cell_of, &h->cell_count, &h->cell_start, &h->cell_fill, &h->cell_atoms, &h->tile_sum, &h->cnt_full,
                       &h->cnt_half, &h->nbr_off, &h->half_off, &h->nbr_j, &h->pair_i, &h->pair_j, &h->pair_eij, &h->pair_eji, &h->pair_img, &h->scalars};
  for (auto *b : ib) b->release();
  h->counters.release();
  h->as_vir.release(); h->as_kin.release(); h->as_en.release(); h->as_send.release(); h->as_recv.release(); h->as_cnt.release(); h->as_epair.release();
  for (auto &e : h->ev) cudaEventDestroy(e);
  for (auto &e : h->ev2) cudaEventDestroy(e);
  h->pool.release(); h->pool_kin.release(); h->pool_base.release(); h->pool_cap.release(); h->split_sc.release(); h->eval_plan.release(); h->slow_list.release();
  h->pd.release(); h->out_zero.release(); h->big_list.release(); h->split_flags.release(); h->inpool.release();
  for (int k = 0; k < 2; k++) { h->cache_hot[k].release(); h->cache_pool[k].release(); }
  h->old_c.release(); h->old_cc0.release(); h->old_cq0.release(); h->old_tag.release(); h->ghost_hash.release(); h->amap.release();
  h->old_half_off.release(); h->old_pair_j.release(); h->fresh_list.release(); h->cache_count.release(); h->cc0.release(); h->cq0.release(); h->drift.release();
  if (h->h_pool_count) { cudaFreeHost(h->h_pool_count); cudaFreeHost(h->h_split_sc); cudaFreeHost(h->h_cache_invalid); cudaEventDestroy(h->ev_sc); }
  if (h->h_pinned) cudaFreeHost(h->h_pinned);
  if (h->h_lagflag) cudaFreeHost(h->h_lagflag);
  if (h->dd.h_int) cudaFreeHost(h->dd.h_int);
  for (auto &e : h->ev_lag) if (e) cudaEventDestroy(e);
  for (auto &e : h->ev_step) cudaEventDestroy(e);
  dd_peer_release(h);
  if (h->dd.peer.d_err) cudaFree(h->dd.peer.d_err);
  h->dd.peer.d_off.release();
  if (h->dd.comm && h->dd.nccl) h->dd.nccl->CommDestroy(h->dd.comm);
  {
    DdCtx &D = h->dd;
    DevBuf<int> *ib2[] = {&D.flag, &D.pos, &D.order, &D.d_int, &D.send_idx, &D.send_slot, &D.shape2};
    for (auto *b : ib2) b->release();
    DevBuf<double> *db2[] = {&D.sendbuf, &D.recvbuf, &D.x2, &D.v2, &D.q2, &D.L2, &h->gf};
    for (auto *b : db2) b->release();
    D.tag2.release(); h->d_tag.release();
  }
  h->stage.release();
  cudaEventDestroy(h->run_e0); cudaEventDestroy(h->run_e1);
  cudaStreamDestroy(h->stream);
  delete h;
  return 0;
}

const char *sh_last_error(const sh_ctx *h) { return h ? h->err.c_str() : "null handle"; }

int sh_set_box(sh_ctx *h, const double lo[3], const double hi[3], const int periodic[3]) {
  for (int d = 0; d < 3; d++) if (!(hi[d] > lo[d])) return fail(h, "box: hi <= lo");
  for (int d = 0; d < 3; d++) { h->lo[d] = lo[d]; h->hi[d] = hi[d]; h->periodic[d] = periodic[d] != 0; }
  // with the domain decomposition on this is the GLOBAL box; the engine-local periodic flags follow from the brick grid
  for (int d = 0; d < 3; d++) { h->dd.glo[d] = lo[d]; h->dd.ghi[d] = hi[d]; h->dd.gper[d] = periodic[d] != 0; }
  h->dd.geometry_ok = false; h->dd.borders_ok = false;
  h->box_set = true; h->forces_valid = false; h->list_valid = false;
  return 0;
}

int sh_set_quadrature(sh_ctx *h, int n_theta, int n_phi) {
  if (!h->shapes.empty()) return fail(h, "set_quadrature must precede add_shape");
  if (n_theta < 2 || n_phi < 4) return fail(h, "quadrature too small");
  if ((long)n_theta * n_phi > 65535) return fail(h, "quadrature has more than 65535 nodes");
  h->n_theta = n_theta; h->n_phi = n_phi;
  return 0;
}

int sh_add_shape(sh_ctx *h, int lmax, const double *a_lm, const double *b_lm, double density, int *shape_id_out) try {
  if ((int)h->shapes.size() >= SH_MAX_SHAPES) return fail(h, "too many shapes");
  ShapeTables t;
  std::string e = build_shape_tables(lmax, a_lm, b_lm, density, h->n_theta, h->n_phi, t, h->cube_n);
  if (!e.empty()) return fail(h, e);
  h->shapes.push_back(std::move(t));
  h->shapes_dirty = true; h->forces_valid = false; h->list_valid = false;
  if (shape_id_out) *shape_id_out = (int)h->shapes.size() - 1;
  return 0;
} catch (...) { return -99; }   // no C++ exception crosses the C ABI (out of memory / internal error)

int sh_get_shape_props(const sh_ctx *h, int shape, double *volume, double com[3], double inertia[3],
                       double quat_principal[4], double *rmax, double *rmin) {
  if (shape < 0 || shape >= (int)h->shapes.size()) return -1;
  const ShapeTables &s = h->shapes[shape];
  if (volume) *volume = s.volume;
  if (com) for (int d = 0; d < 3; d++) com[d] = s.com[d];
  if (inertia) for (int d = 0; d < 3; d++) inertia[d] = s.inertia[d];
  if (quat_principal) for (int d = 0; d < 4; d++) quat_principal[d] = s.quat_principal[d];
  if (rmax) *rmax = s.rmax;
  if (rmin) *rmin = s.rmin;
  return 0;
}

int sh_get_nodes(const sh_ctx *h, int shape, double *p, double *nds) {
  if (shape < 0 || shape >= (int)h->shapes.size()) return -1;
  const ShapeTables &s = h->shapes[shape];
  for (int k = 0; k < s.nq; k++)
    for (int d = 0; d < 3; d++) { if (p) p[3 * k + d] = s.node_p[d][k]; if (nds) nds[3 * k + d] = s.node_n[d][k]; }
  return 0;
}

int sh_set_atoms(sh_ctx *h, int64_t n_in, const int64_t *tag_in, const int *shape_in, const double *x_in, const double *v_in,
                 const double *quat_in, const double *angmom_in) try {
  if (n_in < 0 || n_in > (int64_t)1 << 30) return fail(h, "bad atom count");
  if (n_in > 0 && (!shape_in || !x_in)) return fail(h, "shape and x are required");
  const int ns = (int)h->shapes.size();
  for (int64_t i = 0; i < n_in; i++) if (shape_in[i] < 0 || shape_in[i] >= ns) return fail(h, "atom shape id out of range");
  if (quat_in) for (int64_t i = 0; i < n_in; i++) {
    const double *q = quat_in + 4 * i;
    if (!(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3] > 0)) return fail(h, "zero quaternion");
  }
  CU(cudaSetDevice(h->device));
  // domain decomposition: every rank is handed the same atoms (like create_atoms / read_data) and keeps the ones inside
  // its brick, wrapped into the global box
  std::vector<int64_t> keep;
  std::vector<double> xw, vw;
  const bool dd = h->dd.on;
  if (dd) {
    int rc;
    if ((rc = dd_setup_geometry(h))) return rc;
    dd_refresh_shifts(h);
    const DdGeom &G = h->dd.G;
    xw.assign(x_in, x_in + 3 * n_in);
    if (v_in) vw.assign(v_in, v_in + 3 * n_in); else vw.assign(3 * n_in, 0.0);
    for (int64_t i = 0; i < n_in; i++) {
      double *x = &xw[3 * i];
      if (G.gper[1]) {
        const double ny = std::floor((x[1] - G.glo[1]) / G.L[1]);
        if (ny != 0.0) { x[1] -= G.L[1] * ny; x[0] -= ny * G.le_offset; vw[3 * i] -= ny * G.le_vshear; }
      }
      if (G.gper[0]) x[0] -= G.L[0] * std::floor((x[0] - G.glo[0]) / G.L[0]);
      if (G.gper[2]) x[2] -= G.L[2] * std::floor((x[2] - G.glo[2]) / G.L[2]);
      int gi[3];
      for (int d = 0; d < 3; d++) { const int c = (int)std::floor((x[d] - G.glo[d]) / G.sub[d]); gi[d] = std::min(std::max(c, 0), G.pgrid[d] - 1); }
      if ((gi[0] * G.pgrid[1] + gi[1]) * G.pgrid[2] + gi[2] == h->dd.rank) keep.push_back(i);
    }
  }
  const int64_t n = dd ? (int64_t)keep.size() : n_in;
  const double *x = dd ? xw.data() : x_in, *v = dd ? vw.data() : v_in;
  auto src_index = [&](int64_t i) -> int64_t { return dd ? keep[i] : i; };
  const int st = (int)((n + (dd ? std::max<int64_t>(n / 4, 1024) : 0) + 31) / 32 * 32) + 32;
  try {
    h->x.ensure(3 * (size_t)st); h->v.ensure(3 * (size_t)st); h->q.ensure(4 * (size_t)st); h->L.ensure(3 * (size_t)st);
    h->shape.ensure(st); h->d_tag.ensure(st);
  } catch (std::string &e) { return fail(h, e); }
  { int rc = dd_ensure_derived(h, st); if (rc) return rc; }
  h->n = n; h->stride = st;
  std::vector<double> buf((size_t)4 * st, 0.0);
  auto up = [&](DevBuf<double> &dst, const double *src, int ncomp, bool is_quat) -> cudaError_t {
    std::fill(buf.begin(), buf.end(), 0.0);
    for (int64_t i = 0; i < n; i++) {
      const int64_t k = src_index(i);
      if (src) {
        double nn = 1.0;
        if (is_quat) nn = std::sqrt(src[4 * k] * src[4 * k] + src[4 * k + 1] * src[4 * k + 1] + src[4 * k + 2] * src[4 * k + 2] + src[4 * k + 3] * src[4 * k + 3]);
        for (int d = 0; d < ncomp; d++) buf[(size_t)d * st + i] = is_quat ? src[ncomp * k + d] / nn : src[ncomp * k + d];
      } else if (is_quat) buf[i] = 1.0;
    }
    return cudaMemcpy(dst.p, buf.data(), (size_t)ncomp * st * sizeof(double), cudaMemcpyHostToDevice);
  };
  CU(up(h->x, x, 3, false)); CU(up(h->v, v, 3, false)); CU(up(h->q, quat_in, 4, true)); CU(up(h->L, angmom_in, 3, false));
  CU(cudaMemset(h->f.p, 0, 3 * (size_t)st * 8)); CU(cudaMemset(h->tq.p, 0, 3 * (size_t)st * 8));
  CU(cudaMemset(h->wallf.p, 0, 6 * (size_t)st * 8)); CU(cudaMemset(h->ewall.p, 0, (size_t)st * 8));
  CU(cudaMemset(h->c0.p, 0, 3 * (size_t)st * 8));
  std::vector<int> sh(st, 0);
  for (int64_t i = 0; i < n; i++) sh[i] = shape_in[src_index(i)];
  CU(cudaMemcpy(h->shape.p, sh.data(), (size_t)st * sizeof(int), cudaMemcpyHostToDevice));
  h->tag.resize(n);
  for (int64_t i = 0; i < n; i++) h->tag[i] = tag_in ? tag_in[src_index(i)] : src_index(i) + 1;
  if (n > 0) CU(cudaMemcpy(h->d_tag.p, h->tag.data(), (size_t)n * sizeof(long long), cudaMemcpyHostToDevice));
  h->tags_host_valid = true;
  h->forces_valid = false; h->list_valid = false; h->npairs = 0; h->nentries = 0; h->nghost = 0;
  h->atoms_epoch++; h->cache_state = CACHE_INVALID;
  h->dd.borders_ok = false;
  return 0;
} catch (...) { return -99; }   // no C++ exception crosses the C ABI (out of memory / internal error)

int sh_pair_coeff(sh_ctx *h, int si, int sj, double k, double exponent) {
  if (si < 0 || sj < 0 || si >= SH_MAX_SHAPES || sj >= SH_MAX_SHAPES) return fail(h, "pair_coeff: shape out of range");
  if (!(k >= 0) || !(exponent >= 1.0)) return fail(h, "pair_coeff: need k >= 0, exponent >= 1");
  h->pk[si * SH_MAX_SHAPES + sj] = h->pk[sj * SH_MAX_SHAPES + si] = k;
  h->pm[si * SH_MAX_SHAPES + sj] = h->pm[sj * SH_MAX_SHAPES + si] = exponent;
  h->coeff_dirty = true; h->forces_valid = false;
  return 0;
}

int sh_pair_dissipation(sh_ctx *h, int si, int sj, double gamma_n, double gamma_t, double mu) {
  if (si < 0 || sj < 0 || si >= SH_MAX_SHAPES || sj >= SH_MAX_SHAPES) return fail(h, "pair_dissipation: shape out of range");
  if (!(gamma_n >= 0) || !(gamma_t >= 0) || !(mu >= 0)) return fail(h, "pair_dissipation: need gamma_n, gamma_t, mu >= 0");
  h->pgn[si * SH_MAX_SHAPES + sj] = h->pgn[sj * SH_MAX_SHAPES + si] = gamma_n;
  h->pgt[si * SH_MAX_SHAPES + sj] = h->pgt[sj * SH_MAX_SHAPES + si] = gamma_t;
  h->pmu[si * SH_MAX_SHAPES + sj] = h->pmu[sj * SH_MAX_SHAPES + si] = mu;
  h->dissip = false;
  for (size_t k = 0; k < h->pgn.size(); k++) if (h->pgn[k] > 0 || (h->pgt[k] > 0 && h->pmu[k] > 0)) h->dissip = true;
  const int gv = h->dissip ? 1 : 0;
  if (gv != h->dd.ghost_vel) { h->dd.ghost_vel = gv; h->dd.borders_ok = false; h->list_valid = false; }   // ghost records change width
  h->coeff_dirty = true; h->forces_valid = false;
  return 0;
}

int sh_add_wall(sh_ctx *h, const double point[3], const double normal[3], double k, double exponent) {
  if (h->walls.n >= 16) return fail(h, "too many walls");
  const double nn = std::sqrt(normal[0] * normal[0] + normal[1] * normal[1] + normal[2] * normal[2]);
  if (!(nn > 0)) return fail(h, "wall normal is zero");
  if (!(k >= 0) || !(exponent >= 1.0)) return fail(h, "wall: need k >= 0, exponent >= 1");
  const int w = h->walls.n++;
  for (int d = 0; d < 3; d++) { h->walls.c[w][d] = point[d]; h->walls.nrm[w][d] = normal[d] / nn; }
  h->walls.k[w] = k; h->walls.m[w] = exponent;
  h->forces_valid = false;
  return 0;
}

int sh_set_gravity(sh_ctx *h, const double g[3]) { for (int d = 0; d < 3; d++) h->g[d] = g[d]; return 0; }

int sh_set_neighbor(sh_ctx *h, double skin, int every, int check) {
  if (skin < 0) return fail(h, "skin < 0");
  if (every < 1) return fail(h, "every < 1");
  h->skin = skin; h->neigh_every = every; h->neigh_check = check != 0;
  h->list_valid = false; h->forces_valid = false;
  return 0;
}

int sh_set_damping(sh_ctx *h, double gamma_lin, double gamma_rot) {
  if (gamma_lin < 0 || gamma_rot < 0) return fail(h, "damping < 0");
  h->gamma_lin = gamma_lin; h->gamma_rot = gamma_rot;
  return 0;
}

int sh_set_timestep(sh_ctx *h, double dt) { if (!(dt > 0)) return fail(h, "dt <= 0"); h->dt = dt; return 0; }

int sh_set_pair_tuning(sh_ctx *h, int threads_per_cta, int ctas_per_sm, int variant) {
  if (threads_per_cta != 0 && threads_per_cta != 64 && threads_per_cta != 128 && threads_per_cta != 256 && threads_per_cta != 384 && threads_per_cta != 512)
    return fail(h, "threads_per_cta must be 0, 64, 128, 256 or 512");
  h->tune_threads = threads_per_cta; h->tune_ctas_per_sm = ctas_per_sm; h->tune_variant = variant;
  h->cache_state = CACHE_INVALID;
  return 0;
}

int sh_compute_forces(sh_ctx *h) try {
  CU(cudaSetDevice(h->device));
  int rc = setup_forces(h);
  if (rc) return rc;
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  return 0;
} catch (...) { return -99; }   // no C++ exception crosses the C ABI (out of memory / internal error)

// ---- one timestep in two halves, so that a multi-rank driver can put the ghost exchange between them
namespace {
int launch_integrate_initial(sh_ctx *h, int check_violation) {
  const int n = (int)(h->n - h->nghost);
  const double trig = neighbor_trigger(h), trig2 = trig * trig;
  const double damp_v = 1.0 - 0.5 * h->dt * h->gamma_lin, damp_L = 1.0 - 0.5 * h->dt * h->gamma_rot;
  if (n > 0) {
    integrate_initial_kernel<<<cdiv(n, 256), 256, 0, h->stream>>>(view(h), h->d_shapes.p, h->dt, h->g[0], h->g[1], h->g[2], trig2, h->scalars.p, damp_v, damp_L, check_violation);
    h->kernel_launches++;
  }
  h->time += h->dt;
  h->steps_since_build++;
  return 0;
}

int step_finish(sh_ctx *h, int rebuild) {
  int rc;
  const int n = (int)(h->n - h->nghost);
  const double damp_v = 1.0 - 0.5 * h->dt * h->gamma_lin, damp_L = 1.0 - 0.5 * h->dt * h->gamma_rot;
  if (!h->list_valid) {  // atoms were re-set mid-step (migration): poses of all atoms
    if ((rc = prepare(h))) return rc;
    if (h->n > 0) {
      pose_kernel<<<cdiv(h->n, 256), 256, 0, h->stream>>>(view_all(h), h->d_shapes.p, -1.0, h->scalars.p + 1, 0, (int)h->n);
      h->kernel_launches++;
    }
  } else if (h->nghost > 0) {   // ghost poses from the freshly received x / quat
    pose_kernel<<<cdiv(h->nghost, 256), 256, 0, h->stream>>>(view_all(h), h->d_shapes.p, -1.0, h->scalars.p + 1, n, (int)h->nghost);
    h->kernel_launches++;
  }
  if (rebuild || !h->list_valid) { if ((rc = build_neighbors(h))) return rc; }
  if ((rc = compute_forces_device(h))) return rc;
  if (n > 0) {
    integrate_final_kernel<<<cdiv(n, 256), 256, 0, h->stream>>>(view(h), h->d_shapes.p, h->dt, h->g[0], h->g[1], h->g[2], damp_v, damp_L);
    h->kernel_launches++;
  }
  return 0;
}

// before a decomposed rebuild renumbers the atoms: keep what the candidate cache needs to survive it (old tags and
// origins to recognise the atoms, the cache's reference state, the old pair list, a hash of the old ghosts by tag)
int cache_snapshot(sh_ctx *h) {
  const int n = (int)h->n, nown = (int)(h->n - h->nghost), st = h->stride, ng = (int)h->nghost;
  int hs = 64;
  while (hs < 2 * ng + 2) hs <<= 1;
  try {
    h->old_c.ensure(3 * (size_t)st); h->old_cc0.ensure(3 * (size_t)st); h->old_cq0.ensure(4 * (size_t)st); h->old_tag.ensure((size_t)n + 2);
    h->old_half_off.ensure((size_t)nown + 2); h->old_pair_j.ensure((size_t)h->npairs + 1); h->ghost_hash.ensure(hs);
  } catch (std::string &e) { return fail(h, e); }
  CU(cudaMemcpyAsync(h->old_c.p, h->c.p, 3 * (size_t)st * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  CU(cudaMemcpyAsync(h->old_cc0.p, h->cc0.p, 3 * (size_t)st * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  CU(cudaMemcpyAsync(h->old_cq0.p, h->cq0.p, 4 * (size_t)st * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  CU(cudaMemcpyAsync(h->old_tag.p, h->d_tag.p, (size_t)n * sizeof(long long), cudaMemcpyDeviceToDevice, h->stream));
  CU(cudaMemcpyAsync(h->old_half_off.p, h->half_off.p, ((size_t)nown + 1) * sizeof(int), cudaMemcpyDeviceToDevice, h->stream));
  CU(cudaMemcpyAsync(h->old_pair_j.p, h->pair_j.p, (size_t)h->npairs * sizeof(int), cudaMemcpyDeviceToDevice, h->stream));
  CU(cudaMemsetAsync(h->ghost_hash.p, 0xff, (size_t)hs * sizeof(int), h->stream));
  if (ng > 0) { dd_ghost_hash_kernel<<<cdiv(ng, 256), 256, 0, h->stream>>>(h->old_tag.p, nown, ng, h->ghost_hash.p, hs); h->kernel_launches++; }
  h->old_n = n; h->old_nown = nown; h->old_stride = st; h->ghost_hash_size = hs;
  h->carry = true;
  return 0;
}

// One full timestep of sh_run.  With the lagged neighbor decision (default) the host never waits for the step it is
// enqueuing: whether step s rebuilds was predicted by the integrator of step s-1 (sc[5]) and arrives through a pinned
// slot + event; a misprediction is counted (sc[6]) and reported as an error by sh_run.
int step_once(sh_ctx *h) {
  int rc;
  const bool dd = h->dd.on;
  const bool due = h->steps_since_build + 1 >= h->neigh_every;
  const bool lag = h->lag_mode && h->neigh_check;
  int rebuild = 0;
  bool decided = false;
  if (!due) decided = true;
  else if (!h->neigh_check) { rebuild = 1; decided = true; }
  h->step_index++;
  h->cache_sync_ranks = lag && dd && h->dd.nranks > 1;
  if (lag && h->lag_pending) {   // no prediction in flight (first step, or the step after a rebuild): classic decision below
    CU(cudaEventSynchronize(h->ev_lag[h->lag_slot]));
    const int soft = h->h_lagflag[4 + 2 * h->lag_slot], pred = h->h_lagflag[5 + 2 * h->lag_slot];
    h->lag_pending = false;
    if (!decided && h->lag_pred_valid) { rebuild = pred; decided = true; }
    // cache request of ANY rank, as of two pair phases ago; the flags a cache build resets are stale for one more step
    if (h->cache_sync_ranks && soft && h->cache_state == CACHE_VALID && h->step_index > h->cache_build_step + 2) { h->cache_state = CACHE_INVALID; h->cache_exhausted = true; }
  }
  if ((rc = launch_integrate_initial(h, decided && !rebuild))) return rc;
  if (!decided) {   // classic decision: this step's own displacement flag, one host round trip
    if ((rc = reduce_flag(h, h->scalars.p + 1))) return rc;
    CU(cudaMemcpyAsync(h->h_pinned + 4, h->scalars.p + 1, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    rebuild = h->h_pinned[4] != 0;
  }
  if (lag) {
    // sc[4] (cache nearly used up, sticky until the cache is rebuilt) and sc[5] (prediction) -> MAX over ranks in sc[10..11]
    if (h->cache_sync_ranks || !rebuild) {
      if (dd && h->dd.nranks > 1) NC(h->dd.nccl->AllReduce(h->scalars.p + 4, h->scalars.p + 10, 2, ncclInt, ncclMax, h->dd.comm, h->stream));
      else CU(cudaMemcpyAsync(h->scalars.p + 10, h->scalars.p + 4, 2 * sizeof(int), cudaMemcpyDeviceToDevice, h->stream));
      h->lag_slot ^= 1;
      CU(cudaMemcpyAsync(h->h_lagflag + 4 + 2 * h->lag_slot, h->scalars.p + 10, 2 * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
      CU(cudaEventRecord(h->ev_lag[h->lag_slot], h->stream));
      h->lag_pending = true;
      h->lag_pred_valid = !rebuild;   // a prediction made on a rebuild step refers to the old origins: dropped
    }
    CU(cudaMemsetAsync(h->scalars.p + 5, 0, sizeof(int), h->stream));
  }
  if (dd && rebuild) {
    h->carry = false;
    const bool split = !(h->tune_variant & (1 | 2 | 4 | 8 | 32)) && ((h->tune_variant & 16) || h->npairs >= 16384);
    if (split && h->cache_state == CACHE_VALID && h->list_valid && h->npairs > 0 && h->atoms_epoch == h->cache_epoch &&
        h->cache_level + 1 < SH_CACHE_LEVELS) { if ((rc = cache_snapshot(h))) return rc; }
    const bool carry = h->carry;
    if ((rc = dd_rebuild(h))) return rc;
    h->carry = carry;
  } else if (dd) { if ((rc = dd_forward(h))) return rc; }
  return step_finish(h, rebuild);
}
}  // namespace

int sh_step_begin(sh_ctx *h, int *rebuild_wanted) try {
  CU(cudaSetDevice(h->device));
  int rc;
  if (!h->forces_valid || !h->list_valid) { if ((rc = setup_forces(h))) return rc; }
  if (rebuild_wanted) *rebuild_wanted = 0;
  if (h->n == 0) return 0;
  const bool due = h->steps_since_build + 1 >= h->neigh_every;
  if ((rc = launch_integrate_initial(h, 0))) return rc;
  h->lag_pending = false;
  bool rebuild = false;
  if (due) {
    if (h->neigh_check) {
      CU(cudaMemcpyAsync(h->h_pinned + 4, h->scalars.p + 1, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
      CU(cudaStreamSynchronize(h->stream));
      rebuild = h->h_pinned[4] != 0;
    } else rebuild = true;
  }
  if (rebuild_wanted) *rebuild_wanted = rebuild ? 1 : 0;
  return 0;
} catch (...) { return -99; }   // no C++ exception crosses the C ABI (out of memory / internal error)

int sh_step_end(sh_ctx *h, int rebuild) try {
  CU(cudaSetDevice(h->device));
  if (h->n == 0) return 0;
  return step_finish(h, rebuild);
} catch (...) { return -99; }   // no C++ exception crosses the C ABI (out of memory / internal error)

int sh_run(sh_ctx *h, int64_t nsteps) try {
  CU(cudaSetDevice(h->device));
  int rc;
  if (!h->forces_valid || !h->list_valid) { if ((rc = setup_forces(h))) return rc; }
  if (h->n == 0 && !h->dd.on) return 0;
  CU(cudaEventRecord(h->run_e0, h->stream));
  const bool trace = h->step_trace && nsteps <= 4096;
  if (trace) {
    while ((int64_t)h->ev_step.size() < nsteps + 1) { cudaEvent_t e; CU(cudaEventCreate(&e)); h->ev_step.push_back(e); }
    CU(cudaEventRecord(h->ev_step[0], h->stream));
    h->step_flags.assign(nsteps, 0);
  }
  for (int64_t step = 0; step < nsteps; step++) {
    const int64_t nb0 = h->neighbor_builds, cb0 = h->cache_builds, cr0 = h->cache_remaps;
    const long long al0 = devbuf_stats().allocs;
    if ((rc = step_once(h))) return rc;
    if (trace) {
      CU(cudaEventRecord(h->ev_step[step + 1], h->stream));
      h->step_flags[step] = (h->neighbor_builds > nb0 ? 1 : 0) | (h->cache_builds > cb0 ? 2 : 0) | (h->cache_remaps > cr0 ? 4 : 0) |
                            (devbuf_stats().allocs > al0 ? 8 : 0);
    }
  }
  CU(cudaMemcpyAsync(h->h_lagflag + 2, h->scalars.p + 6, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  if (h->dd.peer.d_err) CU(cudaMemcpyAsync(h->h_lagflag + 3, h->dd.peer.d_err, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaEventRecord(h->run_e1, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  { float ms = 0; cudaEventElapsedTime(&ms, h->run_e0, h->run_e1); h->sec_run_last = ms * 1e-3; h->sec_run_total += h->sec_run_last; }
  if (trace) {
    h->step_ms.assign(nsteps, 0.f);
    for (int64_t k = 0; k < nsteps; k++) cudaEventElapsedTime(&h->step_ms[k], h->ev_step[k], h->ev_step[k + 1]);
    h->step_flags_last = h->step_flags;
  } else h->step_ms.clear();
  if (h->dd.peer.d_err && h->h_lagflag[3] != 0) return fail(h, "ghost exchange over peer memory timed out waiting for a neighbour rank");
  if (h->h_lagflag[2] != 0) {
    CU(cudaMemset(h->scalars.p + 6, 0, sizeof(int)));
    return fail(h, "neighbor skin violated: an atom moved more than half the skin on a step the lagged neighbor decision did not "
                   "rebuild on (increase the skin, or sh_set_tuning \"sync_rebuild\" 1)");
  }
  return 0;
} catch (...) { return -99; }   // no C++ exception crosses the C ABI (out of memory / internal error)

// ---- multi-rank support: the last nghost atoms of the arrays are ghosts (copies of atoms owned by
// other ranks / periodic images): they take part in pairs with owned atoms but receive no force,
// are not integrated and carry no neighbor-list rows.  Device-pointer pack / unpack for the per-step
// forward exchange of ghost x and quat (SURVEY §5.8, §8 a12); the transport itself is NCCL
// point-to-point issued by the host driver (lammps-spherharm_b200/decomp.py).
int sh_set_ghost_count(sh_ctx *h, int64_t nghost) {
  if (nghost < 0 || nghost > h->n) return fail(h, "ghost count out of range");
  h->nghost = nghost; h->forces_valid = false; h->list_valid = false;
  return 0;
}
int sh_pack_atoms(sh_ctx *h, int64_t m, const int *d_idx, const double *d_shift, double *d_out) {
  CU(cudaSetDevice(h->device));
  if (m > 0) {
    pack_atoms_kernel<<<cdiv(m, 256), 256, 0, h->stream>>>(view_all(h), (int)m, d_idx, d_shift, d_out);
    h->kernel_launches++;
  }
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}
int sh_unpack_ghosts(sh_ctx *h, int64_t first, int64_t m, const double *d_in) {
  CU(cudaSetDevice(h->device));
  if (first < 0 || first + m > h->n) return fail(h, "unpack range out of bounds");
  if (m > 0) {
    unpack_atoms_kernel<<<cdiv(m, 256), 256, 0, h->stream>>>(view_all(h), (int)first, (int)m, d_in);
    h->kernel_launches++;
  }
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}
// CUDA-event stopwatch on the library's stream (for drivers that step through sh_step_begin/end)
int sh_mark_begin(sh_ctx *h) {
  CU(cudaSetDevice(h->device));
  CU(cudaEventRecord(h->run_e0, h->stream));
  return 0;
}
int sh_mark_end(sh_ctx *h, double *seconds) {
  CU(cudaSetDevice(h->device));
  CU(cudaEventRecord(h->run_e1, h->stream));
  CU(cudaEventSynchronize(h->run_e1));
  float ms = 0;
  CU(cudaEventElapsedTime(&ms, h->run_e0, h->run_e1));
  if (seconds) *seconds = ms * 1e-3;
  return 0;
}
int sh_synchronize(sh_ctx *h) {
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaGetLastError());
  return 0;
}

int sh_get_run_time(const sh_ctx *h, double *seconds_last_run, double *seconds_total) {
  if (seconds_last_run) *seconds_last_run = h->sec_run_last;
  if (seconds_total) *seconds_total = h->sec_run_total;
  return 0;
}

// Pair::compute-style offload: the caller owns the atoms, pushes x / quat (and optionally v, angmom)
// every step, keeps the neighbor list alive across calls (rebuilt when the skin is exhausted).
int sh_put_state(sh_ctx *h, int64_t n, const double *x, const double *v, const double *quat, const double *angmom) try {
  if (n != h->n) return fail(h, "put_state: n mismatch");
  CU(cudaSetDevice(h->device));
  if (n == 0) return 0;
  const int st = h->stride, nb = cdiv(n, 256);
  try { h->stage.ensure((size_t)4 * n); } catch (std::string &e) { return fail(h, e); }
  struct Item { const double *src; double *dst; int nc; int norm; } items[4] = {
      {x, h->x.p, 3, 0}, {v, h->v.p, 3, 0}, {quat, h->q.p, 4, 1}, {angmom, h->L.p, 3, 0}};
  for (auto &it : items) {
    if (!it.src) continue;
    CU(cudaMemcpyAsync(h->stage.p, it.src, (size_t)it.nc * n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    aos_to_soa_kernel<<<nb, 256, 0, h->stream>>>(h->stage.p, it.dst, (int)n, it.nc, st, it.norm);
    h->kernel_launches++;
  }
  CU(cudaStreamSynchronize(h->stream));
  h->forces_valid = false;
  return 0;
} catch (...) { return -99; }   // no C++ exception crosses the C ABI (out of memory / internal error)

int sh_get_forces(const sh_ctx *hc, int64_t n, double *f, double *torque) try {
  sh_ctx *h = const_cast<sh_ctx *>(hc);
  if (n < 0 || n > h->n) return fail(h, "get_forces: n out of range");
  CU(cudaSetDevice(h->device));
  if (n == 0) return 0;
  const int st = h->stride, nb = cdiv(n, 256);
  try { h->stage.ensure((size_t)6 * n); } catch (std::string &e) { return fail(h, e); }
  soa_to_aos_kernel<<<nb, 256, 0, h->stream>>>(h->f.p, h->stage.p, (int)n, 3, st);
  soa_to_aos_kernel<<<nb, 256, 0, h->stream>>>(h->tq.p, h->stage.p + 3 * n, (int)n, 3, st);
  h->kernel_launches += 2;
  if (f) CU(cudaMemcpyAsync(f, h->stage.p, (size_t)3 * n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (torque) CU(cudaMemcpyAsync(torque, h->stage.p + 3 * n, (size_t)3 * n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
} catch (...) { return -99; }   // no C++ exception crosses the C ABI (out of memory / internal error)

// ---- checkpoint / resume (write_restart / read_restart of the atom style: AtomVec::pack_restart): binary
// snapshot of the owned atoms.  Shapes, coefficients and fixes are re-issued by the input script, as in LAMMPS.
namespace {
struct SnapHeader { char magic[8]; int32_t version, nshapes; int64_t n, step; double lo[3], hi[3]; int32_t periodic[3], pad; };
}
int sh_write_snapshot(const sh_ctx *hc, const char *path, int64_t step) try {
  sh_ctx *h = const_cast<sh_ctx *>(hc);
  const int64_t n = h->n - h->nghost;
  { int rc = sync_tags_host(h); if (rc) return rc; }
  std::vector<double> x(3 * n), v(3 * n), q(4 * n), L(3 * n);
  if (n > 0) { int rc = sh_get_atoms(h, n, x.data(), v.data(), q.data(), L.data(), nullptr, nullptr); if (rc) return rc; }
  std::vector<int> shp(h->stride > 0 ? h->stride : 1);
  if (n > 0) CU(cudaMemcpy(shp.data(), h->shape.p, n * sizeof(int), cudaMemcpyDeviceToHost));
  FILE *f = fopen(path, "wb");
  if (!f) return fail(h, std::string("cannot open snapshot file ") + path);
  SnapHeader hd{};
  std::memcpy(hd.magic, "SHGPUSNP", 8);
  hd.version = 1; hd.nshapes = (int)h->shapes.size(); hd.n = n; hd.step = step;
  for (int d = 0; d < 3; d++) { hd.lo[d] = h->dd.glo[d]; hd.hi[d] = h->dd.ghi[d]; hd.periodic[d] = h->dd.gper[d]; }   // the global box
  bool ok = fwrite(&hd, sizeof hd, 1, f) == 1;
  ok = ok && (n == 0 || (fwrite(h->tag.data(), sizeof(int64_t), n, f) == (size_t)n && fwrite(shp.data(), sizeof(int), n, f) == (size_t)n &&
                         fwrite(x.data(), 8, 3 * n, f) == (size_t)(3 * n) && fwrite(v.data(), 8, 3 * n, f) == (size_t)(3 * n) &&
                         fwrite(q.data(), 8, 4 * n, f) == (size_t)(4 * n) && fwrite(L.data(), 8, 3 * n, f) == (size_t)(3 * n)));
  fclose(f);
  if (!ok) return fail(h, "short write to snapshot file");
  return 0;
} catch (...) { return -99; }   // no C++ exception crosses the C ABI (out of memory / internal error)
int sh_read_snapshot(sh_ctx *h, const char *path, int64_t *step_out) try {
  FILE *f = fopen(path, "rb");
  if (!f) return fail(h, std::string("cannot open snapshot file ") + path);
  SnapHeader hd{};
  if (fread(&hd, sizeof hd, 1, f) != 1 || std::memcmp(hd.magic, "SHGPUSNP", 8) != 0 || hd.version != 1) { fclose(f); return fail(h, "not a shgpu snapshot (bad header)"); }
  if (hd.nshapes != (int)h->shapes.size()) { fclose(f); return fail(h, "snapshot was written with a different number of shapes"); }
  const int64_t n = hd.n;
  if (n < 0 || n > ((int64_t)1 << 30)) { fclose(f); return fail(h, "bad atom count in snapshot"); }
  {   // the payload must really be there before anything is allocated for it (ADVICE r1)
    const long pos = ftell(f);
    fseek(f, 0, SEEK_END);
    const long end = ftell(f);
    fseek(f, pos, SEEK_SET);
    if (end - pos < (long)(n * (int64_t)(sizeof(int64_t) + sizeof(int) + 13 * sizeof(double)))) { fclose(f); return fail(h, "truncated snapshot file"); }
  }
  std::vector<int64_t> tag(n); std::vector<int> shp(n);
  std::vector<double> x(3 * n), v(3 * n), q(4 * n), L(3 * n);
  bool ok = n == 0 || (fread(tag.data(), sizeof(int64_t), n, f) == (size_t)n && fread(shp.data(), sizeof(int), n, f) == (size_t)n &&
                       fread(x.data(), 8, 3 * n, f) == (size_t)(3 * n) && fread(v.data(), 8, 3 * n, f) == (size_t)(3 * n) &&
                       fread(q.data(), 8, 4 * n, f) == (size_t)(4 * n) && fread(L.data(), 8, 3 * n, f) == (size_t)(3 * n));
  fclose(f);
  if (!ok) return fail(h, "truncated snapshot file");
  int rc = sh_set_box(h, hd.lo, hd.hi, hd.periodic);
  if (rc) return rc;
  rc = sh_set_atoms(h, n, tag.data(), shp.data(), x.data(), v.data(), q.data(), L.data());
  if (rc) return rc;
  if (step_out) *step_out = hd.step;
  return 0;
} catch (...) { return -99; }   // no C++ exception crosses the C ABI (out of memory / internal error)

int sh_get_natoms(const sh_ctx *h, int64_t *n) { if (n) *n = h->n; return 0; }

int sh_get_atoms(const sh_ctx *hc, int64_t n, double *x, double *v, double *quat, double *angmom, double *f, double *torque) try {
  sh_ctx *h = const_cast<sh_ctx *>(hc);
  if (n < 0 || n > h->n) return fail(h, "get_atoms: n out of range");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  const int st = h->stride;
  std::vector<double> buf((size_t)4 * st);
  auto down = [&](const DevBuf<double> &src, double *dst, int ncomp) -> cudaError_t {
    if (!dst) return cudaSuccess;
    cudaError_t e = cudaMemcpy(buf.data(), src.p, (size_t)ncomp * st * sizeof(double), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return e;
    for (int64_t i = 0; i < n; i++) for (int d = 0; d < ncomp; d++) dst[ncomp * i + d] = buf[(size_t)d * st + i];
    return cudaSuccess;
  };
  CU(down(h->x, x, 3)); CU(down(h->v, v, 3)); CU(down(h->q, quat, 4)); CU(down(h->L, angmom, 3));
  CU(down(h->f, f, 3)); CU(down(h->tq, torque, 3));
  return 0;
} catch (...) { return -99; }   // no C++ exception crosses the C ABI (out of memory / internal error)

int sh_get_pairs(const sh_ctx *hc, int64_t cap, int64_t *npairs, int64_t *tag_i, int64_t *tag_j, double *V, double *F,
                 double *tau_i, double *tau_j, double *centroid) try {
  sh_ctx *h = const_cast<sh_ctx *>(hc);
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  const int np = h->forces_valid ? h->npairs : 0;
  if (npairs) *npairs = np;
  { int rc = sync_tags_host(h); if (rc) return rc; }
  const int m = (int)std::min<int64_t>(np, cap);
  if (m <= 0) return 0;
  std::vector<int> pi(m), pj(m);
  CU(cudaMemcpy(pi.data(), h->pair_i.p, m * sizeof(int), cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(pj.data(), h->pair_j.p, m * sizeof(int), cudaMemcpyDeviceToHost));
  std::vector<double> buf((size_t)14 * m);
  for (int r = 0; r < 14; r++)
    CU(cudaMemcpy(buf.data() + (size_t)r * m, h->pres.p + (size_t)r * h->pres_stride, m * sizeof(double), cudaMemcpyDeviceToHost));
  for (int k = 0; k < m; k++) {
    if (tag_i) tag_i[k] = h->tag[pi[k]];
    if (tag_j) tag_j[k] = h->tag[pj[k]];
    if (V) V[k] = buf[k];
    for (int r = 0; r < 3; r++) {
      if (F) F[3 * k + r] = buf[(size_t)(2 + r) * m + k];
      if (tau_i) tau_i[3 * k + r] = buf[(size_t)(5 + r) * m + k];
      if (tau_j) tau_j[3 * k + r] = buf[(size_t)(8 + r) * m + k];
      if (centroid) centroid[3 * k + r] = buf[(size_t)(11 + r) * m + k];
    }
  }
  return 0;
} catch (...) { return -99; }   // no C++ exception crosses the C ABI (out of memory / internal error)

int sh_get_energy(const sh_ctx *hc, double *ke_trans, double *ke_rot, double *e_contact) try {
  sh_ctx *h = const_cast<sh_ctx *>(hc);
  CU(cudaSetDevice(h->device));
  const int n = (int)(h->n - h->nghost);
  double kt = 0, kr = 0, ec = 0;
  if (n > 0) {
    int rc = prepare(h);
    if (rc) return rc;
    energy_kernel<<<cdiv(n, 256), 256, 0, h->stream>>>(view(h), h->d_shapes.p, h->ke.p);
    h->kernel_launches++;
    CU(cudaStreamSynchronize(h->stream));
    std::vector<double> buf(2 * (size_t)n);
    CU(cudaMemcpy(buf.data(), h->ke.p, 2 * (size_t)n * sizeof(double), cudaMemcpyDeviceToHost));
    for (int i = 0; i < n; i++) { kt += buf[i]; kr += buf[n + i]; }
    if (h->forces_valid) {
      if (h->npairs > 0) {
        std::vector<double> e(h->npairs);
        CU(cudaMemcpy(e.data(), h->pres.p + (size_t)h->pres_stride, h->npairs * sizeof(double), cudaMemcpyDeviceToHost));
        for (double vv : e) ec += vv;
      }
      if (h->walls.n > 0) {
        std::vector<double> e(n);
        CU(cudaMemcpy(e.data(), h->ewall.p, n * sizeof(double), cudaMemcpyDeviceToHost));
        for (double vv : e) ec += vv;
      }
    }
  }
  if (ke_trans) *ke_trans = kt;
  if (ke_rot) *ke_rot = kr;
  if (e_contact) *e_contact = ec;
  return 0;
} catch (...) { return -99; }   // no C++ exception crosses the C ABI (out of memory / internal error)

// pressure-tensor sums of this rank (compute pressure in LAMMPS terms): fixed-order two-level reduction, no FP atomics
int sh_get_stress(const sh_ctx *hc, double virial[9], double kinetic[9]) try {
  sh_ctx *h = const_cast<sh_ctx *>(hc);
  CU(cudaSetDevice(h->device));
  const int n = (int)(h->n - h->nghost), np = h->forces_valid ? h->npairs : 0;
  const int nb_atoms = std::max(1, cdiv(n, 256)), nb_pairs = std::max(1, cdiv(np, 256));
  try { h->stress_part.ensure((size_t)9 * (nb_atoms + nb_pairs)); } catch (std::string &e) { return fail(h, e); }
  double K[9] = {0}, W[9] = {0};
  if (n > 0) {
    int rc = prepare(h);
    if (rc) return rc;
    stress_kinetic_kernel<<<nb_atoms, 256, 0, h->stream>>>(view(h), h->d_shapes.p, h->stress_part.p);
    h->kernel_launches++;
  }
  if (np > 0) {
    // newton on: a pair with a ghost is evaluated by one rank only and counts fully there
    stress_virial_kernel<<<nb_pairs, 256, 0, h->stream>>>(view_all(h), np, h->nrows > n ? (int)h->n : n, h->pair_i.p, h->pair_j.p, h->pair_img.p, h->pres.p, h->pres_stride,
                                                          h->hi[0] - h->lo[0], h->hi[1] - h->lo[1], h->hi[2] - h->lo[2], h->stress_part.p + (size_t)9 * nb_atoms);
    h->kernel_launches++;
  }
  CU(cudaStreamSynchronize(h->stream));
  std::vector<double> part((size_t)9 * (nb_atoms + nb_pairs), 0.0);
  CU(cudaMemcpy(part.data(), h->stress_part.p, part.size() * sizeof(double), cudaMemcpyDeviceToHost));
  if (n > 0) for (int b = 0; b < nb_atoms; b++) for (int k = 0; k < 9; k++) K[k] += part[(size_t)9 * b + k];
  if (np > 0) for (int b = 0; b < nb_pairs; b++) for (int k = 0; k < 9; k++) W[k] += part[(size_t)9 * (nb_atoms + b) + k];
  for (int k = 0; k < 9; k++) { if (virial) virial[k] = W[k]; if (kinetic) kinetic[k] = K[k]; }
  return 0;
} catch (...) { return -99; }   // no C++ exception crosses the C ABI (out of memory / internal error)

// per-atom virial / kinetic tensor / contact energy / contact count of the owned atoms (compute stress/atom, pe/atom,
// contact/atom).  Fixed-order sums over the CSR rows, no FP atomics; nothing here is part of a step.  Newton on in the
// in-library decomposition: the ghost rows' halves go back to their owners through the reverse plan (collective).
int sh_get_atom_stress(const sh_ctx *hc, int64_t n, int mode, double *virial, double *kinetic, double *energy, int *contacts) try {
  sh_ctx *h = const_cast<sh_ctx *>(hc);
  const int nown = (int)(h->n - h->nghost);
  if (n < 0 || n > nown) return fail(h, "get_atom_stress: n out of range");
  if (mode != 0 && mode != 1) return fail(h, "get_atom_stress: mode must be 0 (centre-to-centre) or 1 (contact centroid)");
  CU(cudaSetDevice(h->device));
  int rc = prepare(h);
  if (rc) return rc;
  DdCtx &D = h->dd;
  const bool newton_dd = D.on && D.newton && D.borders_ok && (h->nghost > 0 || D.nsend > 0);
  const bool pairs = h->forces_valid && h->list_valid && h->npairs > 0;
  const int nall = newton_dd ? (int)h->n : nown;
  const int nrows = pairs ? std::min(h->nrows, nall) : 0;
  try {
    h->as_vir.ensure((size_t)9 * std::max(nown, 1)); h->as_kin.ensure((size_t)9 * std::max(nown, 1));
    h->as_en.ensure(std::max(nown, 1)); h->as_cnt.ensure(std::max(nown, 1));
    if (pairs) h->as_epair.ensure((size_t)h->nentries + 1);
    if (newton_dd) { h->as_send.ensure((size_t)11 * std::max<int64_t>(h->nghost, 1)); h->as_recv.ensure((size_t)11 * std::max(D.nsend, 1)); }
  } catch (std::string &e) { return fail(h, e); }
  if (pairs) {
    CU(cudaMemsetAsync(h->as_epair.p, 0xff, (size_t)h->nentries * sizeof(int), h->stream));
    atom_stress_entry_pair_kernel<<<cdiv(h->npairs, 256), 256, 0, h->stream>>>(h->npairs, h->pair_eij.p, h->pair_eji.p, h->as_epair.p);
    h->kernel_launches++;
  }
  if (nall > 0) {
    AtomStressArgs S;
    S.A = view(h); S.shapes = h->d_shapes.p; S.nall = nall; S.nrows = nrows; S.mode = mode;
    S.nbr_off = h->nbr_off.p; S.epair = h->as_epair.p; S.pair_i = h->pair_i.p; S.pair_j = h->pair_j.p; S.pair_img = h->pair_img.p;
    S.pres = h->pres.p; S.pres_stride = h->pres_stride;
    for (int d = 0; d < 3; d++) S.L[d] = h->hi[d] - h->lo[d];
    S.ewall = h->forces_valid && h->walls.n > 0 ? h->ewall.p : nullptr;
    S.vir = h->as_vir.p; S.kin = h->as_kin.p; S.en = h->as_en.p; S.cnt = h->as_cnt.p; S.ghost_rec = h->as_send.p;
    atom_stress_row_kernel<<<cdiv(nall, 128), 128, 0, h->stream>>>(S);
    h->kernel_launches++;
  }
  if (newton_dd) {
    if ((rc = dd_sendrecv(h, D.nbr_rank, h->as_send.p, D.recv_cnt, h->as_recv.p, D.send_cnt, 11))) return rc;
    if (D.nsend > 0 && nown > 0) {
      atom_stress_add_returned_kernel<<<cdiv(nown, 256), 256, 0, h->stream>>>(nown, D.rev_off.p, D.rev_k.p, h->as_recv.p, h->as_vir.p,
                                                                            h->as_en.p, h->as_cnt.p);
      h->kernel_launches++;
    }
  }
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(h->stream));
  if (n > 0) {
    if (virial) CU(cudaMemcpy(virial, h->as_vir.p, (size_t)9 * n * sizeof(double), cudaMemcpyDeviceToHost));
    if (kinetic) CU(cudaMemcpy(kinetic, h->as_kin.p, (size_t)9 * n * sizeof(double), cudaMemcpyDeviceToHost));
    if (energy) CU(cudaMemcpy(energy, h->as_en.p, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost));
    if (contacts) CU(cudaMemcpy(contacts, h->as_cnt.p, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost));
  }
  return 0;
} catch (...) { return -99; }   // no C++ exception crosses the C ABI (out of memory / internal error)

int sh_get_ghost_pair_evals(const sh_ctx *hc, int64_t *ghost_pair_evals) {
  sh_ctx *h = const_cast<sh_ctx *>(hc);
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  unsigned long long c = 0;
  CU(cudaMemcpy(&c, h->counters.p + 4, sizeof c, cudaMemcpyDeviceToHost));
  if (h->dd.on && h->dd.newton) c = 0;   // newton on: no pair is evaluated twice
  if (ghost_pair_evals) *ghost_pair_evals = (int64_t)c;
  return 0;
}

int sh_get_counters(const sh_ctx *hc, int64_t *pair_evals, int64_t *nodes_transformed, int64_t *nodes_evaluated,
                    int64_t *nodes_inside, int64_t *neighbor_builds, int64_t *kernel_launches) {
  sh_ctx *h = const_cast<sh_ctx *>(hc);
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  unsigned long long c[4];
  CU(cudaMemcpy(c, h->counters.p, sizeof c, cudaMemcpyDeviceToHost));
  if (pair_evals) *pair_evals = (int64_t)c[0];
  if (nodes_transformed) *nodes_transformed = (int64_t)c[1];
  if (nodes_evaluated) *nodes_evaluated = (int64_t)c[2];
  if (nodes_inside) *nodes_inside = (int64_t)c[3];
  if (neighbor_builds) *neighbor_builds = h->neighbor_builds;
  if (kernel_launches) *kernel_launches = h->kernel_launches;
  return 0;
}

int sh_get_timers(const sh_ctx *hc, double *seconds_pair, int64_t *pair_launches, double *seconds_neigh, double *seconds_other) {
  sh_ctx *h = const_cast<sh_ctx *>(hc);
  CU(cudaSetDevice(h->device));
  int rc = drain_events(h);
  if (rc) return rc;
  if (seconds_pair) *seconds_pair = h->sec_pair;
  if (pair_launches) *pair_launches = h->pair_launches;
  if (seconds_neigh) *seconds_neigh = h->sec_neigh;
  if (seconds_other) *seconds_other = h->sec_comm;   // ghost exchange, reverse communication, migration + borders
  return 0;
}

int sh_get_counter_raw(const sh_ctx *hc, int index, int64_t *value) {
  sh_ctx *h = const_cast<sh_ctx *>(hc);
  if (index < 0 || index >= 8) return fail(h, "counter index out of range");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  unsigned long long c = 0;
  CU(cudaMemcpy(&c, h->counters.p + index, sizeof c, cudaMemcpyDeviceToHost));
  if (value) *value = (int64_t)c;
  return 0;
}

int sh_get_split_times(const sh_ctx *hc, double *seconds_cull, double *seconds_eval, double *seconds_reduce, double *seconds_deep) {
  sh_ctx *h = const_cast<sh_ctx *>(hc);
  CU(cudaSetDevice(h->device));
  int rc = drain_events(h);
  if (rc) return rc;
  if (seconds_cull) *seconds_cull = h->sec_cull;
  if (seconds_eval) *seconds_eval = h->sec_eval;
  if (seconds_reduce) *seconds_reduce = h->sec_reduce;
  if (seconds_deep) *seconds_deep = h->sec_deep;
  return 0;
}

int sh_get_split_stats(const sh_ctx *hc, double *seconds_eval, int64_t *eval_launches, int64_t *deep_pairs, int64_t *pool_redos,
                       int64_t *cache_builds) {
  sh_ctx *h = const_cast<sh_ctx *>(hc);
  CU(cudaSetDevice(h->device));
  int rc = drain_events(h);
  if (rc) return rc;
  if ((rc = absorb_split_feedback(h))) return rc;
  if (seconds_eval) *seconds_eval = h->sec_eval;
  if (eval_launches) *eval_launches = h->eval_launches;
  if (deep_pairs) *deep_pairs = h->big_pairs;
  if (pool_redos) *pool_redos = h->pool_grows;
  if (cache_builds) *cache_builds = h->cache_builds;
  return 0;
}

int sh_reset_timers(sh_ctx *h) {
  CU(cudaSetDevice(h->device));
  int rc = drain_events(h);
  if (rc) return rc;
  h->sec_pair = h->sec_neigh = h->sec_comm = h->sec_other = 0; h->pair_launches = 0; h->sec_run_total = 0;
  h->sec_eval = h->sec_cull = h->sec_reduce = h->sec_deep = 0; h->eval_launches = 0; h->big_pairs = 0; h->slow_pairs = 0; h->pool_grows = 0; h->cache_builds = 0; h->cache_remaps = 0; h->sec_cache = 0;
  h->neighbor_builds = 0; h->kernel_launches = 0;
  CU(cudaMemset(h->counters.p, 0, 16 * sizeof(unsigned long long)));
  return 0;
}

int sh_get_cache_stats(const sh_ctx *hc, int64_t *cache_builds, double *seconds_cache, int *level, int64_t *slow_pairs,
                       int64_t *cache_remaps) {
  sh_ctx *h = const_cast<sh_ctx *>(hc);
  CU(cudaSetDevice(h->device));
  int rc = drain_events(h);
  if (rc) return rc;
  if ((rc = absorb_split_feedback(h))) return rc;
  if (cache_builds) *cache_builds = h->cache_builds;
  if (seconds_cache) *seconds_cache = h->sec_cache;
  if (level) *level = h->cache_level;
  if (slow_pairs) *slow_pairs = h->slow_pairs;
  if (cache_remaps) *cache_remaps = h->cache_remaps;
  return 0;
}

int sh_set_tuning(sh_ctx *h, const char *key, double value) try {
  if (!h || !key) return -1;
  const std::string k(key);
  const int v = (int)value;
  if (k == "cull_wpb") { if (v != 0 && v != 1 && v != 2 && v != 4 && v != 8) return fail(h, "cull_wpb must be 0, 1, 2, 4 or 8"); h->tune_cull_wpb = v; }
  else if (k == "cull_lpp") { if (v != 0 && v != 16 && v != 32) return fail(h, "cull_lpp must be 0, 16 or 32"); h->tune_cull_lpp = v; }
  else if (k == "eval_pts") { if (v != 0 && v != 2 && v != 4) return fail(h, "eval_pts must be 0, 2 or 4"); h->eval_pts = v; }
  else if (k == "eval_occ") { if (v != 0 && v != 3 && v != 4) return fail(h, "eval_occ must be 0, 3 or 4"); h->eval_occ = v; }
  else if (k == "eval_mode") { if (v < 0 || v > 2) return fail(h, "eval_mode must be 0 (default), 1 (one block per CTA) or 2 (persistent chunks)"); h->eval_mode = v; }
  else if (k == "cache_level") { if (v < -1 || v >= SH_CACHE_LEVELS) return fail(h, "cache_level must be -1 (adaptive) .. 2"); if (v > 2) return fail(h, "cache_level must be -1 (adaptive) .. 2"); h->cache_level_pin = v; h->cache_state = CACHE_INVALID; }
  else if (k == "cube_n") {
    if (!h->shapes.empty()) return fail(h, "cube_n must be set before add_shape");
    if (v != 0 && (v < 8 || v > 144)) return fail(h, "cube_n must be 0 (default) or 8..144");
    h->cube_n = v;
  } else if (k == "peer_exchange") { h->dd.peer.want = v != 0; if (!h->dd.peer.want && h->dd.peer.enabled) return fail(h, "peer_exchange can only be switched off before the first run"); }
  else if (k == "newton") { h->dd.newton = v != 0; h->list_valid = false; h->forces_valid = false; }
  else if (k == "step_trace") { h->step_trace = v != 0; }
  else if (k == "dd_self_ghosts") { h->dd.self_ghosts = v != 0; h->dd.geometry_ok = false; h->dd.borders_ok = false; }
  else if (k == "sync_rebuild") { h->lag_mode = v == 0; h->lag_pending = false; }
  else return fail(h, "unknown tuning key: " + k);
  return 0;
} catch (...) { return -99; }   // no C++ exception crosses the C ABI (out of memory / internal error)

int sh_measure_fp64_peak(sh_ctx *h, double *flops_per_s, double *sm_clock_mhz_est) {
  CU(cudaSetDevice(h->device));
  const int threads = 256, blocks = h->sm_count * 8, iters = 4096;
  DevBuf<double> out;
  try { out.ensure((size_t)threads * blocks); } catch (std::string &e) { return fail(h, e); }
  cudaEvent_t e0, e1;
  CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
  double best = 0;
  for (int rep = 0; rep < 5; rep++) {
    CU(cudaEventRecord(e0, h->stream));
    dfma_peak_kernel<<<blocks, threads, 0, h->stream>>>(out.p, iters, 1.0000001, 1e-9);
    CU(cudaEventRecord(e1, h->stream));
    CU(cudaEventSynchronize(e1));
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    const double fl = 2.0 * 64.0 * iters * (double)threads * blocks / (ms * 1e-3);
    if (rep > 0) best = std::max(best, fl);
  }
  h->kernel_launches += 5;
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  out.release();
  if (flops_per_s) *flops_per_s = best;
  if (sm_clock_mhz_est) *sm_clock_mhz_est = best / (2.0 * 64.0 * h->sm_count) * 1e-6;  // if 64 FP64 lanes/SM
  CU(cudaGetLastError());
  return 0;
}

// ---- multi-GPU behind the C ABI (SURVEY §8b): one handle per rank; NCCL inside the library ------------------------
int sh_dd_unique_id(char *id, int cap) {
  if (!id || cap < (int)sizeof(ncclUniqueId)) return -1;
  NcclApi *api = nccl_api();
  if (!api) return -8;
  ncclUniqueId u;
  if (api->GetUniqueId(&u) != ncclSuccess) return -9;
  std::memcpy(id, &u, sizeof u);
  return 0;
}

int sh_dd_init(sh_ctx *h, int rank, int nranks, const char *id, const int *pgrid) try {
  if (!h) return -1;
  if (nranks < 1 || nranks > DD_MAX_RANKS || rank < 0 || rank >= nranks) return fail(h, "dd_init: bad rank / nranks (at most 64 ranks)");
  if (h->dd.on) return fail(h, "dd_init: already initialised");
  CU(cudaSetDevice(h->device));
  DdCtx &D = h->dd;
  D.rank = rank; D.nranks = nranks;
  if (nranks > 1) {
    if (!id) return fail(h, "dd_init: a unique id is required for more than one rank");
    D.nccl = nccl_api();
    if (!D.nccl) return fail(h, "dd_init: NCCL is not available (libnccl.so.2)");
    ncclUniqueId u;
    std::memcpy(&u, id, sizeof u);
    NC(D.nccl->CommInitRank(&D.comm, nranks, u, rank));
  }
  if (pgrid && pgrid[0] > 0 && pgrid[1] > 0 && pgrid[2] > 0) { for (int d = 0; d < 3; d++) D.pgrid[d] = pgrid[d]; D.pgrid_set = true; }
  D.on = true; D.geometry_ok = false; D.borders_ok = false;
  h->forces_valid = false; h->list_valid = false;
  if (h->n > 0) return fail(h, "dd_init must precede sh_set_atoms");
  return 0;
} catch (...) { return -99; }   // no C++ exception crosses the C ABI (out of memory / internal error)

int sh_dd_get_info(const sh_ctx *hc, int pgrid[3], int brick[3], int64_t *nlocal, int64_t *nghost, int64_t *migrated,
                   int64_t *border_builds) {
  sh_ctx *h = const_cast<sh_ctx *>(hc);
  if (!h) return -1;
  if (pgrid) for (int d = 0; d < 3; d++) pgrid[d] = h->dd.pgrid[d];
  if (brick) for (int d = 0; d < 3; d++) brick[d] = h->dd.g[d];
  if (nlocal) *nlocal = h->n - h->nghost;
  if (nghost) *nghost = h->nghost;
  if (migrated) *migrated = h->dd.migrated_out;
  if (border_builds) *border_builds = h->dd.border_builds;
  return 0;
}

int sh_get_step_trace(const sh_ctx *h, int64_t cap, int64_t *nsteps, double *ms, int *flags) {
  if (!h) return -1;
  const int64_t n = (int64_t)h->step_ms.size();
  if (nsteps) *nsteps = n;
  for (int64_t k = 0; k < std::min(n, cap); k++) { if (ms) ms[k] = h->step_ms[k]; if (flags) flags[k] = h->step_flags_last[k]; }
  return 0;
}

int sh_get_tags(const sh_ctx *hc, int64_t n, int64_t *tags) try {
  sh_ctx *h = const_cast<sh_ctx *>(hc);
  if (n < 0 || n > h->n) return fail(h, "get_tags: n out of range");
  CU(cudaSetDevice(h->device));
  int rc = sync_tags_host(h);
  if (rc) return rc;
  for (int64_t i = 0; i < n; i++) tags[i] = h->tag[i];
  return 0;
} catch (...) { return -99; }   // no C++ exception crosses the C ABI (out of memory / internal error)

// Lees-Edwards shear (fix deform xy ... remap v): flow along x, gradient along y, rate = d(v_x)/dy.  Images across the
// periodic y boundary are ghosts displaced by rate * Ly * t along x; uses the decomposition machinery even on one GPU.
int sh_set_shear(sh_ctx *h, double rate) {
  if (!h) return -1;
  if (h->n > 0) return fail(h, "set_shear must precede sh_set_atoms");
  if (!h->dd.on) { int rc = sh_dd_init(h, 0, 1, nullptr, nullptr); if (rc) return rc; }
  h->dd.le_rate = rate; h->dd.le_off_build = 0.0; h->dd.le_time_build = h->time;
  h->dd.geometry_ok = false; h->dd.borders_ok = false;
  return 0;
}

}  // extern "C"
