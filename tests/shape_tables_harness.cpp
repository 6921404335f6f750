// Test harness (tests/ only): C wrappers around the product's host-side shape-table builder so that the conservative
// direction-cell tables can be checked on the CPU against the oracle's exact radius evaluation.
#include <cstring>
#include <string>
#include "../lammps-spherharm_b200/csrc/shape_tables.h"

extern "C" {
void *sth_build(int lmax, const double *a, const double *b, double density, int nt, int np, int cube_n, char *err, int errlen) {
  auto *t = new shgpu::ShapeTables();
  std::string e = shgpu::build_shape_tables(lmax, a, b, density, nt, np, *t, cube_n);
  if (!e.empty()) { std::strncpy(err, e.c_str(), errlen - 1); delete t; return nullptr; }
  return t;
}
void sth_free(void *p) { delete static_cast<shgpu::ShapeTables *>(p); }
int sth_cube_n(void *p) { return static_cast<shgpu::ShapeTables *>(p)->cube_n; }
void sth_scalars(void *p, double *out) {   // rmax, rmin, volume, h1, h2, sample_step, sample_pad, r_sup, r_inf, cache_delta[4]
  auto *t = static_cast<shgpu::ShapeTables *>(p);
  out[0] = t->rmax; out[1] = t->rmin; out[2] = t->volume; out[3] = t->h1_bound; out[4] = t->h2_bound;
  out[5] = t->sample_step; out[6] = t->sample_pad; out[7] = t->r_sup; out[8] = t->r_inf;
  for (int lv = 0; lv < 4; lv++) out[9 + lv] = t->cache_delta[lv];
}
void sth_cube(void *p, float *ub2, float *lb2, float *wide2 /* 4 levels, concatenated */) {
  auto *t = static_cast<shgpu::ShapeTables *>(p);
  const size_t nc = t->cube_ub2.size();
  std::memcpy(ub2, t->cube_ub2.data(), nc * sizeof(float));
  std::memcpy(lb2, t->cube_lb2.data(), nc * sizeof(float));
  for (int lv = 0; lv < 4; lv++) std::memcpy(wide2 + lv * nc, t->cube_wide2[lv].data(), nc * sizeof(float));
}
void sth_frame(void *p, double *out) {   // volume, com[3], inertia[3], quat_principal[4]
  auto *t = static_cast<shgpu::ShapeTables *>(p);
  out[0] = t->volume;
  for (int d = 0; d < 3; d++) { out[1 + d] = t->com[d]; out[4 + d] = t->inertia[d]; }
  for (int d = 0; d < 4; d++) out[7 + d] = t->quat_principal[d];
}
void sth_nodes(void *p, double *pts, double *nds) {
  auto *t = static_cast<shgpu::ShapeTables *>(p);
  for (int k = 0; k < t->nq; k++) for (int d = 0; d < 3; d++) { pts[3 * k + d] = t->node_p[d][k]; nds[3 * k + d] = t->node_n[d][k]; }
}
}
