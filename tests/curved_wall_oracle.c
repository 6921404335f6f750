/* curved_wall_oracle.c — TEST INFRASTRUCTURE ONLY: the CPU oracle (oracle/sh_oracle.c, compiled into this unit
 * unchanged) extended by the curved container walls of sh_add_cylinder_wall / sh_add_sphere_wall, so that the tests have
 * a checker for curved_wall_kernel (csrc/curved_wall_kernels.cuh) and for trajectories with curved walls.  Built by
 * tests/test_curved_walls_cpu.py with the oracle's flags (-ffp-contract=off: every fused operation is an explicit fma()).
 *
 * A cw_ctx owns an orc_ctx; every orc_* call works on cw_oracle(cw).  cw_compute_forces / cw_run replace
 * orc_compute_forces / orc_run: the oracle's pair and plane-wall forces, then the curved walls in insertion order with the
 * kernel's operation sequence, cull and body frame.  V = sum over the nodes past the wall of phi(P).N with
 *   cylinder phi = (|rho|^2 - R^2) / (2 |rho|^2) rho  (rho: the part of P - a normal to the unit axis u)
 *   sphere   phi = (|r|^3 - R^3) / (3 |r|^3) r        (r = P - centre). */
#include "../oracle/sh_oracle.c"

#define CW_MAX 8

typedef struct { int cyl; double c[3], u[3], R, k, m; } cwall_t;
typedef struct { orc_ctx *o; int n; cwall_t w[CW_MAX]; } cw_ctx;

cw_ctx *cw_create(void) {
  cw_ctx *cw = (cw_ctx *)calloc(1, sizeof *cw);
  cw->o = orc_create();
  return cw;
}
void cw_destroy(cw_ctx *cw) { if (cw) { orc_destroy(cw->o); free(cw); } }
orc_ctx *cw_oracle(cw_ctx *cw) { return cw->o; }

static int cw_add(cw_ctx *cw, int cyl, const double p[3], const double u[3], double R, double k, double m) {
  if (cw->n >= CW_MAX) return fail(cw->o, "too many curved walls");
  if (!(R > 0)) return fail(cw->o, "curved wall: need radius > 0");
  if (!(k >= 0) || !(m >= 1.0)) return fail(cw->o, "curved wall: need k >= 0, exponent >= 1");
  cwall_t *w = &cw->w[cw->n++];
  w->cyl = cyl;
  for (int d = 0; d < 3; d++) { w->c[d] = p[d]; w->u[d] = u[d]; }
  w->R = R; w->k = k; w->m = m; cw->o->forces_valid = 0;
  return 0;
}
int cw_add_cylinder_wall(cw_ctx *cw, const double point[3], const double axis[3], double R, double k, double m) {
  double nn = sqrt(axis[0] * axis[0] + axis[1] * axis[1] + axis[2] * axis[2]);
  if (!(nn > 0)) return fail(cw->o, "cylinder wall axis is zero");
  double u[3] = {axis[0] / nn, axis[1] / nn, axis[2] / nn};
  return cw_add(cw, 1, point, u, R, k, m);
}
int cw_add_sphere_wall(cw_ctx *cw, const double center[3], double R, double k, double m) {
  double u[3] = {0, 0, 0};
  return cw_add(cw, 0, center, u, R, k, m);
}

int cw_compute_forces(cw_ctx *cw) {
  orc_ctx *c = cw->o;
  if (orc_compute_forces(c)) return -1;
  double ec = c->e_contact;
  for (int w = 0; w < cw->n; w++) {
    const cwall_t *wl = &cw->w[w];
    const double R2 = wl->R * wl->R, R3 = R2 * wl->R;
    for (int64_t i = 0; i < c->n; i++) {
      const shape_t *s = &c->shp[c->shape[i]];
      const double *R = &c->Rs[9 * i];
      double dc[3] = {c->c[3 * i] - wl->c[0], c->c[3 * i + 1] - wl->c[1], c->c[3 * i + 2] - wl->c[2]};
      double e[3] = {dc[0], dc[1], dc[2]};
      if (wl->cyl) {
        double t = fma(dc[2], wl->u[2], fma(dc[1], wl->u[1], dc[0] * wl->u[0]));
        for (int r = 0; r < 3; r++) e[r] = fma(-t, wl->u[r], dc[r]);
      }
      if (sqrt(fma(e[2], e[2], fma(e[1], e[1], e[0] * e[0]))) + s->rmax < wl->R) continue;
      double d[3], ub[3];
      for (int r = 0; r < 3; r++) {
        double t = R[r] * dc[0]; t = fma(R[3 + r], dc[1], t); d[r] = fma(R[6 + r], dc[2], t);
        double v = R[r] * wl->u[0]; v = fma(R[3 + r], wl->u[1], v); ub[r] = fma(R[6 + r], wl->u[2], v);
      }
      double S[3] = {0, 0, 0}, A = 0, T[3] = {0, 0, 0}; int nin = 0;
      for (int k = 0; k < s->nq; k++) {
        const double *p = &s->p[3 * k], *n = &s->nds[3 * k];
        double r0 = d[0] + p[0], r1 = d[1] + p[1], r2 = d[2] + p[2];
        if (wl->cyl) {
          double t = fma(r2, ub[2], fma(r1, ub[1], r0 * ub[0]));
          r0 = fma(-t, ub[0], r0); r1 = fma(-t, ub[1], r1); r2 = fma(-t, ub[2], r2);
        }
        double q2 = fma(r2, r2, fma(r1, r1, r0 * r0));
        if (!(q2 > R2)) continue;
        nin++;
        double rn = fma(r2, n[2], fma(r1, n[1], r0 * n[0])), g;
        if (wl->cyl) g = (q2 - R2) / (2.0 * q2);
        else { double q3 = q2 * sqrt(q2); g = (q3 - R3) / (3.0 * q3); }
        A += g * rn;
        S[0] += n[0]; S[1] += n[1]; S[2] += n[2];
        T[0] += fma(p[1], n[2], -(p[2] * n[1]));
        T[1] += fma(p[2], n[0], -(p[0] * n[2]));
        T[2] += fma(p[0], n[1], -(p[1] * n[0]));
      }
      if (nin == 0 || !(A > 0)) continue;
      double E, p = contact_pressure(wl->k, wl->m, A, &E);
      ec += E;
      double Ss[3], Ts[3], l[3];
      for (int r = 0; r < 3; r++) {
        Ss[r] = R[3 * r] * S[0] + R[3 * r + 1] * S[1] + R[3 * r + 2] * S[2];
        Ts[r] = R[3 * r] * T[0] + R[3 * r + 1] * T[1] + R[3 * r + 2] * T[2];
        l[r] = c->c[3 * i + r] - c->x[3 * i + r];
      }
      double Tt[3] = {Ts[0] + (l[1] * Ss[2] - l[2] * Ss[1]), Ts[1] + (l[2] * Ss[0] - l[0] * Ss[2]), Ts[2] + (l[0] * Ss[1] - l[1] * Ss[0])};
      for (int r = 0; r < 3; r++) { c->f[3 * i + r] += -p * Ss[r]; c->tq[3 * i + r] += -p * Tt[r]; }
    }
  }
  c->e_contact = ec;
  return 0;
}

/* orc_run with cw_compute_forces in place of orc_compute_forces */
int cw_run(cw_ctx *cw, int64_t nsteps) {
  orc_ctx *c = cw->o;
  if (!c->forces_valid) if (cw_compute_forces(cw)) return -1;
  double dt = c->dt, dth = 0.5 * dt;
  const double damp_v = 1.0 - 0.5 * dt * c->gamma_lin, damp_L = 1.0 - 0.5 * dt * c->gamma_rot;
  for (int64_t step = 0; step < nsteps; step++) {
#pragma omp parallel for num_threads(c->nthreads)
    for (int64_t i = 0; i < c->n; i++) {
      const shape_t *s = &c->shp[c->shape[i]];
      double im = 1.0 / s->mass;
      for (int d = 0; d < 3; d++) {
        c->v[3 * i + d] = (c->v[3 * i + d] + dth * (c->f[3 * i + d] * im + c->g[d])) * damp_v;
        c->x[3 * i + d] += dt * c->v[3 * i + d];
        c->L[3 * i + d] = (c->L[3 * i + d] + dth * c->tq[3 * i + d]) * damp_L;
      }
      richardson(&c->q[4 * i], &c->L[3 * i], s->inertia, dth);
    }
    c->time += dt;
    if (cw_compute_forces(cw)) return -1;
#pragma omp parallel for num_threads(c->nthreads)
    for (int64_t i = 0; i < c->n; i++) {
      const shape_t *s = &c->shp[c->shape[i]];
      double im = 1.0 / s->mass;
      for (int d = 0; d < 3; d++) {
        c->v[3 * i + d] = (c->v[3 * i + d] + dth * (c->f[3 * i + d] * im + c->g[d])) * damp_v;
        c->L[3 * i + d] = (c->L[3 * i + d] + dth * c->tq[3 * i + d]) * damp_L;
      }
    }
  }
  return 0;
}
