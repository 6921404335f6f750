// curved_wall_kernels.cuh — static, elastic container walls of curved shape (fix wall/spherharm zcylinder | sphere):
// particles inside an infinite cylinder of any axis, or inside a sphere.  One warp per atom, lanes striding over the
// surface nodes, the same contact law, force and torque as the plane walls (wall_kernel, step_kernels.cuh).
//
// Submerged volume by the divergence theorem with a field phi of divergence 1 that vanishes on the wall surface, so the
// cut face carries no flux and  V = sum over the nodes past the wall of phi(P_k) . N_k:
//   cylinder, rho = P - a less its component along the unit axis u:   phi = (|rho|^2 - R^2) / (2 |rho|^2) rho
//   sphere,   r = P - centre:                                            phi = (|r|^3 - R^3) / (3 |r|^3) r
// phi is evaluated only at nodes past the wall (|rho|, |r| > R > 0), never at its singularity on the axis / centre.
// For a fixed wall dV/dx = sum N over the same nodes: F = -p sum N, tau = -p sum (P - x) x N, p = m k V^(m-1), E = k V^m.
#pragma once
#include "step_kernels.cuh"

namespace shgpu {

#define SH_MAX_CURVED_WALLS 8
enum { CWALL_CYLINDER = 0, CWALL_SPHERE = 1 };

struct CurvedWallSet {
  int n;
  int type[SH_MAX_CURVED_WALLS];
  double c[SH_MAX_CURVED_WALLS][3];   // a point of the axis (cylinder) / the centre (sphere)
  double u[SH_MAX_CURVED_WALLS][3];   // unit axis (cylinder)
  double R[SH_MAX_CURVED_WALLS], k[SH_MAX_CURVED_WALLS], m[SH_MAX_CURVED_WALLS];
};

// add = 1: the plane walls have written wallf / e_wall of every owned atom and the curved walls add to them (planes in
// insertion order, then curved walls in insertion order); add = 0: there are no plane walls and this kernel writes them.
__global__ void curved_wall_kernel(AtomView A, const DevShape *shapes, CurvedWallSet W, double *e_wall, int add) {
  const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (gw >= A.n) return;
  const int i = gw, st = A.stride;
  const DevShape &s = shapes[A.shape[i]];
  double f[3] = {0, 0, 0}, tq[3] = {0, 0, 0}, esum = 0;
  if (add) {
#pragma unroll
    for (int r = 0; r < 3; r++) { f[r] = A.wallf[r * st + i]; tq[r] = A.wallf[(3 + r) * st + i]; }
    esum = e_wall[i];
  }
  for (int w = 0; w < W.n; w++) {
    const bool cyl = W.type[w] == CWALL_CYLINDER;
    const double dc[3] = {A.c[i] - W.c[w][0], A.c[st + i] - W.c[w][1], A.c[2 * st + i] - W.c[w][2]};
    const double u[3] = {W.u[w][0], W.u[w][1], W.u[w][2]};
    double e[3] = {dc[0], dc[1], dc[2]};
    if (cyl) {
      const double t = fma(dc[2], u[2], fma(dc[1], u[1], dc[0] * u[0]));
#pragma unroll
      for (int r = 0; r < 3; r++) e[r] = fma(-t, u[r], dc[r]);
    }
    const double Rw = W.R[w];
    if (sqrt(fma(e[2], e[2], fma(e[1], e[1], e[0] * e[0]))) + s.rmax < Rw) continue;   // every node inside the wall
    double Rm[9], d[3], ub[3];
#pragma unroll
    for (int q = 0; q < 9; q++) Rm[q] = A.Rs[q * st + i];
#pragma unroll
    for (int r = 0; r < 3; r++) {   // body frame: d = Rs^T (c - a), ub = Rs^T u
      double t = Rm[r] * dc[0];
      t = fma(Rm[3 + r], dc[1], t);
      d[r] = fma(Rm[6 + r], dc[2], t);
      double v = Rm[r] * u[0];
      v = fma(Rm[3 + r], u[1], v);
      ub[r] = fma(Rm[6 + r], u[2], v);
    }
    const double R2 = Rw * Rw, R3 = R2 * Rw;
    double S0 = 0, S1 = 0, S2 = 0, Av = 0, T0 = 0, T1 = 0, T2 = 0;
    int cnt = 0;
    for (int k = lane; k < s.nq; k += 32) {
      const double2 a = s.pn[4 * k], b = s.pn[4 * k + 1], cc = s.pn[4 * k + 2];
      const double p0 = a.x, p1 = a.y, p2 = b.x, n0 = b.y, n1 = cc.x, n2 = cc.y;
      double r0 = d[0] + p0, r1 = d[1] + p1, r2 = d[2] + p2;
      if (cyl) {
        const double t = fma(r2, ub[2], fma(r1, ub[1], r0 * ub[0]));
        r0 = fma(-t, ub[0], r0); r1 = fma(-t, ub[1], r1); r2 = fma(-t, ub[2], r2);
      }
      const double q2 = fma(r2, r2, fma(r1, r1, r0 * r0));
      if (q2 > R2) {
        const double rn = fma(r2, n2, fma(r1, n1, r0 * n0));
        double g;
        if (cyl) g = (q2 - R2) / (2.0 * q2);
        else { const double q3 = q2 * sqrt(q2); g = (q3 - R3) / (3.0 * q3); }
        Av += g * rn;
        S0 += n0; S1 += n1; S2 += n2;
        T0 += fma(p1, n2, -(p2 * n1));
        T1 += fma(p2, n0, -(p0 * n2));
        T2 += fma(p0, n1, -(p1 * n0));
        cnt++;
      }
    }
    S0 = warp_sum(S0); S1 = warp_sum(S1); S2 = warp_sum(S2); Av = warp_sum(Av);
    T0 = warp_sum(T0); T1 = warp_sum(T1); T2 = warp_sum(T2);
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    const double V = Av;
    if (cnt == 0 || !(V > 0)) continue;
    double E, pr;
    if (W.m[w] == 1.0) { E = W.k[w] * V; pr = W.k[w]; }
    else { const double pw = pow(V, W.m[w] - 1.0); E = W.k[w] * pw * V; pr = W.m[w] * W.k[w] * pw; }
    esum += E;
    double Ss[3], Ts[3], l[3];
#pragma unroll
    for (int r = 0; r < 3; r++) {
      Ss[r] = Rm[3 * r] * S0 + Rm[3 * r + 1] * S1 + Rm[3 * r + 2] * S2;
      Ts[r] = Rm[3 * r] * T0 + Rm[3 * r + 1] * T1 + Rm[3 * r + 2] * T2;
      l[r] = A.c[r * st + i] - A.x[r * st + i];
    }
    const double Tt[3] = {Ts[0] + (l[1] * Ss[2] - l[2] * Ss[1]), Ts[1] + (l[2] * Ss[0] - l[0] * Ss[2]),
                          Ts[2] + (l[0] * Ss[1] - l[1] * Ss[0])};
#pragma unroll
    for (int r = 0; r < 3; r++) { f[r] += -pr * Ss[r]; tq[r] += -pr * Tt[r]; }
  }
  if (lane == 0) {
#pragma unroll
    for (int r = 0; r < 3; r++) { A.wallf[r * st + i] = f[r]; A.wallf[(3 + r) * st + i] = tq[r]; }
    e_wall[i] = esum;
  }
}

}  // namespace shgpu
