// device_math.cuh — FP64 device arithmetic of the SPHERHARM contact path (sm_100a).
//
// Compiled with -fmad=false: the compiler never contracts a*b+c on its own; every fused
// multiply-add below is an explicit fma() (DFMA).  The sequence of operations on the node
// decision path (pose -> relative pose -> node transform -> rho^2 -> folded SH radius) is the
// contract of DESIGN.md §3, shared with (but not included from) the CPU oracle, so that the
// inside/outside decision of every surface node is bit-identical on both sides.
// Reference source (pair_style spherharm, SPHERHARM math namespace): NOT IN MOUNT.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace shgpu {

struct DevShape {
  int lmax, nterms, nq, nchunks;          // nchunks = ceil(nq/32)
  double rmax, rmin, rmax2, rmin2, mass, inv_mass;
  double inertia[3], com[3], Rp[9];       // Rp row-major: principal frame -> shape frame
  const double *Ap;                       // folded recurrence multipliers, m-major
  const double2 *ab;                      // folded (a,b) coefficients, m-major
  const double *px, *py, *pz;             // node points, shape frame
  const double *nx, *ny, *nz;             // oriented area elements n dS, shape frame
  const double2 *pn;                      // the same per node in one 64 B record: (px,py) (pz,nx) (ny,nz) (0,0)
  int n_theta, n_phi;                     // node k = row*n_phi + col; phi_col = (col+1/2) 2pi/n_phi
  int tab_off;                            // offset (in records) of this shape in the concatenated table
  int nterms4;                            // nterms rounded up to a multiple of 4; tables hold nterms4+4 records
  const float *row_x;                     // cos(theta_row), float copy for the conservative window
  const float2 *cube_ul;                  // per cube-map direction cell: {ub2, lb2} = proven bounds of r^2 over the cell
  int cube_n, pad2_;                      // cells per face edge
  const float4 *pf4;                      // FP32 copy of the node points (x,y,z,0) for the conservative pre-cull
  const float *cube_w2[4];                // candidate-cache tables per margin level (inflated wide bound^2 per cell)
  double cache_delta[4];                  // node displacement margin of the candidate cache per level
};

// rotation matrix (row-major R[3*r+c]) of unit quaternion (w,x,y,z); plain mul/add, fixed order
__device__ __forceinline__ void quat_to_mat(const double q[4], double R[9]) {
  const double w2 = q[0] * q[0], i2 = q[1] * q[1], j2 = q[2] * q[2], k2 = q[3] * q[3];
  const double twoij = (2.0 * q[1]) * q[2], twoik = (2.0 * q[1]) * q[3], twojk = (2.0 * q[2]) * q[3];
  const double twoiw = (2.0 * q[1]) * q[0], twojw = (2.0 * q[2]) * q[0], twokw = (2.0 * q[3]) * q[0];
  R[0] = ((w2 + i2) - j2) - k2;  R[1] = twoij - twokw;          R[2] = twojw + twoik;
  R[3] = twoij + twokw;          R[4] = ((w2 - i2) + j2) - k2;  R[5] = twojk - twoiw;
  R[6] = twoik - twojw;          R[7] = twojk + twoiw;          R[8] = ((w2 - i2) - j2) + k2;
}

// Folded, trig-free spherical-harmonic radius (SURVEY A.2 / App. B "folded form").
// s = point in the shape frame, rho2 = |s|^2 (already computed by the caller with the
// contract's fma chain).  Tables may live in shared or global memory.
// Per (l,m) term: 1 DMUL + 3 DFMA.
__device__ __forceinline__ double sh_radius_folded(int L, const double *__restrict__ Ap,
                                                   const double2 *__restrict__ ab, double s0, double s1,
                                                   double s2, double rho2, double &rho_out) {
  const double rho = sqrt(rho2);
  const double inv = 1.0 / rho;
  const double x = s2 * inv, zx = s0 * inv, zy = s1 * inv;
  double u = 1.0, v = 0.0, r = 0.0;
  int base = 0;
  for (int m = 0; m <= L; m++) {
    if (m > 0) {
      const double t1 = v * zy, un = fma(u, zx, -t1);
      const double t2 = v * zx, vn = fma(u, zy, t2);
      u = un; v = vn;
    }
    const double2 c0 = ab[base];
    double C = c0.x, S = c0.y;
    const int len = L - m;
    if (len >= 1) {
      double q1 = Ap[base + 1] * x, q2 = 1.0;
      const double2 c1 = ab[base + 1];
      C = fma(c1.x, q1, C); S = fma(c1.y, q1, S);
#pragma unroll 4
      for (int i = 2; i <= len; i++) {
        const double tx = Ap[base + i] * x;
        const double q = fma(tx, q1, -q2);
        const double2 ci = ab[base + i];
        C = fma(ci.x, q, C); S = fma(ci.y, q, S);
        q2 = q1; q1 = q;
      }
    }
    r = fma(u, C, r); r = fma(v, S, r);
    base += len + 1;
  }
  rho_out = rho;
  return r;
}

// Two points per thread against the SAME shape: the coefficient loads (1 LDS.64 + 1 LDS.128 per
// term) are shared by both points and the two recurrences are independent dependency chains.
// Measured on B200 (tools/dfma_probe.cu): 67-73 % FP64-pipe utilisation against 57-61 % for the
// one-point loop at 16-32 warps/SM.  Per point the operation sequence is exactly that of
// sh_radius_folded, so each result is bit-identical to the one-point evaluation.
__device__ __forceinline__ void sh_radius_folded_x2(int L, const double *__restrict__ Ap,
                                                    const double2 *__restrict__ ab, const double sA[3],
                                                    double rhoA2, const double sB[3], double rhoB2, double &rhoA,
                                                    double &rhoB, double &rA_out, double &rB_out) {
  const double rA = sqrt(rhoA2), iA = 1.0 / rA, rB = sqrt(rhoB2), iB = 1.0 / rB;
  const double xA = sA[2] * iA, zxA = sA[0] * iA, zyA = sA[1] * iA;
  const double xB = sB[2] * iB, zxB = sB[0] * iB, zyB = sB[1] * iB;
  double uA = 1.0, vA = 0.0, rrA = 0.0, uB = 1.0, vB = 0.0, rrB = 0.0;
  int base = 0;
  for (int m = 0; m <= L; m++) {
    if (m > 0) {
      const double a1 = vA * zyA, un = fma(uA, zxA, -a1), a2 = vA * zxA, vn = fma(uA, zyA, a2);
      uA = un; vA = vn;
      const double b1 = vB * zyB, wn = fma(uB, zxB, -b1), b2 = vB * zxB, yn = fma(uB, zyB, b2);
      uB = wn; vB = yn;
    }
    const double2 c0 = ab[base];
    double CA = c0.x, SA = c0.y, CB = c0.x, SB = c0.y;
    const int len = L - m;
    if (len >= 1) {
      const double ap1 = Ap[base + 1];
      double qA1 = ap1 * xA, qA2 = 1.0, qB1 = ap1 * xB, qB2 = 1.0;
      const double2 c1 = ab[base + 1];
      CA = fma(c1.x, qA1, CA); SA = fma(c1.y, qA1, SA);
      CB = fma(c1.x, qB1, CB); SB = fma(c1.y, qB1, SB);
#pragma unroll 4
      for (int i = 2; i <= len; i++) {
        const double ap = Ap[base + i];
        const double2 ci = ab[base + i];
        const double txA = ap * xA, txB = ap * xB;
        const double qA = fma(txA, qA1, -qA2), qB = fma(txB, qB1, -qB2);
        CA = fma(ci.x, qA, CA); CB = fma(ci.x, qB, CB);
        SA = fma(ci.y, qA, SA); SB = fma(ci.y, qB, SB);
        qA2 = qA1; qA1 = qA; qB2 = qB1; qB1 = qB;
      }
    }
    rrA = fma(uA, CA, rrA); rrA = fma(vA, SA, rrA);
    rrB = fma(uB, CB, rrB); rrB = fma(vB, SB, rrB);
    base += len + 1;
  }
  rhoA = rA; rhoB = rB; rA_out = rrA; rB_out = rrB;
}

// N points per thread against the same shape (N = 4: one LDS.64 + one LDS.128 per term for 16 FP64 instructions,
// four independent dependency chains per lane).  Per point the operation sequence is exactly that of
// sh_radius_folded: results are bit-identical to the one-point evaluation.
template <int N>
__device__ __forceinline__ void sh_radius_folded_n(int L, const double *__restrict__ Ap, const double2 *__restrict__ ab,
                                                   const double (&s)[N][3], const double (&rho2)[N], double (&rho)[N],
                                                   double (&r_out)[N]) {
  double x[N], zx[N], zy[N], u[N], v[N], rr[N];
#pragma unroll
  for (int p = 0; p < N; p++) {
    rho[p] = sqrt(rho2[p]);
    const double inv = 1.0 / rho[p];
    x[p] = s[p][2] * inv; zx[p] = s[p][0] * inv; zy[p] = s[p][1] * inv;
    u[p] = 1.0; v[p] = 0.0; rr[p] = 0.0;
  }
  int base = 0;
  for (int m = 0; m <= L; m++) {
    if (m > 0) {
#pragma unroll
      for (int p = 0; p < N; p++) {
        const double t1 = v[p] * zy[p], un = fma(u[p], zx[p], -t1), t2 = v[p] * zx[p], vn = fma(u[p], zy[p], t2);
        u[p] = un; v[p] = vn;
      }
    }
    const double2 c0 = ab[base];
    double C[N], S[N];
#pragma unroll
    for (int p = 0; p < N; p++) { C[p] = c0.x; S[p] = c0.y; }
    const int len = L - m;
    if (len >= 1) {
      const double ap1 = Ap[base + 1];
      const double2 c1 = ab[base + 1];
      double q1[N], q2[N];
#pragma unroll
      for (int p = 0; p < N; p++) {
        q1[p] = ap1 * x[p]; q2[p] = 1.0;
        C[p] = fma(c1.x, q1[p], C[p]); S[p] = fma(c1.y, q1[p], S[p]);
      }
#pragma unroll 2
      for (int i = 2; i <= len; i++) {
        const double ap = Ap[base + i];
        const double2 ci = ab[base + i];
        double q[N];
#pragma unroll
        for (int p = 0; p < N; p++) { const double tx = ap * x[p]; q[p] = fma(tx, q1[p], -q2[p]); }
#pragma unroll
        for (int p = 0; p < N; p++) C[p] = fma(ci.x, q[p], C[p]);
#pragma unroll
        for (int p = 0; p < N; p++) S[p] = fma(ci.y, q[p], S[p]);
#pragma unroll
        for (int p = 0; p < N; p++) { q2[p] = q1[p]; q1[p] = q[p]; }
      }
    }
#pragma unroll
    for (int p = 0; p < N; p++) { rr[p] = fma(u[p], C[p], rr[p]); rr[p] = fma(v[p], S[p], rr[p]); }
    base += len + 1;
  }
#pragma unroll
  for (int p = 0; p < N; p++) r_out[p] = rr[p];
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// angular velocity in the space frame from the angular momentum: w = R(q) diag(1/I) R(q)^T L (q: principal -> space)
__device__ __forceinline__ void omega_from_angmom(const double q[4], const double L[3], const double I[3],
                                                  double w[3]) {
  double R[9];
  quat_to_mat(q, R);
  double wb[3];
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const double lb = R[k] * L[0] + R[3 + k] * L[1] + R[6 + k] * L[2];
    wb[k] = (I[k] > 0) ? lb / I[k] : 0.0;
  }
#pragma unroll
  for (int r = 0; r < 3; r++) w[r] = R[3 * r] * wb[0] + R[3 * r + 1] * wb[1] + R[3 * r + 2] * wb[2];
}

}  // namespace shgpu
