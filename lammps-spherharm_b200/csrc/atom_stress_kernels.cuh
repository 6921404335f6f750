// atom_stress_kernels.cuh — per-atom virial, kinetic tensor, contact energy and contact count (sh_get_atom_stress;
// LAMMPS compute stress/atom, pe/atom, contact/atom).  Read-only on the state of the last pair phase: every value is
// derived from the per-pair records pres[14][P], walked through the fixed-order CSR rows, so two calls on the same state
// are bitwise equal (no floating-point atomics).
#pragma once
#include "step_kernels.cuh"

namespace shgpu {

// the pair behind every CSR entry: epair[pair_eij[p]] = epair[pair_eji[p]] = p (4 B per entry instead of a per-entry
// copy of the pair record)
__global__ void atom_stress_entry_pair_kernel(int npairs, const int *pair_eij, const int *pair_eji, int *epair) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= npairs) return;
  epair[pair_eij[p]] = p;
  const int e = pair_eji[p];
  if (e >= 0) epair[e] = p;
}

struct AtomStressArgs {
  AtomView A;                 // A.n = owned atoms
  const DevShape *shapes;
  int nall;                   // rows handled: the owned atoms, plus the ghosts when their halves go back to the owners
  int nrows;                  // rows that have CSR entries (0 = no valid forces: the pair parts are zero)
  int mode;                   // 0: (x_i - x_j) / 2 (x) F_ij; 1: contact branch vector (x_i - x_c) (x) F_ij
  const int *nbr_off, *epair, *pair_i, *pair_j, *pair_img;
  const double *pres;
  int pres_stride;
  double L[3];
  const double *ewall;        // per owned atom wall energy, or nullptr (no walls)
  double *vir, *kin, *en;     // owned atom i: vir[9 i + 3a + b], kin[9 i + 3a + b], en[i]
  int *cnt;                   // owned atom i: contacts
  double *ghost_rec;          // ghost g = i - A.n: 11 doubles (virial 9, energy, contacts) owed to its owner
};

// One thread per row, summing the row's entries in CSR order.  Mode 0 evaluates the separation exactly as
// stress_virial_kernel does, identically for both atoms of a pair, so each gets the same half.  Mode 1 takes the branch
// vector from the row atom's own image to the overlap centroid, which pres stores in the frame of pair_i.
__global__ void atom_stress_row_kernel(const __grid_constant__ AtomStressArgs S) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= S.nall) return;
  const AtomView &A = S.A;
  const int st = A.stride;
  const size_t ps = (size_t)S.pres_stride;
  double W[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, e = 0.0;
  int ncon = 0;
  if (r < S.nrows) {
    for (int k = S.nbr_off[r]; k < S.nbr_off[r + 1]; k++) {
      const int p = S.epair[k];
      if (p < 0) continue;
      const double V = S.pres[p];
      if (!(V > 0)) continue;   // no contact: no force, and the centroid is undefined
      const int i = S.pair_i[p], j = S.pair_j[p], img = S.pair_img[p];
      double F[3], b[3];
#pragma unroll
      for (int a = 0; a < 3; a++) F[a] = S.pres[(2 + a) * ps + p];
      if (S.mode == 0) {
#pragma unroll
        for (int a = 0; a < 3; a++) {
          double d = A.c[a * st + i] - A.c[a * st + j];
          const int n = ((img >> (2 * a)) & 3) - 1;
          if (n != 0) d = d - S.L[a] * (double)n;
          b[a] = 0.5 * (d - (A.c[a * st + i] - A.x[a * st + i]) + (A.c[a * st + j] - A.x[a * st + j]));
        }
      } else if (i == r) {
#pragma unroll
        for (int a = 0; a < 3; a++) b[a] = A.x[a * st + i] - S.pres[(11 + a) * ps + p];
      } else {
#pragma unroll
        for (int a = 0; a < 3; a++) {
          double xj = A.x[a * st + j];
          const int n = ((img >> (2 * a)) & 3) - 1;
          if (n != 0) xj = xj + S.L[a] * (double)n;   // the image of j that touches i
          b[a] = xj - S.pres[(11 + a) * ps + p];
          F[a] = -F[a];
        }
      }
#pragma unroll
      for (int a = 0; a < 3; a++)
#pragma unroll
        for (int c = 0; c < 3; c++) W[3 * a + c] += b[a] * F[c];
      e += 0.5 * S.pres[ps + p];
      ncon++;
    }
  }
  if (r < A.n) {
    if (S.ewall) e += S.ewall[r];
    const double m = S.shapes[A.shape[r]].mass, vv[3] = {A.v[r], A.v[st + r], A.v[2 * st + r]};
#pragma unroll
    for (int a = 0; a < 3; a++)
#pragma unroll
      for (int c = 0; c < 3; c++) {
        S.vir[9 * (size_t)r + 3 * a + c] = W[3 * a + c];
        S.kin[9 * (size_t)r + 3 * a + c] = m * vv[a] * vv[c];
      }
    S.en[r] = e;
    S.cnt[r] = ncon;
  } else {
    double *o = S.ghost_rec + 11 * (size_t)(r - A.n);
#pragma unroll
    for (int k = 0; k < 9; k++) o[k] = W[k];
    o[9] = e;
    o[10] = (double)ncon;
  }
}

// newton on: the halves that ghost rows collected on the neighbouring ranks, added to their owners in the fixed order of
// the reverse-communication plan (rev_off / rev_k, as dd_add_returned_forces_kernel)
__global__ void atom_stress_add_returned_kernel(int nown, const int *rev_off, const int *rev_k, const double *in, double *vir,
                                                double *en, int *cnt) {
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= nown) return;
  const int e0 = rev_off[a], e1 = rev_off[a + 1];
  if (e0 == e1) return;
  double acc[11];
#pragma unroll
  for (int k = 0; k < 9; k++) acc[k] = vir[9 * (size_t)a + k];
  acc[9] = en[a];
  int c = cnt[a];
  for (int e = e0; e < e1; e++) {
    const double *rec = in + 11 * (size_t)rev_k[e];
#pragma unroll
    for (int k = 0; k < 10; k++) acc[k] += rec[k];
    c += (int)rec[10];
  }
#pragma unroll
  for (int k = 0; k < 9; k++) vir[9 * (size_t)a + k] = acc[k];
  en[a] = acc[9];
  cnt[a] = c;
}

}  // namespace shgpu
