// pair_split_kernels.cuh — split form of the SPHERHARM pair phase (default for large systems), sm_100a.
//
// Same arithmetic contract and the same inside/outside decision for every surface node as pair_warp_kernel.cuh and
// the oracle; the work is cut so that each kernel runs at the occupancy its bottleneck wants:
//   cache  pair_cache_build_kernel  (on neighbor rebuilds / when a particle used up the cache margin)  a Verlet list of
//          surface nodes: per (pair, direction) the node indices that can pass the exact tests before the next rebuild.
//   A      pair_cull_cached_kernel  (latency bound -> written for memory-level parallelism)  one warp per pair, both
//          directions in ONE flattened candidate list: 128 candidates per iteration are in flight at once (index load,
//          one 16 B FP32 node gather, FP32 transform, direction-cell lookup), survivors of this conservative FP32
//          stage (relative margins) are staged as 2-byte indices, and only they go through the exact FP64 stage
//          (transform, bounding sphere, inscribed sphere, proven per-cell lower / upper bound of r).  The records
//          (s-vector in b's frame + node index, 32 B) are written straight from registers into one contiguous run per
//          (pair, direction) of the pool of the TARGET shape (one atomicAdd per run).
//          pair_cull_window_kernel  (persistent, slow path)  pairs without a cache entry, or every pair on a step whose
//          cache is invalid: conservative window on a's node grid + FP32 pre-cull + the same exact stage.
//   B      pair_eval_kernel  (FP64 FMA-pipe bound)  every pool holds records against ONE shape, so warps are full and
//          shape-uniform whatever pair a record came from; persistent CTAs over contiguous chunks of the pools (the
//          shape's folded table is staged in shared memory only when the shape changes), 2 or 4 points per lane sharing
//          every coefficient load.  The work plan is computed ON THE DEVICE from the pool counters (no host round trip).
//   C      pair_reduce_kernel  (store bound)  a CTA takes 256 pairs, compacts those with nodes to sum in shared memory,
//          and one thread per such pair walks its node indices in a fixed order (bitwise reproducible), accumulates the
//          inside nodes, applies the contact law, writes the outputs; outputs that already hold zeros are not rewritten.
// Pairs that do not fit (more than SURV_CAP staged survivors, or a full pool) go to a device list that the fused
// warp kernel (pair_warp_kernel.cuh) processes afterwards: a full pool costs time, never correctness.
// No floating-point atomics anywhere; pool offsets vary from run to run but never enter the arithmetic.
#pragma once
#include "pair_kernel.cuh"

namespace shgpu {

#define SPLIT_CAP 88      // window kernel: staged records per direction
#define SURV_CAP 320      // cached kernel: staged FP32-stage survivors per pair (both directions)
#define CACHE_CAP 384     // cache build: candidates per direction

struct __align__(16) SurvRec {
  double s0, s1, s2;
  int k;       // node index in a's table
  int flag;    // 0 = to be evaluated, 2 = inside (decided by the cull: inscribed sphere / per-cell lower bound), 3 = dead
};

// one run of records per (pair, direction).  Nodes that the cull already proved inside (inscribed sphere / per-cell lower
// bound) need no evaluation: up to 7 of them are kept inline here instead of occupying lanes of pair_eval_kernel.
// Further proven-inside nodes go to a separate index pool (`inpool`, 4 B per node) that pair_eval_kernel never sees: a deep
// overlap on a fine quadrature (80x160 nodes) has dozens of them per pair.
struct __align__(16) PdEntry {
  long long off;            // first record of the run (absolute index into the pool)
  int cnt;                  // records in the run; -1 = the pair is on the deep-contact list
  unsigned short ntrans;    // candidate nodes the cull transformed for this direction (counter [1])
  unsigned short cnt2;      // proven-inside nodes of this direction in the index pool
  unsigned int off2;        // ... starting here
  unsigned short nin;       // inline inside nodes
  unsigned short in[5];
};
#define PD_INLINE 5

// everything the cached cull needs to start a pair, in one 32 B sector (written by the cache build)
struct __align__(16) PairHot {
  int i, j, n0, n1;         // atoms; cached candidates per direction (n0 < 0: no cache entry)
  long long off;            // first candidate in the cache pool (direction 0, then direction 1)
  int img;                  // periodic image (PairArgs::pair_img)
  unsigned char shp_i, shp_j, pad0, pad1;
};

struct EvalPlanDev {
  int total_blocks, nshape;
  int blk_start[SH_MAX_SHAPES + 1];
  long long count[SH_MAX_SHAPES];
};

// per-step device scalars of the split pipeline (zeroed by one memset at the start of the pair phase)
struct SplitScalars {
  unsigned long long pool_count[SH_MAX_SHAPES];   // records appended this step (may exceed cap -> host grows the pool)
  unsigned long long in_count;                    // entries appended to the inside-node index pool (same rule)
  int nbig;            // pairs on the deep-contact list
  int nslow;           // pairs without a cache entry
  int slow_counter;    // work counter of the window kernel
  int deep_counter;    // work counter of the fused kernel on the deep-contact list
};

struct SplitArgs {
  SurvRec *pool;                  // all shapes' pools in one buffer
  int *pool_kin;                  // per record: its node index if the node is inside, else -1 (own array: the reduction
                                  // reads one contiguous int run per direction instead of the 32 B records)
  const long long *pool_base;     // [nshape] first record of the shape's pool
  const long long *pool_cap;      // [nshape]
  SplitScalars *sc;
  PdEntry *pd;                    // [2P] record run + inline inside nodes per (pair, direction)
  unsigned char *out_zero;        // [P] 1: the pair's outputs (pres, both CSR slots) hold the zero record written by the
                                  // reduction (cleared by the host whenever the list is rebuilt or another kernel wrote them)
  int *big_list;                  // [P]
  int *slow_list;                 // [P]
  int *inpool;                    // node indices proven inside by the cull beyond the inline capacity
  long long in_cap;
};

struct CacheArgs {
  unsigned short *pool;            // candidate node indices; one run per PAIR: direction 0 then direction 1
  PairHot *hot;                    // [P]  n0 = -1: not cached (too many candidates), the pair takes the window path
  unsigned long long *count;       // appended entries (may exceed cap -> host grows and rebuilds)
  long long cap;
  int *overflow;
  const int *invalid;              // device flag raised by cache_check_kernel: the cached kernel stands down when set
  int enabled;
  int level;                       // margin level (DevShape::cache_delta / cube_w2 index)
};

// ---- conservative FP32 margin on rho^2.  The FP32 transform of a node has an absolute error below
// 4 * 2^-24 * (|t| + rmax_a) per component, so |rho2_f32 - rho2| < 16 * 2^-23 * (|t| + rmax_a)^2 with a wide safety
// factor; relative to the pair's own length scale, so it holds for any unit system (ADVICE r1).
__device__ __forceinline__ float fp32_margin(float t0, float t1, float t2, float ra) {
  const float sc = sqrtf(fmaf(t2, t2, fmaf(t1, t1, t0 * t0))) + ra;
  return 1.9073486e-6f * sc * sc;
}

// ---- conservative window on a's node grid (FP32 with margins), shared by the window and cache-build kernels.
// Rb = radius of the sphere around b's origin that a node must enter (rmax_b, or rmax_b + delta for the cache).
struct NodeWindow { bool skip; float cosA, xe, se, phie; };

__device__ __forceinline__ NodeWindow make_window(const DevShape &sa, double Rb, const double *x0) {
  NodeWindow w;
  const double e0 = 2.0 * x0[0], e1 = 2.0 * x0[1], e2 = 2.0 * x0[2];   // b's origin in a's frame
  const double D2 = e0 * e0 + e1 * e1 + e2 * e2, D = sqrt(D2);
  w.skip = D >= (sa.rmax + Rb) * (1.0 + 1e-9);
  w.cosA = -2.0f; w.xe = 1.0f; w.se = 0.0f; w.phie = 0.0f;
  if (!w.skip && D > 1e-9 * (sa.rmax + Rb)) {
    const double q = D2 - Rb * Rb;
    double rc = sa.rmin;
    if (q > 0) rc = fmin(fmax(sqrt(q), sa.rmin), sa.rmax);
    const double g = (rc * rc + q) / (2.0 * rc * D);
    w.cosA = (float)g - 3e-5f;
    if (w.cosA >= 1.0f) w.skip = true;
    w.xe = fminf(1.0f, fmaxf(-1.0f, (float)(e2 / D)));
    w.se = sqrtf(fmaxf(0.0f, 1.0f - w.xe * w.xe));
    w.phie = atan2f((float)e1, (float)e0);
    if (w.phie < 0.0f) w.phie += 6.2831853f;
  }
  return w;
}

__device__ __forceinline__ void classify_row(const DevShape &sa, const NodeWindow &w, int row, int &c0, int &ccount) {
  c0 = 0; ccount = 0;
  const int nph = sa.n_phi;
  if (row >= sa.n_theta) return;
  if (w.cosA <= -1.0f) { ccount = nph; return; }
  const float xa = sa.row_x[row];
  const float sarow = sqrtf(fmaxf(0.0f, 1.0f - xa * xa));
  const float ss = sarow * w.se, xx = xa * w.xe;
  if (xx + ss < w.cosA) return;
  const float cd = (ss > 1e-12f) ? (w.cosA - xx) / ss : -2.0f;
  if (cd <= -1.0f) { ccount = nph; return; }
  const float inv_dphi = (float)nph * 0.15915494f;
  const float dl = acosf(fminf(cd, 1.0f)) + 2e-4f;
  const int b0 = (int)ceilf((w.phie - dl) * inv_dphi - 0.5f);
  const int b1 = (int)floorf((w.phie + dl) * inv_dphi - 0.5f);
  ccount = b1 - b0 + 1;
  if (ccount >= nph) { ccount = nph; c0 = 0; }
  else if (ccount > 0) { c0 = b0 % nph; if (c0 < 0) c0 += nph; }
  else ccount = 0;
}

// cube-map direction cell of a vector (FP32); the tables cover a border strip that absorbs the FP32 index error
__device__ __forceinline__ int cube_cell(float f0, float f1, float f2, int cn) {
  const float ax = fabsf(f0), ay = fabsf(f1), az = fabsf(f2);
  int face; float ma, uu, vv;
  if (ax >= ay && ax >= az) { face = f0 > 0 ? 0 : 1; ma = ax; uu = f1; vv = f2; }
  else if (ay >= az) { face = f1 > 0 ? 2 : 3; ma = ay; uu = f0; vv = f2; }
  else { face = f2 > 0 ? 4 : 5; ma = az; uu = f0; vv = f1; }
  // (approximate reciprocal, 2 ulp: the tables' border strip of 1e-5 in (u, v) absorbs the index error)
  const float im = __fdividef(1.0f, fmaxf(ma, 1e-30f)), hn = 0.5f * (float)cn;
  const int iu = min(cn - 1, max(0, (int)((uu * im + 1.0f) * hn)));
  const int iv = min(cn - 1, max(0, (int)((vv * im + 1.0f) * hn)));
  return (face * cn + iu) * cn + iv;
}

// one element (index l < 15) of the relative pose of direction a -> b: M[9], t[3], x0[3] (same fma chains as the oracle)
__device__ __forceinline__ double pose_element(const PairArgs &A, int a, int b, double dd0, double dd1, double dd2, int l) {
  const int st = A.stride;
  if (l < 9) {
    const int r = l / 3, k = l - 3 * r;
    double m = A.Rs[(0 + r) * st + b] * A.Rs[(0 + k) * st + a];
    m = fma(A.Rs[(3 + r) * st + b], A.Rs[(3 + k) * st + a], m);
    m = fma(A.Rs[(6 + r) * st + b], A.Rs[(6 + k) * st + a], m);
    return m;
  } else if (l < 12) {
    const int r = l - 9;
    double tt = A.Rs[(0 + r) * st + b] * dd0;
    tt = fma(A.Rs[(3 + r) * st + b], dd1, tt);
    tt = fma(A.Rs[(6 + r) * st + b], dd2, tt);
    return tt;
  }
  const int r = l - 12;
  double hx = A.Rs[(0 + r) * st + a] * dd0;
  hx = fma(A.Rs[(3 + r) * st + a], dd1, hx);
  hx = fma(A.Rs[(6 + r) * st + a], dd2, hx);
  return -0.5 * hx;
}
__device__ __forceinline__ void pose_to_smem(const PairArgs &A, int a, int b, double dd0, double dd1, double dd2, int lane,
                                             double *pose) {
  __syncwarp();
  if (lane < 15) pose[lane] = pose_element(A, a, b, dd0, dd1, dd2, lane);
  __syncwarp();
}

// exact FP64 decision stage for one node (DESIGN §3.3 + the proven per-cell bounds): returns the record flag
//   -1 outside (bounding sphere / per-cell upper bound), 2 inside (inscribed sphere / per-cell lower bound), 0 evaluate
__device__ __forceinline__ int exact_node_stage(const double *M, const double *t, double p0, double p1, double p2, double rmax2,
                                                double rmin2, const float2 *__restrict__ cube, int cn, int use_bounds,
                                                double &s0, double &s1, double &s2) {
  s0 = fma(M[0], p0, t[0]); s0 = fma(M[1], p1, s0); s0 = fma(M[2], p2, s0);
  s1 = fma(M[3], p0, t[1]); s1 = fma(M[4], p1, s1); s1 = fma(M[5], p2, s1);
  s2 = fma(M[6], p0, t[2]); s2 = fma(M[7], p1, s2); s2 = fma(M[8], p2, s2);
  const double rho2 = fma(s2, s2, fma(s1, s1, s0 * s0));
  if (!(rho2 < rmax2)) return -1;
  if (rho2 <= rmin2) return 2;
  if (!use_bounds) return 0;
  const float2 ul = __ldg(&cube[cube_cell((float)s0, (float)s1, (float)s2, cn)]);
  if (rho2 <= (double)ul.y) return 2;
  return rho2 < (double)ul.x ? 0 : -1;
}

// ---- candidate cache build: window + FP32 tests against the INFLATED bounds (rmax_b + delta; cube_w2[level]), no FP64
// node work.  Both directions are staged in shared memory and appended as ONE run per pair.
// list == nullptr: every pair; else the pairs list[0 .. *nlist) (pairs that join a live cache after a neighbor rebuild).
template <int WPB>
__global__ void __launch_bounds__(WPB * 32) pair_cache_build_kernel(PairArgs A, CacheArgs C, const int *list, const int *nlist) {
  __shared__ unsigned short s_buf[WPB][2][CACHE_CAP];
  __shared__ double s_pose[WPB][16];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nwork = list ? *nlist : A.npairs;
  for (int w = blockIdx.x * WPB + warp; w < nwork; w += gridDim.x * WPB) {
  const int p = list ? list[w] : w;
  const int i = A.pair_i[p], j = A.pair_j[p];
  double d[3];
  pair_separation(A, p, i, j, d);
  const int shp_i = A.shape[i], shp_j = A.shape[j];
  double *pose = s_pose[warp];
  int cnt0 = 0, cnt1 = 0;
  bool over = false;
  for (int dir = 0; dir < 2 && !over; dir++) {
    const int a = dir ? j : i, b = dir ? i : j;
    const DevShape &sa = A.shapes[dir ? shp_j : shp_i];
    const DevShape &sb = A.shapes[dir ? shp_i : shp_j];
    const double sgn = dir ? -1.0 : 1.0;
    pose_to_smem(A, a, b, sgn * d[0], sgn * d[1], sgn * d[2], lane, pose);
    const double *M = pose, *t = pose + 9, *x0 = pose + 12;
    const double delta = sb.cache_delta[C.level], Rb = sb.rmax + delta;
    const NodeWindow w = make_window(sa, Rb, x0);
    const float4 *__restrict__ pf = sa.pf4;
    const float *__restrict__ cube = sb.cube_w2[C.level];
    const int cn = sb.cube_n, nph = sa.n_phi, nth = sa.n_theta;
    const float fM0 = (float)M[0], fM1 = (float)M[1], fM2 = (float)M[2], fM3 = (float)M[3], fM4 = (float)M[4],
                fM5 = (float)M[5], fM6 = (float)M[6], fM7 = (float)M[7], fM8 = (float)M[8];
    const float ft0 = (float)t[0], ft1 = (float)t[1], ft2 = (float)t[2];
    const float eps = fp32_margin(ft0, ft1, ft2, (float)sa.rmax);
    const float fR2 = (float)(Rb * Rb) + eps;
    const float fin = (float)((sb.rmin + 2.0 * delta) * (sb.rmin + 2.0 * delta)) + eps;
    unsigned short *buf = s_buf[warp][dir];
    int n = 0;
    if (!w.skip) {
      for (int rb = 0; rb < nth && !over; rb += 32) {
        int c0, ccount;
        classify_row(sa, w, rb + lane, c0, ccount);
        unsigned rows = __ballot_sync(0xffffffffu, ccount > 0);
        while (rows && !over) {
          const int rl = __ffs(rows) - 1;
          rows &= rows - 1;
          const int rc0 = __shfl_sync(0xffffffffu, c0, rl), rcount = __shfl_sync(0xffffffffu, ccount, rl);
          const int rowbase = (rb + rl) * nph;
          for (int cb = 0; cb < rcount; cb += 32) {
            const int cc = cb + lane;
            bool pass = false;
            int k = 0;
            if (cc < rcount) {
              int col = rc0 + cc;
              if (col >= nph) col -= nph;
              k = rowbase + col;
              const float4 q = __ldg(&pf[k]);
              const float f0 = fmaf(fM2, q.z, fmaf(fM1, q.y, fmaf(fM0, q.x, ft0)));
              const float f1 = fmaf(fM5, q.z, fmaf(fM4, q.y, fmaf(fM3, q.x, ft1)));
              const float f2 = fmaf(fM8, q.z, fmaf(fM7, q.y, fmaf(fM6, q.x, ft2)));
              const float r2 = fmaf(f2, f2, fmaf(f1, f1, f0 * f0));
              if (r2 < fR2) pass = (r2 < fin) || (r2 < __ldg(&cube[cube_cell(f0, f1, f2, cn)]) + eps);
            }
            const unsigned pm = __ballot_sync(0xffffffffu, pass);
            if (pm) {
              const int nnew = __popc(pm);
              if (n + nnew > CACHE_CAP) { over = true; break; }
              if (pass) buf[n + __popc(pm & ((1u << lane) - 1u))] = (unsigned short)k;
              n += nnew;
            }
          }
        }
      }
    }
    if (dir) cnt1 = n; else cnt0 = n;
    __syncwarp();
  }
  const int ntot = cnt0 + cnt1;
  long long off = 0;
  if (lane == 0 && !over && ntot > 0) off = (long long)atomicAdd(C.count, (unsigned long long)ntot);
  off = __shfl_sync(0xffffffffu, off, 0);
  if (!over && ntot > 0) {
    if (off + ntot <= C.cap) {
      for (int r = lane; r < cnt0; r += 32) C.pool[off + r] = s_buf[warp][0][r];
      for (int r = lane; r < cnt1; r += 32) C.pool[off + cnt0 + r] = s_buf[warp][1][r];
    } else { if (lane == 0) *C.overflow = 1; over = true; }
  }
  if (lane == 0) {
    PairHot hrec;
    hrec.i = i; hrec.j = j; hrec.n0 = over ? -1 : cnt0; hrec.n1 = over ? -1 : cnt1; hrec.off = off; hrec.img = A.pair_img[p];
    hrec.shp_i = (unsigned char)shp_i; hrec.shp_j = (unsigned char)shp_j; hrec.pad0 = 0; hrec.pad1 = 0;
    C.hot[p] = hrec;
  }
  __syncwarp();
  }  // work loop
}

// ---- candidate cache after a neighbor rebuild (same atoms, same indices): a pair that was in the old list keeps its
// candidates (the cache's reference state and validity test are unchanged); pairs that are new go to `fresh_list` and
// are built by pair_cache_build_kernel with the next larger margin (they start from a state that may already have used
// up half of the current one).  One thread per new pair; the pool space of a warp is allocated with one atomic.
__global__ void cache_remap_kernel(PairArgs A, const int *old_half_off, const int *old_pair_j, int old_nown, const PairHot *old_hot,
                                   const unsigned short *old_pool, CacheArgs C, int *fresh_list, int *nfresh, const int *amap) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  int ntot = 0, q = -1;
  PairHot hrec;
  hrec.i = hrec.j = 0; hrec.n0 = hrec.n1 = 0; hrec.off = 0; hrec.img = 0; hrec.shp_i = hrec.shp_j = 0; hrec.pad0 = hrec.pad1 = 0;
  if (p < A.npairs) {
    const int i = A.pair_i[p], j = A.pair_j[p], img = A.pair_img[p];
    // amap (decomposed rebuild): the atoms were renumbered; stayers keep their relative order and a ghost only ever
    // matches an old ghost, so a surviving pair keeps its orientation (oi < oj)
    const int oi = amap ? amap[i] : i, oj = amap ? amap[j] : j;
    if (oi >= 0 && oj >= 0 && oi < old_nown && oi < oj)
      for (int e = old_half_off[oi]; e < old_half_off[oi + 1]; e++)
        if (old_pair_j[e] == oj) { q = e; break; }
    if (q >= 0) {
      hrec = old_hot[q];
      if (hrec.n0 < 0 || hrec.img != img || hrec.i != oi || hrec.j != oj) q = -1;
      hrec.i = i; hrec.j = j;
    }
    if (q >= 0) ntot = hrec.n0 + hrec.n1;
    else fresh_list[atomicAdd(nfresh, 1)] = p;
  }
  // warp-aggregated allocation
  int pre = ntot;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, pre, o); if (lane >= o) pre += t; }
  const int wtot = __shfl_sync(0xffffffffu, pre, 31);
  long long base = 0;
  if (lane == 31 && wtot > 0) base = (long long)atomicAdd(C.count, (unsigned long long)wtot);
  base = __shfl_sync(0xffffffffu, base, 31);
  if (q >= 0) {
    const long long off = base + (pre - ntot);
    if (off + ntot <= C.cap) {
      const unsigned short *src = old_pool + hrec.off;
      for (int r = 0; r < ntot; r++) C.pool[off + r] = src[r];
      hrec.off = off;
    } else { *C.overflow = 1; hrec.n0 = -1; hrec.n1 = -1; hrec.off = 0; }   // no room: the pair takes the window path
    C.hot[p] = hrec;
  }
}

// ---- A (fast path): cull from the candidate cache.  LPP lanes per pair (16: two pairs per warp; the typical pair has
// ~40 candidates and ~15 survivors, so half warps keep the lanes busy and halve the dependent-load rounds per pair).
__device__ __forceinline__ void store_pd(PdEntry *dst, long long off, int cnt, int ntrans, int nin, const unsigned short *in,
                                         unsigned int off2 = 0, int cnt2 = 0) {
  PdEntry e;
  e.off = off; e.cnt = cnt; e.ntrans = (unsigned short)ntrans; e.nin = (unsigned short)nin; e.off2 = off2; e.cnt2 = (unsigned short)cnt2;
#pragma unroll
  for (int q = 0; q < PD_INLINE; q++) e.in[q] = (in && q < nin) ? in[q] : (unsigned short)0;
  *dst = e;
}

// the per-shape fields the cached cull touches, handed over in the kernel's constant parameter space: a runtime-indexed
// constant load instead of a chain of dependent global loads (pair -> shape id -> shape record -> table pointer -> table)
struct ShapeLite {
  const float4 *pf4; const float2 *cube_ul; const double *px, *py, *pz;
  int cube_n, pad_;
  double rmax, rmax2, rmin2;
};
struct ShapeLiteTable { ShapeLite s[SH_MAX_SHAPES]; };

template <int WPB, int LPP>
__global__ void __launch_bounds__(WPB * 32, 32 / WPB) pair_cull_cached_kernel(PairArgs A, SplitArgs S, CacheArgs C, int use_bounds,
                                                                              const __grid_constant__ ShapeLiteTable T) {
  constexpr int PPW = 32 / LPP, U = 2;
  constexpr unsigned FULLSUB = LPP == 32 ? 0xffffffffu : ((1u << LPP) - 1u);
  __shared__ double s_dpose[WPB][PPW][2][12];
  __shared__ float s_fpose[WPB][PPW][2][12];
  __shared__ unsigned short s_surv[WPB][PPW][SURV_CAP];
  __shared__ signed char s_flag[WPB][PPW][SURV_CAP];
  __shared__ unsigned short s_in[WPB][PPW][2][8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane / LPP, sl = lane % LPP, shift = sub * LPP;
  const int p = (blockIdx.x * WPB + warp) * PPW + sub;
  if (*C.invalid) return;                 // margin used up: the window kernel takes every pair of this step
  const bool inrange = p < A.npairs;
  PairHot hot;
  hot.i = hot.j = 0; hot.n0 = hot.n1 = 0; hot.off = 0; hot.img = 21; hot.shp_i = hot.shp_j = 0;
  if (inrange) {
    const int4 *hp = reinterpret_cast<const int4 *>(C.hot + p);
    const int4 h0 = __ldg(hp), h1 = __ldg(hp + 1);
    hot.i = h0.x; hot.j = h0.y; hot.n0 = h0.z; hot.n1 = h0.w;
    hot.off = (long long)(((unsigned long long)(unsigned)h1.y << 32) | (unsigned)h1.x);
    hot.img = h1.z; hot.shp_i = (unsigned char)(h1.w & 255); hot.shp_j = (unsigned char)((h1.w >> 8) & 255);
  }
  if (inrange && hot.n0 < 0 && sl == 0) S.slow_list[atomicAdd(&S.sc->nslow, 1)] = p;   // no cache entry: slow path
  const bool cached = inrange && hot.n0 >= 0;
  const int n0 = cached ? hot.n0 : 0, n1 = cached ? hot.n1 : 0, ntot = n0 + n1;
  if (cached && ntot == 0 && sl < 2) store_pd(&S.pd[2 * p + sl], 0, 0, 0, 0, nullptr);   // bounding spheres too far apart
  const int maxtot = __reduce_max_sync(0xffffffffu, ntot);
  if (maxtot == 0) return;
  const bool work = ntot > 0;
  const int i = hot.i, j = hot.j, shp_i = hot.shp_i, shp_j = hot.shp_j;
  const ShapeLite &si = T.s[shp_i], &sj = T.s[shp_j];
  if (work) {   // relative poses of both directions (M, t): 24 elements spread over the pair's lanes
    const int st = A.stride;
    double d[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
      double dk = A.c[k * st + i] - A.c[k * st + j];
      const int n = ((hot.img >> (2 * k)) & 3) - 1;
      if (n != 0) dk = dk - A.boxlen[k] * (double)n;
      d[k] = dk;
    }
    // M of direction 1 (= Rs_i^T Rs_j) is the transpose of M of direction 0 (= Rs_j^T Rs_i), bit for bit: the same three
    // products in the same order, and a product does not depend on the order of its factors.  15 elements, one per lane:
    // 0..8 M0 (and its transpose), 9..11 t0, 12..14 t1.
    if (sl < 15) {
      const int half = sl >= 12, l = half ? sl - 3 : sl;
      const double sgn = half ? -1.0 : 1.0;
      const double val = pose_element(A, half ? j : i, half ? i : j, sgn * d[0], sgn * d[1], sgn * d[2], l);
      s_dpose[warp][sub][half][l] = val;
      s_fpose[warp][sub][half][l] = (float)val;
      if (sl < 9) {
        const int r = sl / 3, k = sl - 3 * r;
        s_dpose[warp][sub][1][3 * k + r] = val;
        s_fpose[warp][sub][1][3 * k + r] = (float)val;
      }
    }
  }
  __syncwarp();
  const float4 *__restrict__ pf_i = si.pf4, *__restrict__ pf_j = sj.pf4;
  const float2 *__restrict__ cube_i = si.cube_ul, *__restrict__ cube_j = sj.cube_ul;
  const int cn_i = si.cube_n, cn_j = sj.cube_n;
  // per-direction FP32 thresholds (direction 0 tests nodes of i against j)
  const float eps0 = fp32_margin(s_fpose[warp][sub][0][9], s_fpose[warp][sub][0][10], s_fpose[warp][sub][0][11], (float)si.rmax);
  const float eps1 = fp32_margin(s_fpose[warp][sub][1][9], s_fpose[warp][sub][1][10], s_fpose[warp][sub][1][11], (float)sj.rmax);
  const float fR20 = (float)sj.rmax2 + eps0, fR21 = (float)si.rmax2 + eps1;
  const unsigned short *__restrict__ cl = C.pool + hot.off;
  unsigned short *surv = s_surv[warp][sub];
  signed char *sflag = s_flag[warp][sub];
  int nsurv = 0, ns0 = 0;
  bool big = false;
  // ---- conservative FP32 stage over the cached candidates
  for (int base = 0; base < maxtot; base += LPP * U) {
    int k[U];
    float4 q[U];
    bool pass[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const int g = base + LPP * u + sl;
      k[u] = (work && !big && g < ntot) ? (int)__ldg(&cl[g]) : -1;
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const int dirc = (base + LPP * u + sl) >= n0;
      q[u] = k[u] >= 0 ? __ldg(&(dirc ? pf_j : pf_i)[k[u]]) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const int dirc = (base + LPP * u + sl) >= n0;
      const float *fp = s_fpose[warp][sub][dirc];
      const float f0 = fmaf(fp[2], q[u].z, fmaf(fp[1], q[u].y, fmaf(fp[0], q[u].x, fp[9])));
      const float f1 = fmaf(fp[5], q[u].z, fmaf(fp[4], q[u].y, fmaf(fp[3], q[u].x, fp[10])));
      const float f2 = fmaf(fp[8], q[u].z, fmaf(fp[7], q[u].y, fmaf(fp[6], q[u].x, fp[11])));
      const float r2 = fmaf(f2, f2, fmaf(f1, f1, f0 * f0));
      bool ok = k[u] >= 0 && r2 < (dirc ? fR21 : fR20);
      if (ok && use_bounds) ok = r2 < __ldg(&(dirc ? cube_i : cube_j)[cube_cell(f0, f1, f2, dirc ? cn_i : cn_j)]).x + (dirc ? eps1 : eps0);
      pass[u] = ok;
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const unsigned mine = (__ballot_sync(0xffffffffu, pass[u]) >> shift) & FULLSUB;
      if (mine) {
        const int nnew = __popc(mine);
        if (nsurv + nnew > SURV_CAP) big = true;
        else {
          if (pass[u]) surv[nsurv + __popc(mine & ((1u << sl) - 1u))] = (unsigned short)k[u];
          const int nd0 = n0 - (base + LPP * u);       // lanes below nd0 belong to direction 0
          ns0 += nd0 >= LPP ? nnew : (nd0 <= 0 ? 0 : __popc(mine & ((1u << nd0) - 1u)));
          nsurv += nnew;
        }
      }
    }
  }
  __syncwarp();
  // ---- exact FP64 stage, pass 1: decide every survivor (0 evaluate, 2 inside, -1 outside), count per direction
  const bool live = work && !big;
  const int maxs = __reduce_max_sync(0xffffffffu, live ? nsurv : 0);
  int c0d0 = 0, c0d1 = 0, c2d0 = 0, c2d1 = 0;
  for (int gb = 0; gb < maxs; gb += LPP) {
    const int g = gb + sl;
    int fl = -1;
    if (live && g < nsurv) {
      const int dirc = g >= ns0, k = surv[g];
      const ShapeLite &sa = dirc ? sj : si;
      const ShapeLite &sb = dirc ? si : sj;
      const double *M = s_dpose[warp][sub][dirc];
      double s0, s1, s2;
      fl = exact_node_stage(M, M + 9, sa.px[k], sa.py[k], sa.pz[k], sb.rmax2, sb.rmin2, sb.cube_ul, sb.cube_n, use_bounds, s0, s1, s2);
      sflag[g] = (signed char)fl;
    }
    const unsigned m0 = (__ballot_sync(0xffffffffu, fl == 0) >> shift) & FULLSUB;
    const unsigned m2 = (__ballot_sync(0xffffffffu, fl == 2) >> shift) & FULLSUB;
    const int nd0 = ns0 - gb;
    const unsigned md0 = nd0 >= LPP ? FULLSUB : (nd0 <= 0 ? 0u : ((1u << nd0) - 1u));
    c0d0 += __popc(m0 & md0); c0d1 += __popc(m0 & ~md0);
    c2d0 += __popc(m2 & md0); c2d1 += __popc(m2 & ~md0);
  }
  // ---- one contiguous run per direction: [records to evaluate][inside nodes beyond the inline capacity]
  // records to evaluate -> the target shape's pool; proven-inside nodes beyond the inline capacity -> the index pool
  const int r0 = c0d0, r1 = c0d1, x0 = max(0, c2d0 - PD_INLINE), x1 = max(0, c2d1 - PD_INLINE);
  long long off0 = 0, off1 = 0, xoff = 0;
  if (live && sl == 0 && r0 > 0) off0 = (long long)atomicAdd(&S.sc->pool_count[shp_j], (unsigned long long)r0);
  if (live && sl == 1 && r1 > 0) off1 = (long long)atomicAdd(&S.sc->pool_count[shp_i], (unsigned long long)r1);
  if (live && sl == 2 && x0 + x1 > 0) xoff = (long long)atomicAdd(&S.sc->in_count, (unsigned long long)(x0 + x1));
  off0 = __shfl_sync(0xffffffffu, off0, shift);
  off1 = __shfl_sync(0xffffffffu, off1, shift + 1);
  xoff = __shfl_sync(0xffffffffu, xoff, shift + 2);
  if (live && (off0 + r0 > S.pool_cap[shp_j] || off1 + r1 > S.pool_cap[shp_i] || xoff + x0 + x1 > S.in_cap)) big = true;   // a pool is full (the host grows it)
  if (work && big && sl == 0) {   // deep contact or full pool: the fused kernel evaluates this pair (and counts it)
    store_pd(&S.pd[2 * p], 0, -1, 0, 0, nullptr);
    store_pd(&S.pd[2 * p + 1], 0, -1, 0, 0, nullptr);
    S.big_list[atomicAdd(&S.sc->nbig, 1)] = p;
  }
  const bool wr = work && !big;
  const long long base0 = S.pool_base[shp_j] + off0, base1 = S.pool_base[shp_i] + off1;
  // ---- pass 2: write the records (s recomputed: 12 DFMA), inline the first inside nodes
  int w0d0 = 0, w0d1 = 0, w2d0 = 0, w2d1 = 0;
  for (int gb = 0; gb < maxs; gb += LPP) {
    const int g = gb + sl;
    const bool v = wr && g < nsurv;
    const int fl = v ? (int)sflag[g] : -1;
    const unsigned m0 = (__ballot_sync(0xffffffffu, fl == 0) >> shift) & FULLSUB;
    const unsigned m2 = (__ballot_sync(0xffffffffu, fl == 2) >> shift) & FULLSUB;
    const int nd0 = ns0 - gb;
    const unsigned md0 = nd0 >= LPP ? FULLSUB : (nd0 <= 0 ? 0u : ((1u << nd0) - 1u));
    const unsigned lt = (1u << sl) - 1u;
    if (fl >= 0) {
      const int dirc = g >= ns0, k = surv[g];
      const unsigned dm = dirc ? ~md0 : md0;
      const int rank0 = (dirc ? w0d1 : w0d0) + __popc(m0 & dm & lt);
      const int rank2 = (dirc ? w2d1 : w2d0) + __popc(m2 & dm & lt);
      int slot = -1;
      if (fl == 0) slot = rank0;
      else if (rank2 < PD_INLINE) s_in[warp][sub][dirc][rank2] = (unsigned short)k;
      else S.inpool[xoff + (dirc ? x0 : 0) + (rank2 - PD_INLINE)] = k;
      if (slot >= 0) {
        const ShapeLite &sa = dirc ? sj : si;
        const double *M = s_dpose[warp][sub][dirc], *t = M + 9;
        const double p0 = sa.px[k], p1 = sa.py[k], p2 = sa.pz[k];
        SurvRec r;
        r.s0 = fma(M[0], p0, t[0]); r.s0 = fma(M[1], p1, r.s0); r.s0 = fma(M[2], p2, r.s0);
        r.s1 = fma(M[3], p0, t[1]); r.s1 = fma(M[4], p1, r.s1); r.s1 = fma(M[5], p2, r.s1);
        r.s2 = fma(M[6], p0, t[2]); r.s2 = fma(M[7], p1, r.s2); r.s2 = fma(M[8], p2, r.s2);
        r.k = k; r.flag = fl;
        const long long idx = (dirc ? base1 : base0) + slot;
        S.pool[idx] = r;
        S.pool_kin[idx] = -1;
      }
    }
    w0d0 += __popc(m0 & md0); w0d1 += __popc(m0 & ~md0);
    w2d0 += __popc(m2 & md0); w2d1 += __popc(m2 & ~md0);
  }
  __syncwarp();
  if (wr && sl < 2) {
    if (sl == 0) store_pd(&S.pd[2 * p], base0, r0, n0, min(c2d0, PD_INLINE), s_in[warp][sub][0], (unsigned int)xoff, x0);
    else store_pd(&S.pd[2 * p + 1], base1, r1, n1, min(c2d1, PD_INLINE), s_in[warp][sub][1], (unsigned int)(xoff + x0), x1);
  }
}

// ---- A (slow path, persistent): window + FP32 pre-cull + exact stage.  Takes the pairs of the slow list, or every
// pair when the cache is off / invalid this step.
template <int WPB>
__global__ void __launch_bounds__(WPB * 32) pair_cull_window_kernel(PairArgs A, SplitArgs S, CacheArgs C, int use_bounds) {
  __shared__ __align__(16) SurvRec s_rec[WPB][2][SPLIT_CAP];
  __shared__ double s_pose[WPB][16];
  __shared__ unsigned short s_cand[WPB][64];
  __shared__ unsigned short s_in[WPB][2][8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool all = !C.enabled || *C.invalid != 0;
  for (;;) {
    int w = 0;
    if (lane == 0) w = atomicAdd(&S.sc->slow_counter, 1);
    w = __shfl_sync(0xffffffffu, w, 0);
    // nslow is final: the cached kernel that fills the list has completed before this kernel starts
    const int nwork = all ? A.npairs : *(volatile int *)&S.sc->nslow;
    if (w >= nwork) break;
    const int p = all ? w : S.slow_list[w];
    const int i = A.pair_i[p], j = A.pair_j[p];
    double d[3];
    pair_separation(A, p, i, j, d);
    const int shp_i = A.shape[i], shp_j = A.shape[j];
    double *pose = s_pose[warp];
    int cnt0 = 0, cnt1 = 0, nin0 = 0, nin1 = 0, nt0 = 0, nt1 = 0;
    bool big = false;
    for (int dir = 0; dir < 2 && !big; dir++) {
      const int a = dir ? j : i, b = dir ? i : j;
      const DevShape &sa = A.shapes[dir ? shp_j : shp_i];
      const DevShape &sb = A.shapes[dir ? shp_i : shp_j];
      const double sgn = dir ? -1.0 : 1.0;
      pose_to_smem(A, a, b, sgn * d[0], sgn * d[1], sgn * d[2], lane, pose);
      const double *M = pose, *t = pose + 9, *x0 = pose + 12;
      const double rmax2 = sb.rmax2, rmin2 = sb.rmin2;
      const double *__restrict__ nodes = sa.px;
      const int nq = sa.nq;
      const float2 *__restrict__ cube = sb.cube_ul;
      const int cn = sb.cube_n;
      SurvRec *buf = s_rec[warp][dir];
      unsigned short *cand = s_cand[warp], *inl = s_in[warp][dir];
      int queued = 0, nin = 0, n_trans = 0;
      auto exact_stage = [&](bool valid, int k) {
        int flag = -1;
        double s0 = 0, s1 = 0, s2 = 0;
        if (valid) flag = exact_node_stage(M, t, nodes[k], nodes[nq + k], nodes[2 * nq + k], rmax2, rmin2, cube, cn, use_bounds, s0, s1, s2);
        // nodes already proven inside go inline into the run descriptor (up to PD_INLINE), the rest become records
        const unsigned m2 = __ballot_sync(0xffffffffu, flag == 2);
        const int rank2 = nin + __popc(m2 & ((1u << lane) - 1u));
        const bool inline_it = flag == 2 && rank2 < PD_INLINE;
        if (inline_it) inl[rank2] = (unsigned short)k;
        nin = min(PD_INLINE, nin + __popc(m2));
        const bool rec = flag >= 0 && !inline_it;
        const unsigned sm = __ballot_sync(0xffffffffu, rec);
        if (sm) {
          const int nnew = __popc(sm);
          if (queued + nnew > SPLIT_CAP) { big = true; return; }
          if (rec) {
            SurvRec r; r.s0 = s0; r.s1 = s1; r.s2 = s2; r.k = k; r.flag = flag;
            buf[queued + __popc(sm & ((1u << lane) - 1u))] = r;
          }
          queued += nnew;
        }
      };
      const NodeWindow wd = make_window(sa, sb.rmax, x0);
      if (!wd.skip) {
        const float4 *__restrict__ pf = sa.pf4;
        const float fM0 = (float)M[0], fM1 = (float)M[1], fM2 = (float)M[2], fM3 = (float)M[3], fM4 = (float)M[4],
                    fM5 = (float)M[5], fM6 = (float)M[6], fM7 = (float)M[7], fM8 = (float)M[8];
        const float ft0 = (float)t[0], ft1 = (float)t[1], ft2 = (float)t[2];
        const float eps = fp32_margin(ft0, ft1, ft2, (float)sa.rmax);
        const float frmax2 = (float)rmax2 + eps;
        const int nth = sa.n_theta, nph = sa.n_phi;
        int ncand = 0;
        for (int rb = 0; rb < nth && !big; rb += 32) {
          int c0, ccount;
          classify_row(sa, wd, rb + lane, c0, ccount);
          unsigned rows = __ballot_sync(0xffffffffu, ccount > 0);
          while (rows && !big) {
            const int rl = __ffs(rows) - 1;
            rows &= rows - 1;
            const int rc0 = __shfl_sync(0xffffffffu, c0, rl), rcount = __shfl_sync(0xffffffffu, ccount, rl);
            const int rowbase = (rb + rl) * nph;
            for (int cb = 0; cb < rcount && !big; cb += 32) {
              const int cc = cb + lane;
              bool pass = false;
              int k = 0;
              if (cc < rcount) {
                int col = rc0 + cc;
                if (col >= nph) col -= nph;
                k = rowbase + col;
                const float4 q = __ldg(&pf[k]);
                const float f0 = fmaf(fM2, q.z, fmaf(fM1, q.y, fmaf(fM0, q.x, ft0)));
                const float f1 = fmaf(fM5, q.z, fmaf(fM4, q.y, fmaf(fM3, q.x, ft1)));
                const float f2 = fmaf(fM8, q.z, fmaf(fM7, q.y, fmaf(fM6, q.x, ft2)));
                const float r2 = fmaf(f2, f2, fmaf(f1, f1, f0 * f0));
                if (r2 < frmax2) pass = !use_bounds || r2 < __ldg(&cube[cube_cell(f0, f1, f2, cn)]).x + eps;
              }
              n_trans += min(32, rcount - cb);
              const unsigned pm = __ballot_sync(0xffffffffu, pass);
              if (pm) {
                if (pass) cand[ncand + __popc(pm & ((1u << lane) - 1u))] = (unsigned short)k;
                ncand += __popc(pm);
                __syncwarp();
                if (ncand >= 32) {
                  exact_stage(true, (int)cand[lane]);
                  __syncwarp();
                  const int rem = ncand - 32;
                  unsigned short mv = 0;
                  if (lane < rem) mv = cand[32 + lane];
                  __syncwarp();
                  if (lane < rem) cand[lane] = mv;
                  ncand = rem;
                  __syncwarp();
                }
              }
            }
          }
        }
        if (!big && ncand > 0) { exact_stage(lane < ncand, lane < ncand ? (int)cand[lane] : 0); __syncwarp(); }
      }
      if (dir) { cnt1 = queued; nin1 = nin; nt1 = n_trans; } else { cnt0 = queued; nin0 = nin; nt0 = n_trans; }
    }
    __syncwarp();
    long long off0 = 0, off1 = 0;
    if (!big) {
      if (lane == 0 && cnt0 > 0) off0 = (long long)atomicAdd(&S.sc->pool_count[shp_j], (unsigned long long)cnt0);
      if (lane == 1 && cnt1 > 0) off1 = (long long)atomicAdd(&S.sc->pool_count[shp_i], (unsigned long long)cnt1);
      off0 = __shfl_sync(0xffffffffu, off0, 0);
      off1 = __shfl_sync(0xffffffffu, off1, 1);
      if (off0 + cnt0 > S.pool_cap[shp_j] || off1 + cnt1 > S.pool_cap[shp_i]) big = true;
    }
    if (big) {   // the fused kernel re-does (and counts) this pair
      if (lane == 0) {
        store_pd(&S.pd[2 * p], 0, -1, 0, 0, nullptr);
        store_pd(&S.pd[2 * p + 1], 0, -1, 0, 0, nullptr);
        S.big_list[atomicAdd(&S.sc->nbig, 1)] = p;
      }
    } else {
      const long long base0 = S.pool_base[shp_j] + off0, base1 = S.pool_base[shp_i] + off1;
      for (int r = lane; r < cnt0; r += 32) { const SurvRec q = s_rec[warp][0][r]; S.pool[base0 + r] = q; S.pool_kin[base0 + r] = q.flag == 2 ? q.k : -1; }
      for (int r = lane; r < cnt1; r += 32) { const SurvRec q = s_rec[warp][1][r]; S.pool[base1 + r] = q; S.pool_kin[base1 + r] = q.flag == 2 ? q.k : -1; }
      if (lane == 0) store_pd(&S.pd[2 * p], base0, cnt0, nt0, nin0, s_in[warp][0]);
      if (lane == 1) store_pd(&S.pd[2 * p + 1], base1, cnt1, nt1, nin1, s_in[warp][1]);
    }
    __syncwarp();
  }
}

// ---- B: evaluate pooled records.  The plan (records and CTA-sized blocks per shape) is computed on the device.
__global__ void eval_plan_kernel(SplitArgs S, int nshape, int recs_per_block, EvalPlanDev *plan) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  int nblk = 0;
  for (int s = 0; s < nshape; s++) {
    const long long cnt = min((long long)S.sc->pool_count[s], S.pool_cap[s]);
    plan->blk_start[s] = nblk;
    plan->count[s] = cnt;
    nblk += (int)((cnt + recs_per_block - 1) / recs_per_block);
  }
  plan->blk_start[nshape] = nblk;
  plan->total_blocks = nblk;
  plan->nshape = nshape;
}

template <int WPB, int PTS, int MINB>
__global__ void __launch_bounds__(WPB * 32, MINB) pair_eval_kernel(const DevShape *shapes, SplitArgs S, const EvalPlanDev *plan,
                                                                   unsigned long long *counters, int chunked) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int RPW = 32 * PTS;               // records per warp task
  const int total = plan->total_blocks, nshape = plan->nshape;
  // chunked: persistent CTAs over contiguous chunks (a table is staged only when the shape changes);
  // else: one block per CTA, grid-stride for whatever the host's grid estimate did not cover
  const int chunk = (total + (int)gridDim.x - 1) / (int)gridDim.x;
  const int b0 = chunked ? blockIdx.x * chunk : blockIdx.x, b1 = chunked ? min(total, b0 + chunk) : total;
  const int bstep = chunked ? 1 : (int)gridDim.x;
  if (b0 >= b1) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double2 *s_ab = reinterpret_cast<double2 *>(smem_raw);
  double *s_Ap = nullptr;
  int cur = -1, s = 0;
  unsigned long long nev_total = 0;
  for (int blk = b0; blk < b1; blk += bstep) {
    while (s + 1 < nshape && blk >= plan->blk_start[s + 1]) s++;
    const DevShape &sh = shapes[s];
    if (s != cur) {
      __syncthreads();
      s_Ap = reinterpret_cast<double *>(s_ab + sh.nterms4 + 4);
      for (int t = threadIdx.x; t < sh.nterms4 + 4; t += WPB * 32) { s_ab[t] = sh.ab[t]; s_Ap[t] = sh.Ap[t]; }
      __syncthreads();
      cur = s;
    }
    const long long n = plan->count[s];
    const long long r0 = ((long long)(blk - plan->blk_start[s]) * WPB + warp) * RPW;
    if (r0 >= n) continue;
    SurvRec *rec = S.pool + S.pool_base[s];
    int *kin = S.pool_kin + S.pool_base[s];
    const int L = sh.lmax;
    int nev = 0;
    if (PTS == 2) {
      const long long ia = r0 + lane, ib = r0 + 32 + lane;
      const bool va = ia < n, vb = ib < n;
      if (__ballot_sync(0xffffffffu, vb)) {
        const long long ja = va ? ia : r0, jb = vb ? ib : ja;
        const SurvRec ra = rec[ja], rb = rec[jb];
        const double sA[3] = {ra.s0, ra.s1, ra.s2}, sB[3] = {rb.s0, rb.s1, rb.s2};
        const double rhoA2 = fma(sA[2], sA[2], fma(sA[1], sA[1], sA[0] * sA[0]));
        const double rhoB2 = fma(sB[2], sB[2], fma(sB[1], sB[1], sB[0] * sB[0]));
        double rhoA, rhoB, rA, rB;
        sh_radius_folded_x2(L, s_Ap, s_ab, sA, rhoA2, sB, rhoB2, rhoA, rhoB, rA, rB);
        if (va && ra.flag == 0) { kin[ia] = rhoA < rA ? ra.k : -1; nev++; }
        if (vb && rb.flag == 0) { kin[ib] = rhoB < rB ? rb.k : -1; nev++; }
      } else if (va) {
        const SurvRec ra = rec[ia];
        const double rho2 = fma(ra.s2, ra.s2, fma(ra.s1, ra.s1, ra.s0 * ra.s0));
        double rho;
        const double r = sh_radius_folded(L, s_Ap, s_ab, ra.s0, ra.s1, ra.s2, rho2, rho);
        if (ra.flag == 0) { kin[ia] = rho < r ? ra.k : -1; nev++; }
      }
    } else {
      double sv[PTS][3], rho2[PTS], rho[PTS], rr[PTS];
      int fl[PTS], kk[PTS];
      long long idx[PTS];
#pragma unroll
      for (int q = 0; q < PTS; q++) {
        idx[q] = r0 + 32 * q + lane;
        const bool v = idx[q] < n;
        const SurvRec r = rec[v ? idx[q] : r0];
        sv[q][0] = r.s0; sv[q][1] = r.s1; sv[q][2] = r.s2;
        fl[q] = v ? r.flag : 3;
        kk[q] = r.k;
        rho2[q] = fma(r.s2, r.s2, fma(r.s1, r.s1, r.s0 * r.s0));
      }
      sh_radius_folded_n<PTS>(L, s_Ap, s_ab, sv, rho2, rho, rr);
#pragma unroll
      for (int q = 0; q < PTS; q++)
        if (fl[q] == 0) { kin[idx[q]] = rho[q] < rr[q] ? kk[q] : -1; nev++; }
    }
    nev_total += nev;
  }
  // records preset by the cull (flag 2 / 3) are not "evaluated"
  nev_total = __reduce_add_sync(0xffffffffu, (unsigned)nev_total);
  if (lane == 0 && nev_total) { atomicAdd(&counters[2], nev_total); atomicAdd(&counters[5], nev_total); }
}

// ---- C: per-pair reduction + contact law (SURVEY A.5).  One THREAD per pair: the node lists are short (a few records, a
// few of them inside) and each direction is summed sequentially in a fixed order: the records of the run, then the
// index-pool run, then the inline nodes.  Fewer than half of the pairs have any node to sum: a CTA compacts those of its
// 256 pairs in shared memory, so that its lanes are full while they sum.  The kernel is bound by its output stores (the
// CSR slot of the reverse entry is a scattered 8 B store per component), and about 80 % of the pairs write the zero record
// step after step: out_zero marks the pairs whose outputs already hold it, and their stores are skipped.  Deep-contact
// pairs (cnt = -1) are done (and counted) by the fused kernel.
struct NodeSums { double S0, S1, S2, Av, T0, T1, T2, G0, G1, G2; int n; };

// one node of the packed table, (px,py) (pz,nx) (ny,nz); the same operations in the same order as the oracle
__device__ __forceinline__ void add_node(NodeSums &a, double2 q0, double2 q1, double2 q2, const double x0[3]) {
  const double p0 = q0.x, p1 = q0.y, p2 = q1.x;
  const double n0 = q1.y, n1 = q2.x, n2 = q2.y;
  const double dp0 = p0 - x0[0], dp1 = p1 - x0[1], dp2 = p2 - x0[2];
  const double dn = fma(dp2, n2, fma(dp1, n1, dp0 * n0));
  a.S0 += n0; a.S1 += n1; a.S2 += n2;
  a.Av += dn;
  a.T0 += fma(p1, n2, -(p2 * n1));
  a.T1 += fma(p2, n0, -(p0 * n2));
  a.T2 += fma(p0, n1, -(p1 * n0));
  a.G0 = fma(dp0, dn, a.G0); a.G1 = fma(dp1, dn, a.G1); a.G2 = fma(dp2, dn, a.G2);
  a.n++;
}

// the 14-double pair record (coalesced across pairs) and the force / torque of the pair's two CSR slots
__device__ __forceinline__ void store_pair_outputs(const PairArgs &A, int p, const double out[14]) {
#pragma unroll
  for (int r = 0; r < 14; r++) A.pres[(size_t)r * A.pres_stride + p] = out[r];
  const int eij = A.pair_eij[p], eji = A.pair_eji[p];
#pragma unroll
  for (int r = 0; r < 3; r++) {
    A.slot[(size_t)r * A.slot_stride + eij] = out[2 + r];
    A.slot[(size_t)(3 + r) * A.slot_stride + eij] = out[5 + r];
    if (eji >= 0) {
      A.slot[(size_t)r * A.slot_stride + eji] = -out[2 + r];
      A.slot[(size_t)(3 + r) * A.slot_stride + eji] = out[8 + r];
    }
  }
}

// writes the pair's outputs unless they are zero and already hold zeros
__device__ __forceinline__ void store_pair_outputs_once(const PairArgs &A, const SplitArgs &S, int p, bool zero, const double out[14]) {
  const bool held = S.out_zero[p] != 0;
  if (zero && held) return;
  store_pair_outputs(A, p, out);
  if (zero != held) S.out_zero[p] = zero ? 1 : 0;
}

// one pair with nodes to sum.  Per direction the node indices come from three sources in order (run records through
// pool_kin, index pool, inline); RB of them are fetched, then their nodes loaded, then summed in order, so that a pair's
// node loads are in flight together.  Returns the number of inside nodes.
__device__ __forceinline__ int reduce_contact_pair(const PairArgs &A, const SplitArgs &S, int p) {
  constexpr int RB = 2;
  {
    const int4 *ep = reinterpret_cast<const int4 *>(S.pd + 2 * (size_t)p);
    const int4 e0a = __ldg(ep), e0b = __ldg(ep + 1), e1a = __ldg(ep + 2), e1b = __ldg(ep + 3);
    const int i = A.pair_i[p], j = A.pair_j[p];
    const int st = A.stride;
    double d[3];
    pair_separation(A, p, i, j, d);
    const int shp_i = A.shape[i], shp_j = A.shape[j];
    double out[14];
#pragma unroll
    for (int r = 0; r < 14; r++) out[r] = 0.0;
    double Ss[2][3], Ts[2][3], Gs[2][3], Asum[2];
    int ninside_pair = 0;
#pragma unroll
    for (int dir = 0; dir < 2; dir++) {
      const int a = dir ? j : i;
      const DevShape &sa = A.shapes[dir ? shp_j : shp_i];
      const double sgn = dir ? -1.0 : 1.0;
      const int4 ea = dir ? e1a : e0a, eb = dir ? e1b : e0b;
      const long long off = (long long)(((unsigned long long)(unsigned)ea.y << 32) | (unsigned)ea.x);
      const int cnt = ea.z, xc = (ea.w >> 16) & 0xffff, nin = eb.y & 0xffff;   // run records, index-pool and inline nodes
      const int nrx = cnt + xc, ntot = nrx + nin;
      const int *__restrict__ kin = S.pool_kin + off;
      const int *__restrict__ xin = S.inpool + (unsigned)eb.x;
      const double2 *__restrict__ pn = sa.pn;
      NodeSums acc;
      acc.S0 = acc.S1 = acc.S2 = acc.Av = acc.T0 = acc.T1 = acc.T2 = acc.G0 = acc.G1 = acc.G2 = 0.0; acc.n = 0;
      double Ra[9];
#pragma unroll
      for (int e = 0; e < 9; e++) Ra[e] = A.Rs[e * st + a];
      double x0[3];
#pragma unroll
      for (int r = 0; r < 3; r++) {
        double hx = Ra[0 + r] * (sgn * d[0]);
        hx = fma(Ra[3 + r], sgn * d[1], hx);
        hx = fma(Ra[6 + r], sgn * d[2], hx);
        x0[r] = -0.5 * hx;
      }
      for (int b = 0; b < ntot; b += RB) {
        int k[RB];
#pragma unroll
        for (int u = 0; u < RB; u++) {
          const int g = b + u;
          if (g < cnt) k[u] = kin[g];                  // -1: the record's node is outside
          else if (g < nrx) k[u] = xin[g - cnt];
          else if (g < ntot) {
            const int h = g - nrx + 3;                 // halfword index inside the second 16 B of the entry (off2, nin, in[])
            const unsigned w = (h >> 1) == 1 ? (unsigned)eb.y : (h >> 1) == 2 ? (unsigned)eb.z : (unsigned)eb.w;
            k[u] = (int)((w >> (16 * (h & 1))) & 0xffffu);
          } else k[u] = -1;
        }
        double2 q[RB][3];
#pragma unroll
        for (int u = 0; u < RB; u++) {
          if (k[u] >= 0) { q[u][0] = pn[4 * k[u]]; q[u][1] = pn[4 * k[u] + 1]; q[u][2] = pn[4 * k[u] + 2]; }
          else q[u][0] = q[u][1] = q[u][2] = make_double2(0.0, 0.0);
        }
#pragma unroll
        for (int u = 0; u < RB; u++)
          if (k[u] >= 0) add_node(acc, q[u][0], q[u][1], q[u][2], x0);
      }
#pragma unroll
      for (int r = 0; r < 3; r++) {
        Ss[dir][r] = Ra[3 * r] * acc.S0 + Ra[3 * r + 1] * acc.S1 + Ra[3 * r + 2] * acc.S2;
        Ts[dir][r] = Ra[3 * r] * acc.T0 + Ra[3 * r + 1] * acc.T1 + Ra[3 * r + 2] * acc.T2;
        Gs[dir][r] = 0.25 * (Ra[3 * r] * acc.G0 + Ra[3 * r + 1] * acc.G1 + Ra[3 * r + 2] * acc.G2);
      }
      Asum[dir] = acc.Av;
      ninside_pair += acc.n;
    }
    const double V = Asum[0] / 3.0 + Asum[1] / 3.0;
    const bool contact = ninside_pair > 0 && V > 0;
    if (contact) {
      const double kk = A.pk[shp_i * SH_MAX_SHAPES + shp_j], mm = A.pm[shp_i * SH_MAX_SHAPES + shp_j];
      double E, pr;
      if (mm == 1.0) { E = kk * V; pr = kk; }
      else { const double pw = pow(V, mm - 1.0); E = kk * pw * V; pr = mm * kk * pw; }
      out[0] = V; out[1] = E;
      double li[3], lj[3];
#pragma unroll
      for (int r = 0; r < 3; r++) {
        li[r] = A.c[r * st + i] - A.x[r * st + i];
        lj[r] = A.c[r * st + j] - A.x[r * st + j];
      }
      const double *Sij = Ss[0], *Sji = Ss[1], *Tij = Ts[0], *Tji = Ts[1];
      const double Ti[3] = {Tij[0] + (li[1] * Sij[2] - li[2] * Sij[1]), Tij[1] + (li[2] * Sij[0] - li[0] * Sij[2]),
                            Tij[2] + (li[0] * Sij[1] - li[1] * Sij[0])};
      const double Tj[3] = {Tji[0] + (lj[1] * Sji[2] - lj[2] * Sji[1]), Tji[1] + (lj[2] * Sji[0] - lj[0] * Sji[2]),
                            Tji[2] + (lj[0] * Sji[1] - lj[1] * Sji[0])};
#pragma unroll
      for (int r = 0; r < 3; r++) {
        out[2 + r] = -pr * (0.5 * (Sij[r] - Sji[r]));
        out[5 + r] = -pr * Ti[r];
        out[8 + r] = -pr * Tj[r];
        out[11 + r] = (A.c[r * st + i] - 0.5 * d[r]) + (Gs[0][r] + Gs[1][r]) / V;
      }
      if (A.dissip) contact_dissipation(A, i, j, shp_i, shp_j, d, lj, out);
    }
    store_pair_outputs_once(A, S, p, !contact, out);
    return ninside_pair;
  }
}

__global__ void __launch_bounds__(128, 4) pair_reduce_kernel(PairArgs A, SplitArgs S) {
  constexpr int PPT = 2;   // pairs per thread in the CTA's range
  __shared__ int s_list[PPT * 128];
  __shared__ int s_n;
  if (threadIdx.x == 0) s_n = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  int c_pairs = 0, c_trans = 0, c_ghost = 0;
#pragma unroll
  for (int q = 0; q < PPT; q++) {
    const int p = (blockIdx.x * PPT + q) * 128 + threadIdx.x;
    bool hit = false;
    if (p < A.npairs) {
      const int4 *ep = reinterpret_cast<const int4 *>(S.pd + 2 * (size_t)p);
      const int4 e0a = __ldg(ep), e0b = __ldg(ep + 1), e1a = __ldg(ep + 2), e1b = __ldg(ep + 3);
      if (e0a.z >= 0) {
        c_pairs++; c_trans += (e0a.w & 0xffff) + (e1a.w & 0xffff); c_ghost += A.pair_j[p] >= A.nlocal;
        // records, index-pool or inline inside nodes in either direction
        hit = e0a.z + e1a.z + ((e0a.w >> 16) & 0xffff) + ((e1a.w >> 16) & 0xffff) + (e0b.y & 0xffff) + (e1b.y & 0xffff) > 0;
        if (!hit) {
          double out[14];
#pragma unroll
          for (int r = 0; r < 14; r++) out[r] = 0.0;
          store_pair_outputs_once(A, S, p, true, out);
        }
      } else if (S.out_zero[p]) S.out_zero[p] = 0;   // the fused kernel writes this pair's outputs
    }
    const unsigned m = __ballot_sync(0xffffffffu, hit);
    int base = 0;
    if (lane == 0 && m) base = atomicAdd(&s_n, __popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (hit) s_list[base + __popc(m & ((1u << lane) - 1u))] = p;
  }
  // counters: one atomic per warp and counter
  c_pairs = __reduce_add_sync(0xffffffffu, c_pairs); c_trans = __reduce_add_sync(0xffffffffu, c_trans);
  c_ghost = __reduce_add_sync(0xffffffffu, c_ghost);
  if (lane == 0) {
    if (c_pairs) atomicAdd(&A.counters[0], (unsigned long long)c_pairs);
    if (c_trans) atomicAdd(&A.counters[1], (unsigned long long)c_trans);
    if (c_ghost) atomicAdd(&A.counters[4], (unsigned long long)c_ghost);
  }
  __syncthreads();
  const int n = s_n;
  int c_inside = 0;
  for (int t = threadIdx.x; t < n; t += 128) c_inside += reduce_contact_pair(A, S, s_list[t]);
  c_inside = __reduce_add_sync(0xffffffffu, c_inside);
  if (lane == 0 && c_inside) atomicAdd(&A.counters[3], (unsigned long long)c_inside);
}

}  // namespace shgpu
