// GLCM fast path: kernelRadius 1, full 3-D, distances [1] (13 angles), symmetrical, unweighted,
// 8-bit levels.  Same semantics as glcm_voxel<> in vox_features.cuh (which stays the generic
// fallback and the in-repo cross-check), restructured for the GPU:
//   * the 27 window levels are compared once (351 compares) into per-position equality bitmasks;
//   * co-occurrence multiplicities come from pairwise compares of (|a-b|, a+b) keys instead of a
//     merged entry list; all "linear in p" features are exact integer sums;
//   * every log2 is a table lookup (arguments are ratios of small integers);
//   * MCC: the level graph's connectivity and 2-colourability are decided with bitmask propagation; only a
//     connected, non-bipartite graph needs an eigen-solve of the symmetric n x n matrix P/sqrt(px px), n <= 18:
//     dense Householder + Laguerre in registers up to 12 levels (glcm_small_solve), a register-resident Lanczos
//     recurrence above (glcm_lanczos.cuh).
// __host__ __device__ so tests/host_emul can check the arithmetic on the CPU (test-only).
#pragma once
#include "vox_features.cuh"
#include "straightline.inc"
#ifndef __CUDACC__
#include <algorithm>
using std::max;
using std::min;
#endif

#ifdef __CUDA_ARCH__
#define RB_CTZ(x) (__ffs((int)(x)) - 1)
#define RB_POPC(x) __popc((unsigned)(x))
#else
#define RB_CTZ(x) __builtin_ctz((unsigned)(x))
#define RB_POPC(x) __builtin_popcount((unsigned)(x))
#endif

#if (defined(__CUDA_ARCH__) || defined(RB_EMULATE_BLOCK)) && defined(RB_GLCM_BLOCK_SYNC)
#define RB_ANGLE_SYNC() __syncthreads()
#else
#define RB_ANGLE_SYNC() ((void)0)
#endif

namespace rb {

constexpr int GF_NA = 13;
constexpr int GF_LOGT = 40;       // log2 table covers 0..2*18+1
constexpr int GF_KT = 256;        // |a-b| tables
#ifndef GF_DENSE_SMALL
#define GF_DENSE_SMALL 1
#endif
#ifndef GF_DENSE_MAX_CLS
#define GF_DENSE_MAX_CLS 10     // n <= 12 solved densely in registers
#endif
#ifndef GF_BREAKDOWN
#define GF_BREAKDOWN 1e-10
#endif

struct GlcmFastTables {
  // per angle (in processing order: 3 axis, 6 face-diagonal, 4 body-diagonal)
  uint8_t orig[GF_NA];            // index of the angle in the reference order (alive bit)
  uint8_t np[GF_NA];              // pairs per angle: 18 / 12 / 8
  uint8_t pA[GF_NA][18], pB[GF_NA][18];      // window positions (z*9+y*3+x) of the two pair ends
  double log2t[GF_LOGT];          // log2(c), log2t[0] = 0 (never used with weight)
  double idm[GF_KT], idmn[GF_KT], id[GF_KT], idn[GF_KT], inv[GF_KT];   // by k = |i-j|
  double lz0[19];                 // Lanczos start vector (see kLanczosStart0)
  double rsq[GF_LOGT];            // 1 / sqrt(c) for the small integer row sums
};

// Lanczos start vector: a fixed table of unstructured components in [0.25, 1.25) (drawn once from a
// PRNG; anything "generic" works -- arithmetic progressions and Weyl sequences do NOT, they are exactly
// deficient for symmetric level graphs).
static const double kLanczosStart0[19] = {0.47733602246716966, 0.56675833970975287, 1.047365457332734, 0.92625467075097456, 0.641109550601909, 0.58281392786638453, 0.84830875358718982, 0.43673418560371335, 0.9227560440146213, 1.1918028652699371, 0.49824571462957101, 1.1988811518333182, 0.91723745310037241, 0.34589793559411208, 0.69183966616781278, 1.1364799193275177, 0.9474534998820221, 0.57647286407011211, 0.9839281633300665};

// Host-side construction (Ng = max gray level of the ROI, as used by Idmn / Idn).
inline void glcm_fast_build_tables(GlcmFastTables& T, int Ng) {
  // reference order of the 13 unidirectional distance-1 angles (cmatrices.c:843-860)
  int ang[13][3], k = 0;
  for (int z = 1; z >= -1; z--) for (int y = 1; y >= -1; y--) for (int x = 1; x >= -1; x--) {
    if (k < 13) { ang[k][0] = z; ang[k][1] = y; ang[k][2] = x; k++; }
  }
  int slot = 0;
  for (int want = 1; want <= 3; want++)        // number of moving dimensions
    for (int a = 0; a < 13; a++) {
      int nm = (ang[a][0] != 0) + (ang[a][1] != 0) + (ang[a][2] != 0);
      if (nm != want) continue;
      T.orig[slot] = (uint8_t)a;
      int n = 0;
      for (int z = 0; z < 3; z++) for (int y = 0; y < 3; y++) for (int x = 0; x < 3; x++) {
        int z2 = z + ang[a][0], y2 = y + ang[a][1], x2 = x + ang[a][2];
        if (z2 < 0 || z2 > 2 || y2 < 0 || y2 > 2 || x2 < 0 || x2 > 2) continue;
        T.pA[slot][n] = (uint8_t)(z * 9 + y * 3 + x);
        T.pB[slot][n] = (uint8_t)(z2 * 9 + y2 * 3 + x2);
        n++;
      }
      T.np[slot] = (uint8_t)n;
      for (int t = n; t < 18; t++) { T.pA[slot][t] = 0; T.pB[slot][t] = 0; }
      slot++;
    }
  for (int i = 0; i < 19; i++) T.lz0[i] = kLanczosStart0[i];
  T.log2t[0] = 0; T.rsq[0] = 0;
  for (int c = 1; c < GF_LOGT; c++) { T.log2t[c] = log2((double)c); T.rsq[c] = 1.0 / sqrt((double)c); }
  for (int d = 0; d < GF_KT; d++) {
    double kk = d;
    T.idm[d] = 1.0 / (1.0 + kk * kk);
    T.idmn[d] = 1.0 / (1.0 + kk * kk / ((double)Ng * Ng));
    T.id[d] = 1.0 / (1.0 + kk);
    T.idn[d] = 1.0 / (1.0 + kk / (double)Ng);
    T.inv[d] = d ? 1.0 / (kk * kk) : 0.0;
  }
}

// the part of the tables the eigen-solver needs (1.1 KB; the solve kernel keeps only this in shared
// memory so that the L1 carve-out goes to the per-thread Lanczos state)
struct GlcmSolveTables {
  uint8_t np[GF_NA];
  uint8_t pA[GF_NA][18], pB[GF_NA][18];
  double lz0[19];
  double rsq[GF_LOGT];
  double rinv[GF_LOGT];           // 1 / c (rinv[0] = 0): row-sum reciprocals of the register Lanczos solver
  // pairs of an angle as bit sets over the 27 window positions: every pair is (p, p + dshift) for a
  // position p in lo_mask
  uint32_t lo_mask[GF_NA];
  uint8_t dshift[GF_NA];
};
RB_HD void glcm_solve_tables_from(const GlcmFastTables& T, GlcmSolveTables& S) {
  for (int a = 0; a < GF_NA; a++) {
    S.np[a] = T.np[a];
    for (int t = 0; t < 18; t++) { S.pA[a][t] = T.pA[a][t]; S.pB[a][t] = T.pB[a][t]; }
    uint32_t lo = 0;
    for (int t = 0; t < T.np[a]; t++) lo |= 1u << (T.pA[a][t] < T.pB[a][t] ? T.pA[a][t] : T.pB[a][t]);
    S.lo_mask[a] = lo;
    S.dshift[a] = (uint8_t)(T.pA[a][0] < T.pB[a][0] ? T.pB[a][0] - T.pA[a][0] : T.pA[a][0] - T.pB[a][0]);
  }
  for (int i = 0; i < 19; i++) S.lz0[i] = T.lz0[i];
  for (int i = 0; i < GF_LOGT; i++) { S.rsq[i] = T.rsq[i]; S.rinv[i] = i ? 1.0 / (double)i : 0.0; }
}

// ---------------------------------------------------------------------------------------------
// Small level graphs (n <= N <= 8, the bulk of the eigen-tasks of smooth images): dense solve held
// entirely in registers.  Level classes are 27-bit position masks, the co-occurrence counts are
// popcounts of shifted masks, the normalised matrix is deflated by its known top eigenpair
// (1, sqrt(R/S)), tridiagonalised by fully unrolled Householder reflections, and the two extreme
// eigenvalues of the tridiagonal are located by Laguerre's iteration.  No local memory, no
// start-vector or orthogonality questions (a bipartite graph simply yields the eigenvalue -1).
#ifdef __CUDA_ARCH__
#define RB_VCMPEQ4_LSB(a, b) (__vcmpeq4((a), (b)) & 0x01010101u)
#else
static inline uint32_t rb_vcmpeq4_lsb(uint32_t a, uint32_t b) {
  const uint32_t x = a ^ b;                                  // zero byte <=> equal
  const uint32_t t = ((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x | 0x7F7F7F7Fu;
  return (~t) >> 7;                                         // 0x01 per equal byte
}
#define RB_VCMPEQ4_LSB(a, b) rb_vcmpeq4_lsb((a), (b))
#endif

// W7: the 27 window levels packed 4 per word (byte p & 3 of word p >> 2; the 28th byte is 0).
RB_HD void glcm_pack_window(const uint8_t* w, int ws, uint32_t* W7) {
#pragma unroll
  for (int k = 0; k < 7; k++) {
    uint32_t v = 0;
#pragma unroll
    for (int b = 0; b < 4; b++) if (4 * k + b < 27) v |= (uint32_t)w[(4 * k + b) * ws] << (8 * b);
    W7[k] = v;
  }
}
// bit p set <=> window position p holds `lev`
RB_HD uint32_t glcm_eq_positions(const uint32_t* W7, uint32_t lev) {
  const uint32_t rep = lev * 0x01010101u;
  uint32_t m = 0;
#pragma unroll
  for (int k = 0; k < 7; k++) m |= ((RB_VCMPEQ4_LSB(W7[k], rep) * 0x01020408u) >> 24) << (4 * k);
  return m & 0x7FFFFFFu;
}

// both extreme eigenvalues of the symmetric tridiagonal (d[0..N-1], e[1..N-1]) held in registers:
// two Laguerre iterations from outside the spectrum (monotone; cubic for a simple root, linear for
// a repeated one) advanced in one loop, Sturm bisection for an end that has not settled.
template <int N>
RB_HD double tridiag_bisect_static(const double* d, const double* e, double lo, double hi, int k) {
  for (int it = 0; it < 36; it++) {
    const double xm = 0.5 * (lo + hi);
    double pm2 = 1.0, pm1 = d[0] - xm;
    int cnt = pm1 <= 0;
#pragma unroll
    for (int i = 1; i < N; i++) {
      const double e2 = e[i] * e[i];
      if (e2 == 0) { pm2 = 1.0; pm1 = d[i] - xm; cnt += pm1 <= 0; continue; }
      const double p = (d[i] - xm) * pm1 - e2 * pm2;
      const bool neg_prev = pm1 < 0 || (pm1 == 0 && pm2 > 0);
      const bool neg_cur = p < 0 || (p == 0 && !neg_prev);
      cnt += neg_cur != neg_prev;
      pm2 = pm1; pm1 = p;
    }
    if (cnt > k) hi = xm; else lo = xm;
  }
  return 0.5 * (lo + hi);
}
// SYNC (device, block-uniform callers only): the iteration count is agreed across the block and every
// iteration starts at a barrier, so the block's warps stream this code together (see RB_ANGLE_SYNC).
template <int N, bool SYNC>
RB_HD void tridiag_extreme_pair_static(const double* d, const double* e, double* hi_out, double* lo_out, bool live) {
  double lo = d[0], hi = d[0];
#pragma unroll
  for (int i = 0; i < N; i++) {
    const double r = (i > 0 ? fabs(e[i]) : 0.0) + (i + 1 < N ? fabs(e[i + 1]) : 0.0);
    lo = fmin(lo, d[i] - r); hi = fmax(hi, d[i] + r);
  }
  double x[2] = {hi + 1e-9, lo - 1e-9};
  bool done[2] = {!live, !live};
  for (int it = 0; it < 24; it++) {
    const bool pending = !(done[0] && done[1]);
#if defined(__CUDA_ARCH__) || defined(RB_EMULATE_BLOCK)
    if (SYNC) { if (!__syncthreads_or(pending)) break; } else
#endif
    if (!pending) break;
#pragma unroll
    for (int c = 0; c < 2; c++) {
      double p0 = 1.0, p1 = d[0] - x[c], q0 = 0.0, q1 = -1.0, r0 = 0.0, r1 = 0.0;   // p, p', p''
#pragma unroll
      for (int i = 1; i < N; i++) {
        const double a = d[i] - x[c], b = e[i] * e[i];
        const double p2 = a * p1 - b * p0;
        const double q2 = a * q1 - p1 - b * q0;
        const double r2 = a * r1 - 2.0 * q1 - b * r0;
        p0 = p1; p1 = p2; q0 = q1; q1 = q2; r0 = r1; r1 = r2;
      }
      if (done[c]) continue;
      if (p1 == 0) { done[c] = true; continue; }
      const double G = q1 / p1, H = G * G - r1 / p1;
      const double disc = (double)(N - 1) * ((double)N * H - G * G);
      const double sq = sqrt(disc > 0 ? disc : 0.0);
      const double den = fabs(G + sq) > fabs(G - sq) ? G + sq : G - sq;
      if (den == 0 || den != den) continue;            // stalls: left to the bisection below
      const double step = (double)N / den;
      x[c] -= step;
      if (fabs(step) < 1e-10) done[c] = true;
    }
  }
  *hi_out = done[0] ? x[0] : tridiag_bisect_static<N>(d, e, lo - 1e-9, hi + 1e-9, N - 1);
  *lo_out = done[1] ? x[1] : tridiag_bisect_static<N>(d, e, lo - 1e-9, hi + 1e-9, 0);
  if (!live) { *hi_out = 0; *lo_out = 0; }
}

// second largest |eigenvalue| of the normalised co-occurrence matrix of angle slot s whose level
// graph has at most N nodes.  *ok = false (nothing computed) if it has more.
#if defined(__CUDA_ARCH__) || defined(RB_EMULATE_BLOCK)      // RB_EMULATE_BLOCK: tests/host_emul/solve_kernel_emul.cpp
#define RB_SOLVE_SYNC() do { if (SYNC) __syncthreads(); } while (0)
#else
#define RB_SOLVE_SYNC() do { } while (0)
#endif
template <int N, bool SYNC = false, class TT>
RB_HD double glcm_small_solve(const uint8_t* w, int ws, const uint32_t* W7, const TT& T, int s, bool* ok, bool live = true) {
  RB_SOLVE_SYNC();
  const int dsh = T.dshift[s];
  const uint32_t NZ = ~glcm_eq_positions(W7, 0u) & 0x7FFFFFFu;
  const uint32_t VL = NZ & (NZ >> dsh) & T.lo_mask[s];        // valid pairs, by their lower position
  uint32_t U = VL | (VL << dsh);                               // positions of all pair ends
  uint32_t El[N], Eh[N];
  int R[N];
#pragma unroll
  for (int i = 0; i < N; i++) {
    uint32_t E = 0;
    if (U) { E = glcm_eq_positions(W7, w[RB_CTZ(U) * ws]); U &= ~E; }
    El[i] = E & VL;                 // pairs whose lower end is in class i
    Eh[i] = (E >> dsh) & VL;        // pairs whose upper end is in class i
    R[i] = RB_POPC(El[i]) + RB_POPC(Eh[i]);
  }
  *ok = U == 0;
  if (!SYNC && U) return 0.0;                 // (block-uniform callers carry on: no divergent exit before a barrier)
  if (U) live = false;
  RB_SOLVE_SYNC();
  const double invS = 1.0 / (2.0 * RB_POPC(VL));
  double v1[N], rs[N];
#pragma unroll
  for (int i = 0; i < N; i++) { rs[i] = T.rsq[R[i]]; v1[i] = sqrt(R[i] * invS); }
  // deflated matrix A = M - v1 v1^T (lower triangle used)
  double a[N][N];
#pragma unroll
  for (int i = 0; i < N; i++)
#pragma unroll
    for (int j = 0; j <= i; j++) {
      const int c = (i == j) ? 2 * RB_POPC(El[i] & Eh[i]) : RB_POPC(El[i] & Eh[j]) + RB_POPC(El[j] & Eh[i]);
      a[i][j] = c * rs[i] * rs[j] - v1[i] * v1[j];
    }
  // Householder tridiagonalisation, column by column (k = column being reduced)
  double d[N], e[N];
  e[0] = 0;
#pragma unroll
  for (int k = 0; k + 2 < N; k++) {
    RB_SOLVE_SYNC();
    double sigma = 0;
#pragma unroll
    for (int i = k + 2; i < N; i++) sigma += a[i][k] * a[i][k];
    const double x0 = a[k + 1][k];
    d[k] = a[k][k];
    if (sigma < 1e-30) { e[k + 1] = x0; continue; }      // column already tridiagonal
    const double nrm = sqrt(x0 * x0 + sigma);
    const double alpha = x0 > 0 ? -nrm : nrm;
    double v[N], pv[N];
    v[k + 1] = x0 - alpha;
#pragma unroll
    for (int i = k + 2; i < N; i++) v[i] = a[i][k];
    const double beta = -1.0 / (alpha * v[k + 1]);            // 2 / v^T v
    double K = 0;
#pragma unroll
    for (int i = k + 1; i < N; i++) {
      double acc = 0;
#pragma unroll
      for (int j = k + 1; j < N; j++) acc += (j <= i ? a[i][j] : a[j][i]) * v[j];
      pv[i] = beta * acc;
      K += v[i] * pv[i];
    }
    K *= 0.5 * beta;
#pragma unroll
    for (int i = k + 1; i < N; i++) pv[i] -= K * v[i];
#pragma unroll
    for (int i = k + 1; i < N; i++)
#pragma unroll
      for (int j = k + 1; j <= i; j++) a[i][j] -= v[i] * pv[j] + pv[i] * v[j];
    e[k + 1] = alpha;
  }
  d[N - 2] = a[N - 2][N - 2]; e[N - 1] = a[N - 1][N - 2]; d[N - 1] = a[N - 1][N - 1];
  double hi, lo;
  RB_SOLVE_SYNC();
  tridiag_extreme_pair_static<N, SYNC>(d, e, &hi, &lo, live);
  return fmax(fabs(hi), fabs(lo));
}

}  // namespace rb
#include "glcm_lanczos.cuh"
namespace rb {

// large eigen-task (n >= 13 levels) of angle slot s by size class; sm = LZ_NARR*18 doubles of per-thread scratch with
// element stride st.  Only the three axis angles (slots 0..2, 18 pairs) can carry a connected NON-bipartite graph on
// 13+ levels: a 12-pair angle reaches 13 levels only as a tree, and 19 levels on 18 pairs is a tree too -- trees are
// bipartite, eigenvalue -1, MCC term 1 (phase A filters them; answered here as well so the function is total).
template <class TT>
RB_HD double glcm_lanczos_solve(const uint8_t* w, int ws, const TT& T, int s, int cls, double* sm, int st) {
  if (s > 2) return 1.0;
  int n = 0;
  double r;
  if (cls <= 12) r = glcm_lanczos_task<14>(w, ws, T, s, sm, st, &n);
  else if (cls <= 14) r = glcm_lanczos_task<16>(w, ws, T, s, sm, st, &n);
  else { r = glcm_lanczos_task<18>(w, ws, T, s, sm, st, &n); if (n == 19) r = 1.0; }
  return r;
}

// eigen-task entry point of the single-thread composition (host emulation / generic callers).  cls = n - 2
// (glcm_task_class).  The device kernels call glcm_small_solve / glcm_lanczos_task directly, one size at a time.
template <class TT>
RB_HD double glcm_fast_solve(const uint8_t* w, int ws, const TT& T, int s, int cls) {
  if (cls <= GF_DENSE_MAX_CLS) {
    uint32_t W7[7];
    glcm_pack_window(w, ws, W7);
    bool ok = false;
    double r;
    if (cls <= 2) r = glcm_small_solve<4>(w, ws, W7, T, s, &ok);
    else if (cls <= 4) r = glcm_small_solve<6>(w, ws, W7, T, s, &ok);
    else if (cls <= 6) r = glcm_small_solve<8>(w, ws, W7, T, s, &ok);
    else if (cls <= 8) r = glcm_small_solve<10>(w, ws, W7, T, s, &ok);
    else r = glcm_small_solve<12>(w, ws, W7, T, s, &ok);
    return ok ? r : NAN;               // (cannot fail: cls is the exact node count)
  }
  double sm[LZ_NARR * 18];
  return glcm_lanczos_solve(w, ws, T, s, cls, sm, 1);
}

// size class of an eigen-task (number of level nodes) -- tasks of one class share a warp
// (16 keys: n - 2, clamped; ncu showed 11 of 32 lanes active with 8 coarser classes because the loop
// lengths of the sparse solver follow n)
constexpr int GF_NCLS = 16, GF_CLS_BITS = 4;
RB_HD int glcm_task_class(int n) { return n <= 2 ? 0 : n >= 17 ? 15 : n - 2; }

struct GlcmAcc {
  double sum[GLCM_NF];
  int n_ok, n_imc2;
  uint32_t tasks;      // bit s set: angle slot s needs an MCC eigen-solve (added to sum[G_MCC] later)
  unsigned long long tcls;   // GF_CLS_BITS per slot: size class of the task (see glcm_task_class)
  bool ja_nan;
};

// one angle (slot s) of one voxel.  w: the 27 window levels (stride ws), eq: equality masks.
template <int NP>
RB_HD void glcm_fast_angle(const uint8_t* w, int ws, const uint32_t* eq, int es,
                           const GlcmFastTables& T, int s, const VoxParams& P, GlcmAcc& acc) {
  const uint8_t* pA = T.pA[s];
  const uint8_t* pB = T.pB[s];
  // key1 = (a+b) << 8 | |a-b| identifies the unordered level pair; key2 = |a-b|.  Invalid pairs
  // (an end outside the mask / volume) get distinct large keys and sort behind the n valid ones.
  int key1[NP], key2[NP];
  uint32_t valid = 0, EA = 0, EB = 0;
  int n = 0, Ssum = 0, Sab = 0, Sq = 0, Skd = 0;
  bool selfpair = false;               // a level paired with itself: the level graph has a self-loop
#pragma unroll
  for (int t = 0; t < NP; t++) {
    const int a = w[pA[t] * ws], b = w[pB[t] * ws];
    const bool ok = a != 0 && b != 0;
    const int kd = a > b ? a - b : b - a, ks = a + b;
    key1[t] = ok ? (ks << 8 | kd) : (0x100000 + t);
    key2[t] = ok ? kd : (0x1000 + t);
    if (ok) {
      valid |= 1u << t; EA |= 1u << pA[t]; EB |= 1u << pB[t];
      n++; Ssum += ks; Sab += a * b; Sq += a * a + b * b; Skd += kd;
      selfpair |= kd == 0;
    }
  }
  const int orig = T.orig[s];
  if (n == 0) {
    if (P.alive[orig >> 5] >> (orig & 31) & 1u) acc.ja_nan = true;
    return;
  }
  // ---- level classes of the pair ends: marginal entropy and the level graph of this angle.
  // R(level) = number of matrix entries in its row = popcount(class & EA) + popcount(class & EB);
  // sum_levels R log2 R = sum over the 2n pair ends of log2 R(their level).
  // (Straight-line per-pair code on purpose: a loop over the classes with its shared-memory load in the carried
  // dependence measured 25 % slower for the whole kernel -- 8 to 16 warps per SM cannot hide a 30-cycle chain per class.)
  double rl = 0;
  uint32_t reps = 0, all = 0, comp = 0;
  uint32_t em[NP];
#pragma unroll
  for (int t = 0; t < NP; t++) {
    em[t] = 0;
    if (valid >> t & 1u) {
      const uint32_t ea = eq[pA[t] * es], eb = eq[pB[t] * es];
      rl += T.log2t[RB_POPC(ea & EA) + RB_POPC(ea & EB)] + T.log2t[RB_POPC(eb & EA) + RB_POPC(eb & EB)];
      reps |= (ea & (0u - ea)) | (eb & (0u - eb));          // lowest position of each class
      em[t] = ea | eb;
      all |= em[t];
      if (!comp) comp = em[t];
    }
  }
  const int nlev = RB_POPC(reps);
  // ---- MCC classification (glcm.py:679-707, see file header): several components -> 1; a connected bipartite
  // level graph (no level paired with itself, no odd cycle: 29 % of the connected graphs of i.i.d. uniform levels,
  // all trees among them) has the eigenvalue -1 next to +1 -> 1 without a solve; else an eigen-task for phase B.
  double mcc;
  if (P.n_roi_levels < 2) mcc = 1.0;
  else if (nlev < 2) mcc = 0.0;
  else {
    for (int sweep = 0; sweep < NP; sweep++) {
      const uint32_t before = comp;
#pragma unroll
      for (int t = 0; t < NP; t++) if (em[t] & comp) comp |= em[t];
      if (comp == before) break;
    }
    bool bipartite = false;
    if (comp == all && !selfpair) {
      // 2-colouring by a breadth-first sweep over class masks (<= 2 nlev closure steps; round 1 swept the pair list
      // instead -- 18 % of this kernel's instructions -- and had moved the test into the solver thread for that reason)
      bool connected;
      glcm_graph_scan(eq, es, EA, (int)pB[0] - (int)pA[0], EA | EB, false, &connected, &bipartite, true);
    }
    if (comp != all || bipartite) mcc = 1.0;
    else {
      // connected, not bipartite: queued for phase B
      mcc = 0.0; acc.tasks |= 1u << s;
      acc.tcls |= (unsigned long long)glcm_task_class(nlev) << (GF_CLS_BITS * s);
    }
  }
  if (NP == 18) { RB_SORTNET_18(key1); RB_SORTNET_18(key2); }
  else if (NP == 12) { RB_SORTNET_12(key1); RB_SORTNET_12(key2); }
  else { RB_SORTNET_8(key1); RB_SORTNET_8(key2); }
  // S = 2n entries' worth of counts.  Every moment below is an exact integer numerator over a
  // power of S (no cancellation between rounded quantities).
  const int S2 = 2 * n;
  const double S = (double)S2, invS = 1.0 / S, invS2 = invS * invS;
  const double ux = Ssum * invS;
  const double ac = 2.0 * Sab * invS;
  const double contrast = 2.0 * (double)(Sq - 2 * Sab) * invS;
  const int vnum = S2 * Sq - Ssum * Ssum;                       // S^2 * var_x  (>= 0, exact)
  const double sxx = vnum * invS2;
  const double sxy = (double)(2 * Sab * S2 - Ssum * Ssum) * invS2;
  const double ct = (double)(2 * (Sq + 2 * Sab) * S2 - 4 * Ssum * Ssum) * invS2;
  const double da = 2.0 * Skd * invS;
  const double dvar = (double)(2 * (Sq - 2 * Sab) * S2 - 4 * Skd * Skd) * invS2;
  // scan the sorted keys: runs of equal key1 = merged matrix entries (length nn), runs of equal
  // a+b = p_{x+y} bins, runs of equal key2 = p_{x-y} bins (the |i-j| table features are taken per run)
  double cs = 0, cp = 0, idm = 0, idmn = 0, id = 0, idn = 0, inv = 0, lgE = 0, lgD = 0, lgS = 0;
  int E2 = 0, cmax = 0, runK = 0, runS = 0, runD = 0;
#pragma unroll
  for (int i = 0; i < NP; i++) {
    if (i < n) {
      const int k1 = key1[i], ks = k1 >> 8, kd = k1 & 255, k2 = key2[i];
      const double dn = (double)(ks * n - Ssum), d2 = dn * dn;   // (i+j-ux-uy) * n, an integer
      cs += d2 * dn; cp += d2 * d2;
      const int nx1 = (i + 1 < NP) ? key1[i + 1 < NP ? i + 1 : i] : -1;
      const int nx2 = (i + 1 < NP) ? key2[i + 1 < NP ? i + 1 : i] : -1;
      const bool last = (i + 1 == n);
      runK++; runS++; runD++;
      if (last || nx1 != k1) {                 // end of a merged-entry run
        const int c = kd ? runK : 2 * runK;    // count of the matrix entry (both orders when i != j)
        E2 += kd ? 2 * runK * runK : 4 * runK * runK;
        if (c > cmax) cmax = c;
        lgE += runK * T.log2t[c];
        runK = 0;
      }
      if (last || (nx1 >> 8) != ks) { lgS += runS * T.log2t[2 * runS]; runS = 0; }
      if (last || nx2 != k2) {                 // end of a |i-j| bin
        const double r = (double)runD;
        lgD += r * T.log2t[2 * runD];
        idm += r * T.idm[k2]; idmn += r * T.idmn[k2]; id += r * T.id[k2]; idn += r * T.idn[k2]; inv += r * T.inv[k2];
        runD = 0;
      }
    }
  }
  const double invn = 1.0 / n, invn2 = invn * invn;
  const double lS = T.log2t[2 * n];
  const double hxy = -2.0 * invS * (lgE - n * lS);
  const double dent = -2.0 * invS * (lgD - n * lS);
  const double sent = -2.0 * invS * (lgS - n * lS);
  const double hx0 = nlev > 1 ? lS - rl * invS : 0.0;   // one level: exactly 0 (avoids 0/rounding in Imc1)
  // HX = HY = hx0 and HXY1 = HXY2 = 2*hx0 (sum_ij p log2(px py) = sum_i px log2 px + sum_j py log2 py);
  // the reference's "+eps" inside each log2 shifts these by < 1e-13 and is dropped consistently.
  const double hx = hx0, hxy2 = 2.0 * hx0, hxy1 = hxy2;
  double f[GLCM_NF];
  f[G_Autocorrelation] = ac; f[G_JointAverage] = ux;
  f[G_ClusterProminence] = cp * invn2 * invn2 * invn; f[G_ClusterShade] = cs * invn2 * invn2; f[G_ClusterTendency] = ct;
  f[G_Contrast] = contrast;
  f[G_Correlation] = (vnum == 0) ? 1.0 : sxy / (sxx + EPS);
  f[G_DifferenceAverage] = da; f[G_DifferenceEntropy] = dent; f[G_DifferenceVariance] = dvar;
  f[G_JointEnergy] = E2 * invS2; f[G_JointEntropy] = hxy;
  f[G_Imc1] = (hx != 0) ? (hxy - hxy1) / hx : 0.0;
  // exactly independent margins give HXY2 == HXY in the reference (value 0); here the two are
  // built from different table sums, so "equal" means equal to rounding
  const double dxy = hxy2 - hxy;
  f[G_Imc2] = (fabs(dxy) < 1e-12) ? 0.0 : sqrt(1.0 - exp(-2.0 * dxy));
  f[G_Idm] = 2.0 * idm * invS; f[G_Idmn] = 2.0 * idmn * invS; f[G_Id] = 2.0 * id * invS; f[G_Idn] = 2.0 * idn * invS;
  f[G_InverseVariance] = 2.0 * inv * invS;
  f[G_MaximumProbability] = cmax * invS; f[G_SumAverage] = 2.0 * ux; f[G_SumEntropy] = sent; f[G_SumSquares] = sxx;
  f[G_MCC] = mcc;
#pragma unroll
  for (int k = 0; k < GLCM_NF; k++) if (k != G_Imc2) acc.sum[k] += f[k];
  acc.n_ok++;
  if (f[G_Imc2] == f[G_Imc2]) { acc.sum[G_Imc2] += f[G_Imc2]; acc.n_imc2++; }
}

// Phase A of one voxel: everything except the MCC eigen-solves.  w: the 27 window levels (0 =
// unmasked / outside); eq: scratch for 27 equality masks, element stride es (shared memory on the
// device).  Writes the 24 means (MCC without the pending tasks) and returns the task bitmask.
RB_HD uint32_t glcm_fast_voxel_phaseA(const uint8_t* w, int ws, uint32_t* eq, int es, const GlcmFastTables& T,
                                      const VoxParams& P, double* out, int* n_ok_out, unsigned long long* tcls_out = nullptr) {
  uint32_t e[27];
  int wl[27];
#pragma unroll
  for (int p = 0; p < 27; p++) wl[p] = w[p * ws];
  RB_EQMASKS_27(wl, e);
#pragma unroll
  for (int p = 0; p < 27; p++) eq[p * es] = e[p];
  GlcmAcc acc;
#pragma unroll
  for (int k = 0; k < GLCM_NF; k++) acc.sum[k] = 0;
  acc.n_ok = 0; acc.n_imc2 = 0; acc.ja_nan = false; acc.tasks = 0; acc.tcls = 0;
  // RB_ANGLE_SYNC: on the device the block re-converges before every angle so that its warps walk
  // the (large, fully unrolled) angle bodies together and share instruction-cache lines -- without
  // it the kernel is instruction-fetch bound (ncu: 15 "no_instruction" stall cycles per issue).
  for (int s = 0; s < 3; s++) { RB_ANGLE_SYNC(); glcm_fast_angle<18>(w, ws, eq, es, T, s, P, acc); }
  for (int s = 3; s < 9; s++) { RB_ANGLE_SYNC(); glcm_fast_angle<12>(w, ws, eq, es, T, s, P, acc); }
  for (int s = 9; s < 13; s++) { RB_ANGLE_SYNC(); glcm_fast_angle<8>(w, ws, eq, es, T, s, P, acc); }
  *n_ok_out = acc.n_ok;
  if (tcls_out) *tcls_out = acc.tcls;
  const double inv = acc.n_ok ? 1.0 / acc.n_ok : NAN;
#pragma unroll
  for (int k = 0; k < GLCM_NF; k++) out[k] = acc.n_ok ? acc.sum[k] * inv : NAN;
  out[G_Imc2] = acc.n_imc2 ? acc.sum[G_Imc2] / acc.n_imc2 : NAN;
  if (acc.ja_nan) out[G_JointAverage] = NAN;
  if (P.n_roi_levels < 2) out[G_MCC] = 1.0;      // flat ROI: 1 for every centre, with or without pairs (glcm.py:702)
  return acc.tasks;
}

// finish MCC: add the solved eigen-tasks (in slot order) to the partial mean written by phase A
RB_HD double glcm_fast_finish_mcc(double partial_mean, int n_ok, uint32_t tasks, const double* solved, int ss) {
  double add = 0;
  for (int s = 0; s < GF_NA; s++) if (tasks >> s & 1u) add += solved[s * ss];
  return n_ok ? partial_mean + add / n_ok : partial_mean;
}

// single-thread composition (host emulation / reference for the two-phase kernel)
RB_HD void glcm_fast_voxel(const uint8_t* w, int ws, uint32_t* eq, int es, const GlcmFastTables& T,
                           const VoxParams& P, double* out) {
  int n_ok = 0;
  unsigned long long tcls = 0;
  const uint32_t tasks = glcm_fast_voxel_phaseA(w, ws, eq, es, T, P, out, &n_ok, &tcls);
  double solved[GF_NA];
  GlcmSolveTables ST;
  glcm_solve_tables_from(T, ST);
  for (int s = 0; s < GF_NA; s++) solved[s] = (tasks >> s & 1u) ? glcm_fast_solve(w, ws, ST, s, (int)(tcls >> (GF_CLS_BITS * s) & (GF_NCLS - 1))) : 0.0;
  out[G_MCC] = glcm_fast_finish_mcc(out[G_MCC], n_ok, tasks, solved, 1);
}

}  // namespace rb
