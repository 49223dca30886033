// Per-voxel (kernel-window) texture feature math for the fused voxel-based kernels.
//
// Every function here is __host__ __device__: the CUDA kernels in voxel_kernels.cu call them
// with one thread per centre voxel, and tests/host_emul compiles the very same header with g++
// to check the arithmetic against the oracle without a GPU (test-only; the product has no CPU
// path).  Nothing is materialised per voxel except a sparse entry list: the reference's dense
// Nvox x Ng x Ng x Na matrix (reference radiomics/src/_cmatrices.c:143-146,163,185) never exists.
//
// Semantics follow (file:line in /root/reference):
//   window / clipping      radiomics/src/_cmatrices.c:1120-1147 (set_bb): a clipped box equals the
//                          full (2r+1)^3 window with out-of-volume voxels treated as unmasked
//   GLCM counting          radiomics/src/cmatrices.c:31-89;   features radiomics/glcm.py:149-887
//   GLRLM runs             radiomics/src/cmatrices.c:340-535; features radiomics/glrlm.py:120-523
//   GLSZM zones            radiomics/src/cmatrices.c:144-260; features radiomics/glszm.py:108-434
//   GLDM dependence        radiomics/src/cmatrices.c:687-750; features radiomics/gldm.py:103-430
//   NGTDM                  radiomics/src/cmatrices.c:582-654; features radiomics/ngtdm.py:112-287
#pragma once
#include <math.h>
#include <stdint.h>

#ifdef __CUDACC__
#define RB_HD __host__ __device__ __forceinline__
#define RB_HDN __host__ __device__ __noinline__
#else
#define RB_HD inline
#define RB_HDN inline
#endif

namespace rb {

constexpr int NA_MAX = 344;      // bidirectional offsets for distances subset of {1,2,3}
constexpr int NW_MAX = 172;      // unidirectional (weights exist for GLCM/GLRLM only)
constexpr double EPS = 2.220446049250313e-16;  // np.spacing(1)
constexpr uint16_t NOLEV = 0xFFFF;

enum GlcmF { G_Autocorrelation, G_ClusterProminence, G_ClusterShade, G_ClusterTendency, G_Contrast,
             G_Correlation, G_DifferenceAverage, G_DifferenceEntropy, G_DifferenceVariance, G_Id, G_Idm,
             G_Idmn, G_Idn, G_Imc1, G_Imc2, G_InverseVariance, G_JointAverage, G_JointEnergy,
             G_JointEntropy, G_MCC, G_MaximumProbability, G_SumAverage, G_SumEntropy, G_SumSquares,
             GLCM_NF };
enum GlrlmF { R_GrayLevelNonUniformity, R_GrayLevelNonUniformityNormalized, R_GrayLevelVariance,
              R_HighGrayLevelRunEmphasis, R_LongRunEmphasis, R_LongRunHighGrayLevelEmphasis,
              R_LongRunLowGrayLevelEmphasis, R_LowGrayLevelRunEmphasis, R_RunEntropy,
              R_RunLengthNonUniformity, R_RunLengthNonUniformityNormalized, R_RunPercentage,
              R_RunVariance, R_ShortRunEmphasis, R_ShortRunHighGrayLevelEmphasis,
              R_ShortRunLowGrayLevelEmphasis, GLRLM_NF };
// generic "level x size" quantities shared by GLSZM and GLDM
enum SizeF { S_GLN, S_GLNN, S_GLV, S_HGLE, S_LargeE, S_LargeHGLE, S_LargeLGLE, S_LGLE, S_SizeNU,
             S_SizeNUN, S_SmallE, S_SmallHGLE, S_SmallLGLE, S_Entropy, S_Percentage, S_SizeVar, SIZE_NF };
constexpr int GLSZM_NF = 16;   // alphabetical order of the reference feature names == SizeF order
constexpr int GLDM_NF = 14;
enum NgtdmF { N_Busyness, N_Coarseness, N_Complexity, N_Contrast, N_Strength, NGTDM_NF };

struct VoxParams {
  int Z, Y, X;              // volume dims
  long long sz, sy;         // element strides of the level volume (x stride 1)
  int rz, ry, rx;           // window radius per dimension (0 in the force2D dimension)
  int na;                   // number of offsets in ang[]
  int symmetric;            // GLCM: symmetricalGLCM
  int weighted;             // GLCM/GLRLM: weightingNorm given -> angles pooled with wgt[]
  int alpha;                // GLDM
  int Ng;                   // max gray level of the ROI (coefficients["Ng"])
  int n_roi_levels;         // number of distinct levels in the ROI (MCC: <2 -> 1)
  uint32_t alive[(NW_MAX + 31) / 32];  // GLCM: angles that are non-empty for at least one voxel
  double init_value;
  int8_t ang[NA_MAX][3];
  double wgt[NW_MAX];
};

// --------------------------------------------------------------------------------------------
// window + level compaction
template <typename T>
RB_HD void load_window(const T* __restrict__ lev, const VoxParams& P, int cz, int cy, int cx, uint16_t* w) {
  int k = 0;
  for (int dz = -P.rz; dz <= P.rz; dz++)
    for (int dy = -P.ry; dy <= P.ry; dy++)
      for (int dx = -P.rx; dx <= P.rx; dx++) {
        int z = cz + dz, y = cy + dy, x = cx + dx;
        bool in = z >= 0 && z < P.Z && y >= 0 && y < P.Y && x >= 0 && x < P.X;
        w[k++] = in ? (uint16_t)lev[(long long)z * P.sz + (long long)y * P.sy + x] : (uint16_t)0;
      }
}

struct WinGeom {
  int wz, wy, wx, n;
  RB_HD WinGeom(const VoxParams& P) : wz(2 * P.rz + 1), wy(2 * P.ry + 1), wx(2 * P.rx + 1) { n = wz * wy * wx; }
  RB_HD bool inside(int z, int y, int x) const { return z >= 0 && z < wz && y >= 0 && y < wy && x >= 0 && x < wx; }
  RB_HD int idx(int z, int y, int x) const { return (z * wy + y) * wx + x; }
};

// first-occurrence compaction: lidx[p] = local level index (NOLEV if unmasked), val[k] = level
template <int WCAP>
RB_HD int compact_levels(const uint16_t* w, int wn, int* val, uint16_t* lidx) {
  int n = 0;
  for (int p = 0; p < wn; p++) {
    int g = w[p];
    if (!g) { lidx[p] = NOLEV; continue; }
    int k = 0;
    for (; k < n; k++) if (val[k] == g) break;
    if (k == n) val[n++] = g;
    lidx[p] = (uint16_t)k;
  }
  return n;
}

// merged sparse entry list keyed by a 32-bit key
template <int CAP, typename W>
struct Entries {
  uint32_t key[CAP];
  W w[CAP];
  int n;
  bool overflow;
  RB_HD void clear() { n = 0; overflow = false; }
  RB_HD void add(uint32_t k, W v) {
    for (int e = 0; e < n; e++) if (key[e] == k) { w[e] += v; return; }
    if (n < CAP) { key[n] = k; w[n] = v; n++; } else overflow = true;
  }
};

RB_HD double xlog2(double p) { return p * log2(p + EPS); }

// --------------------------------------------------------------------------------------------
// Small dense symmetric eigenvalue machinery for MCC: Householder reduction to tridiagonal form
// followed by Sturm-sequence bisection for ONE eigenvalue by index (no eigenvectors, no sweeps
// to convergence: fixed trip counts, so a warp's lanes stay in step).
//
// Reduce the symmetric n x n matrix A (row-major, leading dimension ld, lower triangle used,
// destroyed) to tridiagonal: diagonal d[0..n-1], sub-diagonal e[1..n-1] (e[0] = 0).
static RB_HDN void sym_tridiagonalize(double* A, int n, int ld, double* d, double* e) {
  for (int i = n - 1; i >= 1; i--) {
    const int l = i - 1;
    double h = 0, scale = 0;
    if (l > 0) {
      for (int k = 0; k <= l; k++) scale += fabs(A[i * ld + k]);
      if (scale == 0) {
        e[i] = A[i * ld + l];
      } else {
        const double inv = 1.0 / scale;
        for (int k = 0; k <= l; k++) { A[i * ld + k] *= inv; h += A[i * ld + k] * A[i * ld + k]; }
        double f = A[i * ld + l];
        double g = f >= 0 ? -sqrt(h) : sqrt(h);
        e[i] = scale * g;
        h -= f * g;
        A[i * ld + l] = f - g;
        f = 0;
        for (int j = 0; j <= l; j++) {
          g = 0;
          for (int k = 0; k <= j; k++) g += A[j * ld + k] * A[i * ld + k];
          for (int k = j + 1; k <= l; k++) g += A[k * ld + j] * A[i * ld + k];
          e[j] = g / h;
          f += e[j] * A[i * ld + j];
        }
        const double hh = f / (h + h);
        for (int j = 0; j <= l; j++) {
          f = A[i * ld + j];
          e[j] = g = e[j] - hh * f;
          for (int k = 0; k <= j; k++) A[j * ld + k] -= f * e[k] + g * A[i * ld + k];
        }
      }
    } else {
      e[i] = A[i * ld + l];
    }
    d[i] = h;
  }
  e[0] = 0;
  for (int i = 0; i < n; i++) d[i] = A[i * ld + i];
}

// k-th smallest eigenvalue (k = 0..n-1) of the symmetric tridiagonal (d, e) inside [lo, hi],
// by bisection on the number of sign changes of the division-free Sturm sequence.
template <typename TD>
static RB_HDN double tridiag_kth_eigenvalue(const TD* d, const TD* e, int n, int k, double lo, double hi,
                                            int iters) {
  for (int it = 0; it < iters; it++) {
    const double x = 0.5 * (lo + hi);
    // p0 = 1, p1 = d0 - x, p_i = (d_i - x) p_{i-1} - e_i^2 p_{i-2}; #eigenvalues < x = sign changes
    double pm2 = 1.0, pm1 = d[0] - x;
    int cnt = pm1 <= 0;                      // a zero counts as an eigenvalue <= x
    for (int i = 1; i < n; i++) {
      const double e2 = (double)e[i] * (double)e[i];
      if (e2 == 0) {                         // decoupled block: restart the sequence
        pm2 = 1.0; pm1 = d[i] - x;
        cnt += pm1 <= 0;
        continue;
      }
      double p = (d[i] - x) * pm1 - e2 * pm2;
      const bool neg_prev = pm1 < 0 || (pm1 == 0 && pm2 > 0);
      const bool neg_cur = p < 0 || (p == 0 && !neg_prev);
      cnt += neg_cur != neg_prev;
      // rescale to stay far from over/underflow (signs are all that matter)
      const double m = fabs(p) > fabs(pm1) ? fabs(p) : fabs(pm1);
      if (m > 1e100 || (m < 1e-100 && m > 0)) { const double sc = 1.0 / m; p *= sc; pm1 *= sc; }
      pm2 = pm1; pm1 = p;
    }
    if (cnt > k) hi = x; else lo = x;
  }
  return 0.5 * (lo + hi);
}

// Extreme eigenvalue (largest if `top`, else smallest) of an UNREDUCED symmetric tridiagonal (d, e)
// by Laguerre's iteration on the characteristic polynomial p(x) = det(T - x I), started outside the
// spectrum at a Gershgorin bound: for a polynomial with only real roots it converges monotonically
// and cubically to the nearest (= extreme) root.  p, p', p'' come from the three-term recurrence.
// Falls back to Sturm bisection if it has not converged after 40 steps.
template <typename TD>
static RB_HDN double tridiag_extreme_eigenvalue(const TD* d, const TD* e, int n, bool top) {
  double lo = d[0], hi = d[0];
  for (int i = 0; i < n; i++) {
    const double r = (i > 0 ? fabs(e[i]) : 0.0) + (i + 1 < n ? fabs(e[i + 1]) : 0.0);
    lo = fmin(lo, d[i] - r); hi = fmax(hi, d[i] + r);
  }
  if (n == 1) return d[0];
  double x = top ? hi + 1e-9 : lo - 1e-9;
  for (int it = 0; it < 40; it++) {
    double p0 = 1.0, p1 = d[0] - x, q0 = 0.0, q1 = -1.0, r0 = 0.0, r1 = 0.0;   // p, p', p''
    for (int i = 1; i < n; i++) {
      const double a = d[i] - x, b = (double)e[i] * (double)e[i];
      const double p2 = a * p1 - b * p0;
      const double q2 = a * q1 - p1 - b * q0;
      const double r2 = a * r1 - 2.0 * q1 - b * r0;
      p0 = p1; p1 = p2; q0 = q1; q1 = q2; r0 = r1; r1 = r2;
    }
    if (p1 == 0) return x;
    const double G = q1 / p1, H = G * G - r1 / p1;
    const double disc = (double)(n - 1) * ((double)n * H - G * G);
    const double sq = sqrt(disc > 0 ? disc : 0.0);
    const double den = fabs(G + sq) > fabs(G - sq) ? G + sq : G - sq;
    if (den == 0 || den != den) break;
    const double step = (double)n / den;
    x -= step;
    if (fabs(step) < 1e-11) return x;
  }
  return tridiag_kth_eigenvalue(d, e, n, top ? n - 1 : 0, lo - 1e-9, hi + 1e-9, 40);
}

// Both extreme eigenvalues of an unreduced symmetric tridiagonal in one Laguerre loop (one pass over
// d, e per iteration serves both ends; lanes of a warp do not serialise "top" and "bottom" calls).
template <typename TD>
static RB_HDN void tridiag_extreme_pair(const TD* d, const TD* e, int n, double* hi_out, double* lo_out, int st = 1) {
  double lo = d[(0) * st], hi = d[(0) * st];
  for (int i = 0; i < n; i++) {
    const double r = (i > 0 ? fabs((double)e[(i) * st]) : 0.0) + (i + 1 < n ? fabs((double)e[(i + 1) * st]) : 0.0);
    lo = fmin(lo, d[(i) * st] - r); hi = fmax(hi, d[(i) * st] + r);
  }
  if (n == 1) { *hi_out = d[(0) * st]; *lo_out = d[(0) * st]; return; }
  double xh = hi + 1e-9, xl = lo - 1e-9;
  bool dh = false, dl = false;
  for (int it = 0; it < 40 && !(dh && dl); it++) {
    const double d0 = d[(0) * st];
    double hp0 = 1.0, hp1 = d0 - xh, hq0 = 0.0, hq1 = -1.0, hr0 = 0.0, hr1 = 0.0;
    double lp0 = 1.0, lp1 = d0 - xl, lq0 = 0.0, lq1 = -1.0, lr0 = 0.0, lr1 = 0.0;
    for (int i = 1; i < n; i++) {
      const double di = d[(i) * st], b = (double)e[(i) * st] * (double)e[(i) * st];
      {
        const double a = di - xh;
        const double p2 = a * hp1 - b * hp0, q2 = a * hq1 - hp1 - b * hq0, r2 = a * hr1 - 2.0 * hq1 - b * hr0;
        hp0 = hp1; hp1 = p2; hq0 = hq1; hq1 = q2; hr0 = hr1; hr1 = r2;
      }
      {
        const double a = di - xl;
        const double p2 = a * lp1 - b * lp0, q2 = a * lq1 - lp1 - b * lq0, r2 = a * lr1 - 2.0 * lq1 - b * lr0;
        lp0 = lp1; lp1 = p2; lq0 = lq1; lq1 = q2; lr0 = lr1; lr1 = r2;
      }
    }
    if (!dh) {
      if (hp1 == 0) dh = true;
      else {
        const double G = hq1 / hp1, H = G * G - hr1 / hp1;
        const double disc = (double)(n - 1) * ((double)n * H - G * G);
        const double sq = sqrt(disc > 0 ? disc : 0.0);
        const double den = fabs(G + sq) > fabs(G - sq) ? G + sq : G - sq;
        if (den == 0 || den != den) break;
        const double step = (double)n / den;
        xh -= step;
        if (fabs(step) < 1e-11) dh = true;
      }
    }
    if (!dl) {
      if (lp1 == 0) dl = true;
      else {
        const double G = lq1 / lp1, H = G * G - lr1 / lp1;
        const double disc = (double)(n - 1) * ((double)n * H - G * G);
        const double sq = sqrt(disc > 0 ? disc : 0.0);
        const double den = fabs(G + sq) > fabs(G - sq) ? G + sq : G - sq;
        if (den == 0 || den != den) break;
        const double step = (double)n / den;
        xl -= step;
        if (fabs(step) < 1e-11) dl = true;
      }
    }
  }
  if (dh && dl) { *hi_out = xh; *lo_out = xl; return; }
  double dc[24], ec[24];                       // rare: Sturm bisection on a contiguous copy
  for (int i = 0; i < n && i < 24; i++) { dc[i] = d[i * st]; ec[i] = e[i * st]; }
  *hi_out = dh ? xh : tridiag_kth_eigenvalue(dc, ec, n, n - 1, lo - 1e-9, hi + 1e-9, 40);
  *lo_out = dl ? xl : tridiag_kth_eigenvalue(dc, ec, n, 0, lo - 1e-9, hi + 1e-9, 40);
}

// Second-largest eigenvalue of a symmetric positive semi-definite matrix with spectrum in [0, 1+]
// (the generic MCC path: A = M M^T).  n >= 2.
static RB_HDN double sym_psd_second_largest(double* A, int n, int ld, double* d, double* e) {
  if (n == 2) {                        // closed form: the two roots of the characteristic quadratic
    const double tr = A[0] + A[ld + 1], det = A[0] * A[ld + 1] - A[ld] * A[ld];
    const double disc = sqrt(fmax(tr * tr - 4.0 * det, 0.0));
    return 0.5 * (tr - disc);
  }
  sym_tridiagonalize(A, n, ld, d, e);
  return tridiag_kth_eigenvalue(d, e, n, n - 2, -1e-6, 1.0 + 1e-6, 46);
}

// Second-largest |eigenvalue| of a symmetric matrix with spectrum in [-1, 1] (the fast MCC path,
// A = normalised co-occurrence D^-1/2 P D^-1/2 whose top eigenvalue is 1).  n >= 2.
static RB_HDN double sym_second_largest_abs(double* A, int n, int ld, double* d, double* e) {
  if (n == 2) return fabs(A[0] + A[ld + 1] - 1.0);     // eigenvalues are 1 and trace - 1
  sym_tridiagonalize(A, n, ld, d, e);
  const double top2 = tridiag_kth_eigenvalue(d, e, n, n - 2, -1.0 - 1e-6, 1.0 + 1e-6, 46);
  const double bot = tridiag_kth_eigenvalue(d, e, n, 0, -1.0 - 1e-6, 1.0 + 1e-6, 46);
  return fmax(fabs(top2), fabs(bot));
}

// --------------------------------------------------------------------------------------------
// GLCM: 24 features of ONE normalised matrix given as merged ordered entries (li<<16|lj, weight).
// Returns false if the matrix is empty (sum 0 -> the reference's NaN angle).
template <int ECAP, int NCAP, int NJCAP, typename W>
RB_HDN bool glcm_angle_features(const Entries<ECAP, W>& E, int n, const int* val, const VoxParams& P,
                                double* f, int* status) {
  double S = 0;
  for (int e = 0; e < E.n; e++) S += (double)E.w[e];
  if (S == 0) return false;
  double px[NCAP], py[NCAP];
  for (int k = 0; k < n; k++) { px[k] = 0; py[k] = 0; }
  double ux = 0, uy = 0;
  for (int e = 0; e < E.n; e++) {
    double p = (double)E.w[e] / S;
    int li = E.key[e] >> 16, lj = E.key[e] & 0xFFFF;
    px[li] += p; py[lj] += p;
    ux += p * val[li]; uy += p * val[lj];
  }
  // difference / sum histograms (merged by k)
  constexpr int KCAP = ECAP < 1024 ? ECAP : 1024;
  Entries<KCAP, double> D, Sm;
  D.clear(); Sm.clear();
  double ac = 0, cp = 0, cs = 0, ct = 0, con = 0, sxx = 0, syy = 0, sxy = 0, da = 0, idm = 0, idmn = 0,
         id = 0, idn = 0, inv = 0, ene = 0, maxp = 0, hxy = 0, hxy1 = 0, sa = 0;
  const double ng = (double)P.Ng;
  for (int e = 0; e < E.n; e++) {
    double p = (double)E.w[e] / S;
    int li = E.key[e] >> 16, lj = E.key[e] & 0xFFFF;
    double i = val[li], j = val[lj];
    ac += p * i * j;
    double d = (i + j) - ux - uy, d2 = d * d;
    ct += p * d2; cs += p * d2 * d; cp += p * d2 * d2;
    double k = fabs(i - j);
    con += p * k * k;
    double dx = i - ux, dy = j - uy;
    sxx += p * dx * dx; syy += p * dy * dy; sxy += p * dx * dy;
    da += p * k;
    idm += p / (1.0 + k * k);
    idmn += p / (1.0 + k * k / (ng * ng));
    id += p / (1.0 + k);
    idn += p / (1.0 + k / ng);
    if (k > 0) inv += p / (k * k);
    ene += p * p;
    if (p > maxp) maxp = p;
    hxy -= xlog2(p);
    hxy1 -= p * log2(px[li] * py[lj] + EPS);
    sa += p * (i + j);
    D.add((uint32_t)k, p);
    Sm.add((uint32_t)(i + j), p);
  }
  if ((D.overflow || Sm.overflow) && status) *status |= 2;
  double dvar = 0, dent = 0, sent = 0;
  for (int e = 0; e < D.n; e++) { double k = (double)D.key[e]; dvar += D.w[e] * (k - da) * (k - da); dent -= xlog2(D.w[e]); }
  for (int e = 0; e < Sm.n; e++) sent -= xlog2(Sm.w[e]);
  double hx = 0, hy = 0, hx0 = 0, hy0 = 0; int nx = 0, ny = 0;
  for (int k = 0; k < n; k++) {
    if (px[k] > 0) { hx -= xlog2(px[k]); hx0 -= px[k] * log2(px[k]); nx++; }
    if (py[k] > 0) { hy -= xlog2(py[k]); hy0 -= py[k] * log2(py[k]); ny++; }
  }
  // HXY2 = -sum_ij px_i py_j log2(px_i py_j + eps); expanded to first order in eps (exact to
  // O(eps^2/(px py))): = HX0 + HY0 - nx*ny*eps/ln2
  double hxy2 = hx0 + hy0 - (double)nx * (double)ny * EPS * 1.4426950408889634;
  f[G_Autocorrelation] = ac;
  f[G_JointAverage] = ux;
  f[G_ClusterProminence] = cp; f[G_ClusterShade] = cs; f[G_ClusterTendency] = ct;
  f[G_Contrast] = con;
  {
    double sx = sqrt(sxx), sy = sqrt(syy);
    f[G_Correlation] = (sx * sy == 0) ? 1.0 : sxy / (sx * sy + EPS);
  }
  f[G_DifferenceAverage] = da; f[G_DifferenceEntropy] = dent; f[G_DifferenceVariance] = dvar;
  f[G_JointEnergy] = ene; f[G_JointEntropy] = hxy;
  {
    double div = hx > hy ? hx : hy;
    f[G_Imc1] = (div != 0) ? (hxy - hxy1) / div : 0.0;
    double arg = 1.0 - exp(-2.0 * (hxy2 - hxy));
    f[G_Imc2] = (hxy2 == hxy) ? 0.0 : sqrt(arg);  // arg<0 -> NaN, dropped by the nanmean as in numpy
  }
  f[G_Idm] = idm; f[G_Idmn] = idmn; f[G_Id] = id; f[G_Idn] = idn; f[G_InverseVariance] = inv;
  f[G_MaximumProbability] = maxp; f[G_SumAverage] = sa; f[G_SumEntropy] = sent; f[G_SumSquares] = sxx;

  // ---- MCC = sqrt(2nd largest eigenvalue of Q), Q = Dx^-1 P Dy^-1 P^T (glcm.py:679-707).
  // Q is similar to M M^T with M = P / sqrt(px py + eps): eigenvalues are the squared singular
  // values of M; every connected component of the bipartite (row level, column level) graph
  // contributes one singular value 1, so >=2 components -> lambda2 = 1 without an eigen-solve.
  if (P.n_roi_levels < 2) { f[G_MCC] = 1.0; return true; }
  uint16_t ridx[NCAP], cidx[NCAP];
  int nr = 0, nc = 0;
  for (int k = 0; k < n; k++) { ridx[k] = px[k] > 0 ? (uint16_t)nr++ : NOLEV; cidx[k] = py[k] > 0 ? (uint16_t)nc++ : NOLEV; }
  if (nr < 2) { f[G_MCC] = 0.0; return true; }  // eigenvalues {1,0,...}: second largest is 0
  {
    uint16_t parent[2 * NCAP];
    for (int k = 0; k < nr + nc; k++) parent[k] = (uint16_t)k;
    for (int e = 0; e < E.n; e++) {
      int a = ridx[E.key[e] >> 16], b = nr + cidx[E.key[e] & 0xFFFF];
      while (parent[a] != a) a = parent[a];
      while (parent[b] != b) b = parent[b];
      if (a != b) parent[a > b ? a : b] = (uint16_t)(a > b ? b : a);
    }
    int comps = 0;
    for (int k = 0; k < nr + nc; k++) if (parent[k] == k) comps++;
    if (comps >= 2) { f[G_MCC] = 1.0; return true; }
  }
  if (nr > NJCAP) { f[G_MCC] = NAN; if (status) *status |= 1; return true; }
  double A[NJCAP * NJCAP];
  for (int k = 0; k < nr * nr; k++) A[k] = 0;
  for (int e1 = 0; e1 < E.n; e1++) {
    int l1 = E.key[e1] >> 16, c1 = E.key[e1] & 0xFFFF;
    double m1 = ((double)E.w[e1] / S) / sqrt(px[l1] * py[c1] + EPS);
    for (int e2 = 0; e2 < E.n; e2++) {
      if ((int)(E.key[e2] & 0xFFFF) != c1) continue;
      int l2 = E.key[e2] >> 16;
      double m2 = ((double)E.w[e2] / S) / sqrt(px[l2] * py[c1] + EPS);
      A[ridx[l1] * nr + ridx[l2]] += m1 * m2;
    }
  }
  double dd[NJCAP], ee[NJCAP];
  const double l2 = sym_psd_second_largest(A, nr, nr, dd, ee);
  f[G_MCC] = sqrt(l2 > 0 ? l2 : 0.0);
  return true;
}

// all 24 GLCM feature values of one centre voxel
template <int WCAP, bool WEIGHTED>
RB_HD void glcm_voxel(const uint16_t* w, const VoxParams& P, double* out, int* status) {
  constexpr int NJCAP = WCAP < 32 ? WCAP : 32;
  constexpr int ECAP = WEIGHTED ? (WCAP <= 27 ? WCAP * WCAP : 2048) : 2 * WCAP;
  const WinGeom G(P);
  int val[WCAP]; uint16_t lidx[WCAP];
  const int n = compact_levels<WCAP>(w, G.n, val, lidx);
  double f[GLCM_NF];
  if (WEIGHTED) {
    Entries<ECAP, double> E; E.clear();
    for (int a = 0; a < P.na; a++) {
      const int az = P.ang[a][0], ay = P.ang[a][1], ax = P.ang[a][2];
      for (int z = 0; z < G.wz; z++) for (int y = 0; y < G.wy; y++) for (int x = 0; x < G.wx; x++) {
        if (!G.inside(z + az, y + ay, x + ax)) continue;
        uint16_t li = lidx[G.idx(z, y, x)], lj = lidx[G.idx(z + az, y + ay, x + ax)];
        if (li == NOLEV || lj == NOLEV) continue;
        E.add(((uint32_t)li << 16) | lj, P.wgt[a]);
        if (P.symmetric) E.add(((uint32_t)lj << 16) | li, P.wgt[a]);
      }
    }
    bool ok = glcm_angle_features<ECAP, WCAP, NJCAP, double>(E, n, val, P, f, status);
    if (E.overflow) { ok = false; if (status) *status |= 2; }
    for (int k = 0; k < GLCM_NF; k++) out[k] = ok ? f[k] : NAN;
    if (P.n_roi_levels < 2) out[G_MCC] = 1.0;    // flat ROI: 1 for every centre, with or without pairs (glcm.py:702)
    return;
  }
  double sum[GLCM_NF]; int cnt[GLCM_NF];
  for (int k = 0; k < GLCM_NF; k++) { sum[k] = 0; cnt[k] = 0; }
  bool ja_nan = false;
  for (int a = 0; a < P.na; a++) {
    const int az = P.ang[a][0], ay = P.ang[a][1], ax = P.ang[a][2];
    Entries<ECAP, int> E; E.clear();
    for (int z = 0; z < G.wz; z++) for (int y = 0; y < G.wy; y++) for (int x = 0; x < G.wx; x++) {
      if (!G.inside(z + az, y + ay, x + ax)) continue;
      uint16_t li = lidx[G.idx(z, y, x)], lj = lidx[G.idx(z + az, y + ay, x + ax)];
      if (li == NOLEV || lj == NOLEV) continue;
      E.add(((uint32_t)li << 16) | lj, 1);
      if (P.symmetric) E.add(((uint32_t)lj << 16) | li, 1);
    }
    bool ok = glcm_angle_features<ECAP, WCAP, NJCAP, int>(E, n, val, P, f, status);
    if (!ok) { if (P.alive[a >> 5] >> (a & 31) & 1u) ja_nan = true; continue; }
    for (int k = 0; k < GLCM_NF; k++) if (f[k] == f[k]) { sum[k] += f[k]; cnt[k]++; }
  }
  for (int k = 0; k < GLCM_NF; k++) out[k] = cnt[k] ? sum[k] / cnt[k] : NAN;
  // JointAverage is a plain mean over the kept angles (glcm.py:292): NaN propagates
  if (ja_nan) out[G_JointAverage] = NAN;
  if (P.n_roi_levels < 2) out[G_MCC] = 1.0;
}

// --------------------------------------------------------------------------------------------
// GLRLM
template <int ECAP, int NCAP, typename W>
RB_HDN bool glrlm_angle_features(const Entries<ECAP, W>& E, int n, const int* val, double* f) {
  constexpr int RLCAP = 8;
  double Nr = 0;
  for (int e = 0; e < E.n; e++) Nr += (double)E.w[e];
  if (Nr == 0) return false;
  double pr[RLCAP], pg[NCAP];
  for (int k = 0; k < RLCAP; k++) pr[k] = 0;
  for (int k = 0; k < n; k++) pg[k] = 0;
  double re = 0, srlgle = 0, srhgle = 0, lrlgle = 0, lrhgle = 0;
  for (int e = 0; e < E.n; e++) {
    double c = (double)E.w[e];
    int li = E.key[e] >> 16, len = (E.key[e] & 0xFFFF) + 1;
    pr[len - 1] += c; pg[li] += c;
    re -= xlog2(c / Nr);
    double i2 = (double)val[li] * val[li], j2 = (double)len * len;
    srlgle += c / (i2 * j2); srhgle += c * i2 / j2; lrlgle += c * j2 / i2; lrhgle += c * i2 * j2;
  }
  double sre = 0, lre = 0, rln = 0, np_ = 0, ur = 0;
  for (int k = 0; k < RLCAP; k++) {
    double j = k + 1;
    sre += pr[k] / (j * j); lre += pr[k] * j * j; rln += pr[k] * pr[k]; np_ += pr[k] * j; ur += pr[k] / Nr * j;
  }
  double rv = 0;
  for (int k = 0; k < RLCAP; k++) { double j = k + 1; rv += pr[k] / Nr * (j - ur) * (j - ur); }
  double gln = 0, ug = 0, lgl = 0, hgl = 0;
  for (int k = 0; k < n; k++) {
    double i = val[k];
    gln += pg[k] * pg[k]; ug += pg[k] / Nr * i; lgl += pg[k] / (i * i); hgl += pg[k] * i * i;
  }
  double glv = 0;
  for (int k = 0; k < n; k++) { double i = val[k]; glv += pg[k] / Nr * (i - ug) * (i - ug); }
  f[R_ShortRunEmphasis] = sre / Nr; f[R_LongRunEmphasis] = lre / Nr;
  f[R_GrayLevelNonUniformity] = gln / Nr; f[R_GrayLevelNonUniformityNormalized] = gln / (Nr * Nr);
  f[R_RunLengthNonUniformity] = rln / Nr; f[R_RunLengthNonUniformityNormalized] = rln / (Nr * Nr);
  f[R_RunPercentage] = Nr / np_;
  f[R_GrayLevelVariance] = glv; f[R_RunVariance] = rv; f[R_RunEntropy] = re;
  f[R_LowGrayLevelRunEmphasis] = lgl / Nr; f[R_HighGrayLevelRunEmphasis] = hgl / Nr;
  f[R_ShortRunLowGrayLevelEmphasis] = srlgle / Nr; f[R_ShortRunHighGrayLevelEmphasis] = srhgle / Nr;
  f[R_LongRunLowGrayLevelEmphasis] = lrlgle / Nr; f[R_LongRunHighGrayLevelEmphasis] = lrhgle / Nr;
  return true;
}

template <int WCAP, bool WEIGHTED>
RB_HD void glrlm_voxel(const uint16_t* w, const VoxParams& P, double* out) {
  const WinGeom G(P);
  int val[WCAP]; uint16_t lidx[WCAP];
  const int n = compact_levels<WCAP>(w, G.n, val, lidx);
  double f[GLRLM_NF], sum[GLRLM_NF]; int cnt[GLRLM_NF];
  for (int k = 0; k < GLRLM_NF; k++) { sum[k] = 0; cnt[k] = 0; }
  Entries<WCAP, double> EW; EW.clear();
  for (int a = 0; a < P.na; a++) {
    const int az = P.ang[a][0], ay = P.ang[a][1], ax = P.ang[a][2];
    Entries<WCAP, int> E; E.clear();
    bool multi = false;
    for (int z = 0; z < G.wz; z++) for (int y = 0; y < G.wy; y++) for (int x = 0; x < G.wx; x++) {
      if (G.inside(z - az, y - ay, x - ax)) continue;  // not a line start
      int cz = z, cy = y, cx = x, gl = -1, rl = 0, elements = 0;
      while (G.inside(cz, cy, cx)) {
        uint16_t l = lidx[G.idx(cz, cy, cx)];
        if (l != NOLEV) {
          elements++;
          if (gl < 0) { gl = l; rl = 0; }
          else if (l == gl) rl++;
          else { E.add(((uint32_t)gl << 16) | (uint32_t)rl, 1); gl = l; rl = 0; }
        } else if (gl >= 0) { E.add(((uint32_t)gl << 16) | (uint32_t)rl, 1); gl = -1; rl = 0; }
        cz += az; cy += ay; cx += ax;
      }
      if (gl >= 0) E.add(((uint32_t)gl << 16) | (uint32_t)rl, 1);
      if (elements > 1) multi = true;
    }
    if (!multi) continue;  // cmatrices.c:524-534: the angle's (only) run-length-1 column is zeroed
    if (WEIGHTED) {
      for (int e = 0; e < E.n; e++) EW.add(E.key[e], P.wgt[a] * E.w[e]);
    } else {
      if (!glrlm_angle_features<WCAP, WCAP, int>(E, n, val, f)) continue;
      for (int k = 0; k < GLRLM_NF; k++) if (f[k] == f[k]) { sum[k] += f[k]; cnt[k]++; }
    }
  }
  if (WEIGHTED) {
    bool ok = glrlm_angle_features<WCAP, WCAP, double>(EW, n, val, f);
    for (int k = 0; k < GLRLM_NF; k++) out[k] = ok ? f[k] : NAN;
  } else {
    for (int k = 0; k < GLRLM_NF; k++) out[k] = cnt[k] ? sum[k] / cnt[k] : NAN;
  }
}

// --------------------------------------------------------------------------------------------
// "level x size" feature block shared by GLSZM (size = zone size) and GLDM (size = dep + 1)
template <int ECAP, int NCAP, int JCAP>
RB_HDN void size_matrix_features(const Entries<ECAP, int>& E, int n, const int* val, double* f) {
  double Nz = 0;
  for (int e = 0; e < E.n; e++) Nz += E.w[e];
  double NzDiv = Nz == 0 ? 1.0 : Nz;
  double pj[JCAP + 1], pg[NCAP];
  int jmax = 0;
  for (int k = 0; k <= JCAP; k++) pj[k] = 0;
  for (int k = 0; k < n; k++) pg[k] = 0;
  double ent = 0, sl = 0, sh = 0, ll = 0, lh = 0;
  for (int e = 0; e < E.n; e++) {
    double c = E.w[e];
    int li = E.key[e] >> 16, j = E.key[e] & 0xFFFF;
    pj[j] += c; pg[li] += c; if (j > jmax) jmax = j;
    ent -= xlog2(c / NzDiv);
    double i2 = (double)val[li] * val[li], j2 = (double)j * j;
    sl += c / (i2 * j2); sh += c * i2 / j2; ll += c * j2 / i2; lh += c * i2 * j2;
  }
  double se = 0, le = 0, snu = 0, np_ = 0, uj = 0;
  for (int j = 1; j <= jmax; j++) {
    double jj = j;
    se += pj[j] / (jj * jj); le += pj[j] * jj * jj; snu += pj[j] * pj[j]; np_ += pj[j] * jj; uj += pj[j] / NzDiv * jj;
  }
  double sv = 0;
  for (int j = 1; j <= jmax; j++) sv += pj[j] / NzDiv * (j - uj) * (j - uj);
  double gln = 0, ug = 0, lgl = 0, hgl = 0;
  for (int k = 0; k < n; k++) { double i = val[k]; gln += pg[k] * pg[k]; ug += pg[k] / NzDiv * i; lgl += pg[k] / (i * i); hgl += pg[k] * i * i; }
  double glv = 0;
  for (int k = 0; k < n; k++) { double i = val[k]; glv += pg[k] / NzDiv * (i - ug) * (i - ug); }
  f[S_GLN] = gln / NzDiv; f[S_GLNN] = gln / (NzDiv * NzDiv); f[S_GLV] = glv; f[S_HGLE] = hgl / NzDiv;
  f[S_LargeE] = le / NzDiv; f[S_LargeHGLE] = lh / NzDiv; f[S_LargeLGLE] = ll / NzDiv; f[S_LGLE] = lgl / NzDiv;
  f[S_SizeNU] = snu / NzDiv; f[S_SizeNUN] = snu / (NzDiv * NzDiv); f[S_SmallE] = se / NzDiv;
  f[S_SmallHGLE] = sh / NzDiv; f[S_SmallLGLE] = sl / NzDiv; f[S_Entropy] = ent;
  f[S_Percentage] = NzDiv / (np_ == 0 ? 1.0 : np_); f[S_SizeVar] = sv;
}

template <int WCAP>
RB_HD void glszm_voxel(const uint16_t* w, const VoxParams& P, double* out) {
  const WinGeom G(P);
  int val[WCAP]; uint16_t lidx[WCAP];
  const int n = compact_levels<WCAP>(w, G.n, val, lidx);
  Entries<WCAP, int> E; E.clear();
  uint16_t stack[WCAP];
  for (int s = 0; s < G.n; s++) {
    uint16_t gl = lidx[s];
    if (gl == NOLEV) continue;
    int top = 0, region = 0;
    stack[top++] = (uint16_t)s; lidx[s] = NOLEV;
    while (top) {
      int k = stack[--top];
      region++;
      int kz = k / (G.wy * G.wx), ky = (k / G.wx) % G.wy, kx = k % G.wx;
      for (int a = 0; a < P.na; a++) {
        int z = kz + P.ang[a][0], y = ky + P.ang[a][1], x = kx + P.ang[a][2];
        if (!G.inside(z, y, x)) continue;
        int j = G.idx(z, y, x);
        if (lidx[j] == gl) { stack[top++] = (uint16_t)j; lidx[j] = NOLEV; }
      }
    }
    E.add(((uint32_t)gl << 16) | (uint32_t)region, 1);
  }
  double f[SIZE_NF];
  size_matrix_features<WCAP, WCAP, WCAP>(E, n, val, f);
  for (int k = 0; k < GLSZM_NF; k++) out[k] = f[k];
}

// GLDM feature order (alphabetical) in terms of the generic block
RB_HD void gldm_from_size(const double* f, double* out) {
  out[0] = f[S_Entropy]; out[1] = f[S_SizeNU]; out[2] = f[S_SizeNUN]; out[3] = f[S_SizeVar];
  out[4] = f[S_GLN]; out[5] = f[S_GLV]; out[6] = f[S_HGLE]; out[7] = f[S_LargeE];
  out[8] = f[S_LargeHGLE]; out[9] = f[S_LargeLGLE]; out[10] = f[S_LGLE]; out[11] = f[S_SmallE];
  out[12] = f[S_SmallHGLE]; out[13] = f[S_SmallLGLE];
}

template <int WCAP>
RB_HD void gldm_voxel(const uint16_t* w, const VoxParams& P, double* out) {
  const WinGeom G(P);
  int val[WCAP]; uint16_t lidx[WCAP];
  const int n = compact_levels<WCAP>(w, G.n, val, lidx);
  Entries<WCAP, int> E; E.clear();
  for (int z = 0; z < G.wz; z++) for (int y = 0; y < G.wy; y++) for (int x = 0; x < G.wx; x++) {
    uint16_t li = lidx[G.idx(z, y, x)];
    if (li == NOLEV) continue;
    int dep = 0;
    for (int a = 0; a < P.na; a++) {
      int z2 = z + P.ang[a][0], y2 = y + P.ang[a][1], x2 = x + P.ang[a][2];
      if (!G.inside(z2, y2, x2)) continue;
      uint16_t lj = lidx[G.idx(z2, y2, x2)];
      if (lj == NOLEV) continue;
      int d = val[li] - val[lj];
      if (d < 0) d = -d;
      if (d <= P.alpha) dep++;
    }
    E.add(((uint32_t)li << 16) | (uint32_t)(dep + 1), 1);
  }
  double f[SIZE_NF];
  size_matrix_features<WCAP, WCAP, NA_MAX + 1>(E, n, val, f);
  gldm_from_size(f, out);
}

// --------------------------------------------------------------------------------------------
// A product rounded on its own, never contracted into a following subtraction: where numpy's i*p_i - j*p_j is exactly 0
// (equal products) a fused multiply-add leaves the rounding error of one product, and a zero denominator becomes ~1e-17.
RB_HD double mul_rn(double a, double b) {
#ifdef __CUDA_ARCH__
  return __dmul_rn(a, b);
#else
  return a * b;
#endif
}

template <int WCAP>
RB_HD void ngtdm_voxel(const uint16_t* w, const VoxParams& P, double* out) {
  const WinGeom G(P);
  int val[WCAP]; uint16_t lidx[WCAP];
  const int n = compact_levels<WCAP>(w, G.n, val, lidx);
  double cnt[WCAP], s[WCAP];
  for (int k = 0; k < n; k++) { cnt[k] = 0; s[k] = 0; }
  for (int z = 0; z < G.wz; z++) for (int y = 0; y < G.wy; y++) for (int x = 0; x < G.wx; x++) {
    uint16_t li = lidx[G.idx(z, y, x)];
    if (li == NOLEV) continue;
    double c = 0, sum = 0;
    for (int a = 0; a < P.na; a++) {
      int z2 = z + P.ang[a][0], y2 = y + P.ang[a][1], x2 = x + P.ang[a][2];
      if (!G.inside(z2, y2, x2)) continue;
      uint16_t lj = lidx[G.idx(z2, y2, x2)];
      if (lj == NOLEV) continue;
      c += 1; sum += val[lj];
    }
    double diff = c == 0 ? 0.0 : (double)val[li] - sum / c;
    cnt[li] += 1; s[li] += fabs(diff);
  }
  double Nvp = 0, ssum = 0;
  for (int k = 0; k < n; k++) { Nvp += cnt[k]; ssum += s[k]; }
  // every level of the window has n_i > 0, so Ngp == n and the reference's p_zero masks are no-ops
  double ps = 0, con = 0, busy_den = 0, cpx = 0, str = 0;
  for (int a = 0; a < n; a++) {
    double pa = cnt[a] / Nvp, ia = val[a];
    ps += pa * s[a];
    for (int b = 0; b < n; b++) {
      double pb = cnt[b] / Nvp, ib = val[b], d = ia - ib;
      con += pa * pb * d * d;
      busy_den += fabs(mul_rn(ia, pa) - mul_rn(ib, pb));
      cpx += fabs(d) * (pa * s[a] + pb * s[b]) / (pa + pb);
      str += (pa + pb) * d * d;
    }
  }
  double div = (double)n * (n - 1);
  out[N_Coarseness] = ps != 0 ? 1.0 / ps : 1e6;
  out[N_Contrast] = div != 0 ? con * ssum / Nvp / div : 0.0;
  out[N_Busyness] = busy_den != 0 ? ps / busy_den : 0.0;
  out[N_Complexity] = cpx / Nvp;
  out[N_Strength] = ssum != 0 ? str / ssum : 0.0;
}

}  // namespace rb
