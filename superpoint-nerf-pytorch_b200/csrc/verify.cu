// spn_verify_pairs (include/spn_verify.h): RANSAC for a fundamental matrix (7-point) or a homography (4-point) per
// image pair, over the compacted matches of spn_match_pairs.
//
//   verify_kernel<MODEL>   one 256-thread CTA per pair.  The pair's match coordinates are staged in shared memory as
//                          int16 (8 bytes a match, 128 KB at cap = 16384) next to a byte mask.  Each round draws 256
//                          hypotheses, one per thread: sample, solve in registers (Householder QR), score every match
//                          in match order.  The round's best is found with a shuffle / shared-memory argmax on (count,
//                          hypothesis), so no atomics; refinement sums the normal matrix with one thread per entry in
//                          match order and takes the smallest eigenvector with a fixed-sweep Jacobi on one thread.
#include <math.h>

#include "spn_common.cuh"
#include "../../include/spn_verify.h"

namespace {

constexpr int kT = 256;   // threads per CTA = hypotheses per round
constexpr int kMaxN = 1 << 20, kMaxCap = 16384, kMaxPairs = 65535, kMaxIters = 1 << 24, kMaxDraws = 1024;
constexpr int kMaxRefits = 3, kJacobiSweeps = 12;
constexpr double kPivotTol = 1e-9, kLeadTol = 1e-12, kH22Tol = 1e-12;

struct VerifyParams {
  const int* kp;            // [N][cap][2] (row, col)
  const int* pairs;         // [P][2] (a, b), uploaded
  const long long* offsets; // [P+1]
  const int* matches;       // [M][2]
  long long M;
  int cap;
  double t2, log1mc;        // t^2, log(1 - confidence)
  int max_hyp;              // max_iters rounded up to a whole round
  unsigned long long seed;
  double* model;
  int* num;
  int* hyp;
  int* best;
  uint8_t* inlier;
};

struct Norm {   // x_hat = s (x - c), per image of the pair
  double sa, cxa, cya, sb, cxb, cyb;
};

// ---------------------------------------------------------------------------------------------------- inlier tests
__device__ __forceinline__ bool inlier_f(const double* F, double xa, double ya, double xb, double yb, double t2) {
  const double l0 = F[0] * xa + F[1] * ya + F[2], l1 = F[3] * xa + F[4] * ya + F[5], l2 = F[6] * xa + F[7] * ya + F[8];
  const double m0 = F[0] * xb + F[3] * yb + F[6], m1 = F[1] * xb + F[4] * yb + F[7];
  const double e = xb * l0 + yb * l1 + l2;
  return e * e <= t2 * (l0 * l0 + l1 * l1 + m0 * m0 + m1 * m1);
}

__device__ __forceinline__ bool inlier_h(const double* H, double xa, double ya, double xb, double yb, double t2) {
  const double p0 = H[0] * xa + H[1] * ya + H[2], p1 = H[3] * xa + H[4] * ya + H[5], p2 = H[6] * xa + H[7] * ya + H[8];
  const double u = p0 - xb * p2, v = p1 - yb * p2;
  return u * u + v * v <= t2 * (p2 * p2);
}

template <int MODEL>
__device__ __forceinline__ bool is_inlier(const double* m, short4 c, double t2) {
  return MODEL == 0 ? inlier_f(m, c.x, c.y, c.z, c.w, t2) : inlier_h(m, c.x, c.y, c.z, c.w, t2);
}

// ---------------------------------------------------------------------------------------------------- reductions
__device__ double block_sum(double v, double* red) {
#pragma unroll
  for (int off = 16; off; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = 0.0;
#pragma unroll
  for (int w = 0; w < kT / 32; ++w) s += red[w];
  __syncthreads();
  return s;
}

__device__ unsigned long long block_max(unsigned long long v, unsigned long long* red) {
#pragma unroll
  for (int off = 16; off; off >>= 1) {
    const unsigned long long o = __shfl_xor_sync(0xffffffffu, v, off);
    v = o > v ? o : v;
  }
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  unsigned long long m = red[0];
#pragma unroll
  for (int w = 1; w < kT / 32; ++w) m = red[w] > m ? red[w] : m;
  __syncthreads();
  return m;
}

// ---------------------------------------------------------------------------------------------------- sampler
__device__ __forceinline__ bool draw_sample(unsigned long long key, int h, int n, int s, int* idx) {
  int got = 0;
  for (int j = 0; j < kMaxDraws && got < s; ++j) {
    const unsigned long long r = splitmix64(key ^ splitmix64(((unsigned long long)(unsigned)h << 32) | (unsigned)j));
    const int k = (int)(((r >> 32) * (unsigned long long)n) >> 32);
    bool dup = false;
#pragma unroll
    for (int u = 0; u < 7; ++u) dup |= u < got && idx[u] == k;
    if (dup) continue;
#pragma unroll
    for (int u = 0; u < 7; ++u)
      if (u == got) idx[u] = k;
    ++got;
  }
  return got == s;
}

// ---------------------------------------------------------------------------------------------------- denormalise
// F = T_b^T F_hat T_a
__device__ void denorm_f(const double* f, const Norm& T, double* F) {
  double g[9];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    g[3 * i] = T.sa * f[3 * i];
    g[3 * i + 1] = T.sa * f[3 * i + 1];
    g[3 * i + 2] = f[3 * i + 2] - T.sa * T.cxa * f[3 * i] - T.sa * T.cya * f[3 * i + 1];
  }
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    F[j] = T.sb * g[j];
    F[3 + j] = T.sb * g[3 + j];
    F[6 + j] = g[6 + j] - T.sb * T.cxb * g[j] - T.sb * T.cyb * g[3 + j];
  }
}

// H = T_b^-1 H_hat T_a, scaled to H[2][2] = 1; false when |H[2][2]| is negligible
__device__ bool denorm_h(const double* h, const Norm& T, double* H) {
  double g[9];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    g[3 * i] = T.sa * h[3 * i];
    g[3 * i + 1] = T.sa * h[3 * i + 1];
    g[3 * i + 2] = h[3 * i + 2] - T.sa * T.cxa * h[3 * i] - T.sa * T.cya * h[3 * i + 1];
  }
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    H[j] = g[j] / T.sb + T.cxb * g[6 + j];
    H[3 + j] = g[3 + j] / T.sb + T.cyb * g[6 + j];
    H[6 + j] = g[6 + j];
  }
  double mx = 0.0;
#pragma unroll
  for (int k = 0; k < 9; ++k) mx = fmax(mx, fabs(H[k]));
  if (!(fabs(H[8]) >= kH22Tol * mx) || H[8] == 0.0) return false;
  const double d = H[8];
#pragma unroll
  for (int k = 0; k < 9; ++k) H[k] /= d;
  return isfinite(H[0] + H[1] + H[2] + H[3] + H[4] + H[5] + H[6] + H[7]);
}

// ---------------------------------------------------------------------------------------------------- 7-point F
__device__ __forceinline__ void cofactors(const double* A, double* c) {
  c[0] = A[4] * A[8] - A[5] * A[7]; c[1] = A[5] * A[6] - A[3] * A[8]; c[2] = A[3] * A[7] - A[4] * A[6];
  c[3] = A[2] * A[7] - A[1] * A[8]; c[4] = A[0] * A[8] - A[2] * A[6]; c[5] = A[1] * A[6] - A[0] * A[7];
  c[6] = A[1] * A[5] - A[2] * A[4]; c[7] = A[2] * A[3] - A[0] * A[5]; c[8] = A[0] * A[4] - A[1] * A[3];
}

// Real roots of c3 x^3 + c2 x^2 + c1 x + c0, ascending -> count (0 when the cubic degenerates)
__device__ int cubic_roots(double c3, double c2, double c1, double c0, double* x) {
  const double mx = fmax(fmax(fabs(c0), fabs(c1)), fmax(fabs(c2), fabs(c3)));
  if (!(fabs(c3) > kLeadTol * mx)) return 0;
  const double b = c2 / c3, c = c1 / c3, d = c0 / c3;
  const double Q = (b * b - 3.0 * c) / 9.0, R = (2.0 * b * b * b - 9.0 * b * c + 27.0 * d) / 54.0;
  const double Q3 = Q * Q * Q;
  int nr;
  if (R * R < Q3) {
    const double th = acos(R / sqrt(Q3)), sq = -2.0 * sqrt(Q), tp = 6.283185307179586;
    x[0] = sq * cos(th / 3.0) - b / 3.0;
    x[1] = sq * cos((th + tp) / 3.0) - b / 3.0;
    x[2] = sq * cos((th - tp) / 3.0) - b / 3.0;
    nr = 3;
  } else {
    const double A = -copysign(cbrt(fabs(R) + sqrt(R * R - Q3)), R);
    const double B = A != 0.0 ? Q / A : 0.0;
    x[0] = A + B - b / 3.0;
    x[1] = x[2] = 0.0;
    nr = 1;
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    if (k >= nr) break;
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const double v = ((c3 * x[k] + c2) * x[k] + c1) * x[k] + c0, dv = (3.0 * c3 * x[k] + 2.0 * c2) * x[k] + c1;
      if (dv != 0.0) x[k] -= v / dv;
    }
  }
  if (nr == 3) {   // sort the three roots ascending
    double t;
    if (x[1] < x[0]) { t = x[0]; x[0] = x[1]; x[1] = t; }
    if (x[2] < x[1]) { t = x[1]; x[1] = x[2]; x[2] = t; }
    if (x[1] < x[0]) { t = x[0]; x[0] = x[1]; x[1] = t; }
  }
  return nr;
}

__device__ int solve7(const short4* pts, const int* idx, const Norm& T, double (&m)[3][9]) {
  double A[9][7];   // column j: the epipolar constraint of sample point j
#pragma unroll
  for (int j = 0; j < 7; ++j) {
    const short4 c = pts[idx[j]];
    const double xa = T.sa * (c.x - T.cxa), ya = T.sa * (c.y - T.cya), xb = T.sb * (c.z - T.cxb), yb = T.sb * (c.w - T.cyb);
    A[0][j] = xb * xa; A[1][j] = xb * ya; A[2][j] = xb;
    A[3][j] = yb * xa; A[4][j] = yb * ya; A[5][j] = yb;
    A[6][j] = xa;      A[7][j] = ya;      A[8][j] = 1.0;
  }
  double beta[7];
#pragma unroll
  for (int k = 0; k < 7; ++k) {   // Householder QR of A (9 x 7); v_k overwrites A[k..8][k]
    double nrm = 0.0;
#pragma unroll
    for (int r = k; r < 9; ++r) nrm += A[r][k] * A[r][k];
    nrm = sqrt(nrm);
    if (!(nrm > kPivotTol)) return 0;
    const double alpha = A[k][k] >= 0.0 ? -nrm : nrm;
    A[k][k] -= alpha;
    double vv = 0.0;
#pragma unroll
    for (int r = k; r < 9; ++r) vv += A[r][k] * A[r][k];
    beta[k] = 2.0 / vv;
#pragma unroll
    for (int j = k + 1; j < 7; ++j) {
      double dot = 0.0;
#pragma unroll
      for (int r = k; r < 9; ++r) dot += A[r][k] * A[r][j];
      dot *= beta[k];
#pragma unroll
      for (int r = k; r < 9; ++r) A[r][j] -= dot * A[r][k];
    }
  }
  double f1[9], f2[9];   // Q e_7 and Q e_8: the null space of the 7 x 9 system
#pragma unroll
  for (int r = 0; r < 9; ++r) { f1[r] = r == 7 ? 1.0 : 0.0; f2[r] = r == 8 ? 1.0 : 0.0; }
#pragma unroll
  for (int k = 6; k >= 0; --k) {
    double d1 = 0.0, d2 = 0.0;
#pragma unroll
    for (int r = k; r < 9; ++r) { d1 += A[r][k] * f1[r]; d2 += A[r][k] * f2[r]; }
    d1 *= beta[k];
    d2 *= beta[k];
#pragma unroll
    for (int r = k; r < 9; ++r) { f1[r] -= d1 * A[r][k]; f2[r] -= d2 * A[r][k]; }
  }
  double D[9], cA[9], cD[9];   // det(F2 + alpha D), D = F1 - F2
#pragma unroll
  for (int k = 0; k < 9; ++k) D[k] = f1[k] - f2[k];
  cofactors(f2, cA);
  cofactors(D, cD);
  double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
#pragma unroll
  for (int k = 0; k < 3; ++k) { c0 += f2[k] * cA[k]; c3 += D[k] * cD[k]; }
#pragma unroll
  for (int k = 0; k < 9; ++k) { c1 += cA[k] * D[k]; c2 += cD[k] * f2[k]; }
  double x[3];
  const int nr = cubic_roots(c3, c2, c1, c0, x);
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    if (r >= nr) break;
    double f[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) f[k] = x[r] * f1[k] + (1.0 - x[r]) * f2[k];
    denorm_f(f, T, m[r]);
  }
  return nr;
}

// ---------------------------------------------------------------------------------------------------- 4-point H
__device__ int solve4(const short4* pts, const int* idx, const Norm& T, double (&m)[3][9]) {
  short4 c[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) c[j] = pts[idx[j]];
#pragma unroll
  for (int u = 0; u < 4; ++u) {   // any three of the four collinear in a or in b: exact on integer coordinates
    const int i0 = u == 0 ? 1 : 0, i1 = u <= 1 ? 2 : 1, i2 = u <= 2 ? 3 : 2;
    const long long da = (long long)(c[i1].x - c[i0].x) * (c[i2].y - c[i0].y) - (long long)(c[i1].y - c[i0].y) * (c[i2].x - c[i0].x);
    const long long db = (long long)(c[i1].z - c[i0].z) * (c[i2].w - c[i0].w) - (long long)(c[i1].w - c[i0].w) * (c[i2].z - c[i0].z);
    if (da == 0 || db == 0) return 0;
  }
  double A[8][9];   // [A | rhs]
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const double xa = T.sa * (c[j].x - T.cxa), ya = T.sa * (c[j].y - T.cya), xb = T.sb * (c[j].z - T.cxb), yb = T.sb * (c[j].w - T.cyb);
    const double r0[9] = {xa, ya, 1.0, 0.0, 0.0, 0.0, -xa * xb, -ya * xb, xb};
    const double r1[9] = {0.0, 0.0, 0.0, xa, ya, 1.0, -xa * yb, -ya * yb, yb};
#pragma unroll
    for (int k = 0; k < 9; ++k) { A[2 * j][k] = r0[k]; A[2 * j + 1][k] = r1[k]; }
  }
  double R[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    double nrm = 0.0;
#pragma unroll
    for (int r = k; r < 8; ++r) nrm += A[r][k] * A[r][k];
    nrm = sqrt(nrm);
    if (!(nrm > kPivotTol)) return 0;
    const double alpha = A[k][k] >= 0.0 ? -nrm : nrm;
    A[k][k] -= alpha;
    double vv = 0.0;
#pragma unroll
    for (int r = k; r < 8; ++r) vv += A[r][k] * A[r][k];
    const double beta = 2.0 / vv;
#pragma unroll
    for (int j = k + 1; j < 9; ++j) {
      double dot = 0.0;
#pragma unroll
      for (int r = k; r < 8; ++r) dot += A[r][k] * A[r][j];
      dot *= beta;
#pragma unroll
      for (int r = k; r < 8; ++r) A[r][j] -= dot * A[r][k];
    }
    R[k] = alpha;
  }
  double h[9];
  h[8] = 1.0;
#pragma unroll
  for (int k = 7; k >= 0; --k) {   // R h = Q^T rhs; R's off-diagonal is A above the diagonal
    double s = A[k][8];
#pragma unroll
    for (int j = k + 1; j < 8; ++j) s -= A[k][j] * h[j];
    h[k] = s / R[k];
  }
  return denorm_h(h, T, m[0]) ? 1 : 0;
}

// ---------------------------------------------------------------------------------------------------- refinement
// Smallest-eigenvalue eigenvector of the symmetric n x n matrix A (destroyed) by cyclic Jacobi; V is n x n scratch.
__device__ void jacobi_min(double* A, double* V, int n, double* out) {
  for (int i = 0; i < n * n; ++i) V[i] = (i / n == i % n) ? 1.0 : 0.0;
  for (int sw = 0; sw < kJacobiSweeps; ++sw)
    for (int p = 0; p < n - 1; ++p)
      for (int q = p + 1; q < n; ++q) {
        const double apq = A[p * n + q];
        if (apq == 0.0) continue;
        const double th = (A[q * n + q] - A[p * n + p]) / (2.0 * apq);
        const double t = fabs(th) > 1e150 ? 0.5 / th : copysign(1.0, th) / (fabs(th) + sqrt(th * th + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < n; ++k) {   // A <- A J (columns p, q)
          const double akp = A[k * n + p], akq = A[k * n + q];
          A[k * n + p] = c * akp - s * akq;
          A[k * n + q] = s * akp + c * akq;
        }
        for (int k = 0; k < n; ++k) {   // A <- J^T A (rows p, q)
          const double apk = A[p * n + k], aqk = A[q * n + k];
          A[p * n + k] = c * apk - s * aqk;
          A[q * n + k] = s * apk + c * aqk;
        }
        for (int k = 0; k < n; ++k) {
          const double vkp = V[k * n + p], vkq = V[k * n + q];
          V[k * n + p] = c * vkp - s * vkq;
          V[k * n + q] = s * vkp + c * vkq;
        }
      }
  int mi = 0;
  for (int i = 1; i < n; ++i)
    if (A[i * n + i] < A[mi * n + mi]) mi = i;
  for (int k = 0; k < n; ++k) out[k] = V[k * n + mi];
}

struct Shared {
  double red[kT / 32];
  unsigned long long redu[kT / 32];
  double best[9];          // the current model, pixels
  double ata[81], vec[81]; // normal matrix, Jacobi scratch
  double v[9], u[3], f[9]; // eigenvectors, rank-2 F (normalised coordinates)
  double fit[9];           // refit, pixels
  int fit_ok;
};

// Element j of the design-matrix row(s) of one match in normalised coordinates: the epipolar constraint for F; for H
// the two DLT rows of x_b x (H x_a) = 0 (row 0 when second == false).
template <int MODEL>
__device__ __forceinline__ double design(int j, bool second, double xa, double ya, double xb, double yb) {
  if (MODEL == 0) {
    switch (j) {
      case 0: return xb * xa; case 1: return xb * ya; case 2: return xb;
      case 3: return yb * xa; case 4: return yb * ya; case 5: return yb;
      case 6: return xa;      case 7: return ya;      default: return 1.0;
    }
  }
  const double z = second ? yb : xb;
  switch (j) {
    case 0: return second ? 0.0 : -xa; case 1: return second ? 0.0 : -ya; case 2: return second ? 0.0 : -1.0;
    case 3: return second ? -xa : 0.0; case 4: return second ? -ya : 0.0; case 5: return second ? -1.0 : 0.0;
    case 6: return z * xa;             case 7: return z * ya;             default: return z;
  }
}

// mask[i] = inlier of m; returns the count (all threads)
template <int MODEL>
__device__ int score_mask(const short4* pts, int n, const double* m, double t2, uint8_t* mask, Shared& S) {
  double cnt = 0.0;
  for (int i = threadIdx.x; i < n; i += kT) {
    const bool in = is_inlier<MODEL>(m, pts[i], t2);
    mask[i] = in;
    cnt += in;
  }
  return (int)block_sum(cnt, S.red);
}

// Refit on the inliers in mask -> S.fit (pixels), S.fit_ok
template <int MODEL>
__device__ void refit(const short4* pts, int n, const uint8_t* mask, const Norm& T, Shared& S) {
  const int tid = threadIdx.x;
  if (tid < 45) {   // entry (j, k), j <= k, of the normal matrix, summed in match order
    int j = 0, e = tid;
    while (e >= 9 - j) { e -= 9 - j; ++j; }
    const int k = j + e;
    double acc = 0.0;
    for (int i = 0; i < n; ++i) {
      if (!mask[i]) continue;
      const short4 c = pts[i];
      const double xa = T.sa * (c.x - T.cxa), ya = T.sa * (c.y - T.cya), xb = T.sb * (c.z - T.cxb), yb = T.sb * (c.w - T.cyb);
      acc += design<MODEL>(j, false, xa, ya, xb, yb) * design<MODEL>(k, false, xa, ya, xb, yb);
      if (MODEL == 1) acc += design<MODEL>(j, true, xa, ya, xb, yb) * design<MODEL>(k, true, xa, ya, xb, yb);
    }
    S.ata[j * 9 + k] = acc;
    S.ata[k * 9 + j] = acc;
  }
  __syncthreads();
  if (tid == 0) {
    double* v = S.v;
    jacobi_min(S.ata, S.vec, 9, v);
    if (MODEL == 0) {   // rank 2: F (I - u u^T), u the smallest eigenvector of F^T F
      double* g = S.ata;
      for (int a = 0; a < 3; ++a)
        for (int b = 0; b < 3; ++b) g[a * 3 + b] = v[a] * v[b] + v[3 + a] * v[3 + b] + v[6 + a] * v[6 + b];
      jacobi_min(g, S.vec, 3, S.u);
      for (int r = 0; r < 3; ++r) {
        const double fu = v[3 * r] * S.u[0] + v[3 * r + 1] * S.u[1] + v[3 * r + 2] * S.u[2];
        for (int c = 0; c < 3; ++c) S.f[3 * r + c] = v[3 * r + c] - fu * S.u[c];
      }
      denorm_f(S.f, T, S.fit);
      S.fit_ok = 1;
    } else {
      S.fit_ok = denorm_h(v, T, S.fit) ? 1 : 0;
    }
  }
  __syncthreads();
}

template <int MODEL>
__global__ void __launch_bounds__(kT, 1) verify_kernel(const VerifyParams p) {
  constexpr int kS = MODEL == 0 ? 7 : 4;      // minimal sample
  constexpr int kMin = MODEL == 0 ? 8 : 4;    // matches needed for a model (and for a refit)
  extern __shared__ __align__(16) uint8_t smem[];
  short4* pts = reinterpret_cast<short4*>(smem);           // (col_a, row_a, col_b, row_b)
  uint8_t* mask = smem + (size_t)p.cap * sizeof(short4);
  __shared__ Shared S;
  const int q = blockIdx.x, tid = threadIdx.x;
  const int a = p.pairs[2 * q], b = p.pairs[2 * q + 1];
  const long long o0 = p.offsets[q], o1 = p.offsets[q + 1];
  if (!(o0 >= 0 && o0 <= o1 && o1 <= p.M && o1 - o0 <= p.cap)) {   // uniform per CTA
    if (tid < 9) p.model[(size_t)q * 9 + tid] = 0.0;
    if (tid == 0) { p.num[q] = -1; p.hyp[q] = 0; p.best[q] = -1; }
    return;
  }
  const int n = (int)(o1 - o0);
  int bad = 0;
  for (int i = tid; i < n; i += kT) {
    const int ia = p.matches[2 * (o0 + i)], ib = p.matches[2 * (o0 + i) + 1];
    short4 c = make_short4(0, 0, 0, 0);
    if (ia >= 0 && ia < p.cap && ib >= 0 && ib < p.cap) {
      const int* ka = p.kp + ((size_t)a * p.cap + ia) * 2;
      const int* kb = p.kp + ((size_t)b * p.cap + ib) * 2;
      const int ra = ka[0], ca = ka[1], rb = kb[0], cb = kb[1];
      if ((unsigned)ra <= 32767u && (unsigned)ca <= 32767u && (unsigned)rb <= 32767u && (unsigned)cb <= 32767u)
        c = make_short4((short)ca, (short)ra, (short)cb, (short)rb);
      else
        bad = 1;
    } else {
      bad = 1;
    }
    pts[i] = c;
    mask[i] = 0;
  }
  bad = __syncthreads_or(bad);
  double* out_m = p.model + (size_t)q * 9;
  if (bad || n < kMin) {
    for (int i = tid; i < n; i += kT) p.inlier[o0 + i] = 0;
    if (tid < 9) out_m[tid] = 0.0;
    if (tid == 0) { p.num[q] = bad ? -1 : 0; p.hyp[q] = 0; p.best[q] = -1; }
    return;
  }
  // Hartley normalisation over all of the pair's matches
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  for (int i = tid; i < n; i += kT) { const short4 c = pts[i]; s0 += c.x; s1 += c.y; s2 += c.z; s3 += c.w; }
  Norm T;
  T.cxa = block_sum(s0, S.red) / n; T.cya = block_sum(s1, S.red) / n;
  T.cxb = block_sum(s2, S.red) / n; T.cyb = block_sum(s3, S.red) / n;
  double da = 0.0, db = 0.0;
  for (int i = tid; i < n; i += kT) {
    const short4 c = pts[i];
    da += sqrt((c.x - T.cxa) * (c.x - T.cxa) + (c.y - T.cya) * (c.y - T.cya));
    db += sqrt((c.z - T.cxb) * (c.z - T.cxb) + (c.w - T.cyb) * (c.w - T.cyb));
  }
  const double mda = block_sum(da, S.red) / n, mdb = block_sum(db, S.red) / n;
  if (!(mda > 0.0 && mdb > 0.0)) {   // all points coincide in a or in b
    for (int i = tid; i < n; i += kT) p.inlier[o0 + i] = 0;
    if (tid < 9) out_m[tid] = 0.0;
    if (tid == 0) { p.num[q] = 0; p.hyp[q] = 0; p.best[q] = -1; }
    return;
  }
  T.sa = 1.4142135623730951 / mda;
  T.sb = 1.4142135623730951 / mdb;
  const unsigned long long key = splitmix64(p.seed ^ splitmix64(((unsigned long long)(unsigned)a << 32) | (unsigned)b));
  int best_cnt = -1, best_h = -1, drawn = 0;
  for (int r = 0;; ++r) {
    const int h = r * kT + tid;
    int idx[7];
    double m[3][9];
    int nm = 0;
    if (draw_sample(key, h, n, kS, idx)) nm = MODEL == 0 ? solve7(pts, idx, T, m) : solve4(pts, idx, T, m);
    int cnt[3] = {0, 0, 0};
    if (nm > 0) {
      for (int i = 0; i < n; ++i) {
        const short4 c = pts[i];
#pragma unroll
        for (int k = 0; k < (MODEL == 0 ? 3 : 1); ++k)
          if (k < nm) cnt[k] += is_inlier<MODEL>(m[k], c, p.t2);
      }
    }
    int tc = -1, tk = 0;
#pragma unroll
    for (int k = 0; k < 3; ++k)
      if (k < nm && cnt[k] > tc) { tc = cnt[k]; tk = k; }
    // (count desc, hypothesis asc): the largest key wins
    const unsigned long long win = block_max(((unsigned long long)(unsigned)(tc + 1) << 32) | (unsigned)(kT - 1 - tid), S.redu);
    const int wc = (int)(win >> 32) - 1, wt = kT - 1 - (int)(win & 0xffffffffu);
    if (wc > best_cnt) {   // earlier rounds hold lower hypotheses: only a strictly larger count replaces the best
      if (tid == wt) {
#pragma unroll
        for (int k = 0; k < 3; ++k)
          if (k == tk)
#pragma unroll
            for (int e = 0; e < 9; ++e) S.best[e] = m[k][e];
      }
      best_cnt = wc;
      best_h = r * kT + wt;
    }
    drawn = (r + 1) * kT;
    bool stop = drawn >= p.max_hyp;
    if (!stop && best_cnt > 0) {
      const double w = (double)best_cnt / n;
      double ws = w;
#pragma unroll
      for (int k = 1; k < kS; ++k) ws *= w;
      const double l = log(1.0 - ws);
      stop = l < 0.0 && (double)drawn >= p.log1mc / l;
    }
    __syncthreads();   // S.best is written
    if (stop) break;
  }
  if (best_cnt < 0) {   // every sample was degenerate
    for (int i = tid; i < n; i += kT) p.inlier[o0 + i] = 0;
    if (tid < 9) out_m[tid] = 0.0;
    if (tid == 0) { p.num[q] = 0; p.hyp[q] = drawn; p.best[q] = -1; }
    return;
  }
  // refinement
  int cur = score_mask<MODEL>(pts, n, S.best, p.t2, mask, S);
  for (int it = 0; it < kMaxRefits && cur >= kMin; ++it) {
    refit<MODEL>(pts, n, mask, T, S);
    if (!S.fit_ok) break;
    double c2 = 0.0;
    for (int i = tid; i < n; i += kT) c2 += is_inlier<MODEL>(S.fit, pts[i], p.t2);
    const int cnt2 = (int)block_sum(c2, S.red);
    if (cnt2 < cur) break;
    if (tid < 9) S.best[tid] = S.fit[tid];
    __syncthreads();
    const bool rising = cnt2 > cur;
    cur = score_mask<MODEL>(pts, n, S.best, p.t2, mask, S);
    if (!rising) break;
  }
  for (int i = tid; i < n; i += kT) p.inlier[o0 + i] = mask[i];
  if (tid == 0) {
    double f[9];
    for (int k = 0; k < 9; ++k) f[k] = S.best[k];
    if (MODEL == 0) {   // ||F||_F = 1, largest-magnitude element positive (first in row-major order on ties)
      double ss = 0.0;
      int im = 0;
      for (int k = 0; k < 9; ++k) {
        ss += f[k] * f[k];
        if (fabs(f[k]) > fabs(f[im])) im = k;
      }
      const double sc = (f[im] < 0.0 ? -1.0 : 1.0) / sqrt(ss);
      for (int k = 0; k < 9; ++k) f[k] *= sc;
    }
    for (int k = 0; k < 9; ++k) out_m[k] = f[k];
    p.num[q] = cur;
    p.hyp[q] = drawn;
    p.best[q] = best_h;
  }
}

}  // namespace

extern "C" int spn_verify_pairs(spn_ctx* ctx, const int32_t* d_kp, int N, int cap, const int32_t* h_pairs, int P,
                                const int64_t* d_offsets, const int32_t* d_matches, int64_t M, int model, double threshold_px,
                                double confidence, int max_iters, uint64_t seed, double* d_model, int32_t* d_num_inliers,
                                int32_t* d_hypotheses, int32_t* d_best, uint8_t* d_inlier, spn_stream stream) {
  SPN_REQUIRE(ctx, "spn_verify_pairs: null pointer (ctx)");
  SPN_REQUIRE(N > 0 && N <= kMaxN, "spn_verify_pairs: N = %d keypoint sets outside [1, %d]", N, kMaxN);
  SPN_REQUIRE(cap > 0 && cap <= kMaxCap, "spn_verify_pairs: cap = %d outside [1, %d]", cap, kMaxCap);
  SPN_REQUIRE(P >= 0 && P <= kMaxPairs, "spn_verify_pairs: P = %d pairs outside [0, %d]", P, kMaxPairs);
  SPN_REQUIRE(M >= 0, "spn_verify_pairs: M = %lld matches must be >= 0", (long long)M);
  SPN_REQUIRE(model == 0 || model == 1, "spn_verify_pairs: model = %d must be 0 (fundamental) or 1 (homography)", model);
  SPN_REQUIRE(isfinite(threshold_px) && threshold_px > 0.0, "spn_verify_pairs: threshold = %g px must be finite and > 0",
              threshold_px);
  SPN_REQUIRE(confidence > 0.0 && confidence < 1.0, "spn_verify_pairs: confidence = %g outside (0, 1)", confidence);
  SPN_REQUIRE(max_iters >= 1 && max_iters <= kMaxIters, "spn_verify_pairs: max_iters = %d outside [1, %d]", max_iters, kMaxIters);
  if (P == 0) return SPN_OK;
  SPN_REQUIRE(d_kp && h_pairs && d_offsets && d_model && d_num_inliers && d_hypotheses && d_best,
              "spn_verify_pairs: null pointer (kp / pairs / offsets / outputs)");
  SPN_REQUIRE(M == 0 || (d_matches && d_inlier), "spn_verify_pairs: null pointer (matches / inlier with M = %lld)", (long long)M);
  for (int q = 0; q < P; ++q)
    SPN_REQUIRE(h_pairs[2 * q] >= 0 && h_pairs[2 * q] < N && h_pairs[2 * q + 1] >= 0 && h_pairs[2 * q + 1] < N,
                "spn_verify_pairs: pair %d = (%d, %d) has an image index outside [0, %d)", q, h_pairs[2 * q], h_pairs[2 * q + 1], N);
  SpnDeviceGuard guard(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  const size_t pair_bytes = (size_t)P * 2 * sizeof(int32_t);
  int rc = spn_ensure_aux(ctx, pair_bytes, s);
  if (rc) return rc;
  // pageable source: the call returns once the bytes are staged
  SPN_CUDA(cudaMemcpyAsync(ctx->aux, h_pairs, pair_bytes, cudaMemcpyHostToDevice, s));
  VerifyParams p;
  p.kp = d_kp; p.pairs = (const int*)ctx->aux; p.offsets = (const long long*)d_offsets; p.matches = d_matches; p.M = M;
  p.cap = cap; p.t2 = threshold_px * threshold_px; p.log1mc = log(1.0 - confidence);
  p.max_hyp = spn_cdiv(max_iters, kT) * kT; p.seed = seed;
  p.model = d_model; p.num = d_num_inliers; p.hyp = d_hypotheses; p.best = d_best; p.inlier = d_inlier;
  const size_t smem = (((size_t)cap * (sizeof(short4) + 1)) + 15) / 16 * 16;
  if (model == 0) {
    SPN_CUDA(cudaFuncSetAttribute(verify_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    verify_kernel<0><<<P, kT, smem, s>>>(p);
  } else {
    SPN_CUDA(cudaFuncSetAttribute(verify_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    verify_kernel<1><<<P, kT, smem, s>>>(p);
  }
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}
