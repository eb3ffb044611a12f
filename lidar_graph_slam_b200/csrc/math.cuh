// Small dense linear algebra shared by host drivers and device kernels (__host__ __device__).
// These are the algorithms the reference reaches through Eigen (un-vendored): two-sided Jacobi SVD
// (JacobiSVD, NDT:127 and FG:273), tridiagonal QR symmetric eigensolver (SelfAdjointEigenSolver, VGC:333),
// cofactor 3x3 inverse (VGC:355,359; FG:149), pivoted LDLT (LSQ:111,136), eulerAngles(0,1,2) (NDT:109).
// Matrices are row-major unless noted.  No FMA contraction (build uses -fmad=false).
#pragma once
#include <cfloat>
#include <cmath>
#include <cstring>

#if defined(__CUDACC__)
#define LGS_HD __host__ __device__ __forceinline__
#else
#define LGS_HD inline
#endif

namespace lgs {
namespace m {

template <typename T>
struct Lim;
template <>
struct Lim<double> {
  static LGS_HD double eps() { return DBL_EPSILON; }
  static LGS_HD double tiny() { return DBL_MIN; }
};
template <>
struct Lim<float> {
  static LGS_HD float eps() { return FLT_EPSILON; }
  static LGS_HD float tiny() { return FLT_MIN; }
};

// clears the sign bit, as std::fabs: -0.0 -> +0.0 (a compare-and-negate keeps -0.0, and S / eigenvalues would differ in sign)
LGS_HD double tabs(double v) { return fabs(v); }
LGS_HD float tabs(float v) { return fabsf(v); }
// std::max / std::min (and Eigen's maxi / mini): the first argument unless the second compares larger (smaller), so a NaN
// second argument is skipped, and maxima are taken left to right as the reference's loops take them
template <typename T>
LGS_HD T tmax(T a, T b) { return a < b ? b : a; }
template <typename T>
LGS_HD T tmin(T a, T b) { return b < a ? b : a; }
LGS_HD double tsqrt(double v) { return sqrt(v); }
LGS_HD float tsqrt(float v) { return sqrtf(v); }

// plane rotation [c s; -s c]
template <typename T>
struct Givens {
  T c, s;
};

template <int N, typename T>
LGS_HD void rot_rows(T* a, int p, int q, T c, T s) {  // rows p,q: x' = c x + s y, y' = -s x + c y
  for (int i = 0; i < N; i++) {
    T x = a[p * N + i], y = a[q * N + i];
    a[p * N + i] = c * x + s * y;
    a[q * N + i] = -s * x + c * y;
  }
}
template <int N, typename T>
LGS_HD void rot_cols(T* a, int p, int q, T c, T s) {  // cols p,q: x' = c x - s y, y' = s x + c y
  for (int i = 0; i < N; i++) {
    T x = a[i * N + p], y = a[i * N + q];
    a[i * N + p] = c * x - s * y;
    a[i * N + q] = s * x + c * y;
  }
}

// Two-sided Jacobi SVD of a square matrix: A = U diag(S) V^T, S descending.
template <int N, typename T>
LGS_HD void svd_jacobi(const T* A, T* U, T* S, T* V) {
  const T precision = T(2) * Lim<T>::eps();
  const T tiny = Lim<T>::tiny();
  T W[N * N];
  T scale = T(0);
  for (int i = 0; i < N * N; i++) scale = tmax(scale, tabs(A[i]));
  if (scale == T(0)) scale = T(1);
  for (int i = 0; i < N * N; i++) W[i] = A[i] / scale;
  for (int i = 0; i < N; i++)
    for (int j = 0; j < N; j++) U[i * N + j] = V[i * N + j] = (i == j) ? T(1) : T(0);
  T max_diag = T(0);
  for (int i = 0; i < N; i++) max_diag = tmax(max_diag, tabs(W[i * N + i]));
  bool done = false;
  for (int sweep = 0; !done && sweep < 1000; sweep++) {
    done = true;
    for (int p = 1; p < N; ++p) {
      for (int q = 0; q < p; ++q) {
        T thr = tmax(tiny, precision * max_diag);
        if (tabs(W[p * N + q]) > thr || tabs(W[q * N + p]) > thr) {
          done = false;
          // 2x2 SVD of [[W_pp W_pq][W_qp W_qq]]: first symmetrise with a rotation, then diagonalise
          T m00 = W[p * N + p], m01 = W[p * N + q], m10 = W[q * N + p], m11 = W[q * N + q];
          T r1c, r1s;
          {
            T t = m00 + m11, d = m10 - m01;
            if (tabs(d) < tiny) {
              r1s = T(0);
              r1c = T(1);
            } else {
              T u = t / d;
              T tmp = tsqrt(T(1) + u * u);
              r1s = T(1) / tmp;
              r1c = u / tmp;
            }
          }
          {
            T x0 = r1c * m00 + r1s * m10, x1 = r1c * m01 + r1s * m11;
            T y0 = -r1s * m00 + r1c * m10, y1 = -r1s * m01 + r1c * m11;
            m00 = x0; m01 = x1; m10 = y0; m11 = y1;
          }
          T jrc, jrs;
          {
            T deno = T(2) * tabs(m01);
            if (deno < tiny) {
              jrc = T(1);
              jrs = T(0);
            } else {
              T tau = (m00 - m11) / deno;
              T w = tsqrt(tau * tau + T(1));
              T t = (tau > T(0)) ? T(1) / (tau + w) : T(1) / (tau - w);
              T sign_t = t > T(0) ? T(1) : T(-1);
              T n = T(1) / tsqrt(t * t + T(1));
              jrs = -sign_t * (m01 / tabs(m01)) * tabs(t) * n;
              jrc = n;
            }
          }
          // j_left = rot1 * j_right^T
          T jlc = r1c * jrc - r1s * (-jrs);
          T jls = r1c * (-jrs) + r1s * jrc;
          rot_rows<N, T>(W, p, q, jlc, jls);
          rot_cols<N, T>(U, p, q, jlc, -jls);
          rot_cols<N, T>(W, p, q, jrc, jrs);
          rot_cols<N, T>(V, p, q, jrc, jrs);
          max_diag = tmax(max_diag, tmax(tabs(W[p * N + p]), tabs(W[q * N + q])));
        }
      }
    }
  }
  for (int i = 0; i < N; i++) {
    T a = tabs(W[i * N + i]);
    S[i] = a;
    if (a != T(0)) {
      T f = W[i * N + i] / a;
      for (int r = 0; r < N; r++) U[r * N + i] *= f;
    }
  }
  for (int i = 0; i < N; i++) S[i] *= scale;
  for (int i = 0; i < N; i++) {
    int pos = i;
    T mx = S[i];
    for (int k = i + 1; k < N; k++)
      if (S[k] > mx) {
        mx = S[k];
        pos = k;
      }
    if (mx == T(0)) break;
    if (pos != i) {
      T t = S[i]; S[i] = S[pos]; S[pos] = t;
      for (int r = 0; r < N; r++) {
        t = U[r * N + i]; U[r * N + i] = U[r * N + pos]; U[r * N + pos] = t;
        t = V[r * N + i]; V[r * N + i] = V[r * N + pos]; V[r * N + pos] = t;
      }
    }
  }
}

// Minimum-norm solve through the SVD with Eigen's default rank threshold (N * eps * sigma_max).
template <int N>
LGS_HD void svd_solve(const double* A, const double* b, double* x) {
  double U[N * N], S[N], V[N * N];
  svd_jacobi<N, double>(A, U, S, V);
  double thr = tmax(S[0] * (double(N) * DBL_EPSILON), DBL_MIN);
  int rank = N;
  while (rank > 0 && S[rank - 1] < thr) --rank;
  double t[N];
  for (int i = 0; i < rank; i++) {
    double acc = 0.0;
    for (int r = 0; r < N; r++) acc += U[r * N + i] * b[r];
    t[i] = acc / S[i];
  }
  for (int r = 0; r < N; r++) {
    double acc = 0.0;
    for (int i = 0; i < rank; i++) acc += V[r * N + i] * t[i];
    x[r] = acc;
  }
}

// 3x3 inverse by cofactors along column 0.
LGS_HD void inv3(const double* a, double* r) {
#define LGS_COF(i, j) (a[((i + 1) % 3) * 3 + (j + 1) % 3] * a[((i + 2) % 3) * 3 + (j + 2) % 3] - a[((i + 1) % 3) * 3 + (j + 2) % 3] * a[((i + 2) % 3) * 3 + (j + 1) % 3])
  double c00 = LGS_COF(0, 0), c10 = LGS_COF(1, 0), c20 = LGS_COF(2, 0);
  double det = (c00 * a[0] + c10 * a[3]) + c20 * a[6];
  double id = 1.0 / det;
  r[0] = c00 * id;            r[1] = c10 * id;            r[2] = c20 * id;
  r[3] = LGS_COF(0, 1) * id;  r[4] = LGS_COF(1, 1) * id;  r[5] = LGS_COF(2, 1) * id;
  r[6] = LGS_COF(0, 2) * id;  r[7] = LGS_COF(1, 2) * id;  r[8] = LGS_COF(2, 2) * id;
#undef LGS_COF
}

LGS_HD void mul3(const double* a, const double* b, double* c) {
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) c[i * 3 + j] = (a[i * 3] * b[j] + a[i * 3 + 1] * b[3 + j]) + a[i * 3 + 2] * b[6 + j];
}

// Symmetric 3x3 eigen decomposition (lower triangle read): Householder tridiagonalisation specialised
// for 3x3 followed by implicit-shift QR steps with Wilkinson shifts; eigenvalues ascending, eigenvectors
// in the columns of Q.
LGS_HD bool eig_sym3(const double* A, double* w, double* Q) {
  double a00 = A[0], a10 = A[3], a11 = A[4], a20 = A[6], a21 = A[7], a22 = A[8];
  double scale = tmax(tmax(tmax(tmax(tmax(tmax(0.0, tabs(a00)), tabs(a10)), tabs(a11)), tabs(a20)), tabs(a21)), tabs(a22));
  if (scale == 0.0) scale = 1.0;
  a00 /= scale; a10 /= scale; a11 /= scale; a20 /= scale; a21 /= scale; a22 /= scale;
  double d[3], e[2];
  d[0] = a00;
  double v1n2 = a20 * a20;
  if (v1n2 <= DBL_MIN) {
    d[1] = a11; d[2] = a22; e[0] = a10; e[1] = a21;
    for (int i = 0; i < 9; i++) Q[i] = (i % 4 == 0) ? 1.0 : 0.0;
  } else {
    double beta = sqrt(a10 * a10 + v1n2);
    double ib = 1.0 / beta;
    double m01 = a10 * ib, m02 = a20 * ib;
    double q = 2.0 * m01 * a21 + m02 * (a22 - a11);
    d[1] = a11 + m02 * q;
    d[2] = a22 - m02 * q;
    e[0] = beta;
    e[1] = a21 - m01 * q;
    Q[0] = 1; Q[1] = 0;   Q[2] = 0;
    Q[3] = 0; Q[4] = m01; Q[5] = m02;
    Q[6] = 0; Q[7] = m02; Q[8] = -m01;
  }
  const int n = 3, max_it = 30;
  int end = n - 1, start = 0, iter = 0;
  const double pinv = 1.0 / DBL_EPSILON;
  while (end > 0) {
    for (int i = start; i < end; ++i) {
      if (tabs(e[i]) < DBL_MIN) {
        e[i] = 0.0;
      } else {
        double se = pinv * e[i];
        if (se * se <= (tabs(d[i]) + tabs(d[i + 1]))) e[i] = 0.0;
      }
    }
    while (end > 0 && e[end - 1] == 0.0) end--;
    if (end <= 0) break;
    iter++;
    if (iter > max_it * n) break;
    start = end - 1;
    while (start > 0 && e[start - 1] != 0.0) start--;
    double td = (d[end - 1] - d[end]) * 0.5;
    double ee = e[end - 1];
    double mu = d[end];
    if (td == 0.0) {
      mu -= tabs(ee);
    } else if (ee != 0.0) {
      double e2 = ee * ee;
      double ax = tabs(td), ay = tabs(ee);
      double pp = tmax(ax, ay);
      double h = 0.0;
      if (pp != 0.0) {
        double qp = tmin(ax, ay) / pp;
        h = pp * sqrt(1.0 + qp * qp);
      }
      if (e2 == 0.0)
        mu -= ee / ((td + (td > 0.0 ? h : -h)) / ee);
      else
        mu -= e2 / (td + (td > 0.0 ? h : -h));
    }
    double x = d[start] - mu;
    double z = e[start];
    for (int k = start; k < end && z != 0.0; ++k) {
      double c, s;
      if (z == 0.0) {
        c = x < 0.0 ? -1.0 : 1.0; s = 0.0;
      } else if (x == 0.0) {
        c = 0.0; s = z < 0.0 ? 1.0 : -1.0;
      } else if (tabs(x) > tabs(z)) {
        double t = z / x;
        double u = sqrt(1.0 + t * t);
        if (x < 0.0) u = -u;
        c = 1.0 / u; s = -t * c;
      } else {
        double t = x / z;
        double u = sqrt(1.0 + t * t);
        if (z < 0.0) u = -u;
        s = -1.0 / u; c = -t * s;
      }
      double sdk = s * d[k] + c * e[k];
      double dkp1 = s * e[k] + c * d[k + 1];
      d[k] = c * (c * d[k] - s * e[k]) - s * (c * e[k] - s * d[k + 1]);
      d[k + 1] = s * sdk + c * dkp1;
      e[k] = c * sdk - s * dkp1;
      if (k > start) e[k - 1] = c * e[k - 1] - s * z;
      x = e[k];
      if (k < end - 1) {
        z = -s * e[k + 1];
        e[k + 1] = c * e[k + 1];
      }
      rot_cols<3, double>(Q, k, k + 1, c, s);
    }
  }
  bool ok = iter <= max_it * n;
  if (ok) {
    for (int i = 0; i < n - 1; ++i) {
      int k = 0;
      double mn = d[i];
      for (int j = 1; j < n - i; j++)
        if (d[i + j] < mn) {
          mn = d[i + j];
          k = j;
        }
      if (k > 0) {
        double t = d[i]; d[i] = d[k + i]; d[k + i] = t;
        for (int r = 0; r < 3; r++) {
          t = Q[r * 3 + i]; Q[r * 3 + i] = Q[r * 3 + k + i]; Q[r * 3 + k + i] = t;
        }
      }
    }
  }
  for (int i = 0; i < 3; i++) w[i] = d[i] * scale;
  return ok;
}

// Robust Cholesky (LDL^T with symmetric diagonal pivoting, lower triangle, in place) and solve, 6x6.
// Pivot = largest |diagonal| of the trailing block; D is applied through a pseudo-inverse.
LGS_HD void ldlt_solve6(const double* Ain, const double* b, double* x) {
  const int N = 6;
  double A[36];
  for (int i = 0; i < 36; i++) A[i] = Ain[i];
  int tr[N];
  for (int k = 0; k < N; k++) {
    int piv = k;
    double big = tabs(A[k * N + k]);
    for (int i = k + 1; i < N; i++) {
      double v = tabs(A[i * N + i]);
      if (v > big) {
        big = v;
        piv = i;
      }
    }
    tr[k] = piv;
    if (piv != k) {
      double t;
      for (int j = 0; j < k; j++) { t = A[k * N + j]; A[k * N + j] = A[piv * N + j]; A[piv * N + j] = t; }
      for (int i = piv + 1; i < N; i++) { t = A[i * N + k]; A[i * N + k] = A[i * N + piv]; A[i * N + piv] = t; }
      t = A[k * N + k]; A[k * N + k] = A[piv * N + piv]; A[piv * N + piv] = t;
      for (int i = k + 1; i < piv; i++) { t = A[i * N + k]; A[i * N + k] = A[piv * N + i]; A[piv * N + i] = t; }
    }
    if (k > 0) {
      double tmp[N];
      for (int j = 0; j < k; j++) tmp[j] = A[j * N + j] * A[k * N + j];
      double acc = 0.0;
      for (int j = 0; j < k; j++) acc += A[k * N + j] * tmp[j];
      A[k * N + k] -= acc;
      for (int i = k + 1; i < N; i++) {
        double a2 = 0.0;
        for (int j = 0; j < k; j++) a2 += A[i * N + j] * tmp[j];
        A[i * N + k] -= a2;
      }
    }
    double pivot = A[k * N + k];
    if (k == 0 && !(tabs(pivot) > 0.0)) {
      for (int j = 0; j < N; j++) tr[j] = j;
      break;
    }
    if (tabs(pivot) > 0.0)
      for (int i = k + 1; i < N; i++) A[i * N + k] /= pivot;
  }
  double y[N];
  for (int i = 0; i < N; i++) y[i] = b[i];
  for (int k = 0; k < N; k++) { double t = y[k]; y[k] = y[tr[k]]; y[tr[k]] = t; }
  for (int i = 0; i < N; i++) {
    double acc = y[i];
    for (int j = 0; j < i; j++) acc -= A[i * N + j] * y[j];
    y[i] = acc;
  }
  for (int i = 0; i < N; i++) {
    double d = A[i * N + i];
    y[i] = (tabs(d) > DBL_MIN) ? y[i] / d : 0.0;
  }
  for (int i = N - 1; i >= 0; i--) {
    double acc = y[i];
    for (int j = i + 1; j < N; j++) acc -= A[j * N + i] * y[j];
    y[i] = acc;
  }
  for (int k = N - 1; k >= 0; k--) { double t = y[k]; y[k] = y[tr[k]]; y[tr[k]] = t; }
  for (int i = 0; i < N; i++) x[i] = y[i];
}

}  // namespace m

// Host 4x4 transforms, column-major.  mul4f keeps Matrix4f's f32 order ((a0 b0 + a1 b1) + a2 b2) + a3 b3: the registration
// results built from it are compared bit for bit with the reference.  C may alias A or B.
inline void identity16f(float* T) {
  for (int i = 0; i < 16; i++) T[i] = (i % 5 == 0) ? 1.0f : 0.0f;
}
inline void mul4f(const float* A, const float* B, float* C) {
  float R[16];
  for (int c = 0; c < 4; c++)
    for (int r = 0; r < 4; r++) R[c * 4 + r] = ((A[r] * B[c * 4] + A[4 + r] * B[c * 4 + 1]) + A[8 + r] * B[c * 4 + 2]) + A[12 + r] * B[c * 4 + 3];
  memcpy(C, R, sizeof(R));
}

}  // namespace lgs
