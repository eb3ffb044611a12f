// The optimiser of pclomp::NormalDistributionsTransform as a resumable state machine, one source for the host and the
// device: computeTransformation (NDT:80-171: Newton step, exit rules), computeStepLengthMT / updateIntervalMT /
// trialValueSelectionMT (NDT:771-931, 647-685, 688-768: More-Thuente line search), computeAngleDerivatives
// (NDT:288-394) and convertTransform (NDT.h:214-231).
//
// An align is a chain of derivative evaluations, each of which needs the sums of the one before it to choose its pose.
// The machine is fed the sums of the pending evaluation (advance) and answers with the next evaluation to run - a pose, its
// f32 transform and angular tables, and a mode - or with "done".  Driven
//   * by the host (ndt.cu, one kernel launch per evaluation): small clouds, profiling, the parity hooks;
//   * by CTA 0 of ndt_align_kernel (ndt_deriv.cuh): the whole align is ONE launch, the grid stays resident, and nothing
//     crosses PCIe between the first evaluation and the result record.
// All state is f64 and every expression keeps the reference's operation order (no FMA contraction: -fmad=false), so both
// drivers walk the same path.
#pragma once
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "math.cuh"

namespace lgs {
namespace ndtopt {

// ---- trigonometry ------------------------------------------------------------------------------------------------
// The reference takes sinf / cosf of the f32 angles (Eigen::AngleAxisf, NDT.h:222-224) and sin / cos of the f64 angles
// (NDT:293-326) from the C library.  A one-ulp difference in a sine moves every transformed point, so the device-resident
// optimiser must produce the libm's bits, not merely a good sine.  sinf_libm / cosf_libm restate glibc's single-precision
// routines (sysdeps/ieee754/flt-32/s_sincosf.h, the ARM optimized-routines algorithm, glibc 2.28+; pinned here against
// glibc 2.39 on x86-64 with FMA: quadrant reduction x - n * pi/2 with n = round(x * 2/pi) taken from a 2^24-scaled
// conversion, then a degree-7 / degree-8 polynomial in f64 with the constants below, multiply-adds fused as the library's
// FMA build fuses them) and agree with it bit for bit for every |x| < 120 (2.2e9 values, tests/sincos_check.cpp runs a
// sample of that sweep).  The f64 sine / cosine of the angular tables are the platform's own (libm on the host,
// libdevice on the GPU, which may differ by an ulp): they reach the f32 terms only through a cast that absorbs it.
struct SinCosTab {
  double c0, c1, s1, c2, s2, c3, s3, c4;
};
LGS_HD double fma_rn(double a, double b, double c) {
#if defined(__CUDA_ARCH__)
  return __fma_rn(a, b, c);
#else
  return fma(a, b, c);
#endif
}
LGS_HD float sincosf_poly(double x, double x2, bool negated, int n) {
  const SinCosTab t0 = {0x1p0, -0x1.ffffffd0c621cp-2, -0x1.555545995a603p-3, 0x1.55553e1068f19p-5, 0x1.1107605230bc4p-7, -0x1.6c087e89a359dp-10,
                        -0x1.994eb3774cf24p-13, 0x1.99343027bf8c3p-16};
  const SinCosTab t1 = {-0x1p0, 0x1.ffffffd0c621cp-2, -0x1.555545995a603p-3, -0x1.55553e1068f19p-5, 0x1.1107605230bc4p-7, 0x1.6c087e89a359dp-10,
                        -0x1.994eb3774cf24p-13, -0x1.99343027bf8c3p-16};
  const SinCosTab& p = negated ? t1 : t0;
  if ((n & 1) == 0) {
    const double x3 = x * x2;
    const double s1 = fma_rn(x2, p.s3, p.s2);
    const double x7 = x3 * x2;
    const double s = fma_rn(x3, p.s1, x);
    return static_cast<float>(fma_rn(x7, s1, s));
  }
  const double x4 = x2 * x2;
  const double c2 = fma_rn(x2, p.c4, p.c3);
  const double c1 = fma_rn(x2, p.c1, p.c0);
  const double x6 = x4 * x2;
  const double c = fma_rn(x4, p.c2, c1);
  return static_cast<float>(fma_rn(x6, c2, c));
}
LGS_HD unsigned abstop12(float x) {
#if defined(__CUDA_ARCH__)
  return (__float_as_uint(x) >> 20) & 0x7ffu;
#else
  unsigned u;
  memcpy(&u, &x, 4);
  return (u >> 20) & 0x7ffu;
#endif
}
// which = 0: sinf(y), 1: cosf(y)
LGS_HD float sincosf_libm(float y, int which) {
  double x = y;
  if (abstop12(y) < abstop12(0x1.921FB6p-1f)) {
    if (abstop12(y) < abstop12(0x1p-12f)) return which ? 1.0f : y;
    return sincosf_poly(x, x * x, false, which);
  }
  if (abstop12(y) < abstop12(120.0f)) {
    const double r = x * 0x1.45F306DC9C883p+23;
    const int n = (static_cast<int>(r) + 0x800000) >> 24;
    x = fma_rn(-static_cast<double>(n), 0x1.921FB54442D18p0, x);
    const int q = n + which;
    const double sign = ((q & 3) == 1 || (q & 3) == 2) ? -1.0 : 1.0;
    return sincosf_poly(x * sign, x * x, (q & 2) != 0, n ^ which);
  }
  // |y| >= 120 rad never occurs for roll / pitch / yaw (the library switches to a Payne-Hanek style reduction there): f64 function, rounded
  return static_cast<float>(which ? cos(x) : sin(x));
}
LGS_HD float sinf_libm(float y) { return sincosf_libm(y, 0); }
LGS_HD float cosf_libm(float y) { return sincosf_libm(y, 1); }

struct Trig {
  float sf[3], cf[3];  // sinf / cosf of (float) roll, pitch, yaw
  double f[8];         // 1, 0, then cos / sin of the f64 roll, pitch, yaw (cx, sx, cy, sy, cz, sz) with the small-angle snap
                       // of NDT:293-326: the factors of the angular tables, addressed by angle_entry
};

// the twelve values of a pose, one at a time (k = 0..2: sinf, 3..5: cosf, 6..8: sin, 9..11: cos of roll / pitch / yaw) so
// that the device can spread them over threads; trig_of_pose is the same arithmetic in a loop
LGS_HD void trig_value(const double x[6], int k, Trig* t) {
  const int a = k % 3;
  if (k < 3) {
    t->sf[a] = sinf_libm(static_cast<float>(x[3 + a]));
  } else if (k < 6) {
    t->cf[a] = cosf_libm(static_cast<float>(x[3 + a]));
  } else {
    const bool snap = fabs(x[3 + a]) < 10e-5;  // NDT:293-326
    if (k < 9)
      t->f[3 + 2 * a] = snap ? 0.0 : sin(x[3 + a]);
    else
      t->f[2 + 2 * a] = snap ? 1.0 : cos(x[3 + a]);
    if (k == 6) {
      t->f[0] = 1.0;
      t->f[1] = 0.0;
    }
  }
}
LGS_HD void trig_of_pose(const double x[6], Trig* t) {
  for (int k = 0; k < 12; k++) trig_value(x, k, t);
}

// Eigen::AngleAxis<float>(angle, Unit{X,Y,Z}).toRotationMatrix() from the angle's sine and cosine: note (1-c)*1 + c on
// the axis diagonal
template <int AXIS>
LGS_HD void angle_axis_unit(float s, float c, float* R) {
  const float ax[3] = {AXIS == 0 ? 1.0f : 0.0f, AXIS == 1 ? 1.0f : 0.0f, AXIS == 2 ? 1.0f : 0.0f};
  const float sa[3] = {s * ax[0], s * ax[1], s * ax[2]};
  const float ca[3] = {(1.0f - c) * ax[0], (1.0f - c) * ax[1], (1.0f - c) * ax[2]};
  float tmp = ca[0] * ax[1];
  R[1] = tmp - sa[2];
  R[3] = tmp + sa[2];
  tmp = ca[0] * ax[2];
  R[2] = tmp + sa[1];
  R[6] = tmp - sa[1];
  tmp = ca[1] * ax[2];
  R[5] = tmp - sa[0];
  R[7] = tmp + sa[0];
  for (int a = 0; a < 3; a++) R[a * 4] = ca[a] * ax[a] + c;
}

LGS_HD float mul3f_entry(const float* a, const float* b, int i, int j) { return (a[i * 3] * b[j] + a[i * 3 + 1] * b[3 + j]) + a[i * 3 + 2] * b[6 + j]; }
LGS_HD void mul3f(const float* a, const float* b, float* c) {
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) c[i * 3 + j] = mul3f_entry(a, b, i, j);
}

// NDT.h:214-231: Translation * AngleAxis(X) * AngleAxis(Y) * AngleAxis(Z) in f32, column-major out
LGS_HD void pose_to_matrix(const double x[6], const Trig& t, float* T) {
  float Rx[9], Ry[9], Rz[9], Rxy[9], R[9];
  angle_axis_unit<0>(t.sf[0], t.cf[0], Rx);
  angle_axis_unit<1>(t.sf[1], t.cf[1], Ry);
  angle_axis_unit<2>(t.sf[2], t.cf[2], Rz);
  mul3f(Rx, Ry, Rxy);
  mul3f(Rxy, Rz, R);
  for (int i = 0; i < 16; i++) T[i] = (i % 5 == 0) ? 1.0f : 0.0f;
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) T[c * 4 + r] = R[r * 3 + c];
  T[12] = static_cast<float>(x[0]);
  T[13] = static_cast<float>(x[1]);
  T[14] = static_cast<float>(x[2]);
}

// computeAngleDerivatives (NDT:329-392): rows a..h of j_ang (entries 0..23) and a2..f3 of h_ang (entries 24..68), f64 and
// their f32 casts.  Every entry of the reference is s1 * f1 * f2 * f3 [+ s2 * f4 * f5 * f6] with the factors taken from
// {1, 0, cx, sx, cy, sy, cz, sz}, products evaluated left to right; the encoding below (generated from the expressions of
// angle_tables_explicit, 3 bits per factor, 1 sign bit per term, 1 bit "has a second term") lets one thread evaluate one
// entry without a 69-way branch.  Multiplying by 1.0 and negating are exact, so each entry has the bits of its expression.
#define LGS_ANGLE_CODES                                                                                                       \
  0x16aa3b, 0x1faa33, 0x000222, 0x16ac3a, 0x1fac32, 0x000223, 0x000235, 0x00003d, 0x000004, 0x0001a3, 0x0003e3, 0x00002b,     \
      0x0003a2, 0x0001e2, 0x00022a, 0x00023c, 0x000234, 0x000001, 0x1fac32, 0x1eae3a, 0x000001, 0x17a833, 0x18edaa, 0x000001, \
      0x1eae3a, 0x17ae32, 0x000023, 0x16aa3b, 0x18cfea, 0x000222, 0x0001a2, 0x0003e2, 0x00002a, 0x0001a3, 0x0003e3, 0x00002b, \
      0x1faa33, 0x1ea83b, 0x000001, 0x1fac32, 0x18ebab, 0x000001, 0x000234, 0x00003c, 0x000005, 0x0003ab, 0x0001eb, 0x000023, \
      0x0001aa, 0x0003ea, 0x000222, 0x00003d, 0x000035, 0x000001, 0x0003e3, 0x0003a3, 0x000001, 0x0001e2, 0x0001a2, 0x000001, \
      0x000234, 0x00003c, 0x000001, 0x1eae3a, 0x17ae32, 0x000001, 0x16aa3b, 0x18cfea, 0x000001
#if defined(__CUDACC__)
__constant__ unsigned kAngleCodeDev[69] = {LGS_ANGLE_CODES};
#endif
// the encoding table; on the device a driver copies it next to the state it works on (Machine::codes, shared memory):
// 69 threads reading 69 different words of __constant__ memory would be serialised by the constant cache
LGS_HD void angle_codes(unsigned* out) {
#if defined(__CUDA_ARCH__)
  for (int e = 0; e < 69; e++) out[e] = kAngleCodeDev[e];
#else
  static const unsigned code[69] = {LGS_ANGLE_CODES};
  for (int e = 0; e < 69; e++) out[e] = code[e];
#endif
}
LGS_HD double angle_entry(const Trig& t, unsigned c) {
  const double* f = t.f;
  double t1 = (f[c & 7] * f[(c >> 3) & 7]) * f[(c >> 6) & 7];
  if (c & (1u << 9)) t1 = -t1;
  if (!(c & (1u << 20))) return t1;
  double t2 = (f[(c >> 10) & 7] * f[(c >> 13) & 7]) * f[(c >> 16) & 7];
  if (c & (1u << 19)) t2 = -t2;
  return t1 + t2;
}
LGS_HD void angle_table_store(const Trig& t, const unsigned* codes, int e, double (*Jd)[3], double (*Hd)[3], float (*Jf)[3], float (*Hf)[3]) {
  const double v = angle_entry(t, codes[e]);
  if (e < 24) {
    (&Jd[0][0])[e] = v;
    (&Jf[0][0])[e] = static_cast<float>(v);
  } else {
    (&Hd[0][0])[e - 24] = v;
    (&Hf[0][0])[e - 24] = static_cast<float>(v);
  }
}
LGS_HD void angle_tables(const Trig& t, double (*Jd)[3], double (*Hd)[3], float (*Jf)[3], float (*Hf)[3]) {
  unsigned codes[69];
  angle_codes(codes);
  for (int e = 0; e < 69; e++) angle_table_store(t, codes, e, Jd, Hd, Jf, Hf);
}

// The same tables written out as in the reference (NDT:329-392).  Only tests/ndt_opt_check.cpp calls this: it pins the
// table-driven form above to these expressions bit for bit (signed zeros included).
LGS_HD void angle_tables_explicit(const Trig& t, double (*Jd)[3], double (*Hd)[3], float (*Jf)[3], float (*Hf)[3]) {
  const double cx = t.f[2], sx = t.f[3], cy = t.f[4], sy = t.f[5], cz = t.f[6], sz = t.f[7];
  const double J[8][3] = {{(-sx * sz + cx * sy * cz), (-sx * cz - cx * sy * sz), (-cx * cy)},
                          {(cx * sz + sx * sy * cz), (cx * cz - sx * sy * sz), (-sx * cy)},
                          {(-sy * cz), sy * sz, cy},
                          {sx * cy * cz, (-sx * cy * sz), sx * sy},
                          {(-cx * cy * cz), cx * cy * sz, (-cx * sy)},
                          {(-cy * sz), (-cy * cz), 0},
                          {(cx * cz - sx * sy * sz), (-cx * sz - sx * sy * cz), 0},
                          {(sx * cz + cx * sy * sz), (cx * sy * cz - sx * sz), 0}};
  const double H[15][3] = {{(-cx * sz - sx * sy * cz), (-cx * cz + sx * sy * sz), sx * cy},
                           {(-sx * sz + cx * sy * cz), (-cx * sy * sz - sx * cz), (-cx * cy)},
                           {(cx * cy * cz), (-cx * cy * sz), (cx * sy)},
                           {(sx * cy * cz), (-sx * cy * sz), (sx * sy)},
                           {(-sx * cz - cx * sy * sz), (sx * sz - cx * sy * cz), 0},
                           {(cx * cz - sx * sy * sz), (-sx * sy * cz - cx * sz), 0},
                           {(-cy * cz), (cy * sz), (sy)},
                           {(-sx * sy * cz), (sx * sy * sz), (sx * cy)},
                           {(cx * sy * cz), (-cx * sy * sz), (-cx * cy)},
                           {(sy * sz), (sy * cz), 0},
                           {(-sx * cy * sz), (-sx * cy * cz), 0},
                           {(cx * cy * sz), (cx * cy * cz), 0},
                           {(-cy * cz), (cy * sz), 0},
                           {(-cx * sz - sx * sy * cz), (-cx * cz + sx * sy * sz), 0},
                           {(-sx * sz + cx * sy * cz), (-cx * sy * sz - sx * cz), 0}};
  for (int r = 0; r < 8; r++)
    for (int c = 0; c < 3; c++) {
      Jd[r][c] = J[r][c];
      Jf[r][c] = static_cast<float>(J[r][c]);
    }
  for (int r = 0; r < 15; r++)
    for (int c = 0; c < 3; c++) {
      Hd[r][c] = H[r][c];
      Hf[r][c] = static_cast<float>(H[r][c]);
    }
}

// ---- More-Thuente pieces ---------------------------------------------------------------------------------------------
// std::min / std::max as the reference's expressions evaluate them (the argument order decides what a NaN does)
LGS_HD double std_min(double a, double b) { return (b < a) ? b : a; }
LGS_HD double std_max(double a, double b) { return (a < b) ? b : a; }

LGS_HD double dot6(const double* a, const double* b) {
  double s = 0;
  for (int i = 0; i < 6; i++) s += a[i] * b[i];
  return s;
}

// updateIntervalMT (NDT:647-685)
LGS_HD bool update_interval(double& a_l, double& f_l, double& g_l, double& a_u, double& f_u, double& g_u, double a_t, double f_t, double g_t) {
  if (f_t > f_l) {
    a_u = a_t; f_u = f_t; g_u = g_t;
    return false;
  }
  if (g_t * (a_l - a_t) > 0) {
    a_l = a_t; f_l = f_t; g_l = g_t;
    return false;
  }
  if (g_t * (a_l - a_t) < 0) {
    a_u = a_l; f_u = f_l; g_u = g_l;
    a_l = a_t; f_l = f_t; g_l = g_t;
    return false;
  }
  return true;
}

LGS_HD double mt_cubic(double a0, double f0, double g0, double a1, double f1, double g1) {
  const double z = 3 * (f1 - f0) / (a1 - a0) - g1 - g0;
  const double w = sqrt(z * z - g1 * g0);
  return a0 + (a1 - a0) * (w - g0 - z) / (g1 - g0 + 2 * w);
}

// trialValueSelectionMT (NDT:688-768)
LGS_HD double trial_value(double a_l, double f_l, double g_l, double a_u, double f_u, double g_u, double a_t, double f_t, double g_t) {
  if (f_t > f_l) {
    const double a_c = mt_cubic(a_l, f_l, g_l, a_t, f_t, g_t);
    const double a_q = a_l - 0.5 * (a_l - a_t) * g_l / (g_l - (f_l - f_t) / (a_l - a_t));
    return fabs(a_c - a_l) < fabs(a_q - a_l) ? a_c : 0.5 * (a_q + a_c);
  }
  if (g_t * g_l < 0) {
    const double a_c = mt_cubic(a_l, f_l, g_l, a_t, f_t, g_t);
    const double a_s = a_l - (a_l - a_t) / (g_l - g_t) * g_l;
    return fabs(a_c - a_t) >= fabs(a_s - a_t) ? a_c : a_s;
  }
  if (fabs(g_t) <= fabs(g_l)) {
    const double a_c = mt_cubic(a_l, f_l, g_l, a_t, f_t, g_t);
    const double a_s = a_l - (a_l - a_t) / (g_l - g_t) * g_l;
    const double a_next = fabs(a_c - a_t) < fabs(a_s - a_t) ? a_c : a_s;
    const double lim = a_t + 0.66 * (a_u - a_t);
    return a_t > a_l ? std_min(lim, a_next) : std_max(lim, a_next);
  }
  return mt_cubic(a_u, f_u, g_u, a_t, f_t, g_t);
}

// ---- Newton step ------------------------------------------------------------------------------------------------------
// delta = -H^-1 g (NDT:127-129).  H is the FULL 6x6 of the reference: its f32 terms are not symmetric - entry (i,j) is
// e * ((-d2 * g_i) * g_j + ... + JCJ(j,i)), entry (j,i) rounds the same products in the other order (NDT:521-531) - so the
// two triangles differ by ~1e-8 relative, and the JacobiSVD of the reference sees both.  (Mirroring one triangle moves the
// Newton step by that much: enough to flip the f32 rounding of an entry of the next transform every few evaluations, after
// which the two optimisers walk different paths.)
// The reference goes through Eigen's two-sided JacobiSVD: ~80 dependent plane rotations, each a chain of f64 divisions and
// square roots - 5 us on a CPU core, 30-40 us on a GPU thread, more than the derivative evaluation it sits between;
// Gaussian elimination still chains six reciprocals (measured: 5.8k SM cycles).  The solution only enters the align
// through p -> (f32 transform, f32 tables), so the machine solves the regular case by block elimination on
// H = [A B; C D] (A: translations, D: rotations): A^-1 and the inverse of the Schur complement S = D - C A^-1 B in closed
// form (adjugate / determinant) - two reciprocals in the whole dependency chain.  It agrees with the SVD solution to
// ~cond * 1e-16 relative, orders below the f32 quantisation of the transform.  Whenever a determinant is small against the
// products it is summed from (cancellation = ill-conditioning), the refinement step below reports more than ~1e-10 of
// error (cond(H) >~ 1e6), or anything is not finite, the machine falls back to the JacobiSVD with Eigen's rank threshold,
// whose minimum-norm semantics then matter.  Both drivers use this rule.  Two different solvers agree only to ~cond * 1e-16:
// driven by the oracle's evaluations on thousands of fuzzed problems (tests/ndt_machine_host.cpp), the machine takes the
// oracle's iteration counts but ends one f32 ulp away in some entry of the transform in ~1.5 % of the aligns (rarely more);
// with `exact_solve` every step goes through the JacobiSVD restatement and all of them are bit-identical.
// H: row-major 6x6; b: right-hand side; x: solution.

// adjugate (row-major) and determinant of a 3x3; false when the determinant cancels
LGS_HD bool mat3_adjugate(const double* a, double* adj, double* det) {
  adj[0] = a[4] * a[8] - a[5] * a[7];
  adj[1] = a[2] * a[7] - a[1] * a[8];
  adj[2] = a[1] * a[5] - a[2] * a[4];
  adj[3] = a[5] * a[6] - a[3] * a[8];
  adj[4] = a[0] * a[8] - a[2] * a[6];
  adj[5] = a[2] * a[3] - a[0] * a[5];
  adj[6] = a[3] * a[7] - a[4] * a[6];
  adj[7] = a[1] * a[6] - a[0] * a[7];
  adj[8] = a[0] * a[4] - a[1] * a[3];
  const double t0 = a[0] * adj[0], t1 = a[1] * adj[3], t2 = a[2] * adj[6];
  *det = (t0 + t1) + t2;
  const double mag = (fabs(t0) + fabs(t1)) + fabs(t2);
  return fabs(*det) > 1e-10 * mag && mag < 1.7976931348623157e308;  // NaN fails the first comparison
}
LGS_HD void mat3_mul_vec(const double* m, const double* v, double* out) {
  out[0] = (m[0] * v[0] + m[1] * v[1]) + m[2] * v[2];
  out[1] = (m[3] * v[0] + m[4] * v[1]) + m[5] * v[2];
  out[2] = (m[6] * v[0] + m[7] * v[1]) + m[8] * v[2];
}
struct Schur6 {
  double Ai[9], W[3][3], Si[9];  // A^-1, A^-1 B, S^-1
};
LGS_HD bool schur_factor6(const double* H, Schur6* f) {
  const double A[9] = {H[0], H[1], H[2], H[6], H[7], H[8], H[12], H[13], H[14]};
  double adjA[9], detA;
  if (!mat3_adjugate(A, adjA, &detA)) return false;
  const double rA = 1.0 / detA;
  for (int k = 0; k < 9; k++) f->Ai[k] = adjA[k] * rA;
  for (int c = 0; c < 3; c++) {  // column c of B = H[0..2][3 + c]
    const double col[3] = {H[3 + c], H[6 + 3 + c], H[12 + 3 + c]};
    double w[3];
    mat3_mul_vec(f->Ai, col, w);
    f->W[0][c] = w[0];
    f->W[1][c] = w[1];
    f->W[2][c] = w[2];
  }
  double S[9];  // D - C W   (C = H[3..5][0..2])
  for (int i = 0; i < 3; i++) {
    const double* ci = H + (3 + i) * 6;
    for (int j = 0; j < 3; j++) S[i * 3 + j] = ci[3 + j] - ((ci[0] * f->W[0][j] + ci[1] * f->W[1][j]) + ci[2] * f->W[2][j]);
  }
  double adjS[9], detS;
  if (!mat3_adjugate(S, adjS, &detS)) return false;
  const double rS = 1.0 / detS;
  for (int k = 0; k < 9; k++) f->Si[k] = adjS[k] * rS;
  return true;
}
LGS_HD void schur_apply6(const double* H, const Schur6& f, const double* b, double* x) {
  double u[3], r[3];
  mat3_mul_vec(f.Ai, b, u);
  for (int i = 0; i < 3; i++) {
    const double* ci = H + (3 + i) * 6;
    r[i] = b[3 + i] - ((ci[0] * u[0] + ci[1] * u[1]) + ci[2] * u[2]);
  }
  mat3_mul_vec(f.Si, r, x + 3);
  for (int i = 0; i < 3; i++) x[i] = u[i] - ((f.W[i][0] * x[3] + f.W[i][1] * x[4]) + f.W[i][2] * x[5]);
}
// Elimination without pivoting loses the digits the determinants cancel (at most ten under mat3_adjugate's rule): one step of iterative refinement on the f64 residual brings the solution back to ~cond * 1e-16.
LGS_HD bool schur_solve6(const double* H, const double* b, double* x) {
  Schur6 f;
  if (!schur_factor6(H, &f)) return false;
  schur_apply6(H, f, b, x);
  double res[6], dx[6];
  for (int i = 0; i < 6; i++) {
    const double* h = H + i * 6;
    res[i] = b[i] - (((h[0] * x[0] + h[1] * x[1]) + (h[2] * x[2] + h[3] * x[3])) + (h[4] * x[4] + h[5] * x[5]));
  }
  schur_apply6(H, f, res, dx);
  // the correction measures the error of the first solve, ~cond(H) * 1e-16: two different algorithms agree on the solution
  // of an ill-conditioned system only to that much, and past ~1e-10 the difference to the reference's JacobiSVD starts to
  // reach the f32 transform (measured on a fuzzed align with cond(H) = 4e8: another iteration count).  Such systems go to
  // the JacobiSVD restatement, which repeats the reference's operations.
  double n_dx = 0, n_x = 0;
  for (int i = 0; i < 6; i++) {
    n_dx += dx[i] * dx[i];
    n_x += x[i] * x[i];
  }
  if (!(n_dx <= 1e-20 * n_x)) return false;
  for (int i = 0; i < 6; i++) x[i] += dx[i];
  for (int i = 0; i < 6; i++)
    if (!(fabs(x[i]) < 1.7976931348623157e308)) return false;
  return true;
}

// JacobiSVD with Eigen's rank threshold, as the reference; out of line on the device (rare, large stack frame).  inline:
// several translation units include this header.
#if defined(__CUDACC__)
__host__ __device__ __noinline__ inline
#else
inline
#endif
void svd_fallback(const double* H, const double* b, double* x) {
  m::svd_solve<6>(H, b, x);
}

// where the evaluation kernels leave entry (i,j) of the Hessian in their row of sums (mode 0): the upper triangle row by
// row from 7, the strict lower triangle row by row from 28
LGS_HD int hess_sum_index(int i, int j) { return i <= j ? 7 + i * 6 - (i * (i - 1)) / 2 + (j - i) : 28 + (i * (i - 1)) / 2 + j; }

// ---- the pose of the guess (host only: once per align) ------------------------------------------------------------
// p = [translation, eulerAngles(0,1,2)] of an Affine3f (NDT:103-111): rotation() is the polar factor
// U V^T of the linear part (f32 Jacobi SVD), then Eigen's eulerAngles branch convention.
inline void matrix_to_pose(const float* T, double p[6]) {
  float L[9], U[9], S[3], V[9], UVt[9], R[9];
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) L[r * 3 + c] = T[c * 4 + r];
  m::svd_jacobi<3, float>(L, U, S, V);
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) UVt[i * 3 + j] = (U[i * 3] * V[j * 3] + U[i * 3 + 1] * V[j * 3 + 1]) + U[i * 3 + 2] * V[j * 3 + 2];
  float det = UVt[0] * (UVt[4] * UVt[8] - UVt[5] * UVt[7]) - UVt[1] * (UVt[3] * UVt[8] - UVt[5] * UVt[6]) +
              UVt[2] * (UVt[3] * UVt[7] - UVt[4] * UVt[6]);
  float sgn = det < 0.0f ? -1.0f : 1.0f;
  for (int r = 0; r < 3; r++) U[r * 3 + 2] *= sgn;
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) R[i * 3 + j] = (U[i * 3] * V[j * 3] + U[i * 3 + 1] * V[j * 3 + 1]) + U[i * 3 + 2] * V[j * 3 + 2];
  const float pi = static_cast<float>(M_PI);
  float r0 = std::atan2(R[1 * 3 + 2], R[2 * 3 + 2]);
  float c2 = std::sqrt(R[0] * R[0] + R[1] * R[1]);
  float r1;
  if (r0 > 0.0f) {
    r0 -= pi;
    r1 = std::atan2(-R[2], -c2);
  } else {
    r1 = std::atan2(-R[2], c2);
  }
  float s1 = std::sin(r0), c1 = std::cos(r0);
  float r2 = std::atan2(s1 * R[2 * 3 + 0] - c1 * R[1 * 3 + 0], c1 * R[1 * 3 + 1] - s1 * R[2 * 3 + 1]);
  p[0] = T[12];
  p[1] = T[13];
  p[2] = T[14];
  p[3] = -r0;
  p[4] = -r1;
  p[5] = -r2;
}

// ---- the machine ------------------------------------------------------------------------------------------------------
struct Command {       // the evaluation to run next
  int mode;            // 0: score + g + H (f32 terms), 1: score + g, 2: computeHessian in f64; < 0: the align is done
  float T[16];         // column-major transform applied to the source points
  float j_ang[8][3];   // NDT:339-346, f32
  float h_ang[15][3];  // NDT:373-392, f32
  double j_ang_d[8][3];
  double h_ang_d[15][3];
};

enum Action { kDone = 0, kSolve = 1, kPose = 2, kHessian = 3 };

struct Machine {
  // parameters
  double step_size, trans_eps, n_in;
  int max_iter;
  int exact_solve;  // every Newton step through the JacobiSVD restatement (lgs_ndt_set_exact_newton_step / LGS_NDT_EXACT_SOLVE=1)
  // optimiser state (NDT:103-171)
  double p[6], score, g[6], H[36];  // H: row-major, both triangles (see "Newton step")
  int nr_iterations, converged, early_exit;
  double trans_probability;
  int evals, trials, hess_recomputes;
  float final_T[16];
  // line-search state (NDT:771-931)
  double dir[6], x_t[6];
  double phi_0, d_phi_0, a_l, f_l, g_l, a_u, f_u, g_u, a_t, step_min, step_max;
  double phi_t, d_phi_t, psi_t, d_psi_t;
  int interval_converged, open_interval, step_iterations;
  int pending;  // what the evaluation in flight is: 0 initial (NDT:119), 1 first of a line search, 2 trial, 3 computeHessian
  double delta_p[6];  // solution of the Newton system
  // work areas of the steps a driver may run in parallel
  int pose_mode;  // kPose: evaluation mode of the pose x_t
  Trig trig;
  float Rx[9], Ry[9], Rz[9], Rxy[9], R[9];
  unsigned codes[69];  // angle_codes, next to the state (see there)

  // NDT:103-119: the first evaluation, at the pose of the guess (T0 = the guess itself, p0 its translation + Euler angles)
  LGS_HD void begin(const double p0[6], const float T0[16], double step_size_, double trans_eps_, int max_iter_, double n_in_, Command* c,
                    int exact_solve_ = 0) {
    exact_solve = exact_solve_;
    step_size = step_size_;
    trans_eps = trans_eps_;
    max_iter = max_iter_;
    n_in = n_in_;
    for (int i = 0; i < 6; i++) p[i] = p0[i];
    for (int i = 0; i < 16; i++) final_T[i] = T0[i];
    score = 0;
    for (int i = 0; i < 6; i++) g[i] = 0;
    for (int i = 0; i < 36; i++) H[i] = 0;
    nr_iterations = converged = early_exit = 0;
    trans_probability = 0;
    evals = 1;
    trials = hess_recomputes = 0;
    pending = 0;
    trig_of_pose(p0, &trig);
    for (int i = 0; i < 16; i++) c->T[i] = T0[i];
    angle_codes(codes);
    for (int e = 0; e < 69; e++) angle_table_store(trig, codes, e, c->j_ang_d, c->h_ang_d, c->j_ang, c->h_ang);
    c->mode = 0;
  }

  LGS_HD void take_sums(const double* s, int mode) {
    // mode 0: score, g[6], upper triangle of H (21), strict lower triangle (15); mode 1: score, g[6]; mode 2: upper
    // triangle of the f64 Hessian (computeHessian's two triangles differ by f64 rounding only: mirrored).  (The reference
    // zeroes H in a gradient-only evaluation, NDT:201; computeHessian always overwrites it before its next use, NDT:927.)
    if (mode == 2) {
      int k = 0;
      for (int i = 0; i < 6; i++)
        for (int j = i; j < 6; j++) H[i * 6 + j] = H[j * 6 + i] = s[k++];
      return;
    }
    score = s[0];
    for (int i = 0; i < 6; i++) g[i] = s[1 + i];
    if (mode == 0)
      for (int i = 0; i < 6; i++)
        for (int j = 0; j < 6; j++) H[i * 6 + j] = s[hess_sum_index(i, j)];
  }

  // NDT:127-129
  LGS_HD void solve() {
    double neg_g[6];
    for (int i = 0; i < 6; i++) neg_g[i] = -g[i];
    if (exact_solve) {  // the reference's own solver for every step (see "Newton step"): bit-identical paths, ~20x the time
      svd_fallback(H, neg_g, delta_p);
      return;
    }
    if (schur_solve6(H, neg_g, delta_p)) return;
    svd_fallback(H, neg_g, delta_p);
  }
  LGS_HD int request_pose(int mode) {
    for (int i = 0; i < 6; i++) x_t[i] = p[i] + dir[i] * a_t;
    pose_mode = mode;
    evals++;
    pending = mode == 0 ? 1 : 2;
    return kPose;
  }
  // NDT:144-162 after a line search that returned `step`; then the next Newton step or the end
  LGS_HD int outer_update(double step) {
    for (int i = 0; i < 6; i++) p[i] = p[i] + dir[i] * step;
    if (nr_iterations > max_iter || (nr_iterations && (fabs(step) < trans_eps))) converged = 1;
    nr_iterations++;
    if (converged) {
      trans_probability = score / n_in;  // NDT:170
      return kDone;
    }
    return kSolve;
  }

  // Feeds the sums of the pending evaluation.  kSolve: call solve, then after_solve.  kPose: build the
  // transform and the tables of x_t (build_pose), mode pose_mode.  kHessian: computeHessian at the pose of the last
  // command (its transform and tables are re-used).  kDone: results in nr_iterations / converged / trans_probability /
  // final_T / p.
  LGS_HD int consume(const double* sums) {
    const double mu = 1.e-4, nu = 0.9;
    const int max_step_iterations = 10;
    if (pending == 0) {
      take_sums(sums, 0);
      return kSolve;
    }
    if (pending == 3) {
      take_sums(sums, 2);
      return outer_update(a_t);
    }
    take_sums(sums, pending == 1 ? 0 : 1);
    phi_t = -score;
    d_phi_t = -dot6(g, dir);
    psi_t = phi_t - phi_0 - mu * d_phi_0 * a_t;
    d_psi_t = d_phi_t - mu * d_phi_0;
    if (pending == 2) {
      if (open_interval && (psi_t <= 0 && d_psi_t >= 0)) {
        open_interval = 0;
        f_l = f_l + phi_0 - mu * d_phi_0 * a_l;
        g_l = g_l + mu * d_phi_0;
        f_u = f_u + phi_0 - mu * d_phi_0 * a_u;
        g_u = g_u + mu * d_phi_0;
      }
      if (open_interval)
        interval_converged = update_interval(a_l, f_l, g_l, a_u, f_u, g_u, a_t, psi_t, d_psi_t) ? 1 : 0;
      else
        interval_converged = update_interval(a_l, f_l, g_l, a_u, f_u, g_u, a_t, phi_t, d_phi_t) ? 1 : 0;
      step_iterations++;
    }
    // the loop condition of NDT:861
    if (!interval_converged && step_iterations < max_step_iterations && !(psi_t <= 0 && d_phi_t <= -nu * d_phi_0)) {
      trials++;
      if (open_interval)
        a_t = trial_value(a_l, f_l, g_l, a_u, f_u, g_u, a_t, psi_t, d_psi_t);
      else
        a_t = trial_value(a_l, f_l, g_l, a_u, f_u, g_u, a_t, phi_t, d_phi_t);
      a_t = std_max(std_min(a_t, step_max), step_min);
      return request_pose(1);
    }
    if (step_iterations) {  // NDT:927-928: the line search iterated, re-evaluate the Hessian in f64 at x_t
      hess_recomputes++;
      pending = 3;
      return kHessian;
    }
    return outer_update(a_t);
  }

  // with the Newton step in delta_p: NDT:130-139, then computeStepLengthMT (NDT:771-931) up to its first evaluation
  LGS_HD int after_solve() {
    const double mu = 1.e-4;
    const double delta_p_norm = sqrt(dot6(delta_p, delta_p));
    if (delta_p_norm == 0 || delta_p_norm != delta_p_norm) {
      trans_probability = score / n_in;
      converged = delta_p_norm == delta_p_norm ? 1 : 0;
      early_exit = 1;
      return kDone;
    }
    for (int i = 0; i < 6; i++) dir[i] = delta_p[i] / delta_p_norm;
    step_max = step_size;
    step_min = trans_eps / 2;
    phi_0 = -score;
    d_phi_0 = -dot6(g, dir);
    if (d_phi_0 >= 0) {
      if (d_phi_0 == 0) return outer_update(0.0);  // NDT:790-791: no step
      d_phi_0 *= -1;
      for (int i = 0; i < 6; i++) dir[i] *= -1;
    }
    step_iterations = 0;
    a_l = 0;
    a_u = 0;
    f_l = phi_0 - phi_0 - mu * d_phi_0 * a_l;  // auxiliaryFunction_PsiMT (NDT.h:430-436)
    g_l = d_phi_0 - mu * d_phi_0;              // auxiliaryFunction_dPsiMT (NDT.h:438-447)
    f_u = phi_0 - phi_0 - mu * d_phi_0 * a_u;
    g_u = d_phi_0 - mu * d_phi_0;
    interval_converged = (step_max - step_min) < 0 ? 1 : 0;
    open_interval = 1;
    a_t = std_max(std_min(delta_p_norm, step_max), step_min);
    return request_pose(0);
  }

  // kPose in three stages a driver may spread over threads (every index of a stage is independent of the others):
  //   stage 0: trig_value(x_t, k, &trig), k = 0..11
  //   stage 1: pose_stage1(i), i = 0..2 (the three axis rotations) and angle_table_store(trig, codes, e, ...), e = 0..68
  //   stage 2: pose_stage2(i), i = 0..8 (Rx * Ry);  stage 3: pose_stage3(i), i = 0..8 ((Rx * Ry) * Rz);  stage 4: pose_stage4(i), i = 0..15
  LGS_HD void pose_stage1(int i) {
    if (i == 0) angle_axis_unit<0>(trig.sf[0], trig.cf[0], Rx);
    else if (i == 1) angle_axis_unit<1>(trig.sf[1], trig.cf[1], Ry);
    else angle_axis_unit<2>(trig.sf[2], trig.cf[2], Rz);
  }
  LGS_HD void pose_stage2(int i) { Rxy[i] = mul3f_entry(Rx, Ry, i / 3, i % 3); }
  LGS_HD void pose_stage3(int i) { R[i] = mul3f_entry(Rxy, Rz, i / 3, i % 3); }
  // stages 1-4 for ONE entry of the transform without any exchange between threads: thread i (0..15) builds the three axis
  // rotations and row (i & 3) of Rx * Ry in registers - redundantly, with the functions the staged form calls, so the bits
  // are the same - and finishes its own entry.  No barriers, no shared-memory round trips: the dependency chain is what counts
  // on a GPU thread.
  LGS_HD void pose_entry(int i, Command* c) {
    const int col = i >> 2, row = i & 3;
    float v = (i % 5 == 0) ? 1.0f : 0.0f;
    if (row < 3 && col < 3) {
      float ax_[9], ay_[9], az_[9];
      angle_axis_unit<0>(trig.sf[0], trig.cf[0], ax_);
      angle_axis_unit<1>(trig.sf[1], trig.cf[1], ay_);
      angle_axis_unit<2>(trig.sf[2], trig.cf[2], az_);
      float rxy[9];
      rxy[row * 3 + 0] = mul3f_entry(ax_, ay_, row, 0);
      rxy[row * 3 + 1] = mul3f_entry(ax_, ay_, row, 1);
      rxy[row * 3 + 2] = mul3f_entry(ax_, ay_, row, 2);
      v = mul3f_entry(rxy, az_, row, col);
    }
    if (col == 3 && row < 3) v = static_cast<float>(x_t[row]);
    final_T[i] = v;
    c->T[i] = v;
    if (i == 0) c->mode = pose_mode;
  }
  LGS_HD void pose_stage4(int i, Command* c) {  // entry i of the column-major transform (NDT.h:214-231); i = 0..15
    const int col = i >> 2, row = i & 3;
    float v = (i % 5 == 0) ? 1.0f : 0.0f;
    if (row < 3 && col < 3) v = R[row * 3 + col];
    if (col == 3 && row < 3) v = static_cast<float>(x_t[row]);
    final_T[i] = v;
    c->T[i] = v;
    if (i == 0) c->mode = pose_mode;
  }

  // the whole step on one thread (host driver): returns true and fills *c when another evaluation is needed.  *c must be
  // the object the previous call (or begin) filled: computeHessian re-uses its transform and tables.
  LGS_HD bool advance(const double* sums, Command* c) {
    int action = consume(sums);
    while (action == kSolve) {
      solve();
      action = after_solve();
    }
    if (action == kDone) return false;
    if (action == kHessian) {
      c->mode = 2;
      return true;
    }
    trig_of_pose(x_t, &trig);
    for (int i = 0; i < 3; i++) pose_stage1(i);
    for (int e = 0; e < 69; e++) angle_table_store(trig, codes, e, c->j_ang_d, c->h_ang_d, c->j_ang, c->h_ang);
    for (int i = 0; i < 9; i++) pose_stage2(i);
    for (int i = 0; i < 9; i++) pose_stage3(i);
    for (int i = 0; i < 16; i++) pose_stage4(i, c);
    return true;
  }
};

}  // namespace ndtopt
}  // namespace lgs
