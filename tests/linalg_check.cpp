// The small dense solvers of csrc/math.cuh and csrc/ndt_opt.cuh compiled for the host, behind the op codes and layouts of
// lgs_linalg_batch (include/lgs_c.h), as a shared library for ctypes.  tests/test_linalg_reference.py compares it bit for
// bit with the oracle's Eigen restatement; tests/test_gpu_linalg.py compares the device's Schur / Newton steps with it.
//   g++ -O2 -std=c++17 -ffp-contract=off -fPIC -shared -I lidar_graph_slam_b200/csrc tests/linalg_check.cpp -o liblinalg_check.so
// Besides the device ops 0..5 it has the host-only uses of the header: 16 = svd_jacobi<3, float> (ICP's Umeyama,
// matrix_to_pose; inputs rounded to float, results widened exactly) and 17 = ldlt_solve6 (the LM step).
#include <cstring>

#include "ndt_opt.cuh"

extern "C" int linalg_check_batch(int op, long n, const double* in, double* out) {
  using namespace lgs;
  int nin, nout;
  switch (op) {
    case 0: case 16: nin = 9; nout = 21; break;
    case 1: nin = 9; nout = 13; break;
    case 2: nin = 9; nout = 9; break;
    case 3: case 17: nin = 42; nout = 6; break;
    case 4: nin = 42; nout = 7; break;
    case 5: nin = 42; nout = 12; break;
    default: return -1;
  }
  for (long t = 0; t < n; t++) {
    const double* a = in + t * nin;
    double* o = out + t * nout;
    switch (op) {
      case 0: m::svd_jacobi<3, double>(a, o, o + 9, o + 12); break;
      case 1: o[12] = m::eig_sym3(a, o, o + 3) ? 1.0 : 0.0; break;
      case 2: m::inv3(a, o); break;
      case 3: m::svd_solve<6>(a, a + 36, o); break;
      case 4: {
        for (int i = 0; i < 6; i++) o[i] = 0.0;
        o[6] = ndtopt::schur_solve6(a, a + 36, o) ? 1.0 : 0.0;
        break;
      }
      case 5: {
        ndtopt::Machine mc;
        std::memcpy(mc.H, a, sizeof(mc.H));
        for (int i = 0; i < 6; i++) mc.g[i] = -a[36 + i];
        for (int e = 0; e < 2; e++) {
          mc.exact_solve = e;
          mc.solve();
          for (int i = 0; i < 6; i++) o[6 * e + i] = mc.delta_p[i];
        }
        break;
      }
      case 16: {
        float af[9], U[9], S[3], V[9];
        for (int i = 0; i < 9; i++) af[i] = static_cast<float>(a[i]);
        m::svd_jacobi<3, float>(af, U, S, V);
        for (int i = 0; i < 9; i++) o[i] = U[i];
        for (int i = 0; i < 3; i++) o[9 + i] = S[i];
        for (int i = 0; i < 9; i++) o[12 + i] = V[i];
        break;
      }
      default: m::ldlt_solve6(a, a + 36, o); break;
    }
  }
  return 0;
}
