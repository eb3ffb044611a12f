// Compile-and-link check of the C++ multi-align entry points of include/lgs/registration.hpp (alignGuesses, alignMany) against
// liblgs_b200.so.  With --run (needs a GPU) every record is compared bitwise with the single align from the same guess.
#include <cmath>
#include <cstdio>
#include <cstring>

#include "lgs/registration.hpp"

static bool same(const lgs_align_result& a, const lgs_align_result& b) {
  return std::memcmp(a.T, b.T, sizeof(a.T)) == 0 && std::memcmp(&a.trans_probability, &b.trans_probability, sizeof(double)) == 0 &&
         a.iterations == b.iterations && a.converged == b.converged && a.evaluations == b.evaluations &&
         a.line_search_trials == b.line_search_trials && a.hessian_recomputes == b.hessian_recomputes;
}

int main(int argc, char** argv) {
  const bool run = argc > 1 && std::strcmp(argv[1], "--run") == 0;
  if (!run) {
    std::printf("shim compiled; version %s\n", lgs_version());
    return 0;
  }
  auto target = std::make_shared<lgs::PointCloud>();
  for (int i = 0; i < 20000; i++) {
    const float a = 0.0005f * i;
    target->push_back(lgs::PointXYZI{10.0f * std::cos(a) + 0.3f * std::sin(7 * a), 10.0f * std::sin(a), 0.0001f * (i % 997), 1.0f, 0, 0, 0, 0});
  }
  auto source = std::make_shared<lgs::PointCloud>();
  for (size_t i = 0; i < target->size(); i += 3) source->push_back((*target)[i]);
  lgs::NormalDistributionsTransform a, b, single;
  for (auto* x : {&a, &b, &single}) {
    x->setResolution(1.0f);
    x->setTransformationEpsilon(0.01);
    x->setMaximumIterations(64);
    x->setInputTarget(target);
    x->setInputSource(source);
  }
  std::vector<lgs::Matrix4f> guesses;
  for (int k = 0; k < 5; k++) {
    lgs::Matrix4f T = lgs::Identity4f();
    const float yaw = 0.01f * (k - 2);
    T[0] = T[5] = std::cos(yaw);
    T[1] = std::sin(yaw);
    T[4] = -T[1];
    T[12] = 0.1f * k;
    T[13] = -0.05f * k;
    guesses.push_back(T);
  }
  const auto rec = a.alignGuesses(guesses, 1.0);
  if (!a.hasConverged() || rec.size() != guesses.size()) return 1;
  lgs::PointCloud out;
  for (size_t k = 0; k < guesses.size(); k++) {
    single.align(out, guesses[k]);
    if (!same(rec[k], single.result()) || rec[k].pair_id != static_cast<int>(k) || rec[k].fitness != single.getFitnessScore(1.0)) return 2;
  }
  const auto many = lgs::alignMany({&a, &b, &a}, {guesses[0], guesses[1], guesses[2]});
  if (many.size() != 3 || !same(many[0], rec[0]) || !same(many[1], rec[1]) || !same(many[2], rec[2])) return 3;
  if (!same(a.result(), rec[2]) || !same(b.result(), rec[1])) return 4;
  std::printf("align_many ok: %zu seeds, iterations", rec.size());
  for (const auto& r : rec) std::printf(" %d", r.iterations);
  std::printf("\n");
  return 0;
}
