// hp_gibbs.cpp -- batch_scorer::hp_gibbs from C++: a fixed (bool, uint32, float) dataset in 3 groups, a grid on every
// feature and on alpha, one Gibbs step.  Prints the drawn indices ([D + 1], alpha last) on one line; tests/test_gpu_hyper.py
// builds the same state through Python and compares.
//
//   hp_gibbs <seed> <counter>
#include <cstdio>
#include <cstdlib>

#include "microscopes_b200/gpu_models.hpp"

using namespace microscopes;
using namespace microscopes::common;
using namespace microscopes::models;

int main(int argc, char **argv) {
  if (argc < 3) { std::fprintf(stderr, "usage: hp_gibbs <seed> <counter>\n"); return 2; }
  const uint64_t seed = std::strtoull(argv[1], nullptr, 10), counter = std::strtoull(argv[2], nullptr, 10);
  const size_t N = 90, K = 3;
  struct __attribute__((packed)) rec { bool b; uint32_t c; float f; };
  std::vector<rec> rows(N);
  std::vector<int64_t> z(N);
  for (size_t i = 0; i < N; i++) {  // the formula the test restates
    rows[i].b = (i * 7) % 10 < 3 + 2 * (i % K);
    rows[i].c = (uint32_t)((i * 13) % 9 + 3 * (i % K));
    rows[i].f = (float)(i % K) + 0.125f * (float)(i % 7);
    z[i] = (int64_t)(i % K);
  }
  std::vector<runtime_type> t = {runtime_type(TYPE_B), runtime_type(TYPE_U32), runtime_type(TYPE_F32)};
  std::vector<std::shared_ptr<gpu_model>> ms = {std::make_shared<gpu_model>(MSB_FAMILY_BB), std::make_shared<gpu_model>(MSB_FAMILY_GP),
                                               std::make_shared<gpu_model>(MSB_FAMILY_NICH)};
  try {
    batch_scorer bs(ms, reinterpret_cast<const uint8_t *>(rows.data()), nullptr, N, t, K + 1);
    bs.set_alpha(1.0);
    for (size_t k = 0; k < K; k++) bs.create_group();
    bs.add_values(z);
    bs.set_hp_grid(0, {0.5, 0.5, 1.0, 1.0, 2.0, 3.0}, {0.0, -0.5, -1.0});
    bs.set_hp_grid(1, {1.0, 1.0, 2.0, 0.5, 4.0, 1.0, 0.5, 2.0}, {0.0, 0.0, -0.25, 0.1});
    bs.set_hp_grid(2, {0.0, 1.0, 1.0, 1.0, 1.0, 0.5, 2.0, 3.0}, {0.0, 0.0});
    bs.set_cluster_hp_grid({0.25, 1.0, 4.0, 16.0}, {0.0, 0.0, 0.0, -2.0});
    const std::vector<int64_t> c = bs.hp_gibbs(seed, counter);
    for (size_t i = 0; i < c.size(); i++) std::printf("%s%lld", i ? " " : "", (long long)c[i]);
    std::printf("\n");
  } catch (const std::runtime_error &e) {
    std::printf("error %s\n", e.what());
    return 1;
  }
  return 0;
}
