// theta.cpp -- batch_scorer::redraw_empty and batch_scorer::theta from C++: a fixed three-feature (bbnc, bb, bbnc) boolean
// dataset in 3 groups plus one empty group, redraw_empty(seed, counter), then theta(widths, seed, counter + 1).  Prints
// the bits of every group's p (feature 0, then feature 2; ascending gid) as unsigned integers on one line;
// tests/test_gpu_theta.py builds the same state through Python and compares.
//
//   theta <seed> <counter>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "microscopes_b200/gpu_models.hpp"

using namespace microscopes;
using namespace microscopes::common;
using namespace microscopes::models;

int main(int argc, char **argv) {
  if (argc < 3) { std::fprintf(stderr, "usage: theta <seed> <counter>\n"); return 2; }
  const uint64_t seed = std::strtoull(argv[1], nullptr, 10), counter = std::strtoull(argv[2], nullptr, 10);
  const size_t N = 90, K = 3;
  struct __attribute__((packed)) rec { bool f0, f1, f2; };
  std::vector<rec> rows(N);
  std::vector<int64_t> z(N);
  for (size_t i = 0; i < N; i++) {  // the formula the test restates
    rows[i].f0 = (i * 7) % 10 < 3 + 2 * (i % K);
    rows[i].f1 = (i * 13) % 9 < 2 + 3 * (i % K);
    rows[i].f2 = (i * 5) % 11 < 4;
    z[i] = (int64_t)(i % K);
  }
  std::vector<runtime_type> t = {runtime_type(TYPE_B), runtime_type(TYPE_B), runtime_type(TYPE_B)};
  std::vector<std::shared_ptr<gpu_model>> ms = {std::make_shared<gpu_model>(MSB_FAMILY_BBNC), std::make_shared<gpu_model>(MSB_FAMILY_BB),
                                               std::make_shared<gpu_model>(MSB_FAMILY_BBNC)};
  try {
    batch_scorer bs(ms, reinterpret_cast<const uint8_t *>(rows.data()), nullptr, N, t, K + 2);
    bs.set_alpha(1.0);
    const double a = 2.0, b = 0.5;  // before create_group: the groups' first p is drawn from these
    b200::check(msb_state_set_hp(bs.handle(), 0, "alpha", &a, 1));
    b200::check(msb_state_set_hp(bs.handle(), 0, "beta", &b, 1));
    std::vector<size_t> gids;
    for (size_t k = 0; k <= K; k++) gids.push_back(bs.create_group());  // the last one stays empty
    bs.add_values(z);
    bs.redraw_empty(seed, counter);
    bs.theta({0.25, 0.0, 1.5}, seed, counter + 1);
    bool first = true;
    for (size_t d : {0, 2})
      for (size_t g : gids) {
        double p;
        b200::check(msb_state_get_ss(bs.handle(), d, g, "p", &p, 1));
        uint64_t bits;
        std::memcpy(&bits, &p, sizeof(bits));
        std::printf("%s%llu", first ? "" : " ", (unsigned long long)bits);
        first = false;
      }
    std::printf("\n");
  } catch (const std::runtime_error &e) {
    std::printf("error %s\n", e.what());
    return 1;
  }
  return 0;
}
