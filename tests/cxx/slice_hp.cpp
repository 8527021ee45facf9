// slice_hp.cpp -- batch_scorer::slice_hp from C++: a fixed three-feature (bb, gp, nich) dataset in 3 groups plus one empty
// group, then one slice_hp(specs, seed, counter) over bb's (alpha, beta) under the non-informative prior, gp's inv_beta,
// nich's mu and nu, and alpha.  Prints the bits of each spec's value as unsigned integers on one line;
// tests/test_gpu_hpslice.py builds the same state through Python and compares.
//
//   slice_hp <seed> <counter>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "microscopes_b200/gpu_models.hpp"

using namespace microscopes;
using namespace microscopes::common;
using namespace microscopes::models;

static msb_slice_hp_spec spec(size_t feature, const char *key, double width, int32_t prior, double a, double b) {
  msb_slice_hp_spec s;
  s.feature = feature; s.key = key; s.width = width; s.prior = prior; s.a = a; s.b = b;
  return s;
}

int main(int argc, char **argv) {
  if (argc < 3) { std::fprintf(stderr, "usage: slice_hp <seed> <counter>\n"); return 2; }
  const uint64_t seed = std::strtoull(argv[1], nullptr, 10), counter = std::strtoull(argv[2], nullptr, 10);
  const size_t N = 90, K = 3;
  struct __attribute__((packed)) rec { bool f0; uint32_t f1; float f2; };
  std::vector<rec> rows(N);
  std::vector<int64_t> z(N);
  for (size_t i = 0; i < N; i++) {  // the formula the test restates
    rows[i].f0 = (i * 7) % 10 < 3 + 2 * (i % K);
    rows[i].f1 = (uint32_t)((i * 13) % 9 + 3 * (i % K));
    rows[i].f2 = (float)((double)(i % K) + 0.125 * (double)(i % 7));
    z[i] = (int64_t)(i % K);
  }
  std::vector<runtime_type> t = {runtime_type(TYPE_B), runtime_type(TYPE_U32), runtime_type(TYPE_F32)};
  std::vector<std::shared_ptr<gpu_model>> ms = {std::make_shared<gpu_model>(MSB_FAMILY_BB), std::make_shared<gpu_model>(MSB_FAMILY_GP),
                                               std::make_shared<gpu_model>(MSB_FAMILY_NICH)};
  try {
    batch_scorer bs(ms, reinterpret_cast<const uint8_t *>(rows.data()), nullptr, N, t, K + 1);
    bs.set_alpha(1.0);
    std::vector<size_t> gids;
    for (size_t k = 0; k <= K; k++) gids.push_back(bs.create_group());  // the last one stays empty
    bs.add_values(z);
    const std::vector<msb_slice_hp_spec> specs = {
        spec(0, "alpha", 1.0, MSB_HPRIOR_NONINFORMATIVE_BETA, 0.0, 0.0), spec(0, "beta", 1.0, MSB_HPRIOR_NONINFORMATIVE_BETA, 0.0, 0.0),
        spec(1, "inv_beta", 0.5, MSB_HPRIOR_EXPONENTIAL, 2.0, 0.0), spec(2, "mu", 0.25, MSB_HPRIOR_NORMAL, 0.5, 2.0),
        spec(2, "nu", 2.0, MSB_HPRIOR_FLAT, 0.5, 30.0), spec(3, "alpha", 1.0, MSB_HPRIOR_EXPONENTIAL, 1.0, 0.0)};
    size_t capped = 0;
    const std::vector<double> v = bs.slice_hp(specs, seed, counter, &capped);
    for (size_t i = 0; i < v.size(); i++) {
      uint64_t bits;
      std::memcpy(&bits, &v[i], sizeof(bits));
      std::printf("%s%llu", i ? " " : "", (unsigned long long)bits);
    }
    std::printf("\n");
  } catch (const std::runtime_error &e) {
    std::printf("error %s\n", e.what());
    return 1;
  }
  return 0;
}
