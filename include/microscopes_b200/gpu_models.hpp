// gpu_models.hpp -- C++ host adapters over the C ABI (include/mscope_b200.h).
//
//   gpu_model / gpu_hypers / gpu_group implement the reference's plugin interface
//   (include/microscopes/models/base.hpp:21-62) the way distributions_model<T> /
//   distributions_hypers<T> / distributions_group<T> do
//   (include/microscopes/models/distributions.hpp:256-509): the hypers and the group
//   own their field vectors on the host, exposed through get_hp_mutator / get_ss_mutator
//   with the reference's key names, and every score_value / add_value / remove_value is
//   evaluated ON THE DEVICE through msb_value_score / msb_value_add / msb_value_remove.
//   There is no host arithmetic and no CPU fallback.
//
//   batch_scorer is the data-parallel form of the same loop: one row_major_dataview-shaped
//   record array, K groups x D features, scored / swept in one call.
//
// Header-only; link with -lmscope_b200.
#pragma once

#include <algorithm>
#include <cstring>
#include <map>
#include <sstream>

#include "../mscope_b200.h"
#include "plugin_api.hpp"
#include "wire.hpp"

namespace microscopes {
namespace models {

namespace b200 {

inline void check(int status) {
  if (status != MSB_OK) throw std::runtime_error(msb_last_error());
}

// one context per process and device, shared by every adapter object
inline msb_ctx *default_ctx(int device = 0) {
  static std::map<int, msb_ctx *> ctxs;
  auto it = ctxs.find(device);
  if (it != ctxs.end()) return it->second;
  msb_ctx *c = nullptr;
  check(msb_ctx_create(device, nullptr, &c));
  ctxs[device] = c;
  return c;
}

struct field { size_t off, cnt; };

inline field hp_field(const msb_model_desc &m, const std::string &key) {
  const size_t d = m.dim;
  switch (m.family) {
    case MSB_FAMILY_BB: if (key == "alpha") return {0, 1}; if (key == "beta") return {1, 1}; break;
    case MSB_FAMILY_BNB: if (key == "alpha") return {0, 1}; if (key == "beta") return {1, 1}; if (key == "r") return {2, 1}; break;
    case MSB_FAMILY_GP: if (key == "alpha") return {0, 1}; if (key == "inv_beta") return {1, 1}; break;
    case MSB_FAMILY_NICH:
      if (key == "mu") return {0, 1}; if (key == "kappa") return {1, 1};
      if (key == "sigmasq") return {2, 1}; if (key == "nu") return {3, 1}; break;
    case MSB_FAMILY_DD: case MSB_FAMILY_DM: if (key == "alphas") return {0, d}; break;  // dm.hpp get_hp_mutator
    case MSB_FAMILY_BBNC: if (key == "alpha") return {0, 1}; if (key == "beta") return {1, 1}; break;  // bbnc.cpp:143-153
    case MSB_FAMILY_NIW:  // beyond the reference: its generic template throws "not supported" (distributions.hpp:112-118)
      if (key == "mu") return {0, d}; if (key == "kappa") return {d, 1};
      if (key == "psi") return {d + 1, d * d}; if (key == "nu") return {d + 1 + d * d, 1}; break;
  }
  throw std::runtime_error("Unknown shared HP param key: " + key);  // distributions.hpp:140
}
inline field ss_field(const msb_model_desc &m, const std::string &key) {
  const size_t d = m.dim;
  switch (m.family) {
    case MSB_FAMILY_BB: if (key == "heads") return {0, 1}; if (key == "tails") return {1, 1}; break;
    case MSB_FAMILY_BNB: if (key == "count") return {0, 1}; if (key == "sum") return {1, 1}; break;
    case MSB_FAMILY_GP: if (key == "count") return {0, 1}; if (key == "sum") return {1, 1}; if (key == "log_prod") return {2, 1}; break;
    case MSB_FAMILY_NICH: if (key == "count") return {0, 1}; if (key == "mean") return {1, 1}; if (key == "count_times_variance") return {2, 1}; break;
    case MSB_FAMILY_DD: if (key == "count_sum") return {0, 1}; if (key == "counts") return {1, d}; break;
    case MSB_FAMILY_BBNC: if (key == "p") return {0, 1}; if (key == "heads") return {1, 1}; if (key == "tails") return {2, 1}; break;  // bbnc.cpp:107-118
    case MSB_FAMILY_DM: if (key == "counts") return {0, d}; if (key == "ratio") return {d, 1}; break;  // schema.proto:25-28
    case MSB_FAMILY_NIW: if (key == "count") return {0, 1}; if (key == "sum_x") return {1, d}; if (key == "sum_xxT") return {1 + d, d * d}; break;
  }
  throw std::runtime_error("Unknown group SS param key: " + key);  // distributions.hpp:152
}

// value_accessor hides its pointer (runtime_value.hpp:58-61): read the value the way every model does,
// through get<T>() / runtime_cast, and hand it to the ABI as doubles
struct value_f64 {
  std::vector<double> x;
  msb_runtime_type type;
  explicit value_f64(const common::value_accessor &v) : x(v.shape()) {
    for (unsigned i = 0; i < v.shape(); i++) x[i] = v.get<double>(i);
    type.prim = MSB_TYPE_F64; type.n = v.shape(); type.vec = v.shape() > 1 ? 1 : 0;
  }
};

inline msb_runtime_type abi_type(const common::runtime_type &t) {
  msb_runtime_type r;
  r.prim = (int32_t)t.t(); r.n = t.n(); r.vec = t.vec() ? 1 : 0;
  return r;
}

}  // namespace b200

class gpu_hypers;

// the field vectors are doubles: the mutators hand out TYPE_F64 views (any primitive type may
// back a field on the caller's side, runtime_cast converts: runtime_type.hpp:143-211)
class gpu_group : public group {
public:
  gpu_group(const msb_model_desc &m) : desc_(m), ss_(msb_model_ss_size(&m), 0.0) {}

  void add_value(const hypers &m, const common::value_accessor &value, common::rng_t &) override;
  void remove_value(const hypers &m, const common::value_accessor &value, common::rng_t &) override;
  float score_value(const hypers &m, const common::value_accessor &value, common::rng_t &) const override;
  float score_data(const hypers &m, common::rng_t &) const override;
  // one draw from the posterior predictive (distributions.hpp:293-298); the caller's rng supplies the counter of the
  // device's Philox stream, so the engine advances as it would upstream.  dm throws, as dm.cpp:100-111 does.
  void sample_value(const hypers &m, common::value_mutator &value, common::rng_t &rng) const override;
  // the serialized Group message, as distributions.hpp:300-306 / bbnc.cpp, dm.cpp return it (wire.hpp)
  common::suffstats_bag_t get_ss() const override { return b200::wire::encode(b200::wire::group_fields(desc_), ss_); }
  void set_ss(const common::suffstats_bag_t &ss) override {  // distributions.hpp:308-314
    std::vector<double> s = ss_;
    b200::wire::decode(b200::wire::group_fields(desc_), ss, s);
    if (desc_.family == MSB_FAMILY_DD) {  // count_sum is not on the wire: it is the sum of the counts
      s[0] = 0.0;
      for (size_t i = 1; i < s.size(); i++) s[0] += s[i];
    }
    ss_ = s;
  }
  void set_ss(const group &g) override { ss_ = static_cast<const gpu_group &>(g).ss_; }  // unchecked cast, as distributions.hpp:316-320
  common::value_mutator get_ss_mutator(const std::string &key) override {
    const b200::field f = b200::ss_field(desc_, key);
    return f.cnt == 1 ? common::value_mutator(&ss_[f.off])
                      : common::value_mutator(reinterpret_cast<uint8_t *>(&ss_[f.off]), common::runtime_type(TYPE_F64, (unsigned)f.cnt));
  }
  std::string debug_str() const override {
    std::ostringstream o;
    o << "{ss=[";
    for (size_t i = 0; i < ss_.size() && i < 8; i++) o << (i ? ", " : "") << ss_[i];
    o << (ss_.size() > 8 ? ", ...]}" : "]}");
    return o.str();
  }
  const std::vector<double> &ss() const { return ss_; }

private:
  msb_model_desc desc_;
  std::vector<double> ss_;
};

class gpu_hypers : public hypers {
public:
  gpu_hypers(const msb_model_desc &m) : desc_(m), hp_(msb_model_hp_size(&m), 0.0) {
    // defaults of microscopes/models.pyx:189,211,223,238,264-269
    switch (m.family) {
      case MSB_FAMILY_BB: case MSB_FAMILY_GP: case MSB_FAMILY_BBNC: hp_[0] = hp_[1] = 1.0; break;
      case MSB_FAMILY_BNB: hp_[0] = hp_[1] = hp_[2] = 1.0; break;
      case MSB_FAMILY_NICH: hp_[1] = hp_[2] = hp_[3] = 1.0; break;
      case MSB_FAMILY_DD: case MSB_FAMILY_DM: for (auto &a : hp_) a = 1.0; break;
      case MSB_FAMILY_NIW:
        hp_[m.dim] = 1.0;
        for (unsigned i = 0; i < m.dim; i++) hp_[m.dim + 1 + (size_t)i * m.dim + i] = 1.0;
        hp_[m.dim + 1 + (size_t)m.dim * m.dim] = (double)m.dim;
        break;
    }
  }
  // the serialized Shared message (distributions.hpp:355-369)
  common::hyperparam_bag_t get_hp() const override { return b200::wire::encode(b200::wire::shared_fields(desc_), hp_); }
  void set_hp(const common::hyperparam_bag_t &hp) override {
    std::vector<double> h = hp_;
    b200::wire::decode(b200::wire::shared_fields(desc_), hp, h);  // throws "wrong dimension" like distributions.hpp:436
    hp_ = h;
  }
  void set_hp(const hypers &s) override { hp_ = static_cast<const gpu_hypers &>(s).hp_; }
  common::value_mutator get_hp_mutator(const std::string &key) override {
    const b200::field f = b200::hp_field(desc_, key);
    return f.cnt == 1 ? common::value_mutator(&hp_[f.off])
                      : common::value_mutator(reinterpret_cast<uint8_t *>(&hp_[f.off]), common::runtime_type(TYPE_F64, (unsigned)f.cnt));
  }
  std::shared_ptr<group> create_group(common::rng_t &) const override { return std::make_shared<gpu_group>(desc_); }
  std::string debug_str() const override { return "{hp}"; }
  const std::vector<double> &hp() const { return hp_; }
  const msb_model_desc &desc() const { return desc_; }

private:
  msb_model_desc desc_;
  std::vector<double> hp_;
};

inline void gpu_group::add_value(const hypers &m, const common::value_accessor &value, common::rng_t &) {
  const gpu_hypers &h = static_cast<const gpu_hypers &>(m);
  const b200::value_f64 v(value);
  b200::check(msb_value_add(b200::default_ctx(), &desc_, h.hp().data(), h.hp().size(), ss_.data(), ss_.size(), v.x.data(), &v.type));
}
inline void gpu_group::remove_value(const hypers &m, const common::value_accessor &value, common::rng_t &) {
  const gpu_hypers &h = static_cast<const gpu_hypers &>(m);
  const b200::value_f64 v(value);
  b200::check(msb_value_remove(b200::default_ctx(), &desc_, h.hp().data(), h.hp().size(), ss_.data(), ss_.size(), v.x.data(), &v.type));
}
inline float gpu_group::score_value(const hypers &m, const common::value_accessor &value, common::rng_t &) const {
  const gpu_hypers &h = static_cast<const gpu_hypers &>(m);
  const b200::value_f64 v(value);
  float out = 0.f;
  b200::check(msb_value_score(b200::default_ctx(), &desc_, h.hp().data(), h.hp().size(), ss_.data(), ss_.size(), v.x.data(), &v.type, &out));
  return out;
}

inline float gpu_group::score_data(const hypers &m, common::rng_t &) const {
  const gpu_hypers &h = static_cast<const gpu_hypers &>(m);
  float out = 0.f;
  b200::check(msb_value_score_data(b200::default_ctx(), &desc_, h.hp().data(), h.hp().size(), ss_.data(), ss_.size(), &out));
  return out;
}
inline void gpu_group::sample_value(const hypers &m, common::value_mutator &value, common::rng_t &rng) const {
  const gpu_hypers &h = static_cast<const gpu_hypers &>(m);
  const uint64_t hi = (uint64_t)rng(), lo = (uint64_t)rng();
  std::vector<double> x(desc_.family == MSB_FAMILY_NIW ? desc_.dim : 1u);
  b200::check(msb_value_sample(b200::default_ctx(), &desc_, h.hp().data(), h.hp().size(), ss_.data(), ss_.size(),
                               0x6d73625f64726177ull, (hi << 32) ^ lo, 1, x.data()));
  if (value.shape() != x.size()) throw std::runtime_error("shapes do not match");  // distributions.hpp:243
  for (size_t i = 0; i < x.size(); i++) value.set<double>(x[i], i);
}

// model handles: what microscopes/_models.pyx:22-44 constructs (bb, gp, nich, dd(size), niw(dim))
class gpu_model : public model {
public:
  gpu_model(int family, unsigned dim = 0) {
    desc_.family = family; desc_.dim = dim;
    if ((family == MSB_FAMILY_DD || family == MSB_FAMILY_NIW || family == MSB_FAMILY_DM) && dim == 0) throw std::runtime_error("no elements");  // distributions.hpp:429,478
  }
  std::shared_ptr<hypers> create_hypers() const override { return std::make_shared<gpu_hypers>(desc_); }
  common::runtime_type get_runtime_type() const override {
    switch (desc_.family) {  // the Value types of SURVEY.md section 2a
      case MSB_FAMILY_BB: case MSB_FAMILY_BBNC: return common::runtime_type(TYPE_B);  // bbnc.cpp:180-184
      case MSB_FAMILY_DM: return common::runtime_type(TYPE_I32, desc_.dim);             // dm.hpp:186-190
      case MSB_FAMILY_BNB: case MSB_FAMILY_GP: return common::runtime_type(TYPE_U32);
      case MSB_FAMILY_NICH: return common::runtime_type(TYPE_F32);
      case MSB_FAMILY_DD: return common::runtime_type(TYPE_I32);
      default: return common::runtime_type(TYPE_F32, desc_.dim);  // distributions.hpp:498-505
    }
  }
  const msb_model_desc &desc() const { return desc_; }

private:
  msb_model_desc desc_;
};

// ---------------------------------------------------------------------------------------------
// batch_scorer: K groups x D features against N rows in one call.  Construct it from the same
// objects the reference's loop uses: the models, the row_major_dataview arguments
// (recarray/dataview.hpp:196-199) and, per group, the per-feature gpu_group objects.
// ---------------------------------------------------------------------------------------------
class batch_scorer {
public:
  batch_scorer(const std::vector<std::shared_ptr<gpu_model>> &models, const uint8_t *data, const bool *mask, size_t n,
               const std::vector<common::runtime_type> &types, size_t max_groups, int device = 0)
      : ctx_(b200::default_ctx(device)), dv_(nullptr), st_(nullptr), D_(models.size()) {
    std::vector<msb_runtime_type> t;
    for (const auto &x : types) t.push_back(b200::abi_type(x));
    std::vector<msb_model_desc> m;
    for (const auto &x : models) m.push_back(x->desc());
    b200::check(msb_dataview_create(ctx_, data, mask, n, t.data(), t.size(), 0, &dv_));
    b200::check(msb_state_create(ctx_, m.data(), m.size(), max_groups, &st_));
    b200::check(msb_state_bind(st_, dv_));
    descs_ = m;
  }
  ~batch_scorer() { msb_state_destroy(st_); msb_dataview_destroy(dv_); }
  batch_scorer(const batch_scorer &) = delete;
  batch_scorer &operator=(const batch_scorer &) = delete;

  void set_alpha(double a) { b200::check(msb_state_set_cluster_hp(st_, "alpha", a)); }
  void set_hypers(size_t feature, const gpu_hypers &h) {
    static const char *keys[8][4] = {{"alpha", "beta", 0, 0}, {"alpha", "beta", "r", 0}, {"alpha", "inv_beta", 0, 0},
                                     {"mu", "kappa", "sigmasq", "nu"}, {"alphas", 0, 0, 0}, {"mu", "kappa", "psi", "nu"},
                                     {"alpha", "beta", 0, 0}, {"alphas", 0, 0, 0}};
    for (int i = 0; i < 4 && keys[descs_[feature].family][i]; i++) {
      const b200::field f = b200::hp_field(descs_[feature], keys[descs_[feature].family][i]);
      b200::check(msb_state_set_hp(st_, feature, keys[descs_[feature].family][i], h.hp().data() + f.off, f.cnt));
    }
  }
  size_t create_group() { size_t g; b200::check(msb_state_create_group(st_, &g)); return g; }
  void add_values(const std::vector<int64_t> &gids) { b200::check(msb_state_add_values(st_, gids.data(), gids.size())); }
  // scores[i * K + c] for every row, columns in ascending gid order (entity_state.hpp:60-72 for all entities at once)
  std::vector<float> score_rows(std::vector<size_t> *gids = nullptr) {
    size_t k = 0, n = 0;
    b200::check(msb_state_ngroups(st_, &k));
    b200::check(msb_state_nentities(st_, &n));
    std::vector<float> out(n * k);
    std::vector<size_t> g(k);
    size_t ncols = 0;
    b200::check(msb_state_score_rows(st_, 0, n, out.data(), k, 0, g.data(), k, &ncols));
    if (gids) *gids = g;
    return out;
  }
  // posterior predictive of rows [row_lo, row_hi) (msb_state_predict): logp always; resp ([nrows][K]), map / draw gids and
  // the imputed values ([nrows][W], masked cells drawn from the drawn group) when the pointer is non-null
  std::vector<double> predict(size_t row_lo, size_t row_hi, uint64_t seed = 0, uint64_t counter = 0,
                              std::vector<float> *resp = nullptr, std::vector<int64_t> *map_gid = nullptr,
                              std::vector<int64_t> *draw_gid = nullptr, std::vector<double> *values = nullptr,
                              std::vector<size_t> *gids = nullptr) {
    size_t k = 0;
    b200::check(msb_state_ngroups(st_, &k));
    size_t w = 0;
    for (const auto &m : descs_) w += (m.family == MSB_FAMILY_NIW || m.family == MSB_FAMILY_DM) ? m.dim : 1;
    const size_t n = row_hi - row_lo;
    std::vector<double> logp(n);
    msb_predict_opts o;
    std::memset(&o, 0, sizeof(o));
    o.seed = seed; o.counter = counter;
    msb_predict_out out;
    std::memset(&out, 0, sizeof(out));
    out.logp = logp.data();
    if (resp) { resp->assign(n * k, 0.f); out.resp = resp->data(); out.resp_ld = k; }
    if (map_gid) { map_gid->assign(n, -1); out.map_gid = map_gid->data(); }
    if (draw_gid) { draw_gid->assign(n, -1); out.draw_gid = draw_gid->data(); }
    if (values) { values->assign(n * w, 0.0); out.values = values->data(); out.values_ld = w; }
    std::vector<size_t> g(k);
    size_t ncols = 0;
    b200::check(msb_state_predict(st_, row_lo, row_hi, &o, &out, g.data(), k, &ncols));
    if (gids) *gids = g;
    return logp;
  }
  // hyperparameter grids (msb_state_set_hp_grid / set_cluster_hp_grid): points[npoints][nhp] in the flat hp layout,
  // log_prior[npoints]; an empty grid removes it
  void set_hp_grid(size_t feature, const std::vector<double> &points, const std::vector<double> &log_prior) {
    const size_t g = log_prior.size();
    b200::check(msb_state_set_hp_grid(st_, feature, points.data(), g, g ? points.size() / g : 0, log_prior.data()));
    grid_sizes_[feature] = g;
  }
  void set_cluster_hp_grid(const std::vector<double> &alphas, const std::vector<double> &log_prior) {
    b200::check(msb_state_set_cluster_hp_grid(st_, alphas.data(), alphas.size(), log_prior.data()));
    grid_sizes_[D_] = alphas.size();
  }
  // one Gibbs step over every grid (msb_state_hp_gibbs), applied to the state: the index drawn per feature, -1 without a
  // grid, [D] = alpha's; logw ([D + 1][*logw_ld], log_prior + log marginal per point) when the pointer is non-null
  std::vector<int64_t> hp_gibbs(uint64_t seed, uint64_t counter, std::vector<double> *logw = nullptr,
                                size_t *logw_ld = nullptr) {
    std::vector<int64_t> choice(D_ + 1, -1);
    msb_hp_gibbs_opts o;
    o.seed = seed; o.counter = counter;
    msb_hp_gibbs_out out;
    std::memset(&out, 0, sizeof(out));
    out.choice = choice.data();
    if (logw) {
      size_t ld = 1;
      for (const auto &g : grid_sizes_) ld = std::max(ld, g.second);
      logw->assign((D_ + 1) * ld, 0.0);
      out.logw = logw->data(); out.logw_ld = ld;
      if (logw_ld) *logw_ld = ld;
    }
    b200::check(msb_state_hp_gibbs(st_, &o, &out));
    return choice;
  }
  // one slice-sampling update of bbnc's p in every group (msb_state_theta): widths[D], 0 leaves a feature alone;
  // returns the number of updates that reached the shrink cap and kept their p
  size_t theta(const std::vector<double> &widths, uint64_t seed, uint64_t counter) {
    msb_theta_opts o;
    o.seed = seed; o.counter = counter; o.widths = widths.data(); o.nwidths = widths.size();
    msb_theta_out out = {0};
    b200::check(msb_state_theta(st_, &o, &out));
    return out.capped;
  }
  // every empty group's bbnc p drawn afresh from Beta(alpha, beta) (msb_state_redraw_empty)
  void redraw_empty(uint64_t seed, uint64_t counter) { b200::check(msb_state_redraw_empty(st_, seed, counter)); }
  // one slice-sampling update per spec of scalar feature hypers and of alpha (feature D), applied to the state
  // (msb_state_slice_hp); returns each spec's value after the call, and the number that reached the shrink cap in *capped
  std::vector<double> slice_hp(const std::vector<msb_slice_hp_spec> &specs, uint64_t seed, uint64_t counter, size_t *capped = nullptr) {
    std::vector<double> values(specs.size());
    msb_slice_hp_opts o;
    o.seed = seed; o.counter = counter; o.specs = specs.data(); o.nspecs = specs.size();
    msb_slice_hp_out out;
    out.capped = 0; out.values = values.data();
    b200::check(msb_state_slice_hp(st_, &o, &out));
    if (capped) *capped = out.capped;
    return values;
  }
  msb_sweep_result sweep(uint64_t seed, uint64_t sweep_id) {
    msb_sweep_opts o;
    std::memset(&o, 0, sizeof(o));
    o.seed = seed; o.sweep = sweep_id;
    msb_sweep_result r;
    size_t n = 0;
    b200::check(msb_state_nentities(st_, &n));
    b200::check(msb_state_sweep(st_, 0, n, &o, &r));
    return r;
  }
  std::vector<int64_t> assignments() {
    size_t n = 0;
    b200::check(msb_state_nentities(st_, &n));
    std::vector<int64_t> a(n);
    b200::check(msb_state_assignments(st_, a.data(), n));
    return a;
  }
  // ---- asynchronous / streaming forms (see INTEGRATION.md 3b) ----------------------------------------------
  // enqueue a sweep and return; sweep_wait() collects rows / moved / units
  void sweep_async(uint64_t seed, uint64_t sweep_id, uint64_t row_id_offset = 0, bool defer_apply = false) {
    msb_sweep_opts o;
    std::memset(&o, 0, sizeof(o));
    o.seed = seed; o.sweep = sweep_id; o.row_id_offset = row_id_offset;
    o.defer_apply = defer_apply ? 1 : 0; o.flags = MSB_SWEEP_ASYNC;
    size_t n = 0;
    b200::check(msb_state_nentities(st_, &n));
    b200::check(msb_state_sweep(st_, 0, n, &o, nullptr));
  }
  msb_sweep_result sweep_wait() { msb_sweep_result r; b200::check(msb_state_sweep_wait(st_, &r)); return r; }
  // a pass over host-resident rows: upload (+ prefetch) on the copy stream, refresh swaps the column buffers
  void upload(const uint8_t *data, const bool *mask = nullptr, bool prefetch = true) {
    b200::check(msb_dataview_upload(dv_, data, mask));
    if (prefetch) b200::check(msb_state_prefetch(st_));
  }
  void refresh() { b200::check(msb_state_refresh(st_)); }
  void assignments_async(int64_t *pinned_out, size_t n) { b200::check(msb_state_assignments_async(st_, pinned_out, n)); }
  void assignments_wait() { b200::check(msb_state_assignments_wait(st_)); }
  // entity_state.hpp:74-86, group_manager.hpp:250-272
  float score_assignment() { float v; b200::check(msb_state_score_assignment(st_, &v)); return v; }
  float score_likelihood(size_t component, size_t gid) { float v; b200::check(msb_state_score_likelihood(st_, component, gid, &v)); return v; }
  float score_likelihood() { float v; b200::check(msb_state_score_likelihood_all(st_, nullptr, 0, &v)); return v; }
  // multi-GPU: flat fp64 delta buffer for ncclAllReduce(sum), then apply_deltas()
  double *delta_buffer(size_t *count) { double *p; b200::check(msb_state_delta_buffer(st_, &p, count)); return p; }
  void apply_deltas() { b200::check(msb_state_apply_deltas(st_)); }
  void *stream() { return msb_ctx_stream(ctx_); }
  msb_state *handle() { return st_; }

private:
  msb_ctx *ctx_;
  msb_dataview *dv_;
  msb_state *st_;
  size_t D_;
  std::vector<msb_model_desc> descs_;
  std::map<size_t, size_t> grid_sizes_;  // feature (D_: alpha) -> grid points registered
};

}  // namespace models
}  // namespace microscopes
