// mscope_b200.cu -- implementation of the C ABI declared in include/mscope_b200.h.
// Host orchestration only; all arithmetic of the hot path runs in the kernels of
// msb_kernels.cuh / msb_niw_tc.cuh on the context's CUDA stream.
#include "../../include/mscope_b200.h"

#include <dlfcn.h>
#include <nccl.h>   // types and prototypes only: the library is resolved at run time (nccl_api below), never linked

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <set>
#include <chrono>
#include <string>
#include <vector>

#include "msb_kernels.cuh"
#include "msb_score.cuh"
#include "msb_niw_tc.cuh"
#include "msb_niw_tc16.cuh"
#include "msb_draw.cuh"
#include "msb_predict.cuh"
#include "msb_hp.cuh"
#include "msb_theta.cuh"
#include "msb_hpslice.cuh"

using namespace msb;

// ---------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------
static thread_local std::string g_last_error;
static int fail(int code, const std::string &msg) { g_last_error = msg; return code; }

#define CU_TRY(expr)                                                                              \
  do {                                                                                            \
    cudaError_t _e = (expr);                                                                      \
    if (_e != cudaSuccess)                                                                        \
      return fail(MSB_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e) + " (" + __FILE__ + ":" + std::to_string(__LINE__) + ")"); \
  } while (0)
#define MSB_TRY(expr)            \
  do {                           \
    int _s = (expr);             \
    if (_s != MSB_OK) return _s; \
  } while (0)
#define REQUIRE(cond, msg) \
  do { if (!(cond)) return fail(MSB_ERR_INVALID, msg); } while (0)

extern "C" MSB_API const char *msb_last_error(void) { return g_last_error.c_str(); }
extern "C" MSB_API int msb_abi_version(void) { return MSB_ABI_VERSION; }

// ---------------------------------------------------------------------------
// objects
// ---------------------------------------------------------------------------
struct msb_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  cudaStream_t copy_stream = nullptr;  // host -> device record uploads run here, overlapping the kernels on `stream`
  // device -> host result copies (msb_state_assignments_async) have a stream of their own: behind the uploads on the copy
  // stream, the NEXT pass's records -- issued right after -- queued behind a copy that waits for the CURRENT sweep to end,
  // which took a whole sweep of look-ahead away from the upload (8 GPUs streaming at once: 3.0 ms per C2 pass for a
  // 2.1 ms step, although the box sustains 24-36 GB/s per GPU with all eight copying, scripts/h2d_contention.py)
  cudaStream_t d2h_stream = nullptr;
  uint64_t launches = 0;
  int sm_count = 0;
  size_t smem_optin = 0;
  KernelProf prof;  // msb_ctx_profile: per-kernel event pairs, off by default
};

struct msb_dataview {
  msb_ctx *ctx = nullptr;
  size_t n = 0, D = 0, rowsize = 0, maskrowsize = 0;
  std::vector<msb_runtime_type> types;
  std::vector<size_t> off, moff;
  std::vector<uint64_t> pi;   // iteration order set by msb_dataview_permute (empty: storage order)
  uint8_t *d_data = nullptr, *d_mask = nullptr;
  bool owns = false;
  // ordering between the copy stream (msb_dataview_upload) and the compute stream (kernels that read the records)
  cudaEvent_t ev_uploaded = nullptr, ev_consumed = nullptr;
  bool upload_pending = false, consumed_recorded = false;
};

// the compute stream is about to read dv's records: wait for an upload still in flight on the copy stream
static cudaError_t dv_acquire(msb_dataview *dv) {
  if (!dv->upload_pending) return cudaSuccess;
  dv->upload_pending = false;
  return cudaStreamWaitEvent(dv->ctx->stream, dv->ev_uploaded, 0);
}
// the compute stream has enqueued its last read of dv's records: the next upload may overwrite them after this point
static cudaError_t dv_release(msb_dataview *dv) {
  if (!dv->ev_consumed) return cudaSuccess;
  dv->consumed_recorded = true;
  return cudaEventRecord(dv->ev_consumed, dv->ctx->stream);
}

struct PhaseEvents { cudaEvent_t e[6]; };

struct msb_state {
  msb_ctx *ctx = nullptr;
  size_t D = 0, kmax = 0;
  std::vector<msb_model_desc> models;
  std::vector<FeatDev> feats;
  FeatDev *d_feats = nullptr;
  FeatDev *d_feats_scalar = nullptr;  // the features the score kernel walks (chunk rows > 0), same order
  size_t n_scalar = 0;
  bool feats_dirty = true;
  // hypers
  std::vector<double> h_hp;
  double *d_hp = nullptr;
  bool hp_dirty = true;
  // suffstats: [counts kmax | per-feature blocks]
  size_t SS = 0;
  double *d_ss = nullptr, *d_delta = nullptr;
  int32_t *d_delta_i32 = nullptr;  // msb_state_delta_buffer_i32
  // CRP bookkeeping (group_manager.hpp:48-306)
  double alpha = 1.0;
  size_t gcount = 0;
  std::map<size_t, int> gid2slot;
  std::vector<int64_t> slot2gid;
  std::vector<int> free_slots;
  std::vector<double> h_counts;
  bool counts_stale = false;      // the device counts (d_ss[0..kmax)) are newer than h_counts
  bool cols_dirty = true;         // groups were created / deleted since the column tables were uploaded
  unsigned long long *h_moved = nullptr;  // pinned + mapped: the moved-row counter of the last sweep lands here
  unsigned long long *h_moved_dev = nullptr;  // its device address (publish_counter_kernel writes it: no copy engine)
  uint32_t *h_flags = nullptr;    // pinned scratch for the bind-time device -> host flags
  uint32_t *d_flags = nullptr;
  int64_t *d_assign64 = nullptr; size_t assign64_cap = 0;
  cudaEvent_t ev_mapped = nullptr, ev_assign_copied = nullptr;  // msb_state_assignments_async
  bool assign_copy_pending = false;
  bool slot2gid_dirty = true;
  msb_sweep_result last_res = {0, 0, 0};
  std::vector<char> slot_dirty;   // suffstats of the slot may be non-zero (set by any update / set_ss)
  bool all_unassigned = true;     // no entity has been assigned since bind
  void *col_slab = nullptr;       // one allocation backing every column
  size_t slab_bytes = 0;
  // Second column buffer (msb_state_prefetch): the next pass's records are converted on the copy stream into the
  // buffer the running sweep does not read; msb_state_refresh then only swaps the two.
  void *col_slab_b = nullptr;
  std::vector<FeatDev> feats_b;
  std::vector<void *> cols_b;
  FeatDev *d_feats_b = nullptr, *d_feats_scalar_b = nullptr;
  uint32_t *d_flags_b = nullptr, *h_flags_b = nullptr;
  cudaEvent_t ev_swap = nullptr, ev_prefetched = nullptr;
  bool prefetch_pending = false, swap_recorded = false, feats_b_dirty = false;
  size_t n_pad = 0;               // rows of the (padded) score columns
  // data
  msb_dataview *dv = nullptr;
  size_t n = 0;
  std::vector<void *> cols;
  int32_t *d_assign = nullptr;
  size_t region_rows = 0, max_chunk_rows = 0;
  std::vector<FeatDev> sc_host;  // the score kernel's walk order (host copy of d_feats_scalar)
  uint64_t bundle_key = 0;       // (tile shape, stage bytes) the bundle layout in d_feats_scalar was made for; 0 = none
  std::vector<FeatDev> sc_host_b;  // the same pair for the second column buffer (msb_state_prefetch): its descriptors point
  uint64_t bundle_key_b = 0;       // into the other slab, so each buffer keeps its own list and its own layout state
  bool has_bbnc = false, has_dm = false;  // has_dm: a vector count feature scored by its own kernel after the scalar ones (like niw)
  uint64_t group_seed = 0x6d73625f62626e63ull;  // Philox key of the per-group parameter draws (bbnc: p ~ Beta(alpha, beta))
  bool has_niw = false, has_scalar = false, tables_only = false, has_dd = false, has_nich = false;
  // workspaces
  float *d_params = nullptr; size_t params_cap = 0;
  float *d_scores = nullptr; size_t scores_cap = 0;
  float *d_base = nullptr; size_t base_cap = 0;
  float *d_base_score = nullptr; size_t base_score_cap = 0;  // base + row-independent nich terms, for the score kernel
  int32_t *d_col2slot = nullptr; size_t col_cap = 0;
  int64_t *d_slot2gid = nullptr;
  int32_t *d_newslot = nullptr, *d_newcol = nullptr; size_t row_cap = 0;
  float *d_uniforms = nullptr;
  unsigned long long *d_counter = nullptr;
  std::vector<float *> d_niwW, d_niwBias, d_niwCoef, d_niwB;
  void *d_niwA16 = nullptr; size_t niw_a16_cap = 0;  // fp16 A operand of the tensor-core NIW kernel (one feature at a time)
  // what d_niwA16 (and the column maxima next to the feature's B operand) currently hold: feature, row range and the
  // version of the column data they were converted from -- rows that did not change between sweeps (bind once, sweep
  // many) are not scanned and converted again
  std::map<std::string, double> pass_host_ns;       // MSB_PASS_TIMING: host nanoseconds per sub-step of msb_state_pass
  int *d_rowmax = nullptr; size_t rowmax_cap = 0;   // per-row score maximum from the bundled score kernel's epilogue (sweep only)
  bool rowmax_valid = false;                        // the last launch_score filled it
  uint64_t col_version = 1, niw_a16_version = 0;
  size_t niw_a16_feat = 0, niw_a16_lo = 0, niw_a16_hi = 0;
  size_t niw_cols_cap = 0;
  // last score
  int tail_g = 0;  // replication width of the last k-tile's table columns (build_params), 0 = none
  int cfg = 1, V = 2; size_t ld = 0, last_rows = 0, last_cols = 0;
  bool last_blocked = false;
  size_t last_skip = 0;  // rows between the score buffer's origin (row_origin) and the first valid row
  std::vector<int32_t> h_col2slot;
  std::vector<size_t> h_colgid;
  // phase events of the last TIMING_RING sweeps (read on demand by msb_state_timings, never inside a sweep)
  static constexpr size_t TIMING_RING = 64;
  std::vector<PhaseEvents> events[TIMING_RING];
  size_t ring_nchunks[TIMING_RING] = {0};
  uint64_t sweep_seq = 0;  // sweeps enqueued so far
  size_t last_allreduce_bytes = 0;  // message size of the last msb_state_allreduce_deltas
  // hyperparameter grids (msb_state_set_hp_grid / set_cluster_hp_grid): [D + 1] host copies, row D = alpha's; the device
  // buffer d_grid = [HpRow rows | points | log priors] is rebuilt whenever a grid is set
  std::vector<std::vector<double>> grid_pts, grid_lp;
  std::vector<HpRow> hp_rows;
  size_t grid_gmax = 0;
  void *d_grid = nullptr;
  double *d_hpwork = nullptr; size_t hpwork_cap = 0;  // msb_state_hp_gibbs scratch
  char *d_theta = nullptr; size_t theta_cap = 0;        // msb_state_theta / redraw_empty scratch (theta_run)
  char *d_hpsl = nullptr; size_t hpsl_cap = 0;          // msb_state_slice_hp scratch
};

#define LAUNCH(ctx, kernel, grid, block, smem, ...)                      \
  do {                                                                   \
    (ctx)->prof.begin(#kernel, (ctx)->stream);                           \
    kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);     \
    (ctx)->prof.end((ctx)->stream);                                      \
    (ctx)->launches++;                                                   \
    CU_TRY(cudaGetLastError());                                          \
  } while (0)

static inline unsigned cdiv(size_t a, size_t b) { return (unsigned)((a + b - 1) / b); }

// device scratch of one call: released on every return path (the CU_TRY / MSB_TRY early returns included)
template <typename T> struct Scratch {
  T *p = nullptr;
  Scratch() = default;
  Scratch(const Scratch &) = delete;
  Scratch &operator=(const Scratch &) = delete;
  ~Scratch() { if (p) cudaFree(p); }
  cudaError_t alloc(size_t count) { return cudaMalloc(&p, sizeof(T) * std::max<size_t>(count, 1)); }
  operator T *() const { return p; }
};

// ---------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------
template <typename K> static cudaError_t opt_in_smem(K kernel, size_t bytes) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

extern "C" MSB_API int msb_ctx_create(int device, void *stream, msb_ctx **out) {
  REQUIRE(out, "msb_ctx_create: out is NULL");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(MSB_ERR_CUDA, std::string("no usable CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e));
  REQUIRE(device >= 0 && device < ndev, "msb_ctx_create: bad device index");
  CU_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10)
    return fail(MSB_ERR_UNSUPPORTED, "this library is built for sm_100a (B200) only; device is sm_" +
                                         std::to_string(prop.major) + std::to_string(prop.minor));
  msb_ctx *c = new msb_ctx();
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  c->smem_optin = prop.sharedMemPerBlockOptin;
  // The sweep's stream outranks the copy streams: the conversion kernel of the NEXT pass's records (copy stream) becomes
  // runnable at the very moment a sweep starts, and at equal priority its blocks were placed first -- the sweep's
  // parameter build and score kernel then waited for them (8 GPUs, C2 passes over host rows: build phase 0.36 instead of
  // 0.03 ms, score 1.50 instead of 1.38 ms).  With priorities the conversion fills what the sweep's kernels leave free.
  int prio_least = 0, prio_greatest = 0;
  CU_TRY(cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest));
  if (stream) c->stream = (cudaStream_t)stream;
  else { CU_TRY(cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, prio_greatest)); c->own_stream = true; }
  CU_TRY(cudaStreamCreateWithPriority(&c->copy_stream, cudaStreamNonBlocking, prio_least));
  CU_TRY(cudaStreamCreateWithPriority(&c->d2h_stream, cudaStreamNonBlocking, prio_least));
  CU_TRY(opt_in_smem(score_kernel<1, 64, 16, false, false>, c->smem_optin));
  CU_TRY(opt_in_smem(score_kernel<2, 32, 16, false, false>, c->smem_optin));
  CU_TRY(opt_in_smem(score_kernel<4, 32, 8, false, false>, c->smem_optin));
  CU_TRY(opt_in_smem(score_kernel<1, 32, 8, false, false>, c->smem_optin));
  CU_TRY(opt_in_smem(score_kernel<1, 64, 16, false, true>, c->smem_optin));
  CU_TRY(opt_in_smem(score_kernel<2, 32, 16, false, true>, c->smem_optin));
  CU_TRY(opt_in_smem(score_kernel<4, 32, 8, false, true>, c->smem_optin));
  CU_TRY(opt_in_smem(score_kernel<1, 32, 8, false, true>, c->smem_optin));
  CU_TRY(opt_in_smem(score_kernel<1, 64, 16, true, false>, c->smem_optin));
  CU_TRY(opt_in_smem(score_kernel<2, 32, 16, true, false>, c->smem_optin));
  CU_TRY(opt_in_smem(score_kernel<4, 32, 8, true, false>, c->smem_optin));
  CU_TRY(opt_in_smem(score_kernel<1, 32, 8, true, false>, c->smem_optin));
  CU_TRY(opt_in_smem(score_kernel<1, 64, 16, true, true>, c->smem_optin));
  CU_TRY(opt_in_smem(score_kernel<2, 32, 16, true, true>, c->smem_optin));
  CU_TRY(opt_in_smem(score_kernel<4, 32, 8, true, true>, c->smem_optin));
  CU_TRY(opt_in_smem(score_kernel<1, 32, 8, true, true>, c->smem_optin));
  CU_TRY(opt_in_smem((score_tables_persistent_kernel<1, 64, 16>), c->smem_optin));
  CU_TRY(opt_in_smem((score_tables_persistent_kernel<2, 32, 16>), c->smem_optin));
  CU_TRY(opt_in_smem((score_tables_persistent_kernel<4, 32, 8>), c->smem_optin));
  CU_TRY(opt_in_smem((score_tables_persistent_kernel<1, 32, 8>), c->smem_optin));
  CU_TRY(opt_in_smem((score_bundle_kernel<2, 32, 16, false>), c->smem_optin));
  CU_TRY(opt_in_smem((score_bundle_kernel<2, 32, 16, true>), c->smem_optin));
  CU_TRY(opt_in_smem((score_bundle_kernel<4, 32, 8, false>), c->smem_optin));
  CU_TRY(opt_in_smem((score_bundle_kernel<4, 32, 8, true>), c->smem_optin));
  CU_TRY(opt_in_smem((score_bundle_kernel<4, 16, 16, false>), c->smem_optin));
  CU_TRY(opt_in_smem((score_bundle_kernel<4, 16, 16, true>), c->smem_optin));
  CU_TRY(opt_in_smem((sample_tile_kernel<4, false>), c->smem_optin));
  CU_TRY(opt_in_smem((sample_tile_kernel<4, true>), c->smem_optin));
  CU_TRY(opt_in_smem((sample_tile_kernel<1, false>), c->smem_optin));
  CU_TRY(opt_in_smem((sample_tile_kernel<1, true>), c->smem_optin));
  CU_TRY(opt_in_smem((predict_tile_kernel<4, false>), c->smem_optin));
  CU_TRY(opt_in_smem((predict_tile_kernel<4, true>), c->smem_optin));
  CU_TRY(opt_in_smem((predict_tile_kernel<1, false>), c->smem_optin));
  CU_TRY(opt_in_smem((predict_tile_kernel<1, true>), c->smem_optin));
  CU_TRY(opt_in_smem((ingest_tile_kernel<512, 1>), c->smem_optin));
  CU_TRY(opt_in_smem((ingest_tile_kernel<256, 2>), c->smem_optin));
  CU_TRY(opt_in_smem((ingest_tile_kernel<128, 4>), c->smem_optin));
  CU_TRY(opt_in_smem((ingest_tile_kernel<64, 8>), c->smem_optin));
  CU_TRY(opt_in_smem(niw_score_data_kernel, c->smem_optin - 1024));
  CU_TRY(opt_in_smem(niw_score_f64_kernel, c->smem_optin - 1024));
  CU_TRY(opt_in_smem(niw_prepare_kernel, c->smem_optin - 1024));  // it also has a few bytes of static shared memory
  CU_TRY(opt_in_smem(niw_score_simt_kernel, c->smem_optin - 1024));
  MSB_TRY(niw_tc_init(c->smem_optin, g_last_error));
  MSB_TRY(niw_tc16_init(c->smem_optin, g_last_error));
  *out = c;
  return MSB_OK;
}

extern "C" MSB_API int msb_ctx_destroy(msb_ctx *ctx) {
  if (!ctx) return MSB_OK;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  cudaStreamSynchronize(ctx->copy_stream);
  cudaStreamSynchronize(ctx->d2h_stream);
  cudaStreamDestroy(ctx->copy_stream);
  cudaStreamDestroy(ctx->d2h_stream);
  if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
  ctx->prof.destroy();
  delete ctx;
  return MSB_OK;
}
extern "C" MSB_API int msb_ctx_synchronize(msb_ctx *ctx) {
  REQUIRE(ctx, "ctx is NULL");
  CU_TRY(cudaStreamSynchronize(ctx->copy_stream));
  CU_TRY(cudaStreamSynchronize(ctx->stream));
  CU_TRY(cudaStreamSynchronize(ctx->d2h_stream));
  return MSB_OK;
}
extern "C" MSB_API void *msb_ctx_stream(msb_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }
extern "C" MSB_API int msb_ctx_launch_count(msb_ctx *ctx, uint64_t *out) {
  REQUIRE(ctx && out, "NULL argument");
  *out = ctx->launches;
  return MSB_OK;
}

// Per-kernel timing.  enable != 0: forget earlier records and put an event pair around every kernel launched on the
// context's compute stream from now on; enable == 0: stop recording (the records stay readable).
extern "C" MSB_API int msb_ctx_profile(msb_ctx *ctx, int enable) {
  REQUIRE(ctx, "ctx is NULL");
  CU_TRY(cudaSetDevice(ctx->device));
  if (enable) { CU_TRY(cudaStreamSynchronize(ctx->stream)); ctx->prof.clear(); }
  ctx->prof.on = enable != 0;
  return MSB_OK;
}
// Text, one line per kernel name in first-launch order: "name\tlaunches\ttotal_ms\n".  *needed = bytes including the
// terminating 0; the text is truncated to cap.
extern "C" MSB_API int msb_ctx_profile_read(msb_ctx *ctx, char *buf, size_t cap, size_t *needed) {
  REQUIRE(ctx && needed, "NULL argument");
  CU_TRY(cudaSetDevice(ctx->device));
  CU_TRY(cudaStreamSynchronize(ctx->stream));
  std::vector<std::string> names;
  std::vector<double> ms;
  std::vector<size_t> cnt;
  for (auto &r : ctx->prof.recs) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, r.a, r.b) != cudaSuccess) { cudaGetLastError(); continue; }
    size_t i = 0;
    for (; i < names.size(); i++) if (names[i] == r.name) break;
    if (i == names.size()) { names.push_back(r.name); ms.push_back(0.0); cnt.push_back(0); }
    ms[i] += t; cnt[i]++;
  }
  std::string out;
  for (size_t i = 0; i < names.size(); i++) {
    char line[512];
    snprintf(line, sizeof line, "%s\t%zu\t%.6f\n", names[i].c_str(), cnt[i], ms[i]);
    out += line;
  }
  *needed = out.size() + 1;
  if (buf && cap) {
    const size_t m = std::min(cap - 1, out.size());
    memcpy(buf, out.data(), m);
    buf[m] = 0;
  }
  return MSB_OK;
}

// ---------------------------------------------------------------------------
// dataview
// ---------------------------------------------------------------------------
static const size_t k_prim_size[MSB_TYPE_NELEMS] = {1, 1, 1, 2, 2, 4, 4, 8, 8, 4, 8};

extern "C" MSB_API int msb_dataview_create(msb_ctx *ctx, const void *data, const void *mask, size_t n,
                                   const msb_runtime_type *types, size_t nfeatures, int on_device,
                                   msb_dataview **out) {
  REQUIRE(ctx && types && out, "msb_dataview_create: NULL argument");
  REQUIRE(data || n == 0, "msb_dataview_create: data is NULL");
  REQUIRE(nfeatures > 0, "msb_dataview_create: no features");
  CU_TRY(cudaSetDevice(ctx->device));
  msb_dataview *dv = new msb_dataview();
  dv->ctx = ctx; dv->n = n; dv->D = nfeatures;
  dv->types.assign(types, types + nfeatures);
  size_t o = 0, mo = 0;
  for (size_t d = 0; d < nfeatures; d++) {  // runtime_type.hpp:123-134
    if (types[d].prim < 0 || types[d].prim >= MSB_TYPE_NELEMS || types[d].n == 0) {
      delete dv;
      return fail(MSB_ERR_INVALID, "msb_dataview_create: bad runtime type for feature " + std::to_string(d));
    }
    dv->off.push_back(o); dv->moff.push_back(mo);
    o += (size_t)types[d].n * k_prim_size[types[d].prim];
    mo += types[d].n;
  }
  dv->rowsize = o; dv->maskrowsize = mo;
  if (on_device) {
    dv->d_data = (uint8_t *)data; dv->d_mask = (uint8_t *)mask; dv->owns = false;
  } else {
    dv->owns = true;
    CU_TRY(cudaEventCreateWithFlags(&dv->ev_uploaded, cudaEventDisableTiming));
    CU_TRY(cudaEventCreateWithFlags(&dv->ev_consumed, cudaEventDisableTiming));
    if (n) {
      CU_TRY(cudaMalloc(&dv->d_data, n * dv->rowsize));
      CU_TRY(cudaMemcpyAsync(dv->d_data, data, n * dv->rowsize, cudaMemcpyHostToDevice, ctx->stream));
      if (mask) {
        CU_TRY(cudaMalloc(&dv->d_mask, n * dv->maskrowsize));
        CU_TRY(cudaMemcpyAsync(dv->d_mask, mask, n * dv->maskrowsize, cudaMemcpyHostToDevice, ctx->stream));
      }
    }
  }
  *out = dv;
  return MSB_OK;
}

extern "C" MSB_API int msb_dataview_upload(msb_dataview *dv, const void *data, const void *mask) {
  REQUIRE(dv && (data || dv->n == 0), "msb_dataview_upload: NULL argument");
  REQUIRE(dv->owns, "msb_dataview_upload: the dataview borrows device memory");
  REQUIRE((mask != nullptr) == (dv->d_mask != nullptr) || dv->n == 0, "msb_dataview_upload: mask presence must match the dataview");
  if (!dv->n) return MSB_OK;
  msb_ctx *ctx = dv->ctx;
  CU_TRY(cudaSetDevice(ctx->device));
  // The copy runs on the context's copy stream, after the last kernel that reads the old records
  // (ev_consumed) and concurrently with everything enqueued on the compute stream since; the next
  // msb_state_refresh / msb_state_bind / msb_dataview_get_row makes the compute stream wait for it.
  if (dv->consumed_recorded) CU_TRY(cudaStreamWaitEvent(ctx->copy_stream, dv->ev_consumed, 0));
  else {  // nothing recorded yet: order after everything enqueued so far (the creating copy included)
    CU_TRY(cudaEventRecord(dv->ev_consumed, ctx->stream));
    CU_TRY(cudaStreamWaitEvent(ctx->copy_stream, dv->ev_consumed, 0));
  }
  CU_TRY(cudaMemcpyAsync(dv->d_data, data, dv->n * dv->rowsize, cudaMemcpyHostToDevice, ctx->copy_stream));
  if (mask) CU_TRY(cudaMemcpyAsync(dv->d_mask, mask, dv->n * dv->maskrowsize, cudaMemcpyHostToDevice, ctx->copy_stream));
  CU_TRY(cudaEventRecord(dv->ev_uploaded, ctx->copy_stream));
  dv->upload_pending = true;
  return MSB_OK;
}

extern "C" MSB_API int msb_dataview_destroy(msb_dataview *dv) {
  if (!dv) return MSB_OK;
  cudaSetDevice(dv->ctx->device);
  cudaStreamSynchronize(dv->ctx->copy_stream);
  cudaStreamSynchronize(dv->ctx->stream);
  if (dv->owns) { cudaFree(dv->d_data); cudaFree(dv->d_mask); }
  if (dv->ev_uploaded) cudaEventDestroy(dv->ev_uploaded);
  if (dv->ev_consumed) cudaEventDestroy(dv->ev_consumed);
  delete dv;
  return MSB_OK;
}
extern "C" MSB_API int msb_dataview_size(const msb_dataview *dv, size_t *n) { REQUIRE(dv && n, "NULL argument"); *n = dv->n; return MSB_OK; }
extern "C" MSB_API int msb_dataview_nfeatures(const msb_dataview *dv, size_t *d) { REQUIRE(dv && d, "NULL argument"); *d = dv->D; return MSB_OK; }
extern "C" MSB_API int msb_dataview_rowsize(const msb_dataview *dv, size_t *rowsize, size_t *maskrowsize) {
  REQUIRE(dv, "NULL argument");
  if (rowsize) *rowsize = dv->rowsize;
  if (maskrowsize) *maskrowsize = dv->maskrowsize;
  return MSB_OK;
}
extern "C" MSB_API int msb_dataview_get_row(msb_dataview *dv, size_t idx, void *row_out, void *mask_out) {
  REQUIRE(dv && row_out, "NULL argument");
  REQUIRE(idx < dv->n, "invalid position");  // dataview.cpp:131
  if (!dv->pi.empty()) idx = (size_t)dv->pi[idx];   // dataview.cpp:127-139: get() reads record pi_[pos_]
  CU_TRY(cudaSetDevice(dv->ctx->device));
  CU_TRY(dv_acquire(dv));
  CU_TRY(cudaMemcpyAsync(row_out, dv->d_data + idx * dv->rowsize, dv->rowsize, cudaMemcpyDeviceToHost, dv->ctx->stream));
  if (mask_out) {
    if (dv->d_mask) CU_TRY(cudaMemcpyAsync(mask_out, dv->d_mask + idx * dv->maskrowsize, dv->maskrowsize, cudaMemcpyDeviceToHost, dv->ctx->stream));
    else memset(mask_out, 0, dv->maskrowsize);
  }
  CU_TRY(cudaStreamSynchronize(dv->ctx->stream));
  return MSB_OK;
}

extern "C" MSB_API int msb_dataview_permute(msb_dataview *dv, uint64_t seed) {
  REQUIRE(dv, "NULL argument");
  // util.hpp:85-94 (Fisher-Yates from the back: swap position i with a uniform position in [0, i]); the draw for
  // position i is word pair 0-1 of Philox(seed, i, 0), reduced by a multiply-high (bias below 2^-32 for n < 2^32)
  dv->pi.resize(dv->n);
  for (size_t i = 0; i < dv->n; i++) dv->pi[i] = i;
  for (size_t i = dv->n; i-- > 1;) {
    uint32_t r[4];
    msb::philox4x32_10(seed, (uint64_t)i, 0, r);
    const uint64_t r64 = ((uint64_t)r[1] << 32) | r[0];
    const size_t j = (size_t)(((unsigned __int128)r64 * (unsigned __int128)(i + 1)) >> 64);
    std::swap(dv->pi[i], dv->pi[j]);
  }
  return MSB_OK;
}
extern "C" MSB_API int msb_dataview_reset_permutation(msb_dataview *dv) {
  REQUIRE(dv, "NULL argument");
  dv->pi.clear();
  return MSB_OK;
}
extern "C" MSB_API int msb_dataview_permutation(const msb_dataview *dv, uint64_t *pi_out, size_t n) {
  REQUIRE(dv && (pi_out || n == 0), "NULL argument");
  REQUIRE(n == dv->n, "wrong length");
  for (size_t i = 0; i < n; i++) pi_out[i] = dv->pi.empty() ? (uint64_t)i : dv->pi[i];
  return MSB_OK;
}

// ---------------------------------------------------------------------------
// model layouts
// ---------------------------------------------------------------------------
static size_t hp_size(const msb_model_desc &m) {
  switch (m.family) {
    case MSB_FAMILY_BB: case MSB_FAMILY_GP: case MSB_FAMILY_BBNC: return 2;
    case MSB_FAMILY_BNB: return 3;
    case MSB_FAMILY_NICH: return 4;
    case MSB_FAMILY_DD: case MSB_FAMILY_DM: return m.dim;
    case MSB_FAMILY_NIW: return (size_t)m.dim * m.dim + m.dim + 2;
    default: return 0;
  }
}
static size_t ss_size(const msb_model_desc &m) {
  switch (m.family) {
    case MSB_FAMILY_BB: case MSB_FAMILY_BNB: return 2;
    case MSB_FAMILY_GP: case MSB_FAMILY_NICH: case MSB_FAMILY_BBNC: return 3;
    case MSB_FAMILY_DD: case MSB_FAMILY_DM: return (size_t)m.dim + 1;
    case MSB_FAMILY_NIW: return (size_t)m.dim * m.dim + m.dim + 1;
    default: return 0;
  }
}
extern "C" MSB_API size_t msb_model_hp_size(const msb_model_desc *m) { return m ? hp_size(*m) : 0; }
extern "C" MSB_API size_t msb_model_ss_size(const msb_model_desc *m) { return m ? ss_size(*m) : 0; }

static int check_model(const msb_model_desc &m, size_t d) {
  switch (m.family) {
    case MSB_FAMILY_BB: case MSB_FAMILY_BNB: case MSB_FAMILY_GP: case MSB_FAMILY_NICH: case MSB_FAMILY_BBNC: return MSB_OK;
    case MSB_FAMILY_DD:
      if (m.dim == 0) return fail(MSB_ERR_INVALID, "no elements");  // distributions.hpp:429
      if (m.dim > 1024) return fail(MSB_ERR_UNSUPPORTED, "dd with more than 1024 categories is not built yet");
      return MSB_OK;
    case MSB_FAMILY_DM:
      if (m.dim == 0) return fail(MSB_ERR_INVALID, "no elements");
      if (m.dim > 1024) return fail(MSB_ERR_UNSUPPORTED, "dm with more than 1024 categories is not built yet");
      return MSB_OK;
    case MSB_FAMILY_NIW:
      if (m.dim == 0) return fail(MSB_ERR_INVALID, "no elements");  // distributions.hpp:478
      if (m.dim > 96) return fail(MSB_ERR_UNSUPPORTED, "niw with dim > 96 is not built yet");
      return MSB_OK;
    default:
      return fail(MSB_ERR_UNSUPPORTED, "model family " + std::to_string(m.family) + " of feature " + std::to_string(d) + " is not built");
  }
}

// key -> (offset, count) inside the flat hp / ss vectors (distributions.hpp:21-56,165-199)
static int hp_field(const msb_model_desc &m, const std::string &key, size_t *off, size_t *cnt) {
  const size_t d = m.dim;
  switch (m.family) {
    case MSB_FAMILY_BB:
      if (key == "alpha") { *off = 0; *cnt = 1; return MSB_OK; }
      if (key == "beta") { *off = 1; *cnt = 1; return MSB_OK; }
      break;
    case MSB_FAMILY_BBNC:  // bbnc.cpp:159-167
      if (key == "alpha") { *off = 0; *cnt = 1; return MSB_OK; }
      if (key == "beta") { *off = 1; *cnt = 1; return MSB_OK; }
      break;
    case MSB_FAMILY_BNB:  // distributions.hpp:29-32
      if (key == "alpha") { *off = 0; *cnt = 1; return MSB_OK; }
      if (key == "beta") { *off = 1; *cnt = 1; return MSB_OK; }
      if (key == "r") { *off = 2; *cnt = 1; return MSB_OK; }
      break;
    case MSB_FAMILY_GP:
      if (key == "alpha") { *off = 0; *cnt = 1; return MSB_OK; }
      if (key == "inv_beta") { *off = 1; *cnt = 1; return MSB_OK; }
      break;
    case MSB_FAMILY_NICH:
      if (key == "mu") { *off = 0; *cnt = 1; return MSB_OK; }
      if (key == "kappa") { *off = 1; *cnt = 1; return MSB_OK; }
      if (key == "sigmasq") { *off = 2; *cnt = 1; return MSB_OK; }
      if (key == "nu") { *off = 3; *cnt = 1; return MSB_OK; }
      break;
    case MSB_FAMILY_DD: case MSB_FAMILY_DM:  // dm.hpp get_hp_mutator("alphas")
      if (key == "alphas") { *off = 0; *cnt = d; return MSB_OK; }
      break;
    case MSB_FAMILY_NIW:
      if (key == "mu") { *off = 0; *cnt = d; return MSB_OK; }
      if (key == "kappa") { *off = d; *cnt = 1; return MSB_OK; }
      if (key == "psi") { *off = d + 1; *cnt = d * d; return MSB_OK; }
      if (key == "nu") { *off = d + 1 + d * d; *cnt = 1; return MSB_OK; }
      break;
    default: break;
  }
  return fail(MSB_ERR_KEY, "Unknown shared HP param key: " + key);
}
static int ss_field(const msb_model_desc &m, const std::string &key, size_t *off, size_t *cnt) {
  const size_t d = m.dim;
  switch (m.family) {
    case MSB_FAMILY_BB:
      if (key == "heads") { *off = 0; *cnt = 1; return MSB_OK; }
      if (key == "tails") { *off = 1; *cnt = 1; return MSB_OK; }
      break;
    case MSB_FAMILY_BBNC:  // bbnc.cpp:112-118 exposes "p"; heads / tails are the message's other fields (schema.proto:14-18)
      if (key == "p") { *off = 0; *cnt = 1; return MSB_OK; }
      if (key == "heads") { *off = 1; *cnt = 1; return MSB_OK; }
      if (key == "tails") { *off = 2; *cnt = 1; return MSB_OK; }
      break;
    case MSB_FAMILY_BNB:  // distributions.hpp:34-36
      if (key == "count") { *off = 0; *cnt = 1; return MSB_OK; }
      if (key == "sum") { *off = 1; *cnt = 1; return MSB_OK; }
      break;
    case MSB_FAMILY_GP:
      if (key == "count") { *off = 0; *cnt = 1; return MSB_OK; }
      if (key == "sum") { *off = 1; *cnt = 1; return MSB_OK; }
      if (key == "log_prod") { *off = 2; *cnt = 1; return MSB_OK; }
      break;
    case MSB_FAMILY_NICH:
      if (key == "count") { *off = 0; *cnt = 1; return MSB_OK; }
      if (key == "mean") { *off = 1; *cnt = 1; return MSB_OK; }
      if (key == "count_times_variance") { *off = 2; *cnt = 1; return MSB_OK; }
      break;
    case MSB_FAMILY_DM:  // the fields of DirichletMultinomial.Group (schema.proto:25-28); dm.hpp itself allows no mutation
      if (key == "counts") { *off = 0; *cnt = d; return MSB_OK; }
      if (key == "ratio") { *off = d; *cnt = 1; return MSB_OK; }
      break;
    case MSB_FAMILY_DD:
      if (key == "count_sum") { *off = 0; *cnt = 1; return MSB_OK; }
      if (key == "counts") { *off = 1; *cnt = d; return MSB_OK; }
      break;
    case MSB_FAMILY_NIW:
      if (key == "count") { *off = 0; *cnt = 1; return MSB_OK; }
      if (key == "sum_x") { *off = 1; *cnt = d; return MSB_OK; }
      if (key == "sum_xxT") { *off = 1 + d; *cnt = d * d; return MSB_OK; }
      break;
    default: break;
  }
  return fail(MSB_ERR_KEY, "Unknown group SS param key: " + key);
}

// ---------------------------------------------------------------------------
// state
// ---------------------------------------------------------------------------
extern "C" MSB_API int msb_state_create(msb_ctx *ctx, const msb_model_desc *models, size_t nfeatures, size_t max_groups,
                                msb_state **out) {
  REQUIRE(ctx && models && out, "msb_state_create: NULL argument");
  REQUIRE(nfeatures > 0 && max_groups > 0, "msb_state_create: empty state");
  REQUIRE(max_groups < (1u << 30), "msb_state_create: too many groups");
  for (size_t d = 0; d < nfeatures; d++) MSB_TRY(check_model(models[d], d));
  CU_TRY(cudaSetDevice(ctx->device));
  msb_state *st = new msb_state();
  st->ctx = ctx; st->D = nfeatures; st->kmax = max_groups;
  st->models.assign(models, models + nfeatures);
  st->feats.resize(nfeatures);
  size_t hpo = 0, sso = max_groups;  // group counts first
  for (size_t d = 0; d < nfeatures; d++) {
    FeatDev &f = st->feats[d];
    memset(&f, 0, sizeof(f));
    const msb_model_desc &m = models[d];
    f.family = m.family; f.dim = m.dim;
    f.hp_off = hpo; f.ss_off = sso; f.ss_w = (uint32_t)ss_size(m);
    hpo += hp_size(m);
    sso += max_groups * ss_size(m);
    switch (m.family) {
      case MSB_FAMILY_BBNC: st->has_bbnc = true;  // fall through: the same two-row table, filled from the group's own p
      case MSB_FAMILY_BB: f.kind = KIND_TABLE; f.coltype = COL_U8; f.ncat = 2; f.dim = 2; st->has_scalar = true; break;
      case MSB_FAMILY_DD:
        f.kind = KIND_TABLE; f.ncat = m.dim; st->has_scalar = true; st->has_dd = true;
        f.coltype = m.dim + 1 <= 256 ? COL_U8 : (m.dim + 1 <= 65536 ? COL_U16 : COL_U32);
        break;
      case MSB_FAMILY_BNB:  // a count family like gp: same lookup-table machinery, its own closed form
      case MSB_FAMILY_GP: f.kind = KIND_GP; f.coltype = COL_U32; f.ncat = 1; st->has_scalar = true; break;
      case MSB_FAMILY_NICH: f.kind = KIND_NICH; f.coltype = COL_F32; st->has_scalar = true; st->has_nich = true; break;
      case MSB_FAMILY_NIW: f.kind = KIND_NIW; f.coltype = COL_F32; st->has_niw = true; break;
      case MSB_FAMILY_DM: f.kind = KIND_DM; f.coltype = COL_U32; st->has_dm = true; break;
    }
  }
  // bb features that sit next to nich features (the general score kernel runs anyway) are scored in binary form
  if (st->has_nich && !getenv("MSB_NO_BINFORM"))
    for (auto &f : st->feats)
      if (f.family == FAM_BB) f.binform = 1;
  st->SS = sso;
  // default hyperparameters: microscopes/models.pyx:189,211,223,238,264-269
  st->h_hp.assign(hpo, 0.0);
  for (size_t d = 0; d < nfeatures; d++) {
    double *h = st->h_hp.data() + st->feats[d].hp_off;
    const msb_model_desc &m = models[d];
    switch (m.family) {
      case MSB_FAMILY_BB: case MSB_FAMILY_GP: case MSB_FAMILY_BBNC: h[0] = h[1] = 1.0; break;
      case MSB_FAMILY_BNB: h[0] = h[1] = h[2] = 1.0; break;  // models.pyx:200
      case MSB_FAMILY_NICH: h[0] = 0.0; h[1] = h[2] = h[3] = 1.0; break;
      case MSB_FAMILY_DM:
      case MSB_FAMILY_DD: for (uint32_t i = 0; i < m.dim; i++) h[i] = 1.0; st->feats[d].asum = (double)m.dim; break;
      case MSB_FAMILY_NIW:
        h[m.dim] = 1.0;
        for (uint32_t i = 0; i < m.dim; i++) h[m.dim + 1 + (size_t)i * m.dim + i] = 1.0;
        h[m.dim + 1 + (size_t)m.dim * m.dim] = (double)m.dim;
        break;
    }
  }
  CU_TRY(cudaMalloc(&st->d_feats, sizeof(FeatDev) * nfeatures));
  CU_TRY(cudaMalloc(&st->d_feats_scalar, sizeof(FeatDev) * nfeatures));
  CU_TRY(cudaMalloc(&st->d_hp, sizeof(double) * std::max<size_t>(hpo, 1)));
  CU_TRY(cudaMalloc(&st->d_ss, sizeof(double) * st->SS));
  CU_TRY(cudaMalloc(&st->d_delta, sizeof(double) * st->SS));
  CU_TRY(cudaMemsetAsync(st->d_ss, 0, sizeof(double) * st->SS, ctx->stream));
  CU_TRY(cudaMemsetAsync(st->d_delta, 0, sizeof(double) * st->SS, ctx->stream));
  CU_TRY(cudaMalloc(&st->d_counter, sizeof(unsigned long long) * 4));
  CU_TRY(cudaMalloc(&st->d_slot2gid, sizeof(int64_t) * max_groups));
  CU_TRY(cudaMalloc(&st->d_flags, sizeof(uint32_t) * 2 * nfeatures));
  CU_TRY(cudaHostAlloc(&st->h_flags, sizeof(uint32_t) * 2 * nfeatures, cudaHostAllocDefault));
  CU_TRY(cudaHostAlloc(&st->h_moved, sizeof(unsigned long long), cudaHostAllocMapped));
  *st->h_moved = 0;
  CU_TRY(cudaHostGetDevicePointer((void **)&st->h_moved_dev, st->h_moved, 0));
  st->slot2gid.assign(max_groups, -1);
  st->h_counts.assign(max_groups, 0.0);
  st->slot_dirty.assign(max_groups, 0);
  for (int s = (int)max_groups - 1; s >= 0; s--) st->free_slots.push_back(s);
  st->cols.assign(nfeatures, nullptr);
  st->d_niwW.assign(nfeatures, nullptr); st->d_niwBias.assign(nfeatures, nullptr);
  st->d_niwCoef.assign(nfeatures, nullptr); st->d_niwB.assign(nfeatures, nullptr);
  *out = st;
  return MSB_OK;
}

extern "C" MSB_API int msb_state_destroy(msb_state *st) {
  if (!st) return MSB_OK;
  cudaSetDevice(st->ctx->device);
  cudaStreamSynchronize(st->ctx->copy_stream);
  cudaStreamSynchronize(st->ctx->stream);
  cudaStreamSynchronize(st->ctx->d2h_stream);
  if (!st->pass_host_ns.empty()) {
    std::string line = "msb_state_pass host ms:";
    for (auto &p : st->pass_host_ns) line += " " + p.first + "=" + std::to_string(p.second * 1e-6);
    fprintf(stderr, "%s\n", line.c_str());
  }
  if (st->ev_mapped) { cudaEventDestroy(st->ev_mapped); cudaEventDestroy(st->ev_assign_copied); }
  if (st->ev_swap) { cudaEventDestroy(st->ev_swap); cudaEventDestroy(st->ev_prefetched); }
  cudaFree(st->col_slab_b); cudaFree(st->d_feats_b); cudaFree(st->d_feats_scalar_b); cudaFree(st->d_flags_b); cudaFreeHost(st->h_flags_b);
  cudaFree(st->col_slab);
  for (size_t d = 0; d < st->D; d++) { cudaFree(st->d_niwW[d]); cudaFree(st->d_niwBias[d]); cudaFree(st->d_niwCoef[d]); cudaFree(st->d_niwB[d]); }
  cudaFree(st->d_niwA16);
  cudaFree(st->d_rowmax);
  cudaFree(st->d_grid); cudaFree(st->d_hpwork); cudaFree(st->d_theta); cudaFree(st->d_hpsl);
  cudaFree(st->d_feats); cudaFree(st->d_feats_scalar); cudaFree(st->d_hp); cudaFree(st->d_ss); cudaFree(st->d_delta); cudaFree(st->d_delta_i32); cudaFree(st->d_counter);
  cudaFree(st->d_slot2gid); cudaFree(st->d_assign64); cudaFree(st->d_flags); cudaFreeHost(st->h_moved); cudaFreeHost(st->h_flags); cudaFree(st->d_assign); cudaFree(st->d_params); cudaFree(st->d_scores);
  cudaFree(st->d_base); cudaFree(st->d_base_score); cudaFree(st->d_col2slot); cudaFree(st->d_newslot); cudaFree(st->d_newcol); cudaFree(st->d_uniforms);
  for (auto &ring : st->events) for (auto &pe : ring) for (auto &e : pe.e) cudaEventDestroy(e);
  delete st;
  return MSB_OK;
}

static int sync_small(msb_state *st) {  // upload hypers / feature descriptors if they changed
  if (st->hp_dirty) {
    CU_TRY(cudaMemcpyAsync(st->d_hp, st->h_hp.data(), sizeof(double) * st->h_hp.size(), cudaMemcpyHostToDevice, st->ctx->stream));
    st->hp_dirty = false;
  }
  if (st->feats_dirty) {
    CU_TRY(cudaMemcpyAsync(st->d_feats, st->feats.data(), sizeof(FeatDev) * st->D, cudaMemcpyHostToDevice, st->ctx->stream));
    // Order in which the score kernel walks the scalar features (a sum, so any order is valid): the
    // FMA-bound ones (nich) are spread evenly between the shared-memory-bound table lookups, so that warps of
    // one block that have drifted apart by a feature keep both pipes busy instead of all queueing on one
    // (C5: 58.8 -> 50.6 ms).  Forcing the overlap with two warp groups that walk each window of features in
    // rotated order was measured too and is not kept: with 2 warps per SM sub-partition neither group
    // saturates its pipe (57.8 ms).
    std::vector<FeatDev> sc, light, heavy;
    for (auto f : st->feats) {
      f.fuse = 0; f.bundle_last = 1; f.sx_off = f.sc_off = 0;
      if (f.rows > 0) (f.kind == KIND_NICH ? heavy : light).push_back(f);
    }
    static const bool no_interleave = getenv("MSB_NO_INTERLEAVE") != nullptr, no_fuse = getenv("MSB_NO_FUSE") != nullptr;
    if (heavy.empty() || light.empty() || no_interleave) {
      for (const auto &f : st->feats) if (f.rows > 0) { sc.push_back(f); sc.back().fuse = 0; }
    } else {
      // Fused quads first (score_bundle_kernel): [bb in binary form, table, table, nich] walked together, one row step
      // doing the two lookups next to the nich arithmetic.  Tables are paired first half with second half of their
      // list, so that a family with big chunks (gp) meets one with small chunks (dd) and every quad fills about the
      // same share of a stage.
      std::vector<FeatDev> bins, tabs, rest;
      for (const auto &f : light) ((f.kind == KIND_TABLE && f.binform) ? bins : tabs).push_back(f);
      const size_t Q = no_fuse ? 0 : std::min(bins.size(), std::min(tabs.size() / 2, heavy.size()));
      const size_t half = tabs.size() / 2;
      for (size_t q = 0; q < Q; q++) {
        sc.push_back(bins[q]); sc.back().fuse = 1;
        sc.push_back(tabs[q]);
        sc.push_back(tabs[half + q]);
        sc.push_back(heavy[q]);
      }
      for (size_t i = Q; i < bins.size(); i++) rest.push_back(bins[i]);
      for (size_t i = 0; i < tabs.size(); i++) if (!(i < Q || (i >= half && i < half + Q))) rest.push_back(tabs[i]);
      // the others: nich features spread evenly between the table lookups
      const size_t nh = heavy.size() - Q;
      size_t li = 0;
      for (size_t h = 0; h < nh; h++) {
        const size_t upto = rest.size() * (h + 1) / nh;
        while (li < upto) sc.push_back(rest[li++]);
        sc.push_back(heavy[Q + h]);
      }
      while (li < rest.size()) sc.push_back(rest[li++]);
    }
    st->n_scalar = sc.size();
    st->sc_host = sc;        // kept: launch_score lays the bundles of score_bundle_kernel out for the tile shape in use
    st->bundle_key = 0;      // ... and uploads the list again when that layout changes
    if (!sc.empty())
      CU_TRY(cudaMemcpy(st->d_feats_scalar, sc.data(), sizeof(FeatDev) * sc.size(), cudaMemcpyHostToDevice));
    st->feats_dirty = false;
  }
  // the host vectors are pageable: the copies above have completed on return
  return MSB_OK;
}

static void layout_chunks(msb_state *st) {
  uint32_t ro = 0, mx = 0;
  for (auto &f : st->feats) {
    switch (f.kind) {
      case KIND_TABLE: f.rows = f.binform ? 2 : f.ncat + 1; break;
      case KIND_GP: f.rows = f.ncat + 4; break;
      case KIND_NICH: f.rows = 4; break;
      default: f.rows = 0; break;
    }
    f.rowoff = ro;
    ro += f.rows;
    mx = std::max(mx, f.rows);
  }
  st->region_rows = ro;
  st->max_chunk_rows = mx;
  st->tables_only = false;  // decided at the end of bind, once the slow-path masks are known
  st->feats_dirty = true;
}

// Fused AoS -> SoA conversion (ingest_tile_kernel): rows per block chosen so that several blocks share an SM (a tile of at
// most 56 KB) -- one block's tile load then overlaps another's conversion; 512 threads per block whatever the tile.
static size_t ingest_tile_bytes(const msb_dataview *dv, size_t TR) {
  return ((size_t)TR * (dv->rowsize / 4 + 1) + (dv->d_mask ? (size_t)TR * (dv->maskrowsize / 4 + 1) : 0)) * 4;
}
static int ingest_rows_per_block(const msb_ctx *ctx, const msb_dataview *dv) {
  for (int TR : {512, 256, 128}) if (ingest_tile_bytes(dv, TR) <= 56 * 1024) return TR;
  return ingest_tile_bytes(dv, 64) <= ctx->smem_optin ? 64 : 0;
}
static cudaError_t launch_ingest_tile(msb_ctx *ctx, cudaStream_t stream, int TR, const msb_dataview *dv, size_t n_pad, const FeatDev *d_feats,
                                      int D, uint32_t *d_flags) {
  const size_t smem = ingest_tile_bytes(dv, TR);
  const unsigned grid = (unsigned)(n_pad / TR);
  const uint32_t rw = (uint32_t)(dv->rowsize / 4), mw = (uint32_t)(dv->maskrowsize / 4);
  ctx->prof.begin("ingest_tile_kernel", stream);
  switch (TR) {
    case 512: ingest_tile_kernel<512, 1><<<grid, 512, smem, stream>>>(dv->d_data, dv->d_mask, dv->n, n_pad, rw, mw, d_feats, D, d_flags); break;
    case 256: ingest_tile_kernel<256, 2><<<grid, 512, smem, stream>>>(dv->d_data, dv->d_mask, dv->n, n_pad, rw, mw, d_feats, D, d_flags); break;
    case 128: ingest_tile_kernel<128, 4><<<grid, 512, smem, stream>>>(dv->d_data, dv->d_mask, dv->n, n_pad, rw, mw, d_feats, D, d_flags); break;
    default: ingest_tile_kernel<64, 8><<<grid, 512, smem, stream>>>(dv->d_data, dv->d_mask, dv->n, n_pad, rw, mw, d_feats, D, d_flags); break;
  }
  ctx->prof.end(stream);
  ctx->launches++;
  return cudaGetLastError();
}

// per-feature "some cell needs the slow path" flags -> host; decides the tables-only kernel variant
static int ingest_flags(msb_state *st, bool force_dirty) {
  msb_ctx *ctx = st->ctx;
  const size_t D = st->D;
  CU_TRY(cudaMemcpyAsync(st->h_flags, st->d_flags, sizeof(uint32_t) * D, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(cudaStreamSynchronize(ctx->stream));
  bool any = false, changed = false;
  for (size_t d = 0; d < D; d++) {
    changed |= st->feats[d].has_slow != st->h_flags[d];
    st->feats[d].has_slow = st->h_flags[d];
    any |= st->h_flags[d] != 0;
  }
  // the tables-only kernel has no slow path and no nich code: gp features qualify when no count exceeds their table
  st->tables_only = !any && !st->has_nich && !getenv("MSB_NO_TABLES_ONLY");
  if (changed || force_dirty) st->feats_dirty = true;
  return MSB_OK;
}

// Reads the bound dataview into the Value-typed columns (pack_kernel) and the score columns + slow-path
// masks (scorecol_kernel).  size_tables: also size the gp lookup tables from the column maxima (bind);
// a refresh keeps the table sizes, counts beyond them take the score kernel's closed-form path.
static int ingest(msb_state *st, bool size_tables) {
  msb_ctx *ctx = st->ctx;
  msb_dataview *dv = st->dv;
  const size_t D = st->D;
  st->col_version++;   // the column data changes: anything derived from it (the fp16 NIW operand) is stale
  MSB_TRY(sync_small(st));
  CU_TRY(dv_acquire(dv));
  // refresh path: one fused pass over the records staged in shared memory (they are read from HBM once)
  const int TR = ingest_rows_per_block(ctx, dv);
  static const bool no_fused = getenv("MSB_NO_FUSED_INGEST") != nullptr;
  if (!size_tables && dv->n && st->has_scalar && dv->rowsize % 4 == 0 && (!dv->d_mask || dv->maskrowsize % 4 == 0) && TR && !no_fused) {
    CU_TRY(cudaMemsetAsync(st->d_flags, 0, sizeof(uint32_t) * D, ctx->stream));
    CU_TRY(launch_ingest_tile(ctx, ctx->stream, TR, dv, st->n_pad, st->d_feats, (int)D, st->d_flags));
    CU_TRY(dv_release(dv));
    return ingest_flags(st, false);
  }
  if (dv->n) {
    dim3 grid(cdiv(dv->n, 256), (unsigned)D);
    LAUNCH(ctx, pack_kernel, grid, 256, 0, dv->d_data, dv->d_mask, dv->n, dv->rowsize, dv->maskrowsize, st->d_feats, (int)D);
  }
  CU_TRY(dv_release(dv));
  if (!size_tables && dv->n)  // refresh without the fused kernel: re-centre the niw rows with the centres chosen at bind
    for (size_t d = 0; d < D; d++) {
      const FeatDev &f = st->feats[d];
      if (f.kind == KIND_NIW)
        LAUNCH(ctx, niw_center_kernel, cdiv(dv->n * (size_t)f.dim, 256), 256, 0, (const float *)f.col, dv->n, (int)f.dim,
               (const float *)f.slowmask, (float *)const_cast<uint32_t *>(f.scol));
    }
  if (size_tables) {
    std::vector<size_t> gp;
    for (size_t d = 0; d < D; d++) if (st->feats[d].kind == KIND_GP) gp.push_back(d);
    if (!gp.empty()) {
      uint32_t *d_max = st->d_flags + D;
      CU_TRY(cudaMemsetAsync(d_max, 0, sizeof(uint32_t) * gp.size(), ctx->stream));
      if (dv->n)
        for (size_t i = 0; i < gp.size(); i++)
          LAUNCH(ctx, colmax_u32_kernel, std::min<unsigned>(cdiv(dv->n, 256), 1024), 256, 0,
                 (const uint32_t *)st->cols[gp[i]], dv->n, d_max + i);
      CU_TRY(cudaMemcpyAsync(st->h_flags + D, d_max, sizeof(uint32_t) * gp.size(), cudaMemcpyDeviceToHost, ctx->stream));
      CU_TRY(cudaStreamSynchronize(ctx->stream));
      const uint32_t cap_limit = 252;  // chunk rows = cap + 4 <= 256
      for (size_t i = 0; i < gp.size(); i++) st->feats[gp[i]].ncat = std::min<uint32_t>(st->h_flags[D + i] + 1, cap_limit);
    }
    // Centre of every niw column, coordinate by coordinate, under the same rule as nich below: the GEMM form
    // |W x - W mu'|^2 never subtracts first, so its fp32 error grows with |x| / sigma (measured: 3e-6 at an offset of
    // 10 sigma, 2.8e-5 at 100, 2.4e-4 at 1000 -- scripts/niw_offset_accuracy.py); the scorers read x - c instead.
    for (size_t d = 0; d < D; d++) {
      const FeatDev &f = st->feats[d];
      if (f.kind != KIND_NIW) continue;
      const int dim = (int)f.dim;
      std::vector<float> cen(dim, 0.f);
      if (dv->n) {
        Scratch<double> d_sum;
        Scratch<uint32_t> d_mm;
        CU_TRY(d_sum.alloc(2 * dim));
        CU_TRY(d_mm.alloc(2 * dim));
        std::vector<uint32_t> h_mm(2 * dim);
        for (int j = 0; j < dim; j++) { h_mm[2 * j] = 0xFFFFFFFFu; h_mm[2 * j + 1] = 0u; }
        CU_TRY(cudaMemsetAsync(d_sum, 0, sizeof(double) * 2 * dim, ctx->stream));
        CU_TRY(cudaMemcpyAsync(d_mm, h_mm.data(), sizeof(uint32_t) * h_mm.size(), cudaMemcpyHostToDevice, ctx->stream));
        dim3 grid(std::min<unsigned>(cdiv(dv->n, 256), 256), (unsigned)dim);
        LAUNCH(ctx, niw_colstats_kernel, grid, 256, 0, (const float *)f.col, dv->n, dim, d_sum.p, d_mm.p);
        std::vector<double> h_sum(2 * dim);
        CU_TRY(cudaMemcpyAsync(h_sum.data(), d_sum, sizeof(double) * h_sum.size(), cudaMemcpyDeviceToHost, ctx->stream));
        CU_TRY(cudaMemcpyAsync(h_mm.data(), d_mm, sizeof(uint32_t) * h_mm.size(), cudaMemcpyDeviceToHost, ctx->stream));
        CU_TRY(cudaStreamSynchronize(ctx->stream));
        auto unkey = [](uint32_t k) { const uint32_t b = (k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k; float v; memcpy(&v, &b, 4); return v; };
        for (int j = 0; j < dim; j++) {
          if (!(h_sum[2 * j + 1] > 0.0)) continue;
          const double mean = h_sum[2 * j] / h_sum[2 * j + 1];
          const double lo = unkey(h_mm[2 * j]), hi = unkey(h_mm[2 * j + 1]);
          if (std::isfinite(mean) && std::max(hi - mean, mean - lo) <= 0.25 * std::fabs(mean)) cen[j] = (float)mean;
        }
      }
      CU_TRY(cudaMemcpyAsync(const_cast<uint32_t *>(f.slowmask), cen.data(), sizeof(float) * dim, cudaMemcpyHostToDevice, ctx->stream));
      CU_TRY(cudaStreamSynchronize(ctx->stream));  // cen is a local
      if (dv->n)
        LAUNCH(ctx, niw_center_kernel, cdiv(dv->n * (size_t)dim, 256), 256, 0, (const float *)f.col, dv->n, dim, (const float *)f.slowmask,
               (float *)const_cast<uint32_t *>(f.scol));
    }
    // Centre of every nich score column.  t = (x - mu') s subtracts first, which is exact near a group's own mean,
    // but the fp32 table entry of mu' carries ulp(mu') of error: for a column that sits far from 0 relative to its
    // spread (all values within |mean| / 4 of the mean) both x and mu' are stored relative to the column mean.
    // Any other column keeps c = 0: centring would cost small values their low bits.
    std::vector<size_t> nc;
    for (size_t d = 0; d < D; d++) if (st->feats[d].kind == KIND_NICH) nc.push_back(d);
    if (!nc.empty()) {
      Scratch<double> d_sum;
      Scratch<uint32_t> d_mm;
      CU_TRY(d_sum.alloc(2 * nc.size()));
      CU_TRY(d_mm.alloc(2 * nc.size()));
      std::vector<uint32_t> h_mm(2 * nc.size());
      for (size_t i = 0; i < nc.size(); i++) { h_mm[2 * i] = 0xFFFFFFFFu; h_mm[2 * i + 1] = 0u; }
      CU_TRY(cudaMemsetAsync(d_sum, 0, sizeof(double) * 2 * nc.size(), ctx->stream));
      CU_TRY(cudaMemcpyAsync(d_mm, h_mm.data(), sizeof(uint32_t) * h_mm.size(), cudaMemcpyHostToDevice, ctx->stream));
      if (dv->n)
        for (size_t i = 0; i < nc.size(); i++)
          LAUNCH(ctx, colstats_f32_kernel, std::min<unsigned>(cdiv(dv->n, 256), 1024), 256, 0, (const float *)st->cols[nc[i]], dv->n,
                 d_sum.p + 2 * i, d_mm.p + 2 * i);
      std::vector<double> h_sum(2 * nc.size());
      CU_TRY(cudaMemcpyAsync(h_sum.data(), d_sum, sizeof(double) * h_sum.size(), cudaMemcpyDeviceToHost, ctx->stream));
      CU_TRY(cudaMemcpyAsync(h_mm.data(), d_mm, sizeof(uint32_t) * h_mm.size(), cudaMemcpyDeviceToHost, ctx->stream));
      CU_TRY(cudaStreamSynchronize(ctx->stream));
      auto unkey = [](uint32_t k) { const uint32_t b = (k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k; float f; memcpy(&f, &b, 4); return f; };
      for (size_t i = 0; i < nc.size(); i++) {
        double c = 0.0;
        if (h_sum[2 * i + 1] > 0.0) {
          const double mean = h_sum[2 * i] / h_sum[2 * i + 1];
          const double lo = unkey(h_mm[2 * i]), hi = unkey(h_mm[2 * i + 1]);
          if (std::isfinite(mean) && std::max(hi - mean, mean - lo) <= 0.25 * std::fabs(mean)) c = (double)(float)mean;
        }
        st->feats[nc[i]].asum = c;
      }
    }
    layout_chunks(st);
  }
  if (st->has_scalar) {  // score columns + slow-path masks (the gp table sizes are known now)
    MSB_TRY(sync_small(st));
    CU_TRY(cudaMemsetAsync(st->d_flags, 0, sizeof(uint32_t) * D, ctx->stream));
    dim3 grid((unsigned)(st->n_pad / 256), (unsigned)D);
    LAUNCH(ctx, scorecol_kernel, grid, 256, 0, st->d_feats, (int)D, dv->n, st->n_pad, st->d_flags);
    return ingest_flags(st, size_tables);
  }
  return MSB_OK;
}

extern "C" MSB_API int msb_state_bind(msb_state *st, msb_dataview *dv) {
  REQUIRE(st && dv, "msb_state_bind: NULL argument");
  REQUIRE(dv->ctx == st->ctx, "msb_state_bind: dataview belongs to another context");
  REQUIRE(dv->D == st->D, "msb_state_bind: feature count mismatch");
  msb_ctx *ctx = st->ctx;
  CU_TRY(cudaSetDevice(ctx->device));
  for (size_t d = 0; d < st->D; d++) {
    const msb_runtime_type &t = dv->types[d];
    const msb_model_desc &m = st->models[d];
    if (m.family == MSB_FAMILY_NIW || m.family == MSB_FAMILY_DM) REQUIRE(t.n == m.dim, "shapes do not match");  // distributions.hpp:218, dm.cpp:11
    else REQUIRE(t.n == 1, "scalar model bound to a vector field");               // distributions.hpp:209
  }
  const size_t n = std::max<size_t>(dv->n, 1);
  const bool same_shape = st->col_slab && st->d_assign && st->n == dv->n;  // the column slab depends on n only
  st->dv = dv; st->n = dv->n;
  if (!same_shape) {
    cudaFree(st->col_slab); st->col_slab = nullptr;
    cudaFree(st->d_assign); st->d_assign = nullptr;
    std::vector<size_t> coff(st->D), soff(st->D), moff(st->D);
    size_t slab = 0;
    const size_t n_pad = (n + 1024 + 1023) / 1024 * 1024;  // tile-granular kernels read whole 1024-row tiles
    st->n_pad = n_pad;
    for (size_t d = 0; d < st->D; d++) {
      const FeatDev &f = st->feats[d];
      const size_t bytes = (f.kind == KIND_NIW || f.kind == KIND_DM) ? n * f.dim * sizeof(float)
                                                                    : n * (f.coltype == COL_U8 ? 1 : f.coltype == COL_U16 ? 2 : 4);
      coff[d] = slab;
      slab += (bytes + 4096 + 255) / 256 * 256;
      if (f.kind == KIND_DM) {  // no score column: dm_score_kernel reads the count rows themselves
        soff[d] = moff[d] = slab;
      } else if (f.kind != KIND_NIW) {
        soff[d] = slab; slab += n_pad * sizeof(uint32_t);
        moff[d] = slab; slab += n_pad / 32 * sizeof(uint32_t);
      } else {  // niw: the centred rows and the centre (FeatDev::scol / slowmask)
        soff[d] = slab; slab += (bytes + 4096 + 255) / 256 * 256;
        moff[d] = slab; slab += ((size_t)f.dim * sizeof(float) + 255) / 256 * 256;
      }
    }
    CU_TRY(cudaMalloc(&st->col_slab, slab));
    st->slab_bytes = slab;
    CU_TRY(cudaStreamSynchronize(ctx->copy_stream));  // a prefetch into the old shadow buffer may still be running
    cudaFree(st->col_slab_b); st->col_slab_b = nullptr;
    for (size_t d = 0; d < st->D; d++) {
      FeatDev &f = st->feats[d];
      st->cols[d] = (char *)st->col_slab + coff[d];
      f.col = st->cols[d];
      f.scol = (const uint32_t *)((char *)st->col_slab + soff[d]);
      f.slowmask = (const uint32_t *)((char *)st->col_slab + moff[d]);
    }
    CU_TRY(cudaMalloc(&st->d_assign, sizeof(int32_t) * n));
  }
  for (size_t d = 0; d < st->D; d++) {
    FeatDev &f = st->feats[d];
    f.has_slow = 0;
    f.src_off = dv->off[d]; f.msk_off = dv->moff[d];
    f.src_prim = (uint32_t)dv->types[d].prim; f.src_n = dv->types[d].n;
  }
  st->feats_dirty = true;
  if (st->prefetch_pending) { CU_TRY(cudaStreamSynchronize(ctx->copy_stream)); st->prefetch_pending = false; }
  st->feats_b.clear();  // the shadow descriptors are rebuilt from the new layout by the next msb_state_prefetch
  MSB_TRY(ingest(st, true));
  CU_TRY(cudaMemsetAsync(st->d_assign, 0xFF, sizeof(int32_t) * n, ctx->stream));  // all -1
  st->all_unassigned = true;
  return MSB_OK;
}

// The bound dataview's records were replaced in place (msb_dataview_upload): convert them again.
// Assignments and suffstats are kept -- the rows are the same entities, streamed from the host again.
extern "C" MSB_API int msb_state_refresh(msb_state *st) {
  REQUIRE(st, "NULL argument");
  REQUIRE(st->dv, "no dataview bound");
  msb_ctx *ctx = st->ctx;
  CU_TRY(cudaSetDevice(ctx->device));
  if (!st->prefetch_pending) return ingest(st, false);
  // the conversion already ran on the copy stream (msb_state_prefetch): make the two column buffers change places
  CU_TRY(cudaEventSynchronize(st->ev_prefetched));                  // its flags are on the host now
  CU_TRY(cudaStreamWaitEvent(ctx->stream, st->ev_prefetched, 0));   // kernels enqueued from here on see the new columns
  st->prefetch_pending = false;
  st->col_version++;
  std::swap(st->col_slab, st->col_slab_b);
  std::swap(st->feats, st->feats_b);
  std::swap(st->cols, st->cols_b);
  std::swap(st->d_feats, st->d_feats_b);
  std::swap(st->d_feats_scalar, st->d_feats_scalar_b);
  std::swap(st->sc_host, st->sc_host_b);
  std::swap(st->bundle_key, st->bundle_key_b);
  bool any = false, changed = st->feats_b_dirty;
  for (size_t d = 0; d < st->D; d++) {
    // fields that are not per buffer follow the buffer that was active until now
    st->feats[d].asum = st->feats_b[d].asum; st->feats[d].ncat = st->feats_b[d].ncat;
    st->feats[d].rows = st->feats_b[d].rows; st->feats[d].rowoff = st->feats_b[d].rowoff;
    changed |= st->feats[d].has_slow != st->h_flags_b[d];
    st->feats[d].has_slow = st->h_flags_b[d];
    any |= st->h_flags_b[d] != 0;
  }
  st->feats_b_dirty = false;
  st->tables_only = !any && !st->has_nich && !getenv("MSB_NO_TABLES_ONLY");
  // the device descriptors of this buffer were last used two passes ago (the prefetch waited for ev_swap), so
  // re-uploading them cannot race with a kernel; needed only when a flag or a shared field changed
  if (changed) st->feats_dirty = true;
  else {  // the feature walk order and count are unchanged: n_scalar stays valid
  }
  CU_TRY(cudaEventRecord(st->ev_swap, ctx->stream));
  st->swap_recorded = true;
  return MSB_OK;
}

// Converts the bound dataview's (re-uploaded) records into the column buffer that the running sweep does not
// read, on the copy stream, right behind the upload.  The following msb_state_refresh swaps the buffers.
extern "C" MSB_API int msb_state_prefetch(msb_state *st) {
  REQUIRE(st, "NULL argument");
  REQUIRE(st->dv, "no dataview bound");
  msb_ctx *ctx = st->ctx;
  msb_dataview *dv = st->dv;
  CU_TRY(cudaSetDevice(ctx->device));
  const size_t D = st->D;
  const int TR = ingest_rows_per_block(ctx, dv);
  const bool fused_ok = dv->n && dv->owns && st->has_scalar && dv->rowsize % 4 == 0 && (!dv->d_mask || dv->maskrowsize % 4 == 0) &&
                        TR && st->col_slab;
  if (!fused_ok || st->prefetch_pending) return MSB_OK;  // msb_state_refresh converts on the compute stream instead
  if (!st->ev_swap) {
    CU_TRY(cudaEventCreateWithFlags(&st->ev_swap, cudaEventDisableTiming));
    CU_TRY(cudaEventCreateWithFlags(&st->ev_prefetched, cudaEventDisableTiming));
    CU_TRY(cudaMalloc(&st->d_feats_b, sizeof(FeatDev) * D));
    CU_TRY(cudaMalloc(&st->d_feats_scalar_b, sizeof(FeatDev) * D));
    CU_TRY(cudaMalloc(&st->d_flags_b, sizeof(uint32_t) * 2 * D));
    CU_TRY(cudaHostAlloc(&st->h_flags_b, sizeof(uint32_t) * 2 * D, cudaHostAllocDefault));
  }
  if (!st->col_slab_b) CU_TRY(cudaMalloc(&st->col_slab_b, st->slab_bytes));
  if (st->feats_b.empty()) {  // shadow descriptors: the same layout, pointers into the second slab
    MSB_TRY(sync_small(st));
    st->feats_b = st->feats;
    st->cols_b = st->cols;
    const ptrdiff_t shift = (char *)st->col_slab_b - (char *)st->col_slab;
    for (size_t d = 0; d < D; d++) {
      FeatDev &f = st->feats_b[d];
      f.col = (char *)f.col + shift;
      st->cols_b[d] = (char *)st->cols_b[d] + shift;
      if (f.scol) f.scol = (const uint32_t *)((const char *)f.scol + shift);
      if (f.slowmask) f.slowmask = (const uint32_t *)((const char *)f.slowmask + shift);
    }
    CU_TRY(cudaStreamSynchronize(ctx->copy_stream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    for (size_t d = 0; d < D; d++)  // the niw centres belong to the layout, not to one buffer
      if (st->feats[d].kind == KIND_NIW)
        CU_TRY(cudaMemcpy(const_cast<uint32_t *>(st->feats_b[d].slowmask), st->feats[d].slowmask, sizeof(float) * st->feats[d].dim,
                          cudaMemcpyDeviceToDevice));
    CU_TRY(cudaMemcpy(st->d_feats_b, st->feats_b.data(), sizeof(FeatDev) * D, cudaMemcpyHostToDevice));
    st->feats_b_dirty = true;  // its walk-order list (d_feats_scalar_b) is built at the first swap
  }
  if (st->swap_recorded) CU_TRY(cudaStreamWaitEvent(ctx->copy_stream, st->ev_swap, 0));  // the last readers of that buffer are done
  CU_TRY(cudaMemsetAsync(st->d_flags_b, 0, sizeof(uint32_t) * D, ctx->copy_stream));
  CU_TRY(launch_ingest_tile(ctx, ctx->copy_stream, TR, dv, st->n_pad, st->d_feats_b, (int)D, st->d_flags_b));
  CU_TRY(cudaMemcpyAsync(st->h_flags_b, st->d_flags_b, sizeof(uint32_t) * D, cudaMemcpyDeviceToHost, ctx->copy_stream));
  CU_TRY(cudaEventRecord(st->ev_prefetched, ctx->copy_stream));
  dv->upload_pending = false;  // the copy stream itself consumed the upload; later uploads queue behind this kernel
  st->prefetch_pending = true;
  return MSB_OK;
}

// ---- hypers / suffstats ------------------------------------------------------
// h_hp[feature][off, off + cnt) = v, and what follows the hypers: dd's alpha sum in both feature tables, the uploads
static void write_hp(msb_state *st, size_t feature, size_t off, const double *v, size_t cnt) {
  double *h = st->h_hp.data() + st->feats[feature].hp_off;
  for (size_t i = 0; i < cnt; i++) h[off + i] = v[i];
  if (st->models[feature].family == MSB_FAMILY_DD) {
    double a = 0.0;
    for (uint32_t i = 0; i < st->models[feature].dim; i++) a += h[i];
    st->feats[feature].asum = a;
    if (!st->feats_b.empty()) { st->feats_b[feature].asum = a; st->feats_b_dirty = true; }
    st->feats_dirty = true;
  }
  st->hp_dirty = true;
}
extern "C" MSB_API int msb_state_set_hp(msb_state *st, size_t feature, const char *key, const double *v, size_t count) {
  REQUIRE(st && key && v, "NULL argument");
  REQUIRE(feature < st->D, "bad feature index");
  size_t off, cnt;
  MSB_TRY(hp_field(st->models[feature], key, &off, &cnt));
  REQUIRE(count == cnt, "wrong dimension");  // distributions.hpp:436
  write_hp(st, feature, off, v, cnt);
  return MSB_OK;
}
extern "C" MSB_API int msb_state_get_hp(msb_state *st, size_t feature, const char *key, double *v, size_t count) {
  REQUIRE(st && key && v, "NULL argument");
  REQUIRE(feature < st->D, "bad feature index");
  size_t off, cnt;
  MSB_TRY(hp_field(st->models[feature], key, &off, &cnt));
  REQUIRE(count == cnt, "wrong dimension");
  const double *h = st->h_hp.data() + st->feats[feature].hp_off;
  for (size_t i = 0; i < cnt; i++) v[i] = h[off + i];
  return MSB_OK;
}
extern "C" MSB_API int msb_state_set_cluster_hp(msb_state *st, const char *key, double v) {
  REQUIRE(st && key, "NULL argument");
  if (std::string(key) != "alpha") return fail(MSB_ERR_KEY, std::string("unknown key: ") + key);  // group_manager.hpp:130
  REQUIRE(v > 0.0, "alpha must be positive");  // group_manager.hpp:120
  st->alpha = v;
  return MSB_OK;
}
extern "C" MSB_API int msb_state_get_cluster_hp(msb_state *st, const char *key, double *v) {
  REQUIRE(st && key && v, "NULL argument");
  if (std::string(key) != "alpha") return fail(MSB_ERR_KEY, std::string("unknown key: ") + key);
  *v = st->alpha;
  return MSB_OK;
}

static int slot_of(msb_state *st, size_t gid, int *slot) {
  auto it = st->gid2slot.find(gid);
  if (it == st->gid2slot.end()) return fail(MSB_ERR_INVALID, "invalid gid");  // group_manager.hpp:157
  *slot = it->second;
  return MSB_OK;
}

// device (additive) <-> reference field representation for one group of one feature
static void ss_to_ref(const msb_model_desc &m, std::vector<double> &s) {
  if (m.family == MSB_FAMILY_NICH) {
    const double n = s[0], mean = n > 0 ? s[1] / n : 0.0;
    double ctv = n > 0 ? s[2] - s[1] * mean : 0.0;
    if (ctv < 0) ctv = 0;
    s[1] = mean; s[2] = ctv;
  }
}
static void ss_from_ref(const msb_model_desc &m, std::vector<double> &s) {
  if (m.family == MSB_FAMILY_NICH) {
    const double n = s[0], mean = s[1], ctv = s[2];
    s[1] = n * mean; s[2] = ctv + n * mean * mean;
  }
}

extern "C" MSB_API int msb_state_get_ss(msb_state *st, size_t feature, size_t gid, const char *key, double *v, size_t count) {
  REQUIRE(st && key && v, "NULL argument");
  REQUIRE(feature < st->D, "bad feature index");
  size_t off, cnt; int slot;
  MSB_TRY(ss_field(st->models[feature], key, &off, &cnt));
  REQUIRE(count == cnt, "wrong dimension");
  MSB_TRY(slot_of(st, gid, &slot));
  const FeatDev &f = st->feats[feature];
  std::vector<double> s(f.ss_w);
  CU_TRY(cudaSetDevice(st->ctx->device));
  CU_TRY(cudaMemcpyAsync(s.data(), st->d_ss + f.ss_off + (size_t)slot * f.ss_w, sizeof(double) * f.ss_w, cudaMemcpyDeviceToHost, st->ctx->stream));
  CU_TRY(cudaStreamSynchronize(st->ctx->stream));
  ss_to_ref(st->models[feature], s);
  for (size_t i = 0; i < cnt; i++) v[i] = s[off + i];
  return MSB_OK;
}
extern "C" MSB_API int msb_state_set_ss(msb_state *st, size_t feature, size_t gid, const char *key, const double *v, size_t count) {
  REQUIRE(st && key && v, "NULL argument");
  REQUIRE(feature < st->D, "bad feature index");
  size_t off, cnt; int slot;
  MSB_TRY(ss_field(st->models[feature], key, &off, &cnt));
  REQUIRE(count == cnt, "wrong dimension");
  MSB_TRY(slot_of(st, gid, &slot));
  const FeatDev &f = st->feats[feature];
  std::vector<double> s(f.ss_w);
  double *dst = st->d_ss + f.ss_off + (size_t)slot * f.ss_w;
  CU_TRY(cudaSetDevice(st->ctx->device));
  CU_TRY(cudaMemcpyAsync(s.data(), dst, sizeof(double) * f.ss_w, cudaMemcpyDeviceToHost, st->ctx->stream));
  CU_TRY(cudaStreamSynchronize(st->ctx->stream));
  ss_to_ref(st->models[feature], s);
  for (size_t i = 0; i < cnt; i++) s[off + i] = v[i];
  if (st->models[feature].family == MSB_FAMILY_DD && off > 0) {
    // count_sum is derived: it follows the counts (dd_score and score_data read it before the next apply refreshes it)
    s[0] = 0.0;
    for (size_t i = 1; i < s.size(); i++) s[0] += s[i];
  }
  ss_from_ref(st->models[feature], s);
  st->slot_dirty[slot] = 1;
  CU_TRY(cudaMemcpyAsync(dst, s.data(), sizeof(double) * f.ss_w, cudaMemcpyHostToDevice, st->ctx->stream));
  CU_TRY(cudaStreamSynchronize(st->ctx->stream));
  return MSB_OK;
}

// ---- groups (group_manager.hpp:133-216) -------------------------------------
// The per-group entity counts live on the device (d_ss[0..kmax)); the host copy is refreshed lazily,
// only when a host-side question needs it, so that sweeps never wait for the stream.
static int host_counts(msb_state *st) {
  if (!st->counts_stale) return MSB_OK;
  CU_TRY(cudaSetDevice(st->ctx->device));
  CU_TRY(cudaMemcpyAsync(st->h_counts.data(), st->d_ss, sizeof(double) * st->kmax, cudaMemcpyDeviceToHost, st->ctx->stream));
  CU_TRY(cudaStreamSynchronize(st->ctx->stream));
  st->counts_stale = false;
  return MSB_OK;
}
extern "C" MSB_API int msb_state_nentities(msb_state *st, size_t *n) { REQUIRE(st && n, "NULL argument"); *n = st->n; return MSB_OK; }
extern "C" MSB_API int msb_state_ngroups(msb_state *st, size_t *n) { REQUIRE(st && n, "NULL argument"); *n = st->gid2slot.size(); return MSB_OK; }
extern "C" MSB_API int msb_state_groups(msb_state *st, size_t *gids, size_t cap, size_t *n) {
  REQUIRE(st && n, "NULL argument");
  *n = st->gid2slot.size();
  if (gids) {
    REQUIRE(cap >= *n, "buffer too small");
    size_t i = 0;
    for (auto &p : st->gid2slot) gids[i++] = p.first;
  }
  return MSB_OK;
}
extern "C" MSB_API int msb_state_empty_groups(msb_state *st, size_t *gids, size_t cap, size_t *n) {
  REQUIRE(st && n, "NULL argument");
  MSB_TRY(host_counts(st));
  size_t c = 0;
  for (auto &p : st->gid2slot)
    if (st->h_counts[p.second] == 0.0) {
      if (gids) { REQUIRE(c < cap, "buffer too small"); gids[c] = p.first; }
      c++;
    }
  *n = c;
  return MSB_OK;
}
extern "C" MSB_API int msb_state_groupsize(msb_state *st, size_t gid, size_t *count) {
  REQUIRE(st && count, "NULL argument");
  int slot;
  MSB_TRY(slot_of(st, gid, &slot));
  MSB_TRY(host_counts(st));
  *count = (size_t)st->h_counts[slot];
  return MSB_OK;
}
// ---- per-group parameter draws (bbnc: p ~ Beta(alpha, beta), bbnc.cpp:120-125) on the host, from the same
// counter-based Philox stream as everything else: key = group_seed, counter = (gid, feature, draw index), so
// every replica of a multi-GPU state draws the same p without communicating.  (The reference draws from its
// std engine; the stream differs, the distribution does not.)
struct PhiloxStream {
  uint64_t seed, a, b;
  uint32_t i = 0;
  double u01() {  // 53-bit uniform in (0, 1)
    uint32_t r[4];
    philox4x32_10(seed, a, (b << 20) | (i++), r);
    const uint64_t bits = ((uint64_t)(r[0] >> 5) << 26) | (uint64_t)(r[1] >> 6);  // 27 + 26 = 53 bits
    return ((double)bits + 0.5) * (1.0 / 9007199254740992.0);
  }
  double normal() { return std::sqrt(-2.0 * std::log(u01())) * std::cos(6.283185307179586 * u01()); }
  double gamma(double k) {  // Marsaglia-Tsang
    if (k < 1.0) return gamma(k + 1.0) * std::pow(u01(), 1.0 / k);
    const double d = k - 1.0 / 3.0, c = 1.0 / std::sqrt(9.0 * d);
    for (;;) {
      double x, v;
      do { x = normal(); v = 1.0 + c * x; } while (v <= 0.0);
      v = v * v * v;
      const double u = u01();
      if (u < 1.0 - 0.0331 * x * x * x * x || std::log(u) < 0.5 * x * x + d * (1.0 - v + std::log(v))) return d * v;
    }
  }
  double beta(double al, double be) { const double x = gamma(al), y = gamma(be); return x / (x + y); }
};

// restore == true: *gid is the identifier to give the group (deserialisation, group_manager.hpp:92-105:
// identifiers are preserved and gcount becomes 1 + the largest one seen)
static int create_group_impl(msb_state *st, size_t *gid, bool restore) {
  REQUIRE(st && gid, "NULL argument");
  if (restore) REQUIRE(st->gid2slot.find(*gid) == st->gid2slot.end(), "group id already in use");
  if (st->free_slots.empty()) return fail(MSB_ERR_NOMEM, "max_groups reached");
  CU_TRY(cudaSetDevice(st->ctx->device));
  const int slot = st->free_slots.back();
  st->free_slots.pop_back();
  size_t g;
  if (restore) { g = *gid; st->gcount = std::max(st->gcount, g + 1); }
  else g = st->gcount++;  // group_manager.hpp:199
  st->gid2slot[g] = slot;
  st->slot2gid[slot] = (int64_t)g;
  st->cols_dirty = st->slot2gid_dirty = true;
  MSB_TRY(host_counts(st));
  st->h_counts[slot] = 0.0;
  // Group::init: zero suffstats (distributions.hpp:351); a slot nobody has written since the state was
  // created is still zero from the initial memset
  if (st->slot_dirty[slot]) {
    CU_TRY(cudaMemsetAsync(st->d_ss + slot, 0, sizeof(double), st->ctx->stream));
    for (auto &f : st->feats)
      CU_TRY(cudaMemsetAsync(st->d_ss + f.ss_off + (size_t)slot * f.ss_w, 0, sizeof(double) * f.ss_w, st->ctx->stream));
    st->slot_dirty[slot] = 0;
  }
  if (st->has_bbnc) {  // hypers::create_group of bbnc samples the group's p (bbnc.cpp:120-125)
    for (size_t d = 0; d < st->D; d++) {
      const FeatDev &f = st->feats[d];
      if (f.family != FAM_BBNC) continue;
      PhiloxStream rng{st->group_seed, (uint64_t)g, (uint64_t)d};
      const double *h = st->h_hp.data() + f.hp_off;
      const double p = rng.beta(h[0], h[1]);
      CU_TRY(cudaMemcpyAsync(st->d_ss + f.ss_off + (size_t)slot * f.ss_w, &p, sizeof(double), cudaMemcpyHostToDevice, st->ctx->stream));
    }
    CU_TRY(cudaStreamSynchronize(st->ctx->stream));  // p is a local
    st->slot_dirty[slot] = 1;
  }
  *gid = g;
  return MSB_OK;
}
extern "C" MSB_API int msb_state_create_group(msb_state *st, size_t *gid) { return create_group_impl(st, gid, false); }
extern "C" MSB_API int msb_state_restore_group(msb_state *st, size_t gid) { return create_group_impl(st, &gid, true); }
extern "C" MSB_API int msb_state_delete_group(msb_state *st, size_t gid) {
  REQUIRE(st, "NULL argument");
  int slot;
  MSB_TRY(slot_of(st, gid, &slot));
  MSB_TRY(host_counts(st));
  if (st->h_counts[slot] != 0.0) return fail(MSB_ERR_STATE, "group not empty");  // group_manager.hpp:211
  st->gid2slot.erase(gid);
  st->slot2gid[slot] = -1;
  st->cols_dirty = st->slot2gid_dirty = true;
  st->free_slots.push_back(slot);
  return MSB_OK;
}

// ---- workspace helpers ---------------------------------------------------------
template <typename T> static int ensure(T **p, size_t *cap, size_t need) {
  if (*cap >= need && *p) return MSB_OK;
  if (*p) { CU_TRY(cudaFree(*p)); *p = nullptr; }
  const size_t ncap = need + need / 8 + 64;
  cudaError_t e = cudaMalloc(p, sizeof(T) * ncap);
  if (e != cudaSuccess) { *cap = 0; return fail(MSB_ERR_NOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e)); }
  *cap = ncap;
  return MSB_OK;
}

static int ensure_rows(msb_state *st, size_t nrows) {
  if (st->row_cap >= nrows && st->d_newslot) return MSB_OK;
  cudaFree(st->d_newslot); cudaFree(st->d_newcol); cudaFree(st->d_uniforms);
  st->d_newslot = st->d_newcol = nullptr; st->d_uniforms = nullptr;
  const size_t cap = nrows + 64;
  CU_TRY(cudaMalloc(&st->d_newslot, sizeof(int32_t) * cap));
  CU_TRY(cudaMalloc(&st->d_newcol, sizeof(int32_t) * cap));
  CU_TRY(cudaMalloc(&st->d_uniforms, sizeof(float) * cap));
  st->row_cap = cap;
  return MSB_OK;
}

// Score-kernel shapes (V groups per lane, RW rows per warp, NW warps per block):
//   0: V=1 RW=64 NW=16  1024 rows x 32 groups  -- big tables (dd with many categories): the table chunk is
//                                                 re-read from L2 once per block, so maximise rows per block
//   1: V=2 RW=32 NW=16   512 rows x 64 groups
//   2: V=4 RW=32 NW=8    256 rows x 128 groups -- small chunks, many groups: fewest instructions per lookup
//   3: V=1 RW=32 NW=8    256 rows x 32 groups  -- K <= 32
//   4: V=4 RW=16 NW=16   256 rows x 128 groups on 16 warps (score_bundle_kernel only)
struct ScoreCfg { int V, RW, NW; };
static const ScoreCfg k_score_cfgs[5] = {{1, 64, 16}, {2, 32, 16}, {4, 32, 8}, {1, 32, 8}, {4, 16, 16}};

static int choose_cfg(const msb_state *st, size_t ncols) {
  if (const char *e = getenv("MSB_SCORE_CFG")) {
    const int c = atoi(e);
    if (c >= 0 && c < 4) return c;
    if (c == 4 && !st->tables_only && st->has_scalar) return c;
  }
  if (ncols <= 32) return 3;
  if (st->max_chunk_rows >= 128) return 0;
  if (ncols >= 256) return 2;
  return 1;
}

// Column order = ascending gid (std::map iteration order of group_manager.hpp:171-178);
// base[c] = log(pseudocount) (group_manager.hpp:274-283).
static int prepare_columns(msb_state *st) {
  msb_ctx *ctx = st->ctx;
  const size_t K = st->gid2slot.size();
  REQUIRE(K > 0, "no groups");
  const int cfg = choose_cfg(st, K);
  st->cfg = cfg;
  st->V = k_score_cfgs[cfg].V;
  const size_t KT = 32 * (size_t)st->V;
  st->ld = (K + KT - 1) / KT * KT;
  if (st->cols_dirty) {  // groups were created / deleted: rebuild and upload the column tables
    st->h_col2slot.resize(K); st->h_colgid.resize(K);
    size_t c = 0;
    for (auto &p : st->gid2slot) { st->h_col2slot[c] = p.second; st->h_colgid[c] = p.first; c++; }
    MSB_TRY(ensure(&st->d_col2slot, &st->col_cap, K));
    CU_TRY(cudaMemcpyAsync(st->d_col2slot, st->h_col2slot.data(), sizeof(int32_t) * K, cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));  // pageable source, reused next time
    st->cols_dirty = false;
  }
  MSB_TRY(ensure(&st->d_base, &st->base_cap, st->ld));
  LAUNCH(ctx, base_kernel, 1, 256, 0, st->d_ss, st->d_col2slot, (int)K, (int)st->ld, (float)st->alpha, st->d_base);
  return MSB_OK;
}

static int build_params(msb_state *st) {
  msb_ctx *ctx = st->ctx;
  const size_t K = st->h_col2slot.size();
  MSB_TRY(sync_small(st));
  const size_t KT = 32 * (size_t)st->V;
  const size_t ktiles = st->ld / KT;
  if (st->has_scalar) {
    MSB_TRY(ensure(&st->d_params, &st->params_cap, ktiles * st->region_rows * KT));
    // enough blocks for a few waves even when D x ktiles is small: big chunks are sliced along z
    const unsigned zs = (unsigned)std::max<size_t>(1, std::min<size_t>(8, st->max_chunk_rows * KT / 2048));
    dim3 grid((unsigned)st->D, (unsigned)ktiles, zs);
    // ragged last k-tile with at most 16 groups (V = 1, tables only): replicated columns, several rows per lookup
    const size_t tail_cols = K - (ktiles - 1) * KT;
    st->tail_g = (st->V == 1 && st->tables_only && tail_cols <= 16 && !getenv("MSB_NO_TAIL_TILE")) ? (tail_cols <= 8 ? 8 : 16) : 0;
    LAUNCH(ctx, build_params_kernel, grid, 256, 0, st->d_feats, (int)st->D, st->d_hp, st->d_ss, st->d_col2slot, (int)K,
           (int)KT, st->region_rows, st->d_params, st->tail_g);
    MSB_TRY(ensure(&st->d_base_score, &st->base_score_cap, st->ld));
    LAUNCH(ctx, copy_f32_kernel, cdiv(st->ld, 256), 256, 0, (const float *)st->d_base, st->d_base_score, st->ld);
    if (st->has_nich) {  // fold sum_d c0 of the nich features into the score kernel's base[]
      LAUNCH(ctx, nich_c0_sum_kernel, cdiv(st->ld, 128), 128, 0, st->d_feats, (int)st->D, st->d_params, st->region_rows,
             (int)KT, (int)st->ld, st->d_base_score);
    }
  }
  if (st->has_niw) {
    for (size_t d = 0; d < st->D; d++) {
      const FeatDev &f = st->feats[d];
      if (f.kind != KIND_NIW) continue;
      if (st->niw_cols_cap < K || !st->d_niwW[d]) {
        // growing K on the sweep path: the kernels of earlier sweeps may still read the old buffers
        CU_TRY(cudaStreamSynchronize(ctx->stream));
        CU_TRY(cudaFree(st->d_niwW[d])); st->d_niwW[d] = nullptr;
        CU_TRY(cudaFree(st->d_niwBias[d])); st->d_niwBias[d] = nullptr;
        CU_TRY(cudaFree(st->d_niwCoef[d])); st->d_niwCoef[d] = nullptr;
        CU_TRY(cudaFree(st->d_niwB[d])); st->d_niwB[d] = nullptr;
        const size_t cap = st->ld + 64;
        CU_TRY(cudaMalloc(&st->d_niwW[d], sizeof(float) * cap * f.dim * f.dim));
        CU_TRY(cudaMalloc(&st->d_niwBias[d], sizeof(float) * cap * f.dim));
        CU_TRY(cudaMalloc(&st->d_niwCoef[d], sizeof(float) * cap * 4));
        CU_TRY(cudaMalloc(&st->d_niwB[d], niw_tc_operand_bytes(cap, f.dim)));
        st->niw_a16_version = 0;   // the column maxima lived in the old buffer
      }
      const size_t smem = (2 * (size_t)f.dim * f.dim + f.dim) * sizeof(double);
      LAUNCH(ctx, niw_prepare_kernel, (unsigned)K, 128, smem, f, st->d_hp, st->d_ss, st->d_col2slot, st->d_niwW[d],
             st->d_niwBias[d], st->d_niwCoef[d]);
    }
    st->niw_cols_cap = std::max(st->niw_cols_cap, K);
  }
  return MSB_OK;
}

// first row the score kernel's grid covers: bulk copies of the row-value tiles need 16-byte aligned sources
static inline size_t row_origin(size_t row_lo) { return row_lo & ~(size_t)127; }

// scores is indexed from row_origin(row_lo): element (row, col) at (row - org) * ld + col (or blocked)
// dm term of the score matrix: the 32-group tile kernel while its transposed e-tile fits in shared memory, else one block per group
template <typename OUT>
static int launch_dm(msb_ctx *ctx, const FeatDev &f, const double *d_hp, const double *d_ss, const int32_t *d_col2slot, size_t K,
                     OUT *scores, size_t ld, size_t row_lo, size_t row_hi) {
  const size_t nrows = row_hi - row_lo;
  const size_t smem = ((size_t)f.dim * 32 + 64) * sizeof(double);
  if (smem <= 200 * 1024 && !getenv("MSB_DM_NO_TILE")) {
    if (smem > 48 * 1024)
      CU_TRY(cudaFuncSetAttribute(dm_score_tile_kernel<OUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(cdiv(nrows, DM_TILE_ROWS), cdiv(K, 32));
    LAUNCH(ctx, dm_score_tile_kernel<OUT>, grid, 256, smem, f, d_hp, d_ss, d_col2slot, (int)K, scores, ld, row_lo, row_hi);
  } else {
    dim3 grid(cdiv(nrows, 128), (unsigned)K);
    LAUNCH(ctx, dm_score_kernel<OUT>, grid, 128, (size_t)f.dim * sizeof(double), f, d_hp, d_ss, d_col2slot, scores, ld, row_lo, row_hi);
  }
  return MSB_OK;
}

static int launch_score(msb_state *st, size_t row_lo, size_t row_hi, float *scores, bool blocked = false, bool want_rowmax = false) {
  msb_ctx *ctx = st->ctx;
  st->rowmax_valid = false;
  const size_t org = row_origin(row_lo);
  const size_t nrows = row_hi - org;
  const size_t K = st->h_col2slot.size();
  const size_t KT = 32 * (size_t)st->V;
  const size_t ktiles = st->ld / KT;
  if (st->has_scalar) {
    const ScoreCfg c = k_score_cfgs[st->cfg];
    const size_t RB = (size_t)c.NW * c.RW;
    const size_t chunk_off = (RB * 4 + RB / 8 + 127) / 128 * 128;
    const size_t fixed = st->n_scalar * sizeof(FeatS) + 2 * 8 * sizeof(uint64_t) + 256;
    size_t stage = (chunk_off + st->max_chunk_rows * KT * sizeof(float) + 127) / 128 * 128;
    if (stage + fixed > ctx->smem_optin) return fail(MSB_ERR_UNSUPPORTED, "parameter chunk does not fit in shared memory");
    const int S = (int)std::max<size_t>(1, std::min<size_t>(8, (ctx->smem_optin - fixed) / stage));
    // the blocked epilogue transposes 32 x KT tiles through the (drained) stage ring
    const size_t tile = RB * (KT + 1) * sizeof(float);   // one 32-row x KT tile per 32 rows of the block
    if (blocked && (size_t)S * stage < tile) stage = ((tile + S - 1) / S + 127) / 128 * 128;
    const size_t smem = (size_t)S * stage + fixed;
    const size_t grid = (size_t)cdiv(nrows, RB) * ktiles;
    if (grid >= (1ull << 31)) return fail(MSB_ERR_UNSUPPORTED, "score grid too large: sweep a smaller row range");
    static const bool no_bundle = getenv("MSB_NO_BUNDLE") != nullptr;
    const bool persistent = getenv("MSB_PERSISTENT") != nullptr;   // read per call: the test switches it
    // The sweep's sampler takes the row maxima from the blocked epilogues of score_bundle_kernel and score_kernel when
    // nothing is added to the matrix afterwards (NIW, dm).  The persistent tables-only kernel stores straight from
    // registers, where a lane holds one group of 32 rows rather than one row, and does not emit them.
    int *rowmax = nullptr;
    if (want_rowmax && blocked && !st->has_niw && !st->has_dm && !(st->tables_only && persistent) && !getenv("MSB_NO_ROWMAX")) {
      const size_t need = nrows + 128;
      if (st->rowmax_cap < need) {
        CU_TRY(cudaFree(st->d_rowmax)); st->d_rowmax = nullptr; st->rowmax_cap = 0;
        CU_TRY(cudaMalloc(&st->d_rowmax, need * sizeof(int)));
        st->rowmax_cap = need;
      }
      CU_TRY(cudaMemsetAsync(st->d_rowmax, 0x80, need * sizeof(int), ctx->stream));   // below every finite float in the ordered encoding
      rowmax = st->d_rowmax;
      st->rowmax_valid = true;
    }
    if (!st->tables_only && !no_bundle && (st->cfg == 1 || st->cfg == 2 || st->cfg == 4)) {
      // General kernel, bundled ring (score_bundle_kernel): three stages of a third of the shared memory each, every
      // stage filled with as many consecutive features of the walk order as fit.
      const size_t fixed_b = st->n_scalar * (sizeof(FeatS) + 8) + 2 * 8 * sizeof(uint64_t) + 256;
      const size_t xm = (RB * 4 + RB / 8 + 127) / 128 * 128;
      const size_t biggest = (xm + st->max_chunk_rows * KT * sizeof(float) + 127) / 128 * 128;
      // stages: measured on C5 (fused quads of ~64 KB) 2 stages 44.4 ms, 3 stages 47.5 ms; on C3 (nich only) 3 and 6 alike
      static const int want_stages = getenv("MSB_BUNDLE_STAGES") ? atoi(getenv("MSB_BUNDLE_STAGES")) : 0;
      bool any_fuse = false;
      for (const auto &f : st->sc_host) any_fuse |= f.fuse != 0;
      int Sb = want_stages ? std::max(2, std::min(8, want_stages)) : ((any_fuse || st->bundle_key == 0) && st->V == 4 && st->max_chunk_rows * KT * sizeof(float) > 16384 ? 2 : 3);
      size_t stage_b = (ctx->smem_optin - fixed_b) / Sb / 128 * 128;
      while (Sb > 2 && stage_b < biggest) { Sb--; stage_b = (ctx->smem_optin - fixed_b) / Sb / 128 * 128; }
      if (stage_b >= biggest && (!blocked || (size_t)Sb * stage_b >= tile)) {
        const uint64_t key = ((uint64_t)st->cfg + 1) << 32 | (uint64_t)stage_b;
        if (st->bundle_key != key) {
          size_t off = 0;
          auto need_of = [&](const FeatDev &f) { return (xm + (size_t)f.rows * KT * sizeof(float) + 127) / 128 * 128; };
          for (size_t i = 0; i < st->sc_host.size(); i++) {
            FeatDev &f = st->sc_host[i];
            size_t need = need_of(f);
            if (f.fuse) {  // a fused quad stays inside one bundle; when it cannot, its features are walked one by one
              size_t quad = 0;
              for (size_t j = 0; j < 4; j++) quad += need_of(st->sc_host[i + j]);
              if (quad > stage_b || st->V != 4) f.fuse = 0;
              else need = quad;
            }
            if (off + need > stage_b) { st->sc_host[i - 1].bundle_last = 1; off = 0; }
            const size_t span = f.fuse ? 4 : 1;
            for (size_t j = 0; j < span; j++) {
              FeatDev &g = st->sc_host[i + j];
              g.sx_off = (uint32_t)off;
              g.sc_off = (uint32_t)(off + xm);
              g.bundle_last = 0;
              off += need_of(g);
            }
            i += span - 1;
          }
          if (!st->sc_host.empty()) st->sc_host.back().bundle_last = 1;
          // kernels of earlier sweeps read the list in stream order: the copy is ordered behind them
          CU_TRY(cudaMemcpyAsync(st->d_feats_scalar, st->sc_host.data(), sizeof(FeatDev) * st->sc_host.size(), cudaMemcpyHostToDevice, ctx->stream));
          CU_TRY(cudaStreamSynchronize(ctx->stream));
          st->bundle_key = key;
        }
        const size_t smem_b = (size_t)Sb * stage_b + fixed_b;
#define MSB_BUNDLE_LAUNCH(V_, RW_, NW_)                                                                                   \
        do {                                                                                                              \
          if (blocked) LAUNCH(ctx, (score_bundle_kernel<V_, RW_, NW_, true>), (unsigned)grid, NW_ * 32, smem_b, MSB_BUNDLE_ARGS); \
          else LAUNCH(ctx, (score_bundle_kernel<V_, RW_, NW_, false>), (unsigned)grid, NW_ * 32, smem_b, MSB_BUNDLE_ARGS);        \
        } while (0)
#define MSB_BUNDLE_ARGS st->d_feats_scalar, (int)st->n_scalar, st->d_params, st->region_rows, (uint32_t)stage_b, Sb, st->d_base_score, \
                        scores, st->ld, org, row_lo, row_hi, st->d_hp, st->d_ss, st->d_col2slot, (int)K, (int)ktiles, rowmax
        if (st->cfg == 1) MSB_BUNDLE_LAUNCH(2, 32, 16);
        else if (st->cfg == 4) MSB_BUNDLE_LAUNCH(4, 16, 16);
        else MSB_BUNDLE_LAUNCH(4, 32, 8);
#undef MSB_BUNDLE_LAUNCH
#undef MSB_BUNDLE_ARGS
        goto scalar_done;
      }
    }
    if (st->cfg == 4) return fail(MSB_ERR_UNSUPPORTED, "score shape 4 exists for the bundled general kernel only");
    if (blocked && st->tables_only && persistent) {
      // The persistent form of the sweep's tables-only kernel (score_tables_persistent_kernel): one CTA per SM walks
      // (row tile, k-tile) items, the ring runs through the item boundaries, a seventeenth warp is the producer, the
      // epilogue stores straight from registers.  Measured on C2 against the one-item-per-block grid (1.378 ms): 1.487 ms
      // with thread 0 as the producer and transposition tiles of its own (4 stages instead of 6), 1.498 with the direct
      // stores (6 stages), 1.974 with a producer that polls instead of waiting, 1.394 with the producer warp (96
      // registers) -- no gain: the kernel sits at 0.79 of the shared-memory wavefront roof either way, and what the block
      // boundaries cost the grid form, the hardware scheduler's dynamic balance gives back.  Opt-in, kept under test.
      const size_t stage_p = (chunk_off + st->max_chunk_rows * KT * sizeof(float) + 127) / 128 * 128;
      const size_t tiles_p = 0;   // the epilogue stores straight from registers
      if (ctx->smem_optin >= fixed + tiles_p + 2 * stage_p) {
        const int Sp = (int)std::min<size_t>(8, (ctx->smem_optin - fixed - tiles_p) / stage_p);
        const size_t smem_p = (size_t)Sp * stage_p + tiles_p + fixed;
        const long long n_items = (long long)grid;
        const unsigned grid_p = (unsigned)std::min<long long>(n_items, ctx->sm_count);
#define MSB_PERSIST_LAUNCH(V_, RW_, NW_)                                                                                        \
        LAUNCH(ctx, (score_tables_persistent_kernel<V_, RW_, NW_>), grid_p, (NW_ + 1) * 32, smem_p, st->d_feats_scalar, (int)st->n_scalar, \
               st->d_params, st->region_rows, (uint32_t)stage_p, Sp, st->d_base_score, scores, st->ld, org, row_lo, row_hi,     \
               (int)ktiles, st->tail_g, n_items)
        switch (st->cfg) {
          case 0: MSB_PERSIST_LAUNCH(1, 64, 16); break;
          case 1: MSB_PERSIST_LAUNCH(2, 32, 16); break;
          case 2: MSB_PERSIST_LAUNCH(4, 32, 8); break;
          default: MSB_PERSIST_LAUNCH(1, 32, 8); break;
        }
#undef MSB_PERSIST_LAUNCH
        goto scalar_done;
      }
    }
    if (smem > ctx->smem_optin) return fail(MSB_ERR_UNSUPPORTED, "score kernel shared memory does not fit");
#define MSB_SCORE_ARGS st->d_feats_scalar, (int)st->n_scalar, st->d_params, st->region_rows, (uint32_t)stage, S, st->d_base_score, \
                       scores, st->ld, org, row_lo, row_hi, st->d_hp, st->d_ss, st->d_col2slot, (int)K, (int)ktiles, st->tail_g, rowmax
#define MSB_SCORE_LAUNCH(V_, RW_, NW_)                                                                         \
    do {                                                                                                       \
      if (blocked && st->tables_only) LAUNCH(ctx, (score_kernel<V_, RW_, NW_, true, true>), (unsigned)grid, NW_ * 32, smem, MSB_SCORE_ARGS);        \
      else if (blocked) LAUNCH(ctx, (score_kernel<V_, RW_, NW_, true, false>), (unsigned)grid, NW_ * 32, smem, MSB_SCORE_ARGS);                     \
      else if (st->tables_only) LAUNCH(ctx, (score_kernel<V_, RW_, NW_, false, true>), (unsigned)grid, NW_ * 32, smem, MSB_SCORE_ARGS);             \
      else LAUNCH(ctx, (score_kernel<V_, RW_, NW_, false, false>), (unsigned)grid, NW_ * 32, smem, MSB_SCORE_ARGS);                                 \
    } while (0)
    switch (st->cfg) {
      case 0: MSB_SCORE_LAUNCH(1, 64, 16); break;
      case 1: MSB_SCORE_LAUNCH(2, 32, 16); break;
      case 2: MSB_SCORE_LAUNCH(4, 32, 8); break;
      default: MSB_SCORE_LAUNCH(1, 32, 8); break;
    }
#undef MSB_SCORE_LAUNCH
#undef MSB_SCORE_ARGS
  }
scalar_done:
  row_lo = org;  // the NIW kernels below index the score matrix from the same origin
  // without scalar features the first NIW feature initialises the matrix: the tensor-core kernel writes
  // base[k] + term directly; the CUDA-core kernel accumulates onto a base-filled matrix
  bool need_init = !st->has_scalar;
  for (size_t d = 0; d < st->D; d++) {
    const FeatDev &f = st->feats[d];
    if (f.kind != KIND_NIW) continue;
    bool done = false;
    const bool tc_ok = f.dim == 64 && !getenv("MSB_NO_TENSOR");
    if (need_init && !tc_ok) {
      LAUNCH(ctx, fill_rows_kernel, cdiv(nrows * st->ld, 256), 256, 0, scores, st->ld, st->d_base, nrows);
      need_init = false;
    }
    if (tc_ok && !getenv("MSB_NIW_TF32") && row_hi > row_lo) {  // fp16 operands (msb_niw_tc16.cuh): the default
      const size_t a_bytes = niw_tc16_a_bytes(row_hi - row_lo);   // the rows of this call, converted once per sweep
      if (st->niw_a16_cap < a_bytes) {
        CU_TRY(cudaFree(st->d_niwA16)); st->d_niwA16 = nullptr; st->niw_a16_cap = 0; st->niw_a16_version = 0;
        CU_TRY(cudaMalloc(&st->d_niwA16, a_bytes));
        st->niw_a16_cap = a_bytes;
      }
      const bool a_valid = st->niw_a16_version == st->col_version && st->niw_a16_feat == d && st->niw_a16_lo == row_lo &&
                           st->niw_a16_hi == row_hi && !getenv("MSB_NIW_NO_A_CACHE");
      MSB_TRY(niw_tc16_score(ctx->stream, &ctx->launches, &ctx->prof, (const float *)f.scol, st->d_niwW[d], st->d_niwBias[d], st->d_niwCoef[d],
                             st->d_niwB[d], (unsigned char *)st->d_niwA16, K, scores, st->ld, row_lo, row_hi, ctx->sm_count,
                             need_init ? st->d_base : nullptr, blocked, a_valid, g_last_error));
      st->niw_a16_version = st->col_version; st->niw_a16_feat = d; st->niw_a16_lo = row_lo; st->niw_a16_hi = row_hi;
      done = true;
    } else {
    st->niw_a16_version = 0;   // the tf32 path packs its own operands over the column maxima kept next to the fp16 B operand
    MSB_TRY(niw_tc_score(ctx->stream, &ctx->launches, (const float *)f.scol, f.dim, st->d_niwW[d], st->d_niwBias[d], st->d_niwCoef[d],
                         st->d_niwB[d], K, scores, st->ld, row_lo, row_hi, ctx->sm_count, need_init ? st->d_base : nullptr,
                         blocked, &done, g_last_error));
    }
    if (blocked && !done) return fail(MSB_ERR_STATE, "internal: blocked score layout without the tensor-core NIW path");
    if (done) need_init = false;
    if (!done) {
      if (need_init) {
        LAUNCH(ctx, fill_rows_kernel, cdiv(nrows * st->ld, 256), 256, 0, scores, st->ld, st->d_base, nrows);
        need_init = false;
      }
      const size_t smem = ((size_t)f.dim * f.dim + f.dim) * sizeof(float);
      dim3 grid(cdiv(nrows, 128), (unsigned)K);
      LAUNCH(ctx, niw_score_simt_kernel, grid, 128, smem, (const float *)f.scol, (int)f.dim, st->d_niwW[d], st->d_niwBias[d],
             st->d_niwCoef[d], scores, st->ld, row_lo, row_hi);
    }
  }
  for (size_t d = 0; d < st->D; d++) {  // dm: one more term per (row, group), accumulated like the CUDA-core niw kernel
    const FeatDev &f = st->feats[d];
    if (f.kind != KIND_DM) continue;
    if (blocked) return fail(MSB_ERR_STATE, "internal: blocked score layout with a dm feature");
    if (need_init) {
      LAUNCH(ctx, fill_rows_kernel, cdiv(nrows * st->ld, 256), 256, 0, scores, st->ld, st->d_base, nrows);
      need_init = false;
    }
    MSB_TRY(launch_dm(ctx, f, st->d_hp, st->d_ss, st->d_col2slot, K, scores, st->ld, row_lo, row_hi));
  }
  return MSB_OK;
}

static void mark_dirty(msb_state *st) {
  for (auto &p : st->gid2slot) st->slot_dirty[p.second] = 1;
}
static int refresh_counts(msb_state *st) {  // the device counts changed: the host copy is re-read on demand (host_counts)
  mark_dirty(st);
  st->counts_stale = true;
  return MSB_OK;
}

static int launch_update(msb_state *st, size_t row_lo, size_t row_hi) {  // old = d_assign, new = d_newslot
  msb_ctx *ctx = st->ctx;
  const size_t nrows = row_hi - row_lo;
  if (st->has_scalar) {
    dim3 grid(cdiv(nrows, 256), cdiv(st->D, UPDATE_SLAB));
    LAUNCH(ctx, update_kernel, grid, 256, 0, st->d_feats, (int)st->D, st->d_assign, st->d_newslot, row_lo, row_hi, st->d_delta);
  }
  for (size_t d = 0; d < st->D; d++) {
    const FeatDev &f = st->feats[d];
    if (f.kind != KIND_NIW) continue;
    LAUNCH(ctx, update_niw_kernel, cdiv(nrows, 8), 256, 0, f, st->d_assign, st->d_newslot, row_lo, row_hi, st->d_delta);
  }
  for (size_t d = 0; d < st->D; d++) {
    const FeatDev &f = st->feats[d];
    if (f.kind != KIND_DM) continue;
    LAUNCH(ctx, update_dm_kernel, cdiv(nrows, 8), 256, 0, f, st->d_assign, st->d_newslot, row_lo, row_hi, st->d_delta);
  }
  LAUNCH(ctx, commit_assign_kernel, cdiv(nrows, 256), 256, st->kmax <= 8192 ? st->kmax * sizeof(int) : 0, st->d_assign,
         st->d_newslot, row_lo, row_hi, st->d_delta, (int)st->kmax, st->d_counter);
  return MSB_OK;
}

static int launch_apply(msb_state *st) {
  LAUNCH(st->ctx, apply_delta_kernel, cdiv(st->SS, 256), 256, 0, st->d_ss, st->d_delta, st->SS);
  if (st->has_dd) {
    dim3 grid(cdiv(st->kmax, 8), (unsigned)st->D);
    LAUNCH(st->ctx, dd_count_sum_kernel, grid, 256, 0, st->d_feats, (int)st->D, (int)st->kmax, st->d_ss);
  }
  return MSB_OK;
}
static int apply_deltas(msb_state *st) {
  MSB_TRY(launch_apply(st));
  return refresh_counts(st);
}

extern "C" MSB_API int msb_state_delta_buffer(msb_state *st, double **dev_ptr, size_t *count) {
  REQUIRE(st && dev_ptr && count, "NULL argument");
  *dev_ptr = st->d_delta; *count = st->SS;
  return MSB_OK;
}
// Count-valued states only (every feature bb or dd: each delta is a number of rows, |delta| <= N < 2^31): the pending
// deltas as int32, exact, half the bytes to all-reduce.  *dev_ptr == NULL (and MSB_OK) for any other state (bnb / gp
// sums of values can exceed int32, nich / niw moments are real).
extern "C" MSB_API int msb_state_delta_buffer_i32(msb_state *st, int32_t **dev_ptr, size_t *count) {
  REQUIRE(st && dev_ptr && count, "NULL argument");
  *dev_ptr = nullptr; *count = st->SS;
  for (const auto &m : st->models)
    if (m.family != MSB_FAMILY_BB && m.family != MSB_FAMILY_DD) return MSB_OK;  // (bbnc's p is not a count)
  if (st->n >= (1ull << 31) || getenv("MSB_NO_I32_DELTAS")) return MSB_OK;
  CU_TRY(cudaSetDevice(st->ctx->device));
  if (!st->d_delta_i32) CU_TRY(cudaMalloc(&st->d_delta_i32, sizeof(int32_t) * st->SS));
  LAUNCH(st->ctx, delta_to_i32_kernel, cdiv(st->SS, 256), 256, 0, st->d_delta, st->SS, st->d_delta_i32);
  *dev_ptr = st->d_delta_i32;
  return MSB_OK;
}
// after the all-reduce of that buffer: back into the fp64 delta buffer, then msb_state_apply_deltas as usual
extern "C" MSB_API int msb_state_delta_from_i32(msb_state *st) {
  REQUIRE(st && st->d_delta_i32, "msb_state_delta_buffer_i32 was not called");
  CU_TRY(cudaSetDevice(st->ctx->device));
  LAUNCH(st->ctx, delta_from_i32_kernel, cdiv(st->SS, 256), 256, 0, st->d_delta_i32, st->SS, st->d_delta);
  return MSB_OK;
}
extern "C" MSB_API int msb_state_suffstat_buffer(msb_state *st, double **dev_ptr, size_t *count) {
  REQUIRE(st && dev_ptr && count, "NULL argument");
  *dev_ptr = st->d_ss; *count = st->SS;
  return MSB_OK;
}
extern "C" MSB_API int msb_state_apply_deltas(msb_state *st) {
  REQUIRE(st, "NULL argument");
  CU_TRY(cudaSetDevice(st->ctx->device));
  return apply_deltas(st);
}

// ---- assignments -------------------------------------------------------------
extern "C" MSB_API int msb_state_assignments(msb_state *st, int64_t *out, size_t n) {
  REQUIRE(st && out, "NULL argument");
  REQUIRE(st->dv, "no dataview bound");
  REQUIRE(n == st->n, "wrong length");
  if (!n) return MSB_OK;
  msb_ctx *ctx = st->ctx;
  CU_TRY(cudaSetDevice(ctx->device));
  MSB_TRY(ensure(&st->d_assign64, &st->assign64_cap, n));
  if (st->slot2gid_dirty) {
    CU_TRY(cudaMemcpyAsync(st->d_slot2gid, st->slot2gid.data(), sizeof(int64_t) * st->kmax, cudaMemcpyHostToDevice, ctx->stream));
    st->slot2gid_dirty = false;  // pageable source: the copy has been staged on return
  }
  LAUNCH(ctx, map_i32_to_i64_kernel, cdiv(n, 256), 256, 0, st->d_assign, st->d_slot2gid, n, st->d_assign64);
  CU_TRY(cudaMemcpyAsync(out, st->d_assign64, sizeof(int64_t) * n, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(cudaStreamSynchronize(ctx->stream));
  return MSB_OK;
}

// The same, without waiting: the gid translation runs on the compute stream, the device -> host copy on the
// copy stream (so it overlaps whatever the compute stream does next, e.g. the next sweep).  `out` should be
// pinned and must not be read before msb_state_assignments_wait returns.  One copy in flight per state.
extern "C" MSB_API int msb_state_assignments_async(msb_state *st, int64_t *out, size_t n) {
  REQUIRE(st && out, "NULL argument");
  REQUIRE(st->dv, "no dataview bound");
  REQUIRE(n == st->n, "wrong length");
  if (!n) return MSB_OK;
  msb_ctx *ctx = st->ctx;
  CU_TRY(cudaSetDevice(ctx->device));
  if (!st->ev_mapped) {
    CU_TRY(cudaEventCreateWithFlags(&st->ev_mapped, cudaEventDisableTiming));
    CU_TRY(cudaEventCreateWithFlags(&st->ev_assign_copied, cudaEventDisableTiming));
  }
  if (st->assign_copy_pending) {  // d_assign64 is still being read by the previous copy
    CU_TRY(cudaStreamWaitEvent(ctx->stream, st->ev_assign_copied, 0));
  }
  MSB_TRY(ensure(&st->d_assign64, &st->assign64_cap, n));
  if (st->slot2gid_dirty) {
    CU_TRY(cudaMemcpyAsync(st->d_slot2gid, st->slot2gid.data(), sizeof(int64_t) * st->kmax, cudaMemcpyHostToDevice, ctx->stream));
    st->slot2gid_dirty = false;
  }
  LAUNCH(ctx, map_i32_to_i64_kernel, cdiv(n, 256), 256, 0, st->d_assign, st->d_slot2gid, n, st->d_assign64);
  CU_TRY(cudaEventRecord(st->ev_mapped, ctx->stream));
  CU_TRY(cudaStreamWaitEvent(ctx->d2h_stream, st->ev_mapped, 0));
  CU_TRY(cudaMemcpyAsync(out, st->d_assign64, sizeof(int64_t) * n, cudaMemcpyDeviceToHost, ctx->d2h_stream));
  CU_TRY(cudaEventRecord(st->ev_assign_copied, ctx->d2h_stream));
  st->assign_copy_pending = true;
  return MSB_OK;
}
extern "C" MSB_API int msb_state_assignments_wait(msb_state *st) {
  REQUIRE(st, "NULL argument");
  if (!st->assign_copy_pending) return MSB_OK;
  CU_TRY(cudaSetDevice(st->ctx->device));
  CU_TRY(cudaEventSynchronize(st->ev_assign_copied));
  st->assign_copy_pending = false;
  return MSB_OK;
}

static int read_assign(msb_state *st, size_t eid, int32_t *slot) {
  CU_TRY(cudaMemcpyAsync(slot, st->d_assign + eid, sizeof(int32_t), cudaMemcpyDeviceToHost, st->ctx->stream));
  CU_TRY(cudaStreamSynchronize(st->ctx->stream));
  return MSB_OK;
}

static int add_values_impl(msb_state *st, const int64_t *gids, size_t n, bool defer) {
  REQUIRE(st && gids, "NULL argument");
  REQUIRE(st->dv, "no dataview bound");
  REQUIRE(n == st->n, "wrong length");
  if (!n) return MSB_OK;
  msb_ctx *ctx = st->ctx;
  CU_TRY(cudaSetDevice(ctx->device));
  std::vector<int32_t> cur, req(n);
  if (st->all_unassigned) cur.assign(n, -1);
  else {
    cur.resize(n);
    CU_TRY(cudaMemcpyAsync(cur.data(), st->d_assign, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
  }
  std::vector<int> g2s;  // dense gid -> slot table: one lookup per entity instead of a map search
  if (!st->gid2slot.empty()) {
    g2s.assign(st->gid2slot.rbegin()->first + 1, -1);
    for (auto &p : st->gid2slot) g2s[p.first] = p.second;
  }
  for (size_t i = 0; i < n; i++) {
    if (gids[i] < 0) { req[i] = cur[i]; continue; }
    if (cur[i] >= 0) return fail(MSB_ERR_STATE, "entity already assigned");  // group_manager.hpp:221
    if ((size_t)gids[i] >= g2s.size() || g2s[(size_t)gids[i]] < 0) return fail(MSB_ERR_INVALID, "invalid gid");
    req[i] = g2s[(size_t)gids[i]];
  }
  st->all_unassigned = false;
  MSB_TRY(ensure_rows(st, n));
  MSB_TRY(sync_small(st));
  CU_TRY(cudaMemcpyAsync(st->d_newslot, req.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(cudaMemsetAsync(st->d_counter, 0, sizeof(unsigned long long), ctx->stream));
  MSB_TRY(launch_update(st, 0, n));
  if (defer) return refresh_counts(st);  // the caller all-reduces the delta buffer, then msb_state_apply_deltas
  return apply_deltas(st);
}

extern "C" MSB_API int msb_state_add_values(msb_state *st, const int64_t *gids, size_t n) { return add_values_impl(st, gids, n, false); }
// multi-GPU replica initialisation: the local rows' contributions stay in the delta buffer; all-reduce it
// (msb_state_delta_buffer), then msb_state_apply_deltas -- the same path as a sweep, so per-group parameters that are
// not sums over rows (bbnc's p) are never touched
extern "C" MSB_API int msb_state_add_values_deferred(msb_state *st, const int64_t *gids, size_t n) { return add_values_impl(st, gids, n, true); }
extern "C" MSB_API int msb_state_add_value(msb_state *st, size_t gid, size_t eid) {
  REQUIRE(st, "NULL argument");
  REQUIRE(st->dv, "no dataview bound");
  REQUIRE(eid < st->n, "invalid eid");
  int slot; int32_t cur;
  MSB_TRY(slot_of(st, gid, &slot));
  CU_TRY(cudaSetDevice(st->ctx->device));
  MSB_TRY(read_assign(st, eid, &cur));
  if (cur != -1) return fail(MSB_ERR_STATE, "entity already assigned");
  st->all_unassigned = false;
  MSB_TRY(ensure_rows(st, 1));
  MSB_TRY(sync_small(st));
  const int32_t s32 = slot;
  CU_TRY(cudaMemcpyAsync(st->d_newslot, &s32, sizeof(int32_t), cudaMemcpyHostToDevice, st->ctx->stream));
  MSB_TRY(launch_update(st, eid, eid + 1));
  return apply_deltas(st);
}

extern "C" MSB_API int msb_state_remove_value(msb_state *st, size_t eid, size_t *gid) {
  REQUIRE(st, "NULL argument");
  REQUIRE(st->dv, "no dataview bound");
  REQUIRE(eid < st->n, "invalid eid");
  int32_t cur;
  CU_TRY(cudaSetDevice(st->ctx->device));
  MSB_TRY(read_assign(st, eid, &cur));
  if (cur == -1) return fail(MSB_ERR_STATE, "entity not assigned");  // group_manager.hpp:238
  if (gid) *gid = (size_t)st->slot2gid[cur];
  MSB_TRY(ensure_rows(st, 1));
  MSB_TRY(sync_small(st));
  const int32_t s32 = -1;
  CU_TRY(cudaMemcpyAsync(st->d_newslot, &s32, sizeof(int32_t), cudaMemcpyHostToDevice, st->ctx->stream));
  MSB_TRY(launch_update(st, eid, eid + 1));
  return apply_deltas(st);
}

// ---- scoring -------------------------------------------------------------------
static int ensure_scores(msb_state *st, size_t nrows) {  // rows padded to the 32-row blocks of the blocked layout
  return ensure(&st->d_scores, &st->scores_cap, (nrows + 31) / 32 * 32 * st->ld + 64);
}

extern "C" MSB_API int msb_state_score_value(msb_state *st, size_t eid, size_t *gids, float *scores, size_t cap, size_t *n) {
  REQUIRE(st && n, "NULL argument");
  REQUIRE(st->dv, "no dataview bound");
  REQUIRE(eid < st->n, "invalid eid");
  msb_ctx *ctx = st->ctx;
  CU_TRY(cudaSetDevice(ctx->device));
  MSB_TRY(prepare_columns(st));
  const size_t K = st->h_col2slot.size();
  *n = K;
  if (!scores && !gids) return MSB_OK;
  REQUIRE(cap >= K, "buffer too small");
  size_t skip = 0;
  if (!st->has_niw && !st->has_dm) {
    MSB_TRY(ensure_scores(st, 1));
    MSB_TRY(sync_small(st));
    LAUNCH(ctx, score_direct_kernel<float>, 1, 128, 0, st->d_feats, (int)st->D, st->d_hp, st->d_ss, st->d_col2slot, (int)K,
           st->d_base, st->d_scores, st->ld, eid, eid + 1);
  } else {
    skip = eid - row_origin(eid);
    MSB_TRY(ensure_scores(st, skip + 1));
    MSB_TRY(build_params(st));
    MSB_TRY(launch_score(st, eid, eid + 1, st->d_scores));
  }
  st->last_rows = 1; st->last_cols = K; st->last_blocked = false; st->last_skip = skip;
  if (scores) CU_TRY(cudaMemcpyAsync(scores, st->d_scores + skip * st->ld, sizeof(float) * K, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(cudaStreamSynchronize(ctx->stream));
  if (gids) for (size_t c = 0; c < K; c++) gids[c] = st->h_colgid[c];
  return MSB_OK;
}

extern "C" MSB_API int msb_state_score_rows(msb_state *st, size_t row_lo, size_t row_hi, float *scores, size_t ld,
                                    int on_device, size_t *gids, size_t cap, size_t *ncols) {
  REQUIRE(st && ncols, "NULL argument");
  REQUIRE(st->dv, "no dataview bound");
  REQUIRE(row_lo <= row_hi && row_hi <= st->n, "bad row range");
  msb_ctx *ctx = st->ctx;
  CU_TRY(cudaSetDevice(ctx->device));
  MSB_TRY(prepare_columns(st));
  const size_t K = st->h_col2slot.size();
  *ncols = K;
  if (gids) { REQUIRE(cap >= K, "buffer too small"); for (size_t c = 0; c < K; c++) gids[c] = st->h_colgid[c]; }
  const size_t nrows = row_hi - row_lo;
  if (!nrows) return MSB_OK;
  const bool direct = getenv("MSB_FORCE_DIRECT") && !st->has_niw && !st->has_dm;
  const size_t skip = direct ? 0 : row_lo - row_origin(row_lo);
  // a device destination with the internal leading dimension is written in place
  float *dst = (on_device && scores && ld == st->ld && skip == 0) ? scores : nullptr;
  if (!dst) { MSB_TRY(ensure_scores(st, nrows + skip)); dst = st->d_scores; }
  if (direct) {
    MSB_TRY(sync_small(st));
    LAUNCH(ctx, score_direct_kernel<float>, (unsigned)nrows, 128, 0, st->d_feats, (int)st->D, st->d_hp, st->d_ss, st->d_col2slot,
           (int)K, st->d_base, dst, st->ld, row_lo, row_hi);
  } else {
    MSB_TRY(build_params(st));
    MSB_TRY(launch_score(st, row_lo, row_hi, dst));
  }
  st->last_rows = nrows; st->last_cols = K; st->last_blocked = false; st->last_skip = dst == st->d_scores ? skip : 0;
  if (scores && dst != scores) {
    REQUIRE(ld >= K, "ld smaller than the number of groups");
    CU_TRY(cudaMemcpy2DAsync(scores, sizeof(float) * ld, dst + skip * st->ld, sizeof(float) * st->ld, sizeof(float) * K, nrows,
                             on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, ctx->stream));
  }
  if (!on_device) CU_TRY(cudaStreamSynchronize(ctx->stream));
  return MSB_OK;
}

// fp64 scores: the closed forms evaluated in double straight from the resident suffstats (no tables, no fp32
// anywhere but the stored values themselves).  The verification path for the 1e-12 tolerance; host output.
extern "C" MSB_API int msb_state_score_rows_f64(msb_state *st, size_t row_lo, size_t row_hi, double *scores, size_t ld,
                                        size_t *gids, size_t cap, size_t *ncols) {
  REQUIRE(st && ncols, "NULL argument");
  REQUIRE(st->dv, "no dataview bound");
  REQUIRE(row_lo <= row_hi && row_hi <= st->n, "bad row range");
  msb_ctx *ctx = st->ctx;
  CU_TRY(cudaSetDevice(ctx->device));
  MSB_TRY(prepare_columns(st));
  MSB_TRY(sync_small(st));
  const size_t K = st->h_col2slot.size();
  *ncols = K;
  if (gids) { REQUIRE(cap >= K, "buffer too small"); for (size_t c = 0; c < K; c++) gids[c] = st->h_colgid[c]; }
  const size_t nrows = row_hi - row_lo;
  if (!nrows || !scores) return MSB_OK;
  REQUIRE(ld >= K, "ld smaller than the number of groups");
  Scratch<double> d_out;
  CU_TRY(d_out.alloc(nrows * K));
  LAUNCH(ctx, score_direct_kernel<double>, (unsigned)nrows, 128, 0, st->d_feats, (int)st->D, st->d_hp, st->d_ss, st->d_col2slot,
         (int)K, st->d_base, d_out, K, row_lo, row_hi);
  for (size_t d = 0; d < st->D; d++) {
    const FeatDev &f = st->feats[d];
    if (f.kind != KIND_NIW) continue;
    const size_t smem = ((size_t)f.dim * f.dim + f.dim) * sizeof(double);
    LAUNCH(ctx, niw_score_f64_kernel, (unsigned)K, 128, smem, f, st->d_hp, st->d_ss, st->d_col2slot, d_out, K, row_lo, row_hi);
  }
  for (size_t d = 0; d < st->D; d++) {
    const FeatDev &f = st->feats[d];
    if (f.kind != KIND_DM) continue;
    MSB_TRY(launch_dm(ctx, f, st->d_hp, st->d_ss, st->d_col2slot, K, d_out.p, K, row_lo, row_hi));
  }
  CU_TRY(cudaMemcpy2DAsync(scores, sizeof(double) * ld, d_out, sizeof(double) * K, sizeof(double) * K, nrows,
                           cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(cudaStreamSynchronize(ctx->stream));
  return MSB_OK;
}

extern "C" MSB_API int msb_state_last_scores(msb_state *st, float **dev_ptr, size_t *ld, size_t *nrows, size_t *ncols) {
  REQUIRE(st, "NULL argument");
  if (dev_ptr) *dev_ptr = st->d_scores + (st->last_blocked ? 0 : st->last_skip * st->ld);
  if (ld) *ld = st->ld;
  if (nrows) *nrows = st->last_rows;
  if (ncols) *ncols = st->last_cols;
  return MSB_OK;
}
extern "C" MSB_API int msb_state_read_last_scores(msb_state *st, float *out, size_t ld_out) {
  REQUIRE(st && out, "NULL argument");
  REQUIRE(ld_out >= st->last_cols, "ld smaller than the number of groups");
  if (!st->last_rows || !st->last_cols) return MSB_OK;
  CU_TRY(cudaSetDevice(st->ctx->device));
  if (st->last_blocked) {
    Scratch<float> tmp;
    CU_TRY(tmp.alloc(st->last_rows * st->last_cols));
    LAUNCH(st->ctx, unblock_kernel, cdiv(st->last_rows * st->last_cols, 256), 256, 0, st->d_scores, st->ld, st->last_skip,
           st->last_rows, (int)st->last_cols, tmp);
    CU_TRY(cudaMemcpy2DAsync(out, sizeof(float) * ld_out, tmp, sizeof(float) * st->last_cols, sizeof(float) * st->last_cols,
                             st->last_rows, cudaMemcpyDeviceToHost, st->ctx->stream));
    CU_TRY(cudaStreamSynchronize(st->ctx->stream));
    return MSB_OK;
  }
  CU_TRY(cudaMemcpy2DAsync(out, sizeof(float) * ld_out, st->d_scores + st->last_skip * st->ld, sizeof(float) * st->ld,
                           sizeof(float) * st->last_cols, st->last_rows, cudaMemcpyDeviceToHost, st->ctx->stream));
  CU_TRY(cudaStreamSynchronize(st->ctx->stream));
  return MSB_OK;
}
// back = 0: the last sweep, 1: the one before it, ... (up to TIMING_RING - 1 sweeps back)
extern "C" MSB_API int msb_state_timings(msb_state *st, size_t back, float *ms, size_t count) {
  REQUIRE(st && ms, "NULL argument");
  for (size_t i = 0; i < count; i++) ms[i] = 0.f;
  REQUIRE(back < msb_state::TIMING_RING && back < st->sweep_seq, "no such sweep in the timing ring");
  const size_t slot = (st->sweep_seq - 1 - back) % msb_state::TIMING_RING;
  std::vector<PhaseEvents> &ev = st->events[slot];
  CU_TRY(cudaSetDevice(st->ctx->device));
  CU_TRY(cudaEventSynchronize(ev[0].e[3]));
  float out[5] = {0, 0, 0, 0, 0}, t = 0.f;
  CU_TRY(cudaEventElapsedTime(&t, ev[0].e[0], ev[0].e[1])); out[0] = t;
  for (size_t c = 0; c < st->ring_nchunks[slot]; c++)
    for (int p = 0; p < 3; p++) { CU_TRY(cudaEventElapsedTime(&t, ev[c + 1].e[p], ev[c + 1].e[p + 1])); out[1 + p] += t; }
  CU_TRY(cudaEventElapsedTime(&t, ev[0].e[2], ev[0].e[3])); out[4] = t;
  for (size_t i = 0; i < count && i < 5; i++) ms[i] = out[i];
  return MSB_OK;
}
extern "C" MSB_API int msb_state_last_timings(msb_state *st, float *ms, size_t count) {
  REQUIRE(st && ms, "NULL argument");
  for (size_t i = 0; i < count; i++) ms[i] = 0.f;
  if (!st->sweep_seq) return MSB_OK;
  return msb_state_timings(st, 0, ms, count);
}

// ---- marginal likelihoods (entity_state.hpp:74-86, group_manager.hpp:250-272) -------------------------------
// out[c * D + d] = group::score_data of (group column c, feature d), columns in ascending gid order
static int score_data_matrix(msb_state *st, std::vector<double> &h) {
  msb_ctx *ctx = st->ctx;
  CU_TRY(cudaSetDevice(ctx->device));
  MSB_TRY(prepare_columns(st));
  MSB_TRY(sync_small(st));
  const size_t K = st->h_col2slot.size(), D = st->D;
  Scratch<double> d_out;
  CU_TRY(d_out.alloc(K * D));
  LAUNCH(ctx, score_data_kernel, cdiv(K * D, 128), 128, 0, st->d_feats, (int)D, st->d_hp, st->d_ss, st->d_col2slot, (int)K, d_out);
  for (size_t d = 0; d < D; d++) {
    const FeatDev &f = st->feats[d];
    if (f.kind != KIND_NIW) continue;
    const size_t smem = ((size_t)f.dim * f.dim + f.dim) * sizeof(double);
    LAUNCH(ctx, niw_score_data_kernel, (unsigned)K, 128, smem, f, (int)d, (int)D, st->d_hp, st->d_ss, st->d_col2slot, d_out);
  }
  h.resize(K * D);
  CU_TRY(cudaMemcpyAsync(h.data(), d_out, sizeof(double) * K * D, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(cudaStreamSynchronize(ctx->stream));
  return MSB_OK;
}

extern "C" MSB_API int msb_state_score_likelihood(msb_state *st, size_t feature, size_t gid, float *out) {
  REQUIRE(st && out, "NULL argument");
  REQUIRE(feature < st->D, "bad feature index");
  int slot;
  MSB_TRY(slot_of(st, gid, &slot));
  std::vector<double> h;
  MSB_TRY(score_data_matrix(st, h));
  for (size_t c = 0; c < st->h_col2slot.size(); c++)
    if (st->h_col2slot[c] == slot) { *out = (float)h[c * st->D + feature]; return MSB_OK; }
  return fail(MSB_ERR_INVALID, "invalid gid");
}

// per_feature[d] = sum over groups of score_data (entity_state.hpp:78-86), total = sum over features
extern "C" MSB_API int msb_state_score_likelihood_all(msb_state *st, float *per_feature, size_t nfeatures, float *total) {
  REQUIRE(st, "NULL argument");
  REQUIRE(!per_feature || nfeatures == st->D, "wrong length");
  std::vector<double> h;
  MSB_TRY(score_data_matrix(st, h));
  double tot = 0.0;
  for (size_t d = 0; d < st->D; d++) {
    float s = 0.f;  // the reference accumulates the per-group floats in a float (entity_state.hpp:81-84)
    for (size_t c = 0; c < st->h_col2slot.size(); c++) s += (float)h[c * st->D + d];
    if (per_feature) per_feature[d] = s;
    tot += s;
  }
  if (total) *total = (float)tot;
  return MSB_OK;
}

extern "C" MSB_API int msb_state_score_assignment(msb_state *st, float *out) {
  REQUIRE(st && out, "NULL argument");
  REQUIRE(st->dv && st->n > 0, "no entities");
  msb_ctx *ctx = st->ctx;
  CU_TRY(cudaSetDevice(ctx->device));
  MSB_TRY(prepare_columns(st));
  Scratch<double> d_out;
  CU_TRY(d_out.alloc(2));
  LAUNCH(ctx, score_assignment_kernel, 1, 256, 0, st->d_ss, st->d_col2slot, (int)st->h_col2slot.size(), st->d_assign, st->alpha, d_out);
  double h[2] = {0, 0};
  CU_TRY(cudaMemcpyAsync(h, d_out, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(cudaStreamSynchronize(ctx->stream));
  if ((size_t)h[1] != st->n) return fail(MSB_ERR_STATE, "not assigned");  // group_manager.hpp:255,260
  *out = (float)h[0];
  return MSB_OK;
}

// ---- sampler ---------------------------------------------------------------------
// 32-row tile staged in shared memory (sample_tile_kernel): scores read from HBM exactly once (bulk copy of the
// blocked layout, or coalesced transposing loads of a row-major one)
static bool tile_sampler_fits(size_t K) { return K * 33 * 4 <= 48 * 1024 && !getenv("MSB_NO_TILE_SAMPLER"); }

static int launch_tile_sampler(msb_ctx *ctx, bool blocked, const float *scores, size_t ld, size_t skip, int K, size_t nrows,
                               const float *d_u, uint64_t seed, uint64_t sweep, uint64_t row_id0, const int32_t *col2slot,
                               int32_t *out_col, int32_t *out_slot, const int *rowmax) {
  const size_t nblk = (skip + nrows + 31) / 32 - skip / 32;
  // The kernel is bound by instruction issue and latency, so what counts is warps per SM, and a warp's tile is what
  // limits them: blocks of four warps waste the remainder (K = 256: 32 KB per warp, one block of four per SM where
  // seven warps fit), blocks of one warp do not: C4 sample 0.566 -> 0.517 ms.  Four-warp blocks stay where they lose
  // little -- at equal occupancy they are the faster form (C2: 8 warps in two blocks 0.416 ms, 9 one-warp blocks 0.501).
  auto warps_per_sm = [&](int sw) {
    return (size_t)sw * std::min<size_t>(32 / sw, ctx->smem_optin / sample_tile_smem(sw, K, !blocked));
  };
  const bool one_warp = 2 * warps_per_sm(1) >= 3 * warps_per_sm(4) && !getenv("MSB_SAMPLER_FOUR_WARPS");
#define MSB_TILE_SAMPLER(SW)                                                                                                      \
  do {                                                                                                                        \
    const size_t smem = sample_tile_smem(SW, K, !blocked);                                                                    \
    const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(32 / SW, ctx->smem_optin / smem));                           \
    const unsigned grid = (unsigned)std::min<size_t>((nblk + SW - 1) / SW, (size_t)ctx->sm_count * per_sm);                   \
    if (blocked)                                                                                                              \
      LAUNCH(ctx, (sample_tile_kernel<SW, false>), grid, SW * 32, smem, scores, ld, skip, K, nrows, d_u, seed, sweep, row_id0,  \
             col2slot, out_col, out_slot, rowmax);                                                                            \
    else                                                                                                                      \
      LAUNCH(ctx, (sample_tile_kernel<SW, true>), grid, SW * 32, smem, scores, ld, skip, K, nrows, d_u, seed, sweep, row_id0,   \
             col2slot, out_col, out_slot, (const int *)nullptr);                                                              \
  } while (0)
  if (one_warp) MSB_TILE_SAMPLER(1);
  else MSB_TILE_SAMPLER(4);
#undef MSB_TILE_SAMPLER
  return MSB_OK;
}

extern "C" MSB_API int msb_sample_discrete_log(msb_ctx *ctx, const float *scores, size_t nrows, size_t k, size_t ld,
                                       const float *uniforms, int32_t *out) {
  REQUIRE(ctx && scores && uniforms && out, "NULL argument");
  REQUIRE(k > 0 && ld >= k && k < (1u << 30), "bad shape");
  if (!nrows) return MSB_OK;
  CU_TRY(cudaSetDevice(ctx->device));
  Scratch<float> d_s, d_u;
  Scratch<int32_t> d_o;
  CU_TRY(d_s.alloc(nrows * ld));
  CU_TRY(d_u.alloc(nrows));
  CU_TRY(d_o.alloc(nrows));
  CU_TRY(cudaMemcpyAsync(d_s, scores, sizeof(float) * nrows * ld, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(cudaMemcpyAsync(d_u, uniforms, sizeof(float) * nrows, cudaMemcpyHostToDevice, ctx->stream));
  if (tile_sampler_fits(k))
    MSB_TRY(launch_tile_sampler(ctx, false, d_s, ld, 0, (int)k, nrows, d_u, 0ull, 0ull, 0ull, nullptr, d_o, nullptr, nullptr));
  else
    LAUNCH(ctx, sample_kernel, cdiv(nrows, 128), 128, 0, (const float *)d_s, ld, (int)k, nrows, (const float *)d_u, 0ull, 0ull, 0ull, (const int32_t *)nullptr, (int32_t *)d_o, (int32_t *)nullptr);
  CU_TRY(cudaMemcpyAsync(out, d_o, sizeof(int32_t) * nrows, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(cudaStreamSynchronize(ctx->stream));
  return MSB_OK;
}

extern "C" MSB_API int msb_philox_uniforms(msb_ctx *ctx, uint64_t seed, uint64_t sweep, uint64_t row_lo, size_t n, float *out) {
  REQUIRE(ctx && out, "NULL argument");
  if (!n) return MSB_OK;
  CU_TRY(cudaSetDevice(ctx->device));
  Scratch<float> d_u;
  CU_TRY(d_u.alloc(n));
  LAUNCH(ctx, philox_fill_kernel, cdiv(n, 256), 256, 0, seed, sweep, row_lo, n, (float *)d_u);
  CU_TRY(cudaMemcpyAsync(out, d_u, sizeof(float) * n, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(cudaStreamSynchronize(ctx->stream));
  return MSB_OK;
}

extern "C" MSB_API int msb_selftest_expf(msb_ctx *ctx, const float *x, size_t n, float *y) {
  REQUIRE(ctx && x && y, "NULL argument");
  if (!n) return MSB_OK;
  CU_TRY(cudaSetDevice(ctx->device));
  Scratch<float> d;
  CU_TRY(d.alloc(2 * n));
  CU_TRY(cudaMemcpyAsync(d, x, sizeof(float) * n, cudaMemcpyHostToDevice, ctx->stream));
  LAUNCH(ctx, selftest_expf_kernel, cdiv(n, 256), 256, 0, (const float *)d, n, d.p + n);
  CU_TRY(cudaMemcpyAsync(y, d.p + n, sizeof(float) * n, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(cudaStreamSynchronize(ctx->stream));
  return MSB_OK;
}

extern "C" MSB_API int msb_selftest_expf2(msb_ctx *ctx, uint64_t *mismatches) {
  REQUIRE(ctx && mismatches, "NULL argument");
  CU_TRY(cudaSetDevice(ctx->device));
  Scratch<unsigned long long> d;
  CU_TRY(d.alloc(1));
  CU_TRY(cudaMemsetAsync(d, 0, sizeof(unsigned long long), ctx->stream));
  LAUNCH(ctx, selftest_expf2_kernel, cdiv((size_t)EXPF2_LAST_BITS / 2 + 1, 256), 256, 0, (unsigned long long *)d);
  unsigned long long h = 0;
  CU_TRY(cudaMemcpyAsync(&h, d, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(cudaStreamSynchronize(ctx->stream));
  *mismatches = h;
  return MSB_OK;
}

extern "C" MSB_API int msb_selftest_skip_rule(msb_ctx *ctx, const uint8_t *e, const float *acc, const float *d, size_t n,
                                             uint8_t *out) {
  REQUIRE(ctx && e && acc && d && out, "NULL argument");
  if (!n) return MSB_OK;
  CU_TRY(cudaSetDevice(ctx->device));
  Scratch<float> df;
  Scratch<uint8_t> db;
  CU_TRY(df.alloc(2 * n));
  CU_TRY(db.alloc(2 * n));
  CU_TRY(cudaMemcpyAsync(df, acc, sizeof(float) * n, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(cudaMemcpyAsync(df.p + n, d, sizeof(float) * n, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(cudaMemcpyAsync(db, e, n, cudaMemcpyHostToDevice, ctx->stream));
  LAUNCH(ctx, selftest_skip_rule_kernel, cdiv(n, 256), 256, 0, (const uint8_t *)db, (const float *)df, (const float *)(df.p + n), n,
         db.p + n);
  CU_TRY(cudaMemcpyAsync(out, db.p + n, n, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(cudaStreamSynchronize(ctx->stream));
  return MSB_OK;
}

extern "C" MSB_API int msb_selftest_division(msb_ctx *ctx, uint64_t seed, size_t n, uint64_t *mismatches) {
  REQUIRE(ctx && mismatches, "NULL argument");
  CU_TRY(cudaSetDevice(ctx->device));
  Scratch<unsigned long long> d;
  CU_TRY(d.alloc(1));
  CU_TRY(cudaMemsetAsync(d, 0, sizeof(unsigned long long), ctx->stream));
  if (n) LAUNCH(ctx, selftest_division_kernel, cdiv(n, 256), 256, 0, seed, n, (unsigned long long *)d);
  unsigned long long h = 0;
  CU_TRY(cudaMemcpyAsync(&h, d, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(cudaStreamSynchronize(ctx->stream));
  *mismatches = h;
  return MSB_OK;
}

// ---- NCCL: the one exchange step of the path (SURVEY.md section 8e) -------------------------------------------------
// Rows are sharded, every rank holds a full replica of the suffstats, and one all-reduce(sum) of the flat delta buffer
// per sweep keeps the replicas identical.  The NCCL library is resolved at run time: a host process that already has
// one loaded (PyTorch ships its own libnccl.so.2) must keep using that copy, so the library is looked up among the
// loaded objects first and dlopen'ed only when there is none.
struct NcclApi {
  bool ok = false;
  std::string err;
  const char *(*GetErrorString)(ncclResult_t) = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*CommCount)(const ncclComm_t, int *) = nullptr;
  ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GetVersion)(int *) = nullptr;
};
static NcclApi &nccl_api() {
  static NcclApi api;
  static bool tried = false;
  if (tried) return api;
  tried = true;
  void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) { api.err = std::string("NCCL is not available: ") + dlerror(); return api; }
#define MSB_NCCL_SYM(field, name)                                         \
  api.field = reinterpret_cast<decltype(api.field)>(dlsym(h, name));      \
  if (!api.field) { api.err = std::string("NCCL symbol missing: ") + name; return api; }
  MSB_NCCL_SYM(GetErrorString, "ncclGetErrorString")
  MSB_NCCL_SYM(GetUniqueId, "ncclGetUniqueId")
  MSB_NCCL_SYM(CommInitRank, "ncclCommInitRank")
  MSB_NCCL_SYM(CommDestroy, "ncclCommDestroy")
  MSB_NCCL_SYM(CommCount, "ncclCommCount")
  MSB_NCCL_SYM(AllReduce, "ncclAllReduce")
  MSB_NCCL_SYM(GetVersion, "ncclGetVersion")
#undef MSB_NCCL_SYM
  api.ok = true;
  return api;
}
#define NCCL_TRY(expr)                                                                                        \
  do {                                                                                                        \
    ncclResult_t _r = (expr);                                                                                 \
    if (_r != ncclSuccess) return fail(MSB_ERR_CUDA, std::string(#expr) + ": " + nccl_api().GetErrorString(_r)); \
  } while (0)

extern "C" MSB_API int msb_nccl_version(int *version) {
  REQUIRE(version, "NULL argument");
  NcclApi &n = nccl_api();
  if (!n.ok) return fail(MSB_ERR_UNSUPPORTED, n.err);
  NCCL_TRY(n.GetVersion(version));
  return MSB_OK;
}
extern "C" MSB_API int msb_nccl_unique_id(void *id128) {
  REQUIRE(id128, "NULL argument");
  NcclApi &n = nccl_api();
  if (!n.ok) return fail(MSB_ERR_UNSUPPORTED, n.err);
  static_assert(sizeof(ncclUniqueId) == MSB_NCCL_UNIQUE_ID_BYTES, "ncclUniqueId size");
  ncclUniqueId id;
  NCCL_TRY(n.GetUniqueId(&id));
  memcpy(id128, &id, sizeof id);
  return MSB_OK;
}
extern "C" MSB_API int msb_nccl_comm_create(msb_ctx *ctx, int nranks, int rank, const void *id128, void **comm) {
  REQUIRE(ctx && id128 && comm, "NULL argument");
  REQUIRE(nranks > 0 && rank >= 0 && rank < nranks, "bad rank");
  NcclApi &n = nccl_api();
  if (!n.ok) return fail(MSB_ERR_UNSUPPORTED, n.err);
  CU_TRY(cudaSetDevice(ctx->device));
  ncclUniqueId id;
  memcpy(&id, id128, sizeof id);
  ncclComm_t c = nullptr;
  NCCL_TRY(n.CommInitRank(&c, nranks, id, rank));
  *comm = c;
  return MSB_OK;
}
extern "C" MSB_API int msb_nccl_comm_destroy(void *comm) {
  if (!comm) return MSB_OK;
  NcclApi &n = nccl_api();
  if (!n.ok) return fail(MSB_ERR_UNSUPPORTED, n.err);
  NCCL_TRY(n.CommDestroy((ncclComm_t)comm));
  return MSB_OK;
}

// every suffstat of the state is a count of rows (bb heads / tails, dd counts): the deltas are integers bounded by the
// GLOBAL row count, so they cross the wire as exact int32 when that count fits
static bool counts_only(const msb_state *st) {
  for (const auto &m : st->models)
    if (m.family != MSB_FAMILY_BB && m.family != MSB_FAMILY_DD) return false;  // (bbnc's p is not a count)
  return true;
}

// Sum the pending suffstat deltas over the ranks of `comm` on the context's stream and apply the sum to the resident
// suffstats: afterwards every replica holds the same state.  global_rows = rows over ALL ranks (0 = unknown: fp64
// deltas).  Every rank must pass the same value -- the element type of the collective depends on it.
extern "C" MSB_API int msb_state_allreduce_deltas(msb_state *st, void *nccl_comm, uint64_t global_rows) {
  REQUIRE(st && nccl_comm, "NULL argument");
  NcclApi &n = nccl_api();
  if (!n.ok) return fail(MSB_ERR_UNSUPPORTED, n.err);
  msb_ctx *ctx = st->ctx;
  CU_TRY(cudaSetDevice(ctx->device));
  static const bool no_i32 = getenv("MSB_NO_I32_DELTAS") != nullptr;
  const bool i32 = counts_only(st) && global_rows > 0 && global_rows < (1ull << 31) && !no_i32;
  if (i32) {
    if (!st->d_delta_i32) CU_TRY(cudaMalloc(&st->d_delta_i32, sizeof(int32_t) * st->SS));
    LAUNCH(ctx, delta_to_i32_kernel, cdiv(st->SS, 256), 256, 0, st->d_delta, st->SS, st->d_delta_i32);
    NCCL_TRY(n.AllReduce(st->d_delta_i32, st->d_delta_i32, st->SS, ncclInt32, ncclSum, (ncclComm_t)nccl_comm, ctx->stream));
    LAUNCH(ctx, delta_from_i32_kernel, cdiv(st->SS, 256), 256, 0, st->d_delta_i32, st->SS, st->d_delta);
  } else {
    NCCL_TRY(n.AllReduce(st->d_delta, st->d_delta, st->SS, ncclFloat64, ncclSum, (ncclComm_t)nccl_comm, ctx->stream));
  }
  st->last_allreduce_bytes = st->SS * (i32 ? sizeof(int32_t) : sizeof(double));
  return apply_deltas(st);
}
extern "C" MSB_API int msb_state_last_allreduce_bytes(msb_state *st, size_t *bytes) {
  REQUIRE(st && bytes, "NULL argument");
  *bytes = st->last_allreduce_bytes;
  return MSB_OK;
}

// ---- sweep -------------------------------------------------------------------------
// rows per chunk of a sweep or a prediction: the score matrix of one chunk stays within MSB_SCORES_MB (default 4 GB)
static size_t score_chunk_rows(const msb_state *st, size_t nrows) {
  size_t budget_mb = 4096;
  if (const char *e = getenv("MSB_SCORES_MB")) budget_mb = std::max(1, atoi(e));
  size_t chunk = std::max<size_t>(1, std::min(nrows, budget_mb * 1024 * 1024 / (st->ld * sizeof(float))));
  if (chunk < nrows) chunk = std::max<size_t>(1024, chunk / 1024 * 1024);
  return chunk;
}

// the sweep keeps the scores in the sampler-friendly blocked layout; the CUDA-core NIW kernel (dim != 64)
// accumulates row-major only
static bool blocked_layout(const msb_state *st) {
  bool niw_tc_only = true;
  for (const auto &f : st->feats) if (f.kind == KIND_NIW && (f.dim != 64 || getenv("MSB_NO_TENSOR"))) niw_tc_only = false;
  if (st->has_dm) niw_tc_only = false;  // dm_score_kernel accumulates row-major
  return niw_tc_only && !getenv("MSB_NO_BLOCKED");
}

// one group per row of the chunk [lo, hi) of a call over [row_lo, row_hi), from the score matrix launch_score left in
// d_scores: column into d_newcol, slot into d_newslot.  uniforms (host, one per row of the call) or NULL -> Philox
// (seed, row_id_offset + row, counter).
static int launch_sampler(msb_state *st, bool blocked, size_t K, size_t row_lo, size_t lo, size_t hi, const float *uniforms,
                          uint64_t seed, uint64_t counter, uint64_t row_id_offset) {
  msb_ctx *ctx = st->ctx;
  const size_t skip = lo - row_origin(lo);
  const float *d_u = nullptr;
  if (uniforms) {
    CU_TRY(cudaMemcpyAsync(st->d_uniforms, uniforms + (lo - row_lo), sizeof(float) * (hi - lo), cudaMemcpyHostToDevice, ctx->stream));
    d_u = st->d_uniforms;
  }
  if (tile_sampler_fits(K))
    MSB_TRY(launch_tile_sampler(ctx, blocked, st->d_scores + (blocked ? 0 : skip * st->ld), st->ld, blocked ? skip : 0, (int)K,
                                hi - lo, d_u, seed, counter, row_id_offset + lo, st->d_col2slot, st->d_newcol,
                                st->d_newslot, blocked && st->rowmax_valid ? st->d_rowmax : nullptr));
  else if (blocked)
    LAUNCH(ctx, sample_blocked_kernel, cdiv(hi - lo, 128), 128, 0, st->d_scores, st->ld, skip, (int)K, hi - lo, d_u, seed,
           counter, row_id_offset + lo, st->d_col2slot, st->d_newcol, st->d_newslot,
           (const int *)(st->rowmax_valid ? st->d_rowmax : nullptr));
  else
    LAUNCH(ctx, sample_kernel, cdiv(hi - lo, 128), 128, 0, st->d_scores + skip * st->ld, st->ld, (int)K, hi - lo, d_u, seed,
           counter, row_id_offset + lo, st->d_col2slot, st->d_newcol, st->d_newslot);
  return MSB_OK;
}

extern "C" MSB_API int msb_state_sweep(msb_state *st, size_t row_lo, size_t row_hi, const msb_sweep_opts *opts,
                               msb_sweep_result *res) {
  REQUIRE(st && opts, "NULL argument");
  REQUIRE(st->dv, "no dataview bound");
  REQUIRE(row_lo <= row_hi && row_hi <= st->n, "bad row range");
  msb_ctx *ctx = st->ctx;
  CU_TRY(cudaSetDevice(ctx->device));
  MSB_TRY(prepare_columns(st));
  const size_t K = st->h_col2slot.size();
  const size_t nrows = row_hi - row_lo;
  if (res) { res->rows = nrows; res->moved = 0; res->units = (uint64_t)nrows * K * st->D; }
  if (!nrows) return MSB_OK;
  const size_t chunk = score_chunk_rows(st, nrows);
  const size_t nchunks = (nrows + chunk - 1) / chunk;
  MSB_TRY(ensure_scores(st, chunk + 128));
  MSB_TRY(ensure_rows(st, chunk));
  const size_t ring = st->sweep_seq % msb_state::TIMING_RING;
  std::vector<PhaseEvents> &ev = st->events[ring];
  while (ev.size() < nchunks + 1) {
    PhaseEvents pe;
    for (auto &e : pe.e) CU_TRY(cudaEventCreate(&e));
    ev.push_back(pe);
  }
  st->ring_nchunks[ring] = nchunks;
  st->sweep_seq++;
  const bool blocked = blocked_layout(st);
  LAUNCH(ctx, zero_u64_kernel, 1, 1, 0, st->d_counter);
  CU_TRY(cudaEventRecord(ev[0].e[0], ctx->stream));
  MSB_TRY(build_params(st));
  CU_TRY(cudaEventRecord(ev[0].e[1], ctx->stream));
  for (size_t c = 0; c < nchunks; c++) {
    const size_t lo = row_lo + c * chunk, hi = std::min(row_hi, lo + chunk);
    PhaseEvents &pe = ev[c + 1];
    CU_TRY(cudaEventRecord(pe.e[0], ctx->stream));
    const size_t skip = lo - row_origin(lo);
    MSB_TRY(launch_score(st, lo, hi, st->d_scores, blocked, true));
    st->last_skip = skip;
    CU_TRY(cudaEventRecord(pe.e[1], ctx->stream));
    MSB_TRY(launch_sampler(st, blocked, K, row_lo, lo, hi, opts->uniforms, opts->seed, opts->sweep, opts->row_id_offset));
    CU_TRY(cudaEventRecord(pe.e[2], ctx->stream));
    MSB_TRY(launch_update(st, lo, hi));
    CU_TRY(cudaEventRecord(pe.e[3], ctx->stream));
  }
  st->last_rows = nchunks == 1 ? nrows : (nrows - (nchunks - 1) * chunk); st->last_cols = K;
  st->last_blocked = blocked;
  CU_TRY(cudaEventRecord(ev[0].e[2], ctx->stream));
  if (!opts->defer_apply) MSB_TRY(launch_apply(st));
  CU_TRY(cudaEventRecord(ev[0].e[3], ctx->stream));
  LAUNCH(ctx, publish_counter_kernel, 1, 1, 0, (const unsigned long long *)st->d_counter, st->h_moved_dev);
  MSB_TRY(refresh_counts(st));  // marks the host copy of the group counts stale; no synchronisation
  st->last_res.rows = nrows; st->last_res.units = (uint64_t)nrows * K * st->D; st->last_res.moved = 0;
  if (opts->flags & MSB_SWEEP_ASYNC) {  // everything is enqueued; msb_state_sweep_wait collects the result
    if (res) res->moved = 0;
    return MSB_OK;
  }
  CU_TRY(cudaStreamSynchronize(ctx->stream));
  st->last_res.moved = *st->h_moved;
  if (res) res->moved = *st->h_moved;
  return MSB_OK;
}

extern "C" MSB_API int msb_state_sweep_wait(msb_state *st, msb_sweep_result *res) {
  REQUIRE(st, "NULL argument");
  CU_TRY(cudaSetDevice(st->ctx->device));
  CU_TRY(cudaStreamSynchronize(st->ctx->stream));
  st->last_res.moved = *st->h_moved;
  if (res) *res = st->last_res;
  return MSB_OK;
}

// ---- posterior predictive of a row range (DESIGN.md section 4.9) ------------------------------------------------------
// logp / resp / MAP from one score matrix: the 32-row tile form where a tile fits (as the sampler), else one thread per row
static int launch_predict(msb_state *st, bool blocked, int K, size_t lo, size_t hi, const double *d_logz, double *logp,
                          int32_t *map_col, float *resp) {
  msb_ctx *ctx = st->ctx;
  const size_t nrows = hi - lo, skip = lo - row_origin(lo);
  const float *scores = st->d_scores + (blocked ? 0 : skip * st->ld);
  const size_t sk = blocked ? skip : 0;
  const int *rowmax = blocked && st->rowmax_valid ? st->d_rowmax : nullptr;
  if (!tile_sampler_fits(K)) {
    if (blocked)
      LAUNCH(ctx, predict_rows_kernel<false>, cdiv(nrows, 128), 128, 0, scores, st->ld, sk, K, nrows, rowmax, d_logz, logp, map_col, resp, (size_t)K);
    else
      LAUNCH(ctx, predict_rows_kernel<true>, cdiv(nrows, 128), 128, 0, scores, st->ld, sk, K, nrows, rowmax, d_logz, logp, map_col, resp, (size_t)K);
    return MSB_OK;
  }
  const size_t nblk = (sk + nrows + 31) / 32 - sk / 32;
  // warps per SM, as launch_tile_sampler chooses them: one-warp blocks where four-warp blocks would waste shared memory
  auto warps_per_sm = [&](int sw) { return (size_t)sw * std::min<size_t>(32 / sw, ctx->smem_optin / predict_tile_smem(sw, K, !blocked)); };
  const bool one_warp = 2 * warps_per_sm(1) >= 3 * warps_per_sm(4);
#define MSB_PREDICT_TILE(SW)                                                                                                  \
  do {                                                                                                                    \
    const size_t smem = predict_tile_smem(SW, K, !blocked);                                                               \
    const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(32 / SW, ctx->smem_optin / smem));                       \
    const unsigned grid = (unsigned)std::min<size_t>((nblk + SW - 1) / SW, (size_t)ctx->sm_count * per_sm);               \
    if (blocked)                                                                                                          \
      LAUNCH(ctx, (predict_tile_kernel<SW, false>), grid, SW * 32, smem, scores, st->ld, sk, K, nrows, rowmax, d_logz, logp, map_col, resp, (size_t)K); \
    else                                                                                                                  \
      LAUNCH(ctx, (predict_tile_kernel<SW, true>), grid, SW * 32, smem, scores, st->ld, sk, K, nrows, (const int *)nullptr, d_logz, logp, map_col, resp, (size_t)K); \
  } while (0)
  if (one_warp) MSB_PREDICT_TILE(1);
  else MSB_PREDICT_TILE(4);
#undef MSB_PREDICT_TILE
  return MSB_OK;
}

extern "C" MSB_API int msb_state_predict(msb_state *st, size_t row_lo, size_t row_hi, const msb_predict_opts *opts,
                                         msb_predict_out *out, size_t *gids, size_t cap, size_t *ncols) {
  REQUIRE(st && opts && out && ncols, "NULL argument");
  REQUIRE(st->dv, "no dataview bound");
  REQUIRE(row_lo <= row_hi && row_hi <= st->n, "bad row range");
  msb_ctx *ctx = st->ctx;
  CU_TRY(cudaSetDevice(ctx->device));
  MSB_TRY(prepare_columns(st));
  const size_t K = st->h_col2slot.size(), D = st->D;
  *ncols = K;
  if (gids) { REQUIRE(cap >= K, "buffer too small"); for (size_t c = 0; c < K; c++) gids[c] = st->h_colgid[c]; }
  REQUIRE(!out->resp || out->resp_ld >= K, "resp_ld smaller than the number of groups");
  std::vector<ImputeFeat> ifeat(D);
  size_t W = 0;
  for (size_t d = 0; d < D; d++) {
    ifeat[d].off = W; ifeat[d].fac = nullptr;
    W += (st->feats[d].kind == KIND_NIW || st->feats[d].kind == KIND_DM) ? st->feats[d].dim : 1;
  }
  const bool impute = out->values != nullptr;
  const bool draw = impute || out->draw_gid;
  if (impute) {
    REQUIRE(out->values_ld >= W, "values_ld smaller than the row width");
    // the draw counters counter * 2^40 + row id * D + d must not overlap between counters
    REQUIRE(opts->counter < (1ull << 24), "counter must be below 2^24 for imputation");
    REQUIRE(opts->row_id_offset + row_hi <= ((1ull << 40) - 1) / std::max<size_t>(D, 1), "row ids times features must stay below 2^40");
  }
  const size_t nrows = row_hi - row_lo;
  if (!nrows) return MSB_OK;
  const size_t chunk = score_chunk_rows(st, nrows);
  const size_t nchunks = (nrows + chunk - 1) / chunk;
  MSB_TRY(ensure_scores(st, chunk + 128));
  MSB_TRY(ensure_rows(st, chunk));
  const bool blocked = blocked_layout(st);
  MSB_TRY(build_params(st));
  Scratch<double> d_logz, d_logp, d_vals;
  Scratch<int32_t> d_map;
  Scratch<float> d_resp;
  Scratch<uint32_t> d_unsupported;
  Scratch<ImputeFeat> d_ifeat;
  std::vector<Scratch<double>> d_fac(D);
  CU_TRY(d_logz.alloc(1));
  CU_TRY(d_logp.alloc(chunk));
  CU_TRY(d_map.alloc(chunk));
  if (out->resp) CU_TRY(d_resp.alloc(chunk * K));
  LAUNCH(ctx, crp_logz_kernel, 1, 256, 0, st->d_ss, st->d_col2slot, (int)K, (float)st->alpha, d_logz.p);
  if (impute) {
    CU_TRY(d_vals.alloc(chunk * W));
    CU_TRY(d_unsupported.alloc(1));
    CU_TRY(cudaMemsetAsync(d_unsupported, 0, sizeof(uint32_t), ctx->stream));
    for (size_t d = 0; d < D; d++) {
      const FeatDev &f = st->feats[d];
      if (f.kind != KIND_NIW) continue;
      const size_t smem = ((size_t)f.dim * f.dim + f.dim) * sizeof(double);
      if (smem > 48 * 1024) CU_TRY(cudaFuncSetAttribute(niw_predictive_factor_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      CU_TRY(d_fac[d].alloc(st->kmax * ((size_t)f.dim * f.dim + f.dim + 1)));
      LAUNCH(ctx, niw_predictive_factor_kernel, (unsigned)K, 128, smem, f, st->d_hp, st->d_ss, st->d_col2slot, d_fac[d].p);
      ifeat[d].fac = d_fac[d].p;
    }
    CU_TRY(d_ifeat.alloc(D));
    CU_TRY(cudaMemcpyAsync(d_ifeat.p, ifeat.data(), sizeof(ImputeFeat) * D, cudaMemcpyHostToDevice, ctx->stream));
  }
  std::vector<int32_t> h_map(chunk), h_draw(draw ? chunk : 0);
  for (size_t c = 0; c < nchunks; c++) {
    const size_t lo = row_lo + c * chunk, hi = std::min(row_hi, lo + chunk), n = hi - lo, r0 = lo - row_lo;
    MSB_TRY(launch_score(st, lo, hi, st->d_scores, blocked, true));
    MSB_TRY(launch_predict(st, blocked, (int)K, lo, hi, d_logz, d_logp, d_map, d_resp));
    if (draw) MSB_TRY(launch_sampler(st, blocked, K, row_lo, lo, hi, opts->uniforms, opts->seed, opts->counter, opts->row_id_offset));
    if (impute)
      LAUNCH(ctx, impute_kernel, dim3(cdiv(n, 128), (unsigned)D), 128, 0, st->d_feats, (const ImputeFeat *)d_ifeat.p, (int)D,
             st->d_hp, st->d_ss, st->d_newslot, lo, n, opts->seed, opts->counter << 40, opts->row_id_offset + lo, d_vals.p, W,
             d_unsupported.p);
    if (out->logp) CU_TRY(cudaMemcpyAsync(out->logp + r0, d_logp, sizeof(double) * n, cudaMemcpyDeviceToHost, ctx->stream));
    if (out->map_gid) CU_TRY(cudaMemcpyAsync(h_map.data(), d_map, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, ctx->stream));
    if (draw) CU_TRY(cudaMemcpyAsync(h_draw.data(), st->d_newcol, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, ctx->stream));
    if (out->resp)
      CU_TRY(cudaMemcpy2DAsync(out->resp + r0 * out->resp_ld, sizeof(float) * out->resp_ld, d_resp, sizeof(float) * K, sizeof(float) * K,
                               n, cudaMemcpyDeviceToHost, ctx->stream));
    if (impute)
      CU_TRY(cudaMemcpy2DAsync(out->values + r0 * out->values_ld, sizeof(double) * out->values_ld, d_vals, sizeof(double) * W,
                               sizeof(double) * W, n, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    for (size_t i = 0; i < n; i++) {
      if (out->map_gid) out->map_gid[r0 + i] = (int64_t)st->h_colgid[h_map[i]];
      if (out->draw_gid) out->draw_gid[r0 + i] = (int64_t)st->h_colgid[h_draw[i]];
    }
    st->last_skip = lo - row_origin(lo);
  }
  st->last_rows = nchunks == 1 ? nrows : (nrows - (nchunks - 1) * chunk); st->last_cols = K;
  st->last_blocked = blocked;
  if (impute) {
    uint32_t bad = 0;
    CU_TRY(cudaMemcpy(&bad, d_unsupported, sizeof(bad), cudaMemcpyDeviceToHost));
    if (bad) return fail(MSB_ERR_UNSUPPORTED, "multinomial sampling unimplemented");  // dm.cpp:100-111
  }
  return MSB_OK;
}

// ---- hyperparameter grids: one Gibbs step over the hypers (DESIGN.md section 4.10) ------------------------------------
// bnb's score_data drops the r-dependent data term (score_data_cell), so the conditional of a grid over r is not the
// one these weights give: every point must carry the feature's current r
static int check_bnb_r(const msb_state *st, size_t feature, const double *pts, size_t npoints) {
  const double r = st->h_hp[st->feats[feature].hp_off + 2];
  for (size_t g = 0; g < npoints; g++)
    if (pts[g * 3 + 2] != r)
      return fail(MSB_ERR_INVALID, "feature " + std::to_string(feature) + ": bnb grid point " + std::to_string(g) +
                                       " changes r; only (alpha, beta) can be resampled on a grid");
  return MSB_OK;
}

static int upload_grids(msb_state *st) {
  std::vector<HpRow> rows;
  size_t npts = 0, nlp = 0, gmax = 0;
  for (size_t d = 0; d <= st->D; d++) {
    const size_t G = st->grid_lp[d].size();
    if (!G) continue;
    HpRow r;
    memset(&r, 0, sizeof(r));
    r.feat = (int32_t)d; r.npoints = (int32_t)G; r.nhp = (uint32_t)(st->grid_pts[d].size() / G);
    r.pt_off = npts; r.lp_off = nlp;
    npts += st->grid_pts[d].size(); nlp += G; gmax = std::max(gmax, G);
    rows.push_back(r);
  }
  const size_t rows_b = (sizeof(HpRow) * rows.size() + 255) / 256 * 256;
  std::vector<char> h(rows_b + sizeof(double) * (npts + nlp));
  if (!rows.empty()) memcpy(h.data(), rows.data(), sizeof(HpRow) * rows.size());
  double *pts = (double *)(h.data() + rows_b), *lp = pts + npts;
  for (const HpRow &r : rows) {
    memcpy(pts + r.pt_off, st->grid_pts[r.feat].data(), sizeof(double) * st->grid_pts[r.feat].size());
    memcpy(lp + r.lp_off, st->grid_lp[r.feat].data(), sizeof(double) * r.npoints);
  }
  CU_TRY(cudaSetDevice(st->ctx->device));
  void *d = nullptr;
  if (!rows.empty()) {
    CU_TRY(cudaMalloc(&d, h.size()));
    cudaError_t e = cudaMemcpyAsync(d, h.data(), h.size(), cudaMemcpyHostToDevice, st->ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st->ctx->stream);  // h is pageable and goes out of scope
    if (e != cudaSuccess) { cudaFree(d); CU_TRY(e); }
  }
  CU_TRY(cudaStreamSynchronize(st->ctx->stream));  // an hp_gibbs still in flight may read the old buffer
  CU_TRY(cudaFree(st->d_grid));
  st->d_grid = d;
  st->hp_rows = rows;
  st->grid_gmax = gmax;
  return MSB_OK;
}

static void grids_resize(msb_state *st) {
  if (st->grid_lp.empty()) { st->grid_pts.resize(st->D + 1); st->grid_lp.resize(st->D + 1); }
}

// grid `row` (a feature, or D for alpha) := (pts, lp); the host copies change only if the device buffer was rebuilt
static int replace_grid(msb_state *st, size_t row, std::vector<double> pts, std::vector<double> lp) {
  st->grid_pts[row].swap(pts);
  st->grid_lp[row].swap(lp);
  const int rc = upload_grids(st);
  if (rc != MSB_OK) { st->grid_pts[row].swap(pts); st->grid_lp[row].swap(lp); }
  return rc;
}

// a grid's points are a launch dimension of the hp kernels (gridDim.y)
constexpr size_t HP_MAX_POINTS = 65535;

extern "C" MSB_API int msb_state_set_hp_grid(msb_state *st, size_t feature, const double *points, size_t npoints, size_t nhp,
                                             const double *log_prior) {
  REQUIRE(st, "NULL argument");
  REQUIRE(feature < st->D, "bad feature index");
  grids_resize(st);
  if (npoints == 0) return replace_grid(st, feature, {}, {});
  REQUIRE(points && log_prior, "NULL argument");
  const msb_model_desc &m = st->models[feature];
  REQUIRE(nhp == hp_size(m), "feature " + std::to_string(feature) + ": a grid point has " + std::to_string(nhp) +
                                 " values, the family takes " + std::to_string(hp_size(m)));
  REQUIRE(npoints <= HP_MAX_POINTS, "too many grid points: at most " + std::to_string(HP_MAX_POINTS));
  for (size_t i = 0; i < npoints * nhp; i++) REQUIRE(std::isfinite(points[i]), "non-finite grid value");
  for (size_t g = 0; g < npoints; g++) REQUIRE(std::isfinite(log_prior[g]), "non-finite log prior");
  if (m.family == MSB_FAMILY_BNB) MSB_TRY(check_bnb_r(st, feature, points, npoints));
  return replace_grid(st, feature, std::vector<double>(points, points + npoints * nhp),
                      std::vector<double>(log_prior, log_prior + npoints));
}

extern "C" MSB_API int msb_state_set_cluster_hp_grid(msb_state *st, const double *alphas, size_t npoints, const double *log_prior) {
  REQUIRE(st, "NULL argument");
  grids_resize(st);
  if (npoints == 0) return replace_grid(st, st->D, {}, {});
  REQUIRE(alphas && log_prior, "NULL argument");
  REQUIRE(npoints <= HP_MAX_POINTS, "too many grid points: at most " + std::to_string(HP_MAX_POINTS));
  for (size_t g = 0; g < npoints; g++) {
    REQUIRE(std::isfinite(alphas[g]) && alphas[g] > 0.0, "alpha must be positive and finite");  // group_manager.hpp:120
    REQUIRE(std::isfinite(log_prior[g]), "non-finite log prior");
  }
  return replace_grid(st, st->D, std::vector<double>(alphas, alphas + npoints), std::vector<double>(log_prior, log_prior + npoints));
}

extern "C" MSB_API int msb_state_hp_gibbs(msb_state *st, const msb_hp_gibbs_opts *opts, msb_hp_gibbs_out *out) {
  REQUIRE(st && opts, "NULL argument");
  REQUIRE(opts->counter < (1ull << 32), "counter must be below 2^32");
  const size_t D = st->D, R = st->hp_rows.size(), G = st->grid_gmax;
  REQUIRE(!out || !out->logw || out->logw_ld >= G, "logw_ld smaller than the largest grid");
  if (out && out->choice)
    for (size_t d = 0; d <= D; d++) out->choice[d] = -1;
  if (!R) return MSB_OK;
  for (const HpRow &r : st->hp_rows)
    if ((size_t)r.feat < D && st->models[r.feat].family == MSB_FAMILY_BNB)
      MSB_TRY(check_bnb_r(st, r.feat, st->grid_pts[r.feat].data(), r.npoints));
  msb_ctx *ctx = st->ctx;
  CU_TRY(cudaSetDevice(ctx->device));
  MSB_TRY(prepare_columns(st));
  MSB_TRY(sync_small(st));
  const size_t K = st->h_col2slot.size();
  const size_t rows_b = (sizeof(HpRow) * R + 255) / 256 * 256;
  const HpRow *d_rows = (const HpRow *)st->d_grid;
  const double *d_pts = (const double *)((const char *)st->d_grid + rows_b);
  size_t npts = 0;
  for (const HpRow &r : st->hp_rows) npts += (size_t)r.npoints * r.nhp;
  const double *d_lp = d_pts + npts;
  // scratch: L [R][G] | logw [R][G] | choice [R] (int64) | niw, for the largest niw grid of P points: ld0 [P] and the
  // per-(point, group) values [P][K]
  size_t niw_pts = 0;
  for (const HpRow &r : st->hp_rows)
    if ((size_t)r.feat < D && st->feats[r.feat].kind == KIND_NIW) niw_pts = std::max(niw_pts, (size_t)r.npoints);
  MSB_TRY(ensure(&st->d_hpwork, &st->hpwork_cap, 2 * R * G + R + niw_pts * (K + 1)));
  double *d_L = st->d_hpwork, *d_logw = d_L + R * G;
  int64_t *d_choice = (int64_t *)(d_logw + R * G);
  double *d_ld0 = (double *)(d_choice + R), *d_niw = d_ld0 + niw_pts;
  LAUNCH(ctx, hp_grid_kernel, dim3((unsigned)R, (unsigned)G), HP_THREADS, 0, st->d_feats, (int)D, d_rows, d_pts, st->d_ss,
         st->d_col2slot, (int)K, G, d_L);
  for (size_t i = 0; i < R; i++) {
    const HpRow &r = st->hp_rows[i];
    const double *pts = d_pts + r.pt_off;
    if ((size_t)r.feat == D) {
      LAUNCH(ctx, hp_alpha_kernel, 1, HP_THREADS, 0, st->d_ss, st->d_col2slot, (int)K, pts, r.npoints, d_L + i * G);
      continue;
    }
    const FeatDev &f = st->feats[r.feat];
    if (f.kind != KIND_NIW) continue;
    const size_t smem0 = (size_t)f.dim * f.dim * sizeof(double), smem = smem0 + f.dim * sizeof(double);
    if (smem > 48 * 1024) {
      CU_TRY(opt_in_smem(niw_hp_prior_kernel, smem0));
      CU_TRY(opt_in_smem(niw_hp_group_kernel, smem));
    }
    LAUNCH(ctx, niw_hp_prior_kernel, (unsigned)r.npoints, 128, smem0, (int)f.dim, pts, r.nhp, d_ld0);
    LAUNCH(ctx, niw_hp_group_kernel, dim3((unsigned)K, (unsigned)r.npoints), 128, smem, f, pts, r.nhp, d_ld0, st->d_ss,
           st->d_col2slot, (int)K, d_niw);
    LAUNCH(ctx, hp_reduce_kernel, (unsigned)r.npoints, HP_THREADS, 0, d_niw, (int)K, d_L + i * G);
  }
  LAUNCH(ctx, hp_draw_kernel, cdiv(R, 32), 32, 0, d_rows, (int)R, d_lp, d_L, G, opts->seed, opts->counter, d_logw, d_choice);
  std::vector<double> h(R * G + R);
  CU_TRY(cudaMemcpyAsync(h.data(), d_logw, sizeof(double) * h.size(), cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(cudaStreamSynchronize(ctx->stream));
  const double *logw = h.data();
  const int64_t *choice = (const int64_t *)(h.data() + R * G);
  for (size_t i = 0; i < R; i++) {
    if (choice[i] >= 0) continue;
    const HpRow &r = st->hp_rows[i];
    const std::string who = (size_t)r.feat == D ? std::string("alpha") : "feature " + std::to_string(r.feat);
    for (int g = 0; g < r.npoints; g++) {
      const double w = logw[i * G + g];
      if (std::isnan(w)) return fail(MSB_ERR_INVALID, who + ": grid point " + std::to_string(g) + " has a NaN weight");
      if (w == HUGE_VAL) return fail(MSB_ERR_INVALID, who + ": grid point " + std::to_string(g) + " has weight +inf");
    }
    return fail(MSB_ERR_INVALID, who + ": every grid point has weight -inf");
  }
  for (size_t i = 0; i < R; i++) {
    const HpRow &r = st->hp_rows[i];
    const double *pt = st->grid_pts[r.feat].data() + (size_t)choice[i] * r.nhp;
    if ((size_t)r.feat == D) st->alpha = *pt;
    else write_hp(st, r.feat, 0, pt, r.nhp);
    if (out && out->choice) out->choice[r.feat] = choice[i];
    if (out && out->logw)
      for (int g = 0; g < r.npoints; g++) out->logw[(size_t)r.feat * out->logw_ld + g] = logw[i * G + g];
  }
  return MSB_OK;
}

// ---- non-conjugate parameters: slice sampling of bbnc's p, fresh p for the empty groups (DESIGN.md section 4.11) ------
// The stream packing (msb_theta.cuh) holds a feature index in 16 bits; a launch covers at most 65535 features (gridDim.y)
constexpr size_t THETA_MAX_FEATURE = 65535;

// One launch of theta_kernel (slice) or redraw_empty_kernel over the features in tf and every group column, then the
// call's one synchronise; the new p are committed into d_ss only if no column was refused.
// d_theta = [flags: 2 x u32 | pad | ThetaFeat[A] | gid per column, u32 [K] | pad | p [A][K] (fp64) | status [A][K] (u8)]
static int theta_run(msb_state *st, bool slice, const std::vector<ThetaFeat> &tf, uint64_t seed, uint64_t counter, size_t *capped) {
  if (capped) *capped = 0;
  if (tf.empty() || st->gid2slot.empty()) return MSB_OK;
  for (const auto &p : st->gid2slot)
    REQUIRE(p.first < (1ull << 32), "gid " + std::to_string(p.first) + " does not fit the stream packing (gids below 2^32)");
  msb_ctx *ctx = st->ctx;
  CU_TRY(cudaSetDevice(ctx->device));
  MSB_TRY(prepare_columns(st));
  MSB_TRY(sync_small(st));
  const size_t K = st->h_col2slot.size(), A = tf.size();
  const size_t off_tf = 16, off_gid = off_tf + sizeof(ThetaFeat) * A, off_p = (off_gid + sizeof(uint32_t) * K + 7) / 8 * 8,
               off_s = off_p + sizeof(double) * A * K;
  std::vector<char> h(off_p, 0);
  const uint32_t flags0[2] = {0u, UINT32_MAX};
  memcpy(h.data(), flags0, sizeof(flags0));
  memcpy(h.data() + off_tf, tf.data(), sizeof(ThetaFeat) * A);
  uint32_t *hg = (uint32_t *)(h.data() + off_gid);
  for (size_t c = 0; c < K; c++) hg[c] = (uint32_t)st->h_colgid[c];
  MSB_TRY(ensure(&st->d_theta, &st->theta_cap, off_s + A * K));
  char *d = st->d_theta;
  uint32_t *d_flags = (uint32_t *)d;
  const ThetaFeat *d_tf = (const ThetaFeat *)(d + off_tf);
  const uint32_t *d_gid = (const uint32_t *)(d + off_gid);
  double *d_p = (double *)(d + off_p);
  uint8_t *d_s = (uint8_t *)(d + off_s);
  CU_TRY(cudaMemcpyAsync(d, h.data(), h.size(), cudaMemcpyHostToDevice, ctx->stream));  // pageable: staged on return
  const dim3 grid(cdiv(K, THETA_THREADS), (unsigned)A);
  if (slice)
    LAUNCH(ctx, theta_kernel, grid, THETA_THREADS, 0, st->d_feats, d_tf, st->d_hp, st->d_ss, st->d_col2slot, d_gid, (int)K, seed,
           counter, d_p, d_s, d_flags);
  else
    LAUNCH(ctx, redraw_empty_kernel, grid, THETA_THREADS, 0, st->d_feats, d_tf, st->d_hp, st->d_ss, st->d_col2slot, d_gid, (int)K,
           seed, counter, d_p, d_s, d_flags);
  uint32_t hf[2];
  CU_TRY(cudaMemcpyAsync(hf, d_flags, sizeof(hf), cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(cudaStreamSynchronize(ctx->stream));
  if (hf[1] != UINT32_MAX) {
    const size_t a = hf[1] / K, c = hf[1] % K;
    const std::string who = "feature " + std::to_string(tf[a].feat) + ": gid " + std::to_string(st->h_colgid[c]);
    return fail(MSB_ERR_INVALID, slice ? who + ": the current p has a non-finite score_data; the slice update needs a finite density there"
                                       : who + ": the Beta(alpha, beta) draw of p underflowed (both gamma variates are 0)");
  }
  LAUNCH(ctx, theta_commit_kernel, grid, THETA_THREADS, 0, st->d_feats, d_tf, st->d_col2slot, (int)K, d_p, d_s, st->d_ss);
  for (size_t c = 0; c < K; c++) st->slot_dirty[st->h_col2slot[c]] = 1;
  if (capped) *capped = hf[0];
  return MSB_OK;
}

extern "C" MSB_API int msb_state_theta(msb_state *st, const msb_theta_opts *opts, msb_theta_out *out) {
  static const char *const family_names[] = {"bb", "bnb", "gp", "nich", "dd", "niw", "bbnc", "dm"};
  REQUIRE(st && opts, "NULL argument");
  REQUIRE(opts->nwidths == st->D, std::to_string(opts->nwidths) + " widths for a state of " + std::to_string(st->D) + " features");
  REQUIRE(opts->widths || st->D == 0, "NULL argument");
  REQUIRE(opts->counter < (1ull << 32), "counter must be below 2^32");
  std::vector<ThetaFeat> tf;
  for (size_t d = 0; d < st->D; d++) {
    const double w = opts->widths[d];
    REQUIRE(std::isfinite(w) && w >= 0.0, "feature " + std::to_string(d) + ": the slice width must be finite and non-negative");
    if (w == 0.0) continue;
    REQUIRE(st->models[d].family == MSB_FAMILY_BBNC, "feature " + std::to_string(d) + ": " + family_names[st->models[d].family] +
                                                         " has no non-conjugate parameter (only bbnc's p is slice-sampled)");
    REQUIRE(d < THETA_MAX_FEATURE, "feature " + std::to_string(d) + ": the index does not fit the stream packing (below 65535)");
    ThetaFeat t;
    t.feat = (int32_t)d; t.pad = 0; t.w = w;
    tf.push_back(t);
  }
  size_t capped = 0;
  MSB_TRY(theta_run(st, true, tf, opts->seed, opts->counter, &capped));
  if (out) out->capped = capped;
  return MSB_OK;
}

extern "C" MSB_API int msb_state_redraw_empty(msb_state *st, uint64_t seed, uint64_t counter) {
  REQUIRE(st, "NULL argument");
  REQUIRE(counter < (1ull << 32), "counter must be below 2^32");
  std::vector<ThetaFeat> tf;
  for (size_t d = 0; d < st->D; d++) {
    if (st->models[d].family != MSB_FAMILY_BBNC) continue;
    REQUIRE(d < THETA_MAX_FEATURE, "feature " + std::to_string(d) + ": the index does not fit the stream packing (below 65535)");
    ThetaFeat t;
    t.feat = (int32_t)d; t.pad = 0; t.w = 0.0;
    tf.push_back(t);
  }
  return theta_run(st, false, tf, seed, counter, nullptr);
}

// ---- slice sampling of continuous hypers (DESIGN.md section 4.12) ----------------------------------------------------
// A spec's target, support and stream: msb_hpslice.cuh.  The feature index (alpha: D) is kept below 65535 like theta's.
constexpr size_t HPSL_MAX_FEATURE = 65535;

extern "C" MSB_API int msb_state_slice_hp(msb_state *st, const msb_slice_hp_opts *opts, msb_slice_hp_out *out) {
  REQUIRE(st && opts, "NULL argument");
  REQUIRE(opts->specs || opts->nspecs == 0, "NULL argument");
  REQUIRE(opts->counter < (1ull << 32), "counter must be below 2^32");
  if (out) out->capped = 0;
  const size_t D = st->D, S = opts->nspecs;
  std::vector<HpSliceFeat> tasks;
  std::vector<std::vector<HpSliceSpec>> specs;     // per task, in the order given
  std::vector<std::vector<size_t>> hp_offs;        // per task and spec: the key's offset in the feature's hp vector
  std::map<size_t, size_t> task_of;
  for (size_t i = 0; i < S; i++) {
    const msb_slice_hp_spec &sp = opts->specs[i];
    REQUIRE(sp.key, "NULL argument");
    const size_t d = sp.feature;
    const std::string key = sp.key;
    REQUIRE(d <= D, "spec " + std::to_string(i) + ": feature index " + std::to_string(d) + " out of range (" + std::to_string(D) +
                        " features; " + std::to_string(D) + " = alpha)");
    const std::string who = d == D ? "alpha" : "feature " + std::to_string(d) + ": key '" + key + "'";
    size_t off = 0, cnt = 1;
    int slot = 0, partner = -1;
    double lo = 0.0;
    const msb_model_desc *m = d < D ? &st->models[d] : nullptr;
    if (!m) {
      if (key != "alpha") return fail(MSB_ERR_KEY, "alpha: unknown cluster hp key: " + key);
    } else {
      const int rc = hp_field(*m, key, &off, &cnt);
      if (rc != MSB_OK) return fail(rc, "feature " + std::to_string(d) + ": " + g_last_error);
      const bool vec = m->family == MSB_FAMILY_DD || m->family == MSB_FAMILY_DM ||
                       (m->family == MSB_FAMILY_NIW && (key == "mu" || key == "psi"));
      if (vec) return fail(MSB_ERR_UNSUPPORTED, who + ": a vector hyper cannot be slice-sampled; resample it on a grid (msb_state_set_hp_grid)");
      REQUIRE(!(m->family == MSB_FAMILY_BNB && key == "r"),
              who + ": bnb's score_data drops the r-dependent data term; only (alpha, beta) can be slice-sampled");
      slot = (int)off;
      if (m->family == MSB_FAMILY_NIW) {
        slot = key == "kappa" ? 0 : 1;
        if (key == "nu") lo = (double)m->dim - 1.0;
      }
      if (m->family == MSB_FAMILY_NICH && key == "mu") lo = -HUGE_VAL;
    }
    REQUIRE(d < HPSL_MAX_FEATURE, who + ": the feature index does not fit the stream packing (below 65535)");
    REQUIRE(std::isfinite(sp.width) && sp.width > 0.0, who + ": the slice width must be finite and positive");
    switch (sp.prior) {
      case MSB_HPRIOR_FLAT:
        REQUIRE(std::isfinite(sp.a) && std::isfinite(sp.b) && sp.a < sp.b, who + ": the flat prior needs finite lo < hi");
        break;
      case MSB_HPRIOR_EXPONENTIAL:
        REQUIRE(std::isfinite(sp.a) && sp.a > 0.0, who + ": the exponential prior needs a finite rate > 0");
        break;
      case MSB_HPRIOR_NORMAL:
        REQUIRE(std::isfinite(sp.a) && std::isfinite(sp.b) && sp.b > 0.0, who + ": the normal prior needs a finite mu and a finite s2 > 0");
        break;
      case MSB_HPRIOR_NONINFORMATIVE_BETA:
        REQUIRE(m && (m->family == MSB_FAMILY_BB || m->family == MSB_FAMILY_BBNC || m->family == MSB_FAMILY_BNB) &&
                    (key == "alpha" || key == "beta"),
                who + ": the non-informative beta prior applies to the alpha and beta of bb, bbnc and bnb only");
        partner = 1 - slot;
        break;
      default: return fail(MSB_ERR_INVALID, who + ": unknown prior kind " + std::to_string(sp.prior));
    }
    auto it = task_of.find(d);
    if (it == task_of.end()) {
      HpSliceFeat t;
      memset(&t, 0, sizeof(t));
      t.feat = (int32_t)d; t.niw = -1;
      if (!m) {
        t.h[0] = st->alpha;
      } else {
        const double *h = st->h_hp.data() + st->feats[d].hp_off;
        if (m->family == MSB_FAMILY_NIW) { t.h[0] = h[m->dim]; t.h[1] = h[m->dim + 1 + (size_t)m->dim * m->dim]; }
        else for (size_t j = 0; j < hp_size(*m); j++) t.h[j] = h[j];
      }
      it = task_of.emplace(d, tasks.size()).first;
      tasks.push_back(t);
      specs.emplace_back();
      hp_offs.emplace_back();
    }
    for (const HpSliceSpec &o : specs[it->second]) REQUIRE(o.slot != slot, who + ": the key appears twice");
    HpSliceSpec s;
    memset(&s, 0, sizeof(s));
    s.slot = slot; s.partner = partner; s.prior = sp.prior; s.out = (uint32_t)i;
    s.w = sp.width; s.a = sp.a; s.b = sp.b; s.lo = lo;
    specs[it->second].push_back(s);
    hp_offs[it->second].push_back(off);
  }
  if (tasks.empty()) return MSB_OK;
  msb_ctx *ctx = st->ctx;
  CU_TRY(cudaSetDevice(ctx->device));
  MSB_TRY(prepare_columns(st));
  MSB_TRY(sync_small(st));
  const size_t K = st->h_col2slot.size(), T = tasks.size();
  std::vector<HpSliceSpec> flat;
  size_t nniw = 0;
  for (size_t i = 0; i < T; i++) {
    tasks[i].first = (uint32_t)flat.size();
    tasks[i].nspecs = (uint32_t)specs[i].size();
    flat.insert(flat.end(), specs[i].begin(), specs[i].end());
    if ((size_t)tasks[i].feat < D && st->feats[tasks[i].feat].kind == KIND_NIW) tasks[i].niw = (int32_t)nniw++;
  }
  // d_hpsl = [HpSliceFeat [T] | HpSliceSpec [S] | value [S] (fp64) | status [S] (u8) | pad | niw prep [nniw][K][3] | log |psi| [nniw]]
  const size_t off_spec = sizeof(HpSliceFeat) * T, off_val = off_spec + sizeof(HpSliceSpec) * S, off_status = off_val + sizeof(double) * S,
               off_prep = (off_status + S + 7) / 8 * 8, off_ld0 = off_prep + sizeof(double) * nniw * K * 3,
               total = off_ld0 + sizeof(double) * nniw;
  std::vector<char> h(off_val);
  memcpy(h.data(), tasks.data(), off_spec);
  memcpy(h.data() + off_spec, flat.data(), sizeof(HpSliceSpec) * S);
  MSB_TRY(ensure(&st->d_hpsl, &st->hpsl_cap, total));
  char *d = st->d_hpsl;
  double *d_val = (double *)(d + off_val), *d_prep = (double *)(d + off_prep), *d_ld0 = (double *)(d + off_ld0);
  uint8_t *d_status = (uint8_t *)(d + off_status);
  CU_TRY(cudaMemcpyAsync(d, h.data(), h.size(), cudaMemcpyHostToDevice, ctx->stream));  // pageable: staged on return
  CU_TRY(cudaMemsetAsync(d_status, 0xff, S, ctx->stream));
  for (const HpSliceFeat &t : tasks) {
    if (t.niw < 0) continue;
    const FeatDev &f = st->feats[t.feat];
    const size_t smem = ((size_t)f.dim * f.dim + f.dim) * sizeof(double);
    if (smem > 48 * 1024) CU_TRY(opt_in_smem(niw_slice_prep_kernel, smem));
    LAUNCH(ctx, niw_slice_prep_kernel, (unsigned)(K + 1), 128, smem, f, st->d_hp, st->d_ss, st->d_col2slot, (int)K,
           d_prep + (size_t)t.niw * K * 3, d_ld0 + t.niw);
  }
  LAUNCH(ctx, hp_slice_kernel, (unsigned)T, HP_THREADS, 0, st->d_feats, (int)D, (const HpSliceFeat *)d,
         (const HpSliceSpec *)(d + off_spec), st->d_ss, st->d_col2slot, (int)K, d_prep, d_ld0, opts->seed, opts->counter, d_val,
         d_status);
  std::vector<char> r(off_status + S - off_val);
  CU_TRY(cudaMemcpyAsync(r.data(), d_val, r.size(), cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(cudaStreamSynchronize(ctx->stream));
  const double *val = (const double *)r.data();
  const uint8_t *status = (const uint8_t *)(r.data() + sizeof(double) * S);
  for (size_t i = 0; i < S; i++)
    if (status[i] == HPSL_BAD) {
      const msb_slice_hp_spec &sp = opts->specs[i];
      return fail(MSB_ERR_INVALID, (sp.feature == D ? std::string("alpha") : "feature " + std::to_string(sp.feature) + ": key '" + sp.key + "'") +
                                       ": the target (log prior + score_data) is not finite at the current value; the slice update needs a finite density there");
    }
  size_t capped = 0;
  for (size_t i = 0; i < T; i++) {
    const size_t f = tasks[i].feat;
    if (f == D) { st->alpha = val[specs[i][0].out]; continue; }
    std::vector<double> v(st->h_hp.begin() + st->feats[f].hp_off, st->h_hp.begin() + st->feats[f].hp_off + hp_size(st->models[f]));
    bool changed = false;
    for (size_t j = 0; j < specs[i].size(); j++) {
      const double x = val[specs[i][j].out];
      changed |= memcmp(&x, &v[hp_offs[i][j]], sizeof(double)) != 0;
      v[hp_offs[i][j]] = x;
    }
    if (changed) write_hp(st, f, 0, v.data(), v.size());
  }
  for (size_t i = 0; i < S; i++) {
    capped += status[i] == HPSL_CAPPED;
    if (out && out->values) out->values[i] = val[i];
  }
  if (out) out->capped = capped;
  return MSB_OK;
}

// ---- one pass over host rows in ONE call ---------------------------------------------------------------------------
// What a caller that re-reads its host rows on every pass (the reference does: recarray/dataview.hpp:194-217) would
// otherwise issue as six calls: refresh (this pass's columns become current) -> upload + prefetch of the NEXT pass's
// records on the copy stream -> sweep (+ the delta all-reduce when a communicator is given) -> wait for the previous
// pass's assignments -> start the copy of this pass's assignments.  Nothing in it waits for the compute stream.
extern "C" MSB_API int msb_state_pass(msb_state *st, const msb_pass_opts *opts, msb_sweep_result *res) {
  REQUIRE(st && opts, "NULL argument");
  REQUIRE(st->dv, "no dataview bound");
  static const bool dbg = getenv("MSB_DEBUG_SYNC") != nullptr;  // diagnostics: wait for the device after every sub-step
  static const bool timing = getenv("MSB_PASS_TIMING") != nullptr;  // diagnostics: host time per sub-step, printed at destroy
#define MSB_PASS_STEP(what, expr)                                                                        \
  do {                                                                                                   \
    const auto t0_ = std::chrono::steady_clock::now();                                                   \
    MSB_TRY(expr);                                                                                       \
    if (timing) st->pass_host_ns[what] += (double)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0_).count(); \
    if (dbg) {                                                                                           \
      const cudaError_t e_ = cudaDeviceSynchronize();                                                    \
      if (e_ != cudaSuccess) return fail(MSB_ERR_CUDA, std::string("msb_state_pass, after ") + what + ": " + cudaGetErrorString(e_)); \
    }                                                                                                    \
  } while (0)
  MSB_PASS_STEP("refresh", msb_state_refresh(st));
  if (opts->next_data) {
    MSB_PASS_STEP("upload", msb_dataview_upload(st->dv, opts->next_data, opts->next_mask));
    MSB_PASS_STEP("prefetch", msb_state_prefetch(st));
  }
  msb_sweep_opts so = opts->sweep;
  so.flags |= MSB_SWEEP_ASYNC;
  if (opts->nccl_comm) so.defer_apply = 1;
  MSB_PASS_STEP("sweep", msb_state_sweep(st, 0, st->n, &so, res));
  if (opts->nccl_comm) MSB_PASS_STEP("allreduce", msb_state_allreduce_deltas(st, opts->nccl_comm, opts->global_rows));
  if (opts->assign_out) {
    MSB_PASS_STEP("assignments_wait", msb_state_assignments_wait(st));
    MSB_PASS_STEP("assignments_async", msb_state_assignments_async(st, opts->assign_out, st->n));
  }
#undef MSB_PASS_STEP
  return MSB_OK;
}

// ---- single-value plugin calls (models/base.hpp:25-27) -------------------------------
static int value_to_doubles(const void *value, const msb_runtime_type *vt, std::vector<double> &x) {
  REQUIRE(value && vt, "NULL argument");
  REQUIRE(vt->prim >= 0 && vt->prim < MSB_TYPE_NELEMS && vt->n > 0, "bad runtime type");
  x.resize(vt->n);
  const uint8_t *p = (const uint8_t *)value;
  for (uint32_t i = 0; i < vt->n; i++, p += k_prim_size[vt->prim]) {
    switch (vt->prim) {
      case MSB_TYPE_B: x[i] = *p != 0; break;
      case MSB_TYPE_I8: x[i] = *(const int8_t *)p; break;
      case MSB_TYPE_U8: x[i] = *p; break;
      case MSB_TYPE_I16: { int16_t v; memcpy(&v, p, 2); x[i] = v; } break;
      case MSB_TYPE_U16: { uint16_t v; memcpy(&v, p, 2); x[i] = v; } break;
      case MSB_TYPE_I32: { int32_t v; memcpy(&v, p, 4); x[i] = v; } break;
      case MSB_TYPE_U32: { uint32_t v; memcpy(&v, p, 4); x[i] = v; } break;
      case MSB_TYPE_I64: { int64_t v; memcpy(&v, p, 8); x[i] = (double)v; } break;
      case MSB_TYPE_U64: { uint64_t v; memcpy(&v, p, 8); x[i] = (double)v; } break;
      case MSB_TYPE_F32: { float v; memcpy(&v, p, 4); x[i] = v; } break;
      default: { double v; memcpy(&v, p, 8); x[i] = v; } break;
    }
  }
  return MSB_OK;
}

static int value_op(msb_ctx *ctx, const msb_model_desc *model, int op, const double *hp, size_t nhp, double *ss,
                    size_t nss, const void *value, const msb_runtime_type *vtype, float *score) {
  REQUIRE(ctx && model && hp && ss, "NULL argument");
  MSB_TRY(check_model(*model, 0));
  REQUIRE(nhp == hp_size(*model) && nss == ss_size(*model), "wrong dimension");
  std::vector<double> x;
  MSB_TRY(value_to_doubles(value, vtype, x));
  REQUIRE(x.size() == ((model->family == MSB_FAMILY_NIW || model->family == MSB_FAMILY_DM) ? model->dim : 1u), "shapes do not match");
  CU_TRY(cudaSetDevice(ctx->device));
  Scratch<double> d_buf;
  Scratch<float> d_score;
  const size_t total = nhp + nss + x.size();
  CU_TRY(d_buf.alloc(total));
  CU_TRY(d_score.alloc(64));
  double *d_hp = d_buf.p, *d_ss = d_buf.p + nhp, *d_x = d_ss + nss;
  CU_TRY(cudaMemcpyAsync(d_hp, hp, sizeof(double) * nhp, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(cudaMemcpyAsync(d_ss, ss, sizeof(double) * nss, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(cudaMemcpyAsync(d_x, x.data(), sizeof(double) * x.size(), cudaMemcpyHostToDevice, ctx->stream));
  int rc = MSB_OK;
  if (model->family == MSB_FAMILY_NIW && op == 0) {
    // one group, one row: the batched NIW kernels with K = 1, N = 1
    const uint32_t d = model->dim;
    FeatDev f; memset(&f, 0, sizeof(f));
    f.family = FAM_NIW; f.kind = KIND_NIW; f.dim = d; f.hp_off = 0; f.ss_off = 0; f.ss_w = (uint32_t)nss;
    Scratch<float> d_W, d_x32;
    Scratch<int32_t> d_c2s;
    std::vector<float> x32(x.begin(), x.end());
    CU_TRY(d_W.alloc((size_t)d * d + d + 4));
    CU_TRY(d_x32.alloc(d));
    CU_TRY(d_c2s.alloc(1));
    CU_TRY(cudaMemsetAsync(d_c2s, 0, sizeof(int32_t), ctx->stream));
    CU_TRY(cudaMemsetAsync(d_score, 0, sizeof(float), ctx->stream));
    CU_TRY(cudaMemcpyAsync(d_x32, x32.data(), sizeof(float) * d, cudaMemcpyHostToDevice, ctx->stream));
    float *d_bias = d_W.p + (size_t)d * d, *d_coef = d_bias + d;
    LAUNCH(ctx, niw_prepare_kernel, 1, 128, (2 * (size_t)d * d + d) * sizeof(double), f, d_hp, d_ss, (const int32_t *)d_c2s, d_W.p, d_bias, d_coef);
    LAUNCH(ctx, niw_score_simt_kernel, dim3(1, 1), 128, ((size_t)d * d + d) * sizeof(float), (const float *)d_x32, (int)d, (const float *)d_W,
           (const float *)d_bias, (const float *)d_coef, d_score.p, (size_t)1, (size_t)0, (size_t)1);
    CU_TRY(cudaMemcpyAsync(score, d_score, sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
  } else {
    LAUNCH(ctx, value_op_kernel, 1, 32, 0, model->family, model->dim, op, d_hp, d_ss, d_x, d_score.p);
    if (op == 0) CU_TRY(cudaMemcpyAsync(score, d_score, sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    else CU_TRY(cudaMemcpyAsync(ss, d_ss, sizeof(double) * nss, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
  }
  return rc;
}

extern "C" MSB_API int msb_value_score(msb_ctx *ctx, const msb_model_desc *model, const double *hp, size_t nhp, const double *ss,
                               size_t nss, const void *value, const msb_runtime_type *vtype, float *score) {
  REQUIRE(score, "NULL argument");
  return value_op(ctx, model, 0, hp, nhp, const_cast<double *>(ss), nss, value, vtype, score);
}
extern "C" MSB_API int msb_value_add(msb_ctx *ctx, const msb_model_desc *model, const double *hp, size_t nhp, double *ss,
                             size_t nss, const void *value, const msb_runtime_type *vtype) {
  return value_op(ctx, model, 1, hp, nhp, ss, nss, value, vtype, nullptr);
}
extern "C" MSB_API int msb_value_remove(msb_ctx *ctx, const msb_model_desc *model, const double *hp, size_t nhp, double *ss,
                                size_t nss, const void *value, const msb_runtime_type *vtype) {
  return value_op(ctx, model, 2, hp, nhp, ss, nss, value, vtype, nullptr);
}

// ---- group::score_data of one group (models/base.hpp:28, distributions.hpp:287-291): the kernels of
// msb_state_score_likelihood on a one-feature, one-group layout
extern "C" MSB_API int msb_value_score_data(msb_ctx *ctx, const msb_model_desc *model, const double *hp, size_t nhp, const double *ss,
                                            size_t nss, float *score) {
  REQUIRE(ctx && model && hp && ss && score, "NULL argument");
  MSB_TRY(check_model(*model, 0));
  REQUIRE(nhp == hp_size(*model) && nss == ss_size(*model), "wrong dimension");
  CU_TRY(cudaSetDevice(ctx->device));
  std::vector<double> s(ss, ss + nss);
  ss_from_ref(*model, s);
  FeatDev f; memset(&f, 0, sizeof(f));
  f.family = model->family; f.dim = model->dim; f.ss_w = (uint32_t)nss;
  switch (model->family) {
    case MSB_FAMILY_GP: case MSB_FAMILY_BNB: f.kind = KIND_GP; break;
    case MSB_FAMILY_NICH: f.kind = KIND_NICH; break;
    case MSB_FAMILY_NIW: f.kind = KIND_NIW; break;
    case MSB_FAMILY_DM: f.kind = KIND_DM; break;
    default: f.kind = KIND_TABLE; break;
  }
  if (model->family == MSB_FAMILY_DD) for (size_t i = 0; i < nhp; i++) f.asum += hp[i];
  Scratch<double> d_buf;
  Scratch<FeatDev> d_f;
  Scratch<int32_t> d_c2s;
  CU_TRY(d_buf.alloc(nhp + nss + 1));
  CU_TRY(d_f.alloc(1));
  CU_TRY(d_c2s.alloc(1));
  double *d_hp = d_buf.p, *d_ss = d_buf.p + nhp, *d_out = d_ss + nss;
  CU_TRY(cudaMemcpyAsync(d_hp, hp, sizeof(double) * nhp, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(cudaMemcpyAsync(d_ss, s.data(), sizeof(double) * nss, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(cudaMemcpyAsync(d_f.p, &f, sizeof(FeatDev), cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(cudaMemsetAsync(d_c2s.p, 0, sizeof(int32_t), ctx->stream));
  if (model->family == MSB_FAMILY_NIW) {
    const size_t smem = ((size_t)f.dim * f.dim + f.dim) * sizeof(double);
    LAUNCH(ctx, niw_score_data_kernel, 1, 128, smem, f, 0, 1, (const double *)d_hp, (const double *)d_ss, (const int32_t *)d_c2s.p, d_out);
  } else {
    LAUNCH(ctx, score_data_kernel, 1, 32, 0, (const FeatDev *)d_f.p, 1, (const double *)d_hp, (const double *)d_ss, (const int32_t *)d_c2s.p, 1, d_out);
  }
  double r;
  CU_TRY(cudaMemcpyAsync(&r, d_out, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(cudaStreamSynchronize(ctx->stream));
  *score = (float)r;
  return MSB_OK;
}

// ---- group::sample_value (models/base.hpp:29, distributions.hpp:293-298) -----------------------------------------
static int launch_draws(msb_ctx *ctx, const msb_model_desc &m, int abi_repr, const double *d_hp, const double *d_ss, uint64_t seed,
                        uint64_t counter, size_t n, double *out) {
  if (m.family == MSB_FAMILY_DM) return fail(MSB_ERR_UNSUPPORTED, "multinomial sampling unimplemented");  // dm.cpp:100-111
  const size_t width = m.family == MSB_FAMILY_NIW ? m.dim : 1;
  Scratch<double> d_out;
  CU_TRY(d_out.alloc(n * width));
  const size_t smem = m.family == MSB_FAMILY_NIW ? ((size_t)m.dim * m.dim + m.dim) * sizeof(double) : 0;
  if (smem > 48 * 1024) CU_TRY(cudaFuncSetAttribute(sample_value_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const unsigned grid = (unsigned)std::min<size_t>(cdiv(n, 128), 148 * 4);
  LAUNCH(ctx, sample_value_kernel, grid, 128, smem, (int)m.family, m.dim, abi_repr, d_hp, d_ss, seed, counter, n, d_out.p);
  CU_TRY(cudaMemcpyAsync(out, d_out, sizeof(double) * n * width, cudaMemcpyDeviceToHost, ctx->stream));
  CU_TRY(cudaStreamSynchronize(ctx->stream));
  return MSB_OK;
}

extern "C" MSB_API int msb_value_sample(msb_ctx *ctx, const msb_model_desc *model, const double *hp, size_t nhp, const double *ss,
                                        size_t nss, uint64_t seed, uint64_t counter, size_t n, double *out) {
  REQUIRE(ctx && model && hp && ss && out, "NULL argument");
  MSB_TRY(check_model(*model, 0));
  REQUIRE(nhp == hp_size(*model) && nss == ss_size(*model), "wrong dimension");
  if (!n) return MSB_OK;
  CU_TRY(cudaSetDevice(ctx->device));
  Scratch<double> d_buf;
  CU_TRY(d_buf.alloc(nhp + nss));
  CU_TRY(cudaMemcpyAsync(d_buf.p, hp, sizeof(double) * nhp, cudaMemcpyHostToDevice, ctx->stream));
  CU_TRY(cudaMemcpyAsync(d_buf.p + nhp, ss, sizeof(double) * nss, cudaMemcpyHostToDevice, ctx->stream));
  return launch_draws(ctx, *model, 1, d_buf.p, d_buf.p + nhp, seed, counter, n, out);
}

extern "C" MSB_API int msb_state_sample_value(msb_state *st, size_t feature, size_t gid, uint64_t seed, uint64_t counter, size_t n,
                                              double *out) {
  REQUIRE(st && out, "NULL argument");
  REQUIRE(feature < st->D, "bad feature index");
  int slot;
  MSB_TRY(slot_of(st, gid, &slot));
  if (!n) return MSB_OK;
  msb_ctx *ctx = st->ctx;
  CU_TRY(cudaSetDevice(ctx->device));
  MSB_TRY(sync_small(st));
  const FeatDev &f = st->feats[feature];
  return launch_draws(ctx, st->models[feature], 0, st->d_hp + f.hp_off, st->d_ss + f.ss_off + (size_t)slot * f.ss_w, seed, counter, n, out);
}

#ifdef MSB_NIW_TRACE
extern "C" MSB_API int msb_debug_niw_trace(long long *out, int n) {
  return (int)cudaMemcpyFromSymbol(out, msb::niw_trace, (size_t)n * sizeof(long long));
}
#endif
