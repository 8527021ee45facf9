/*
 * mscope_b200.h -- C ABI of the B200-native hot path of microscopes-common.
 *
 * One shared library (common_b200/csrc/libmscope_b200.so) exports exactly the
 * symbols declared here.  No C++ or torch types cross this boundary: plain
 * pointers, sizes, opaque handles, int status codes + msb_last_error().
 *
 * What each entry point replaces in the reference (paths relative to the
 * reference tree, datamicroscopes/common):
 *
 *   msb_dataview_*        include/microscopes/common/recarray/dataview.hpp:194-217
 *                         (row_major_dataview ctor: data, mask, n, types) and
 *                         src/common/recarray/dataview.cpp:81-139 (row addressing)
 *   msb_runtime_type      include/microscopes/common/runtime_type.hpp:65-141
 *   msb_prim              include/microscopes/common/type_info.h:10-44
 *   msb_state_set/get_hp  models/distributions.hpp:128-144,165-181 (get_hp_mutator keys)
 *   msb_state_set/get_ss  models/distributions.hpp:146-160,183-199 (get_ss_mutator keys)
 *   msb_state_create_group / delete_group / groups / groupsize / empty_groups
 *                         common/group_manager.hpp:133-216
 *   msb_state_add_value / remove_value / score_value
 *                         common/entity_state.hpp:57-72 (which loop over
 *                         models/base.hpp:25-27 group::add_value/remove_value/score_value)
 *   msb_state_score_likelihood / score_assignment
 *                         common/entity_state.hpp:74-86, common/group_manager.hpp:250-272
 *   msb_state_score_rows  the same K x D loop of base.hpp:27 for a whole row range
 *   msb_sample_discrete_log
 *                         common/util.hpp:125-156 (scores_to_probs + sample_discrete)
 *   msb_state_sweep       one batched (synchronous, approximate) reassignment pass: score/sample/update
 *                         (SURVEY.md section 3b) against frozen suffstats
 *   msb_state_predict     mixturemodel's score_value (logsumexp of one inplace_score_value over the groups), the
 *                         responsibilities, and sample_post_pred's imputation of masked cells, for a row range
 *   msb_state_hp_gibbs    mixturemodel's grid feature-hp and cluster-hp kernels: one Gibbs step over gridded hypers
 *   msb_state_theta / redraw_empty
 *                         mixturemodel's theta kernel (slice sampling of bbnc's p) and the auxiliary-parameter
 *                         step of its assign_resample kernel (Neal's algorithm 8: the empty groups' p from the prior)
 *   msb_state_slice_hp    mixturemodel's slice hp kernel: one slice update of scalar feature hypers and of alpha
 *   msb_value_*           single-value group::score_value/add_value/remove_value/score_data/sample_value
 *                         (models/base.hpp:25-27), executed on the device
 *
 * Semantics notes
 *  - A masked (row, feature) cell contributes 0 to every score and nothing to
 *    the suffstats (the reference leaves this to the caller and asserts
 *    !anymasked, distributions.hpp:269,276,283).
 *  - Values cross the ABI as double (integers are exact); device storage is
 *    described in DESIGN.md.
 *  - All calls on one msb_ctx are ordered on its CUDA stream; calls returning
 *    host data synchronise that stream before returning.
 *  - There is no CPU fallback: without a usable CUDA device msb_ctx_create
 *    fails with MSB_ERR_CUDA.
 */
#ifndef MSCOPE_B200_H
#define MSCOPE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSB_ABI_VERSION 1

#if defined(__GNUC__)
#define MSB_API __attribute__((visibility("default")))
#else
#define MSB_API
#endif

typedef struct msb_ctx msb_ctx;           /* device + stream */
typedef struct msb_dataview msb_dataview; /* device copy of a row_major_dataview */
typedef struct msb_state msb_state;       /* K groups x D features of suffstats + hypers + assignments */

enum msb_status {
  MSB_OK = 0,
  MSB_ERR_INVALID = 1,     /* bad argument (the reference throws std::runtime_error) */
  MSB_ERR_CUDA = 2,        /* CUDA runtime error, see msb_last_error() */
  MSB_ERR_NOMEM = 3,
  MSB_ERR_UNSUPPORTED = 4,
  MSB_ERR_KEY = 5,         /* unknown hp/ss key: distributions.hpp:140,152 */
  MSB_ERR_STATE = 6        /* call not valid in the current state (e.g. entity already assigned) */
};

/* type_info.h:10-34, same order, same values */
enum msb_prim {
  MSB_TYPE_B = 0, MSB_TYPE_I8, MSB_TYPE_U8, MSB_TYPE_I16, MSB_TYPE_U16,
  MSB_TYPE_I32, MSB_TYPE_U32, MSB_TYPE_I64, MSB_TYPE_U64, MSB_TYPE_F32, MSB_TYPE_F64,
  MSB_TYPE_NELEMS
};

/* runtime_type.hpp:65-141: (primitive, n, vec) */
typedef struct msb_runtime_type {
  int32_t prim;  /* enum msb_prim */
  uint32_t n;    /* number of elements (1 for scalars) */
  int32_t vec;   /* 0 scalar, 1 vector */
} msb_runtime_type;

/* DISTRIB_FOR_EACH_DISTRIBUTION, distributions.hpp:58-64, + NormalInverseWishart (distributions.hpp:449-509) */
enum msb_family {
  MSB_FAMILY_BB = 0,   /* BetaBernoulli             hp: alpha beta            ss: heads tails */
  MSB_FAMILY_BNB = 1,  /* BetaNegativeBinomial      hp: alpha beta r          ss: count sum */
  MSB_FAMILY_GP = 2,   /* GammaPoisson              hp: alpha inv_beta        ss: count sum log_prod */
  MSB_FAMILY_NICH = 3, /* NormalInverseChiSq        hp: mu kappa sigmasq nu   ss: count mean count_times_variance */
  MSB_FAMILY_DD = 4,   /* DirichletDiscrete(dim)    hp: alphas[dim]           ss: count_sum counts[dim] */
  MSB_FAMILY_NIW = 5,  /* NormalInverseWishart(dim) hp: mu[dim] kappa psi[dim*dim] nu
                                                    ss: count sum_x[dim] sum_xxT[dim*dim] */
  MSB_FAMILY_BBNC = 6, /* BetaBernoulliNonConj (in-tree model, src/models/bbnc.cpp)
                                                    hp: alpha beta            ss: p heads tails
                          p is the group's own parameter, drawn from Beta(alpha, beta) when the group is created */
  MSB_FAMILY_DM = 7    /* DirichletMultinomial(dim) (in-tree model, src/models/dm.cpp): the value is a vector of dim counts
                                                    hp: alphas[dim]           ss: counts[dim] ratio */
};

typedef struct msb_model_desc {
  int32_t family; /* enum msb_family */
  uint32_t dim;   /* dd: number of categories (runtime, not capped at 128); niw: dimension; else 0 */
} msb_model_desc;

MSB_API const char *msb_last_error(void);
MSB_API int msb_abi_version(void);

/* ---- context ------------------------------------------------------------ */
/* stream: a cudaStream_t owned by the caller, or NULL to create a private one */
MSB_API int msb_ctx_create(int device, void *stream, msb_ctx **out);
MSB_API int msb_ctx_destroy(msb_ctx *ctx);
MSB_API int msb_ctx_synchronize(msb_ctx *ctx);
MSB_API void *msb_ctx_stream(msb_ctx *ctx);
/* number of kernels this library has launched on ctx since creation */
MSB_API int msb_ctx_launch_count(msb_ctx *ctx, uint64_t *out);
/* diagnostics (the reference's only profiling is common/timer.hpp:20-126 around its loop): enable != 0 puts a CUDA event
 * pair around every kernel launched on the context's stream from now on (earlier records are dropped); 0 stops.
 * msb_ctx_profile_read: one text line per kernel, "name\tlaunches\ttotal_ms\n"; *needed = bytes incl. the final 0. */
MSB_API int msb_ctx_profile(msb_ctx *ctx, int enable);
MSB_API int msb_ctx_profile_read(msb_ctx *ctx, char *buf, size_t cap, size_t *needed);

/* ---- dataview (recarray/dataview.hpp:194-217) --------------------------- */
/* data: n records, AoS, field offsets = running sum of type sizes
 *       (runtime_type.hpp:123-134); mask: n x sum(type.n) bytes of bool or NULL.
 * on_device != 0: data/mask are device pointers (no host copy). */
MSB_API int msb_dataview_create(msb_ctx *ctx, const void *data, const void *mask, size_t n,
                        const msb_runtime_type *types, size_t nfeatures, int on_device,
                        msb_dataview **out);
/* replace the records (and mask) of a host-created dataview in place: same n, same types.  Asynchronous on the
 * context's stream when the host buffers are pinned.  Follow with msb_state_refresh on the states bound to it. */
MSB_API int msb_dataview_upload(msb_dataview *dv, const void *data, const void *mask);
MSB_API int msb_dataview_destroy(msb_dataview *dv);
MSB_API int msb_dataview_size(const msb_dataview *dv, size_t *n);
MSB_API int msb_dataview_nfeatures(const msb_dataview *dv, size_t *d);
MSB_API int msb_dataview_rowsize(const msb_dataview *dv, size_t *rowsize, size_t *maskrowsize);
/* copy record idx (and its mask row, may be NULL) back to the host: dataview::get(idx) */
MSB_API int msb_dataview_get_row(msb_dataview *dv, size_t idx, void *row_out, void *mask_out);
/* row_major_dataview::permute / reset_permutation (src/common/recarray/dataview.cpp:141-151, util.hpp:85-94): a
 * Fisher-Yates order for iteration, drawn from the counter-based Philox stream (key = seed, counter = position).  While
 * a permutation is set, msb_dataview_get_row(idx) returns record pi[idx]; the stored records -- and the entity ids of a
 * state bound to the dataview -- keep their order, as in the reference.  msb_dataview_permutation reads pi back (the
 * identity when none is set): the order in which a caller visits the entities of a sequential pass. */
MSB_API int msb_dataview_permute(msb_dataview *dv, uint64_t seed);
MSB_API int msb_dataview_reset_permutation(msb_dataview *dv);
MSB_API int msb_dataview_permutation(const msb_dataview *dv, uint64_t *pi_out, size_t n);

/* ---- state -------------------------------------------------------------- */
MSB_API int msb_state_create(msb_ctx *ctx, const msb_model_desc *models, size_t nfeatures,
                     size_t max_groups, msb_state **out);
MSB_API int msb_state_destroy(msb_state *st);
/* converts the AoS records to columnar Value-typed device columns (the
 * runtime_cast of runtime_type.hpp:145-166 applied once per cell) and sizes the
 * assignment vector (all -1, group_manager.hpp:64-69). */
MSB_API int msb_state_bind(msb_state *st, msb_dataview *dv);
/* the bound dataview was re-uploaded (msb_dataview_upload): convert its records again, keeping the
 * assignments and the suffstats (the reference re-reads its borrowed host rows on every pass,
 * recarray/dataview.hpp:194-217; here the pass over host rows is upload + refresh + sweep). */
MSB_API int msb_state_refresh(msb_state *st);
/* optional, right after msb_dataview_upload: convert the new records on the copy stream into a second column
 * buffer while the compute stream is still sweeping the current one; the next msb_state_refresh then only swaps
 * the buffers (no conversion, no wait on the compute stream).  A no-op when the fused conversion does not apply. */
MSB_API int msb_state_prefetch(msb_state *st);

MSB_API int msb_state_set_hp(msb_state *st, size_t feature, const char *key, const double *v, size_t count);
MSB_API int msb_state_get_hp(msb_state *st, size_t feature, const char *key, double *v, size_t count);
MSB_API int msb_state_set_ss(msb_state *st, size_t feature, size_t gid, const char *key, const double *v, size_t count);
MSB_API int msb_state_get_ss(msb_state *st, size_t feature, size_t gid, const char *key, double *v, size_t count);
/* CRP hyperparameter "alpha": group_manager.hpp:107-131 */
MSB_API int msb_state_set_cluster_hp(msb_state *st, const char *key, double v);
MSB_API int msb_state_get_cluster_hp(msb_state *st, const char *key, double *v);

MSB_API int msb_state_nentities(msb_state *st, size_t *n);
MSB_API int msb_state_ngroups(msb_state *st, size_t *n);
MSB_API int msb_state_groups(msb_state *st, size_t *gids, size_t cap, size_t *n); /* ascending gid */
MSB_API int msb_state_empty_groups(msb_state *st, size_t *gids, size_t cap, size_t *n);
MSB_API int msb_state_groupsize(msb_state *st, size_t gid, size_t *count);
MSB_API int msb_state_create_group(msb_state *st, size_t *gid);
MSB_API int msb_state_delete_group(msb_state *st, size_t gid); /* must be empty */
/* deserialisation (group_manager.hpp:71-105): create the group with the identifier it had when it was saved */
MSB_API int msb_state_restore_group(msb_state *st, size_t gid);

/* assignments: gid per entity, -1 = unassigned (group_manager.hpp:133-137) */
MSB_API int msb_state_assignments(msb_state *st, int64_t *out, size_t n);
/* the same without waiting: gid translation on the compute stream, device -> host copy on the copy stream (it
 * overlaps the next sweep).  `out` (pinned) is valid once msb_state_assignments_wait returns. */
MSB_API int msb_state_assignments_async(msb_state *st, int64_t *out, size_t n);
MSB_API int msb_state_assignments_wait(msb_state *st);
/* bulk add_value of every currently unassigned entity whose gids[i] != -1 */
MSB_API int msb_state_add_values(msb_state *st, const int64_t *gids, size_t n);
/* the same, leaving the suffstat changes in the delta buffer (multi-GPU replica initialisation: all-reduce the
 * buffer of msb_state_delta_buffer, then msb_state_apply_deltas) */
MSB_API int msb_state_add_values_deferred(msb_state *st, const int64_t *gids, size_t n);

/* single-entity calls, entity_state.hpp:57-72 */
MSB_API int msb_state_add_value(msb_state *st, size_t gid, size_t eid);
MSB_API int msb_state_remove_value(msb_state *st, size_t eid, size_t *gid);
MSB_API int msb_state_score_value(msb_state *st, size_t eid, size_t *gids, float *scores, size_t cap, size_t *n);

/* batched scoring: scores[(i - row_lo) * ld + c] for column c <-> gids[c]
 * (all groups, ascending gid), = log(pseudocount) + sum_d score_value.
 * on_device != 0: scores is a device pointer. */
MSB_API int msb_state_score_rows(msb_state *st, size_t row_lo, size_t row_hi, float *scores, size_t ld,
                         int on_device, size_t *gids, size_t cap, size_t *ncols);

/* the same matrix in fp64 (host output): the closed forms in double straight from the resident suffstats,
 * no tables and no tensor cores -- the path the 1e-12 fp64 tolerance is checked on */
MSB_API int msb_state_score_rows_f64(msb_state *st, size_t row_lo, size_t row_hi, double *scores, size_t ld,
                             size_t *gids, size_t cap, size_t *ncols);

/* entity_state.hpp:74-86: score_likelihood(component, gid) = group::score_data (models/base.hpp:28), the log
 * marginal likelihood of the group's data under the component's hypers; and its sum over the groups per
 * component (per_feature[nfeatures], may be NULL) and over everything (total, may be NULL).  fp64 closed forms
 * on the device from the resident suffstats. */
MSB_API int msb_state_score_likelihood(msb_state *st, size_t feature, size_t gid, float *out);
MSB_API int msb_state_score_likelihood_all(msb_state *st, float *per_feature, size_t nfeatures, float *total);
/* group_manager.hpp:250-272: log CRP probability of the current partition; every entity must be assigned */
MSB_API int msb_state_score_assignment(msb_state *st, float *out);

/* util.hpp:125-156 on the device, one uniform per row; host pointers */
MSB_API int msb_sample_discrete_log(msb_ctx *ctx, const float *scores, size_t nrows, size_t k, size_t ld,
                            const float *uniforms, int32_t *out);
/* the uniform the sweep draws for (seed, global row id, sweep): Philox4x32-10 */
MSB_API int msb_philox_uniforms(msb_ctx *ctx, uint64_t seed, uint64_t sweep, uint64_t row_lo, size_t n, float *out);

/* y[i] = the sampler's exp (DESIGN.md, sampler contract) of x[i], evaluated on the device: the checker's own copy
 * must give the same bits */
MSB_API int msb_selftest_expf(msb_ctx *ctx, const float *x, size_t n, float *y);
/* device self-test of the sampler's packed exp (DESIGN.md, sampler contract): every float x in [-86, 0] through the
 * two-at-a-time form and through the scalar one; counts the results whose bits differ.  Must report 0. */
MSB_API int msb_selftest_expf2(msb_ctx *ctx, uint64_t *mismatches);
/* out[i] = 1 where the sampler's dart walk would skip a batch whose largest p has the biased exponent e[i], for a sum
 * acc[i] and a dart d[i] (DESIGN.md, sampler contract), else 0; evaluated on the device so that the host can check the
 * rule exactly */
MSB_API int msb_selftest_skip_rule(msb_ctx *ctx, const uint8_t *e, const float *acc, const float *d, size_t n, uint8_t *out);
/* device self-test of the sampler's division sequence (DESIGN.md, sampler contract), scalar and packed: n pseudo-random
 * operand sets, counts the results that differ from the IEEE division.  Must report 0. */
MSB_API int msb_selftest_division(msb_ctx *ctx, uint64_t seed, size_t n, uint64_t *mismatches);

typedef struct msb_sweep_opts {
  uint64_t seed;          /* Philox key */
  uint64_t sweep;         /* Philox counter word 2 */
  uint64_t row_id_offset; /* global id of local row 0 (multi-GPU row sharding) */
  const float *uniforms;  /* host array, one per row of [row_lo,row_hi), or NULL -> Philox */
  int32_t defer_apply;    /* 1: leave the suffstat deltas unapplied (all-reduce them, then msb_state_apply_deltas) */
  int32_t flags;          /* MSB_SWEEP_* */
} msb_sweep_opts;

/* enqueue the sweep on the context's stream and return without waiting; res->moved is then reported by
 * msb_state_sweep_wait (or read as 0).  Uniforms passed with an asynchronous sweep must stay valid until then. */
#define MSB_SWEEP_ASYNC 1

typedef struct msb_sweep_result {
  uint64_t rows;   /* rows processed */
  uint64_t moved;  /* rows whose group changed (local) */
  uint64_t units;  /* rows x groups x features scored */
} msb_sweep_result;

/* score rows [row_lo,row_hi) against the frozen suffstats, draw a group per row,
 * then apply remove_value(old)/add_value(new) for every row that moved.
 * This is a BATCHED (synchronous) pass, not the sequential kernel of entity_state.hpp:57-72: every row is scored
 * against suffstats and CRP counts that still contain the row itself, and all rows move at once, so the row's current
 * group is over-weighted (visibly for tiny groups) and the pass is an approximate Gibbs kernel -- it does not leave
 * the posterior exactly invariant (tests/test_gpu_parity.py puts the deviation on record on an enumerated example).
 * The exact chain is the per-entity sequence msb_state_remove_value -> msb_state_score_value -> draw ->
 * msb_state_add_value, which the same test file holds to the enumerated posterior. */
MSB_API int msb_state_sweep(msb_state *st, size_t row_lo, size_t row_hi, const msb_sweep_opts *opts,
                    msb_sweep_result *res);

/* waits for the stream and reports the last sweep (rows, moved, units) */
MSB_API int msb_state_sweep_wait(msb_state *st, msb_sweep_result *res);

/* ---- posterior predictive of rows [row_lo, row_hi) of the bound dataview (DESIGN.md section 4.9) ---------------------
 * The rows are scored against the current suffstats exactly as msb_state_score_rows scores them (columns c <-> gids[c],
 * ascending gid).  An assigned row's own contribution is part of the suffstats it is scored against: this is not a
 * leave-one-out predictive.  Held-out rows are bound unassigned (add_values with -1) and swept around.
 * For a row with fp32 scores s_c: m = max s_c, p_c = the sampler's exp(s_c - m), acc = sum p_c in fp64, column order.
 *   logp      log p(x_observed | state) = m + log(acc) - log(Z), Z = sum of the pseudocounts (fp64): with an empty group
 *             Z = N_assigned + alpha and logp is the DP posterior predictive (the existing clusters and a new one); with
 *             none it is the finite mixture over the present groups.  Replaces score_rows + the CRP normaliser + a host
 *             logsumexp (mixturemodel's score_value).
 *   resp      RN(p_c / (float)acc): bit for bit the probabilities the sampler walks (util.hpp:125-136).  Replaces
 *             score_rows + scores_to_probs on the host.
 *   map_gid   the gid of the first column with s_c = m.
 *   draw_gid  the sweep's draw for the row, uniform philox_u01(seed, row_id_offset + row, counter) or uniforms[row - row_lo].
 *             Replaces score_rows + msb_sample_discrete_log.
 *   values    [nrows][values_ld >= W], W = sum of the feature widths (dim for niw and dm, else 1), feature order: an
 *             observed cell is the value the device holds (the cast column value); a masked one (as the scorer sees it:
 *             a dd category outside [0, C), a niw vector with any masked element) is drawn from the posterior predictive
 *             of the row's drawn group, equal to msb_state_sample_value(d, gid, seed, counter * 2^40 + (row_id_offset +
 *             row) * D + d, n = 1).  Implies the draw.  counter >= 2^24 or (row_id_offset + row_hi) * D >= 2^40:
 *             MSB_ERR_INVALID.  A masked dm cell: MSB_ERR_UNSUPPORTED, "multinomial sampling unimplemented".  Replaces
 *             one msb_state_sample_value call per masked cell (sample_post_pred).
 * Every output is optional (NULL: not wanted).  Nothing of the state changes: assignments, suffstats, deltas, counts
 * and the sweep timing ring stay as they are; msb_state_last_scores describes the matrix of the last row chunk scored. */
typedef struct msb_predict_opts {
  uint64_t seed, counter, row_id_offset;
  const float *uniforms;              /* host, one per row of [row_lo, row_hi), or NULL -> Philox */
} msb_predict_opts;
typedef struct msb_predict_out {      /* host pointers; NULL = not wanted */
  double *logp;                       /* [nrows] */
  float *resp; size_t resp_ld;        /* [nrows][resp_ld >= K], column c <-> gids[c] */
  int64_t *map_gid;                   /* [nrows] */
  int64_t *draw_gid;                  /* [nrows] */
  double *values; size_t values_ld;   /* [nrows][values_ld >= W] */
} msb_predict_out;
MSB_API int msb_state_predict(msb_state *st, size_t row_lo, size_t row_hi, const msb_predict_opts *opts,
                              msb_predict_out *out, size_t *gids, size_t cap, size_t *ncols);

/* ---- hyperparameter inference on a grid (DESIGN.md section 4.10) -----------------------------------------------------
 * The mixturemodel runner's grid feature-hp kernel and its cluster-hp kernel, on the device.  Grids are registered once
 * and stay resident; the caller supplies the log hyperprior of every point (msb_state_slice_hp, below, evaluates its own).
 *
 * msb_state_set_hp_grid: feature `feature` gets npoints >= 1 grid points, each a complete hp vector in the flat layout
 * msb_value_score_data takes (nhp doubles; bb: alpha, beta; bnb: alpha, beta, r; gp: alpha, inv_beta; nich: mu, kappa,
 * sigmasq, nu; dd / dm: alphas[C]; niw: mu[d], kappa, psi[d*d], nu; bbnc: alpha, beta), points[npoints][nhp] row-major,
 * log_prior[npoints].  npoints == 0 removes the feature's grid.  msb_state_set_cluster_hp_grid: the same for the CRP
 * concentration, alphas[npoints] > 0.  A grid holds at most 65535 points.
 * Refused with MSB_ERR_INVALID, the state untouched: nhp that is not the family's, a non-finite value or log prior, an
 * alpha <= 0, more than 65535 points, a bnb point whose r differs from the feature's current r (bnb's score_data drops the r-dependent data
 * term, so only (alpha, beta) can be resampled).
 *
 * msb_state_hp_gibbs: one Gibbs step for every feature that has a grid, and for alpha if it has one.
 *   feature d:  L[g] = sum over every group column (ascending gid, empty groups included) of score_data(theta_g), fp64
 *               -- the set msb_state_score_likelihood_all sums, nothing rounded to float
 *   alpha:      L[g] = (#non-empty groups - 1) log alpha_g + lgamma(1 + alpha_g) - lgamma(n + alpha_g), n = assigned entities
 *   w_g = log_prior[g] + L[g], m = max w, p_g = exp(w_g - m) summed in index order in fp64; the draw is the first g whose
 *   running sum exceeds u * sum p, u a 53-bit uniform from philox4x32_10(key = seed, counter = (d, HP_TAG | counter))
 *   (alpha: d = D; its two first words a, b give u = ((a >> 5) 2^26 + (b >> 6)) 2^-53).  counter >= 2^32: MSB_ERR_INVALID.
 *   The sums over groups have a fixed order and no atomics: identical suffstats give identical weights and draws, so
 *   replicas after msb_state_allreduce_deltas draw the same hypers without a collective.
 *   The drawn points are written as msb_state_set_hp / msb_state_set_cluster_hp write them; assignments, suffstats,
 *   deltas and the sweep timing ring do not change.  Pending deferred deltas are not included (as for score_likelihood).
 *   A NaN or +inf weight (e.g. a niw psi that is not positive definite) or a grid whose weights are all -inf: MSB_ERR_INVALID,
 *   naming the feature and the point, and no hyper is changed.
 *   out (host pointers, each may be NULL): choice[D + 1] = the index drawn per feature, -1 without a grid, [D] = alpha's;
 *   logw[(D + 1) * logw_ld], logw_ld >= the largest grid: row d holds w_g of feature d (row D: alpha); rows without a
 *   grid are not written. */
MSB_API int msb_state_set_hp_grid(msb_state *st, size_t feature, const double *points, size_t npoints, size_t nhp,
                                  const double *log_prior);
MSB_API int msb_state_set_cluster_hp_grid(msb_state *st, const double *alphas, size_t npoints, const double *log_prior);
typedef struct msb_hp_gibbs_opts { uint64_t seed, counter; } msb_hp_gibbs_opts;
typedef struct msb_hp_gibbs_out {     /* host pointers; NULL = not wanted */
  int64_t *choice;                    /* [D + 1] */
  double *logw; size_t logw_ld;       /* [D + 1][logw_ld] */
} msb_hp_gibbs_out;
MSB_API int msb_state_hp_gibbs(msb_state *st, const msb_hp_gibbs_opts *opts, msb_hp_gibbs_out *out);

/* ---- non-conjugate parameters (DESIGN.md section 4.11) ---------------------------------------------------------------
 * msb_state_theta: one univariate slice-sampling update (Neal 2003: stepping out with width w, then shrinkage) of bbnc's
 * p in every group column, empty groups included, for every feature whose width widths[d] > 0 (0 leaves the feature
 * alone; nwidths must be D).  The target is the group's score_data with p substituted, the function
 * msb_state_score_likelihood evaluates.  An update that reaches the cap of 200 shrink steps (or 2^20 stepping-out
 * steps on a side) keeps its p and is counted in out->capped.  Draws come from
 * philox4x32_10(key = seed, counter = (counter << 32 | gid, THETA_TAG | d << 16 | block)): identical suffstats give
 * identical p, on every replica and after deserialisation.  Pending deferred deltas are not included.
 * msb_state_redraw_empty: every bbnc feature's p of every group whose resident count is 0 becomes a fresh
 * Beta(alpha, beta) draw x / (x + y) from the same packing under AUX_TAG; groups with members keep their p bit for bit.
 * Without a bbnc feature it does nothing.
 * Both write p into the suffstats (msb_state_get_ss "p") after the call's one synchronise, and only if no column was
 * refused.  Refused with MSB_ERR_INVALID, the state untouched: a width that is negative or not finite, a width > 0 on a
 * family other than bbnc, nwidths != D, counter >= 2^32, a feature index >= 65535 or a gid >= 2^32, a group whose
 * current p has a non-finite score_data (e.g. p set to 0 or 1 by hand), a Beta draw that underflowed (the message names
 * the feature and the gid). */
typedef struct msb_theta_opts {
  uint64_t seed, counter;
  const double *widths; size_t nwidths;   /* [D] slice widths; 0 = leave the feature alone */
} msb_theta_opts;
typedef struct msb_theta_out { size_t capped; } msb_theta_out;
MSB_API int msb_state_theta(msb_state *st, const msb_theta_opts *opts, msb_theta_out *out);
MSB_API int msb_state_redraw_empty(msb_state *st, uint64_t seed, uint64_t counter);

/* ---- slice sampling of continuous hypers (DESIGN.md section 4.12) ----------------------------------------------------
 * msb_state_slice_hp: the mixturemodel runner's slice hp kernel.  Each spec gets one univariate slice update (Neal 2003)
 * of one scalar hyper of one feature, or of the CRP concentration (feature == D, key "alpha").  The target is
 *   f(x) = log prior(x) + sum over every group column (ascending gid, empty groups included) of score_data with x
 *          substituted -- fp64, the set msb_state_hp_gibbs sums, with its fixed order and no atomics;
 *   alpha: log prior(x) + (#non-empty groups - 1) log x + lgamma(1 + x) - lgamma(n + x), n = assigned entities;
 * and -inf outside the key's support.  Sliceable keys and supports: bb, bbnc, bnb alpha, beta (0, inf) -- bbnc's given
 * the groups' p; gp alpha, inv_beta (0, inf); nich mu (real line), kappa, sigmasq, nu (0, inf); niw(d) kappa (0, inf),
 * nu (d - 1, inf); alpha (0, inf).
 * The update: y = f(x0) + log u; L = x0 - w u', R = L + w; bounded stepping out with m = 128 (L at most floor(m V)
 * times, R at most m - 1 - floor(m V) times, while f > y); then shrinkage, at most 200 steps.  A spec that reaches the cap
 * keeps x0 and is counted in out->capped.  A feature's specs run in the order given, each conditioning on the values its
 * predecessors drew; features and alpha are independent given the partition.  Spec j (its index among its feature's
 * specs) of feature d reads philox4x32_10(key = seed, counter = (counter << 32 | d, HPSL_TAG | j << 16 | block)),
 * HPSL_TAG = "HPSL" << 32: identical suffstats and hypers give identical values, on every replica.
 * After the call's one synchronise, and only if nothing was refused, every changed feature's hp vector is written as
 * msb_state_set_hp writes it and alpha as msb_state_set_cluster_hp does; assignments, suffstats, deltas and the sweep
 * timing ring do not change.  Pending deferred deltas are not included.
 * Refused, the state untouched, with MSB_ERR_KEY for a key the family does not have, MSB_ERR_UNSUPPORTED for a vector
 * key (dd / dm alphas, niw mu / psi: resample them on a grid with msb_state_set_hp_grid), and MSB_ERR_INVALID (the
 * message names the feature and the key) for: bnb's r (score_data drops its data term), a width <= 0 or not finite,
 * prior parameters outside the ranges below, the non-informative prior on anything but the alpha / beta of bb, bbnc or
 * bnb, a key twice for one feature, a feature index > D or >= 65535, counter >= 2^32, a current value where f is not
 * finite (e.g. outside the flat prior's interval, niw nu <= d - 1, a bbnc group whose p is 0 while it has heads), and
 * no groups. */
enum msb_hprior {                       /* the reference's in-tree hyperpriors, plus a flat interval */
  MSB_HPRIOR_FLAT = 0,                  /* a = lo, b = hi:      0 on (lo, hi), -inf outside; lo < hi, both finite */
  MSB_HPRIOR_EXPONENTIAL = 1,           /* a = rate > 0:        log(rate) - rate x for x >= 0, -inf below (log_exponential) */
  MSB_HPRIOR_NORMAL = 2,                /* a = mu, b = s2 > 0:  -0.5 log(2 pi s2) - (x - mu)^2 / (2 s2)   (log_normal) */
  MSB_HPRIOR_NONINFORMATIVE_BETA = 3    /* -2.5 log(alpha + beta), the partner at its current value (log_noninformative_beta_prior) */
};
typedef struct msb_slice_hp_spec {
  size_t feature;                       /* < D, or D for the CRP concentration (key "alpha") */
  const char *key;                      /* a scalar hp key of the family, as msb_state_set_hp names it */
  double width;                         /* slice width w > 0 */
  int32_t prior;                        /* enum msb_hprior */
  double a, b;                          /* the prior's parameters */
} msb_slice_hp_spec;
typedef struct msb_slice_hp_opts {
  uint64_t seed, counter;
  const msb_slice_hp_spec *specs; size_t nspecs;
} msb_slice_hp_opts;
typedef struct msb_slice_hp_out {
  size_t capped;                        /* specs that reached the shrink cap and kept their value */
  double *values;                       /* [nspecs] or NULL: each spec's value after the call */
} msb_slice_hp_out;
MSB_API int msb_state_slice_hp(msb_state *st, const msb_slice_hp_opts *opts, msb_slice_hp_out *out);

/* multi-GPU: flat fp64 buffer [group counts | per-feature suffstat deltas] on the device */
MSB_API int msb_state_delta_buffer(msb_state *st, double **dev_ptr, size_t *count);
MSB_API int msb_state_apply_deltas(msb_state *st);
/* count-valued states (every feature bb or dd): the same deltas as exact int32, half the bytes to all-reduce;
 * *dev_ptr is NULL for any other state.  After the all-reduce call
 * msb_state_delta_from_i32, then msb_state_apply_deltas. */
MSB_API int msb_state_delta_buffer_i32(msb_state *st, int32_t **dev_ptr, size_t *count);
MSB_API int msb_state_delta_from_i32(msb_state *st);
/* the resident suffstats themselves, same layout (replica initialisation: all-reduce, then apply_deltas) */
MSB_API int msb_state_suffstat_buffer(msb_state *st, double **dev_ptr, size_t *count);

/* ---- the exchange step (SURVEY.md section 8e: rows sharded over the GPUs of one box, suffstat replicas) ----------
 * NCCL is resolved at run time (the copy already loaded in the process, else libnccl.so.2); MSB_ERR_UNSUPPORTED
 * when there is none.  A host that already owns an ncclComm_t passes it as nccl_comm; the helpers below create
 * one from a 128-byte ncclUniqueId that rank 0 generates and hands to the other ranks by its own means. */
#define MSB_NCCL_UNIQUE_ID_BYTES 128
MSB_API int msb_nccl_version(int *version);
MSB_API int msb_nccl_unique_id(void *id128);
MSB_API int msb_nccl_comm_create(msb_ctx *ctx, int nranks, int rank, const void *id128, void **nccl_comm);
MSB_API int msb_nccl_comm_destroy(void *nccl_comm);
/* ncclAllReduce(sum) of the pending suffstat deltas on the context's stream, then msb_state_apply_deltas: every
 * replica ends with the same suffstats.  global_rows = rows over ALL ranks (every rank passes the same value);
 * count-valued states (every feature bb or dd) whose global row count fits int32 exchange exact int32 deltas,
 * anything else fp64.  nccl_comm is an ncclComm_t. */
MSB_API int msb_state_allreduce_deltas(msb_state *st, void *nccl_comm, uint64_t global_rows);
MSB_API int msb_state_last_allreduce_bytes(msb_state *st, size_t *bytes);

/* one pass over host rows in one call: msb_state_refresh -> msb_dataview_upload(next_data, next_mask) +
 * msb_state_prefetch (skipped when next_data is NULL) -> msb_state_sweep over every row, asynchronous
 * (-> msb_state_allreduce_deltas when nccl_comm is given) -> msb_state_assignments_wait + _async into assign_out
 * (pinned, n int64; skipped when NULL).  Returns without waiting for the compute stream. */
typedef struct msb_pass_opts {
  msb_sweep_opts sweep;
  const void *next_data;  /* host records of the NEXT pass (pinned), or NULL */
  const void *next_mask;
  int64_t *assign_out;    /* or NULL */
  void *nccl_comm;        /* ncclComm_t or NULL */
  uint64_t global_rows;   /* rows over all ranks (see msb_state_allreduce_deltas) */
} msb_pass_opts;
MSB_API int msb_state_pass(msb_state *st, const msb_pass_opts *opts, msb_sweep_result *res);

/* device pointer + leading dimension of the scores the last sweep/score wrote (diagnostics, tests) */
MSB_API int msb_state_last_scores(msb_state *st, float **dev_ptr, size_t *ld, size_t *nrows, size_t *ncols);
/* host copy of that matrix: out[r * ld_out + c], r < nrows, c < ncols */
MSB_API int msb_state_read_last_scores(msb_state *st, float *out, size_t ld_out);
/* events recorded around the kernels of the last sweep; ms per phase:
 * [0] table build, [1] score, [2] sample, [3] update, [4] apply */
MSB_API int msb_state_last_timings(msb_state *st, float *ms, size_t count);
/* the same for an earlier sweep: back = 0 is the last one, 1 the one before ... (a ring of 64 sweeps), so a
 * caller can enqueue many asynchronous sweeps and read every one's phase times afterwards */
MSB_API int msb_state_timings(msb_state *st, size_t back, float *ms, size_t count);

/* ---- single-value plugin calls (models/base.hpp:25-27), run on the device -- */
/* hp/ss are the flat field vectors in the order listed at enum msb_family */
MSB_API int msb_value_score(msb_ctx *ctx, const msb_model_desc *model, const double *hp, size_t nhp,
                    const double *ss, size_t nss, const void *value, const msb_runtime_type *vtype,
                    float *score);
MSB_API int msb_value_add(msb_ctx *ctx, const msb_model_desc *model, const double *hp, size_t nhp,
                  double *ss, size_t nss, const void *value, const msb_runtime_type *vtype);
MSB_API int msb_value_remove(msb_ctx *ctx, const msb_model_desc *model, const double *hp, size_t nhp,
                     double *ss, size_t nss, const void *value, const msb_runtime_type *vtype);
/* group::score_data (models/base.hpp:28; distributions.hpp:287-291; src/models/dm.cpp:79-95, bbnc.cpp:61-73): the marginal
 * likelihood of the data summarised by one group's suffstats */
MSB_API int msb_value_score_data(msb_ctx *ctx, const msb_model_desc *model, const double *hp, size_t nhp,
                         const double *ss, size_t nss, float *score);
/* group::sample_value (models/base.hpp:29; distributions.hpp:293-298; src/models/bbnc.cpp:75-83): n draws from the group's
 * posterior predictive into out[n * width] (width = dim for niw, else 1).  Draw i reads the Philox stream
 * (key = seed, counter = counter + i): the same (seed, counter) gives the same value on every device and in the checker.
 * dm: MSB_ERR_UNSUPPORTED, "multinomial sampling unimplemented", as src/models/dm.cpp:100-111 throws. */
MSB_API int msb_value_sample(msb_ctx *ctx, const msb_model_desc *model, const double *hp, size_t nhp,
                     const double *ss, size_t nss, uint64_t seed, uint64_t counter, size_t n, double *out);
/* the same from the suffstats resident in HBM: feature `feature` of group `gid` */
MSB_API int msb_state_sample_value(msb_state *st, size_t feature, size_t gid, uint64_t seed, uint64_t counter,
                           size_t n, double *out);
MSB_API size_t msb_model_hp_size(const msb_model_desc *model);
MSB_API size_t msb_model_ss_size(const msb_model_desc *model);

#ifdef __cplusplus
}
#endif
#endif /* MSCOPE_B200_H */
