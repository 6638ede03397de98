/* brie_b200 C ABI -- the drop-in boundary under the reference's Python object protocol.
 *
 * The reference (huangyh09/brie v2.3.0) has no FFI: `fit_BRIE_matrix`
 * (brie/models/model_wrap.py:138-146, 174-187) talks to `BRIE2`
 * (brie/models/model_TFProb.py:35-273) through Python attributes.  This ABI is
 * what a `BRIE2`-compatible class binds with ctypes instead of TensorFlow; each
 * entry names the reference code it replaces.  Plain pointers and sizes only.
 *
 * Conventions
 *  - All array pointers are DEVICE pointers unless the name ends in `_host`.
 *  - Every (cells, events) matrix is row-major with leading dimension `ld`
 *    floats (ld % 4 == 0, ld >= n_events); columns >= n_events are padding and
 *    must hold zero counts.  Same layout as the reference's (Nc, Ng) tensors.
 *    Counts are non-negative (read counts plus the pseudo-count); the step kernel relies on it.
 *  - `n_models` independent models (the full/base fit plus the LRT refits of
 *    model_wrap.py:155-187) are batched in every launch; model-major arrays are
 *    (n_models, ...).  Every model has its own design matrix Xc[model] (Nc, Kc):
 *    the columns that model uses (np.delete / np.append of model_wrap.py:161, 167),
 *    in model order, zero-padded to the common width Kc; bit k of
 *    `xc_mask[model]` says column k is in use (a padded column's Wc row stays 0).
 *  - The caller owns every buffer; the library allocates no persistent device
 *    memory.  Handles own small host structs only.
 *  - Every function returns 0 on success, <0 on error; brie_last_error() gives
 *    the message (thread-local).  No exceptions cross the ABI.
 *  - `stream` is a cudaStream_t passed as void*; all work is enqueued on it,
 *    nothing synchronises unless documented.
 */
#ifndef BRIE_B200_H
#define BRIE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BRIE_ABI_VERSION 12
#define BRIE_MAX_MODELS 32
#define BRIE_MAX_KC 16   /* widest design whose covariate contraction stays in registers / shared memory */
#define BRIE_MAX_KG 8
#define BRIE_MAX_K_WIDE 4096 /* any wider Kc or Kg up to this runs the wide form (see brie_fit_desc.Kc) */

#define BRIE_TARGET_ELBO 0
#define BRIE_TARGET_MARGINLIK 1

#define BRIE_OK 0
#define BRIE_ERR_ARG (-1)
#define BRIE_ERR_CUDA (-2)
#define BRIE_ERR_UNSUPPORTED (-3)

typedef struct brie_fit_desc {
  int64_t n_cells;        /* Nc  (model_TFProb.py:46) */
  int64_t n_events;       /* Ng of this shard (model_TFProb.py:47) */
  int64_t ld;             /* leading dimension of (cells, events) arrays */
  int64_t event_offset;   /* global index of local event 0 (RNG counters) */
  uint64_t seed;          /* noise / init key */
  int32_t n_models;       /* 1 + number of LRT refits batched (model_wrap.py:156) */
  int32_t Kc;             /* common (padded) width of the per-model Xc (model_TFProb.py:48): 0, 1, 2, 4, 8 or 16 for the
                             register-resident contraction; anything else up to BRIE_MAX_K_WIDE (or Kg > BRIE_MAX_KG)
                             selects the WIDE form: prior mean Xc Wc + Wg Xg^T and the gradients -Xc^T r, -r Xg are
                             GEMMs (cuBLAS SGEMM, fp32) around the fused kernel, which then reads / writes one extra
                             (cells, events) array each -- the reference accepts any Kc, Kg (:84-85, 121-126) */
  int32_t Kg;             /* columns of Xg (model_TFProb.py:49): 0, 4 or 8, or the wide form */
  int32_t mc_size;        /* MC_size (model_TFProb.py:130) */
  int32_t n_layers;       /* 2 or 3 count layers (model_TFProb.py:184) */
  int32_t has_efflen;     /* 0: binomial branch :162-167; 1: effLen branch :168-185 */
  int32_t cell_mode;      /* 0: intercept/sigma (1,Ng); 1: (Nc,1) (model_TFProb.py:53-60) */
  int32_t train_intercept;/* intercept is a Variable (model_TFProb.py:67-71) */
  int32_t train_sigma;    /* sigma_log is a Variable (model_TFProb.py:73-78) */
  int32_t trace_cap;      /* slots in loss_trace per model */
  int32_t target;         /* BRIE_TARGET_ELBO (model_TFProb.py:206-211) or BRIE_TARGET_MARGINLIK (:202-205) */
  int32_t rows_per_cta;   /* 0: library picks the cell rows per CTA; > 0: use this value (a gathered sub-fit of
                             brie_fit_bind's event_ids keeps its parent's value, so the float32 partial sums over
                             cells associate the same way and its results stay bit-identical to the parent's) */
  int32_t model_id[BRIE_MAX_MODELS]; /* RNG model word of each batched model */
  uint32_t xc_mask[BRIE_MAX_MODELS]; /* bit k set: column k of Xc[model] is a real covariate (Kc <= BRIE_MAX_KC) */
  int32_t xc_width[BRIE_MAX_MODELS]; /* wide form: columns [0, xc_width[model]) of Xc[model] are real covariates */
} brie_fit_desc;

typedef struct brie_fit_sizes {
  size_t scratch_bytes;     /* brie_fit_buffers.scratch */
  size_t adam_small_floats; /* brie_fit_buffers.adam_small */
  int32_t rows_per_cta;
  int32_t n_row_chunks;
  int32_t n_col_tiles;
  int32_t reserved;
} brie_fit_sizes;

typedef struct brie_fit_buffers {
  const float* counts[3]; /* (Nc, ld) isoform1, isoform2, ambiguous (NULL if n_layers == 2),
                             pseudo-count already applied (model_wrap.py:113-117) */
  const float* efflen3;   /* (3, ld): columns 0, 4, 5 of varm['effLen'] (model_TFProb.py:176); NULL if !has_efflen */
  const float* Xc;        /* (M, Nc, Kc) row-major: per-model design matrices (model_TFProb.py:220) */
  const float* Xg;        /* (Ng, Kg) row-major (model_TFProb.py:221) */
  float* Z_loc;           /* (M, Nc, ld)  (model_TFProb.py:80) */
  float* Z_std_log;       /* (M, Nc, ld)  (model_TFProb.py:82) */
  float* adam_Z;          /* (4, M, Nc, ld): m(Z_loc), v(Z_loc), m(Z_std_log), v(Z_std_log) */
  float* Wc;              /* (M, Kc, ld)  (model_TFProb.py:84) */
  float* intercept;       /* (M, ld) or, cell_mode, (M, Nc)  (model_TFProb.py:68) */
  float* sigma_log;       /* same shape as intercept (model_TFProb.py:74) */
  float* Wg;              /* (M, Nc, Kg)  (model_TFProb.py:85) */
  float* adam_small;      /* Adam moments of Wc, intercept, sigma_log, Wg */
  const uint8_t* active;  /* (M, ld): 1 = this model still optimises this event */
  float* loss_trace;      /* (M, trace_cap, ld): per-step per-event loss (pre-update) */
  void* scratch;
  /* Gathered sub-fit (the convergence-extension rounds of model_TFProb.py:250-258 on the events whose reference
   * batch has not converged yet, physically compacted so that every 32-byte sector moved holds active events).
   * Each model then has its OWN column -> event map and therefore its own gathered count / length tiles:
   *  event_ids (M, ld) int32: global event id of every column (the RNG counter word), NULL = event_offset + column;
   *  counts_model_stride: floats between the count tiles of consecutive models, 0 = all models share one tile;
   *  efflen_model_stride: likewise for efflen3 ((3, ld) per model), 0 = shared.
   * Only the step entry points work on such a fit (Kg = 0, cell_mode = 0, target ELBO); results go back with
   * brie_scatter_events.  A sub-fit that steps on packed count codes (brie_fit_set_count_codes) may leave counts[]
   * all NULL. */
  const int32_t* event_ids;
  int64_t counts_model_stride;
  int64_t efflen_model_stride;
} brie_fit_buffers;

typedef struct brie_fit brie_fit; /* opaque */

int brie_abi_version(void);
const char* brie_last_error(void);

/* Replaces BRIE2.__init__ bookkeeping (model_TFProb.py:42-85): validates the
 * description, picks the launch geometry and reports scratch sizes. */
int brie_fit_create(const brie_fit_desc* desc, brie_fit** out);
int brie_fit_destroy(brie_fit* fit);
int brie_fit_get_sizes(const brie_fit* fit, brie_fit_sizes* out);
int brie_fit_bind(brie_fit* fit, const brie_fit_buffers* buffers);

/* Replaces Model_init (model_TFProb.py:12-31): Z_loc ~ N(0,1), Z_std_log ~ N(0,1),
 * Wc ~ N(0,1) on rows in use (row index = position among the model's own columns),
 * Wg ~ N(0,1), intercept ~ N(0,1) if trained else `intercept_const`,
 * sigma_log = log(sigma_const) (1 -> 0).  Counter-based, see brie_philox.h. */
int brie_fit_init_params(brie_fit* fit, float intercept_const, float sigma_const, void* stream);

/* Replaces `tf.optimizers.Adam(learning_rate=lr)` (model_TFProb.py:237): zero
 * all Adam moments and reset the step count t of every model. */
int brie_fit_begin_stage(brie_fit* fit, float lr, void* stream);

/* Continue an optimiser that already took `adam_t` steps in its stage (the extension rounds keep using the last
 * stage's optimizer, model_TFProb.py:255): like brie_fit_begin_stage but the Adam moments are left as they are,
 * the Adam step count starts at adam_t and the RNG step word at global_step.  brie_fit_get_step reads both. */
int brie_fit_resume_stage(brie_fit* fit, float lr, int64_t adam_t, uint32_t global_step);
int brie_fit_get_step(const brie_fit* fit, int64_t* adam_t, uint32_t* global_step);

/* Replaces `tfp.math.minimize(loss_fn, num_steps, optimizer)` (model_TFProb.py:239,
 * 255): n_steps fused ELBO forward + backward + Adam steps (get_loss :194-211,
 * logLik_MC :130-191, Z_prior :118-127, constraint clips :68-69, :80-81).
 * If trace_slot0 >= 0 the pre-update per-event loss of step i is written to
 * loss_trace[:, trace_slot0 + i, :]; if < 0 the loss is not evaluated. */
int brie_fit_run_steps(brie_fit* fit, int32_t n_steps, int32_t trace_slot0, void* stream);

/* Packed count codes for the fused step kernel (brie_encode_counts).  From now on the step kernel reads one 32-bit
 * code word per element from `codes` ((Nc, ld) per model, codes_model_stride words apart, 0 = one tile shared by all
 * models, as counts_model_stride) and decodes the counts of elements with reads from dict (DEVICE, (3, 256) floats),
 * instead of streaming the float32 count tiles: 4 B of counts per element and step instead of 12 (8 with two layers).
 * The decoded values are the tiles' own bit patterns, so results are bit-identical.  Everything else that reads
 * counts (loss_gene, element terms, target marginLik) keeps reading the float32 tiles.  codes = NULL returns to the
 * float32 tiles.  Both arrays must stay valid while set. */
int brie_fit_set_count_codes(brie_fit* fit, const uint32_t* codes, int64_t codes_model_stride, const float* dict);

/* Column compaction for the convergence-extension rounds (model_TFProb.py:250-258).  The
 * reference extends each event batch on its own (model_wrap.py:241-260); batches that have
 * converged stay frozen through `active`.  Once most are frozen the step kernel can visit only
 * the 8-event column blocks (one 32-byte sector of every f32 array) that still hold an active
 * event: blk_ids (DEVICE, (n_models, blk_stride) int32, ascending block indices col / 8) lists
 * them per model, n_blk_host (HOST, n_models) their counts.  Results are bit-identical to the
 * uncompacted step.  blk_ids = NULL restores the dense walk.  The list must cover every event
 * with active = 1 and must stay valid until replaced.  Needs ld % 8 == 0, Kg = 0, cell_mode = 0,
 * target ELBO. */
int brie_fit_set_active_blocks(brie_fit* fit, const int32_t* blk_ids, int64_t blk_stride,
                               const int32_t* n_blk_host);

/* Which models the step entry points step: bit m of `mask` set = model m steps (brie_fit_create starts with all
 * models).  A step leaves a cleared model alone: its fused or marginLik step CTAs, wide-form GEMMs, per-cell reduce
 * and per-cell Adam update are skipped.  A shared-parameter fit (Kg > 0 or cell_mode) clears the bit of
 * every model whose convergence-extension rounds (model_TFProb.py:250-258) have ended: its `active` flags keep its
 * per-event state put, but only the mask keeps Wg and a per-cell intercept / sigma_log put.  Refuses bits at or
 * beyond n_models and an open split step. */
int brie_fit_set_model_mask(brie_fit* fit, uint32_t mask);

/* All-reduce hook for event-sharded fits with shared per-cell parameters
 * (Kg > 0 or cell_mode).  brie_fit_step_phase runs ONE step in two halves:
 * phase 0 leaves the summed per-cell gradients in cell_grad (M, Nc, n_cell_acc)
 * (pointer returned by brie_fit_cell_grad) for the caller to all-reduce; phase 1
 * applies Adam to Wg / per-cell intercept / sigma_log. */
int brie_fit_step_phase(brie_fit* fit, int32_t phase, int32_t trace_slot, void* stream);
int brie_fit_cell_grad(brie_fit* fit, float** ptr, int64_t* n_floats);

/* Event-sharded fits with shared per-cell parameters WITHOUT a host round trip per step: a
 * communicator spanning the ranks that hold the event shards of one fit (one process per GPU).
 * The reference has no counterpart (single process); the exchange follows from its model: Wg is
 * (Nc, Kg), shared by all events (model_TFProb.py:85, 124-125), and with intercept_mode 'cell'
 * so are intercept and sigma_log (:53-55), while events are the shard axis (model_wrap.py:241-260).
 *  brie_comm_unique_id : rank 0 fills 128 bytes (ncclUniqueId) that the caller ships to every rank;
 *  brie_comm_create    : collective over all `world` ranks, on the calling thread's current device;
 *  brie_fit_set_comm   : from now on brie_fit_run_steps all-reduces (sum) the per-cell gradient
 *                        buffer (M, Nc, Kg + 2 * cell_mode) with NCCL on `stream` between the fused
 *                        step kernel and the per-cell Adam update; NULL detaches.
 *  brie_comm_allreduce_f32 / _f64 : in-place sum on `stream` (group loss traces, tests).
 * NCCL is bound at run time (dlopen of libnccl.so.2, preferring the copy already in the process);
 * without it these return BRIE_ERR_UNSUPPORTED and brie_comm_nccl_version() returns 0. */
typedef struct brie_comm brie_comm; /* opaque */
int brie_comm_nccl_version(void);
int brie_comm_unique_id(void* id_host /* 128 bytes */);
int brie_comm_create(const void* id_host, int32_t rank, int32_t world, brie_comm** out);
int brie_comm_destroy(brie_comm* comm);
int brie_comm_allreduce_f32(brie_comm* comm, float* buf, int64_t n, void* stream);
int brie_comm_allreduce_f64(brie_comm* comm, double* buf, int64_t n, void* stream);
int64_t brie_comm_allreduce_count(const brie_comm* comm);
int brie_fit_set_comm(brie_fit* fit, brie_comm* comm);

/* Replaces the 500x `get_loss(axis=0)` averaging (model_TFProb.py:261-264):
 * loss_gene[m, g] = sum_c KL - mean over n_eval evaluations, each with `mc_size` fresh-noise
 * samples, of sum_c loglik.  The reference's loop calls get_loss without the fit's **kwargs,
 * so its evaluations use logLik_MC's default MC_size = 1 (model_TFProb.py:130), not --MCsize. */
int brie_fit_eval_loss_gene(brie_fit* fit, int32_t n_eval, int32_t mc_size, float* loss_gene /* (M, ld) */,
                            void* stream);

/* Replaces the Psi / Psi95CI / Z_std properties (model_TFProb.py:88-106) for one model. */
int brie_fit_posterior(brie_fit* fit, int32_t model, float* Psi, float* Psi95CI, float* Z_std,
                       void* stream);

/* Observed information of model `model`'s per-event regression parameters from its fitted posterior (no reference
 * counterpart; DESIGN §2.2).  Given W, b and sigma the exact posterior of Z factorises over (cell, event), so Louis'
 * missing-information formula gives, per event g,
 *   I_g = sum_c w_cg x~_c x~_c^T,  w_cg = max(sigma^2 - s_cg^2, 0) / sigma^4,  s_cg = exp(Z_std_log[model, c, g]),
 * sigma = exp(sigma_log) of the event (or, cell_mode, of the cell).  x~_c is the model's design row: its Xc columns in
 * mask order (xc_mask bits, or the first xc_width columns of the wide form: the order of its Wc rows), then a 1 when
 * the intercept is per-event and trained (cell_mode 0, train_intercept 1).  Wg and a per-cell intercept / sigma are
 * known offsets.  K~ = that width.
 *  brie_fit_wald_sizes : scratch bytes and K~ of `model`;
 *  brie_fit_wald_info  : info (DEVICE, (n_events, K~ (K~ + 1) / 2) float64, row-major) receives the upper triangle
 *                        of each I_g, pairs (k <= l) row-major over x~; scratch needs the size above.  Reads only
 *                        the step entry points' state (Z_std_log, sigma_log, Xc), so it works on a fit whose
 *                        extension rounds ran on gathered sub-fits (not on a sub-fit itself).  Deterministic: no
 *                        atomics, repeated calls give bit-identical output.  Target ELBO only (marginLik trains no
 *                        posterior). */
int brie_fit_wald_sizes(const brie_fit* fit, int32_t model, size_t* scratch_bytes, int32_t* k_tilde);
int brie_fit_wald_info(brie_fit* fit, int32_t model, double* info, void* scratch, void* stream);

/* Score-test parts of n_cand candidate cell covariates against model `model` as the null model (no reference
 * counterpart; DESIGN §2.3), from its fitted posterior with no refit.  With x~_c as above, the prior mean m_cg, sigma
 * the event's (or, cell_mode, the cell's) and x_cj = X[c * ldx + j]:
 *   r_cg = (Z_loc[model, c, g] - m_cg) / sigma^2,   w_cg = max(sigma^2 - s_cg^2, 0) / sigma^4   (as in the Wald pass)
 *   U[g, j] = sum_c x_cj r_cg,   A[g, j] = sum_c w_cg x_cj^2,   B[g, j, k] = sum_c w_cg x_cj x~_ck,
 *   Utheta[g, k] = sum_c x~_ck r_cg
 * in float64 (the prior mean too).  With I_g of brie_fit_wald_info the efficient information of candidate j is
 * A - B I^-1 B^T and its efficient score U - B I^-1 Utheta.
 *  brie_fit_score_sizes : scratch bytes and K~ of `model` for n_cand candidates (the scratch grows with n_cand:
 *                         up to 64 row chunks x n_cand (K~ + 2) x ld doubles; callers split the candidates);
 *  brie_fit_score_parts : X (DEVICE, (n_cells, ldx) float32, ldx >= n_cand); U, A (DEVICE, (n_events, n_cand)),
 *                         B (DEVICE, (n_events, n_cand, K~)), Utheta (DEVICE, (n_events, K~)), all float64 and
 *                         8-byte aligned (B and Utheta may be NULL when K~ = 0).  The row chunks are the Wald pass's,
 *                         a function of n_cells alone; no atomics: repeated calls, event chunks and shards give the
 *                         same bits.  Works on a fit whose extension rounds ran on gathered sub-fits (not on a
 *                         sub-fit itself).  Target ELBO only. */
int brie_fit_score_sizes(const brie_fit* fit, int32_t model, int32_t n_cand, size_t* scratch_bytes, int32_t* k_tilde);
int brie_fit_score_parts(brie_fit* fit, int32_t model, const float* X, int32_t n_cand, int64_t ldx, double* U,
                         double* A, double* B, double* Utheta, void* scratch, void* stream);

/* Cross terms of the joint score test of groups of candidates (DESIGN §2.4), from model `model`'s fitted posterior:
 *   out[g, p] = sum_c w_cg x_c,j x_c,j'   for pair p = (j, j') = (pairs[2 p], pairs[2 p + 1])
 * with w_cg the Louis weight of brie_fit_wald_info, in float64.  The pairs j = j' are brie_fit_score_parts' A; the
 * joint efficient information of a group G is V_GG = A_GG - B_G I^-1 B_G^T.
 *  brie_fit_score_cross_sizes : scratch bytes of `model` for n_pairs pairs (up to 64 row chunks x n_pairs x ld
 *                               doubles, plus the pair table; callers split the pairs);
 *  brie_fit_score_cross       : X (DEVICE, (n_cells, ldx) float32), pairs (HOST, (n_pairs, 2) int32, each
 *                               0 <= j < j' < ldx, copied into the scratch with cudaMemcpyAsync on `stream`), out
 *                               (DEVICE, (n_events, n_pairs) float64).  out and scratch 8-byte aligned.  The row chunks
 *                               are the Wald pass's, a function of n_cells alone; no atomics: repeated calls, pair
 *                               blocks, event chunks and shards give the same bits.
 * Both refuse what brie_fit_score_parts refuses (a null or unbound fit, a model out of range, a gathered sub-fit,
 * target marginLik) and n_pairs <= 0; brie_fit_score_cross also refuses pairs out of range, before any launch. */
int brie_fit_score_cross_sizes(const brie_fit* fit, int32_t model, int32_t n_pairs, size_t* scratch_bytes);
int brie_fit_score_cross(brie_fit* fit, int32_t model, const float* X, int64_t ldx, const int32_t* pairs,
                         int32_t n_pairs, double* out, void* scratch, void* stream);

/* Replaces the tensors the public model API returns for one model (BRIE2.logLik_MC model_TFProb.py:130-191,
 * Z_prior :118-127, the KL of get_loss :208), as dense (Nc, ld) arrays; any output may be NULL.
 *   loglik     : mean over mc_size samples of the element's log-likelihood, z ~ N(Z_loc, Z_std) (:159, :191);
 *                margin != 0: z ~ the prior, log-mean-exp over the samples (:157, :189)
 *   kl         : KL(N(Z_loc, Z_std) || N(prior mean, sigma))
 *   prior_mean : Xc Wc + Wg Xg^T + intercept
 * c1, c2, c3 are the caller's count tiles ((Nc, ld), c3 may be NULL) -- get_loss / logLik_MC take count_layers
 * as an argument, not the fitted ones.  Noise: counter (event, cell, noise_step) of the EVAL phase. */
int brie_fit_element_terms(brie_fit* fit, int32_t model, const float* c1, const float* c2, const float* c3,
                           int32_t mc_size, uint32_t noise_step, int32_t margin, float* loglik, float* kl,
                           float* prior_mean, void* stream);

/* Replaces `tfd.Multinomial(total_counts, probs=Phi).sample()` of brie.models.simulator (simulator.py:54-73):
 * (c1, c2, c3)[c, g] ~ Multinomial(total[c, g], [psi L1, (1 - psi) L2, L3] / sum) with total, psi (Nc, ld) device
 * arrays (total holds integral values), efflen3 (3, ld) or NULL (L = 1, 1, 0), c3 may be NULL. */
int brie_resample_counts(uint64_t seed, int64_t n_cells, int64_t n_events, int64_t ld, int64_t event_offset,
                         const float* total, const float* psi, const float* efflen3, float* c1, float* c2, float* c3,
                         void* stream);

/* Sum the per-event loss trace over reference batches (model_wrap.py:241-246:
 * group g covers events [g*group_size, (g+1)*group_size) in GLOBAL event index):
 * out[m, grp, slot] for slot in [0, n_slots).  Feeds the convergence rule of
 * model_TFProb.py:250-251 and uns['brie_losses']. */
int brie_fit_group_trace(brie_fit* fit, int32_t n_slots, int64_t group_size, int64_t n_groups,
                         double* out /* (M, n_groups, n_slots) */, void* stream);

/* Total kernels launched by this handle so far (bench.py's gpu_launches). */
int64_t brie_fit_launch_count(const brie_fit* fit);

/* Measurement aid (no reference counterpart): bracket the next `capacity` launches of
 * the fused step kernel with CUDA events on the launching stream; _time_ms waits for
 * them, returns their summed duration and count, and re-arms the same capacity. */
int brie_fit_kernel_timing(brie_fit* fit, int32_t capacity);
int brie_fit_kernel_time_ms(brie_fit* fit, double* total_ms, int32_t* n_launches);

/* Noise dumps (tests): eps[s, r, c] for rows [0,n_rows), global cols col_offset + [0,n_cols). */
int brie_philox_normals_host(uint64_t seed, uint32_t phase, uint32_t model, uint32_t step,
                             int32_t n_samples, int64_t n_rows, int64_t n_cols, int64_t col_offset,
                             float* out_host);
int brie_philox_normals_device(uint64_t seed, uint32_t phase, uint32_t model, uint32_t step,
                               int32_t n_samples, int64_t n_rows, int64_t n_cols, int64_t col_offset,
                               float* out, void* stream);

/* Synthetic counts on the device, following brie/models/simulator.py:54-73 and
 * simulator/simuPSI.py:129-130 (bench.py workloads too large for host RAM):
 * z = logit_mean[g] + Xc[c,:] Wc[:,g] + logit_sd[g] N(0,1) clipped to +-9, psi = sigmoid(z),
 * n ~ Poisson(lam[g]) Bernoulli(cdr[g]), (c1,c2,c3) ~ Multinomial(n, [psi L1, (1-psi) L2, L3] / sum),
 * then the pseudo-count of model_wrap.py:113-117.  Per-event vectors have ld entries, Wc is
 * (Kc, ld), efflen3 (3, ld) or NULL (L = 1,1,0), c3 may be NULL; outputs are (n_cells, ld). */
int brie_simulate_counts(uint64_t seed, int64_t n_cells, int64_t n_events, int64_t ld,
                         int64_t event_offset, const float* logit_mean, const float* logit_sd,
                         const float* Xc, const float* Wc, int32_t Kc, const float* efflen3,
                         const float* lam, const float* cdr, float pseudo_count, float* c1, float* c2,
                         float* c3, void* stream);

/* ---- count ingest in front of the fit (SURVEY f1) --------------------------------------
 * Replaces the host densification of sparse layers (`data[i].toarray()`,
 * model_wrap.py:108-111; model_TFProb.py:135-137): scatter a CSC slab (events = columns,
 * the format brie-count writes, io_utils.py:107) or a CSR matrix into the dense
 * (n_cells, ld) float32 tile the fit reads.  `out` is zero-filled first; duplicate
 * entries sum (as toarray() does); indices outside the tile are ignored.
 *  csc: colptr has n_events + 1 entries relative to rows/vals (colptr[0] == 0 for a slab
 *       cut out of a larger matrix), rows are cell ids.
 *  csr: rowptr has n_cells + 1 entries, cols are GLOBAL event ids; the tile keeps
 *       events [event_begin, event_begin + n_events).
 * rows/cols/vals may be NULL for an empty layer. */
int brie_ingest_csc(int64_t n_cells, int64_t n_events, int64_t ld, const int64_t* colptr,
                    const int32_t* rows, const float* vals, float* out, void* stream);
int brie_ingest_csr(int64_t n_cells, int64_t event_begin, int64_t n_events, int64_t ld,
                    const int64_t* rowptr, const int32_t* cols, const float* vals, float* out,
                    void* stream);

/* Replaces the pseudo-count of model_wrap.py:113-117, in place on the device tiles:
 * where c1 + c2 > 0 (float32), c1 += pseudo_count and c2 += pseudo_count. */
int brie_add_pseudo_count(int64_t n_cells, int64_t ld, float pseudo_count, float* c1, float* c2,
                          void* stream);

/* Replaces the dense float64 accumulation of filter_genes (preprocessing.py:38-61): per event
 * stats[0..2, g] = column sums of c1, c2, c3 (c3 may be NULL), stats[3, g] = number of cells
 * with c1 + c2 > 0, stats[4, g] = number of cells with c1 + c2 + c3 > 0; all float64, (5, ld).
 * `scratch` needs brie_gene_stats_scratch_bytes(n_cells, ld) bytes.  Deterministic. */
size_t brie_gene_stats_scratch_bytes(int64_t n_cells, int64_t ld);
int brie_gene_stats(int64_t n_cells, int64_t ld, const float* c1, const float* c2, const float* c3,
                    double* stats, void* scratch, void* stream);

/* Dictionary coding of the count tiles for brie_fit_set_count_codes.  Read counts (plus the pseudo-count) take few
 * distinct values, so each element's layers fit one 32-bit word: byte l (l = 0, 1, 2) is the index of layer l's
 * value in dict[l * 256 + .], byte 3 is 0.  dict[l * 256] = 0.0f (+0 and -0 both map to it), so a word is non-zero
 * iff c1 + c2 + c3 > 0; the other entries are the layer's distinct non-zero values in ascending order, bit for bit.
 * One pass over the (n_cells, ld) tiles (c3 may be NULL: its byte is 0) collects each layer's values, a second
 * writes the code words.  n_values (DEVICE, 3 int32) receives the number of distinct non-zero values per layer; a
 * value above 255 means the tiles cannot be coded -- more than 255 distinct non-zero values in a layer, or a
 * negative or NaN count -- and then `codes` is left unwritten.  dict: (3, 256) floats.  scratch needs
 * brie_encode_counts_scratch_bytes() bytes.  Nothing synchronises: read n_values after the stream. */
size_t brie_encode_counts_scratch_bytes(void);
int brie_encode_counts(int64_t n_cells, int64_t ld, const float* c1, const float* c2, const float* c3,
                       uint32_t* codes, float* dict, int32_t* n_values, void* scratch, void* stream);

/* Column gather of a dense tile (`adata._inplace_subset_var`, preprocessing.py:63, without a
 * host round trip): out[r, j] = in[r, src[j]] for j < n_out, zero padding up to ld_out. */
int brie_gather_events(int64_t n_cells, int64_t ld_in, const float* in, const int64_t* src,
                       int64_t n_out, int64_t ld_out, float* out, void* stream);

/* Inverse of brie_gather_events: out[r, dst[j]] = in[r, j] for j < n_in; other columns of `out` are untouched.
 * dst entries must be distinct. */
int brie_scatter_events(int64_t n_cells, int64_t ld_in, const float* in, const int64_t* dst,
                        int64_t n_in, int64_t ld_out, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BRIE_B200_H */
