/*
 * ncf_b200.h — C ABI of the B200-native NCF training / leave-one-out evaluation hot path.
 *
 * The reference (YonkaMayonkaZ/NCF) has no FFI: its hot path is stock PyTorch ops driven
 * from Python (SURVEY.md §8b).  This header is the boundary a maintainer would bind instead:
 * plain pointers and sizes, no torch types.  Every entry point cites the reference code it
 * replaces (paths relative to the reference root).
 *
 * Conventions
 *  - All pointers are DEVICE pointers unless the name ends in _host.  The library never
 *    allocates persistent memory and never frees caller memory; scratch comes from the
 *    caller through (workspace, workspace_bytes) sized by the *_workspace_bytes queries.
 *  - Every call is asynchronous on `stream` (a cudaStream_t passed as void*), performs no
 *    host synchronisation and is CUDA-graph capturable.
 *  - Return value: 0 = OK, NCF_ERR_ARG (-1) bad argument, NCF_ERR_CUDA (-2) CUDA error,
 *    NCF_ERR_WORKSPACE (-3) workspace too small.  ncf_last_error() returns a thread-local
 *    message for the last failing call on this thread.
 *  - There is no CPU fallback: without a CUDA device every compute entry returns NCF_ERR_CUDA.
 *  - Tables are fp32 row-major [rows, dim]; Linear weights are [out, in] row-major (the
 *    nn.Linear layout, reference src/ncf/models.py:24,34); indices are int64 (torch default).
 */
#ifndef NCF_B200_H
#define NCF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NCF_ABI_VERSION 1
#define NCF_MAX_LAYERS 8

#define NCF_OK 0
#define NCF_ERR_ARG (-1)
#define NCF_ERR_CUDA (-2)
#define NCF_ERR_WORKSPACE (-3)

/* model_type of reference src/ncf/models.py:5,30-33 ("NeuMF-end" and "NeuMF-pre" compute alike) */
#define NCF_GMF 0
#define NCF_MLP 1
#define NCF_NEUMF 2

/* tower_math: arithmetic of the tower contractions (embedding path, loss and optimiser are always
 * fp32).  NCF_MATH_FP32 keeps fp32 accuracy (error-compensated 3xTF32 on the tensor pipe, or fp32
 * FMA for shapes the tensor path does not cover) and is what the 1e-5 parity bar is stated for;
 * NCF_MATH_TF32 is single-pass TF32 (10-bit mantissa inputs, fp32 accumulate), ~3x fewer MMAs. */
#define NCF_MATH_FP32 0
#define NCF_MATH_TF32 1

/* Parameters of one NCF model (reference src/ncf/models.py:11-34).  mlp_dim = factor_num *
 * 2^(num_layers-1); tower layer k maps width factor_num*2^(num_layers-k) -> half of it. */
typedef struct NcfModel {
  int32_t model_type;
  int32_t factor_num;
  int32_t num_layers;
  int32_t mlp_dim;
  int32_t tower_math; /* NCF_MATH_* */
  int32_t reserved;
  int64_t user_num;
  int64_t item_num;
  float* embed_user_gmf; /* [user_num, factor_num]  embed_user_GMF.weight */
  float* embed_item_gmf; /* [item_num, factor_num]  embed_item_GMF.weight */
  float* embed_user_mlp; /* [user_num, mlp_dim]     embed_user_MLP.weight */
  float* embed_item_mlp; /* [item_num, mlp_dim]     embed_item_MLP.weight */
  float* mlp_w[NCF_MAX_LAYERS]; /* MLP_layers.{3k+1}.weight [out_k, in_k] */
  float* mlp_b[NCF_MAX_LAYERS]; /* MLP_layers.{3k+1}.bias   [out_k]       */
  float* predict_w;             /* predict_layer.weight [1, f | 2f]       */
  float* predict_b;             /* predict_layer.bias   [1]               */
} NcfModel;

/* Gradients of one training step.  The embedding gradients live in zero-initialised buffers
 * addressed like the tables (only touched rows are ever non-zero; the optimiser re-zeroes
 * them) plus a list of the distinct rows touched since the last optimiser step — the
 * deduplicated replacement of autograd's dense embedding grad (reference
 * scripts/train_neumf.py:114, SURVEY.md §8 a9).  Tower gradients are one flat buffer laid out
 * [W_0, b_0, W_1, b_1, ..., W_{L-1}, b_{L-1}, predict_w, predict_b]. */
typedef struct NcfGrads {
  float* g_user_gmf;
  float* g_item_gmf;
  float* g_user_mlp;
  float* g_item_mlp;
  float* g_tower;         /* flat, ncf_tower_param_count() floats */
  int32_t* user_flag;     /* [user_num] 0/1 */
  int32_t* item_flag;     /* [item_num] 0/1 */
  int64_t* user_list;     /* capacity >= max distinct users per optimiser step */
  int64_t* item_list;
  int32_t* touched_count; /* [4]: {n_user_rows, n_item_rows, ticket of the step-closing kernel (zero between calls), reserved} */
} NcfGrads;

/* Adam state (reference optim.Adam defaults, scripts/train_neumf.py:90).  The reference Adam is
 * DENSE: a row touched once keeps moving every later step through its momentum.  We update
 * only touched rows and replay the skipped zero-gradient steps lazily (last_step per row), so
 * results equal the dense update (SURVEY.md §7 H1).  ncf_adam_flush() brings every row up to
 * date before weights are read (evaluation, checkpoint). */
typedef struct NcfAdamState {
  float* m_user_gmf; float* v_user_gmf;
  float* m_item_gmf; float* v_item_gmf;
  float* m_user_mlp; float* v_user_mlp;
  float* m_item_mlp; float* v_item_mlp;
  float* m_tower;    float* v_tower;
  int32_t* user_last_step; /* [user_num], 0 = never touched */
  int32_t* item_last_step; /* [item_num] */
  int64_t* step;           /* [1] device step counter (number of optimiser steps taken) */
} NcfAdamState;

typedef struct NcfAdamHyper {
  float lr, beta1, beta2, eps;
} NcfAdamHyper;

/* ---- library ------------------------------------------------------------------------- */
int ncf_version(void);
const char* ncf_last_error(void);
/* which tile-kernel family the calling thread's last forward / training call ran on:
 * 0 none yet, 1 generic (FMA), 2 mma.sync tensor path, 3 tcgen05/TMEM path, 4 thread-per-sample FMA kernel
 * for narrow towers (factor_num 8) (diagnostic; tests) */
int ncf_last_tile_path(void);
/* Measurement aid for bench.py: with profiling on, every training step on the tcgen05 path records
 * the CUDA-event time of each of its launches (and synchronises the stream).  ncf_profile_read
 * copies the last step's times (milliseconds) and, if names != NULL, their labels as cap strings of
 * name_len bytes; returns the number of entries. */
/* Data-parallel overlap: makes `stream` wait until the embedding-row gradients (g_user_*, g_item_*) of
 * the calling thread's last ncf_train_step_grads / ncf_backward call are complete.  On the tcgen05
 * path that is before the weight-gradient kernel has run, so an all-reduce of the row gradients on
 * another stream overlaps with it; the tower gradients are complete when the call's stream is. */
int ncf_wait_embedding_grads(void* stream);
int ncf_profile_enable(int32_t on);
int ncf_profile_read(float* ms, char* names, int32_t cap, int32_t name_len);
/* number of floats in the flat tower buffer for this shape */
int64_t ncf_tower_param_count(int32_t model_type, int32_t factor_num, int32_t num_layers);

/* ---- a1: observed-pair structure --------------------------------------------------------
 * Replaces the dok_matrix fill loop of reference src/data/datasets.py:20-24 by a CSR with
 * sorted columns: rowptr int64[user_num+1], col int32[P].  Duplicate pairs are kept.  Pairs whose user
 * is outside [0, user_num) are left out; *bad_flag (device int32, nullable) is set to 1 when there was
 * such a pair or an item outside int32 (the reference's dok_matrix raises IndexError there).
 * Rows are sorted in shared memory (bitonic; one warp per row <= 256 items, one CTA per row <= 32 768).
 * workspace: ncf_csr_workspace_bytes(P, user_num). */
int64_t ncf_csr_workspace_bytes(int64_t P, int64_t user_num);
int ncf_csr_build(const int64_t* pos_user, const int64_t* pos_item, int64_t P, int64_t user_num,
                  int64_t* rowptr, int32_t* col, int32_t* bad_flag, void* workspace,
                  int64_t workspace_bytes, void* stream);

/* ---- (f) data side: the reference's on-disk formats and its leave-one-out preprocessing -------------------
 * Text: u.train.rating (`user<TAB>item` per line) and u.test.negative (`(user,pos)<TAB>neg1<TAB>...`, no
 * trailing newline) as written by reference src/data/preprocessing.py:137-154 and read by load_all
 * (src/data/datasets.py:9-36).  ncf_text_line_starts: positions of the first byte of every non-empty line
 * (a byte after '\n', or byte 0, that is not '\n' / '\r'); *n_lines (device) receives their number; with
 * line_start == NULL only the count is produced (call once to size the array, once to fill it).
 * ncf_text_parse_ints: out[line, j] = j-th integer (maximal digit run, optional leading '-') of the line,
 * j < K; *status (device) bit 0 = a line had fewer than K integers (missing ones are -1: the reference
 * would silently misalign its users there, SURVEY.md H5), bit 1 = (exact != 0) a line had more than K. */
int64_t ncf_text_workspace_bytes(int64_t nbytes);
int ncf_text_line_starts(const uint8_t* text, int64_t nbytes, int64_t* line_start, int64_t cap, int64_t* n_lines,
                         void* workspace, int64_t workspace_bytes, void* stream);
int ncf_text_parse_ints(const uint8_t* text, int64_t nbytes, const int64_t* line_start, int64_t n_lines, int32_t K,
                        int32_t exact, int64_t* out, int32_t* status, void* stream);
/* LeaveOneOutPreprocessor.temporal_split (reference src/data/preprocessing.py:45-90): ratings sorted by
 * (user, timestamp, position in the file); the last one of every user with at least two ratings goes to
 * (test_user, test_item) [ordered by user], everything else to (train_user, train_item) in sorted order.
 * totals (device int64[2]) = {n_train, n_test}; train_* need room for n entries, test_* for user_num.
 * *bad_flag (device, nullable): 1 = a user id outside [0, user_num) or a timestamp outside [0, 2^32),
 * 2 = a user with more than 16 384 ratings (the shared-memory row sort does not take it). */
int64_t ncf_split_workspace_bytes(int64_t n, int64_t user_num);
int ncf_leave_one_out_split(const int64_t* user, const int64_t* item, const int64_t* timestamp, int64_t n,
                            int64_t user_num, int64_t* train_user, int64_t* train_item, int64_t* test_user,
                            int64_t* test_item, int64_t* totals, int32_t* bad_flag, void* workspace,
                            int64_t workspace_bytes, void* stream);
/* generate_test_negatives (reference src/data/preprocessing.py:92-135): for test row r, up to K DISTINCT
 * items uniform over [0, num_items) that are not in row test_user[r] of the CSR (train and test items of the
 * user), at most 10 K draws, written ascending into out[r, :] (unused slots -1); count[r] = how many.
 * Draw a uses word a % 4 of Philox4x32-10(counter = {r (lo), r (hi), a / 4, 'NEGS'}, key = seed). */
int ncf_eval_negatives(const int64_t* rowptr, const int32_t* col, const int64_t* test_user, int64_t n,
                       int64_t user_num, int64_t num_items, int32_t K, uint64_t seed, int64_t* out, int32_t* count,
                       void* stream);

/* ---- a2: negative sampler ---------------------------------------------------------------
 * Replaces NCFData.ng_sample (reference src/data/datasets.py:53-69): for positive p and
 * t < num_ng, out_neg_item[p*num_ng + t] is drawn uniformly from [0, item_num) and redrawn
 * while (pos_user[p], j) is an observed pair.  Draw a of sample s = p_offset+p, t uses word
 * a%4 of Philox4x32-10(counter = {s*num_ng+t (lo), (hi), a/4, epoch}, key = seed), mapped to an
 * item by mulhi32(word, item_num).  p_offset lets shards sample disjoint global sample ids.
 * A positive whose user is outside [0, user_num), or whose 65 536 draws were all observed pairs (the
 * reference loops forever on a user who interacted with every item), gets -1: the training kernels
 * then report a bad index instead of training on an observed pair. */
int ncf_sample_neg(const int64_t* rowptr, const int32_t* col, const int64_t* pos_user, int64_t P,
                   int64_t p_offset, int64_t user_num, int32_t num_ng, int64_t item_num, uint64_t seed,
                   uint64_t epoch, int64_t* out_neg_item, void* stream);

/* ---- a3: epoch shuffle + batching ---------------------------------------------------------
 * Replaces DataLoader(shuffle=True) over NCFData.__getitem__ (reference
 * src/data/datasets.py:71-83, scripts/train_neumf.py:55): position q of the epoch stream holds
 * sample perm(q), where perm is a keyed bijection of [0, S), S = P*(1+num_ng); sample s < P is
 * positive s with label 1, sample s >= P is negative s-P with label 0 (positives-then-negatives
 * order of datasets.py:68).  Writes positions [q_begin, q_begin+count). */
int ncf_shuffle_epoch(const int64_t* pos_user, const int64_t* pos_item, const int64_t* neg_item,
                      int64_t P, int32_t num_ng, uint64_t seed, uint64_t epoch, int64_t q_begin,
                      int64_t count, int64_t* out_user, int64_t* out_item, float* out_label,
                      void* stream);

/* ---- a6: forward (inference) --------------------------------------------------------------
 * Replaces NCF.forward (reference src/ncf/models.py:97-118): logits[b] for (user[b], item[b]). */
int64_t ncf_forward_workspace_bytes(const NcfModel* m_host, int64_t B);
int ncf_forward(const NcfModel* m_host, const int64_t* user, const int64_t* item, int64_t B,
                float* logits, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- a7/a8: loss and its gradient w.r.t. the logits -----------------------------------------
 * Replaces nn.BCEWithLogitsLoss (reference scripts/train_neumf.py:86,113) and, when
 * teacher_logits != NULL, ResponseDistillation.combined_loss (reference
 * src/distillation/base.py:40-50 + response.py:28-32):
 *   loss = alpha * mean BCE(x, y) + (1-alpha) * mean (x - t)^2     (alpha ignored without teacher)
 * Adds the batch loss to *loss_accum (double) and, if dlogit != NULL, writes dloss/dx. */
int ncf_loss_grad(const float* logits, const float* label, const float* teacher_logits,
                  float alpha, int64_t B, double* loss_accum, float* dlogit, void* stream);
/* The other distillation objectives of the reference (src/distillation/base.py:26-50, response.py:34-61 and
 * the logit-level terms of feature.py:125-146 / attention.py:81-101): per-sample
 *   w_task * BCE(x, y) + w_kd * KD(x, t),   KD = (x - t)^2 (kd_mode 0) or
 *   KD = T^2 * (sigmoid(x/T) - sigmoid(t/T))^2 (kd_mode 1: BaseDistillation.knowledge_distillation_loss),
 * both means over the batch.  *loss_accum += loss; dlogit (nullable) receives dloss/dlogit for ncf_backward. */
int ncf_loss_grad_kd(const float* logits, const float* label, const float* teacher_logits, float w_task,
                     float w_kd, float temperature, int32_t kd_mode, int64_t B, double* loss_accum,
                     float* dlogit, void* stream);
/* Feature matching (reference src/distillation/feature.py:56-67,83-123) on one of the two embedding-level
 * features: kind 0 = gmf_features (E_uG[u] * E_iG[i]), kind 1 = mlp_input ([E_uM[u] ; E_iM[i]]).
 * *loss_accum += weight * mse(adapter(student feature), teacher feature); the gradient is added to the
 * student's embedding-gradient rows in g (the rows must have been registered by the step: ncf_mark_rows /
 * ncf_adam_prepare).  adapter_w [teacher width, student width] / adapter_b are the fixed nn.Linear the
 * reference creates when the widths differ (feature.py:36-46; never optimised, train_student.py:131);
 * NULL = identity (equal widths).  The tower-level features (mlp_linear_k / mlp_relu_k) only match for
 * equal architectures and are served by the autograd path (ncf_b200.distillation.FeatureDistillation). */
int ncf_feature_kd(const NcfModel* student_host, const NcfModel* teacher_host, const NcfGrads* g_host,
                   const int64_t* user, const int64_t* item, int64_t B, int32_t kind, const float* adapter_w,
                   const float* adapter_b, float weight, double* loss_accum, void* stream);

/* ---- a6+a7+a8+a9: fused training step (forward, loss, backward) --------------------------------
 * Replaces `prediction = model(user,item); loss = criterion(...); loss.backward()` (reference
 * scripts/train_neumf.py:112-114; with teacher_logits: scripts/train_student.py:154-155).
 * Accumulates into g (which must be zero for a fresh step), adds the batch loss to *loss_accum,
 * optionally writes the logits.  workspace: ncf_train_workspace_bytes(m, B). */
int64_t ncf_train_workspace_bytes(const NcfModel* m_host, int64_t B);
int ncf_train_step_grads(const NcfModel* m_host, const NcfGrads* g_host, const int64_t* user,
                         const int64_t* item, const float* label, const float* teacher_logits,
                         float alpha, int64_t B, double* loss_accum, float* logits_out,
                         void* workspace, int64_t workspace_bytes, void* stream);

/* Same as ncf_train_step_grads, but the loss mean (and hence dloss/dlogit) is taken over B_norm >= B
 * samples: the B local samples of this rank are a slice of a global batch of B_norm (multi-GPU). */
int ncf_train_step_grads_norm(const NcfModel* m_host, const NcfGrads* g_host, const int64_t* user,
                              const int64_t* item, const float* label, const float* teacher_logits,
                              float alpha, int64_t B, int64_t B_norm, double* loss_accum,
                              float* logits_out, void* workspace, int64_t workspace_bytes,
                              void* stream);

/* ---- a9 alone: backward from a caller-supplied dloss/dlogit ---------------------------------------
 * Replaces autograd's backward through NCF.forward (reference scripts/train_neumf.py:114) when the
 * loss was computed elsewhere (e.g. by torch in an unmodified reference loop): recomputes the
 * forward for the batch inside the fused kernel and accumulates the gradients into g. */
int ncf_backward(const NcfModel* m_host, const NcfGrads* g_host, const int64_t* user,
                 const int64_t* item, const float* dlogit, int64_t B, void* workspace,
                 int64_t workspace_bytes, void* stream);

/* ---- a10: optimisers --------------------------------------------------------------------------
 * ncf_adam_step: optim.Adam(lr, betas=(0.9,0.999), eps=1e-8).step() (reference
 * scripts/train_neumf.py:90,115) on the tower (dense) and on the touched rows (lazy, dense-
 * equivalent); consumes and re-zeroes g, increments *s->step.
 * ncf_adam_flush: replays pending zero-gradient steps for every row (call before reading weights).
 * ncf_sgd_step: optim.SGD(lr).step() (reference scripts/train_neumf.py:88), no momentum. */
/* ncf_mark_rows: registers the distinct (user, item) rows of a batch in g's touched lists — the
 * dedup the optimisers iterate over.  Every optimiser step must be preceded by ncf_adam_prepare
 * (Adam; it marks and catches up) or ncf_mark_rows (SGD) on the same batch. */
int ncf_mark_rows(const NcfModel* m_host, const NcfGrads* g_host, const int64_t* user,
                  const int64_t* item, int64_t B, void* stream);
/* One side at a time (side 0 = users, 1 = items), for row lists that do not pair up: row-sharded
 * tables register a rank's own users and the item rows other ranks requested separately. */
int ncf_mark_rows_side(const NcfModel* m_host, const NcfGrads* g_host, const int64_t* rows, int64_t n,
                       int32_t side, void* stream);
/* Replays the pending zero-gradient Adam steps of every row currently in g's touched lists. */
int ncf_adam_catchup(const NcfModel* m_host, const NcfGrads* g_host, const NcfAdamState* s_host,
                     NcfAdamHyper h, void* stream);
/* ncf_adam_prepare: call BEFORE ncf_train_step_grads of the same batch.  Registers the batch's
 * distinct rows in g's touched lists and replays their pending zero-gradient steps, so that the
 * forward reads the rows exactly as the reference's dense Adam would have left them. */
int ncf_adam_prepare(const NcfModel* m_host, const NcfGrads* g_host, const NcfAdamState* s_host,
                     NcfAdamHyper h, const int64_t* user, const int64_t* item, int64_t B,
                     void* stream);
int ncf_adam_step(const NcfModel* m_host, const NcfGrads* g_host, const NcfAdamState* s_host,
                  NcfAdamHyper h, void* stream);
/* The same optimiser step taken over EVERY row of the tables (the reference's dense Adam literally):
 * rows without gradient take their zero-gradient step now instead of being replayed later.  Cheaper
 * than list + catch-up + row gather once a step touches a large share of the rows (large batches,
 * data-parallel global batches).  After it every row is current: the next step needs no
 * ncf_adam_prepare (ncf_mark_rows is not needed for this entry either). */
int ncf_adam_step_dense(const NcfModel* m_host, const NcfGrads* g_host, const NcfAdamState* s_host,
                        NcfAdamHyper h, void* stream);
/* The all-rows step restricted to user rows [user_lo, user_hi) (and every item row): data-parallel
 * ranks that each train on the samples of their own range of users (new design, SURVEY.md 8e) own
 * those user rows - the other user rows are never read or written on this rank.  parts: mask of 1 (user
 * tables), 2 (item tables), 4 (tower) = what this call updates; the rest was updated by another path of
 * the same step (the peer-memory exchange ncf_adam_p2p for the replicated item tables and the tower).
 * Whatever parts is, user rows [user_lo, user_hi) and every item row are stamped as current (last step =
 * the new step, flags cleared), the step counter is incremented and the touched counts are zeroed; user rows
 * outside the range are not touched.  Gradients are consumed (zeroed) only in the parts updated.  Partial
 * parts need row widths that are multiples of 4 floats. */
int ncf_adam_step_dense_range(const NcfModel* m_host, const NcfGrads* g_host, const NcfAdamState* s_host,
                              NcfAdamHyper h, int64_t user_lo, int64_t user_hi, int32_t parts, void* stream);
/* Optimiser sharding for replicated data parallelism (new design, SURVEY.md 8e): with parameters,
 * gradients and moments laid out as flat buffers, every rank reduce-scatters the gradients, updates
 * its own slice with ncf_adam_range (elementwise Adam at step *step + 1; zeroes g; every row must be
 * current, i.e. the all-rows mode) and all-gathers the parameters; ncf_adam_finish_dense then stamps
 * every row as current and increments the step counter. */
int ncf_adam_range(float* p, float* m, float* v, float* g, int64_t n, const int64_t* step, NcfAdamHyper h,
                   void* stream);
int ncf_adam_finish_dense(const NcfModel* m_host, const NcfGrads* g_host, const NcfAdamState* s_host,
                          void* stream);
/* The same sharded step with the gradient exchange inside the kernel, for ranks on one NVLink node
 * (experimental, NCF_DP_P2P=1 in ncf_b200.dist): grad_bufs / param_bufs are HOST arrays of `world`
 * device pointers - entry r is rank r's flat gradient / parameter buffer, entry `rank` the caller's own,
 * the others mapped with ncf_ipc_open.  The caller owns elements [lo, lo + n): the kernel sums that slice
 * over every rank's gradients (peer loads) times grad_scale (1/world for rank-mean gradients, 1 when every
 * rank already divided by the global batch), updates m / v (n elements, local) and stores the
 * new parameters into every rank's buffer (peer stores).  Bracket it with rank barriers: all gradients
 * complete before, all ranks done after (then zero the local gradient buffer). */
int ncf_adam_p2p(const void* const* grad_bufs, void* const* param_bufs, float* m, float* v, int64_t lo, int64_t n,
                 int32_t world, int32_t rank, float grad_scale, const int64_t* step, NcfAdamHyper h, void* stream);
/* Rank barrier over peer memory for the exchanges above (instead of a one-element NCCL all-reduce): flag_peers
 * is a HOST array of `world` device pointers to every rank's flag array (uint32[world], zero-initialised,
 * ncf_peer_alloc + ncf_ipc_open); epoch_counter is a local device uint32 (zero-initialised) that counts this
 * rank's barriers, so the call can be captured in a CUDA graph.  Every rank must issue the same sequence of
 * barriers on its stream.  Release / acquire at system scope: writes of earlier kernels on the stream are
 * visible to what the peers launch after their barrier.  The wait is bounded (trap, not hang). */
int ncf_peer_barrier(void* const* flag_peers, int32_t world, int32_t rank, uint32_t* epoch_counter, void* stream);
/* Buffers shared between ranks have to be allocations of their own (CUDA IPC exports whole
 * allocations): ncf_peer_alloc returns zero-filled device memory of the current device, the only
 * memory this library ever owns; ncf_ipc_export writes its 64-byte handle, which the peers turn into
 * a pointer valid on their current device with ncf_ipc_open (undo: ncf_ipc_close, ncf_peer_free). */
int ncf_peer_alloc(int64_t bytes, void** dev_ptr_out);
int ncf_peer_free(void* dev_ptr);
int ncf_ipc_export(const void* dev_ptr, void* handle64);
int ncf_ipc_open(const void* handle64, void** dev_ptr_out);
int ncf_ipc_close(void* dev_ptr);
int ncf_adam_flush(const NcfModel* m_host, const NcfAdamState* s_host, NcfAdamHyper h,
                   void* stream);
int ncf_sgd_step(const NcfModel* m_host, const NcfGrads* g_host, float lr, void* stream);

/* ---- (e) row-sharded tables: pack / unpack around the NCCL all-to-alls ----------------------------------
 * New design (the reference is single-process, SURVEY.md 8e).  Row r lives on rank r % world at
 * local index r / world.
 * ncf_bucket_by_owner: groups the n samples by the owner of their item: perm[pos] = sample index,
 *   local_idx[pos] = item / world, counts[w] = samples whose item lives on rank w; cursor is
 *   int32[world] scratch.  A negative item (ncf_sample_neg's -1) counts for owner 0 with local_idx = -1, so
 *   counts and perm still cover all n samples; ncf_gather_rows zero-fills its row and ncf_scatter_add_rows
 *   skips it.  1 <= world <= 64.  ncf_permute_*: out[i] = in[perm[i]].
 * ncf_gather_rows: out[i][:] = table[idx[i]][:].  ncf_scatter_add_rows: table[idx[i]][:] += in[i][:]. */
int ncf_bucket_by_owner(const int64_t* item, int64_t n, int32_t world, int64_t* perm,
                        int64_t* local_idx, int32_t* counts, int32_t* cursor, void* stream);
int ncf_permute_i64(const int64_t* in, const int64_t* perm, int64_t n, int64_t* out, void* stream);
int ncf_permute_f32(const float* in, const int64_t* perm, int64_t n, float* out, void* stream);
int ncf_gather_rows(const float* table, const int64_t* idx, int64_t n, int32_t dim, int64_t rows,
                    float* out, void* stream);
int ncf_scatter_add_rows(float* table, const int64_t* idx, int64_t n, int32_t dim, int64_t rows,
                         const float* in, void* stream);

/* The same exchange over peer memory on one NVLink node (no NCCL all-to-all, no split sizes on the host):
 * every rank maps the others' buffers through CUDA IPC (ncf_peer_alloc / ncf_ipc_export / ncf_ipc_open) and
 * passes arrays of `world` device addresses (entry r = rank r's buffer as seen from this device).
 *   inbox        int64 [world][cap] per rank: entry (source r, j) = (local row << 32) | slot
 *   inbox_count  int32 [world]      per rank: requests of source r
 * ncf_shard_request (requester): writes one request per sample into the inbox of the owner of its item
 *   (item % world) and then the per-owner counts; slot = the sample's position in the batch.  cursor:
 *   int32[world] local scratch.  ncf_shard_mark_requests (owner): registers the requested rows in the item
 *   side of the touched list (then ncf_adam_catchup).  ncf_shard_push_rows (owner): stores each requested
 *   row of its item tables into the requester's receive buffers [cap, f] / [cap, d] at `slot`.
 * ncf_shard_push_grads (requester): g_gmf[s] / g_mlp[s] (per-sample item-row gradients of the fused step)
 *   are added (red.sys over NVLink) to row item[s] / world of the gradient tables of rank item[s] % world.
 * The caller separates request | mark + catch-up + push rows | fused step + push grads | optimiser by rank
 * barriers. */
int ncf_shard_request(const int64_t* item, int64_t n, int32_t world, int32_t rank, int64_t cap, int64_t item_num,
                      void* const* inbox_peers, void* const* inbox_count_peers, int32_t* cursor, void* stream);
int ncf_shard_mark_requests(const NcfModel* m_host, const NcfGrads* g_host, const int64_t* inbox,
                            const int32_t* inbox_count, int32_t world, int64_t cap, void* stream);
int ncf_shard_push_rows(const NcfModel* m_host, const int64_t* inbox, const int32_t* inbox_count, int32_t world,
                        int64_t cap, void* const* rows_gmf_peers, void* const* rows_mlp_peers, void* stream);
int ncf_shard_push_grads(const int64_t* item, int64_t n, int32_t world, int64_t item_num, const float* g_gmf,
                         const float* g_mlp, int32_t f, int32_t d, void* const* grad_gmf_peers,
                         void* const* grad_mlp_peers, void* stream);

/* ---- a11: leave-one-out evaluation --------------------------------------------------------------
 * Replaces metrics() (reference src/training/metrics.py:4-25).  scores is [n, C]; column 0 is the
 * held-out positive (reference src/data/datasets.py:31-34).  Per user: topk_idx[k] = indices of the
 * k largest scores in descending order, ties (-0.0 == +0.0) broken towards the LOWER candidate index;
 * NaN is not a candidate, and a row with fewer than k non-NaN scores is padded with -1.  This is the
 * order of ncf_topk_rows.  rank = position of candidate 0 in that order, or -1 when it is not among
 * the first k or is NaN; hit = rank >= 0; ndcg = 1/log2(rank+2) or 0.  (torch.topk, which the
 * reference uses, ranks NaN above every number, so there a NaN held-out score counts as a hit.)
 * Any of hit / rank / ndcg / topk_idx may be NULL.  Requires 1 <= k <= C <= 1024. */
int ncf_eval_rank(const float* scores, int64_t n, int32_t C, int32_t k, uint8_t* hit,
                  int32_t* rank, float* ndcg, int32_t* topk_idx, void* stream);
/* Scores every user's C candidates with the model, then ranks as above.
 * workspace: ncf_eval_workspace_bytes(m, n, C). */
int64_t ncf_eval_workspace_bytes(const NcfModel* m_host, int64_t n, int32_t C);
int ncf_eval_users(const NcfModel* m_host, const int64_t* users, const int64_t* cands, int64_t n,
                   int32_t C, int32_t k, uint8_t* hit, int32_t* rank, float* ndcg,
                   int32_t* topk_idx, float* scores_out, void* workspace, int64_t workspace_bytes,
                   void* stream);

/* ---- full-catalog recommendation and full-ranking evaluation ---------------------------------------
 * New capability (the reference ranks only the sampled candidates of metrics()).
 * ncf_mask_items excludes items from per-row scores: for row r, every col[j], j in
 * [rowptr[users[r]], rowptr[users[r]+1]), with 0 <= col[j] < C sets scores[r, col[j]] = NaN.  A row whose
 * users[r] is outside [0, user_num) is set to NaN entirely.  rowptr/col: the sorted CSR of ncf_csr_build
 * (duplicates allowed). */
int ncf_mask_items(float* scores, int64_t n, int64_t C, const int64_t* users, int64_t user_num,
                   const int64_t* rowptr, const int32_t* col, void* stream);

/* Per row of scores [n, C]: the k best candidates, best first.  NaN = not a candidate.  Order: larger score
 * first; equal scores (-0.0 == +0.0) -> lower column first (the rule of ncf_eval_rank).  topk_item[r, j] is
 * the column, topk_score[r, j] the score as stored in the row.  Rows with fewer than k candidates are padded
 * with item -1 / score NaN.  target (nullable, [n]): target_rank[r] = number of candidates that precede
 * column target[r] in that order (full rank, not capped by k); -1 when the target is outside [0, C), not a
 * candidate, or target is NULL (target_rank nullable only then).  1 <= k <= 1024, k <= C < 2^31.
 * Every score is read four times whatever k is (radix select in shared memory: the workspace query returns 0
 * for valid arguments, -1 otherwise). */
int64_t ncf_topk_rows_workspace_bytes(int64_t n, int64_t C, int32_t k);
int ncf_topk_rows(const float* scores, int64_t n, int64_t C, int32_t k, const int64_t* target,
                  int64_t* topk_item, float* topk_score, int32_t* target_rank,
                  void* workspace, int64_t workspace_bytes, void* stream);

/* Scores users[0..n) against every item of the model (the forward kernels of ncf_forward), excludes each
 * user's CSR row (rowptr/col with user_num + 1 row pointers; both NULL: no exclusion) and selects as
 * ncf_topk_rows, with columns = item ids.  Users are processed min(chunk_users, n) at a time, at most 2^28
 * (user, item) pairs per chunk: workspace = scores [chunk, item_num] + item ids [chunk * item_num] + forward
 * workspace, sized by ncf_recommend_workspace_bytes(m, min(chunk_users, n), k).  k <= item_num < 2^31. */
int64_t ncf_recommend_workspace_bytes(const NcfModel* m, int64_t chunk_users, int32_t k);
int ncf_recommend(const NcfModel* m, const int64_t* users, int64_t n, int32_t k,
                  const int64_t* rowptr, const int32_t* col, const int64_t* target, int64_t chunk_users,
                  int64_t* topk_item, float* topk_score, int32_t* target_rank,
                  void* workspace, int64_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NCF_B200_H */
