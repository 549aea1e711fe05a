/* glove_b200.h -- C ABI of libglove_b200.so: the B200-native (sm_100a) GloVe training / eval / top-k hot path.
 *
 * The reference (yxtay/glove-tensorflow) has NO native plugin / FFI interface: every FLOP of its hot path runs inside
 * stock TensorFlow 2.11 ops reached from Python.  The seam this library slots under is therefore the internal one
 *     model_fn(features, labels, mode, params) -> EstimatorSpec      [ref src/models/estimator.py:13-56]
 *     input_fn() -> tf.data.Dataset                                  [ref src/models/data_utils.py:4-26]
 * with mode TRAIN -> glove_prepare_batches + glove_train_step, EVAL -> glove_eval_loss, PREDICT -> glove_topk_cosine.
 * Each entry point below cites the reference call site it replaces.
 *
 * Conventions
 *   - extern "C", plain C types only; every entry returns int (0 = GLOVE_OK, < 0 = error, text via glove_last_error()).
 *   - All buffers are CALLER-OWNED DEVICE pointers (e.g. torch tensors); the library never allocates user-visible
 *     memory.  Scratch is caller-provided; sizes come from the *_bytes() queries.  (Exceptions: the *_host entry points
 *     at the bottom take HOST buffers and do their own staging -- they are the end-to-end convenience boundary.)
 *   - All work is enqueued asynchronously on the caller's cudaStream_t (passed as void*); no hidden synchronisation;
 *     every launch sequence is CUDA-graph capturable (the step index lives in device memory, see glove_scalars).
 *   - No global mutable state except the thread-local error string.
 *
 * Table layout ("packed table"): one buffer per side (row / col), float32 [V][P][S]:
 *     S = glove_table_stride(d) = roundup(d + 2, 8) floats (so every plane row is a whole number of 32-byte sectors)
 *     P = glove_table_planes(optimizer): Adam 3 (x, m, v); Adagrad 2 (x, accumulator); SGD 1 (x)
 *     plane 0 row = [ x_0 .. x_{d-1} | c_d | c_{d+1} | 0 .. ] with, for side s (0 = row table, 1 = col table),
 *                   the bias in column d+s and the last_step word (int32 bits) in column d+1-s.  The two sides are
 *                   mirrored so that the dot product of a row-side and a col-side snapshot row needs no masking.
 *     plane p>0   = optimizer slot for the same columns (bias slot in column d+s)
 *   The reference keeps 4 Keras Embedding variables (R,C [V,d]; rb,cb [V,1]; src/models/model_utils.py:31-39) plus Keras
 *   optimizer slots; glove_pack_plane / glove_unpack_plane convert between the two layouts.
 */
#ifndef GLOVE_B200_H_
#define GLOVE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* 2: glove_step_args starts with struct_size and ends with peer_gather (n_shards, shard, peer_gather were appended in
 *    round 1 without a bump); adam_mode gained GLOVE_ADAM_REPLAY_EXACT and GLOVE_ADAM_REPLAY became the closed-form
 *    replay; glove_train_steps_host takes a caller-owned glove_host_pipe; glove_step_graph_* added. */
#define GLOVE_B200_ABI_VERSION 2

enum { GLOVE_OK = 0, GLOVE_EINVAL = -1, GLOVE_ECUDA = -2, GLOVE_EWORKSPACE = -3, GLOVE_EUNSUPPORTED = -4 };

/* head: which estimator head builds the loss.
 *   GLOVE_HEAD_GLOVE    tf.estimator.RegressionHead(weight_column)                 [ref src/models/estimator.py:48-56]
 *   GLOVE_HEAD_LOGISTIC BinaryClassHead x2 + MultiHead([pos, neg], [1, neg_factor]) [ref src/models/logistic_matrix_factorisation.py:50-54] */
enum { GLOVE_HEAD_GLOVE = 0, GLOVE_HEAD_LOGISTIC = 1 };

/* optimizer: tf.keras.optimizers.get({"class_name": name, ...}) legacy OptimizerV2 classes [ref src/models/train_utils.py:13-16] */
enum { GLOVE_OPT_ADAM = 0, GLOVE_OPT_ADAGRAD = 1, GLOVE_OPT_SGD = 2 };

/* adam_mode:
 *   GLOVE_ADAM_REPLAY  reference semantics (legacy Keras Adam decays m, v and moves x on ALL rows every step) obtained
 *                      without dense sweeps: the zero-gradient steps a row missed are applied when it is next touched
 *                      (and by glove_flush_lazy_state before eval / export / checkpoint), in CLOSED FORM: the run
 *                      sum_j alpha_j b1^j m0 / (b2^(j/2) sqrt(v0) + eps) is a cubic in q = sqrt(v0)/(sqrt(v0)+eps) with
 *                      per-row coefficients, so a run of any length costs one sqrt + one reciprocal per element.  Equal to
 *                      the sequential recurrence to fp32 resolution (closer to its fp64 value than the fp32 recurrence is).
 *   GLOVE_ADAM_REPLAY_EXACT  the same schedule with the run replayed step by step with exactly the fp32 operations of the
 *                      dense sweep: bit-identical to flushing after every step (the literal legacy-Keras schedule), at the
 *                      price of O(gap) arithmetic per element.  Kept as the arithmetic ground truth of the tests.
 *   GLOVE_ADAM_LAZY    LazyAdam: untouched rows frozen.  NOT the reference's arithmetic; kept for measurement. */
enum { GLOVE_ADAM_REPLAY = 0, GLOVE_ADAM_LAZY = 1, GLOVE_ADAM_REPLAY_EXACT = 2 };

/* Device-resident scalars (32 bytes).  step = global_step = number of optimizer steps applied so far
 * [ref src/models/estimator.py:44-45].  g = MatrixFactorisation.global_bias [ref src/models/model_utils.py:39]. */
typedef struct glove_scalars {
    int32_t step;
    int32_t error;      /* sticky device-side error flag (0 = ok) */
    float g, g_s0, g_s1; /* global bias and its optimizer slots (Adam m, v / Adagrad accumulator) */
    float loss;         /* loss of the most recent train step */
    int32_t ticket;     /* internal */
    int32_t reserved;
} glove_scalars;

const char *glove_last_error(void);
int32_t glove_abi_version(void);

/* ---- packed tables ------------------------------------------------------------------------------------------ */
int32_t glove_table_stride(int32_t d);
int32_t glove_table_planes(int32_t optimizer);
/* zero the table, last_step = 0, Adagrad accumulator plane = 0.1 (Keras initial_accumulator_value) */
int glove_table_init(float *table, int64_t V, int32_t d, int32_t optimizer, int32_t side, void *stream);
/* plane <- (emb [V,d], bias [V] (may be NULL)) ; replaces 4x ResourceGather-able Keras variables [ref model_utils.py:31-37] */
int glove_pack_plane(float *table, int64_t V, int32_t d, int32_t planes, int32_t plane, int32_t side, const float *emb,
                     const float *bias, void *stream);
int glove_unpack_plane(const float *table, int64_t V, int32_t d, int32_t planes, int32_t plane, int32_t side,
                       float *emb, float *bias, void *stream);
/* read / write the per-row last_step column (int32 [V]) -- checkpoint / resume */
int glove_get_last_step(const float *table, int64_t V, int32_t d, int32_t planes, int32_t side, int32_t *out,
                        void *stream);
int glove_set_last_step(float *table, int64_t V, int32_t d, int32_t planes, int32_t side, const int32_t *in,
                        void *stream);

/* ---- input pipeline: replaces make_csv_dataset shuffle/batch [ref src/models/data_utils.py:4-26] -------------- */
/* out[k] = position in the COO of global sample (first + k): epoch e = n / nnz uses the keyed bijection with key
 * (key + e) on n % nnz.  Deterministic, stateless, O(1) memory. */
int glove_shuffle_indices(uint32_t key, int64_t nnz, int64_t first, int64_t count, int64_t *out, void *stream);

size_t glove_plan_bytes(int32_t K, int32_t B);
size_t glove_prepare_workspace_bytes(int32_t K, int32_t B);
/* Builds the plan for K consecutive batches of B samples: gathers the triples (explicit sample_idx [K*B] if non-NULL,
 * else the keyed shuffle starting at global sample first_sample), sorts each batch by row id and by col id (stable),
 * and emits segment / work-item lists.  colA/colB = (glove_value, glove_weight) or (value, neg_weight).
 * first_step = the optimizer step that batch 0 of this plan belongs to. */
int glove_prepare_batches(void *plan, void *workspace, size_t workspace_bytes, const int32_t *row, const int32_t *col,
                          const float *colA, const float *colB, int64_t nnz, const int64_t *sample_idx,
                          int64_t first_sample, uint32_t shuffle_key, int32_t first_step, int32_t K, int32_t B,
                          int32_t V, void *stream);
/* Same, for row-sharded tables (n_shards owners, owner of id = id % n_shards, local row = id / n_shards): ids are
 * remapped owner-major so that every owner's rows form one block of slots; slot positions are padded so that all
 * owners' blocks have the same size (see glove_plan_shard_info).  n_shards = 1 is glove_prepare_batches. */
int glove_prepare_batches_sharded(void *plan, void *workspace, size_t workspace_bytes, const int32_t *row,
                                  const int32_t *col, const float *colA, const float *colB, int64_t nnz,
                                  const int64_t *sample_idx, int64_t first_sample, uint32_t shuffle_key,
                                  int32_t first_step, int32_t K, int32_t B, int32_t V, int32_t n_shards, void *stream);
/* Host view of batch k's shard layout: out20[10*side + r] (r = 0..8) = first slot owned by shard r (entries past
 * n_shards = number of segments), out20[10*side + 9] = padded slots per shard.  Synchronises the stream. */
int glove_plan_shard_info(const void *plan, int32_t K, int32_t B, int32_t k, int32_t *out20, void *stream);
/* Debug / test view of a plan: copies per-batch counts to host-visible ints: out[0..3] = {n_row_segments,
 * n_col_segments, n_row_items, n_col_items} of batch k.  Synchronises the stream. */
int glove_plan_batch_counts(const void *plan, int32_t K, int32_t B, int32_t k, int32_t *out4, void *stream);

/* ---- TRAIN: model_fn(mode=TRAIN) + optimizer.get_updates [ref src/models/estimator.py:13-56] ------------------- */
typedef struct glove_step_args {
    uint32_t struct_size;         /* = sizeof(glove_step_args) as compiled by the CALLER (glove_step_args_size() is the
                                   * library's): every entry point refuses a mismatch instead of reading past the struct */
    float *row_table, *col_table; /* packed tables */
    glove_scalars *scalars;       /* device */
    const void *plan;             /* from glove_prepare_batches; the batch used is (scalars->step - plan.first_step) */
    void *workspace;              /* glove_step_workspace_bytes(B, d); ZERO-FILLED before its first use */
    size_t workspace_bytes;
    const float *alpha;           /* device fp32 [alpha_len]: Adam step size per 0-based step (lr*sqrt(1-b2^t)/(1-b1^t)) */
    int32_t alpha_len;
    float *loss_out;              /* device fp32 [loss_cap]: loss_out[step % loss_cap] = pre-update loss; may be NULL */
    int32_t loss_cap;
    int32_t plan_K;
    int64_t V;
    int32_t d, B;
    int32_t head, optimizer, adam_mode;
    float learning_rate, l2_reg, reg_scale, neg_factor;
    float beta1, beta2, epsilon;
    /* data-parallel: this rank only accumulates triples whose in-batch index p satisfies p / dp_block == dp_rank
     * (dp_world <= 1 disables).  See glove_grad_step / glove_apply_step. */
    int32_t dp_rank, dp_world;
    /* row-sharded tables (n_shards > 1): this process holds the rows with id % n_shards == shard (local row id /
     * n_shards, V_local = ceil(V / n_shards)); the plan must come from glove_prepare_batches_sharded.  0 / 1 = not sharded. */
    int32_t n_shards, shard;
    /* row-sharded tables with peer-mapped workspaces (glove_shard_set_peers): 4 = rows pushed by the owners' stage kernels +
     * device-side synchronisation; 3 = pull + device-side synchronisation (see glove_shard_train_step); 2 = the requested rows are pulled into the
     * local snapshot by glove_shard_pull_step; 1 = no pull, glove_shard_update_step gathers every opposite row straight
     * from its owner's workspace over NVLink; 0 = rows arrive through a collective (pack / unpack or all-gather). */
    int32_t peer_gather;
} glove_step_args;

size_t glove_step_args_size(void);
size_t glove_step_workspace_bytes(int32_t B, int32_t d);
/* one full TRAIN step; increments scalars->step */
int glove_train_step(const glove_step_args *args, void *stream);
/* n_steps consecutive TRAIN steps captured once as a CUDA graph (2 n_steps kernel nodes) and replayed with one launch:
 * the step index and the batch derived from it are read from device memory, so a graph built on `args` is valid for ANY
 * run of n_steps steps that this plan buffer serves (n_steps <= plan_K, starting where scalars->step stands).  Replaces the
 * n_steps session.run(train_op) calls of the reference's hook-driven loop [ref src/models/train_utils.py:39-40] when the
 * batch is small enough for launch overhead to matter (configs/app.ini: BATCH_SIZE = 1024).  The handle is caller-owned;
 * results are bit-identical to n_steps glove_train_step calls. */
typedef struct glove_step_graph glove_step_graph;
int glove_step_graph_create(const glove_step_args *args, int32_t n_steps, glove_step_graph **out);
int glove_step_graph_launch(glove_step_graph *graph, void *stream);
int glove_step_graph_destroy(glove_step_graph *graph);
/* Optional overlap aid for GLOVE_ADAM_REPLAY_EXACT: replays, ahead of time and on ANOTHER stream, the idle Adam steps of the
 * rows of step `step_index`'s batch that are not in the batch of step_index-1 (so the step in flight cannot touch
 * them).  Must be ordered after the completion of step_index-2 and before the start of step_index (events); a no-op
 * for the first batch of a plan and for other optimizers / modes.  Results are bit-identical with or without it. */
int glove_catchup_step(const glove_step_args *args, int32_t step_index, void *stream);
/* same step, with CUDA events recorded around its three kernels on `stream`; synchronises and returns their device
 * durations in milliseconds: ms3 = {stage, update (incl. split-segment combine and step finish), 0}.  Measurement aid for bench.py (roofline). */
int glove_train_step_profiled(const glove_step_args *args, void *stream, float *ms3);
/* data-parallel split of the same step: grad_step writes this rank's partial gradient sums for every global segment
 * into grad_rows / grad_cols ([n_segments][S], dense in slot order) and {sum w*l.., sum e} into grad_scalars[4];
 * the caller all-reduces those three buffers (NCCL), then apply_step applies the optimizer on every replica. */
int glove_grad_step(const glove_step_args *args, float *grad_rows, float *grad_cols, float *grad_scalars,
                    void *stream);
int glove_apply_step(const glove_step_args *args, const float *grad_rows, const float *grad_cols,
                     const float *grad_scalars, void *stream);

/* Row-sharded tables (cfg4, SURVEY 8e), owner-computes.  One step on every rank is
 *   glove_shard_stage_step   stage (and replay) the OWNED rows of the batch into this shard's block of the snapshot
 *   -- all-gather the snapshot blocks (equal-sized, see glove_plan_shard_info) --
 *   glove_shard_update_step  the fused gather-loss-update of the work items of the OWNED segments (both sides), written
 *                            in place to the local tables; loss_scalars[0..2] = this rank's {data loss, sum e, reg} sums
 *   -- all-reduce loss_scalars (3 floats) --
 *   glove_shard_finish_step  loss, replicated global bias, step counter (identical on every rank)
 * No gradient ever crosses the network: the only bulk exchange is the snapshot of the touched rows.
 * The snapshot lives in the step workspace: side s starts at glove_step_snapshot_offset(B, d, s) bytes and holds
 * glove_step_snapshot_rows(B) rows of glove_table_stride(d) floats.
 *
 * Exchange variants between stage and update: (a) all-gather of the shards' snapshot blocks (every row to every rank), or
 * (b) all-to-all of REQUESTED rows only -- glove_shard_pack_step gathers, for every peer, the rows of this shard's block
 * that the peer's work items need (request lists built at plan time, see glove_plan_need_info) into send_buf;
 * all_to_all(v); glove_shard_unpack_step scatters the received rows to their snapshot positions. */
/* (c) peer memory: no NCCL data movement at all.  Every rank allocates its step workspace in peer-mapped memory (CUDA
 * IPC / symmetric memory) and registers all of them once with glove_shard_set_peers.  A step is
 *   stage -> barrier across ranks -> [glove_shard_pull_step] -> glove_shard_update_step -> all-reduce of loss_scalars
 *   (doubles as the barrier that keeps the next stage from overwriting a snapshot block a peer still reads) -> finish.
 * peer_gather = 2: glove_shard_pull_step reads every REQUESTED row once from its owner's snapshot over NVLink and writes
 * it to the same position of the local snapshot (pack + all-to-all + unpack in one launch, no staging buffers);
 * peer_gather = 1: no pull; the update kernel loads each opposite row from the snapshot of its owner (position / padded
 * block size) while it computes -- one launch fewer, but a row is fetched once per triple instead of once per step. */
/* peer_gather = 3: as 2, and the step synchronises ON THE DEVICE: a rank announces "my snapshot block is staged" / "my
 * update is done, here are my loss sums" by writing an epoch (and the sums) into every peer's workspace with system-scope
 * release stores and waits by polling its own memory -- no symmetric-memory barrier, no NCCL all-reduce, no host round
 * trip between the phases (the pull waits owner by owner, the finish adds the ranks' sums in rank order).  A step is
 *   glove_shard_train_step = stage -> glove_shard_signal_staged -> pull -> update -> glove_shard_finish_sync
 * five launches, capturable by glove_step_graph_create.  The two announcements are exposed for callers that drive the phases
 * themselves (N shards emulated on one GPU: every shard must have announced before any shard waits). */
/* peer_gather = 4 (Adam with the closed-form replay): as 3, and the exchange is FUSED INTO THE STAGE: an owner writes every
 * row it stages straight from registers into the snapshot of each shard whose work items read it (request mask per segment,
 * built at plan time) -- posted NVLink writes that overlap the staging of the following rows; there is no pull kernel,
 * glove_shard_wait_staged only waits for the owners' announcements:
 *   glove_shard_train_step = stage(+push) -> glove_shard_signal_staged -> glove_shard_wait_staged -> update -> finish_sync */
int glove_shard_wait_staged(const glove_step_args *args, void *stream);
int glove_shard_signal_staged(const glove_step_args *args, void *stream);
int glove_shard_finish_sync(const glove_step_args *args, const float *loss_scalars, void *stream);
int glove_shard_train_step(const glove_step_args *args, void *stream);
int glove_shard_pull_step(const glove_step_args *args, void *stream);
int glove_shard_set_peers(const glove_step_args *args, const void *const *peer_workspaces, int32_t n_peers, void *stream);
int glove_shard_stage_step(const glove_step_args *args, void *stream);
int glove_shard_pack_step(const glove_step_args *args, float *send_buf, void *stream);
int glove_shard_unpack_step(const glove_step_args *args, const float *recv_buf, void *stream);
/* Host copy of the request-list offsets of a whole plan: out[side][K][8][9] ints; the rows shard r needs from owner q in
 * batch k (for the work items of `side`) number out[side][k][r][q+1] - out[side][k][r][q].  Synchronises the stream. */
int glove_plan_need_info(const void *plan, int32_t K, int32_t B, int32_t *out, void *stream);
/* Shared plan construction (row-sharded tables): a plan of K steps of the GLOBAL batch is built by ONE rank
 * (glove_prepare_batches_sharded into peer-mapped memory) and every rank copies the slice that describes its own block of
 * segments -- offset tables, segment / triple / work-item / long-segment records, request lists of shard `shard` -- from
 * `src_plan` (the builder's buffer as mapped in this process) into the same offsets of `dst_plan` (a local buffer of
 * glove_plan_bytes(K, B)).  The step entry points of shard `shard` then run on `dst_plan` exactly as on a plan built
 * locally (same results bit for bit); per rank the cost of plan construction stops growing with the number of shards.
 * The caller orders the copy after the builder has finished (and the next build after every reader has). */
int glove_plan_pull_slice(void *dst_plan, const void *src_plan, int32_t K, int32_t B, int32_t n_shards, int32_t shard,
                          void *stream);
int glove_shard_update_step(const glove_step_args *args, float *loss_scalars, void *stream);
int glove_shard_finish_step(const glove_step_args *args, const float *loss_scalars, void *stream);
int64_t glove_step_snapshot_rows(int32_t B);
size_t glove_step_snapshot_offset(int32_t B, int32_t d, int32_t side);

/* Applies the missed zero-gradient Adam steps of every row up to (not including) step to_step (closed form, as the
 * stage of GLOVE_ADAM_REPLAY does).  Required before the tables are read from outside the step (eval, export,
 * checkpoint).  glove_flush_lazy_state_exact replays them step by step (GLOVE_ADAM_REPLAY_EXACT); calling it after
 * every step is the literal dense-sweep schedule of legacy Keras Adam. */
int glove_flush_lazy_state(float *table, int64_t V, int32_t d, int32_t optimizer, int32_t side, const float *alpha,
                           int32_t alpha_len, int32_t to_step, float beta1, float beta2, float epsilon, void *stream);
int glove_flush_lazy_state_exact(float *table, int64_t V, int32_t d, int32_t optimizer, int32_t side, const float *alpha,
                                 int32_t alpha_len, int32_t to_step, float beta1, float beta2, float epsilon, void *stream);

/* ---- EVAL: model_fn(mode=EVAL), RegressionHead metrics [ref src/models/estimator.py:87-92] -------------------- */
/* Forward-only pass over COO positions [first, first+count) in file order in batches of batch_size.  out: double
 * [n_batches][8] = {sum w*l, sum w, sum w*y, sum w*z, sum |R_i|^2, sum |C_j|^2, sum rb_i^2, sum cb_j^2} per batch
 * (logistic head: {sum p*softplus(-z), sum p, sum n*softplus(z), sum n, ...}).  workspace: glove_eval_workspace_bytes. */
size_t glove_eval_workspace_bytes(int64_t count, int32_t batch_size);
int glove_eval_loss(const float *row_table, const float *col_table, const glove_scalars *scalars, int32_t planes,
                    int32_t d, const int32_t *row, const int32_t *col, const float *colA, const float *colB,
                    int64_t first, int64_t count, int32_t batch_size, int32_t head, double *out, void *workspace,
                    size_t workspace_bytes, void *stream);

/* ---- PREDICT: cosine_similarity + tf.math.top_k [ref src/models/utils.py:12-19, src/models/model_utils.py:81-110] */
/* normalised bf16 copy of the row table for the tensor-core pass: out_bf16 [V_pad][Kp] (Kp = glove_topk_kpad(d), rows
 * >= V zero), inv_norm [V] = rsqrt(max(sum x^2, 1e-12)) in fp32. */
int32_t glove_topk_kpad(int32_t d);
int64_t glove_topk_vpad(int64_t V);
int glove_normalize_rows(const float *table, int64_t V, int32_t d, int32_t planes, void *out_bf16, float *inv_norm,
                         void *stream);
size_t glove_topk_workspace_bytes(int64_t V, int32_t d, int32_t n_queries, int32_t k);
/* For each query id q: top-k over all V rows of cosine(x_q, x_v) in fp32, sorted descending, ties -> lower id.
 * out_sim fp32 [n_queries][k], out_idx int32 [n_queries][k].  Candidates come from the tcgen05 bf16 pass over
 * norm_bf16 and are re-scored exactly in fp32 from the table. */
int glove_topk_cosine(const float *table, int64_t V, int32_t d, int32_t planes, const void *norm_bf16,
                      const float *inv_norm, const int32_t *query_ids, int32_t n_queries, int32_t k, float *out_sim,
                      int32_t *out_idx, void *workspace, size_t workspace_bytes, void *stream);
/* Same, with the query vectors taken from ANOTHER packed table (qtable, qplanes, its normalised bf16 copy qnorm_bf16;
 * query_ids index qtable): what a shard of a row-sharded table runs on the gathered query rows.  Candidate ids are rows
 * of `table`. */
int glove_topk_cosine_queries(const float *table, int64_t V, int32_t d, int32_t planes, const void *norm_bf16,
                              const float *inv_norm, const float *qtable, int32_t qplanes, const void *qnorm_bf16,
                              const int32_t *query_ids, int32_t n_queries, int32_t k, float *out_sim, int32_t *out_idx,
                              void *workspace, size_t workspace_bytes, void *stream);
/* k best of n_cand candidates per query (cand_idx < 0 = empty slot): descending similarity, ties -> lower id.  Last step
 * of a row-sharded top-k (every shard contributes the top-k of its rows with ids made global). */
int glove_topk_merge(const float *cand_sim, const int32_t *cand_idx, int32_t n_queries, int32_t n_cand, int32_t k,
                     float *out_sim, int32_t *out_idx, void *stream);
/* Diagnostics: number of queries of the last glove_topk_cosine call on `workspace` that failed the candidate guarantee
 * check and were recomputed by the exact scan (0 in the common case).  Synchronises. */
int glove_topk_flagged(const void *workspace, int64_t V, int32_t d, int32_t n_queries, int32_t k, int32_t *host_count,
                       void *stream);
/* exact fp32 CUDA-core reference implementation of the same contract (no tensor cores); used by tests and as the
 * fallback for shapes the tensor-core path does not cover */
int glove_topk_cosine_fp32(const float *table, int64_t V, int32_t d, int32_t planes, const float *inv_norm,
                           const int32_t *query_ids, int32_t n_queries, int32_t k, float *out_sim, int32_t *out_idx,
                           void *workspace, size_t workspace_bytes, void *stream);

/* ---- Intrinsic evaluation: word analogies and word-pair similarity over the row table --------------------------------
 * Conventions of Stanford GloVe eval/python/evaluate.py: rows are l2-normalised (here with the 1e-12 floor of
 * tf.math.l2_normalize, as the top-k), the question (a, b, c) -> d is answered by the best row outside {a, b, c} (only
 * those ids are excluded: a duplicate row of b under another id stays a candidate), ties -> lower id.
 *   GLOVE_ANALOGY_ADD (3CosAdd): cosine of x with q = b^ - a^ + c^, ranked by the cosine top-k (tensor-core candidate
 *     pass when norm_bf16 is given, exact fp32 scan when it is NULL) for k + 3 entries, then a, b, c dropped: exact,
 *     since the top-k outside three ids is a subset of the top-(k+3).
 *   GLOVE_ANALOGY_MUL (3CosMul, Levy & Goldberg 2014, "Linguistic Regularities in Sparse and Explicit Word
 *     Representations"): score = ((1+cos(x,b))/2 * (1+cos(x,c))/2) / ((1+cos(x,a))/2 + 1e-3), exact fp32 scan, in a
 *     fixed operation order (bit-identical from run to run).
 * Candidates are rows [0, V) of table (V may be smaller than the table: the most frequent words of a frequency-ordered
 * vocabulary); abc int32 [n][3] device, ids < V (checked by the caller); 1 <= k <= 29 and k + 3 <= V; out_score fp32 and
 * out_idx int32 [n][k], descending. inv_norm as glove_normalize_rows computes it for the table. */
enum { GLOVE_ANALOGY_ADD = 0, GLOVE_ANALOGY_MUL = 1 };
size_t glove_analogy_workspace_bytes(int64_t V, int32_t d, int32_t n_questions, int32_t k, int32_t method);
int glove_analogy_topk(const float *table, int64_t V, int32_t d, int32_t planes, const void *norm_bf16,
                       const float *inv_norm, const int32_t *abc, int32_t n_questions, int32_t method, int32_t k,
                       float *out_score, int32_t *out_idx, void *workspace, size_t workspace_bytes, void *stream);
/* out[i] = cosine of the rows pairs[2i] and pairs[2i+1] (int32 [n][2] device, ids < V), computed as the top-k computes
 * its similarities (the first row normalised as the query, the second through inv_norm): bit for bit the similarity the
 * top-k of the first row reports for the second. */
int glove_pair_cosine(const float *table, int64_t V, int32_t d, int32_t planes, const float *inv_norm,
                      const int32_t *pairs, int32_t n_pairs, float *out, void *stream);

/* ---- INGEST: interaction.csv text -> device COO (SURVEY 8 f.1) -----------------------------------------------------
 * Replaces tf.data make_csv_dataset(select_columns=...) [ref src/models/data_utils.py:4-26] and the per-step
 * StaticHashTable(TextFileInitializer(vocab.txt), default_value=0) lookup [ref src/models/model_utils.py:121-127,
 * src/models/estimator.py:26-28].  The caller uploads the file bytes (after the header record) chunk by chunk; every
 * chunk must start at a record boundary.  RFC-4180 quoting, "" escapes, \r\n and blank lines are handled on the
 * device; float columns are converted with ONE rounding, decimal text -> float32 (as DecodeCSV does), empty field -> 0. */
enum { GLOVE_CSV_TOKEN = 0, GLOVE_CSV_INT = 1, GLOVE_CSV_FLOAT = 2 };
typedef struct glove_csv_schema {
    int32_t n_cols;      /* fields per record (from the header) */
    int32_t column[4];   /* index of the row, col, colA, colB columns */
    int32_t kind[4];     /* row / col: GLOVE_CSV_TOKEN (string resolved through the vocab table, missing -> 0) or
                          * GLOVE_CSV_INT (a *_token_id column, checked against [0, n_vocab)); colA / colB: GLOVE_CSV_FLOAT */
} glove_csv_schema;
/* Device hash table over the lines of vocab.txt [ref src/data/text8.py:149-150]: vocab_bytes holds every line followed
 * by one '\n', vocab_off[v] .. vocab_off[v+1]-1 delimit line v (n_vocab + 1 offsets).  A duplicated line keeps the
 * lowest line number.  slots = glove_vocab_slots(n_vocab) int32 entries. */
int64_t glove_vocab_slots(int64_t n_vocab);
int glove_vocab_build(int32_t *table, int64_t slots, const uint8_t *vocab_bytes, const int64_t *vocab_off,
                      int64_t n_vocab, void *stream);
size_t glove_csv_workspace_bytes(int64_t nbytes);
/* Pass 1 over a chunk (text: device, 16-byte aligned): number of non-empty TERMINATED records -> *n_records_host.
 * Synchronises the stream.  glove_csv_parse on the same (text, nbytes, workspace) must follow. */
int glove_csv_index(const uint8_t *text, int64_t nbytes, void *workspace, size_t workspace_bytes,
                    int64_t *n_records_host, void *stream);
/* Pass 2 + parse: fills row/col/colA/colB[0 .. *n_rows_host) in file order.  capacity >= n_records + 1 entries in
 * row_ends (scratch) and the four outputs.  final_chunk: an unterminated last record counts; otherwise its bytes are
 * left to the next chunk (*consumed_host = bytes of this chunk that were parsed).  first_record numbers the records
 * in error messages.  Any malformed record fails the call (GLOVE_EINVAL, lowest record reported). Synchronises. */
int glove_csv_parse(const uint8_t *text, int64_t nbytes, int32_t final_chunk, void *workspace, size_t workspace_bytes,
                    const glove_csv_schema *schema, const int32_t *vocab_table, int64_t vocab_slots,
                    const uint8_t *vocab_bytes, const int64_t *vocab_off, int64_t n_vocab, int64_t *row_ends,
                    int32_t *row, int32_t *col, float *colA, float *colB, int64_t capacity, int64_t first_record,
                    int64_t *n_rows_host, int64_t *consumed_host, void *stream);
/* Host entry to the decimal -> float32 routine the parse kernel uses (one field, no blanks); for tests and tools. */
int glove_parse_float32(const char *text, int32_t n, float *out);

/* ---- WORD VECTORS: the GloVe text format <-> device float32 rows (glove_vectors.cu) -------------------------------
 * Format (DESIGN.md 3): one vector per line, "word v_1 ... v_d"; fields separated by runs of ASCII space / tab; trailing
 * blanks and a '\r' before the '\n' ignored; blank lines skipped; the LAST d fields are the numbers and the word is
 * everything before them with the separating blanks trimmed (words may contain spaces or look like numbers).  Numbers are
 * rounded once, decimal text -> float32 (glove_parse_float32); nan / inf and malformed numbers fail the call.  The optional
 * word2vec header "V d" and the choice of d (2 <= d <= 510) are the caller's business (they need the first line only).
 * Import: the caller uploads the file chunk by chunk (text: device, 16-byte aligned, every chunk starts at a line start),
 * glove_vectors_index counts its '\n', glove_vectors_parse (same text, nbytes and workspace) parses it.  Export: rows are
 * printed with the shortest decimal that parses back to the same float32 (glove_format_float32). */
/* n_lines = the count glove_vectors_index returned (0 for the index call itself), or the number of rows to format with
 * nbytes = 0. */
size_t glove_vectors_workspace_bytes(int64_t nbytes, int64_t n_lines);
/* Number of '\n' in the chunk -> *n_lines_host.  Synchronises the stream. */
int glove_vectors_index(const uint8_t *text, int64_t nbytes, void *workspace, size_t workspace_bytes, int64_t *n_lines_host,
                        void *stream);
/* Parses the non-blank lines of the chunk in order: row r of the chunk goes to out + r * ld (ld >= d floats, so that a
 * packed one-plane table, ld = glove_table_stride(d), is filled in place), its word to text[word_start[r] ..
 * + word_len[r]).  A row past row_capacity fails the call (a header's count).  final_chunk: an unterminated last line is
 * parsed; otherwise its bytes are left to the next chunk (*consumed_host = bytes of this chunk that were parsed).
 * first_line = 1-based file line of the chunk's first line (lines of padding in front count), for the error message,
 * which names the lowest offending line.
 * Synchronises. */
int glove_vectors_parse(const uint8_t *text, int64_t nbytes, int32_t final_chunk, int32_t d, int64_t n_lines,
                        void *workspace, size_t workspace_bytes, float *out, int64_t ld, int64_t row_capacity,
                        int64_t *word_start, int32_t *word_len, int64_t first_line, int64_t *n_rows_host,
                        int64_t *consumed_host, void *stream);
/* Export of n rows (rows: device fp32, leading dimension ld) with their words (words[word_off[r] .. word_off[r+1]), word_off
 * device int64 [n + 1]) as n lines "word v_1 ... v_d\n".  format_size computes the line offsets in the workspace
 * (glove_vectors_workspace_bytes(0, n)) and the text size (synchronises); format, on the same arguments and workspace,
 * writes the text (capacity >= that size; asynchronous after one read of the size). */
int glove_vectors_format_size(const float *rows, int64_t ld, int32_t d, int64_t n, const int64_t *word_off, void *workspace,
                              size_t workspace_bytes, int64_t *text_bytes_host, void *stream);
int glove_vectors_format(const float *rows, int64_t ld, int32_t d, int64_t n, const uint8_t *words, const int64_t *word_off,
                         void *workspace, size_t workspace_bytes, uint8_t *text, int64_t capacity, void *stream);
/* Host entry to the float32 -> shortest decimal routine the export kernel uses: out (capacity >= 16) receives *length
 * bytes, no terminating NUL.  For tests and tools. */
int glove_format_float32(float value, char *out, int32_t capacity, int32_t *length);

/* ---- TOKENS: corpus text -> token stream, the front half of the preprocessor (SURVEY 8 f.4) ------------------------
 * text8.split() [ref src/data/text8.py:47], Counter(text_tokens) [ref :62], token2id.get(token, 0) [ref :85-86].
 * Tokens are maximal runs of non-whitespace bytes (ASCII whitespace; the UTF-8 encodings of the other separators that
 * str.split() knows are refused with GLOVE_EUNSUPPORTED).  text: device, < 2^31 bytes per call. */
size_t glove_tokens_workspace_bytes(int64_t nbytes, int64_t n_tokens);
/* starts[i] / lens[i] of every token, in text order; *n_tokens_host is set even when it exceeds capacity.  Workspace:
 * glove_tokens_workspace_bytes(nbytes, 0).  Synchronises. */
int glove_tokens_scan(const uint8_t *text, int64_t nbytes, void *workspace, size_t workspace_bytes, int64_t *starts,
                      int32_t *lens, int64_t capacity, int64_t *n_tokens_host, void *stream);
/* Distinct tokens (radix sort of a 64-bit hash of the bytes, verified byte-wise: a collision fails the call): for each,
 * the start and length of its FIRST occurrence and its count; order = by hash.  Workspace:
 * glove_tokens_workspace_bytes(nbytes, n_tokens).  Synchronises. */
int glove_tokens_count(const uint8_t *text, int64_t nbytes, const int64_t *starts, int64_t n_tokens, void *workspace,
                       size_t workspace_bytes, int64_t *first_start, int32_t *first_len, int64_t *count, int64_t capacity,
                       int64_t *n_distinct_host, void *stream);
/* ids[i] = line of token i in the vocab table built by glove_vocab_build, missing -> 0.  Asynchronous. */
int glove_tokens_lookup(const uint8_t *text, const int64_t *starts, const int32_t *lens, int64_t n_tokens,
                        const int32_t *vocab_table, int64_t vocab_slots, const uint8_t *vocab_bytes, const int64_t *vocab_off,
                        int32_t *ids, void *stream);
/* Stanford GloVe's token stream (corpus.py, scheme "stanford").  glove_text_refused: the lowest offset in text[0, nbytes)
 * of a byte Stanford's tokenizer would glue into a token but glove_tokens_scan splits on (\v, \f, 0x1c-0x1f, a \r not
 * directly before \n; next_byte = the byte after the chunk, -1 at the end of the file), or -1.  scratch: 8 device
 * bytes; text 16-byte aligned.  Synchronises.
 * glove_tokens_stream: the in-vocabulary tokens among the n_tokens of glove_tokens_scan, in text order, as
 * out[j] = (segment << 32) | id (id = line of the vocab table, out-of-vocabulary tokens removed; segment =
 * segment_base + the number of '\n' bytes before the token, counted from text_begin, plus 1 when newline_before; uint32,
 * wrapping).  *last_segment_host: the segment of token n_tokens - 1, kept or not (the segment_base of the next chunk).
 * capacity >= n_tokens.  Workspace: glove_tokens_stream_workspace_bytes(n_tokens).  Synchronises. */
int glove_text_refused(const uint8_t *text, int64_t nbytes, int32_t next_byte, uint64_t *scratch, int64_t *first_host,
                       void *stream);
size_t glove_tokens_stream_workspace_bytes(int64_t n_tokens);
int glove_tokens_stream(const uint8_t *text, int64_t text_begin, const int64_t *starts, const int32_t *lens, int64_t n_tokens,
                        int32_t newline_before, uint32_t segment_base, const int32_t *vocab_table, int64_t vocab_slots,
                        const uint8_t *vocab_bytes, const int64_t *vocab_off, void *workspace, size_t workspace_bytes,
                        uint64_t *out, int64_t capacity, int64_t *n_out_host, uint32_t *last_segment_host, void *stream);

/* ---- PREPROCESS: token-id stream -> symmetric co-occurrence table with the GloVe columns (SURVEY 8 f.4) ------------
 * create_interaction_dataframe + create_glove_dataframe of the reference preprocessor [ref src/data/text8.py:84-139].
 * Partial tables are (keys u64[n] sorted unique, agg i64[2n] = {count, numer} per key) with numer = sum over the pairs of
 * lcm(1..context)/distance, i.e. the reference's sum of 1/distance carried exactly.  All pointers are device memory.
 * workspace: glove_cooc_workspace_bytes(n_items), n_items = the largest of n_positions*context (chunk), n_a+n_b (merge),
 * 2*n (finish).  Every call synchronises the stream. */
size_t glove_cooc_workspace_bytes(int64_t n_items);
/* Pairs (id[p], id[p+k]), p in [0, n_positions), k = 1..context, p + k < n_tokens (token_ids holds n_tokens >= n_positions
 * entries: the chunk plus its look-ahead), equal ids dropped [ref text8.py:90-95,98-102]. */
int glove_cooc_chunk(const int32_t *token_ids, int64_t n_positions, int64_t n_tokens, int32_t V, int32_t context,
                     void *workspace, size_t workspace_bytes, uint64_t *out_keys, int64_t *out_agg, int64_t capacity,
                     int64_t *n_unique_host, void *stream);
/* Union of two partial tables, summed per key.  capacity >= n_a + n_b. */
int glove_cooc_merge(const uint64_t *keys_a, const int64_t *agg_a, int64_t n_a, const uint64_t *keys_b, const int64_t *agg_b,
                     int64_t n_b, int32_t V, void *workspace, size_t workspace_bytes, uint64_t *out_keys, int64_t *out_agg,
                     int64_t capacity, int64_t *n_unique_host, void *stream);
/* Union with the transposed table [ref text8.py:105-110], count >= count_min [ref text8.py:129], columns
 * [ref text8.py:113-117,130-139]: value = numer / lcm (one rounding), neg_weight = vocab_count[row] * (vocab_count[col] /
 * total_tokens), glove_weight = clip((count/100)^0.75, 0, 1), glove_value = log(value).  Records come out in the order
 * of a keyed 64-bit hash of (row, col) (the reference uses Python's salted hash() of the token pair: a random order).
 * *n_out_host is set even when it exceeds capacity (the call then fails and can be repeated with larger outputs). */
int glove_cooc_finish(const uint64_t *keys, const int64_t *agg, int64_t n, int32_t V, int32_t context, int64_t count_min,
                      const int64_t *vocab_count, int64_t total_tokens, uint64_t order_key, void *workspace,
                      size_t workspace_bytes, int32_t *row, int32_t *col, int64_t *count, double *value, double *neg_weight,
                      double *glove_weight, double *glove_value, int64_t capacity, int64_t *n_out_host, void *stream);

/* Streamed preprocessing (glove_tensorflow_b200/corpus.py): the co-occurrence table split into 2^part_bits partitions by
 * the top bits of the record-order hash, each merged and finished on its own; taken in ascending order the partitions'
 * records are the record order of glove_cooc_finish.  glove_cooc_route writes both orientations of every entry of a
 * right-context table (keys, agg as from glove_cooc_chunk) grouped by partition: partition p is the next
 * part_count_host[p] entries of out_keys / out_agg (capacity >= 2n).  part_bits 0..12.  Synchronises. */
size_t glove_cooc_route_workspace_bytes(int64_t n, int32_t part_bits);
int glove_cooc_route(const uint64_t *keys, const int64_t *agg, int64_t n, int32_t V, uint64_t order_key, int32_t part_bits,
                     void *workspace, size_t workspace_bytes, uint64_t *out_keys, int64_t *out_agg, int64_t capacity,
                     int64_t *part_count_host, void *stream);
/* The Stanford GloVe scheme (cooccur's counting rules).  glove_cooc_chunk_stanford: tokens as from glove_tokens_stream;
 * for positions p < n_positions and k = 1..window (1..15) with p + k < n_tokens and both on one segment, the pair
 * (id[p], id[p + k]), self pairs included, with weight lcm(1..window) / k (distance_weighting) or 1; reduced as
 * glove_cooc_chunk.  glove_cooc_route_stanford: glove_cooc_route with both orientations (symmetric) or only (a, b);
 * capacity >= 2n or n.  glove_cooc_finish_stanford: glove_cooc_finish_sorted with count_min 1 and value = numer /
 * lcm(1..window) (distance_weighting) or count.  Same workspaces and synchronisation as their reference counterparts. */
int glove_cooc_chunk_stanford(const uint64_t *tokens, int64_t n_positions, int64_t n_tokens, int32_t V, int32_t window,
                              int32_t distance_weighting, void *workspace, size_t workspace_bytes, uint64_t *out_keys,
                              int64_t *out_agg, int64_t capacity, int64_t *n_unique_host, void *stream);
int glove_cooc_route_stanford(const uint64_t *keys, const int64_t *agg, int64_t n, int32_t V, uint64_t order_key,
                              int32_t part_bits, int32_t symmetric, void *workspace, size_t workspace_bytes, uint64_t *out_keys,
                              int64_t *out_agg, int64_t capacity, int64_t *part_count_host, void *stream);
int glove_cooc_finish_stanford(const uint64_t *keys, const int64_t *agg, int64_t n, int32_t V, int32_t window,
                               int32_t distance_weighting, const int64_t *vocab_count, int64_t total_tokens, uint64_t order_key,
                               void *workspace, size_t workspace_bytes, int32_t *row, int32_t *col, int64_t *count,
                               double *value, double *neg_weight, double *glove_weight, double *glove_value, int64_t capacity,
                               int64_t *n_out_host, void *stream);
/* glove_cooc_finish for a table that is already symmetric (one partition merged from routed entries): no transpose.
 * Workspace: glove_cooc_workspace_bytes(n). */
int glove_cooc_finish_sorted(const uint64_t *keys, const int64_t *agg, int64_t n, int32_t V, int32_t context, int64_t count_min,
                             const int64_t *vocab_count, int64_t total_tokens, uint64_t order_key, void *workspace,
                             size_t workspace_bytes, int32_t *row, int32_t *col, int64_t *count, double *value,
                             double *neg_weight, double *glove_weight, double *glove_value, int64_t capacity,
                             int64_t *n_out_host, void *stream);
/* Pass 1 of the streamed preprocessor: merges the n_chunk distinct tokens of one text chunk (first / first_len / count
 * as from glove_tokens_count; origin = byte offset of text[0] in the corpus) into the global table of distinct tokens
 * (g_*, n_global entries sorted by token hash; g_first = corpus byte offset of the first occurrence, g_off / g_len = the
 * token bytes in pool).  The merged table goes to o_* (capacity >= n_global + n_chunk suffices), new tokens append their
 * bytes to pool[pool_used ..]; *pool_used_host receives the new fill.  Equal hashes of different tokens fail with
 * GLOVE_EUNSUPPORTED.  Synchronises. */
size_t glove_vocab_merge_workspace_bytes(int64_t n_global, int64_t n_chunk);
int glove_vocab_merge(const uint8_t *text, int64_t origin, const int64_t *first, const int32_t *first_len, const int64_t *count,
                      int64_t n_chunk, const uint64_t *g_hash, const int64_t *g_count, const int64_t *g_first,
                      const int64_t *g_off, const int32_t *g_len, int64_t n_global, uint8_t *pool, int64_t pool_used,
                      int64_t pool_capacity, void *workspace, size_t workspace_bytes, uint64_t *o_hash, int64_t *o_count,
                      int64_t *o_first, int64_t *o_off, int32_t *o_len, int64_t capacity, int64_t *n_out_host,
                      int64_t *pool_used_host, void *stream);
/* interaction.csv lines of n finished records (the columns of glove_cooc_finish) in the reference's column order:
 * row_token_id,col_token_id,count,value,row_token,col_token,neg_weight,glove_weight,glove_value.  Token t is
 * token_bytes[token_off[t] .. token_off[t+1]), already quoted as the csv needs; float64 values print as repr(float).
 * glove_cooc_csv_size measures (synchronises), glove_cooc_csv_format (same columns and workspace) writes (asynchronous). */
size_t glove_cooc_csv_workspace_bytes(int64_t n_records);
int glove_cooc_csv_size(const int32_t *row, const int32_t *col, const int64_t *count, const double *value,
                        const double *neg_weight, const double *glove_weight, const double *glove_value, int64_t n,
                        const int64_t *token_off, void *workspace, size_t workspace_bytes, int64_t *text_bytes_host,
                        void *stream);
int glove_cooc_csv_format(const int32_t *row, const int32_t *col, const int64_t *count, const double *value,
                          const double *neg_weight, const double *glove_weight, const double *glove_value, int64_t n,
                          const uint8_t *token_bytes, const int64_t *token_off, void *workspace, size_t workspace_bytes,
                          uint8_t *text, int64_t capacity, void *stream);
/* Host entry to the float64 -> repr(float) routine the csv kernel uses: out (capacity >= 24) receives *length bytes, no
 * terminating NUL.  glove_format_float64_device runs the device build on n bit patterns (device memory): slot i of out
 * (24 bytes each) receives len[i] bytes.  Asynchronous.  For tests and tools. */
int glove_format_float64(double value, char *out, int32_t capacity, int32_t *length);
int glove_format_float64_device(const uint64_t *bits, int64_t n, char *out, int32_t *len, void *stream);

/* Stanford GloVe co-occurrence records (cooccurrence.bin / .shuf.bin, real = double): struct { int32 word1, word2;
 * float64 val; }, little-endian, 16 bytes, ids 1-based lines of the vocabulary.
 * glove_cooc_bin_parse: n records (device memory, 16-byte aligned; record i has the global 0-based index
 * first_record + i) -> row[i] = word1 - 1, col[i] = word2 - 1, target[i] = (float)log(val),
 * weight[i] = (float)(val >= x_max ? 1 : pow(val / x_max, alpha)), computed in float64.  A record with an id outside
 * 1..V or a val that is not finite and > 0 lowers *error (device word; all ones = none) to
 * global_index * 4 + GLOVE_CREC_BAD_*, so after the call it names the lowest bad record seen so far.  Asynchronous.
 * glove_cooc_bin_format: n finished records (row, col, value as from glove_cooc_finish*) -> records (16-byte aligned,
 * 16 n bytes) with ids + 1.  Asynchronous. */
#define GLOVE_CREC_BAD_WORD1 0
#define GLOVE_CREC_BAD_WORD2 1
#define GLOVE_CREC_BAD_VALUE 2
int glove_cooc_bin_parse(const void *records, int64_t n, int64_t first_record, int64_t V, double x_max, double alpha,
                         int32_t *row, int32_t *col, float *target, float *weight, unsigned long long *error, void *stream);
int glove_cooc_bin_format(const int32_t *row, const int32_t *col, const double *value, int64_t n, void *records,
                          void *stream);

/* Stanford GloVe's trainer (glove.c with one thread), exact on the GPU (DESIGN.md section 3).  State in glove.c's layout:
 * W and gradsq are 2V rows of d + 1 doubles (rows 0..V-1 word vectors, V..2V-1 context vectors, last element the bias).
 * glove_sgd_parse: like glove_cooc_bin_parse (same validation and error word), into the trainer's 24-byte records:
 * words[2i .. 2i+1] = {word1 - 1, word2 - 1}, lf[2i .. 2i+1] = {log(val), val > x_max ? 1 : pow(val / x_max, alpha)} in
 * float64 (words 8-byte, lf and records 16-byte aligned).  Asynchronous.
 * glove_sgd_links: prev[2j] = the last record before j with the same word1, prev[2j+1] the same for word2, -1 if none
 * (stable radix sort per side).  Asynchronous.
 * glove_sgd_init: W[i] = (u - 0.5) / d for the 2V(d+1) elements, u = (splitmix64(seed * 0xD1B54A32D192ED03 +
 * i * 0x9E3779B97F4A7C15) >> 11) * 2^-53.  Asynchronous.
 * glove_sgd_epoch: one pass over the n records in file order, exactly glove.c's recurrence (1 <= d <= 512).  done[n]
 * starts at zero and receives `epoch`, which must grow from call to call (1, 2, ...) on the same done array.  grid = 0:
 * every CTA that fits, else that many CTAs (any value gives the same bits).  *cost (device) receives the summed record
 * costs / n.  Synchronises; a dependency link that does not point backwards fails with GLOVE_EINVAL, a wait of about a
 * second with GLOVE_ECUDA.
 * glove_sgd_rows: out (float32, V + unk rows) = per word the row of a vectors file: model 0 = W row and W~ row with
 * biases (2d + 2 values), 1 = W (d values), 2 = W + W~ summed in float64 (d values); unk = 1 adds glove.c's <unk> row
 * from the per-element mean (each term divided by m, then summed) of the last m = min(100, V) rows.  Asynchronous. */
int glove_sgd_parse(const void *records, int64_t n, int64_t first_record, int64_t V, double x_max, double alpha,
                    int32_t *words, double *lf, unsigned long long *error, void *stream);
size_t glove_sgd_links_workspace_bytes(int64_t n);
int glove_sgd_links(const int32_t *words, int64_t n, int64_t V, int32_t *prev, void *workspace, size_t workspace_bytes,
                    void *stream);
int glove_sgd_init(double *W, int64_t V, int32_t d, uint64_t seed, void *stream);
size_t glove_sgd_epoch_workspace_bytes(int64_t n);
int glove_sgd_epoch(double *W, double *gradsq, int64_t V, int32_t d, const int32_t *words, const double *lf,
                    const int32_t *prev, int64_t n, double eta, double grad_clip, int32_t epoch, int32_t *done,
                    int32_t grid, void *workspace, size_t workspace_bytes, double *cost, void *stream);
int glove_sgd_rows(const double *W, int64_t V, int32_t d, int32_t model, int32_t unk, float *out, void *stream);

/* ---- HOST-buffer boundary (end to end): what a non-torch caller of the reference's training path would bind ----- */
/* Runs K TRAIN steps (K a multiple of args->plan_K, at most 4096) on K*B explicit triples held in HOST memory (pinned
 * recommended) and copies the K losses back to host_losses.  Internally a pipeline over the chunks of plan_K steps:
 * H2D + plan construction of chunk c+1 on a helper stream while the steps of chunk c run on `stream`, and (exact-replay
 * Adam) the catch-up of step s+1 on a second helper stream while step s runs (GLOVE_ADAM_REPLAY_EXACT only).  Device state (tables, scalars, plans,
 * workspaces) stays caller-owned: `plan` holds glove_host_plan_bytes(plan_K, B) bytes (two plans), `staging`
 * glove_host_staging_bytes(plan_K, B).  Synchronises the stream on entry and before returning. */
size_t glove_host_staging_bytes(int32_t plan_K, int32_t B);
size_t glove_host_plan_bytes(int32_t plan_K, int32_t B);
/* The helper streams and events of the pipeline live in a CALLER-OWNED handle (created on the current device): the
 * library keeps no process-global state, and two handles can drive two streams / devices concurrently. */
typedef struct glove_host_pipe glove_host_pipe;
int glove_host_pipe_create(glove_host_pipe **out);
int glove_host_pipe_destroy(glove_host_pipe *pipe);
int glove_train_steps_host(glove_host_pipe *pipe, const glove_step_args *args, void *plan, void *prepare_ws, size_t prepare_ws_bytes,
                           void *staging, size_t staging_bytes, const int32_t *host_row, const int32_t *host_col,
                           const float *host_colA, const float *host_colB, int32_t K, float *host_losses,
                           void *stream);

#ifdef __cplusplus
}
#endif
#endif /* GLOVE_B200_H_ */
