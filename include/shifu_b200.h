/*
 * shifu_b200.h - C ABI of the B200-native tabular-DNN train/score hot path.
 *
 * This is the drop-in boundary (SURVEY.md section 8b, seam B3).  The reference has no
 * native boundary of its own for this path: its arithmetic is reached through
 *   - Python  tf.Session.run          shifu-tensorflow-on-yarn/src/main/resources/ssgd_monitor.py:276,281
 *   - Java    TF-Java JNI (libtensorflow_jni 1.4.0)
 *                                     shifu-tensorflow-eval/src/main/java/ml/shifu/shifu/tensorflow/TensorflowModel.java:63-88,169
 * Every entry point below names the reference call it stands in for.  A JNI shim
 * (java/, csrc/jni_shim.c) and a ctypes binding (shifu-tensorflow_b200/_capi.py) sit on top of
 * exactly these symbols; see INTEGRATION.md.
 *
 * Conventions
 *   - every function returns 0 on success, a negative sb_status on failure;
 *     sb_last_error() returns a thread-local message for the last failure on this thread.
 *   - the caller owns all host buffers; the library owns all device memory.
 *   - one handle = one CUDA device.  Handles are not thread-safe except sb_model_score*,
 *     which is re-entrant (the reference scorer is called from many threads,
 *     TensorflowModel.java:53 has no lock).
 *   - flat parameter order is layer-major [W_0 (in x out, row-major), b_0, W_1, b_1, ..., W_out, b_out],
 *     i.e. the variables weight_hidden_layer{l}, biases_hidden_layer{l}, weight_shifu_output_0,
 *     biases_shifu_output_0 of ssgd_monitor.py:59,64,99-104,121.
 *   - there is NO CPU fallback: every compute entry point fails with SB_ERR_CUDA when no
 *     sm_100 device is present.
 */
#ifndef SHIFU_B200_H
#define SHIFU_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SB_MAX_HIDDEN 32

typedef enum {
  SB_OK = 0,
  SB_ERR_INVALID = -1,   /* bad argument                                   */
  SB_ERR_CUDA = -2,      /* CUDA / driver / no device                      */
  SB_ERR_NCCL = -3,
  SB_ERR_IO = -4,        /* SavedModel / checkpoint read or write          */
  SB_ERR_STATE = -5,     /* e.g. scoring before load (IllegalStateException in TensorflowModel.java:55-57) */
  SB_ERR_FORMAT = -6     /* unsupported graph / corrupt file               */
} sb_status;

/* get_activation_fun, ssgd_monitor.py:74-88 */
typedef enum { SB_ACT_SIGMOID = 0, SB_ACT_TANH = 1, SB_ACT_RELU = 2, SB_ACT_LEAKYRELU = 3, SB_ACT_NONE = -1 } sb_act;
/* SB_LOSS_MSE = tf.losses.mean_squared_error on the sigmoid output, SUM_BY_NONZERO_WEIGHTS
 * (ssgd_monitor.py:129) - the reference's loss.  SB_LOSS_SIGMOID_CE = BASELINE.json's wording. */
typedef enum { SB_LOSS_MSE = 0, SB_LOSS_SIGMOID_CE = 1 } sb_loss;
/* ADADELTA: ssgd_monitor.py:138; ADAM: ssgd.py:57; SGD: ssgd_monitor_bk.py:81; MOMENTUM: north star */
typedef enum { SB_OPT_ADADELTA = 0, SB_OPT_ADAM = 1, SB_OPT_SGD = 2, SB_OPT_MOMENTUM = 3 } sb_optimizer;
/* SB_PREC_FP32: fp32 operands and fp32 accumulation end to end (what TF-CPU computes) - parity mode (CUDA cores).
 * SB_PREC_BF16: bf16 operands on tcgen05 tensor cores, fp32 accumulation in TMEM, fp32 master
 *               weights and optimizer state - performance mode.
 * SB_PREC_FP32_TC: fp32-class accuracy ON the tensor cores: every fp32 operand value is split into three bf16 parts
 *               (v = p0 + p1 + p2, exact to ~2^-24), the six part products with i + j < 3 accumulate in fp32 TMEM.  Same
 *               kernels as SB_PREC_BF16 over a six times longer K axis; meets the fp32 tolerances (loss / gradients
 *               1e-4, scores 1e-5).  Parity mode that is not a CUDA-core program.
 * SB_PREC_BF16X2: two parts, three products (~2^-17 relative per product): half the cost of FP32_TC. */
typedef enum { SB_PREC_FP32 = 0, SB_PREC_BF16 = 1, SB_PREC_FP32_TC = 2, SB_PREC_BF16X2 = 3 } sb_precision;

typedef struct {
  int32_t n_features;              /* FEATURE_COUNT = len(SELECTED_COLUMN_NUMS), ssgd_monitor.py:43-44 */
  int32_t n_hidden;                /* train.params.NumHiddenLayers, ssgd_monitor.py:93                 */
  int32_t hidden[SB_MAX_HIDDEN];   /* train.params.NumHiddenNodes,  ssgd_monitor.py:94                 */
  int32_t acts[SB_MAX_HIDDEN];     /* train.params.ActivationFunc,  ssgd_monitor.py:95 (sb_act)        */
  int32_t loss;                    /* sb_loss                                                          */
  int32_t optimizer;               /* sb_optimizer                                                     */
  float learning_rate;             /* train.params.LearningRate, ssgd_monitor.py:133                   */
  float rho;                       /* Adadelta rho (TF default 0.95)                                   */
  float epsilon;                   /* Adadelta / Adam epsilon (TF default 1e-8)                        */
  float beta1, beta2;              /* Adam (TF defaults 0.9 / 0.999)                                   */
  float momentum;                  /* Momentum                                                         */
  int32_t max_batch;               /* largest mini-batch (rows) a step will be given                   */
  int32_t precision;               /* sb_precision                                                     */
} sb_net_desc;

typedef struct sb_trainer sb_trainer_t;
typedef struct sb_model sb_model_t;

/* ---- library ---- */
const char* sb_version(void);
const char* sb_last_error(void);
/* number of visible CUDA devices with compute capability 10.x; <0 on error */
int sb_device_count(void);
/* pinned host memory for callers that want true async H2D (JNI direct buffers) */
int sb_host_alloc(void** ptr, uint64_t bytes);
int sb_host_free(void* ptr);

/* ---- data-parallel rendezvous: replaces tf.train.Server/ClusterSpec (ssgd_monitor.py:152-166).
 * Rank 0 calls sb_nccl_unique_id and ships the 128 bytes to the other ranks by any means. ---- */
#define SB_NCCL_ID_BYTES 128
int sb_nccl_unique_id(void* out128);

/* ---- trainer: replaces model()+MonitoredTrainingSession of the worker branch
 * (ssgd_monitor.py:110-144, 251-257).  nccl_id may be NULL when world == 1. ---- */
int sb_trainer_create(const sb_net_desc* desc, int device, const void* nccl_id, int rank, int world,
                      sb_trainer_t** out);
/* (world > 1 with nccl_id == NULL: replicas driven by ONE process; they must be connected with
 * sb_trainer_set_peer_pointers before the first step, there is no NCCL fallback then.) */
int sb_trainer_destroy(sb_trainer_t* t);
/* Optional faster gradient exchange for ranks on one NVLink/NVSwitch node: a two-shot all-reduce kernel over CUDA-IPC
 * peer memory instead of NCCL.  Every rank exports its exchange buffer (64-byte cudaIpcMemHandle_t), the host
 * all-gathers the handles in rank order and hands the table to every rank.  Must be called on all ranks before the
 * next step; without it the exchange is ncclAllReduce. */
#define SB_IPC_HANDLE_BYTES 64
int sb_trainer_ipc_handle(sb_trainer_t* t, void* out64);
int sb_trainer_set_peer_handles(sb_trainer_t* t, const void* handles /* world x 64 bytes */, int32_t n_handles);
/* back to NCCL: unmap the peers (call on every rank when any rank failed to map, so that no rank runs the peer kernels) */
int sb_trainer_clear_peer_handles(sb_trainer_t* t);
/* The same peer table for trainers that live in ONE process (one host thread driving several GPUs, or several replicas
 * on one GPU in the tests): instead of IPC handles, pass every rank's exchange allocation (sb_trainer_exchange_base) as a
 * plain device pointer, in rank order; peer access between the devices is enabled here.  bases[own rank] is ignored. */
void* sb_trainer_exchange_base(sb_trainer_t* t);
int sb_trainer_set_peer_pointers(sb_trainer_t* t, void* const* bases, int32_t n);
int64_t sb_trainer_param_count(const sb_trainer_t* t);
/* variable init / restore (tf.initialize_all_variables + Saver.restore, ssgd_monitor.py:238,327) */
int sb_trainer_set_params(sb_trainer_t* t, const float* flat, int64_t n);
int sb_trainer_get_params(sb_trainer_t* t, float* flat, int64_t n);
/* xavier-uniform init on weights and biases (ssgd_monitor.py:59-68), seeded */
int sb_trainer_init_xavier(sb_trainer_t* t, uint64_t seed);
/* parity hook: the (all-reduced, mean over ranks) gradient the last step applied */
int sb_trainer_get_grads(sb_trainer_t* t, float* flat, int64_t n);

/* one sess.run([train_step, loss, global_step], feed_dict) (ssgd_monitor.py:272-276) in the
 * "clean" schedule: forward, loss, backward, gradient mean over ranks, one optimizer update.
 * X [rows, n_features] fp32 row-major, y [rows] (labels 0/1 as float), w [rows] sample weights
 * (NULL = all 1.0), all HOST memory.  loss_out (nullable) receives this rank's mini-batch loss. */
int sb_trainer_step(sb_trainer_t* t, const float* X, const float* y, const float* w, int32_t rows,
                    float* loss_out);

/* Wide+deep (BASELINE.json configs[3]; the reference only plumbs the numeric / categorical column lists,
 * TensorflowTaskExecutor.java:213-223, and has no sparse model - spec in oracle/wide_deep.py): the first hidden layer's
 * n_features = n_dense + n_onehot inputs are n_dense numeric columns followed by the one-hot expansion of n_cat categorical
 * columns.  A sparse step feeds the dense block Xd [rows, n_dense] and idx [rows, n_cat] (global one-hot column of each
 * categorical value, -1 = missing) and evaluates the one-hot block as an embedding gather (forward) / scatter-add
 * (gradient) - the SAME parameters, loss and update as sb_trainer_step on the materialised one-hot matrix. */
int sb_trainer_set_sparse(sb_trainer_t* t, int32_t n_dense, int32_t n_onehot, int32_t n_cat);
int sb_trainer_step_sparse(sb_trainer_t* t, const float* Xd, const int32_t* idx, const float* y, const float* w,
                           int32_t rows, float* loss_out);
int sb_trainer_predict_sparse(sb_trainer_t* t, const float* Xd, const int32_t* idx, int64_t rows, float* out);
int sb_trainer_eval_loss_sparse(sb_trainer_t* t, const float* Xd, const int32_t* idx, const float* y, const float* w,
                                int64_t rows, float* loss_out);

/* Same step, pipelined: returns as soon as the work is queued.  The H2D copy of this batch goes through a second
 * staging slot on a copy stream and overlaps the previous step's compute; the loss of the most recent step is read
 * with sb_trainer_last_loss (which waits).  X / y / w must be pinned (sb_host_alloc or equivalent) for the copy to be
 * truly asynchronous and must stay untouched until two further steps have been queued or sb_trainer_sync returned. */
int sb_trainer_step_async(sb_trainer_t* t, const float* X, const float* y, const float* w, int32_t rows);

/* Reference epoch-sync schedule (SyncReplicasOptimizer, ssgd_monitor.py:136-141): accumulate the
 * gradient of one mini-batch without updating; then apply the MEAN of the n accumulated
 * mini-batch gradients (averaged over ranks as well) as ONE optimizer update. */
int sb_trainer_accumulate(sb_trainer_t* t, const float* X, const float* y, const float* w, int32_t rows,
                          float* loss_out);
int sb_trainer_apply_accumulated(sb_trainer_t* t);     /* queued on the trainer's stream; sb_trainer_sync / get_params wait */
/* Same, with the divisor given explicitly: the update uses (sum over ranks of the locally accumulated gradients) /
 * total_pushes.  This is ConditionalAccumulator.take_grad(R) when ranks accepted different numbers of pushes (stale pushes
 * are dropped per worker, ssgd_monitor.py:136-141; the host-side token bookkeeping lives in trainer.py). */
int sb_trainer_apply_accumulated_mean(sb_trainer_t* t, int64_t total_pushes);

/* HBM-resident training set: load_data + np.array_split (ssgd_monitor.py:186-192) keep the whole
 * set in RAM and slice mini-batches from it; here the set lives in HBM and each step reads its
 * rows [row_offset, row_offset+rows) from there.  Calling load again replaces the set. */
int sb_trainer_load_dataset(sb_trainer_t* t, const float* X, const float* y, const float* w, int64_t n_rows);
/* Wide+deep resident set (after sb_trainer_set_sparse): Xd [n_rows, n_dense] fp32, idx [n_rows, n_cat] int32 (global one-hot
 * column, -1 = missing), y, w [n_rows]; HOST or DEVICE pointers, like sb_trainer_load_dataset.  Replaces any resident set;
 * sb_trainer_load_dataset replaces it in turn.  While it is loaded, the resident entry points (step_resident[_async],
 * run_resident, accumulate_resident, loss_resident, profile_step) run sparse steps.  SB_ERR_STATE before set_sparse,
 * SB_ERR_INVALID for an index outside [-1, n_onehot) (checked on the device at load; steps do no per-index host work). */
int sb_trainer_load_dataset_sparse(sb_trainer_t* t, const float* Xd, const int32_t* idx, const float* y, const float* w,
                                   int64_t n_rows);
/* (X / y / w of sb_trainer_load_dataset, sb_trainer_eval_loss and sb_trainer_predict may be HOST or DEVICE pointers on the
 * trainer's device: sb_text_parse_device hands the parsed set over without a host round trip.) */
int sb_trainer_step_resident(sb_trainer_t* t, int64_t row_offset, int32_t rows, float* loss_out);
/* same, but does not wait for the GPU: the loss of step i is readable after sb_trainer_sync */
int sb_trainer_step_resident_async(sb_trainer_t* t, int64_t row_offset, int32_t rows);
/* The inner loop of an epoch in one call (`for i in range(total_batch): sess.run(train_step)`, ssgd_monitor.py:268-276):
 * n_steps consecutive update steps over rows [row_offsets[i], row_offsets[i]+rows) of the resident set, identical to
 * n_steps calls of sb_trainer_step_resident_async.  Does not wait for the GPU; steps are replayed four per captured
 * graph, so the turn-around between two graphs is paid once per four steps. */
int sb_trainer_run_resident(sb_trainer_t* t, const int64_t* row_offsets, int32_t n_steps, int32_t rows);
int sb_trainer_accumulate_resident(sb_trainer_t* t, int64_t row_offset, int32_t rows, float* loss_out);
/* forward + loss only over resident rows, no gradient, no update: what a sess.run whose push the accumulator drops as stale
 * still reports (its loss), ssgd_monitor.py:276 */
int sb_trainer_loss_resident(sb_trainer_t* t, int64_t row_offset, int32_t rows, float* loss_out);
int sb_trainer_last_loss(sb_trainer_t* t, float* loss_out);
/* the loss curve: mini-batch loss of update steps first_step .. first_step + n - 1 (1-based global_step values; the last
 * 8192 steps are kept).  Every step's tail kernel posts its (loss sum, n_nz) into pinned host memory, so asynchronous
 * calls (sb_trainer_run_resident / _step_async) lose no per-step loss (`loss` fetched by every sess.run, ssgd_monitor.py:276).
 * Waits for the queued work. */
int sb_trainer_loss_history(sb_trainer_t* t, int64_t first_step, int32_t n, float* out);
int sb_trainer_sync(sb_trainer_t* t);
/* Make every replica identical to rank `root`: parameters, optimizer state and the step counter (ncclBroadcast on the
 * trainer's communicator).  The reference keeps ONE copy of the variables on the parameter servers, initialised or restored
 * by the chief only (ssgd_monitor.py:203-206, 251-257); replicas get the same effect by calling this on all ranks after
 * init / restore on the root.  No-op when world == 1. */
int sb_trainer_broadcast_state(sb_trainer_t* t, int32_t root);
/* cudaStream_t the trainer launches on (for CUDA-event timing by the caller) */
void* sb_trainer_stream(sb_trainer_t* t);
/* number of this library's kernels launched by one step at this batch size (bench.py's gpu_launches) */
int sb_trainer_kernels_per_step(sb_trainer_t* t, int32_t rows);

/* measurement hook: runs ONE training step over resident rows outside the CUDA graph with a CUDA event after
 * every kernel launch on the trainer's stream; ms[i] is the device time of launch i, names is a '\n'-joined list
 * (load_batch, gemm_fwd, out_layer, gemm_dw, gemm_da, [allreduce], optimizer).  The step is a real step
 * (parameters are updated). */
int sb_trainer_profile_step(sb_trainer_t* t, int64_t row_offset, int32_t rows, char* names, int32_t names_cap,
                            float* ms, int32_t cap, int32_t* n_out);

/* validation pass: sess.run([loss, global_step]) on the valid set (ssgd_monitor.py:281-284);
 * forward + loss only, any number of rows (processed in max_batch chunks with the reduction of
 * ONE big batch: sum w*(..)^2 over all rows / count of non-zero weights over all rows). */
int sb_trainer_eval_loss(sb_trainer_t* t, const float* X, const float* y, const float* w, int64_t rows,
                         float* loss_out);
/* forward only: sigmoid outputs for rows (host) */
int sb_trainer_predict(sb_trainer_t* t, const float* X, int64_t rows, float* out);

/* checkpoint / resume (MonitoredTrainingSession(checkpoint_dir=...), ssgd_monitor.py:251-257):
 * params + optimizer state + step counter as one flat blob. */
int sb_trainer_save_checkpoint(sb_trainer_t* t, const char* path);
int sb_trainer_load_checkpoint(sb_trainer_t* t, const char* path);
int64_t sb_trainer_global_step(const sb_trainer_t* t);

/* simple_save + export_generic_config (ssgd_monitor.py:457-490): SavedModel dir (saved_model.pb with
 * tag "serve", signature "serving_default" shifu_input_0 -> shifu_output_0, variables/ tensor bundle)
 * plus GenericModelConfig.json. */
int sb_trainer_export_savedmodel(sb_trainer_t* t, const char* export_dir);

/* ---- scorer: replaces TensorflowModel.init / compute (TensorflowModel.java:112-172, 53-94) ---- */
/* SavedModelBundle.load(modelPath, tags) + feed/fetch by op name */
int sb_model_load(const char* saved_model_dir, const char* input_name, const char* output_name,
                  const char* tag, int device, int precision, sb_model_t** out);
/* build directly from a topology + flat parameters (no file) */
int sb_model_create(const sb_net_desc* desc, const float* flat_params, int64_t n, int device, sb_model_t** out);
int sb_model_destroy(sb_model_t* m);
int32_t sb_model_n_features(const sb_model_t* m);
int32_t sb_model_n_layers(const sb_model_t* m);
/* batched compute(): X [rows, n_features] fp32 host -> out [rows] fp32 host */
int sb_model_score(sb_model_t* m, const float* X, int64_t rows, float* out);
/* compute(MLData): one row of doubles -> double (double->float cast at TensorflowModel.java:64-68) */
int sb_model_score_row_f64(sb_model_t* m, const double* row, int32_t n, double* out);
/* device-resident scoring (X, out are DEVICE pointers on the model's device), asynchronous on the
 * model's stream; sb_model_sync waits. */
int sb_model_score_device(sb_model_t* m, const float* dX, int64_t rows, float* dOut);
int sb_model_sync(sb_model_t* m);
void* sb_model_stream(sb_model_t* m);

/* ---- text ingest: the per-cell float() loop of load_data (ssgd_monitor.py:387-419) on the GPU ----
 * text: the gunzipped, delim-separated lines (must end with '\n'), HOST memory.  col_map[c] gives the role of text
 * column c: >= 0 feature index (into X [rows, n_feat] row-major), SB_COL_TARGET, SB_COL_WEIGHT, SB_COL_SKIP; columns
 * >= n_map are skipped.  y <- float(target cell); w <- weight cell with "negative -> 1.0", 1.0 when the line has no
 * weight column.  Every value is float32(float64(text)) exactly as numpy feeds the reference's fp32 placeholders.
 * Cells the exact fast path declines (> 15-19 significant digits, |exp| > 22, nan/inf, malformed) are NOT written:
 * they are listed in flags[0..min(n_flags, flag_cap)) for the caller to resolve with its own float(); slot -100 marks
 * a line whose number of feature cells / target cell is wrong. */
#define SB_COL_SKIP (-1)
#define SB_COL_TARGET (-2)
#define SB_COL_WEIGHT (-3)
typedef struct { int64_t row; int32_t slot; int32_t len; int64_t offset; } sb_cell_flag;
int sb_text_parse(const char* text, int64_t n_bytes, char delim, const int32_t* col_map, int32_t n_map, int32_t n_feat,
                  float* X, float* y, float* w, int64_t max_rows, int64_t* n_rows_out, sb_cell_flag* flags,
                  int64_t flag_cap, int64_t* n_flags_out, int device);
/* The same parse with the result left ON THE DEVICE: *dX [rows, n_feat], *dy, *dw are cudaMalloc'ed by the library (release
 * with sb_device_free) and go straight into sb_trainer_load_dataset / sb_trainer_eval_loss; only the flag list (cells for
 * the caller's float(), patched in with sb_device_patch_f32) and 4 bytes per row (weights, for the n_nz prefix counts) ever
 * reach the host.  kernel_ms_out (nullable): device time of the three parsing kernels (HBM-bound: text read twice for the
 * line index, once for the cells; X written once) - bench.py's `ingest` roofline. */
int sb_text_parse_device(const char* text, int64_t n_bytes, char delim, const int32_t* col_map, int32_t n_map, int32_t n_feat,
                         float** dX, float** dy, float** dw, int64_t* n_rows_out, sb_cell_flag* flags, int64_t flag_cap,
                         int64_t* n_flags_out, int device, float* kernel_ms_out);
int sb_device_alloc_f32(float** out, int64_t n, int device);
int sb_device_free(void* p);
int sb_device_patch_f32(float* d_base, int64_t index, float value);
int sb_device_read_f32(const float* d_src, int64_t n, float* host_out);
/* d_dst[i, :] = d_src[rows_host[i], :] - the train / valid split of the parsed set (the Bernoulli coins of
 * ssgd_monitor.py:396 are drawn on the host from the caller's RNG; only the row indices travel) */
int sb_device_gather_rows(const float* d_src, int32_t n_cols, const int64_t* rows_host, int64_t n, float* d_dst, int device);

/* test hook: the same parsing state machine run on the host (CPU unit tests of the number parser; not a product path) */
int sb_debug_text_parse_host(const char* text, int64_t n_bytes, char delim, const int32_t* col_map, int32_t n_map,
                             int32_t n_feat, float* X, float* y, float* w, int64_t max_rows, int64_t* n_rows_out,
                             sb_cell_flag* flags, int64_t flag_cap, int64_t* n_flags_out);

/* ---- file-format helpers used by the host mirrors and tests ---- */
/* write a SavedModel for an arbitrary MLP (host only, no GPU needed) */
int sb_savedmodel_write(const char* export_dir, const sb_net_desc* desc, const float* flat_params, int64_t n);
/* parse a SavedModel into topology + flat parameters (host only).  flat may be NULL to query n_params. */
int sb_savedmodel_read(const char* saved_model_dir, const char* input_name, const char* output_name,
                       const char* tag, sb_net_desc* desc_out, int32_t* out_act, float* flat, int64_t flat_cap,
                       int64_t* n_params);

/* ---- kernel-level test hooks (parity tests of single kernels through the C ABI) ---- */
/* D[M,N] = A[M,K] * B[N,K]^T on the tcgen05 path: A, B are fp32 host arrays that are rounded to
 * bf16 on the device; D fp32 host.  split_k >= 1. */
int sb_debug_gemm_bf16(const float* A, const float* B, float* D, int32_t M, int32_t N, int32_t K,
                       int32_t split_k, int device);
/* same with explicit operand layouts: a_mn = 0: A is [M,K] (K-major), 1: A is [K,M] (MN-major); b_mn likewise for
 * B ([N,K] or [K,N]).  Instantiated combinations: (0,0) dA GEMM, (0,1) forward GEMM, (1,1) dW GEMM. */
int sb_debug_gemm_bf16_ex(const float* A, const float* B, float* D, int32_t M, int32_t N, int32_t K,
                          int32_t split_k, int32_t a_mn, int32_t b_mn, int device);
/* same, forcing the tile configuration: cfg_cg = 1 (one CTA per 128 x cfg_bn tile, cfg_bn 64|128) or 2 (CTA pair per
 * 256 x cfg_bn tile, tcgen05 cta_group::2, cfg_bn 128|256); cfg_cg = 0 lets the planner choose. */
int sb_debug_gemm_bf16_cfg(const float* A, const float* B, float* D, int32_t M, int32_t N, int32_t K,
                           int32_t split_k, int32_t a_mn, int32_t b_mn, int32_t cfg_cg, int32_t cfg_bn, int device);

/* D = A B^T with every fp32 operand value held as np bf16 parts (np = 2: three part products, 3: six; see sb_precision):
 * the tensor-core parity GEMM behind SB_PREC_FP32_TC / SB_PREC_BF16X2. */
int sb_debug_gemm_split(const float* A, const float* B, float* D, int32_t M, int32_t N, int32_t K, int32_t np, int device);

/* micro-benchmark of one tile configuration: average device milliseconds per launch over `iters` back-to-back launches
 * (CUDA events on the launching stream, operands L2-warm) */
/* Timeline of the last step (trainer created with SB_STEP_TRACE=1 in the environment): for each GEMM launch of the
 * step, 16 %globaltimer stamps (ns) of its CTA 0: [0] entry, [1] setup done, [2] dependencies resolved, [3] first TMA
 * issued, [4] first stage landed, [5] MMAs of the first tile issued, [6] first accumulator complete, [7] first
 * epilogue done, [8] exit.  names = comma-separated kernel roles.  Measurement aid; no reference counterpart. */
int sb_debug_step_trace(sb_trainer_t* t, uint64_t* stamps, int32_t cap_kernels, char* names, int32_t names_cap, int32_t* n_kernels);
int sb_debug_gemm_bench(const float* A, const float* B, float* D, int32_t M, int32_t N, int32_t K, int32_t split_k,
                        int32_t a_mn, int32_t b_mn, int32_t cfg_cg, int32_t cfg_bn, int device, int32_t iters,
                        float* ms_out);

#ifdef __cplusplus
}
#endif
#endif /* SHIFU_B200_H */
