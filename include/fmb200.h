/*
 * fmb200.h -- C ABI of libfmb200.so, the B200 (sm_100a) implementation of the FM-family training
 * hot path of haan6/fm-for-online-recommendation.
 *
 * The reference has no FFI layer: its hot path is the Python method surface of
 * models/models_online_deep/*.py and models/models_online/*.py (SURVEY.md section 8b).  Each entry
 * point below names the reference code (file:line, relative to the reference root) it replaces.
 * INTEGRATION.md shows the ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *   - plain pointers and sizes only; `dev` pointers are CUDA device pointers, `host` pointers are
 *     host memory.  Buffers are caller-owned unless they belong to a session handle.
 *   - every function that launches work takes a cudaStream_t and is asynchronous on it, except the
 *     `*_host` entry points, which return after their result has been copied back.
 *   - return value: 0 = ok, <0 = error (FMB_ERR_*); fmb_last_error() returns a thread-local
 *     message.  No exceptions cross the boundary.
 *   - packed parameter table: float[R][rowp], rowp = fmb_rowp(k) = round_up(k+1, 16) (64-byte aligned rows); row r holds
 *     second_order_embeddings row (k floats), then the first_order_embeddings weight, then zero
 *     padding.  R = sum of feature_sizes; global row id = field offset + per-field id.
 *   - S and gvec row pitch: kp4 = fmb_kp4(k) = round_up(k, 4).
 */
#ifndef FMB200_H
#define FMB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* fmb_stream_t; /* == cudaStream_t */
typedef struct fmb_session fmb_session;

#define FMB_OK 0
#define FMB_ERR_ARG (-1)
#define FMB_ERR_CUDA (-2)
#define FMB_ERR_WS (-3)

/* update rules applied to touched rows / dense parameters */
#define FMB_UPDATE_ADAM1 0 /* torch.optim.Adam re-created every call => first-step sign update
                              (fm_adam.py:60,68; SURVEY.md A12) -- the reference behaviour */
#define FMB_UPDATE_SGD 1   /* p -= lr * g (legacy notebooks' torch.optim.SGD; SURVEY.md 8f.4) */
#define FMB_UPDATE_FTRL 2  /* per-coordinate FTRL-Proximal, FM-only steps (fmb_ftrl_t below) */
#define FMB_UPDATE_ADAGRAD 3 /* torch.optim.Adagrad with persistent per-coordinate sums (fmb_adagrad_t below) */
#define FMB_UPDATE_SPARSE_ADAM 4 /* torch.optim.SparseAdam on the tables, torch.optim.Adam on the bias and the tower,
                                    moments kept across calls (fmb_sparse_adam_t below) */

/* loss variants (SURVEY.md A6) */
#define FMB_LOSS_BCE_LOGITS 0         /* F.binary_cross_entropy_with_logits(z, y) */
#define FMB_LOSS_BCE_LOGITS_OF_SIG 1  /* F.binary_cross_entropy_with_logits(sigmoid(z), y) */

/* ---- library identity / errors -------------------------------------------------------------- */
int fmb_version(void);
const char* fmb_last_error(void);
int fmb_device_count(void); /* 0 when no usable GPU: callers must fail, there is no CPU path */
int fmb_rowp(int k);
int fmb_kp4(int k);

/* ---- A1-A3: first_order / second_order / forward_fm ------------------------------------------
 * replaces deepfm_adam.py:46-77 (= nfm_adam.py:45-76, deepfm_onn.py:55-86, nfm_onn.py:57-88,
 * fm_adam.py:34-54).  ids [B,F] int32 global row ids; xv [B,F] or NULL (all ones); bias [1].
 * Outputs (each nullable): first [B,F], S [B,kp4] (sum_f e_f), bi [B,k] (0.5*(S^2 - Q)),
 * sum_first [B], z [B] = (sum_first + sum_j bi) + bias.  When y [B] is non-NULL the loss variant
 * `loss_kind` is evaluated on z as well: delta [B] = dLoss/dz, lossv [B] = per-sample loss. */
int fmb_fm_forward(const int32_t* ids_dev, const float* xv_dev, const float* table_dev, const float* bias_dev,
                   int B, int F, int k, float* first_dev, float* S_dev, float* bi_dev, float* sum_first_dev,
                   float* z_dev, const float* y_dev, int loss_kind, float* delta_dev, float* lossv_dev,
                   fmb_stream_t stream);

/* ---- A6: loss + gradient on the logit (fm_adam.py:63-67, :77-81) ------------------------------- */
int fmb_loss_delta(int loss_kind, const float* z_dev, const float* y_dev, int B, float* delta_dev,
                   float* lossv_dev, fmb_stream_t stream);
/* ---- AFM (SURVEY.md 8f.3; csrc/afm.cu): the reference's afm_adam.py cannot run (afm_adam.py:67,69,121-123), so the model
 * is the AFM paper's (Xiao et al. 2017, eq. 8) with the reference's parameter set (afm_adam.py:34-41); checked against
 * oracle/afm.py.  fmb_afm_step: forward (+ backward when delta_dev != NULL: loss gradient, per-sample dense gradients, per-entry
 * embedding gradients staged in ws at their sorted positions); fmb_afm_dense_update: batch sum + update of W | c | H | P;
 * fmb_fm_backward_runs_all: the FM run kernel over every run (rows hit once included) sums and applies the staged gradients. */
size_t fmb_afm_dense_floats(int k, int A);
int fmb_afm_step(const int32_t* ids_dev, const float* xv_dev, const float* y_dev, const uint32_t* posflag_dev,
                 const float* table_dev, const float* bias_dev, const float* W_dev, const float* c_dev, const float* H_dev,
                 const float* P_dev, const unsigned char* pair_i_dev, const unsigned char* pair_j_dev, int B, int F, int k,
                 int A, int loss_kind, float* z_dev, float* delta_dev, float* lossv_dev, float* dense_g_dev, void* ws_dev,
                 size_t ws_bytes, fmb_stream_t stream);
int fmb_afm_dense_update(const float* dense_g_dev, int B, int k, int A, float* W_dev, float* c_dev, float* H_dev,
                         float* P_dev, float lr, int mode, float* grads_out_dev, fmb_stream_t stream);
int fmb_fm_backward_runs_all(const int32_t* sorted_keys_dev, int64_t N, float* table_dev, int F, int k, float lr, int mode,
                             void* ws_dev, size_t ws_bytes, fmb_stream_t stream);

/* ---- RRF_Online (RRF_Online.py:70-187; SURVEY.md 8f.3): persistent fp64 kernel, one CTA walks the stream in order.
 * gamma_dev [d] (log scale) and w_dev [2D] are updated in place; preds_dev [N] / nvalid_dev: predictions of the samples whose
 * score was not NaN (the reference skips the others).  task 0 = 'reg' (l2 loss), 1 = 'cls' (logit loss). */
int fmb_rrf_run(const double* X_dev, const double* Y_dev, int N, int d, int D, int task, double lr_w, double lr_gamma,
                double* gamma_dev, double* w_dev, const double* eps_dev, double* preds_dev, int* nvalid_dev,
                fmb_stream_t stream);

/* ---- device-resident input pipeline (SURVEY.md 8f.1; csrc/dataset.cu) ------------------------------------------
 * fmb_dataset_encode_ids: per-field local ids (the int64 LongTensor of deepfm_adam.py:47) -> global int32 row ids, with
 *   nn.Embedding's range check (*err_dev = 1 on an id outside [0, feature_sizes[f])); field_off_dev int32 [F+1].
 * fmb_dataset_take: dst row i = src row index_dev[i] -- the batch builders of utils/data_preprocess.py:154-264 and the
 *   balance_* functions (:46-82, :120-151), which append one Python list per sample; xv / y may be NULL; pos_count_dev
 *   (nullable, zeroed by the caller) counts labels == 1 (ratio_list); *err_dev = 1 on an index outside [0, n_src).
 * fmb_dict_encode_first_seen: read_svm_file's vocabulary build (utils/data_preprocess.py:100-108, `list.index` per cell):
 *   codes_dev [N,d] = index of X[i,c] among column c's distinct values in order of first appearance, sizes_dev [d] = their
 *   number (feature_sizes); *err_dev = 2 when X holds a NaN. */
int fmb_dataset_encode_ids(const int64_t* local_dev, int64_t n, int F, const int32_t* field_off_dev, int32_t* ids_dev,
                           int* err_dev, fmb_stream_t stream);
int fmb_dataset_take(const int32_t* ids_src_dev, const float* xv_src_dev, const float* y_src_dev, int F, int64_t n_src,
                     const int64_t* index_dev, int64_t n, int32_t* ids_dst_dev, float* xv_dst_dev, float* y_dst_dev,
                     int32_t* pos_count_dev, int* err_dev, fmb_stream_t stream);
size_t fmb_dict_encode_workspace_bytes(int64_t N, int d);
int fmb_dict_encode_first_seen(const double* X_dev, int64_t N, int d, int32_t* codes_dev, int32_t* sizes_dev, int* err_dev,
                               void* ws_dev, size_t ws_bytes, fmb_stream_t stream);

/* ---- metrics on the device (SURVEY.md 8f.2; csrc/metrics.cu) -------------------------------------------------
 * running curves of utils/metric_manager.py:7-29 (fp64, sequential accumulation like the Python loops), confusion
 * counts of fm_adam.py:101-111 for a batch of predictions, exact ROC AUC ingredients (pair counts), torch.sigmoid of
 * a logit vector (predict_proba). */
int fmb_metric_regression(const double* pred_dev, const double* real_dev, int64_t n, double* out_dev /*[n+1]*/,
                          fmb_stream_t stream);
int fmb_metric_classification(const double* pred_dev, const double* real_dev, int64_t n, double* metric_dev,
                              double* acc_dev, fmb_stream_t stream);
int fmb_confusion(const uint8_t* pred_dev, const float* y_dev, int64_t n, unsigned long long* conf_dev /*tp,fp,tn,fn*/,
                  fmb_stream_t stream);
int fmb_auc_pairs(const float* scores_dev, const float* labels_dev, int64_t n, unsigned long long* counts_dev,
                  fmb_stream_t stream);
int fmb_sigmoid(const float* z_dev, int n, float* p_dev, fmb_stream_t stream);

/* element-wise ATen mirrors (torch 2.11 CPU arithmetic restated on the device, csrc/fmb_aten_math.cuh):
 * op 0 torch.sigmoid of element i of a contiguous [n] tensor (fm_adam.py:80,86), 1 at::log_sigmoid (inside
 * F.binary_cross_entropy_with_logits, fm_adam.py:65), 2 Tensor.sqrt as torch.optim.Adam calls it (fm_adam.py:68),
 * 3 glibc expf.  Exported so that parity tests can sweep them against the oracle. */
int fmb_math_eval(int op, const float* x_dev, float* y_dev, int64_t n, fmb_stream_t stream);
/* sum in ATen's CPU order (loss.mean(), bias gradient): out[0] = sum(x[0:n]) */
int fmb_sum_aten(const float* x_dev, int64_t n, float* out_dev, fmb_stream_t stream);
/* optimizer.step() on dense parameters (bias, hidden_layers): fm_adam.py:68 */
int fmb_update_dense(float* p_dev, const float* g_dev, int64_t n, float lr, int mode, fmb_stream_t stream);
/* _ex: update mode 3 (Adagrad) with the parameters' sums sums_dev [n] (read and written; NULL in the other modes) */
int fmb_update_dense_ex(float* p_dev, const float* g_dev, int64_t n, float lr, int mode, float* sums_dev, float eps,
                        fmb_stream_t stream);
/* bias step from sum(delta) and mean loss; bias_dev / loss_out_dev nullable */
int fmb_finish_step(const float* delta_dev, const float* lossv_dev, int B, float* bias_dev, float lr, int mode,
                    float* loss_out_dev, fmb_stream_t stream);

/* ---- deterministic sort by row id + segments (replaces the implicit ordering of torch's CPU
 * embedding_dense_backward; SURVEY.md A6/A12) -------------------------------------------------- */
size_t fmb_sort_workspace_bytes(int64_t N);
int fmb_sort_segment(const int32_t* keys_dev, int64_t N, int key_bits, void* ws_dev, size_t ws_bytes,
                     int32_t* sorted_keys_dev, int32_t* perm_dev, int32_t* seg_start_dev /*[N+1], nullable*/,
                     int32_t* nseg_dev /*[1], nullable*/, fmb_stream_t stream);

/* fast path for ids laid out [B,F] with column f holding field f (field_off_dev [F+1]): one CTA per
 * field sorts its column in shared memory; output identical to fmb_sort_segment on the flat matrix */
int fmb_sort_fields_max_batch(void);
int fmb_sort_fields(const int32_t* ids_dev, int B, int F, const int32_t* field_off_dev, int32_t* sorted_keys_dev,
                    int32_t* perm_dev, fmb_stream_t stream);
/* Run list: what the sort hands to the run kernel of the FM step (round 2).  One entry of 4 int32 per run of >= 2 equal
 * sorted keys: {first sorted position, key, entries of the run among its first 32 positions (2..32), 1 if the run has
 * at least 128 entries else 0}; entries_dev is
 * [nseg][seg_cap][4], seg_count_dev [2*nseg]: segment g holds seg_count_dev[g] runs of fewer than 128 entries from its
 * start upwards and seg_count_dev[nseg + g] longer runs from its end downwards, in any order (one segment per producer
 * CTA: no global counter, nothing to zero).  fmb_runlist_shape gives the shape fmb_sort_fields_ex fills for a batch. */
typedef struct fmb_runlist_t { int32_t* entries_dev; uint32_t* seg_count_dev; int nseg, seg_cap; } fmb_runlist_t;
void fmb_runlist_shape(int B, int F, int* nseg, int* seg_cap);
/* _ex: the sort kernels also write what the FM step of the NEXT section consumes, saving a kernel behind the sort:
 * posflag_dev [B*F] (as fmb_pos_flags, nullable) and the run list rl (nullable).  flags & FMB_SORT_SPARSE_OK (needs
 * posflag_dev): fields with >= 16*B rows are not sorted at all -- a shared-memory hash pass finds the entries whose row is
 * hit more than once; sorted_keys_dev / perm_dev then hold only those entries, in (key, sample) order at the head of the
 * field's range [f*B, (f+1)*B), sorted_keys_dev is -1 behind them, perm_dev undefined there; posflag_dev of the other
 * entries of those fields is NOT written: the caller clears posflag_dev (cudaMemsetAsync) in front of the call.  That is
 * all the FM step reads (rows hit once are updated inside fmb_fm_step_fused and their position is never used). */
#define FMB_SORT_SPARSE_OK 1
int64_t fmb_sort_fields_sparse_min_rows(int B);   /* rows a field needs to skip its sort at batch B; 0 = never at this B */
int fmb_sort_fields_ex(const int32_t* ids_dev, int B, int F, const int32_t* field_off_dev, int32_t* sorted_keys_dev,
                       int32_t* perm_dev, uint32_t* posflag_dev, const fmb_runlist_t* rl, int flags, fmb_stream_t stream);

/* ---- A1-A3 + A6 fused: the FM-only step with every row read once (csrc/fm_step.cu) ----------------
 * replaces forward_fm + F.binary_cross_entropy_with_logits + loss.backward() + optimizer.step() of
 * fm_adam.py:56-82 (and update_embedding of the other four classes) in three launches:
 *   fmb_pos_flags        per entry: its position in the stable sort | "row hit more than once" flag
 *   fmb_fm_step_fused    gather, logit, loss, gradient; rows hit once are updated from the copy in shared memory,
 *                        the other entries stage their contribution at their sorted position in `ws`
 *   fmb_fm_backward_runs sums every run of >= 2 equal sorted keys in sample order (torch's CPU
 *                        embedding_dense_backward order) and updates those rows
 * followed by fmb_finish_step (bias step, mean loss) on delta/lossv.  ws: fmb_bwd_workspace_bytes(B*F, k). */
/* update mode 2: per-coordinate FTRL-Proximal (z, n, w with L1/L2; McMahan et al. 2013 -- the update BASELINE.json's
 * north_star names; the reference's FM_FTRL.py:76-80 is the linearised form without n and lives in fmb_ftrl_fm_run).
 * zn_dev [R][2][rowp] holds the z and n sub-rows of every packed table row, bias_zn_dev [2] those of the bias.  The _ex
 * entry points are the plain ones plus this state (NULL unless mode == 2); algorithmic bytes grow by 16F(k+1) per sample. */
typedef struct fmb_ftrl_t { float* zn_dev; float* bias_zn_dev; float beta, l1, l2; } fmb_ftrl_t;
/* update mode 3: torch.optim.Adagrad(lr = the step's lr, lr_decay = 0, weight_decay = 0, eps,
 * initial_accumulator_value = the caller's fill of the sums), one optimizer kept across calls.  Per coordinate, in the
 * order torch's CPU _single_tensor_adagrad rounds it:  s' = fma(g, g, s);  p' = p + (-lr * g) / (sqrt(s') + eps).
 * A zero gradient leaves p and s as they are, so updating only the rows a batch hits is the dense optimizer.
 * sums_dev [R][rowp]: row r's sums at row r's offsets of the packed table (padding columns are never written);
 * bias_sum_dev [1]; mlp_sums_dev [fmb_mlp_numel] (tower fit and fmb_online_deep_run_ex, NULL for FM-only steps).
 * Entry points with a state slot (fmb_fm_step_fused_ex, fmb_fm_backward_runs_ex / _list, fmb_finish_step_ex) take it
 * there in mode 3: pass (const fmb_ftrl_t*)&adagrad.  Algorithmic bytes of the FM step grow by 8F(k+1) per sample.
 * The row-sharded steps take each rank's shard of the sums (fmb_shard3_step_ex); the shard2 path, AFM and
 * fmb_fm_backward_runs_all reject mode 3. */
typedef struct fmb_adagrad_t { float* sums_dev; float* bias_sum_dev; float* mlp_sums_dev; float eps; } fmb_adagrad_t;
/* update mode 4: torch.optim.SparseAdam(betas, eps, lr = the step's lr) on the embedding tables -- only the rows a batch
 * hits update their moments and weights, a zero gradient of such a row included -- and torch.optim.Adam(betas, eps) on the
 * bias and the tower, both kept across calls.  Per coordinate, as torch 2.11's CPU kernels round it:
 *   SparseAdam: u1 = (g - m)*(1-b1); m' = m + u1; u2 = (g*g - v)*(1-b2); v' = v + u2;  p' = p + s_e * (m' / (sqrt(v') + eps))
 *   Adam:       m' = fma(1-b1, g - m, m); v' = fma((1-b2)*g, g, v*b2);  p' = p + (s_d * m') / (sqrt(v') / c2 + eps)
 * with the step's float scalars s_e = -lr*sqrt(1-b2^t)/(1-b1^t), s_d = -lr/(1-b1^t), c2 = (1-b2^t)^0.5, computed in double
 * on the host and rounded to float (fmb_adam_scalars).  The tables and the bias count every step (`step`); the tower counts
 * only the steps that give it a gradient (`mlp_step`: tower fit, run_experiment), as torch skips a parameter whose .grad
 * is None.  mv_dev [R][2][rowp]: m and v sub-rows of every packed table row (FTRL's layout; padding never written);
 * bias_mv_dev [2]; mlp_mv_dev [2][fmb_mlp_numel] (m, then v) or NULL.  Zero-fill the moments and counters to start.
 * The entry points with a state slot take it there (pass (const fmb_ftrl_t*)&sa), advanced to the step being run by
 * fmb_sparse_adam_advance; a session step advances it itself (fmb_session_set_sparse_adam).  Algorithmic bytes of the FM
 * step grow by 16F(k+1) per sample.  The row-sharded steps take each rank's shard of the moments (fmb_shard3_step_ex);
 * the shard2 path, AFM and fmb_fm_backward_runs_all reject mode 4. */
typedef struct fmb_adam_step_t { float emb_step, bias_step, bias_bc2s, mlp_step, mlp_bc2s; } fmb_adam_step_t;
typedef struct fmb_sparse_adam_t {
    float* mv_dev; float* bias_mv_dev; float* mlp_mv_dev;
    double beta1, beta2;
    float eps;
    int64_t step, mlp_step;     /* steps taken so far */
    fmb_adam_step_t cur;        /* the scalars of the step being run */
    const float* steps_dev;     /* fmb_online_deep_run_ex: the examples' scalars (fmb_sparse_adam_online_steps) */
} fmb_sparse_adam_t;
/* out[0] = s_e, out[1] = s_d, out[2] = c2 of step t (float), from lr and the betas in double as CPython computes them */
void fmb_adam_scalars(float lr, double beta1, double beta2, int64_t t, float* out);
/* ++step (and ++mlp_step when tower != 0); fills cur */
int fmb_sparse_adam_advance(fmb_sparse_adam_t* sa, float lr, int tower);
/* the scalars of N single-example steps of fmb_online_deep_run_ex into out_host [4 + 5N] ((1-b1, b2, 1-b2, eps), then one
 * fmb_adam_step_t per example), advancing the counters by N; copy it to the device and point steps_dev at it */
int fmb_sparse_adam_online_steps(fmb_sparse_adam_t* sa, float lr, int tower, int N, float* out_host);
/* mode 4's Adam step of the tower's n parameters (mlp_mv_dev and cur.mlp_*) */
int fmb_update_dense_adam(float* p_dev, const float* g_dev, int64_t n, const fmb_sparse_adam_t* sa, fmb_stream_t stream);
int fmb_fm_step_fused_ex(const int32_t* ids_dev, const float* xv_dev, const float* y_dev, float* table_dev,
                         const float* bias_dev, const uint32_t* posflag_dev, int B, int F, int k, int loss_kind, float lr,
                         int mode, const fmb_ftrl_t* ftrl, float* delta_dev, float* lossv_dev, void* ws_dev,
                         size_t ws_bytes, fmb_stream_t stream);
int fmb_fm_backward_runs_ex(const int32_t* sorted_keys_dev, int64_t N, float* table_dev, int F, int k, float lr, int mode,
                            const fmb_ftrl_t* ftrl, void* ws_dev, size_t ws_bytes, fmb_stream_t stream);
int fmb_finish_step_ex(const float* delta_dev, const float* lossv_dev, int B, float* bias_dev, float lr, int mode,
                       const fmb_ftrl_t* ftrl, float* loss_dev, fmb_stream_t stream);
int fmb_pos_flags(const int32_t* sorted_keys_dev, const int32_t* perm_dev, int64_t N, uint32_t* posflag_dev,
                  fmb_stream_t stream);
/* run-list forms (round 2): fmb_pos_flags_ex also appends the runs of >= 2 equal keys to rl, which must be ONE segment
 * (nseg == 1, seg_cap >= N/2) whose counters seg_count_dev[0..1] the caller zeroes beforehand (used behind fmb_sort_segment;
 * fmb_sort_fields_ex needs neither).  fmb_fm_backward_runs_list starts one warp per listed run instead of one per 32
 * sorted positions (all runs of a Criteo-shaped batch in flight at once; the first CTAs of the grid take the runs of
 * >= 128 entries with a deeper ring started at the run's first entry).  rl == NULL: the plain forms. */
int fmb_pos_flags_ex(const int32_t* sorted_keys_dev, const int32_t* perm_dev, int64_t N, uint32_t* posflag_dev,
                     const fmb_runlist_t* rl, fmb_stream_t stream);
int fmb_fm_backward_runs_list(const int32_t* sorted_keys_dev, int64_t N, float* table_dev, int F, int k, float lr, int mode,
                              const fmb_ftrl_t* ftrl, const fmb_runlist_t* rl, void* ws_dev, size_t ws_bytes,
                              fmb_stream_t stream);
int fmb_fm_step_fused(const int32_t* ids_dev, const float* xv_dev /*nullable*/, const float* y_dev, float* table_dev,
                      const float* bias_dev, const uint32_t* posflag_dev, int B, int F, int k, int loss_kind, float lr,
                      int mode, float* delta_dev, float* lossv_dev, void* ws_dev, size_t ws_bytes, fmb_stream_t stream);
int fmb_fm_backward_runs(const int32_t* sorted_keys_dev, int64_t N, float* table_dev, int F, int k, float lr, int mode,
                         void* ws_dev, size_t ws_bytes, fmb_stream_t stream);

/* ---- A6: sparse embedding gradient (segmented, in sample order) fused with the row update ------
 * replaces loss.backward() + optimizer.step() for the embedding tables (fm_adam.py:67-68,
 * deepfm_adam.py:102-103,115-116).  gs [B] = gradient on the FM logit; use_fm2 = it also flows
 * through sum_j bi; gvec [B,kp4] (nullable) = gradient on bi from the MLP (deepfm_adam.py:81). */
size_t fmb_bwd_workspace_bytes(int64_t N, int k);
int fmb_fm_backward_update(const int32_t* sorted_keys_dev, const int32_t* perm_dev, int64_t N,
                           const float* xv_dev, float* table_dev, int F, int k, const float* S_dev,
                           const float* gs_dev, int use_fm2, const float* gvec_dev, float lr, int mode,
                           void* ws_dev, size_t ws_bytes, fmb_stream_t stream);

/* extended form: n_entries = 1 + largest entry index in perm; S/gvec row pitch and gs stride (they may
 * live inside a gathered per-sample context); sorted keys >= key_limit are padding and are skipped */
int fmb_fm_backward_update_ex(const int32_t* sorted_keys_dev, const int32_t* perm_dev, int64_t N, int64_t n_entries,
                              const float* xv_dev, float* table_dev, int F, int k, const float* S_dev, int s_pitch,
                              const float* gs_dev, int gs_stride, int use_fm2, const float* gvec_dev,
                              int32_t key_limit, float lr, int mode, void* ws_dev, size_t ws_bytes,
                              fmb_stream_t stream);
/* _rl: with the run list of the sorted keys (nullable) the run kernel starts one warp per run, the long runs first */
int fmb_fm_backward_update_rl(const int32_t* sorted_keys_dev, const int32_t* perm_dev, int64_t N, int64_t n_entries,
                              const float* xv_dev, float* table_dev, int F, int k, const float* S_dev, int s_pitch,
                              const float* gs_dev, int gs_stride, int use_fm2, const float* gvec_dev, int32_t key_limit,
                              float lr, int mode, const fmb_runlist_t* rl, void* ws_dev, size_t ws_bytes,
                              fmb_stream_t stream);

/* _rl_ex: update mode 3 needs `ada` (its sums_dev), mode 4 an fmb_sparse_adam_t in the same slot (cast), advanced to the
 * step; NULL in the other modes -- the tower fit's backward */
int fmb_fm_backward_update_rl_ex(const int32_t* sorted_keys_dev, const int32_t* perm_dev, int64_t N, int64_t n_entries,
                                 const float* xv_dev, float* table_dev, int F, int k, const float* S_dev, int s_pitch,
                                 const float* gs_dev, int gs_stride, int use_fm2, const float* gvec_dev, int32_t key_limit,
                                 float lr, int mode, const fmb_adagrad_t* ada, const fmb_runlist_t* rl, void* ws_dev,
                                 size_t ws_bytes, fmb_stream_t stream);

/* ---- row-sharded multi-GPU step (BASELINE.json configs[4]; no counterpart in the reference, which is
 * single-device: SURVEY.md 8e).  Row r lives on rank r % G at local row r / G.  See csrc/sharded.cu. */
int fmb_shard_pw(int k); /* floats per pooled partial [S | Q | first]   */
int fmb_shard_cw(int k); /* floats per sample context [S | delta | loss | z] */
int fmb_shard_sort_max_cap(void);
int fmb_transpose_ids(const int32_t* ids_dev /*[B,F]*/, int B, int F, int32_t* out_dev /*[F,B]*/, fmb_stream_t stream);
int fmb_shard_partial_forward(const int32_t* idsT_all_dev /*[G,F,B]*/, const float* table_local_dev, int G, int me,
                              int B, int F, int k, float* partial_dev /* ---- multi-GPU, second design (csrc/shard2.cu): O(B*F) work per rank ------------------------------------------
 * Row r lives on rank r % G at local row r / G.  Every rank steps on its own batch; rows are gathered from the owners'
 * shards through peer-mapped pointers (NVLink), each rank stores one partial gradient per distinct row of its batch into
 * the owner's inbox (slot = [source rank][position in the source's stable sort]), the owner adds the partials in rank
 * order and applies the update.  Pointer arrays hold G peer-mapped addresses (entry `me` = the caller's own buffer).
 *   fmb_shard2_fused       forward + loss + contributions (rows hit once in my batch go straight to the inbox)
 *   fmb_shard2_runs        run kernel: partial gradient of every run of >= 2 equal keys -> inbox
 *   fmb_shard2_push_keys   my sorted keys -> slab `me` of every rank's keys_all [G][N]
 *   fmb_shard2_owner_apply scan keys_all, count the ranks hitting each owned row, rank-ordered add, row update
 * Exchanges are fenced with fmb_shard_signal epochs.  Reference semantics: fm_adam.py:56-69 on the concatenated batch. */
int fmb_shard2_slot_floats(void);
/* every row read of the forward pass is local: hot-field replica (hot_dev [R_hot][16], hot_base_dev [F] = first replica row
 * of a field or -1), own shard, or rowbox_dev [N][16] (filled by the owners: fmb_shard2_push_rows) */
int fmb_shard2_fused(const int32_t* ids_dev, const float* xv_dev, const float* y_dev, const uint32_t* posflag_dev,
                     void* const* tables, void* const* inbox, void* const* dl, const float* rowbox_dev, const float* hot_dev,
                     const int32_t* hot_base_dev, const int32_t* field_off_dev, const float* bias_dev, int G, int me, int B,
                     int F, int k, int loss_kind, void* ws_dev, size_t ws_bytes, const uint32_t* wait_flags_dev,
                     const uint32_t* wait_epoch_dev, int wait_channel, int* error_dev, fmb_stream_t stream);
int fmb_shard2_runs(const int32_t* sorted_keys_dev, int64_t N, int F, int k, void* ws_dev, size_t ws_bytes,
                    void* const* inbox, int G, int me, fmb_stream_t stream);
int fmb_shard2_push_keys(const int32_t* sorted_keys_dev, int64_t N, int G, int me, void* const* keys_all,
                         fmb_stream_t stream);
/* row service for the next forward pass: rows I own that the other ranks' sorted lists name -> their rowboxes */
int fmb_shard2_push_rows(const int32_t* keys_all_dev, float* table_dev, void* const* rowbox, void* const* hot,
                         const int32_t* hot_base_dev, const int32_t* field_off_dev, int G, int me, int B, int F, int k,
                         fmb_stream_t stream);
/* my rows of the hot fields -> every rank's replica (after initialising / loading parameters) */
int fmb_shard2_push_hot(float* table_dev, void* const* hot, const int32_t* hot_base_dev, const int32_t* field_off_dev,
                        int R_hot, int G, int me, int F, int k, fmb_stream_t stream);
/* list_dev [G*N] / nlist_dev [2] / parity: compact list of the owned run starts (built by the count pass so that the
 * apply pass runs full warps).  wait_*: the kernels themselves wait for the peers' epoch on wait_channel (NULL = no wait). */
int fmb_shard2_owner_apply(const int32_t* keys_all_dev, const float* inbox_dev, float* table_dev, uint32_t* cnt_dev,
                           uint32_t* list_dev, uint32_t* nlist_dev, int parity, void* const* hot,
                           const int32_t* hot_base_dev, const int32_t* field_off_dev, int G, int me, int B, int F, int k,
                           float lr, int mode, const uint32_t* wait_flags_dev, const uint32_t* wait_epoch_dev,
                           int wait_channel, int* error_dev, fmb_stream_t stream);

/*[G*B,PW]*/, fmb_stream_t stream);
int fmb_shard_combine(const float* recv_dev /*[G,B,PW]*/, const float* bias_dev, const float* y_dev, int G, int me,
                      int B, int k, int loss_kind, float* ctx_dev /*[B,CW]*/, float* z_dev /*nullable*/, fmb_stream_t stream);
int fmb_shard_unpack_ctx(const float* ctx_all_dev, int64_t n, int k, float* delta_dev, float* lossv_dev,
                         fmb_stream_t stream);
int fmb_shard_sort_fields(const int32_t* idsT_all_dev, int G, int me, int B, int F, const int32_t* field_off_dev,
                          int cap, int32_t* sorted_keys_dev /*[F,cap]*/, int32_t* perm_dev /*[F,cap]*/,
                          int32_t* counts_dev /*[F]*/, int32_t* overflow_dev /*[1]*/, fmb_stream_t stream);
/* _rl: also the run list of every field's sorted owned entries (rl->nseg == F, seg_cap >= cap/2 + 1; nullable) */
int fmb_shard_sort_fields_rl(const int32_t* idsT_all_dev, int G, int me, int B, int F, const int32_t* field_off_dev, int cap,
                             int32_t* skeys_dev, int32_t* perm_dev, int32_t* counts_dev, int32_t* overflow_dev,
                             const fmb_runlist_t* rl, fmb_stream_t stream);
/* The three exchanges without a collective call: with idsT_all, recv, ctx_all and a flag block in symmetric (peer
 * mapped) memory, producers store straight into the consumers' buffers over NVLink.  Every `peers` argument is a
 * HOST array of G (<= 8) device pointers, entry r = where THIS device maps rank r's copy of that buffer.
 *   fmb_shard_transpose_ids_peers   ids [B,F] -> slab `me` of every rank's idsT_all [G,F,B]        (replaces all-gather 1)
 *   fmb_shard_partial_forward_peers block r of the pooled partials -> block `me` of rank r's recv  (replaces the all-to-all)
 *   fmb_shard_combine_peers         fold + ctx rows -> rows [me*B,(me+1)*B) of every rank's ctx_all      (replaces all-gather 2)
 *   fmb_shard_signal                per-channel epoch flags, uint32 [8 channels][8 ranks] in symmetric memory;
 *                                   mode 1 publish (fence.sys + st.release.sys to all peers), 2 wait for all G peers
 *                                   (ld.acquire.sys, bounded spin), 3 both; sync_local uint32 [16] ordinary device
 *                                   memory, zero-initialised (epoch[8] | block counters[8]);
 *                                   error_dev (nullable) receives 1 + channel on a time-out.
 * The producers can publish their channel themselves from their last block (publish_channel >= 0), the fused
 * combine can wait at its start (wait_channel >= 0): then only consumers that are not fused need fmb_shard_signal. */
int fmb_shard_transpose_ids_peers(const int32_t* ids_dev, int B, int F, int G, int me, void* const* idsT_all_peers,
                                  void* const* flag_peers, uint32_t* flags_local_dev, uint32_t* sync_local_dev,
                                  int* error_dev, int publish_channel /* -1: none */, fmb_stream_t stream);
int fmb_shard_partial_forward_peers(const int32_t* idsT_all_dev, const float* table_local_dev, int G, int me, int B,
                                    int F, int k, void* const* recv_peers, void* const* flag_peers,
                                    uint32_t* flags_local_dev, uint32_t* sync_local_dev, int* error_dev,
                                    int publish_channel /* -1: none */, fmb_stream_t stream);
/* fmb_shard_combine fused with its two exchanges: waits for `wait_channel` (the owners' partials), folds, stores
 * the ctx rows into every rank's ctx_all (and ctx_local_dev when given), publishes `publish_channel`.  k <= 16. */
int fmb_shard_combine_peers(const float* recv_dev, const float* bias_dev, const float* y_dev, int G, int me, int B,
                            int k, int loss_kind, void* const* ctx_all_peers, float* ctx_local_dev /*nullable*/,
                            void* const* flag_peers, uint32_t* flags_local_dev, uint32_t* sync_local_dev,
                            int* error_dev, int wait_channel, int publish_channel, fmb_stream_t stream);
int fmb_shard_signal(void* const* flag_peers, uint32_t* flags_local_dev, uint32_t* sync_local_dev, int channel, int G,
                     int me, int mode, int* error_dev, fmb_stream_t stream);

/* ---- the sharded step as ONE kernel per rank (csrc/shard3.cu): a CTA keeps the rows it owns for a tile of 8*G samples in
 * shared memory across both exchanges (partials -> the samples' owner, context -> everyone) and updates from that copy;
 * per-TILE epoch flags in peer-mapped memory instead of per-kernel ones.  Same arithmetic, same order, same results as the
 * three-kernel path above (fm_adam.py:56-69 on the concatenated batch, owner-major fold).
 *   fmb_shard3_tiles        tiles per step (0 = shape not supported: G in {1,2,4,8}, B % (8*G) == 0, G*B <= 65536, k <= 15);
 *                           the tile-flag block holds 2 * tiles uint32 words, zero-initialised, mapped by every peer
 *   fmb_shard_sort_fields_pf  fmb_shard_sort_fields_rl + posflag [F][G*B]: sorted position | 0x80000000 (row hit more than
 *                           once) of every entry this rank owns
 *   fmb_shard3_step         the step up to the staged multi-hit contributions; fmb_fm_backward_runs_list, fmb_shard_unpack_ctx
 *                           and fmb_finish_step follow; epoch_dev: uint32 step counter (device), fmb_shard3_bump adds 1 behind
 *                           the step; *error_dev: 16 + phase on a time-out, 32 when a tile's entry capacity overflowed */
int fmb_shard3_tiles(int G, int B, int F, int k);
int fmb_shard_sort_fields_pf(const int32_t* idsT_all_dev, int G, int me, int B, int F, const int32_t* field_off_dev, int cap,
                             int32_t* skeys_dev, int32_t* perm_dev, int32_t* counts_dev, int32_t* overflow_dev,
                             const fmb_runlist_t* rl, uint32_t* posflag_dev, fmb_stream_t stream);
int fmb_shard3_step(const int32_t* idsT_all_dev, float* table_local_dev, const float* bias_dev, const float* y_dev,
                    const uint32_t* posflag_dev, int G, int me, int B, int F, int k, int cap, int loss_kind, float lr, int mode,
                    void* ws_dev, size_t ws_bytes, void* const* recv_peers, void* const* ctx_peers, void* const* tflag_peers,
                    const float* recv_local_dev, const float* ctx_local_dev, const uint32_t* tflags_local_dev,
                    const uint32_t* epoch_dev, int* error_dev, fmb_stream_t stream);
/* _ex: with the update rule's state (NULL in modes 0 and 1).  Mode 3: an fmb_adagrad_t whose sums_dev is this rank's
 * [R_local + 1][rowp] shard (local row r / G of row r, the local table's layout) and bias_sum_dev the replicated [1];
 * mode 4: an fmb_sparse_adam_t whose mv_dev is this rank's [R_local + 1][2][rowp] shard and bias_mv_dev the replicated
 * [2], advanced to this step by fmb_sparse_adam_advance (once per step on every rank).  Pass the same state to the
 * fmb_fm_backward_runs_list and fmb_finish_step_ex calls that follow.  Mode 3 or 4 without its state is refused. */
int fmb_shard3_step_ex(const int32_t* idsT_all_dev, float* table_local_dev, const float* bias_dev, const float* y_dev,
                       const uint32_t* posflag_dev, int G, int me, int B, int F, int k, int cap, int loss_kind, float lr,
                       int mode, const void* state, void* ws_dev, size_t ws_bytes, void* const* recv_peers,
                       void* const* ctx_peers, void* const* tflag_peers, const float* recv_local_dev,
                       const float* ctx_local_dev, const uint32_t* tflags_local_dev, const uint32_t* epoch_dev,
                       int* error_dev, fmb_stream_t stream);
int fmb_shard3_bump(uint32_t* epoch_dev, fmb_stream_t stream);

/* ---- A4/A5: MLP tower on the Bi-Interaction vector (deepfm_adam.py:79-89, nfm_adam.py:78-88,
 * deepfm_onn.py:88-102).  mlp = W0[H,k] c0[H] W1[H,H] c1[H] ... (nn.Linear layouts, concatenated);
 * act [L,B,H] post-relu activations; head [L,B] = sum_j act[l][b][j]. fp32 SIMT, k-ascending FMA. */
int64_t fmb_mlp_numel(int k, int L, int H);
int fmb_mlp_forward(const float* bi_dev, int ldbi, const float* mlp_dev, int B, int k, int L, int H,
                    float* act_dev, float* head_dev /*nullable*/, fmb_stream_t stream);
size_t fmb_mlp_bwd_workspace_bytes(int B, int H);
/* backward of head `top`: gtop [B] is the gradient on sum_j act[top][b][j]; writes the gradients of
 * layers 0..top into gmlp (same layout as mlp) and, when gbi is non-NULL, d/d(bi) [B,ldgbi]. */
int fmb_mlp_backward(const float* bi_dev, int ldbi, const float* mlp_dev, const float* act_dev,
                     const float* gtop_dev, int top, int B, int k, int L, int H, float* gmlp_dev, float* gbi_dev,
                     int ldgbi, void* ws_dev, size_t ws_bytes, fmb_stream_t stream);
/* Contractions of >= 2^24 multiply-adds (cfg4: B = 8192, H = 400) run on the tcgen05 tensor cores as 3xTF32
 * with fp32 accumulation in tensor memory (csrc/gemm_tc.cu, ~1e-6 relative); smaller ones -- every shape of the
 * reference's scripts -- on the exact SIMT kernel.  fmb_set_tensor_cores(0) forces the exact path. */
void fmb_set_tensor_cores(int on);
int fmb_tensor_cores_enabled(void);
int fmb_tensor_core_threshold_log2(void);
int fmb_gemm_tc_nt(const float* A_dev /*[M,K]*/, const float* B_dev /*[N,K]*/, float* C_dev /*[M,N]*/, int M, int N,
                   int K, fmb_stream_t stream); /* C = A B^T on the tensor cores (tests) */
/* General form: C[m*scm + n] = epi( sum_k A[m*sam + k*sak] * B[k*sbk + n*sbn] ), epi 0 none / 1 relu(x + bias[n]) /
 * 2 keep where mask[m*smm + n] > 0; colsum[m] = sum_k A(m,k) (nullable).  The three tower products
 * (mlp.cu: forward NT, dX NN, dW TN with K = batch split across CTAs) are this call. */
int fmb_gemm_tc_strided(const float* A_dev, int64_t sam, int64_t sak, const float* B_dev, int64_t sbk, int64_t sbn,
                        float* C_dev, int64_t scm, int M, int N, int K, int epi, const float* bias_dev,
                        const float* mask_dev, int64_t smm, float* colsum_dev, fmb_stream_t stream);
int fmb_gemm_tc_error(void);
/* z = base + head, base = z_fm (DeepFM, deepfm_adam.py:88) or sum_first + bias (NFM, nfm_adam.py:79,87) */
int fmb_combine_logit(int nfm, const float* z_fm_dev, const float* sum_first_dev, const float* bias_dev,
                      const float* head_dev, int B, float* z_dev, fmb_stream_t stream);
/* ONN heads p[l,b] = sigmoid(base[b] + head[l,b]) (deepfm_onn.py:95-99) */
int fmb_onn_heads(int nfm, const float* z_fm_dev, const float* sum_first_dev, const float* bias_dev,
                  const float* head_dev, int L, int B, float* p_dev, fmb_stream_t stream);
/* predict threshold sigmoid(z) > 0.5 (fm_adam.py:84-88; deepfm_onn.py:171-175 applies it to p_last) */
int fmb_predict(const float* z_dev, int n, uint8_t* out_dev, fmb_stream_t stream);

/* ---- A7: hedge backpropagation (deepfm_onn.py:109-154, nfm_onn.py:111-156) ---------------------
 * head_grad: BCELoss(p_l, y) per sample (lossv) and its gradient on the head's pre-sigmoid logit;
 * accumulate: w[j] (+)= alpha[i] * grad for layers j <= i; apply: W -= n*w, then the alpha update. */
int fmb_hedge_head_grad(const float* p_dev, const float* y_dev, int B, float* gtop_dev, float* lossv_dev,
                        fmb_stream_t stream);
int fmb_hedge_accumulate(float* acc_dev, const float* gmlp_dev, const float* alpha_dev, int i, int k, int L, int H,
                         fmb_stream_t stream);
int fmb_hedge_apply(float* mlp_dev, const float* acc_dev, float lr, float* alpha_dev, const float* loss_sum_dev,
                    int B, int k, int L, int H, float hb, float hs, fmb_stream_t stream);
/* hedge backpropagation in ONE backward pass (SURVEY.md A7): acc = sum_{i>=l} alpha_i dL_i/dW_l for every layer l, by
 * injecting alpha_i * gtop_all[i] at every head on the way down; replaces the L calls of fmb_mlp_backward +
 * fmb_hedge_accumulate (deepfm_onn.py:127-141) when the tower's products run on the tensor cores (results within
 * tolerance of the L-pass form, not bit-identical to it: each alpha_i * grad_i is no longer rounded separately). */
int fmb_mlp_backward_hedge(const float* bi_dev, int ldbi, const float* mlp_dev, const float* act_dev,
                           const float* gtop_all_dev /*[L,B]*/, const float* alpha_dev /*[L]*/, int B, int k, int L, int H,
                           float* acc_dev, void* ws_dev, size_t ws_bytes, fmb_stream_t stream);

/* ---- A8: per-example online mode as one persistent kernel ---------------------------------------
 * replaces run_experiment (fm_adam.py:90-119, same in all five classes): for each example in order,
 * predict then fit with batch size 1 (Adam family: fm_adam.py:71-82, deepfm_adam.py:106-117,
 * nfm_adam.py:105-116; ONN: deepfm_onn.py:109-154).  kind 0..4 = FMAdam, DeepFMAdam, NFMAdam, DeepFMOnn,
 * NFMOnn.  preds [N] = prediction made before fitting example i; conf [4] = tp, fp, tn, fn. */
int fmb_online_deep_run(int kind, const int32_t* ids_dev /*[N,F]*/, const float* xv_dev, const float* y_dev, int N,
                        int F, int k, int L, int H, float* table_dev, float* bias_dev, float* mlp_dev,
                        float* alpha_dev, float* acc_dev /*[fmb_mlp_numel], ONN*/, float lr, float hb, float hs,
                        int mode, uint8_t* preds_dev, int64_t* conf_dev, fmb_stream_t stream);
/* _ex: update mode 3 of kinds 0-2 reads and writes the sums of `ada` (table, bias and, with a tower, the tower's); the
 * ONN kinds' hedge step uses no optimizer and ignores the mode.  fmb_online_deep_run rejects mode 3 for kinds 0-2.  Mode 4
 * takes an fmb_sparse_adam_t in the same slot (cast) whose steps_dev holds the N examples' scalars. */
int fmb_online_deep_run_ex(int kind, const int32_t* ids_dev, const float* xv_dev, const float* y_dev, int N, int F, int k,
                           int L, int H, float* table_dev, float* bias_dev, float* mlp_dev, float* alpha_dev,
                           float* acc_dev, float lr, float hb, float hs, int mode, const fmb_adagrad_t* ada,
                           uint8_t* preds_dev, int64_t* conf_dev, fmb_stream_t stream);

/* ---- A9-A11: classical fp64 online learners, one persistent launch per stream -------------------
 * fmb_ftrl_fm_run : FM_FTRL.online_learning (models/models_online/FM_FTRL.py:47-92)
 * fmb_sftrl_run   : SFTRL_CCFM.online_learning (SFTRL_CCFM.py:30-121; vanila = 0) and
 *                   SFTRL_Vanila.online_learning (SFTRL_Vanila.py:33-123; vanila = 1)
 * X [N,d] dense fp64, y [N]; task 0 = 'reg', 1 = 'cls'; preds [N]; status [1] = 0 or (index of the
 * first NaN score) + 1 -- the caller raises ValueError('Nan contained') like FM_FTRL.py:64-65. */
int fmb_ftrl_fm_run(const double* X_dev, const double* y_dev, int N, int d, int m2, int task, double eta,
                    double* w1_dev /*[d] in/out*/, double* W2_dev /*[m2,d-1] in/out*/,
                    double* g_w1_dev /*[d] zeroed*/, double* g_W2_dev /*[m2,d-1] zeroed*/, double* preds_dev,
                    int* status_dev, fmb_stream_t stream);
size_t fmb_sftrl_workspace_bytes(int d, int m);
int fmb_sftrl_run(const double* X_dev, const double* y_dev, int N, int d, int m, int task, int vanila, double eta,
                  double* BT_P_dev /*[ds,2m]*/, double* BT_N_dev /*[ds,2m]*/, int* row_counts_dev /*[2]*/,
                  double* w_dev /*[d], vanila*/, double* g_w_dev /*[d], vanila*/, double* preds_dev,
                  int* status_dev, void* ws_dev, size_t ws_bytes, fmb_stream_t stream);

/* ---- training session: one call per step -------------------------------------------------------
 * fmb_session_fm_step      : FMAdam.update_embedding / FMAdam.fit and every class's
 *                            update_embedding (fm_adam.py:56-82, deepfm_adam.py:91-104,
 *                            nfm_adam.py:90-103, deepfm_onn.py:156-169, nfm_onn.py:158-171)
 * fmb_session_fm_step_host : the same with HOST ids/xv/y; copies in, runs, copies the loss out. */
int fmb_session_create(fmb_session** out, int F, int k, int64_t max_batch,
                       const int32_t* field_off_host /*[F+1] global row offset per field, nullable*/);
void fmb_session_destroy(fmb_session* s);
int64_t fmb_session_launches(const fmb_session* s);
int fmb_session_graph_count(const fmb_session* s); /* step graphs currently cached */
int fmb_session_fm_step(fmb_session* s, const int32_t* ids_dev, const float* xv_dev, const float* y_dev, int B,
                        float* table_dev, float* bias_dev, int key_bits, int loss_kind, float lr, int mode,
                        float* loss_dev, fmb_stream_t stream);
int fmb_session_fm_step_host(fmb_session* s, const int32_t* ids_host, const float* xv_host, const float* y_host,
                             int B, float* table_dev, float* bias_dev, int key_bits, int loss_kind, float lr,
                             int mode, float* loss_host, fmb_stream_t stream);

/* pre-sort: the sort of a batch depends on its ids only.  fmb_session_presort(ids) sorts them now on a side
 * stream (overlapping the step in flight); the next fmb_session_fm_step called with the same ids pointer and
 * B skips its own sort.  The ids must stay unchanged until that step has been submitted. */
int fmb_session_presort(fmb_session* s, const int32_t* ids_dev, int B, int key_bits);
/* FTRL-Proximal state of the session's steps (update mode 2) */
int fmb_session_set_ftrl(fmb_session* s, float* zn_dev, float* bias_zn_dev, float beta, float l1, float l2);
/* Adagrad state of the session's steps (update mode 3): sums_dev [R][rowp], bias_sum_dev [1], filled by the caller */
int fmb_session_set_adagrad(fmb_session* s, float* sums_dev, float* bias_sum_dev, float eps);
/* SparseAdam state of the session's steps (update mode 4): the caller's struct, kept by pointer; every mode-4 step
 * advances it (tower = 0) when submitted and takes that step's scalars by value */
int fmb_session_set_sparse_adam(fmb_session* s, fmb_sparse_adam_t* sa);
/* forget a pending pre-sort (the caller cannot vouch that the pre-sorted ids buffer still holds the same batch) */
void fmb_session_presort_invalidate(fmb_session* s);
/* fmb_session_fm_step with the sort of the NEXT batch riding along: next_ids_dev (nullable) are the ids the
 * following call will step on (main_experiment.py:92-105 walks its batches in a known order); their stable sort
 * runs on a side branch of this step's graph and the following call, recognised by its ids pointer, skips its own.
 * One CUDA graph per configuration, re-pointed at each call's batch (cudaGraphExecKernelNodeSetParams). */
int fmb_session_fm_step_next(fmb_session* s, const int32_t* ids_dev, const float* xv_dev, const float* y_dev, int B,
                             float* table_dev, float* bias_dev, int key_bits, int loss_kind, float lr, int mode,
                             const int32_t* next_ids_dev, float* loss_dev, fmb_stream_t stream);

/* pipelined host entry point: fmb_session_host_slots() input slots (slot = 0..3); the H2D copies and the sort of the
 * following steps run on the session's copy / side streams while step t computes.  Pinned / registered host buffers are read in place.  fmb_session_wait_loss
 * blocks until the step last submitted on `slot` has finished and returns its mean loss. */
int fmb_session_fm_step_host_async(fmb_session* s, int slot, const int32_t* ids_host, const float* xv_host,
                                   const float* y_host, int B, float* table_dev, float* bias_dev, int key_bits,
                                   int loss_kind, float lr, int mode, fmb_stream_t stream);
int fmb_session_host_slots(void);   /* input slots of fmb_session_fm_step_host_async (4): a caller cycling through all of
                                      * them and collecting a loss three steps later never waits for the GPU to submit */
int fmb_session_wait_loss(fmb_session* s, int slot, float* loss_host);

#ifdef __cplusplus
}
#endif
#endif /* FMB200_H */
