/* issue_emb_b200 -- C ABI of the B200-native Issue_Embeddings encoder hot path and the Label_Microservice
 * MLP head (libissue_emb_b200.so).  Plain pointers and sizes only; no torch / C++ types.
 *
 * The reference (kubeflow/Code-Intelligence) has no FFI layer for this path: its "operator API" is the Python
 * class InferenceWrapper and sklearn's MLPClassifier behind MLPWrapper.  Each entry point below states the
 * reference interface it replaces (paths relative to the reference tree); INTEGRATION.md shows the ctypes
 * binding a maintainer would add on the reference side.
 *
 * Conventions
 *   - every function returns IE_OK (0) or a negative IE_ERR_* code and never aborts; ie_last_error() returns a
 *     thread-local human-readable message for the last failing call on this thread.  Device-side waits are bounded:
 *     one that exceeds its limit drains the kernel and surfaces as IE_ERR_CUDA (no trap, the CUDA context and the
 *     handle stay usable).
 *   - a handle owns its device weights and workspace; calls on one handle are serialised internally (host mutex; a
 *     call on another stream first waits for the previous call's completion event); handles may be used from any host
 *     thread.  The persistent recurrent kernel is launched cooperatively: it runs only when its whole grid can be
 *     resident, so two handles (or other work) sharing a device serialise instead of deadlocking.
 *   - `flags & IE_FLAG_DEVICE_PTRS`: ids / lengths / out (or X / probs) are device pointers on the handle's
 *     device and the call is asynchronous on `stream`; otherwise they are host pointers (pinned or pageable)
 *     and the call returns after the result has been copied back.  In device-pointer mode data-dependent errors
 *     (token id out of range, length outside [1,T] -- clamped --, wait timeout) cannot be returned by the call itself:
 *     ie_encoder_check_errors() reports them.
 *   - `stream` is a cudaStream_t passed as void*.  With host pointers NULL selects the handle's own stream; with
 *     IE_FLAG_DEVICE_PTRS it is used verbatim (NULL = the legacy default stream, which is torch's default).
 */
#ifndef ISSUE_EMB_B200_H_
#define ISSUE_EMB_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IE_OK 0
#define IE_ERR_INVALID (-1) /* bad argument / shape (Python shim raises ValueError)                        */
#define IE_ERR_CUDA (-2)    /* CUDA runtime / launch failure (RuntimeError)                                  */
#define IE_ERR_OOM (-3)     /* device memory exhausted (RuntimeError, so the reference's batch-halving loop   */
                            /* py/code_intelligence/inference.py:214-223 keeps working)                       */
#define IE_ERR_STATE (-4)   /* weights not loaded, wrong call order                                           */
#define IE_ERR_TOKEN (-5)   /* a token id outside [0, vocab_sz) was seen (ValueError)                         */

#define IE_FLAG_DEVICE_PTRS 1

/* ie_config.flags */
#define IE_CFG_ACCURATE_GATES 1 /* ex2+rcp sigmoid/tanh (abs err ~1e-7) instead of the default single-MUFU          */
                                /* tanh.approx.f32 gates (rel err 2^-11; no measurable effect on the parity metrics) */
#define IE_CFG_FP32 2           /* "fp32-accurate" mode (BASELINE configs[1] as written; the reference computes in    */
                                /* fp32, Issue_Embeddings/flask_app/inference.py:57): every product runs as split-bf16  */
                                /* (x = hi + lo, three tensor-core passes hi*hi + lo*hi + hi*lo, f32 accumulate: ~2^-17 */
                                /* relative per product), input projections kept in f32, IEEE gates.  ~3x the MMAs.    */
#define IE_CFG_F32_GX 4         /* keep the hoisted input projections in f32 instead of fp16 (bf16 mode only)         */

#define IE_MAX_BATCH 3072 /* upper bound of rows per ie_encoder_encode call; the handle's own limit is
                             ie_encoder_max_batch() = 256 x (batches per launch, default 5): that many independent
                             256-row batches ride one launch of the persistent recurrent kernel (each a CTA-pair
                             M=256 UMMA tile); they share the kernel, not their results */

typedef struct ie_encoder ie_encoder;
typedef struct ie_mlp ie_mlp;

/* AWD-LSTM encoder shape.  Replaces what fastai's load_learner() unpickles at
 * Issue_Embeddings/flask_app/inference.py:33-36 (model structure: notebooks/04_Inference.ipynb:157-187):
 * Embedding(vocab_sz, emb_sz, padding_idx=pad_idx) -> n_layers x LSTM, in_0 = emb_sz, hidden = n_hid,
 * out_{L-1} = emb_sz.  Output width is 3*emb_sz. */
typedef struct ie_config {
  int32_t n_layers; /* deployed reference model: 4 (north-star wording: 3) */
  int32_t emb_sz;   /* 800  */
  int32_t n_hid;    /* 2400 */
  int32_t vocab_sz; /* 60000 */
  int32_t pad_idx;  /* 1 (inference.py:36 learn.data.pad_idx) */
  int32_t device;   /* CUDA device ordinal */
  int32_t flags;    /* IE_CFG_* bits, 0 = defaults */
} ie_config;

int ie_version(void);
const char* ie_last_error(void);

/* InferenceWrapper.__init__ (Issue_Embeddings/flask_app/inference.py:29-39): create the encoder ... */
int ie_encoder_create(const ie_config* cfg, ie_encoder** out);
void ie_encoder_destroy(ie_encoder* h);

/* ... and load its weights (host pointers, f32, C-contiguous):
 *   emb   [vocab_sz, emb_sz]                     state_dict key  encoder.weight
 *   w_ih  [4*out_l, in_l]   rows i|f|g|o         rnns.{l}.module.weight_ih_l0
 *   w_hh  [4*out_l, out_l]                       rnns.{l}.weight_hh_l0_raw
 *   b_ih, b_hh [4*out_l]                         rnns.{l}.module.bias_{ih,hh}_l0
 * (torch.nn.LSTM layout; key names per fastai 1.0.53 AWD_LSTM, SURVEY.md section 8c). */
int ie_encoder_load_embedding(ie_encoder* h, const float* emb);
int ie_encoder_load_layer(ie_encoder* h, int32_t layer, const float* w_ih, const float* w_hh, const float* b_ih,
                          const float* b_hh);

/* The hot path.  Replaces InferenceWrapper._forward_pass + batch_seq_pool
 * (Issue_Embeddings/flask_app/inference.py:55-57 and :215-246; bulk loop py/code_intelligence/inference.py:207-212)
 * and, with B == 1 and lengths[0] == T, get_pooled_features (inference.py:71-90):
 *   ids     [B, T] int64, batch-first, right-padded with pad_idx (what pad_sequence builds, inference.py:201)
 *   lengths [B] int32, 1 <= lengths[b] <= T
 *   out     [B, 3*emb_sz] f32 = [mean | max | last] over the first lengths[b] steps of the last layer's hidden
 *           states, zero initial state (encoder.reset(), inference.py:56)
 * 1 <= B <= ie_encoder_max_batch(h).  T is bounded only by the workspace cap B_pad*T <= 2^22 tokens (IE_ERR_OOM
 * beyond; B_pad = B rounded up to 256): the time dimension is processed in chunks, so a single 16k-token issue is
 * fine. */
int ie_encoder_encode(ie_encoder* h, const int64_t* ids, const int32_t* lengths, int32_t B, int32_t T, float* out,
                      int32_t flags, void* stream);

/* InferenceWrapper.get_raw_features (inference.py:59-68): the last layer's hidden states, raw [B, T, emb_sz] f32. */
int ie_encoder_raw_features(ie_encoder* h, const int64_t* ids, int32_t B, int32_t T, float* raw, int32_t flags,
                            void* stream);

/* Number of kernels this handle has launched so far (bench.py reports it as gpu_launches). */
int64_t ie_encoder_launch_count(const ie_encoder* h);

/* Rows one ie_encoder_encode call accepts on this handle: 1280 = five 256-row batches per launch by default
 * (environment variable IE_BATCHES=n at create time, 1 <= n <= 12, changes that to 256 n). */
int32_t ie_encoder_max_batch(const ie_encoder* h);

/* Device-side error state of the last call on this handle (waits for it to finish): IE_OK, IE_ERR_TOKEN (a token id
 * outside [0, vocab_sz) was remapped to 0), IE_ERR_INVALID (a length outside [1,T] was clamped; device-pointer mode
 * only -- host lengths are validated before anything is launched) or IE_ERR_CUDA (a device-side wait timed out and
 * the kernel was drained).  Host-pointer calls report these themselves; device-pointer calls are asynchronous, so
 * their caller asks here.  Clears the state. */
int ie_encoder_check_errors(ie_encoder* h);

/* Device time of each phase of the last encode call on this handle, from CUDA events recorded on the launching
 * stream: ms[0] = embedding gather, then per layer l: ms[1+2l] = input-projection GEMM, ms[2+2l] = the T recurrent
 * step launches, last = pool finalize.  Waits for the call to finish.  Returns the number of phases (or < 0). */
int ie_encoder_last_phase_ms(ie_encoder* h, float* ms, int32_t cap);

/* SM clock (MHz) the recurrent kernel of each layer ran at in the last call, from clock64 / globaltimer stamps taken
 * by the kernel itself (nvidia-smi cannot resolve single phases).  mhz[l] = recurrent kernel of layer l,
 * mhz[n_layers + l] = its input-projection GEMM (0 when the layer had none).  Returns 2 * n_layers (or < 0). */
int ie_encoder_last_phase_mhz(ie_encoder* h, float* mhz, int32_t cap);

/* Debug hook: per-item timeline of one layer of the persistent recurrent kernel (tools/trace_layer.py). */
int64_t ie_debug_seq_trace(ie_encoder* h, int32_t layer, long long* out, int64_t cap);

/* MLP head.  Replaces sklearn MLPClassifier.predict_proba as called by MLPWrapper.predict_probabilities
 * (py/label_microservice/mlp.py:56-63): relu hidden layers, logistic output (multilabel).
 *   dims [n_layers + 1] = {D_in, hidden..., n_labels};  coef_l [dims[l], dims[l+1]] f32 (sklearn coefs_[l],
 *   fan_in major), intercept_l [dims[l+1]].  X [n, D_in] f32 -> probs [n, n_labels] f32. */
int ie_mlp_create(int32_t n_layers, const int32_t* dims, int32_t device, ie_mlp** out);
int ie_mlp_load_layer(ie_mlp* m, int32_t layer, const float* coef, const float* intercept);
int ie_mlp_predict_proba(ie_mlp* m, const float* X, int32_t n, float* probs, int32_t flags, void* stream);
void ie_mlp_destroy(ie_mlp* m);

/* Threshold search.  Replaces the per-label loop of MLPWrapper.find_probability_thresholds
 * (py/label_microservice/mlp.py:81-98: sklearn precision_recall_curve + "highest precision among the points with
 * precision >= precision_threshold and recall >= recall_threshold; first such point in increasing-threshold order").
 *   scores [n, n_labels] f32 (predict_proba of the hold-out set), truth [n, n_labels] uint8 (0/1), n <= 16384
 *   thresholds [n_labels] f32 (NaN: no qualifying point, the label is excluded -- None in the reference),
 *   precisions / recalls [n_labels] f64 at the chosen point (0 when excluded).
 * Host pointers (synchronous) or, with IE_FLAG_DEVICE_PTRS, device pointers on `device` (asynchronous on `stream`). */
int ie_pr_thresholds(const float* scores, const uint8_t* truth, int32_t n, int32_t n_labels, double precision_threshold,
                     double recall_threshold, float* thresholds, double* precisions, double* recalls, int32_t device,
                     int32_t flags, void* stream);

/* Similar-issue search: exact cosine k-nearest neighbours over an index of issue embeddings.  Replaces the host-side
 * brute-force searches of the reference: the one-shot labeler of
 * Issue_Embeddings/notebooks/scratch/Kubeflow-FewShotLearning.ipynb (cell 46, oneshotlabeler.query: CosineSimilarity
 * against every labelled issue, then argsort(descending=True)) and KNeighborsClassifier(n_neighbors=2,
 * weights='distance', metric='cosine') of cell 77 of the same notebook; the duplicate issues noted at
 * Get-GitHub-Issues.ipynb:361 and 01_AcquireData.ipynb:48 are what a self-join finds.  The reference's README lists
 * duplicate detection and reviewer recommendation as uses of the embedding; both are this search.
 *
 * Create: vectors [n, d] f32 (host, or device on `device` with IE_FLAG_DEVICE_PTRS, read on `stream`), 1 <= d <= 4096,
 * all finite.  Synchronous.  The index keeps 4 * round_up(d, 64) bytes per row (split-bf16 residuals), plus 12 B. */
typedef struct ie_knn ie_knn;
int ie_knn_create(const float* vectors, int64_t n, int32_t d, int32_t device, int32_t flags, void* stream, ie_knn** out);
/* Search, as sklearn NearestNeighbors(metric='cosine', algorithm='brute').kneighbors:
 *   queries [m, d] f32 -> distances [m, k] f32 (1 - cos, ascending; ties: smaller id first), ids [m, k] int64.
 *   queries == NULL: the queries are index rows [row0, row0 + m), each excluding itself (kneighbors(X=None)).
 * 1 <= k <= 32 and k <= n (n - 1 for self-queries).  Zero vectors have cosine 0 with everything (distance 1).
 * Host pointers: synchronous, non-finite queries are rejected.  IE_FLAG_DEVICE_PTRS: queries / distances / ids are
 * device pointers and the call is asynchronous on `stream`. */
int ie_knn_search(ie_knn* h, const float* queries, int64_t row0, int32_t m, int32_t k, float* distances, int64_t* ids,
                  int32_t flags, void* stream);
void ie_knn_destroy(ie_knn* h);

/* Debug / test hook: D[M,N] = A[M,K] * B[N,K]^T (+bias) through the same tcgen05 GEMM the encoder uses.
 * a [M,K], b [N,K], bias [N] or NULL: host f32 (rounded to bf16 on the device); d [M,N] host f32. */
int ie_debug_gemm(const float* a, const float* b, const float* bias, int32_t M, int32_t N, int32_t K, int32_t act,
                  float* d, int32_t device);

#ifdef __cplusplus
}
#endif
#endif /* ISSUE_EMB_B200_H_ */
