// Internal launch interfaces between the C-ABI layer (api.cu) and the sm_100a kernels.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace ie {

// ---- TMA descriptor helper (tmap.cu) ---------------------------------------------------------
// 2-D bf16 tensor, inner (contiguous) dimension `inner` elements, `rows` rows, row pitch `ld` elements,
// box {box_inner, box_rows}, 128-byte swizzle (box_inner must be 64).
cudaError_t make_tmap_bf16_2d(CUtensorMap* out, const void* base, uint64_t inner, uint64_t rows, uint64_t ld,
                              uint32_t box_inner, uint32_t box_rows);

// ---- GEMM (gemm.cu) ----------------------------------------------------------------------------
struct GemmArgs {
  const __nv_bfloat16* a;  // [m_pad, lda]   (split-bf16: [hi(k_pad) | lo(k_pad)] per row)
  const __nv_bfloat16* b;  // [n_pad, ldb]
  void* d;                 // [m_store.., ldd] f32 or bf16
  const float* bias;       // [n_pad] or nullptr
  int m_pad, n_pad, k_pad;
  long long lda, ldb, ldd;
  int m_store, n_store;
  int bn;        // N tile (multiple of 16, <= 256, divides n_pad)
  int act;       // 0 none, 1 relu, 2 sigmoid
  int out_bf16;  // output type: 0 f32, 1 bf16, 2 fp16 (act must be 0)
  int num_sms;
  int segs;      // 1: bf16 operands; 3: split-bf16 (K loop over [A_hi|A_lo|A_hi] x [B_hi|B_hi|B_lo], ~fp32 products)
  unsigned* abort_flag;  // optional global word raised when a wait exceeds spin_limit (ptx.cuh abort protocol)
  long long spin_limit;  // SM cycles; 0 = default
  long long* diag;       // optional [4]: {clock64, globaltimer ns} at the start and end of CTA 0
};
cudaError_t launch_gemm_bf16(const GemmArgs& g, cudaStream_t stream);

// ---- fallback recurrent step (lstm.cu): one timestep of one 256-row batch per launch -------------------------------
struct LstmStepArgs {
  CUtensorMap tm_h;  // hidden-state ring of the time chunk [(Tc+1)*b_pad rows, ring cols], box {64, 128}
  CUtensorMap tm_w;  // W_hh [4*out_pad rows, cols], box {64, 128}; rows ordered [slice][unit][gate], 32 units / slice
  const void* gx;    // f32 or bf16 [rows, 4*out_pad] (bias folded in): row t*b_pad + brow of the chunk, or token id
  const int* tok;    // optional time-major token ids of the whole call (per-token input-projection table)
  float* c;          // [b_pad, out_pad] cell state
  __nv_bfloat16* y;  // ring (slot 0 = h before the chunk (zeros at t0 = 0); slot t+1 = h_t, t chunk-local)
  float* raw;        // optional [b_pad, T_total, raw_ld] f32 copy of h (get_raw_features)
  float* pool_sum;   // optional [b_pad, out_pad] (last layer only; formats: lstm_common.cuh)
  float* pool_max;
  float* pool_last;
  const int* lengths;  // [b_pad]
  unsigned* abort_flag;
  long long spin_limit;
  int t, t0, T_total;  // chunk-local timestep, global index of the chunk's first timestep, timesteps of the call
  int b_pad;           // rows per time slot (multiple of 256)
  int g;               // which 256-row batch of the slot
  int u, n_cta, out_pad, kh_pad;
  long long ldy, raw_ld;
  int gate_mode, gx_bf16, segs;
};
cudaError_t launch_lstm_step(const LstmStepArgs& a, cudaStream_t stream);

// ---- persistent recurrent layer (lstm_layer.cu): all timesteps of a layer (or of a time chunk) in one cooperative launch,
//      up to kMaxBatches batches of 256 rows; (timestep, batch, tile) items dealt round-robin over all CTA pairs
constexpr int kMaxBatches = 12;
struct LstmLayerArgs {
  CUtensorMap tm_h, tm_w;  // as LstmStepArgs
  CUtensorMap tm_h64;      // same tensor as tm_h with box {64, 64}: the quarter tile one CTA multicasts (mc != 0)
  CUtensorMap tm_x;        // pre_nkb > 0: the PREVIOUS layer's ring (slot t+1 = this layer's x_t), box {64, 128}
  int pre_nkb;             // > 0: fuse the input projection into the K loop -- pre_nkb = kin_pad / 64 k-blocks of
                           // x_t W_ih^T precede the recurrent ones; tm_w then covers [W_ih | W_hh] (inner kin_pad + kh_pad),
                           // gx is unused and `bias` (b_ih + b_hh, permuted like the weight rows) is added instead
  const float* bias;
  int mc;                  // 1: clusters of two CTA pairs share every h tile by TMA multicast (needs an even number of tiles)
  int mc_pairs;            // CTA pairs that can be co-resident in clusters of four (lstm_layer_max_pairs() of a check_only query)
  const void* gx;
  const int* tok;
  float* c;
  __nv_bfloat16* y;
  float* raw;
  float* pool_sum;
  float* pool_max;
  float* pool_last;
  const int* lengths;
  unsigned* step_done;   // [T*ng] zero-initialised (step, batch) counters of this launch
  unsigned* abort_flag;
  long long spin_limit;
  int T, t0, T_total;    // timesteps in this launch, global index of the first, timesteps of the whole call
  int ng;                // batches of 256 rows
  int u, n_cta, out_pad, kh_pad;
  long long ldy, raw_ld;
  int gate_mode, gx_bf16, segs;
  int num_sms, check_only, cooperative;
  int fault;             // debug: drop one counter update (exercises the abort protocol)
  long long* trace;      // optional [grid][trace_items][12] timeline (debug)
  int trace_items;
  long long* diag;       // optional [4]: {clock64, globaltimer ns} at the start and end of CTA 0 (SM clock of the launch)
};
cudaError_t launch_lstm_layer(const LstmLayerArgs& a, cudaStream_t stream);
int lstm_layer_pairs(const LstmLayerArgs& a);  // CTA pairs the launch will use
int lstm_layer_max_pairs();                    // result of the last check_only query on this thread

// ---- small memory-bound kernels (misc.cu) --------------------------------------------------------
// ids [B, T] int64 (batch-first, right padded) -> x0 [(T*b_pad), ldx] bf16, time-major rows t*b_pad + b
// (t0, Tc): only timesteps [t0, t0+Tc) are gathered, into rows (t - t0)*b_pad + b
cudaError_t launch_embed_gather(const int64_t* ids, int B, int T, int b_pad, const __nv_bfloat16* emb, int vocab,
                                int e_pad, __nv_bfloat16* x0, long long ldx, int pad_idx, int* err_flag, int t0, int Tc,
                                cudaStream_t stream);
// lengths_in [B] (device) -> lengths_out [b_pad]: clamped to [1, T] (err_flag[2] raised if it had to clamp), rows >= B: 1
cudaError_t launch_prep_lengths(const int* lengths_in, int B, int T, int b_pad, int* lengths_out, int* err_flag,
                                cudaStream_t stream);
// out[b] = [sum/len | max | last], b < B, first `e` units
// ids [B, T] int64 -> tok [T*b_pad] int32 time-major (rows >= B: pad_idx), range-checked like launch_embed_gather
cudaError_t launch_tokens_time_major(const int64_t* ids, int B, int T, int b_pad, int vocab, int pad_idx, int* tok,
                                     int* err_flag, cudaStream_t stream);
cudaError_t launch_pool_finalize(const float* pool_sum, const float* pool_max, const float* pool_last,
                                 const int* lengths, int B, int e, int out_pad, float* out, cudaStream_t stream);
// f32 [rows, cols] (row pitch ld_src) -> bf16 [rows_pad, ld_dst] with optional row permutation (src row of dst row r
// = perm[r], or -1 for a zero row); columns >= cols zero filled.
// lo_off > 0: split-bf16 layout -- hi = bf16(x) in columns [0, lo_off), lo = bf16(x - hi) in [lo_off, 2*lo_off)
cudaError_t launch_convert_rows(const float* src, long long ld_src, int cols, const int* perm, int rows_dst,
                                __nv_bfloat16* dst, long long ld_dst, int lo_off, cudaStream_t stream);
cudaError_t launch_fill_f32(float* p, size_t n, float v, cudaStream_t stream);

// ---- precision-recall threshold search (pr_curve.cu): scores [n, n_labels] f32, truth [n, n_labels] u8 (device) ----------
constexpr int kPrMaxSamples = 16384;
cudaError_t launch_pr_thresholds(const float* scores, const uint8_t* truth, int n, int n_labels, double p_thr,
                                 double r_thr, float* out_thr, double* out_prec, double* out_rec, cudaStream_t stream);

// ---- exact cosine k-nearest-neighbour search (knn.cu) ---------------------------------------------------------------
// Index prep: inv[r] = 1 / |x_r| (f64, 0 for a zero row); partial column sums of x * inv over blocks of 512 rows (rows
// of this call land in partial blocks [blk0, blk0 + knn_colsum_blocks(rows))); mu = sum of the blocks in order / n.
long long knn_colsum_blocks(long long rows);
cudaError_t launch_knn_inv_norm(const float* x, long long ldx, int d, int rows, double* inv, cudaStream_t stream);
cudaError_t launch_knn_colsum(const float* x, long long ldx, int d, int rows, const double* inv, double* partial,
                              long long blk0, cudaStream_t stream);
cudaError_t launch_knn_mean(const double* partial, long long nblk, int d, int k_pad, long long n, double* mu,
                            cudaStream_t stream);
// rows [rows, d] f32 -> out [rows, 2*k_pad] bf16 = [hi | lo] of f32(x/|x| - mu); bias[r] = f32(mu . r) (nullptr: not
// written; queries), omc[r] = 1 - (x/|x|) . mu; all dot products in f64
cudaError_t launch_knn_prep_rows(const float* x, long long ldx, int d, int rows, const double* mu, int k_pad,
                                 __nv_bfloat16* out, float* bias, double* omc, cudaStream_t stream);
// *flag = 1 if any of x[rows, d] (row pitch ldx) is NaN or infinite
cudaError_t launch_knn_check_finite(const float* x, long long ldx, int d, long long rows, unsigned* flag,
                                    cudaStream_t stream);
constexpr int kKnnMaxK = 32;
struct KnnSearchArgs {
  const __nv_bfloat16* a;      // query operand [a_rows, 2*k_pad] (split-bf16 residuals); rows a_row0 .. a_row0 + m
  long long a_rows;            // rows of the A tensor (reads past it are zero-filled by the TMA unit)
  int a_row0;
  const __nv_bfloat16* index;  // [n_pad, 2*k_pad]
  const float* bias;           // [n_pad] b_x
  int n_valid, n_pad, k_pad;   // n_pad % 256 == 0, k_pad % 64 == 0
  long long self0;             // >= 0: query i is index row self0 + i and skips itself; -1: external queries
  int m, k;                    // queries of this launch, neighbours per query (1..kKnnMaxK)
  const double* omc;           // [m] 1 - c_q
  float* cand_s;               // workspace [m, knn_search_grid(), k]
  int* cand_i;
  float* dist;                 // [m, k]
  int64_t* ids;                // [m, k]
  int num_sms;
  unsigned* abort_flag;
  long long spin_limit;
};
int knn_search_grid(int n_pad, int num_sms);
cudaError_t launch_knn_search(const KnnSearchArgs& a, cudaStream_t stream);

}  // namespace ie
