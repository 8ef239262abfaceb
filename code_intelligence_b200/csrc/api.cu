// C-ABI layer of libissue_emb_b200.so (declared in include/issue_emb_b200.h): handle management, weight
// re-layout, workspace, and the launch sequence of the encoder hot path and the MLP head.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/issue_emb_b200.h"
#include "kernels.h"

namespace {

thread_local std::string g_last_error;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

int cuda_fail(cudaError_t e, const char* what) {
  const int code = (e == cudaErrorMemoryAllocation) ? IE_ERR_OOM : IE_ERR_CUDA;
  if (e == cudaErrorMemoryAllocation) cudaGetLastError();  // clear the sticky-free OOM
  return fail(code, "%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
}

#define CK(expr)                                              \
  do {                                                        \
    cudaError_t _e = (expr);                                  \
    if (_e != cudaSuccess) return cuda_fail(_e, #expr);       \
  } while (0)

inline long long round_up(long long x, long long m) { return (x + m - 1) / m * m; }

// grow-only device buffer; owns its allocation (freed on destruction, so error paths do not leak)
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
  DevBuf& operator=(DevBuf&& o) noexcept {
    if (this != &o) { release(); p = o.p; cap = o.cap; o.p = nullptr; o.cap = 0; }
    return *this;
  }
  ~DevBuf() { release(); }
  cudaError_t reserve(size_t bytes, bool zero = false) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) { p = nullptr; return e; }
    cap = bytes;
    if (zero) {
      // the handle's streams are non-blocking: make the (legacy-stream) memset complete before anyone uses it
      e = cudaMemset(p, 0, bytes);
      if (e != cudaSuccess) return e;
      return cudaDeviceSynchronize();
    }
    return cudaSuccess;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct Layer {
  int in = 0, out = 0;      // logical dims
  int u = 32, n_cta = 0;    // hidden units per weight slice (CTA), slices (even: CTA pairs own two)
  int out_pad = 0;          // n_cta * u
  int kin_pad = 0;          // padded K of the input projection
  int kh_pad = 0;           // padded K of the recurrent projection
  int bn = 0;               // GEMM N tile for the input projection
  DevBuf w_ih, w_hh, bias;  // sliced layouts
  DevBuf w_cat;             // last layer: rows [W_ih (kin_pad) | W_hh (kh_pad)] for the fused input projection
  bool loaded = false;
};

}  // namespace

struct ie_encoder {
  ie_config cfg{};
  int num_sms = 148;
  int e_pad = 0;  // emb_sz rounded up to 64
  // one weight layout: slices of u = 32 hidden units, rows [slice][unit][gate]; a CTA pair owns two slices = one
  // N = 256 accumulator tile (lstm_layer.cu), the fallback kernel one slice per CTA (lstm.cu)
  std::vector<Layer> layers;
  int segs = 1;            // 1: bf16 operands; 3: split-bf16 ("fp32-accurate", IE_CFG_FP32)
  int gate_mode = 2;       // lstm_common.cuh: 2 tanh.approx, 1 ex2+rcp, 0 IEEE
  int gx_bf16 = 1;         // input projections (Gx, per-token table) stored as 16-bit floats -- IEEE half -- instead of f32
                           // (f32 in the fp32-accurate mode)
  int use_persistent = 1;  // cooperative persistent kernel; 0 (IE_SEQ=0 or not co-resident): per-timestep fallback
  int persist_checked = 0;
  int cooperative = 1;     // launch attribute (IE_COOP=0: plain launch, co-residency by the occupancy check only)
  int use_mc = 0;          // IE_MC=1: sibling CTA pairs share h tiles by TMA multicast (clusters of four)
  int mc_pairs = 0;        // pairs co-resident in clusters of four
  int batches = 5;         // batches of 256 rows one launch takes (IE_BATCHES, <= kMaxBatches)
  int fuse_last = 1;       // the last layer's input projection rides its recurrent K loop (lstm_layer.cu FUSE) instead of a
                           // hoisted GEMM + Gx round trip (IE_FUSE_LAST=0: hoisted like the other layers)
  int max_batch = 1280;
  // layer 0's input projection W_ih0 . Emb[id] + b depends on the token id alone: tabulated once per weight set
  // (proj: [vocab_pad, 4*out_pad], computed by the same GEMM from the same operands => the same bits as gather + GEMM)
  // and the recurrent kernel reads row tok[t, b] of it: no embedding gather, no layer-0 GEMM, no Gx write for layer 0
  int use_proj = 1;
  bool proj_built = false;
  DevBuf proj, tok;
  DevBuf emb;  // bf16 [vocab_pad, e_pad] (split mode: [hi | lo])
  bool emb_loaded = false;
  long long spin_limit = 0;  // SM cycles a device-side wait may take (0: default ~2 s); IE_SPIN_LIMIT_MS
  int fault = 0;             // IE_DEBUG_FAULT: exercise the abort protocol
  long long chunk_t = 0;     // IE_CHUNK_T: force the time-chunk length (testing)
  // workspace
  DevBuf ids, len_in, lengths, x0, y[2], hcarry, gx, c, pool_sum, pool_max, pool_last, out, raw, err, step_done, diag;
  DevBuf trace;           // debug timeline of one layer of the persistent kernel (ie_debug_seq_trace)
  int trace_layer = -1;
  int trace_T = 0, trace_ctas = 0;
  long long y_ld = 0;
  long long ws_tokens = 0;  // largest b_pad*T the workspace was grown for
  int small_calls = 0;      // consecutive calls far below ws_tokens (workspace is released after a few)
  cudaStream_t own_stream = nullptr;
  cudaStream_t last_stream = nullptr;
  cudaEvent_t done_ev = nullptr;  // end of the last call: a call on another stream waits for it (shared workspace)
  bool has_done = false;
  int64_t launches = 0;
  // phase boundary events of the last encode call and what ended at each (0 start, 1 gather, 2+2l gemm_l, 3+2l steps_l,
  // 2+2L finalize)
  std::vector<cudaEvent_t> ev;
  std::vector<int> ev_tag;
  int ev_used = 0;
  int last_T = 0, last_b_pad = 0;
  std::mutex mu;
};

struct ie_mlp {
  int device = 0;
  int num_sms = 148;
  std::vector<int> dims;
  struct L {
    int k_pad = 0, n_pad = 0, bn = 0;
    DevBuf w, b;
    bool loaded = false;
  };
  std::vector<L> layers;
  DevBuf xf, act[2], probs;
  DevBuf xb;                // bf16 copy of one row chunk of X
  long long act_ld = 0;
  int chunk_dev = 1 << 18;  // rows per pass in device-pointer mode (IE_MLP_CHUNK at create time)
  cudaStream_t own_stream = nullptr;
  std::mutex mu;
};

struct ie_knn {
  int device = 0;
  int num_sms = 148;
  long long n = 0;
  int d = 0, k_pad = 0, n_pad = 0;
  DevBuf index;  // bf16 [n_pad, 2*k_pad]: [hi | lo] of the f32 residual x/|x| - mean; padding rows zero
  DevBuf bias;   // f32 [n_pad]: b_x = mean . r_x
  DevBuf omc;    // f64 [n]: 1 - c_x = 1 - (x/|x|) . mean (self-queries)
  DevBuf mean;   // f64 [k_pad]: mean of the unit vectors
  // search workspace
  DevBuf qf, qa, qomc, cand_s, cand_i, dist, ids, err;
  cudaStream_t own_stream = nullptr;
  cudaStream_t last_stream = nullptr;
  cudaEvent_t done_ev = nullptr;  // end of the last call: a call on another stream waits for it (shared workspace)
  bool has_done = false;
  std::mutex mu;
  ~ie_knn() {
    if (done_ev) cudaEventDestroy(done_ev);
    if (own_stream) cudaStreamDestroy(own_stream);
  }
};

namespace {

constexpr int kErrWords = 4;  // err[0] token id out of range, err[1] device-side wait timed out (abort protocol),
                              // err[2] a length had to be clamped (device-pointer mode)

int plan_layers(ie_encoder* h) {
  const ie_config& c = h->cfg;
  h->e_pad = static_cast<int>(round_up(c.emb_sz, 64));
  h->layers.resize(c.n_layers);
  int prev_pad = h->e_pad;
  for (int l = 0; l < c.n_layers; ++l) {
    Layer& L = h->layers[l];
    L.in = (l == 0) ? c.emb_sz : c.n_hid;
    L.out = (l == c.n_layers - 1) ? c.emb_sz : c.n_hid;
    L.u = 32;
    L.n_cta = (L.out + L.u - 1) / L.u;
    if (L.n_cta & 1) ++L.n_cta;  // CTA pairs: the last pair's second slice is pure padding
    L.out_pad = L.n_cta * L.u;
    L.kin_pad = prev_pad;
    L.kh_pad = L.out_pad;        // multiple of 64
    prev_pad = L.kh_pad;
    L.bn = 256;                  // 4*out_pad is a multiple of 256
  }
  return IE_OK;
}

// torch gate-major rows [4*out] -> sliced rows [slice][unit][gate]; -1 marks zero padding rows
std::vector<int> slice_perm(const Layer& L) {
  std::vector<int> perm(4 * static_cast<size_t>(L.out_pad));
  for (int j = 0; j < L.n_cta; ++j)
    for (int i = 0; i < L.u; ++i)
      for (int g = 0; g < 4; ++g) {
        const int unit = j * L.u + i;
        perm[(static_cast<size_t>(j) * L.u + i) * 4 + g] = unit < L.out ? g * L.out + unit : -1;
      }
  return perm;
}

// host f32 [rows_src, cols] -> device bf16 [perm.size(), ld] (split mode: [hi(k_pad) | lo(k_pad)], ld = 2*k_pad)
int upload_sliced(const float* host, int rows_src, int cols, const std::vector<int>& perm, int k_pad, int segs, DevBuf& dst,
                  cudaStream_t s) {
  DevBuf tmp, dperm;
  const int ld_dst = segs > 1 ? 2 * k_pad : k_pad;
  CK(tmp.reserve(static_cast<size_t>(rows_src) * cols * sizeof(float)));
  CK(dperm.reserve(perm.size() * sizeof(int)));
  CK(cudaMemcpyAsync(tmp.p, host, static_cast<size_t>(rows_src) * cols * sizeof(float), cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(dperm.p, perm.data(), perm.size() * sizeof(int), cudaMemcpyHostToDevice, s));
  CK(dst.reserve(perm.size() * static_cast<size_t>(ld_dst) * sizeof(__nv_bfloat16)));
  CK(ie::launch_convert_rows(tmp.as<float>(), cols, cols, dperm.as<int>(), static_cast<int>(perm.size()),
                             dst.as<__nv_bfloat16>(), ld_dst, segs > 1 ? k_pad : 0, s));
  CK(cudaStreamSynchronize(s));
  tmp.release();
  dperm.release();
  return IE_OK;
}

long long max_out_pad(const ie_encoder* h) {
  long long m = 0;
  for (const Layer& L : h->layers) m = std::max<long long>(m, L.out_pad);
  return m;
}

void release_workspace(ie_encoder* h) {
  DevBuf* bufs[] = {&h->ids, &h->x0, &h->y[0], &h->y[1], &h->gx, &h->raw, &h->step_done, &h->tok};
  for (DevBuf* b : bufs) b->release();
  h->ws_tokens = 0;
  h->small_calls = 0;
}

// The time dimension is processed in chunks of chunk_T steps (time-major: every layer runs a chunk before the next
// chunk starts; c and h are carried per layer), so everything but the token ids is bounded by chunk_T * b_pad rows.
int ensure_workspace(ie_encoder* h, int b_pad, int T, int chunk_T, bool want_raw, bool need_x0, bool need_tok) {
  const ie_config& c = h->cfg;
  const long long mop = max_out_pad(h);
  const long long rows = static_cast<long long>(T) * b_pad;
  const long long crow = static_cast<long long>(chunk_T) * b_pad;
  const int ring_mul = h->segs > 1 ? 2 : 1;
  CK(h->ids.reserve(static_cast<size_t>(h->max_batch) * T * sizeof(int64_t)));
  CK(h->len_in.reserve(h->max_batch * sizeof(int)));
  CK(h->lengths.reserve(h->max_batch * sizeof(int)));
  CK(h->err.reserve(kErrWords * sizeof(int), true));
  CK(h->diag.reserve(static_cast<size_t>(c.n_layers) * 8 * sizeof(long long), true));
  if (need_x0) CK(h->x0.reserve(static_cast<size_t>(crow) * ring_mul * h->e_pad * sizeof(__nv_bfloat16)));
  // hidden-state rings of one chunk: (chunk_T + 1) slots of b_pad rows; slot 0 = the layer's h before the chunk (carry).
  // Every column a tensor map can reach is written before it is read (padded units produce exact zeros).
  h->y_ld = ring_mul * mop;
  const size_t ybytes = static_cast<size_t>(crow + b_pad) * h->y_ld * sizeof(__nv_bfloat16);
  for (int i = 0; i < 2; ++i) CK(h->y[i].reserve(ybytes));
  CK(h->hcarry.reserve(static_cast<size_t>(c.n_layers) * h->max_batch * h->y_ld * sizeof(__nv_bfloat16)));
  CK(h->gx.reserve(static_cast<size_t>(crow) * 4 * mop * (h->gx_bf16 ? 2 : 4)));
  CK(h->c.reserve(static_cast<size_t>(c.n_layers) * h->max_batch * mop * sizeof(float)));
  const size_t pb = static_cast<size_t>(h->max_batch) * mop * sizeof(float);
  CK(h->pool_sum.reserve(pb));
  CK(h->pool_max.reserve(pb));
  CK(h->pool_last.reserve(pb));
  CK(h->out.reserve(static_cast<size_t>(h->max_batch) * 3 * c.emb_sz * sizeof(float)));
  if (want_raw) CK(h->raw.reserve(static_cast<size_t>(b_pad) * T * mop * sizeof(float)));
  CK(h->step_done.reserve(static_cast<size_t>(chunk_T) * ie::kMaxBatches * sizeof(unsigned)));
  if (need_tok) CK(h->tok.reserve(static_cast<size_t>(rows) * sizeof(int)));
  h->ws_tokens = std::max(h->ws_tokens, crow);
  return IE_OK;
}

int mark(ie_encoder* h, int tag, cudaStream_t s) {
  if (h->ev_used >= static_cast<int>(h->ev.size())) {
    cudaEvent_t e;
    CK(cudaEventCreate(&e));
    h->ev.push_back(e);
    h->ev_tag.push_back(0);
  }
  h->ev_tag[h->ev_used] = tag;
  CK(cudaEventRecord(h->ev[h->ev_used++], s));
  return IE_OK;
}

bool proj_usable(const ie_encoder* h) {
  if (!h->use_proj) return false;
  const Layer& L = h->layers[0];
  const long long v_pad = round_up(h->cfg.vocab_sz, 256);
  const long long bytes = v_pad * 4ll * L.out_pad * (h->gx_bf16 ? 2 : 4);
  return bytes <= (6ll << 30);  // huge vocabularies fall back to gather + GEMM
}

void fill_gemm(const ie_encoder* h, const Layer& L, ie::GemmArgs& g) {
  g.b = L.w_ih.as<__nv_bfloat16>();
  g.ldb = static_cast<long long>(h->segs > 1 ? 2 : 1) * L.kin_pad;
  g.ldd = 4ll * L.out_pad;
  g.bias = L.bias.as<float>();
  g.n_pad = 4 * L.out_pad;
  g.k_pad = L.kin_pad;
  g.n_store = 4 * L.out_pad;
  g.bn = L.bn;
  g.act = 0;
  g.out_bf16 = h->gx_bf16 ? 2 : 0;  // fp16 or f32
  g.num_sms = h->num_sms;
  g.segs = h->segs;
  g.abort_flag = h->err.as<unsigned>() + 1;
  g.spin_limit = h->spin_limit;
}

// tabulate layer 0's input projection for every token id (once per weight set)
int build_proj_table(ie_encoder* h, cudaStream_t s) {
  const Layer& L = h->layers[0];
  const long long v_pad = round_up(h->cfg.vocab_sz, 256);
  CK(h->proj.reserve(static_cast<size_t>(v_pad) * 4 * L.out_pad * (h->gx_bf16 ? 2 : 4)));
  ie::GemmArgs g{};
  fill_gemm(h, L, g);
  g.a = h->emb.as<__nv_bfloat16>();
  g.lda = static_cast<long long>(h->segs > 1 ? 2 : 1) * h->e_pad;
  g.d = h->proj.p;
  g.m_pad = static_cast<int>(v_pad);
  g.m_store = static_cast<int>(v_pad);
  CK(ie::launch_gemm_bf16(g, s));
  h->launches++;
  h->proj_built = true;
  return IE_OK;
}

int check_persistent(ie_encoder* h, cudaStream_t s) {
  if (h->persist_checked) return IE_OK;
  for (const Layer& L : h->layers) {
    ie::LstmLayerArgs q{};
    q.T = 1; q.ng = 1; q.u = L.u; q.n_cta = L.n_cta; q.out_pad = L.out_pad; q.kh_pad = L.kh_pad; q.segs = 1;
    q.num_sms = h->num_sms; q.check_only = 1;
    if (ie::launch_lstm_layer(q, s) != cudaSuccess) h->use_persistent = 0;
  }
  if (h->use_mc) {
    ie::LstmLayerArgs q{};
    const Layer& L = h->layers[0];
    q.T = 1; q.ng = 1; q.u = L.u; q.n_cta = L.n_cta; q.out_pad = L.out_pad; q.kh_pad = L.kh_pad; q.segs = 1;
    q.num_sms = h->num_sms; q.check_only = 1; q.mc = 1; q.gx_bf16 = 1;
    if (ie::launch_lstm_layer(q, s) == cudaSuccess) h->mc_pairs = ie::lstm_layer_max_pairs() & ~1;
    if (h->mc_pairs < 2) h->use_mc = 0;
  }
  cudaGetLastError();
  h->persist_checked = 1;
  return IE_OK;
}

// the launch sequence shared by encode (pooled) and raw_features
int run_encoder(ie_encoder* h, const int64_t* ids, const int32_t* lengths, int B, int T, float* out, float* raw_out,
                int flags, cudaStream_t s) {
  const ie_config& c = h->cfg;
  if (!h->emb_loaded) return fail(IE_ERR_STATE, "embedding not loaded");
  for (const Layer& L : h->layers)
    if (!L.loaded) return fail(IE_ERR_STATE, "LSTM layer weights not loaded");
  if (B < 1 || B > h->max_batch) return fail(IE_ERR_INVALID, "B=%d outside [1,%d]", B, h->max_batch);
  if (T < 1) return fail(IE_ERR_INVALID, "T=%d must be >= 1", T);
  if (ids == nullptr || (out == nullptr && raw_out == nullptr)) return fail(IE_ERR_INVALID, "null pointer");
  const bool dev = (flags & IE_FLAG_DEVICE_PTRS) != 0;
  const bool pooled = out != nullptr;
  const int ng = (B + 255) / 256;
  const int b_pad = 256 * ng;
  // IE_MAX_TOKENS: artificial cap on B_pad*T (exercises the callers' OOM batch-halving loop); real limits come from
  // cudaMalloc (-> IE_ERR_OOM) -- only the token ids grow with T, everything else is bounded by the time chunk
  long long cap = 1ll << 27;
  if (const char* e = getenv("IE_MAX_TOKENS")) cap = std::max(256ll, atoll(e));
  if (static_cast<long long>(b_pad) * T > cap)
    return fail(IE_ERR_OOM, "B_pad*T = %lld tokens exceeds the workspace cap %lld; use a smaller batch",
                static_cast<long long>(b_pad) * T, cap);
  CK(cudaSetDevice(c.device));
  // <= 2^21 (timestep, row) pairs of Gx at once (40 GB as fp16 at H = 2400); half of that with f32 projections
  long long chunk_T = std::max<long long>(1, ((h->gx_bf16 ? 2ll : 1ll) << 20) / b_pad);
  if (h->chunk_t > 0) chunk_T = h->chunk_t;
  chunk_T = std::min<long long>(chunk_T, T);
  const bool proj = proj_usable(h);
  int rc = ensure_workspace(h, b_pad, T, static_cast<int>(chunk_T), raw_out != nullptr, !proj, proj);
  if (rc != IE_OK) return rc;
  if (h->done_ev == nullptr) CK(cudaEventCreateWithFlags(&h->done_ev, cudaEventDisableTiming));
  // one workspace per handle: a call on another stream first waits for the previous call
  if (h->has_done && h->last_stream != s) CK(cudaStreamWaitEvent(s, h->done_ev, 0));

  CK(cudaMemsetAsync(h->err.p, 0, kErrWords * sizeof(int), s));
  CK(cudaMemsetAsync(h->diag.p, 0, static_cast<size_t>(c.n_layers) * 8 * sizeof(long long), s));
  if (pooled) {
    if (lengths == nullptr) return fail(IE_ERR_INVALID, "lengths is null");
    const int* len_src = lengths;
    if (!dev) {
      for (int b = 0; b < B; ++b)
        if (lengths[b] < 1 || lengths[b] > T)
          return fail(IE_ERR_INVALID, "lengths[%d]=%d outside [1,%d]", b, lengths[b], T);
      CK(cudaMemcpyAsync(h->len_in.p, lengths, B * sizeof(int), cudaMemcpyHostToDevice, s));
      len_src = h->len_in.as<int>();
    }
    CK(ie::launch_prep_lengths(len_src, B, T, b_pad, h->lengths.as<int>(), h->err.as<int>(), s));
  }
  const int64_t* ids_dev = ids;
  if (!dev) {
    CK(cudaMemcpyAsync(h->ids.p, ids, static_cast<size_t>(B) * T * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    ids_dev = h->ids.as<int64_t>();
  }

  h->ev_used = 0;
  h->last_T = T;
  h->last_b_pad = b_pad;
  if (proj && !h->proj_built && (rc = build_proj_table(h, s)) != IE_OK) return rc;
  if ((rc = mark(h, 0, s)) != IE_OK) return rc;
  const int ring_mul = h->segs > 1 ? 2 : 1;
  const long long mop = max_out_pad(h);
  if (proj) {
    CK(ie::launch_tokens_time_major(ids_dev, B, T, b_pad, c.vocab_sz, c.pad_idx, h->tok.as<int>(), h->err.as<int>(), s));
    h->launches++;
  }
  if (h->use_persistent) check_persistent(h, s);
  const bool persistent = h->use_persistent != 0;
  // h_{-1} = 0 for every layer
  const size_t carry_layer = static_cast<size_t>(h->max_batch) * h->y_ld;  // elements
  CK(cudaMemsetAsync(h->hcarry.p, 0, static_cast<size_t>(c.n_layers) * carry_layer * sizeof(__nv_bfloat16), s));
  const size_t slot_bytes = static_cast<size_t>(b_pad) * h->y_ld * sizeof(__nv_bfloat16);

  for (long long t0 = 0; t0 < T; t0 += chunk_T) {
    const int Tc = static_cast<int>(std::min<long long>(chunk_T, T - t0));
    const long long crow = static_cast<long long>(Tc) * b_pad;
    if (!proj) {
      CK(ie::launch_embed_gather(ids_dev, B, T, b_pad, h->emb.as<__nv_bfloat16>(), c.vocab_sz, ring_mul * h->e_pad,
                                 h->x0.as<__nv_bfloat16>(), ring_mul * h->e_pad, c.pad_idx, h->err.as<int>(),
                                 static_cast<int>(t0), Tc, s));
      h->launches++;
    }
    if ((rc = mark(h, 1, s)) != IE_OK) return rc;
    int cur = 0;
    const __nv_bfloat16* layer_in = h->x0.as<__nv_bfloat16>();
    const __nv_bfloat16* prev_ring = nullptr;  // the previous layer's ring (slot 0 included)
    long long layer_in_ld = ring_mul * h->e_pad;
    for (int l = 0; l < c.n_layers; ++l) {
      const bool last = (l == c.n_layers - 1);
      Layer& L = h->layers[l];
      const bool from_table = proj && l == 0;  // Gx rows of layer 0 are rows of the per-token table: no GEMM
      // last layer: input projection fused into the recurrent K loop (no GEMM, no Gx)
      const bool fused = persistent && last && l > 0 && h->segs == 1 && h->fuse_last && L.w_cat.p != nullptr;
      __nv_bfloat16* ybuf = h->y[cur].as<__nv_bfloat16>();
      __nv_bfloat16* carry = h->hcarry.as<__nv_bfloat16>() + static_cast<size_t>(l) * carry_layer;
      float* cstate = h->c.as<float>() + static_cast<size_t>(l) * h->max_batch * mop;
      CUtensorMap tm_h, tm_w;
      CK(ie::make_tmap_bf16_2d(&tm_h, ybuf, static_cast<uint64_t>(ring_mul) * L.kh_pad, static_cast<uint64_t>(crow + b_pad),
                               h->y_ld, 64, 128));
      if (fused)
        CK(ie::make_tmap_bf16_2d(&tm_w, L.w_cat.p, static_cast<uint64_t>(L.kin_pad + L.kh_pad), 4ull * L.out_pad,
                                 static_cast<uint64_t>(L.kin_pad + L.kh_pad), 64, 128));
      else
        CK(ie::make_tmap_bf16_2d(&tm_w, L.w_hh.p, static_cast<uint64_t>(ring_mul) * L.kh_pad, 4ull * L.out_pad,
                                 static_cast<uint64_t>(ring_mul) * L.kh_pad, 64, 128));
      CUtensorMap tm_h64 = tm_h;
      CUtensorMap tm_x = tm_h;
      if (fused)
        CK(ie::make_tmap_bf16_2d(&tm_x, prev_ring, static_cast<uint64_t>(L.kin_pad), static_cast<uint64_t>(crow + b_pad),
                                 h->y_ld, 64, 128));
      if (h->use_mc)
        CK(ie::make_tmap_bf16_2d(&tm_h64, ybuf, static_cast<uint64_t>(ring_mul) * L.kh_pad,
                                 static_cast<uint64_t>(crow + b_pad), h->y_ld, 64, 64));
      // slot 0 of the ring = this layer's h at the end of the previous chunk (zeros before the first)
      CK(cudaMemcpyAsync(ybuf, carry, slot_bytes, cudaMemcpyDeviceToDevice, s));
      if (!from_table && !fused) {
        // hoisted input projection over the chunk's Tc*b_pad rows
        ie::GemmArgs g{};
        fill_gemm(h, L, g);
        g.a = layer_in;
        g.lda = layer_in_ld;
        g.d = h->gx.p;
        g.m_pad = static_cast<int>(crow);
        g.m_store = static_cast<int>(crow);
        g.diag = h->diag.as<long long>() + 8 * l + 4;
        CK(ie::launch_gemm_bf16(g, s));
        h->launches++;
      }
      if ((rc = mark(h, 2 + 2 * l, s)) != IE_OK) return rc;

      if (persistent) {
        CK(cudaMemsetAsync(h->step_done.p, 0, static_cast<size_t>(Tc) * ng * sizeof(unsigned), s));
        ie::LstmLayerArgs q{};
        q.tm_h = tm_h; q.tm_w = tm_w; q.tm_h64 = tm_h64; q.mc = h->use_mc; q.mc_pairs = h->mc_pairs;
        q.tm_x = tm_x; q.pre_nkb = fused ? L.kin_pad / 64 : 0; q.bias = L.bias.as<float>();
        q.gx = from_table ? h->proj.p : h->gx.p;
        q.tok = from_table ? h->tok.as<int>() : nullptr;
        q.c = cstate; q.y = ybuf;
        q.raw = (last && raw_out != nullptr) ? h->raw.as<float>() : nullptr;
        q.pool_sum = (last && pooled) ? h->pool_sum.as<float>() : nullptr;
        q.pool_max = h->pool_max.as<float>(); q.pool_last = h->pool_last.as<float>();
        q.lengths = h->lengths.as<int>();
        q.step_done = h->step_done.as<unsigned>();
        q.abort_flag = h->err.as<unsigned>() + 1; q.spin_limit = h->spin_limit;
        q.T = Tc; q.t0 = static_cast<int>(t0); q.T_total = T; q.ng = ng;
        q.u = L.u; q.n_cta = L.n_cta; q.out_pad = L.out_pad; q.kh_pad = L.kh_pad;
        q.ldy = h->y_ld; q.raw_ld = L.out_pad;
        q.gate_mode = h->gate_mode; q.gx_bf16 = h->gx_bf16; q.segs = h->segs;
        q.num_sms = h->num_sms; q.check_only = 0; q.cooperative = h->cooperative; q.fault = h->fault;
        q.diag = h->diag.as<long long>() + 8 * l;
        q.trace = nullptr;
        if (l == h->trace_layer && t0 == 0) {
          const int pairs = ie::lstm_layer_pairs(q);
          const long long items = (static_cast<long long>(Tc) * ng * (L.n_cta / 2) + pairs - 1) / pairs;
          CK(h->trace.reserve(static_cast<size_t>(2 * pairs) * items * 12 * sizeof(long long), true));
          q.trace = h->trace.as<long long>();
          q.trace_items = static_cast<int>(items);
          h->trace_T = static_cast<int>(items);
          h->trace_ctas = 2 * pairs;
        }
        cudaError_t e = ie::launch_lstm_layer(q, s);
        if (e == cudaErrorCooperativeLaunchTooLarge) {
          cudaGetLastError();
          return fail(IE_ERR_STATE, "the persistent recurrent kernel cannot be co-resident on this device "
                                   "(cooperative launch refused); set IE_SEQ=0 for the per-timestep fallback");
        }
        CK(e);
        h->launches += 1;
      } else {
        ie::LstmStepArgs a{};
        a.tm_h = tm_h; a.tm_w = tm_w;
        a.gx = from_table ? h->proj.p : h->gx.p;
        a.tok = from_table ? h->tok.as<int>() : nullptr;
        a.c = cstate; a.y = ybuf;
        a.raw = (last && raw_out != nullptr) ? h->raw.as<float>() : nullptr;
        a.pool_sum = (last && pooled) ? h->pool_sum.as<float>() : nullptr;
        a.pool_max = h->pool_max.as<float>(); a.pool_last = h->pool_last.as<float>();
        a.lengths = h->lengths.as<int>();
        a.abort_flag = h->err.as<unsigned>() + 1; a.spin_limit = h->spin_limit;
        a.t0 = static_cast<int>(t0); a.T_total = T; a.b_pad = b_pad;
        a.u = L.u; a.n_cta = L.n_cta; a.out_pad = L.out_pad; a.kh_pad = L.kh_pad;
        a.ldy = h->y_ld; a.raw_ld = L.out_pad;
        a.gate_mode = h->gate_mode; a.gx_bf16 = h->gx_bf16; a.segs = h->segs;
        for (int t = 0; t < Tc; ++t)
          for (int g = 0; g < ng; ++g) {
            a.t = t; a.g = g;
            CK(ie::launch_lstm_step(a, s));
          }
        h->launches += static_cast<int64_t>(Tc) * ng;
      }
      if (t0 + Tc < T)  // carry h of the chunk's last step into the next chunk
        CK(cudaMemcpyAsync(carry, ybuf + static_cast<size_t>(Tc) * b_pad * h->y_ld, slot_bytes, cudaMemcpyDeviceToDevice, s));
      if ((rc = mark(h, 3 + 2 * l, s)) != IE_OK) return rc;
      prev_ring = ybuf;
      layer_in = ybuf + static_cast<long long>(b_pad) * h->y_ld;  // slot 1 onwards
      layer_in_ld = h->y_ld;
      cur ^= 1;
    }
  }
  const long long rows = static_cast<long long>(T) * b_pad;

  const Layer& LL = h->layers.back();
  if (pooled) {
    float* out_dev = dev ? out : h->out.as<float>();
    CK(ie::launch_pool_finalize(h->pool_sum.as<float>(), h->pool_max.as<float>(), h->pool_last.as<float>(),
                                h->lengths.as<int>(), B, c.emb_sz, LL.out_pad, out_dev, s));
    h->launches++;
    if ((rc = mark(h, 2 + 2 * c.n_layers, s)) != IE_OK) return rc;
    if (!dev)
      CK(cudaMemcpyAsync(out, out_dev, static_cast<size_t>(B) * 3 * c.emb_sz * sizeof(float), cudaMemcpyDeviceToHost, s));
  }
  if (raw_out != nullptr) {
    // raw workspace is [b_pad, T, out_pad]; compact to [B, T, emb_sz]
    CK(cudaMemcpy2DAsync(raw_out, static_cast<size_t>(c.emb_sz) * sizeof(float), h->raw.p,
                         static_cast<size_t>(LL.out_pad) * sizeof(float), static_cast<size_t>(c.emb_sz) * sizeof(float),
                         static_cast<size_t>(B) * T, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, s));
  }
  CK(cudaEventRecord(h->done_ev, s));
  h->has_done = true;
  h->last_stream = s;
  // a handle that once served a very long sequence does not keep tens of GB for ever
  if (h->ws_tokens > (1ll << 21) && std::min<long long>(rows, chunk_T * b_pad) * 8 < h->ws_tokens) {
    if (++h->small_calls >= 4) {
      CK(cudaStreamSynchronize(s));
      release_workspace(h);
    }
  } else {
    h->small_calls = 0;
  }
  return IE_OK;
}

// read and clear the device error words of the last call (waits for it)
int collect_errors(ie_encoder* h) {
  if (!h->has_done) return IE_OK;
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaEventSynchronize(h->done_ev));
  int w[kErrWords] = {0, 0, 0, 0};
  CK(cudaMemcpy(w, h->err.p, sizeof(w), cudaMemcpyDeviceToHost));
  if (w[0] | w[1] | w[2]) CK(cudaMemset(h->err.p, 0, sizeof(w)));
  if (w[1] != 0) {
    h->use_persistent = h->fault ? h->use_persistent : 0;  // do not walk into the same wall again
    return fail(IE_ERR_CUDA, "a device-side wait exceeded its limit and the kernel was drained (the persistent grid lost "
                             "co-residency, or a protocol error); results of this call are invalid");
  }
  if (w[0] != 0) return fail(IE_ERR_TOKEN, "token id outside [0,%d) in ids", h->cfg.vocab_sz);
  if (w[2] != 0) return fail(IE_ERR_INVALID, "a length outside [1,T] was clamped");
  return IE_OK;
}

}  // namespace

extern "C" {

int ie_version(void) { return 200; }

const char* ie_last_error(void) { return g_last_error.c_str(); }

int ie_encoder_create(const ie_config* cfg, ie_encoder** out) {
  if (cfg == nullptr || out == nullptr) return fail(IE_ERR_INVALID, "null argument");
  if (cfg->n_layers < 1 || cfg->n_layers > 16 || cfg->emb_sz < 1 || cfg->n_hid < 1 || cfg->vocab_sz < 1 ||
      cfg->pad_idx < 0 || cfg->pad_idx >= cfg->vocab_sz)
    return fail(IE_ERR_INVALID, "bad encoder config");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(IE_ERR_CUDA, "no CUDA device available (%s): this library has no CPU fallback",
                cudaGetErrorString(e));
  if (cfg->device < 0 || cfg->device >= ndev) return fail(IE_ERR_INVALID, "device %d not in [0,%d)", cfg->device, ndev);
  CK(cudaSetDevice(cfg->device));
  int major = 0, sms = 0;
  CK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, cfg->device));
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cfg->device));
  if (major != 10) return fail(IE_ERR_CUDA, "device compute capability %d.x is not sm_100 (B200)", major);
  ie_encoder* h = new ie_encoder();
  h->cfg = *cfg;
  h->num_sms = sms;
  if (cfg->flags & IE_CFG_FP32) {  // split-bf16 products (~fp32), f32 Gx, IEEE gates
    h->segs = 3;
    h->gx_bf16 = 0;
    h->gate_mode = 0;
  } else {
    h->gate_mode = (cfg->flags & IE_CFG_ACCURATE_GATES) ? 1 : 2;
    if (cfg->flags & IE_CFG_F32_GX) h->gx_bf16 = 0;
  }
  // development knobs (DESIGN.md section 4); none is needed in production
  if (const char* v = getenv("IE_SEQ")) h->use_persistent = atoi(v);
  if (const char* v = getenv("IE_COOP")) h->cooperative = atoi(v);
  if (const char* v = getenv("IE_MC")) h->use_mc = atoi(v);
  if (const char* v = getenv("IE_EMB_PROJ")) h->use_proj = atoi(v);
  if (const char* v = getenv("IE_GX_BF16")) { if (h->segs == 1) h->gx_bf16 = atoi(v); }
  if (const char* v = getenv("IE_FAST_MATH")) { if (h->segs == 1) h->gate_mode = atoi(v) ? 2 : 1; }
  if (const char* v = getenv("IE_FUSE_LAST")) h->fuse_last = atoi(v);
  if (const char* v = getenv("IE_BATCHES")) h->batches = std::min(ie::kMaxBatches, std::max(1, atoi(v)));
  if (const char* v = getenv("IE_SPIN_LIMIT_MS")) h->spin_limit = static_cast<long long>(atof(v) * 1.9e6);
  if (const char* v = getenv("IE_DEBUG_FAULT")) h->fault = atoi(v);
  if (const char* v = getenv("IE_CHUNK_T")) h->chunk_t = atoll(v);
  h->max_batch = 256 * h->batches;
  int rc = plan_layers(h);
  if (rc != IE_OK) { delete h; return rc; }
  e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) { delete h; return cuda_fail(e, "cudaStreamCreate"); }
  *out = h;
  return IE_OK;
}

void ie_encoder_destroy(ie_encoder* h) {
  if (h == nullptr) return;
  cudaSetDevice(h->cfg.device);
  cudaDeviceSynchronize();
  for (Layer& L : h->layers) { L.w_ih.release(); L.w_hh.release(); L.bias.release(); L.w_cat.release(); }
  DevBuf* bufs[] = {&h->emb, &h->ids, &h->len_in, &h->lengths, &h->x0, &h->y[0], &h->y[1], &h->gx, &h->c, &h->pool_sum,
                    &h->pool_max, &h->pool_last, &h->out, &h->raw, &h->err, &h->step_done, &h->trace, &h->proj, &h->tok,
                    &h->diag, &h->hcarry};
  for (DevBuf* b : bufs) b->release();
  for (cudaEvent_t e : h->ev) cudaEventDestroy(e);
  if (h->done_ev) cudaEventDestroy(h->done_ev);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
}

int ie_encoder_load_embedding(ie_encoder* h, const float* emb) {
  if (h == nullptr || emb == nullptr) return fail(IE_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> lk(h->mu);
  CK(cudaSetDevice(h->cfg.device));
  // the per-token table GEMM reads the embedding as its A operand: rows padded to whole M tiles (zeros)
  const int v_rows = static_cast<int>(round_up(h->cfg.vocab_sz, 256));
  std::vector<int> ident(v_rows);
  for (int i = 0; i < v_rows; ++i) ident[i] = i < h->cfg.vocab_sz ? i : -1;
  int rc = upload_sliced(emb, h->cfg.vocab_sz, h->cfg.emb_sz, ident, h->e_pad, h->segs, h->emb, h->own_stream);
  if (rc != IE_OK) return rc;
  h->emb_loaded = true;
  h->proj_built = false;
  return IE_OK;
}

int ie_encoder_load_layer(ie_encoder* h, int32_t layer, const float* w_ih, const float* w_hh, const float* b_ih,
                          const float* b_hh) {
  if (h == nullptr || w_ih == nullptr || w_hh == nullptr || b_ih == nullptr || b_hh == nullptr)
    return fail(IE_ERR_INVALID, "null argument");
  if (layer < 0 || layer >= h->cfg.n_layers) return fail(IE_ERR_INVALID, "layer %d out of range", layer);
  std::lock_guard<std::mutex> lk(h->mu);
  CK(cudaSetDevice(h->cfg.device));
  Layer& L = h->layers[layer];
  const std::vector<int> perm = slice_perm(L);
  int rc = upload_sliced(w_ih, 4 * L.out, L.in, perm, L.kin_pad, h->segs, L.w_ih, h->own_stream);
  if (rc != IE_OK) return rc;
  rc = upload_sliced(w_hh, 4 * L.out, L.out, perm, L.kh_pad, h->segs, L.w_hh, h->own_stream);
  if (rc != IE_OK) return rc;
  std::vector<float> bias(perm.size());
  for (size_t r = 0; r < perm.size(); ++r) bias[r] = perm[r] < 0 ? 0.0f : b_ih[perm[r]] + b_hh[perm[r]];
  CK(L.bias.reserve(bias.size() * sizeof(float)));
  CK(cudaMemcpy(L.bias.p, bias.data(), bias.size() * sizeof(float), cudaMemcpyHostToDevice));
  if (layer == h->cfg.n_layers - 1 && layer > 0 && h->segs == 1) {
    // [W_ih | W_hh] row by row: the B operand of the fused last layer (one tensor map, K = kin_pad + kh_pad)
    const size_t kc = static_cast<size_t>(L.kin_pad) + L.kh_pad, rows = 4 * static_cast<size_t>(L.out_pad);
    CK(L.w_cat.reserve(rows * kc * sizeof(__nv_bfloat16)));
    CK(cudaMemcpy2D(L.w_cat.p, kc * 2, L.w_ih.p, static_cast<size_t>(L.kin_pad) * 2, static_cast<size_t>(L.kin_pad) * 2, rows,
                    cudaMemcpyDeviceToDevice));
    CK(cudaMemcpy2D(L.w_cat.as<__nv_bfloat16>() + L.kin_pad, kc * 2, L.w_hh.p, static_cast<size_t>(L.kh_pad) * 2,
                    static_cast<size_t>(L.kh_pad) * 2, rows, cudaMemcpyDeviceToDevice));
  }
  L.loaded = true;
  if (layer == 0) h->proj_built = false;
  return IE_OK;
}

int ie_encoder_encode(ie_encoder* h, const int64_t* ids, const int32_t* lengths, int32_t B, int32_t T, float* out,
                      int32_t flags, void* stream) {
  if (h == nullptr) return fail(IE_ERR_INVALID, "null handle");
  if (out == nullptr) return fail(IE_ERR_INVALID, "out is null");
  if (ids == nullptr || lengths == nullptr) return fail(IE_ERR_INVALID, "null pointer");
  std::lock_guard<std::mutex> lk(h->mu);
  // device-pointer mode: `stream` is used verbatim (NULL = the legacy default stream, e.g. torch's default);
  // host-pointer mode: NULL selects the handle's own stream
  const bool dev = (flags & IE_FLAG_DEVICE_PTRS) != 0;
  cudaStream_t s = (stream || dev) ? static_cast<cudaStream_t>(stream) : h->own_stream;
  int rc = run_encoder(h, ids, lengths, B, T, out, nullptr, flags, s);
  if (rc != IE_OK || dev) return rc;
  return collect_errors(h);  // host-pointer mode: synchronous, device-side errors are reported by this call
}

int ie_encoder_raw_features(ie_encoder* h, const int64_t* ids, int32_t B, int32_t T, float* raw, int32_t flags,
                            void* stream) {
  if (h == nullptr) return fail(IE_ERR_INVALID, "null handle");
  if (raw == nullptr) return fail(IE_ERR_INVALID, "raw is null");
  std::lock_guard<std::mutex> lk(h->mu);
  const bool dev = (flags & IE_FLAG_DEVICE_PTRS) != 0;
  cudaStream_t s = (stream || dev) ? static_cast<cudaStream_t>(stream) : h->own_stream;
  int rc = run_encoder(h, ids, nullptr, B, T, nullptr, raw, flags, s);
  if (rc != IE_OK || dev) return rc;
  return collect_errors(h);
}

int ie_encoder_check_errors(ie_encoder* h) {
  if (h == nullptr) return fail(IE_ERR_INVALID, "null handle");
  std::lock_guard<std::mutex> lk(h->mu);
  return collect_errors(h);
}

int64_t ie_encoder_launch_count(const ie_encoder* h) { return h ? h->launches : 0; }

int32_t ie_encoder_max_batch(const ie_encoder* h) { return h ? h->max_batch : IE_MAX_BATCH; }

// debug: request a per-item timeline of `layer` in the persistent kernel on the next encode (layer < 0: off);
// with out != NULL copy the last recorded timeline [ctas][items][12] and return ctas*items
int64_t ie_debug_seq_trace(ie_encoder* h, int32_t layer, long long* out, int64_t cap) {
  if (h == nullptr) return fail(IE_ERR_INVALID, "null handle");
  std::lock_guard<std::mutex> lk(h->mu);
  h->trace_layer = layer;
  if (out == nullptr) return 0;
  const int64_t n = static_cast<int64_t>(h->trace_ctas) * h->trace_T;
  if (n == 0 || n * 12 > cap) return fail(IE_ERR_STATE, "no trace recorded or buffer too small");
  cudaSetDevice(h->cfg.device);
  cudaDeviceSynchronize();
  if (cudaMemcpy(out, h->trace.p, n * 12 * sizeof(long long), cudaMemcpyDeviceToHost) != cudaSuccess)
    return fail(IE_ERR_CUDA, "trace copy failed");
  return n;
}

int ie_encoder_last_phase_ms(ie_encoder* h, float* ms, int32_t cap) {
  if (h == nullptr || ms == nullptr) return fail(IE_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> lk(h->mu);
  if (h->ev_used < 2) return fail(IE_ERR_STATE, "no encode call recorded");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaEventSynchronize(h->ev[h->ev_used - 1]));
  const int n = 2 + 2 * h->cfg.n_layers;  // gather, (gemm_l, steps_l) x L, finalize
  std::vector<float> acc(n, 0.0f);
  for (int i = 1; i < h->ev_used; ++i) {
    float t = 0.0f;
    CK(cudaEventElapsedTime(&t, h->ev[i - 1], h->ev[i]));
    const int tag = h->ev_tag[i];
    if (tag >= 1 && tag <= n) acc[tag - 1] += t;  // time chunks of a layer add up
  }
  for (int i = 0; i < n && i < cap; ++i) ms[i] = acc[i];
  return n;
}

int ie_encoder_last_phase_mhz(ie_encoder* h, float* mhz, int32_t cap) {
  if (h == nullptr || mhz == nullptr) return fail(IE_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> lk(h->mu);
  if (!h->has_done) return fail(IE_ERR_STATE, "no encode call recorded");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaEventSynchronize(h->done_ev));
  const int L = h->cfg.n_layers;
  std::vector<long long> d(static_cast<size_t>(L) * 8);
  CK(cudaMemcpy(d.data(), h->diag.p, d.size() * sizeof(long long), cudaMemcpyDeviceToHost));
  // mhz[l] = recurrent kernel of layer l, mhz[L + l] = its input-projection GEMM (0 when the layer had none)
  for (int i = 0; i < 2 * L && i < cap; ++i) {
    const long long* q = d.data() + 8 * (i % L) + 4 * (i / L);
    const long long dc = q[2] - q[0], dn = q[3] - q[1];
    mhz[i] = (dn > 0 && dc > 0) ? static_cast<float>(1e3 * static_cast<double>(dc) / static_cast<double>(dn)) : 0.0f;
  }
  return 2 * h->cfg.n_layers;
}

// ---------------------------------------------------------------------------------------------
// MLP head
// ---------------------------------------------------------------------------------------------
int ie_mlp_create(int32_t n_layers, const int32_t* dims, int32_t device, ie_mlp** out) {
  if (dims == nullptr || out == nullptr || n_layers < 1 || n_layers > 16) return fail(IE_ERR_INVALID, "bad argument");
  for (int i = 0; i <= n_layers; ++i)
    if (dims[i] < 1) return fail(IE_ERR_INVALID, "dims[%d]=%d", i, dims[i]);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(IE_ERR_CUDA, "no CUDA device available (%s): this library has no CPU fallback",
                cudaGetErrorString(e));
  if (device < 0 || device >= ndev) return fail(IE_ERR_INVALID, "device %d not in [0,%d)", device, ndev);
  CK(cudaSetDevice(device));
  int major = 0, sms = 0;
  CK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  if (major != 10) return fail(IE_ERR_CUDA, "device compute capability %d.x is not sm_100 (B200)", major);
  ie_mlp* m = new ie_mlp();
  m->device = device;
  m->num_sms = sms;
  m->dims.assign(dims, dims + n_layers + 1);
  m->layers.resize(n_layers);
  long long ld = 64;
  for (int l = 0; l < n_layers; ++l) {
    ie_mlp::L& L = m->layers[l];
    L.k_pad = static_cast<int>(round_up(dims[l], 64));
    // N tile: a tcgen05.mma costs about the same whatever its N (profiles/README.md), so wide layers use the full N = 256
    // (a 600-wide hidden layer is padded to 768 = 3 tiles: 123 instead of 185 instruction slots per 128-row tile for the
    // (1600, 600, 600, 256) head) and narrow ones a single tile
    const int n16 = static_cast<int>(round_up(dims[l + 1], 16));
    L.bn = n16 >= 256 ? 256 : n16;
    L.n_pad = static_cast<int>(round_up(dims[l + 1], L.bn));
    ld = std::max<long long>(ld, round_up(std::max(L.n_pad, L.k_pad), 64));
  }
  m->act_ld = ld;
  if (const char* v = getenv("IE_MLP_CHUNK")) m->chunk_dev = static_cast<int>(round_up(std::max(256, atoi(v)), 256));
  e = cudaStreamCreateWithFlags(&m->own_stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) { delete m; return cuda_fail(e, "cudaStreamCreate"); }
  *out = m;
  return IE_OK;
}

int ie_mlp_load_layer(ie_mlp* m, int32_t layer, const float* coef, const float* intercept) {
  if (m == nullptr || coef == nullptr || intercept == nullptr) return fail(IE_ERR_INVALID, "null argument");
  if (layer < 0 || layer >= static_cast<int>(m->layers.size())) return fail(IE_ERR_INVALID, "layer out of range");
  std::lock_guard<std::mutex> lk(m->mu);
  CK(cudaSetDevice(m->device));
  ie_mlp::L& L = m->layers[layer];
  const int fan_in = m->dims[layer], fan_out = m->dims[layer + 1];
  // sklearn coefs_[l] is [fan_in, fan_out]; the GEMM wants B = [fan_out rows, fan_in] (K-major)
  std::vector<float> wt(static_cast<size_t>(fan_out) * fan_in);
  for (int i = 0; i < fan_in; ++i)
    for (int o = 0; o < fan_out; ++o) wt[static_cast<size_t>(o) * fan_in + i] = coef[static_cast<size_t>(i) * fan_out + o];
  std::vector<int> perm(L.n_pad);
  for (int r = 0; r < L.n_pad; ++r) perm[r] = r < fan_out ? r : -1;
  int rc = upload_sliced(wt.data(), fan_out, fan_in, perm, L.k_pad, 1, L.w, m->own_stream);
  if (rc != IE_OK) return rc;
  std::vector<float> b(L.n_pad, 0.0f);
  std::copy(intercept, intercept + fan_out, b.begin());
  CK(L.b.reserve(b.size() * sizeof(float)));
  CK(cudaMemcpy(L.b.p, b.data(), b.size() * sizeof(float), cudaMemcpyHostToDevice));
  L.loaded = true;
  return IE_OK;
}

int ie_mlp_predict_proba(ie_mlp* m, const float* X, int32_t n, float* probs, int32_t flags, void* stream) {
  if (m == nullptr || X == nullptr || probs == nullptr) return fail(IE_ERR_INVALID, "null argument");
  if (n < 1) return fail(IE_ERR_INVALID, "n=%d", n);
  for (const auto& L : m->layers)
    if (!L.loaded) return fail(IE_ERR_STATE, "MLP layer weights not loaded");
  std::lock_guard<std::mutex> lk(m->mu);
  CK(cudaSetDevice(m->device));
  const bool dev = (flags & IE_FLAG_DEVICE_PTRS) != 0;
  cudaStream_t s = (stream || dev) ? static_cast<cudaStream_t>(stream) : m->own_stream;
  const int nl = static_cast<int>(m->layers.size());
  const int d_in = m->dims[0], n_labels = m->dims[nl];
  // rows per pass: host buffers are staged through a 2^16-row device buffer; device pointers take chunk_dev rows
  int chunk = dev ? m->chunk_dev : (1 << 16);
  chunk = static_cast<int>(std::min<long long>(chunk, round_up(n, 256)));
  const ie_mlp::L& LL = m->layers[nl - 1];
  // the last GEMM writes straight into the caller's array when its row pitch is a legal store width
  const bool direct_out = dev && n_labels % 16 == 0 && n_labels == LL.n_pad;
  // (Converting chunk k+1 on a side stream under the GEMMs of chunk k was measured: 6.79 vs 6.84 ms per 2^20 rows at
  // D_in = 2400 -- the HBM-bound convert pass and the tensor-bound GEMMs share the board's power budget, not only the SMs;
  // profiles/README.md.)
  CK(m->act[0].reserve(static_cast<size_t>(chunk) * m->act_ld * sizeof(__nv_bfloat16), true));
  CK(m->act[1].reserve(static_cast<size_t>(chunk) * m->act_ld * sizeof(__nv_bfloat16), true));
  CK(m->xb.reserve(static_cast<size_t>(chunk) * m->act_ld * sizeof(__nv_bfloat16), true));
  if (!direct_out) CK(m->probs.reserve(static_cast<size_t>(chunk) * LL.n_pad * sizeof(float)));
  if (!dev) CK(m->xf.reserve(static_cast<size_t>(chunk) * d_in * sizeof(float)));
  for (long long r0 = 0; r0 < n; r0 += chunk) {
    const int rows = static_cast<int>(std::min<long long>(chunk, n - r0));
    // whole M = 256 tiles when there are enough of them for the CTA-pair GEMM (rows past `rows` hold stale finite data
    // and are never stored)
    const int m_pad = static_cast<int>(rows >= 256 * 40 ? round_up(rows, 256) : round_up(rows, 128));
    const float* xsrc = X + r0 * d_in;
    if (!dev) {
      CK(cudaMemcpyAsync(m->xf.p, xsrc, static_cast<size_t>(rows) * d_in * sizeof(float), cudaMemcpyHostToDevice, s));
      xsrc = m->xf.as<float>();
    }
    __nv_bfloat16* xbuf = m->xb.as<__nv_bfloat16>();
    CK(ie::launch_convert_rows(xsrc, d_in, d_in, nullptr, rows, xbuf, m->act_ld, 0, s));   // f32 -> bf16, K padded with zeros
    const __nv_bfloat16* cur_in = xbuf;
    int cur = 0;
    for (int l = 0; l < nl; ++l) {
      const ie_mlp::L& L = m->layers[l];
      const bool last = (l == nl - 1);
      ie::GemmArgs g{};
      g.a = cur_in;
      g.lda = m->act_ld;
      g.b = L.w.as<__nv_bfloat16>();
      g.ldb = L.k_pad;
      g.bias = L.b.as<float>();
      g.m_pad = m_pad;
      g.n_pad = L.n_pad;
      g.k_pad = L.k_pad;
      g.m_store = rows;
      g.n_store = L.n_pad;
      g.bn = L.bn;
      g.num_sms = m->num_sms;
      if (last) {
        g.d = direct_out ? static_cast<void*>(probs + r0 * n_labels) : m->probs.p;
        g.ldd = L.n_pad;
        g.act = 2;
        g.out_bf16 = 0;
      } else {
        g.d = m->act[cur].p;
        g.ldd = m->act_ld;
        g.act = 1;
        g.out_bf16 = 1;
      }
      CK(ie::launch_gemm_bf16(g, s));
      cur_in = m->act[cur].as<__nv_bfloat16>();
      cur ^= 1;
    }
    if (!direct_out)
      CK(cudaMemcpy2DAsync(probs + r0 * n_labels, static_cast<size_t>(n_labels) * sizeof(float), m->probs.p,
                           static_cast<size_t>(LL.n_pad) * sizeof(float), static_cast<size_t>(n_labels) * sizeof(float),
                           rows, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, s));
    if (!dev) CK(cudaStreamSynchronize(s));  // xf is reused by the next chunk
  }
  return IE_OK;
}

int ie_pr_thresholds(const float* scores, const uint8_t* truth, int32_t n, int32_t n_labels, double precision_threshold,
                     double recall_threshold, float* thresholds, double* precisions, double* recalls, int32_t device,
                     int32_t flags, void* stream) {
  if (scores == nullptr || truth == nullptr || thresholds == nullptr || precisions == nullptr || recalls == nullptr)
    return fail(IE_ERR_INVALID, "null argument");
  if (n < 1 || n_labels < 1) return fail(IE_ERR_INVALID, "n=%d n_labels=%d", n, n_labels);
  if (n > ie::kPrMaxSamples)
    return fail(IE_ERR_INVALID, "n=%d exceeds the %d samples one CTA sorts in shared memory", n, ie::kPrMaxSamples);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(IE_ERR_CUDA, "no CUDA device available (%s): this library has no CPU fallback", cudaGetErrorString(e));
  if (device < 0 || device >= ndev) return fail(IE_ERR_INVALID, "device %d not in [0,%d)", device, ndev);
  CK(cudaSetDevice(device));
  const bool dev = (flags & IE_FLAG_DEVICE_PTRS) != 0;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (dev) {
    CK(ie::launch_pr_thresholds(scores, truth, n, n_labels, precision_threshold, recall_threshold, thresholds, precisions,
                                recalls, s));
    return IE_OK;
  }
  DevBuf ds, dt, dth, dp, dr;
  const size_t cells = static_cast<size_t>(n) * n_labels;
  CK(ds.reserve(cells * sizeof(float)));
  CK(dt.reserve(cells));
  CK(dth.reserve(n_labels * sizeof(float)));
  CK(dp.reserve(n_labels * sizeof(double)));
  CK(dr.reserve(n_labels * sizeof(double)));
  CK(cudaMemcpyAsync(ds.p, scores, cells * sizeof(float), cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(dt.p, truth, cells, cudaMemcpyHostToDevice, s));
  CK(ie::launch_pr_thresholds(ds.as<float>(), dt.as<uint8_t>(), n, n_labels, precision_threshold, recall_threshold,
                              dth.as<float>(), dp.as<double>(), dr.as<double>(), s));
  CK(cudaMemcpyAsync(thresholds, dth.p, n_labels * sizeof(float), cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(precisions, dp.p, n_labels * sizeof(double), cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(recalls, dr.p, n_labels * sizeof(double), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return IE_OK;
}

void ie_mlp_destroy(ie_mlp* m) {
  if (m == nullptr) return;
  cudaSetDevice(m->device);
  cudaDeviceSynchronize();
  for (auto& L : m->layers) { L.w.release(); L.b.release(); }
  m->xf.release(); m->act[0].release(); m->act[1].release(); m->probs.release(); m->xb.release();
  if (m->own_stream) cudaStreamDestroy(m->own_stream);
  delete m;
}

int ie_debug_gemm(const float* a, const float* b, const float* bias, int32_t M, int32_t N, int32_t K, int32_t act,
                  float* d, int32_t device) {
  if (a == nullptr || b == nullptr || d == nullptr || M < 1 || N < 1 || K < 1) return fail(IE_ERR_INVALID, "bad argument");
  CK(cudaSetDevice(device));
  int sms = 148;
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  const int m_pad = static_cast<int>(round_up(M, 128)), k_pad = static_cast<int>(round_up(K, 64));
  const int n16 = static_cast<int>(round_up(N, 16));
  int bn = 16;
  if (n16 >= 240 && n16 % 240 == 0) bn = 240;
  else if (n16 >= 128) bn = 128;
  else bn = n16;
  const int n_pad = static_cast<int>(round_up(N, bn));
  DevBuf fa, fb, ba, bb, dd, db;
  cudaStream_t s = nullptr;
  CK(fa.reserve(static_cast<size_t>(M) * K * 4));
  CK(fb.reserve(static_cast<size_t>(N) * K * 4));
  CK(ba.reserve(static_cast<size_t>(m_pad) * k_pad * 2, true));
  CK(bb.reserve(static_cast<size_t>(n_pad) * k_pad * 2, true));
  CK(dd.reserve(static_cast<size_t>(m_pad) * n_pad * 4));
  CK(cudaMemcpy(fa.p, a, static_cast<size_t>(M) * K * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(fb.p, b, static_cast<size_t>(N) * K * 4, cudaMemcpyHostToDevice));
  CK(ie::launch_convert_rows(fa.as<float>(), K, K, nullptr, M, ba.as<__nv_bfloat16>(), k_pad, 0, s));
  CK(ie::launch_convert_rows(fb.as<float>(), K, K, nullptr, N, bb.as<__nv_bfloat16>(), k_pad, 0, s));
  if (bias) {
    std::vector<float> bp(n_pad, 0.0f);
    std::copy(bias, bias + N, bp.begin());
    CK(db.reserve(n_pad * 4));
    CK(cudaMemcpy(db.p, bp.data(), n_pad * 4, cudaMemcpyHostToDevice));
  }
  ie::GemmArgs g{};
  g.a = ba.as<__nv_bfloat16>(); g.lda = k_pad;
  g.b = bb.as<__nv_bfloat16>(); g.ldb = k_pad;
  g.d = dd.p; g.ldd = n_pad;
  g.bias = bias ? db.as<float>() : nullptr;
  g.m_pad = m_pad; g.n_pad = n_pad; g.k_pad = k_pad;
  g.m_store = M; g.n_store = n_pad; g.bn = bn; g.act = act; g.out_bf16 = 0; g.num_sms = sms;
  CK(ie::launch_gemm_bf16(g, s));
  CK(cudaMemcpy2D(d, static_cast<size_t>(N) * 4, dd.p, static_cast<size_t>(n_pad) * 4, static_cast<size_t>(N) * 4, M,
                  cudaMemcpyDeviceToHost));
  fa.release(); fb.release(); ba.release(); bb.release(); dd.release(); db.release();
  return IE_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// Similar-issue search (knn.cu)
// ---------------------------------------------------------------------------------------------
namespace {

constexpr int kKnnMaxDim = 4096;
constexpr long long kKnnBuildChunk = 1 << 16;  // rows per prep pass (host input is staged through an f32 buffer this big)
constexpr int kKnnQueryChunk = 2048;           // queries per search launch (bounds the candidate workspace)

int knn_build(ie_knn* h, const float* vectors, bool dev, cudaStream_t s) {
  const long long n = h->n;
  const int d = h->d;
  const long long chunk = std::min(n, kKnnBuildChunk);
  const long long nblk = ie::knn_colsum_blocks(n);
  CK(h->index.reserve(static_cast<size_t>(h->n_pad) * 2 * h->k_pad * sizeof(__nv_bfloat16), true));
  CK(h->bias.reserve(static_cast<size_t>(h->n_pad) * sizeof(float), true));
  CK(h->omc.reserve(static_cast<size_t>(n) * sizeof(double)));
  CK(h->mean.reserve(static_cast<size_t>(h->k_pad) * sizeof(double)));
  CK(h->err.reserve(sizeof(unsigned), true));
  DevBuf inv, partial, xf;
  CK(inv.reserve(static_cast<size_t>(chunk) * sizeof(double)));
  CK(partial.reserve(static_cast<size_t>(nblk) * d * sizeof(double)));
  if (!dev) CK(xf.reserve(static_cast<size_t>(chunk) * d * sizeof(float)));
  unsigned* flag = h->err.as<unsigned>();
  auto rows_at = [&](long long r0, int rows) -> const float* {
    if (dev) return vectors + r0 * d;
    if (cudaMemcpyAsync(xf.p, vectors + r0 * d, static_cast<size_t>(rows) * d * sizeof(float), cudaMemcpyHostToDevice,
                        s) != cudaSuccess)
      return nullptr;
    return xf.as<float>();
  };
  // pass 1: norms and fixed-order partial column sums of the unit vectors -> mean
  for (long long r0 = 0; r0 < n; r0 += chunk) {
    const int rows = static_cast<int>(std::min(chunk, n - r0));
    const float* x = rows_at(r0, rows);
    if (x == nullptr) return cuda_fail(cudaGetLastError(), "cudaMemcpyAsync");
    CK(ie::launch_knn_check_finite(x, d, d, rows, flag, s));
    CK(ie::launch_knn_inv_norm(x, d, d, rows, inv.as<double>(), s));
    CK(ie::launch_knn_colsum(x, d, d, rows, inv.as<double>(), partial.as<double>(), r0 / 512, s));
  }
  CK(ie::launch_knn_mean(partial.as<double>(), nblk, d, h->k_pad, n, h->mean.as<double>(), s));
  unsigned bad = 0;
  CK(cudaMemcpyAsync(&bad, flag, sizeof(unsigned), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (bad) return fail(IE_ERR_INVALID, "vectors contain NaN or infinite values");
  // pass 2: split-bf16 residuals, b_x and 1 - c_x
  for (long long r0 = 0; r0 < n; r0 += chunk) {
    const int rows = static_cast<int>(std::min(chunk, n - r0));
    const float* x = rows_at(r0, rows);
    if (x == nullptr) return cuda_fail(cudaGetLastError(), "cudaMemcpyAsync");
    CK(ie::launch_knn_prep_rows(x, d, d, rows, h->mean.as<double>(), h->k_pad,
                                h->index.as<__nv_bfloat16>() + r0 * 2 * h->k_pad, h->bias.as<float>() + r0,
                                h->omc.as<double>() + r0, s));
  }
  CK(cudaStreamSynchronize(s));
  return IE_OK;
}

}  // namespace

extern "C" {

int ie_knn_create(const float* vectors, int64_t n, int32_t d, int32_t device, int32_t flags, void* stream, ie_knn** out) {
  if (vectors == nullptr || out == nullptr) return fail(IE_ERR_INVALID, "null argument");
  if (d < 1 || d > kKnnMaxDim) return fail(IE_ERR_INVALID, "d=%d outside [1,%d]", d, kKnnMaxDim);
  if (n < 1 || n > INT32_MAX - 256) return fail(IE_ERR_INVALID, "n=%lld outside [1,%d]", static_cast<long long>(n), INT32_MAX - 256);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(IE_ERR_CUDA, "no CUDA device available (%s): this library has no CPU fallback", cudaGetErrorString(e));
  if (device < 0 || device >= ndev) return fail(IE_ERR_INVALID, "device %d not in [0,%d)", device, ndev);
  CK(cudaSetDevice(device));
  int major = 0, sms = 0;
  CK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  if (major != 10) return fail(IE_ERR_CUDA, "device compute capability %d.x is not sm_100 (B200)", major);
  ie_knn* h = new ie_knn();
  h->device = device;
  h->num_sms = sms;
  h->n = n;
  h->d = d;
  h->k_pad = static_cast<int>(round_up(d, 64));
  h->n_pad = static_cast<int>(round_up(n, 256));
  e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->done_ev, cudaEventDisableTiming);
  if (e != cudaSuccess) { delete h; return cuda_fail(e, "cudaStreamCreate"); }
  const bool dev = (flags & IE_FLAG_DEVICE_PTRS) != 0;
  const int rc = knn_build(h, vectors, dev, dev ? static_cast<cudaStream_t>(stream) : h->own_stream);
  if (rc != IE_OK) { delete h; return rc; }
  *out = h;
  return IE_OK;
}

int ie_knn_search(ie_knn* h, const float* queries, int64_t row0, int32_t m, int32_t k, float* distances, int64_t* ids,
                  int32_t flags, void* stream) {
  if (h == nullptr || distances == nullptr || ids == nullptr) return fail(IE_ERR_INVALID, "null argument");
  if (m < 1) return fail(IE_ERR_INVALID, "m=%d must be >= 1", m);
  const bool self = queries == nullptr;
  const long long cands = self ? h->n - 1 : h->n;
  if (k < 1 || k > ie::kKnnMaxK) return fail(IE_ERR_INVALID, "k=%d outside [1,%d]", k, ie::kKnnMaxK);
  if (k > cands) return fail(IE_ERR_INVALID, "k=%d exceeds the %lld candidates of the index", k, cands);
  if (self && (row0 < 0 || row0 + m > h->n))
    return fail(IE_ERR_INVALID, "rows [%lld,%lld) outside the index of %lld rows", static_cast<long long>(row0),
                static_cast<long long>(row0) + m, h->n);
  const bool dev = (flags & IE_FLAG_DEVICE_PTRS) != 0;
  const int d = h->d;
  if (!self && !dev) {
    const size_t total = static_cast<size_t>(m) * d;
    for (size_t i = 0; i < total; ++i)
      if (!std::isfinite(queries[i])) return fail(IE_ERR_INVALID, "queries contain NaN or infinite values");
  }
  std::lock_guard<std::mutex> lk(h->mu);
  CK(cudaSetDevice(h->device));
  cudaStream_t s = (stream || dev) ? static_cast<cudaStream_t>(stream) : h->own_stream;
  if (h->has_done && s != h->last_stream) CK(cudaStreamWaitEvent(s, h->done_ev, 0));
  const int grid = ie::knn_search_grid(h->n_pad, h->num_sms);
  const int chunk = std::min(m, kKnnQueryChunk);
  const int chunk_pad = static_cast<int>(round_up(chunk, 128));
  CK(h->cand_s.reserve(static_cast<size_t>(chunk) * grid * k * sizeof(float)));
  CK(h->cand_i.reserve(static_cast<size_t>(chunk) * grid * k * sizeof(int)));
  if (!self) {
    CK(h->qa.reserve(static_cast<size_t>(chunk_pad) * 2 * h->k_pad * sizeof(__nv_bfloat16), true));
    CK(h->qomc.reserve(static_cast<size_t>(chunk) * sizeof(double)));
    if (!dev) CK(h->qf.reserve(static_cast<size_t>(chunk) * d * sizeof(float)));
  }
  if (!dev) {
    CK(h->dist.reserve(static_cast<size_t>(chunk) * k * sizeof(float)));
    CK(h->ids.reserve(static_cast<size_t>(chunk) * k * sizeof(int64_t)));
  }
  CK(cudaMemsetAsync(h->err.p, 0, sizeof(unsigned), s));
  for (long long q0 = 0; q0 < m; q0 += chunk) {
    const int rows = static_cast<int>(std::min<long long>(chunk, m - q0));
    ie::KnnSearchArgs a{};
    a.index = h->index.as<__nv_bfloat16>();
    a.bias = h->bias.as<float>();
    a.n_valid = static_cast<int>(h->n);
    a.n_pad = h->n_pad;
    a.k_pad = h->k_pad;
    a.m = rows;
    a.k = k;
    a.cand_s = h->cand_s.as<float>();
    a.cand_i = h->cand_i.as<int>();
    a.num_sms = h->num_sms;
    a.abort_flag = h->err.as<unsigned>();
    if (self) {
      // the stored residuals of rows [row0 + q0, +rows) are the query operand: no prep
      a.a = h->index.as<__nv_bfloat16>();
      a.a_rows = h->n_pad;
      a.a_row0 = static_cast<int>(row0 + q0);
      a.self0 = row0 + q0;
      a.omc = h->omc.as<double>() + row0 + q0;
    } else {
      const float* x = queries + q0 * d;
      if (!dev) {
        CK(cudaMemcpyAsync(h->qf.p, x, static_cast<size_t>(rows) * d * sizeof(float), cudaMemcpyHostToDevice, s));
        x = h->qf.as<float>();
      }
      CK(ie::launch_knn_prep_rows(x, d, d, rows, h->mean.as<double>(), h->k_pad, h->qa.as<__nv_bfloat16>(), nullptr,
                                  h->qomc.as<double>(), s));
      a.a = h->qa.as<__nv_bfloat16>();
      a.a_rows = chunk_pad;
      a.a_row0 = 0;
      a.self0 = -1;
      a.omc = h->qomc.as<double>();
    }
    a.dist = dev ? distances + q0 * k : h->dist.as<float>();
    a.ids = dev ? ids + q0 * k : h->ids.as<int64_t>();
    CK(ie::launch_knn_search(a, s));
    if (!dev) {
      CK(cudaMemcpyAsync(distances + q0 * k, h->dist.p, static_cast<size_t>(rows) * k * sizeof(float),
                         cudaMemcpyDeviceToHost, s));
      CK(cudaMemcpyAsync(ids + q0 * k, h->ids.p, static_cast<size_t>(rows) * k * sizeof(int64_t), cudaMemcpyDeviceToHost,
                         s));
      CK(cudaStreamSynchronize(s));  // qf and the output staging are reused by the next chunk
    }
  }
  CK(cudaEventRecord(h->done_ev, s));
  h->last_stream = s;
  h->has_done = true;
  if (!dev) {
    unsigned aborted = 0;
    CK(cudaMemcpy(&aborted, h->err.p, sizeof(unsigned), cudaMemcpyDeviceToHost));
    if (aborted) return fail(IE_ERR_CUDA, "a device-side wait of the search kernel exceeded its limit and was drained");
  }
  return IE_OK;
}

void ie_knn_destroy(ie_knn* h) {
  if (h == nullptr) return;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  delete h;
}

}  // extern "C"
