// Exact cosine k-nearest-neighbour search over an issue-embedding index (include/issue_emb_b200.h: ie_knn_*).
//
// Raw cosines between encoder outputs are crowded near 1 (neighbours ranked 1..10 are ~1e-7 apart), so a bf16 or
// even an f32 dot product of unit vectors misranks.  The search uses exact algebra instead (DESIGN.md, "Similar-issue
// search"): with mu the mean of the index's unit vectors, r_x = x^ - mu per index row and s_q = q^ - mu per query,
//
//     cos(q, x) = q^.mu + mu.r_x + s_q.r_x  =  c_q + b_x + s_q.r_x
//
// c_q only shifts a query's distances, b_x is one bias per index row, and the GEMM term multiplies vectors of norm
// ~0.007 instead of 1, so its rounding error shrinks with them.  Norms, unit vectors, mu, b and c are f64; r and s are
// rounded to f32 once and split into bf16 hi / lo, and the GEMM runs the split-bf16 K loop of gemm.cu
// ([A_hi | A_lo | A_hi] x [B_hi | B_hi | B_lo], f32 accumulate).
//
// Kernels:
//   knn_inv_norm_kernel / knn_colsum_kernel / knn_mean_kernel   deterministic f64 mean of the unit vectors (fixed-order
//                                                                partial sums, no float atomics)
//   knn_prep_rows_kernel   rows -> split-bf16 residuals, b (index rows) and 1 - c
//   knn_search_kernel      tcgen05 GEMM (queries x index tiles) fused with a running top-k per query row: the
//                          similarity matrix never leaves the SM
//   knn_merge_kernel       top-k of the per-CTA candidates, distances (1 - c_q) - t in f64
#include <cfloat>
#include <climits>

#include "kernels.h"
#include "ptx.cuh"

namespace ie {

namespace {

constexpr int kKnnBlockM = 128;
constexpr int kKnnBlockN = 256;
constexpr int kKnnBlockK = 64;
constexpr int kKnnThreads = 256;
constexpr int kKnnColRows = 512;  // rows per partial column sum of the mean

// 128-thread block sum in f64; the result (valid in every thread) depends only on the inputs, not on timing
__device__ __forceinline__ double block_sum128(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  const double s = (red[0] + red[1]) + (red[2] + red[3]);
  __syncthreads();
  return s;
}

__device__ __forceinline__ double row_sumsq(const float* __restrict__ xr, int d, double* red) {
  double ss = 0.0;
  for (int c = threadIdx.x; c < d; c += 128) {
    const double v = xr[c];
    ss = fma(v, v, ss);
  }
  return block_sum128(ss, red);
}

__device__ __forceinline__ double inv_norm(double ss) { return ss > 0.0 ? 1.0 / sqrt(ss) : 0.0; }

__global__ void __launch_bounds__(128) knn_inv_norm_kernel(const float* __restrict__ x, long long ldx, int d, int rows,
                                                           double* __restrict__ inv) {
  __shared__ double red[4];
  const int r = blockIdx.x;
  if (r >= rows) return;
  const double ss = row_sumsq(x + static_cast<long long>(r) * ldx, d, red);
  if (threadIdx.x == 0) inv[r] = inv_norm(ss);
}

// partial[blk][c] = sum over rows [blk*kKnnColRows, +kKnnColRows) of x[r][c] * inv[r], rows in order
__global__ void __launch_bounds__(128) knn_colsum_kernel(const float* __restrict__ x, long long ldx, int d, int rows,
                                                         const double* __restrict__ inv, double* __restrict__ partial,
                                                         long long blk0) {
  const int c = blockIdx.x * 128 + threadIdx.x;
  if (c >= d) return;
  const int r0 = blockIdx.y * kKnnColRows;
  const int r1 = min(rows, r0 + kKnnColRows);
  double acc = 0.0;
  for (int r = r0; r < r1; ++r) acc = fma(static_cast<double>(x[static_cast<long long>(r) * ldx + c]), inv[r], acc);
  partial[(blk0 + blockIdx.y) * d + c] = acc;
}

__global__ void knn_mean_kernel(const double* __restrict__ partial, long long nblk, int d, int k_pad, long long n,
                                double* __restrict__ mu) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= k_pad) return;
  double s = 0.0;
  if (c < d)
    for (long long b = 0; b < nblk; ++b) s += partial[b * d + c];
  mu[c] = c < d ? s / static_cast<double>(n) : 0.0;
}

// One row per block: x^ = x / |x| (f64), r = f32(x^ - mu) split into bf16 [hi(k_pad) | lo(k_pad)], b = mu.r (f64 -> f32,
// index rows only) and omc = 1 - x^.mu (f64).  Index rows and queries go through this same code, so an index row queried
// from outside gets the same operand bits as its stored residual.
__global__ void __launch_bounds__(128) knn_prep_rows_kernel(const float* __restrict__ x, long long ldx, int d, int rows,
                                                            const double* __restrict__ mu, int k_pad,
                                                            __nv_bfloat16* __restrict__ out, float* __restrict__ bias,
                                                            double* __restrict__ omc) {
  __shared__ double red[4];
  const int r = blockIdx.x;
  if (r >= rows) return;
  const float* xr = x + static_cast<long long>(r) * ldx;
  const double inv = inv_norm(row_sumsq(xr, d, red));
  __nv_bfloat16* o = out + static_cast<long long>(r) * (2 * k_pad);
  double bs = 0.0, cs = 0.0;
  for (int c = threadIdx.x; c < k_pad; c += 128) {
    float rv = 0.0f;
    if (c < d) {
      const double u = static_cast<double>(xr[c]) * inv;
      const double m = mu[c];
      rv = static_cast<float>(u - m);
      cs = fma(u, m, cs);
      bs = fma(m, static_cast<double>(rv), bs);
    }
    const __nv_bfloat16 hi = __float2bfloat16_rn(rv);
    o[c] = hi;
    o[k_pad + c] = __float2bfloat16_rn(rv - __bfloat162float(hi));
  }
  bs = block_sum128(bs, red);
  cs = block_sum128(cs, red);
  if (threadIdx.x == 0) {
    if (bias != nullptr) bias[r] = static_cast<float>(bs);
    omc[r] = 1.0 - cs;
  }
}

__global__ void knn_check_finite_kernel(const float* __restrict__ x, long long ldx, int d, long long rows,
                                        unsigned* flag) {
  const long long total = rows * d;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / d;
    if (!isfinite(x[r * ldx + (i - r * d)])) {
      atomicExch(flag, 1u);
      return;
    }
  }
}

// (score, id) order of the search: higher score first, then smaller id
__device__ __forceinline__ bool better(float a, int ia, float b, int ib) { return a > b || (a == b && ia < ib); }

// insert (t, id) into the descending list s / ids (static indexing: the lists stay in registers)
template <int KMAX>
__device__ __forceinline__ void topk_insert(float (&s)[KMAX], int (&ids)[KMAX], float t, int id) {
#pragma unroll
  for (int j = 0; j < KMAX; ++j) {
    if (better(t, id, s[j], ids[j])) {
      const float ts = s[j];
      const int ti = ids[j];
      s[j] = t;
      ids[j] = id;
      t = ts;
      id = ti;
    }
  }
}

// Fused similarity GEMM + top-k.  CTA c owns index n-blocks [nb0, nb1) and sweeps them once per 128-query m-block:
//   warp 0      TMA producer: query tile 128 x 64 and index tile 256 x 64 per stage, 128B swizzle
//   warp 1      UMMA issuer : tcgen05.mma kind::f16 M=128 N=256 K=16, split-bf16 K loop, TMEM double buffered
//   warp 2      TMEM allocator
//   warps 4..7  epilogue    : thread = query row; t = acc + b_x, running top-KMAX in registers across the CTA's tiles;
//                             at the end of the m-block the first k entries go to cand[query][cta][k]
template <int KMAX>
__global__ void __launch_bounds__(kKnnThreads, 1)
knn_search_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                  const float* __restrict__ bias, int n_valid, int a_row0, long long self0, int m_valid,
                  int num_m_blocks, int num_n_blocks, int num_k_blocks, int k_pad, int stages, int k,
                  float* __restrict__ cand_s, int* __restrict__ cand_i, unsigned* abort_flag, long long spin_limit) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw & 1023u)) & 1023u);

  constexpr uint32_t a_bytes = kKnnBlockM * kKnnBlockK * 2;
  constexpr uint32_t b_bytes = kKnnBlockN * kKnnBlockK * 2;
  constexpr uint32_t stage_bytes = a_bytes + b_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + static_cast<size_t>(stages) * stage_bytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + stages;
  uint64_t* tfull_bar = bars + 2 * stages;
  uint64_t* tempty_bar = bars + 2 * stages + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * stages + 4);
  uint32_t* abort_s = tmem_slot + 1;
  const Abort ab{abort_s, abort_flag, spin_limit};
  const int nkt = num_k_blocks * 3;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  const int nb0 = static_cast<int>(static_cast<long long>(blockIdx.x) * num_n_blocks / gridDim.x);
  const int nb1 = static_cast<int>(static_cast<long long>(blockIdx.x + 1) * num_n_blocks / gridDim.x);
  const int cnt = nb1 - nb0;
  const int num_tiles = num_m_blocks * cnt;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], 128);
    }
    *abort_s = 0;
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = 0; tile < num_tiles && !aborted(ab); ++tile) {
        const int mb = tile / cnt;
        const int nb = nb0 + (tile - mb * cnt);
        for (int kb = 0; kb < nkt; ++kb) {
          const int seg = kb / num_k_blocks, r = kb - seg * num_k_blocks;
          mbar_wait(&empty_bar[stage], phase ^ 1, ab);
          uint8_t* sa = smem + static_cast<size_t>(stage) * stage_bytes;
          mbar_arrive_expect_tx(&full_bar[stage], stage_bytes);
          // the query tile is re-read by every CTA for every n-block: keep it in L2; the index streams through
          tma_load_2d(sa, &tmA, &full_bar[stage], (seg == 1 ? k_pad : 0) + r * kKnnBlockK, a_row0 + mb * kKnnBlockM,
                      kEvictLast);
          tma_load_2d(sa + a_bytes, &tmB, &full_bar[stage], (seg == 2 ? k_pad : 0) + r * kKnnBlockK, nb * kKnnBlockN,
                      kEvictFirst);
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_bf16(kKnnBlockM, kKnnBlockN);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = 0; tile < num_tiles && !aborted(ab); ++tile) {
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1, ab);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + static_cast<uint32_t>(acc * kKnnBlockN);
        for (int kb = 0; kb < nkt; ++kb) {
          mbar_wait(&full_bar[stage], phase, ab);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + static_cast<size_t>(stage) * stage_bytes);
          const uint64_t da = umma_desc_sw128(sa);
          const uint64_t db = umma_desc_sw128(sa + a_bytes);
#pragma unroll
          for (int kk = 0; kk < kKnnBlockK / 16; ++kk) umma_bf16(tmem_d, da + 2 * kk, db + 2 * kk, idesc, (kb | kk) != 0);
          umma_commit(&empty_bar[stage]);
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tfull_bar[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp >= 4) {
    const int q = warp - 4;  // TMEM lane quarter == warp % 4
    int acc = 0;
    uint32_t acc_phase = 0;
    float s[KMAX];
    int ids[KMAX];
    for (int tile = 0; tile < num_tiles; ++tile) {
      const int mb = tile / cnt;
      const int nbi = tile - mb * cnt;
      const int nb = nb0 + nbi;
      const int qrow = mb * kKnnBlockM + q * 32 + lane;
      // self-queries skip their own index row (no index row has a negative id)
      const long long self_ll = self0 >= 0 ? self0 + qrow : -1;
      const int self_id = self_ll >= 0 && self_ll < INT_MAX ? static_cast<int>(self_ll) : -1;
      if (nbi == 0) {
#pragma unroll
        for (int j = 0; j < KMAX; ++j) { s[j] = -INFINITY; ids[j] = INT_MAX; }
      }
      mbar_wait(&tfull_bar[acc], acc_phase, ab);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(acc * kKnnBlockN);
      for (int c = 0; c < kKnnBlockN; c += 16) {
        uint32_t r[16];
        tmem_ld16(taddr + c, r);
        tmem_ld_wait();
        const int n0 = nb * kKnnBlockN + c;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int n = n0 + j;
          const float t = __uint_as_float(r[j]) + __ldg(bias + n);
          // within a CTA ids arrive in increasing order, so an equal score never displaces an earlier entry
          if (t > s[KMAX - 1] && n < n_valid && n != self_id) topk_insert<KMAX>(s, ids, t, n);
        }
      }
      tc_fence_before();
      mbar_arrive(&tempty_bar[acc]);
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      if (nbi == cnt - 1 && qrow < m_valid) {
        const long long base = (static_cast<long long>(qrow) * gridDim.x + blockIdx.x) * k;
#pragma unroll
        for (int j = 0; j < KMAX; ++j)
          if (j < k) { cand_s[base + j] = s[j]; cand_i[base + j] = ids[j]; }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// One warp per query: top-k of the `per_query` candidates (score desc, id asc), distance = (1 - c_q) - t in f64 stored
// as f32, final order ascending distance with ties broken by the smaller id.
constexpr int kMergeKmax = kKnnMaxK;
__global__ void __launch_bounds__(128) knn_merge_kernel(const float* __restrict__ cand_s, const int* __restrict__ cand_i,
                                                        int per_query, int m, int k, const double* __restrict__ omc,
                                                        float* __restrict__ dist, int64_t* __restrict__ out_ids) {
  __shared__ float sd[4][kMergeKmax];
  __shared__ int si[4][kMergeKmax];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qi = blockIdx.x * 4 + w;
  if (qi >= m) return;
  float s[kMergeKmax];
  int ids[kMergeKmax];
#pragma unroll
  for (int j = 0; j < kMergeKmax; ++j) { s[j] = -INFINITY; ids[j] = INT_MAX; }
  const float* cs = cand_s + static_cast<long long>(qi) * per_query;
  const int* ci = cand_i + static_cast<long long>(qi) * per_query;
  for (int i = lane; i < per_query; i += 32) {
    const float t = cs[i];
    const int id = ci[i];
    if (better(t, id, s[kMergeKmax - 1], ids[kMergeKmax - 1])) topk_insert<kMergeKmax>(s, ids, t, id);
  }
  const double base = omc[qi];
  for (int j = 0; j < k; ++j) {
    float bs = s[0];
    int bi = ids[0];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float os = __shfl_xor_sync(0xffffffffu, bs, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (better(os, oi, bs, bi)) { bs = os; bi = oi; }
    }
    if (ids[0] == bi && s[0] == bs) {  // ids are distinct: exactly one lane owns the winner
#pragma unroll
      for (int jj = 0; jj < kMergeKmax - 1; ++jj) { s[jj] = s[jj + 1]; ids[jj] = ids[jj + 1]; }
      s[kMergeKmax - 1] = -INFINITY;
      ids[kMergeKmax - 1] = INT_MAX;
    }
    if (lane == 0) {
      sd[w][j] = static_cast<float>(base - static_cast<double>(bs));
      si[w][j] = bi;
    }
  }
  __syncwarp();
  if (lane == 0) {
    // distinct scores can round to the same f32 distance: keep ties in id order
    for (int j = 1; j < k; ++j) {
      const float dj = sd[w][j];
      const int ij = si[w][j];
      int p = j;
      while (p > 0 && sd[w][p - 1] == dj && si[w][p - 1] > ij) {
        sd[w][p] = sd[w][p - 1];
        si[w][p] = si[w][p - 1];
        --p;
      }
      sd[w][p] = dj;
      si[w][p] = ij;
    }
  }
  __syncwarp();
  for (int j = lane; j < k; j += 32) {
    dist[static_cast<long long>(qi) * k + j] = sd[w][j];
    out_ids[static_cast<long long>(qi) * k + j] = si[w][j];
  }
}

size_t knn_smem_bytes(int stages) {
  return 1024 + static_cast<size_t>(stages) * (kKnnBlockM + kKnnBlockN) * kKnnBlockK * 2 + (2 * stages + 4) * 8 + 32;
}

}  // namespace

long long knn_colsum_blocks(long long rows) { return (rows + kKnnColRows - 1) / kKnnColRows; }

cudaError_t launch_knn_inv_norm(const float* x, long long ldx, int d, int rows, double* inv, cudaStream_t stream) {
  if (rows < 1) return cudaSuccess;
  knn_inv_norm_kernel<<<rows, 128, 0, stream>>>(x, ldx, d, rows, inv);
  return cudaGetLastError();
}

cudaError_t launch_knn_colsum(const float* x, long long ldx, int d, int rows, const double* inv, double* partial,
                              long long blk0, cudaStream_t stream) {
  if (rows < 1) return cudaSuccess;
  const dim3 grid((d + 127) / 128, static_cast<unsigned>(knn_colsum_blocks(rows)));
  knn_colsum_kernel<<<grid, 128, 0, stream>>>(x, ldx, d, rows, inv, partial, blk0);
  return cudaGetLastError();
}

cudaError_t launch_knn_mean(const double* partial, long long nblk, int d, int k_pad, long long n, double* mu,
                            cudaStream_t stream) {
  knn_mean_kernel<<<(k_pad + 127) / 128, 128, 0, stream>>>(partial, nblk, d, k_pad, n, mu);
  return cudaGetLastError();
}

cudaError_t launch_knn_prep_rows(const float* x, long long ldx, int d, int rows, const double* mu, int k_pad,
                                 __nv_bfloat16* out, float* bias, double* omc, cudaStream_t stream) {
  if (k_pad % kKnnBlockK) return cudaErrorInvalidValue;
  if (rows < 1) return cudaSuccess;
  knn_prep_rows_kernel<<<rows, 128, 0, stream>>>(x, ldx, d, rows, mu, k_pad, out, bias, omc);
  return cudaGetLastError();
}

cudaError_t launch_knn_check_finite(const float* x, long long ldx, int d, long long rows, unsigned* flag,
                                    cudaStream_t stream) {
  if (rows < 1) return cudaSuccess;
  const long long total = rows * d;
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 32) blocks = 148 * 32;
  knn_check_finite_kernel<<<static_cast<unsigned>(blocks), 256, 0, stream>>>(x, ldx, d, rows, flag);
  return cudaGetLastError();
}

int knn_search_grid(int n_pad, int num_sms) {
  const int nnb = n_pad / kKnnBlockN;
  const int sms = num_sms > 0 ? num_sms : 148;
  return nnb < sms ? nnb : sms;
}

cudaError_t launch_knn_search(const KnnSearchArgs& a, cudaStream_t stream) {
  if (a.k < 1 || a.k > kKnnMaxK || a.k_pad % kKnnBlockK || a.n_pad % kKnnBlockN || a.m < 1 || a.n_valid > a.n_pad)
    return cudaErrorInvalidValue;
  CUtensorMap tmA, tmB;
  cudaError_t e = make_tmap_bf16_2d(&tmA, a.a, 2ull * a.k_pad, a.a_rows, 2ull * a.k_pad, kKnnBlockK, kKnnBlockM);
  if (e != cudaSuccess) return e;
  e = make_tmap_bf16_2d(&tmB, a.index, 2ull * a.k_pad, a.n_pad, 2ull * a.k_pad, kKnnBlockK, kKnnBlockN);
  if (e != cudaSuccess) return e;
  int stages = 4;
  while (stages > 2 && knn_smem_bytes(stages) > 227 * 1024) --stages;
  const size_t smem = knn_smem_bytes(stages);
  const int grid = knn_search_grid(a.n_pad, a.num_sms);
  const int num_m_blocks = (a.m + kKnnBlockM - 1) / kKnnBlockM;
  const long long spin_limit = a.spin_limit > 0 ? a.spin_limit : kSpinLimitDefault;
  auto kfn = knn_search_kernel<kKnnMaxK>;
  e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
  if (e != cudaSuccess) return e;
  kfn<<<grid, kKnnThreads, smem, stream>>>(tmA, tmB, a.bias, a.n_valid, a.a_row0, a.self0, a.m, num_m_blocks,
                                           a.n_pad / kKnnBlockN, a.k_pad / kKnnBlockK, a.k_pad, stages, a.k, a.cand_s,
                                           a.cand_i, a.abort_flag, spin_limit);
  e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  knn_merge_kernel<<<(a.m + 3) / 4, 128, 0, stream>>>(a.cand_s, a.cand_i, grid * a.k, a.m, a.k, a.omc, a.dist, a.ids);
  return cudaGetLastError();
}

}  // namespace ie
