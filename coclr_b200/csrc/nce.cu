// MoCo / InfoNCE logits fused with temperature and cross-entropy (model/pretrain.py:175-182 +
// nn.CrossEntropyLoss of main_nce.py:201,314): one launch produces logits = [q.k, q.queue]/T,
// the per-row loss (label 0) and d(mean loss)/d(logits); a second small kernel turns any
// d(logits) into d(q).  Latency-bound (B rows x (1+K) columns x 128), so plain FFMA with
// coalesced reads of the [dim, K] queue (keys are columns, consecutive keys are contiguous).
#include "common.cuh"
#include "coclr_b200.h"

namespace coclr {

static constexpr int kNceThreads = 512;

COCLR_DEVINL float block_reduce(float v, float* sh, bool is_max) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int o = 16; o > 0; o >>= 1) {
    const float t = __shfl_xor_sync(0xffffffffu, v, o);
    v = is_max ? fmaxf(v, t) : v + t;
  }
  __syncthreads();
  if (lane == 0) sh[w] = v;
  __syncthreads();
  if (w == 0) {
    float x = lane < (blockDim.x >> 5) ? sh[lane] : (is_max ? -INFINITY : 0.f);
    for (int o = 16; o > 0; o >>= 1) {
      const float t = __shfl_xor_sync(0xffffffffu, x, o);
      x = is_max ? fmaxf(x, t) : x + t;
    }
    if (lane == 0) sh[0] = x;
  }
  __syncthreads();
  return sh[0];
}

__global__ void __launch_bounds__(kNceThreads) nce_fwd_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                              const float* __restrict__ queue, float T, int B, int D,
                                                              int K, float* __restrict__ logits,
                                                              float* __restrict__ loss_rows,
                                                              float* __restrict__ dlogits) {
  extern __shared__ float sm[];
  float* sq = sm;        // [D]
  float* red = sm + D;   // [32]
  const int b = blockIdx.x;
  for (int c = threadIdx.x; c < D; c += blockDim.x) sq[c] = q[(long)b * D + c];
  __syncthreads();
  float* lrow = logits + (long)b * (K + 1);
  // positive logit
  float pp = 0.f;
  for (int c = threadIdx.x; c < D; c += blockDim.x) pp += sq[c] * k[(long)b * D + c];
  const float lpos = block_reduce(pp, red, false) / T;
  if (threadIdx.x == 0) lrow[0] = lpos;
  float mx = lpos;
  for (int j = threadIdx.x; j < K; j += blockDim.x) {
    float a = 0.f;
#pragma unroll 8
    for (int c = 0; c < D; ++c) a = fmaf(sq[c], __ldg(queue + (long)c * K + j), a);
    a = a / T;
    lrow[1 + j] = a;
    mx = fmaxf(mx, a);
  }
  mx = block_reduce(mx, red, true);
  float se = 0.f;
  for (int j = threadIdx.x; j < K + 1; j += blockDim.x) se += __expf(lrow[j] - mx);  // own writes / thread 0's lpos
  __syncthreads();
  se = block_reduce(se, red, false);
  const float lse = mx + logf(se);
  if (threadIdx.x == 0 && loss_rows) loss_rows[b] = lse - lpos;
  if (dlogits) {
    const float invB = 1.f / (float)B;
    float* drow = dlogits + (long)b * (K + 1);
    for (int j = threadIdx.x; j < K + 1; j += blockDim.x) {
      const float p = __expf(lrow[j] - lse);
      drow[j] = (p - (j == 0 ? 1.f : 0.f)) * invB;
    }
  }
}

// dq[b, c] = ( dlogits[b,0] * k[b,c] + sum_j dlogits[b,1+j] * queue[c, j] ) / T
__global__ void __launch_bounds__(kNceThreads) nce_bwd_kernel(const float* __restrict__ dlogits,
                                                              const float* __restrict__ k,
                                                              const float* __restrict__ queue, float T, int D, int K,
                                                              float* __restrict__ dq) {
  extern __shared__ float sd[];  // [K+1]
  const int b = blockIdx.x;
  for (int j = threadIdx.x; j < K + 1; j += blockDim.x) sd[j] = dlogits[(long)b * (K + 1) + j];
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int c = w; c < D; c += nw) {
    float a = 0.f;
    for (int j = lane; j < K; j += 32) a = fmaf(sd[1 + j], __ldg(queue + (long)c * K + j), a);
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) dq[(long)b * D + c] = (a + sd[0] * k[(long)b * D + c]) / T;
  }
}

// Long queues (config 3: K = 16384): one CTA per row leaves most of the 148 SMs idle and every CTA streams the whole
// [D, K] queue through L2.  The split form cuts a row into K slices of kNceSlice columns on blockIdx.y:
//   pass 1 (nce_fwd_slice_kernel): logits of the slice + the slice's (max, sum exp(l - max)) into ws[b][slice][2];
//   pass 2 (nce_fwd_finish_kernel): every CTA folds the row's partials into the log-sum-exp, then loss / dlogits of its slice.
static constexpr int kNceSlice = 1024;

__global__ void __launch_bounds__(256) nce_fwd_slice_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                            const float* __restrict__ queue, float T, int D, int K,
                                                            float* __restrict__ logits, float* __restrict__ ws) {
  extern __shared__ float sm[];
  float* sq = sm;        // [D]
  float* red = sm + D;   // [32]
  const int b = blockIdx.x, sl = blockIdx.y, nsl = gridDim.y;
  for (int c = threadIdx.x; c < D; c += blockDim.x) sq[c] = q[(long)b * D + c];
  __syncthreads();
  float* lrow = logits + (long)b * (K + 1);
  float mx = -INFINITY;
  if (sl == 0) {   // the positive logit belongs to slice 0
    float pp = 0.f;
    for (int c = threadIdx.x; c < D; c += blockDim.x) pp += sq[c] * k[(long)b * D + c];
    const float lpos = block_reduce(pp, red, false) / T;
    if (threadIdx.x == 0) lrow[0] = lpos;
    mx = lpos;
  }
  const int j0 = sl * kNceSlice, j1 = min(K, j0 + kNceSlice);
  float mine[kNceSlice / 256];
#pragma unroll
  for (int u = 0; u < kNceSlice / 256; ++u) {
    const int j = j0 + u * 256 + threadIdx.x;
    float a = -INFINITY;
    if (j < j1) {
      a = 0.f;
#pragma unroll 8
      for (int c = 0; c < D; ++c) a = fmaf(sq[c], __ldg(queue + (long)c * K + j), a);
      a = a / T;
      lrow[1 + j] = a;
    }
    mine[u] = a;
    mx = fmaxf(mx, a);
  }
  mx = block_reduce(mx, red, true);
  float se = 0.f;
#pragma unroll
  for (int u = 0; u < kNceSlice / 256; ++u) se += __expf(mine[u] - mx);      // exp(-inf) = 0 for the padded tail
  if (sl == 0 && threadIdx.x == 0) se += __expf(lrow[0] - mx);
  __syncthreads();
  se = block_reduce(se, red, false);
  if (threadIdx.x == 0) {
    ws[((long)b * nsl + sl) * 2 + 0] = mx;
    ws[((long)b * nsl + sl) * 2 + 1] = se;
  }
}

__global__ void __launch_bounds__(256) nce_fwd_finish_kernel(const float* __restrict__ logits, const float* __restrict__ ws,
                                                             int B, int K, float* __restrict__ loss_rows,
                                                             float* __restrict__ dlogits) {
  const int b = blockIdx.x, sl = blockIdx.y, nsl = gridDim.y;
  float mx = -INFINITY;
  for (int s = 0; s < nsl; ++s) mx = fmaxf(mx, ws[((long)b * nsl + s) * 2]);
  float se = 0.f;
  for (int s = 0; s < nsl; ++s) se += ws[((long)b * nsl + s) * 2 + 1] * __expf(ws[((long)b * nsl + s) * 2] - mx);
  const float lse = mx + logf(se);
  const float* lrow = logits + (long)b * (K + 1);
  if (sl == 0 && threadIdx.x == 0 && loss_rows) loss_rows[b] = lse - lrow[0];
  if (dlogits) {
    const float invB = 1.f / (float)B;
    float* drow = dlogits + (long)b * (K + 1);
    const int j0 = sl * kNceSlice, j1 = min(K, j0 + kNceSlice);
    if (sl == 0 && threadIdx.x == 0) drow[0] = (__expf(lrow[0] - lse) - 1.f) * invB;
    for (int j = j0 + threadIdx.x; j < j1; j += blockDim.x) drow[1 + j] = __expf(lrow[1 + j] - lse) * invB;
  }
}

// dq for long queues: one warp per (row, channel) sums its whole dot product over the queue, channels spread over
// blockIdx.y, so that the grid fills the SMs like the K slices of the forward.  Every dq element is written once, in a
// fixed summation order: no atomics, and the same dq in every run.
__global__ void __launch_bounds__(256) nce_bwd_cols_kernel(const float* __restrict__ dlogits, const float* __restrict__ k,
                                                           const float* __restrict__ queue, float T, int D, int K,
                                                           float* __restrict__ dq) {
  const int b = blockIdx.x;
  const int lane = threadIdx.x & 31, c = blockIdx.y * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (c >= D) return;
  const float* drow = dlogits + (long)b * (K + 1);
  const float* qrow = queue + (long)c * K;
  float a = 0.f;
  for (int j = lane; j < K; j += 32) a = fmaf(__ldg(drow + 1 + j), __ldg(qrow + j), a);
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  if (lane == 0) dq[(long)b * D + c] = (a + drow[0] * k[(long)b * D + c]) / T;
}

}  // namespace coclr

using namespace coclr;

extern "C" int coclr_nce_logits_ce(const float* q, const float* k, const float* queue, float T, int B, int D, int K,
                                   float* logits, float* loss_rows, float* dlogits, float* ws, coclr_stream_t stream) {
  if (!q || !k || !queue || !logits || B <= 0 || D <= 0 || K <= 0) return COCLR_E_ARG;
  if (ws != nullptr && K > 2 * kNceSlice) {
    const dim3 grid(B, (K + kNceSlice - 1) / kNceSlice);
    nce_fwd_slice_kernel<<<grid, 256, (D + 32) * sizeof(float), (cudaStream_t)stream>>>(q, k, queue, T, D, K, logits, ws);
    nce_fwd_finish_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(logits, ws, B, K, loss_rows, dlogits);
    return cudaGetLastError() == cudaSuccess ? COCLR_OK : COCLR_E_LAUNCH;
  }
  nce_fwd_kernel<<<B, kNceThreads, (D + 32) * sizeof(float), (cudaStream_t)stream>>>(q, k, queue, T, B, D, K, logits,
                                                                                    loss_rows, dlogits);
  return cudaGetLastError() == cudaSuccess ? COCLR_OK : COCLR_E_LAUNCH;
}

extern "C" int coclr_nce_logits_bwd(const float* dlogits, const float* k, const float* queue, float T, int B, int D,
                                    int K, float* dq, coclr_stream_t stream) {
  if (!dlogits || !k || !queue || !dq) return COCLR_E_ARG;
  if (K > 2 * kNceSlice) {
    const dim3 grid(B, (D + 7) / 8);
    nce_bwd_cols_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(dlogits, k, queue, T, D, K, dq);
    return cudaGetLastError() == cudaSuccess ? COCLR_OK : COCLR_E_LAUNCH;
  }
  const size_t smem = (size_t)(K + 1) * sizeof(float);
  if (smem > 200 * 1024) return COCLR_E_ARG;
  if (smem > 48 * 1024) {
    if (cudaFuncSetAttribute(nce_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
      return COCLR_E_LAUNCH;
  }
  nce_bwd_kernel<<<B, kNceThreads, smem, (cudaStream_t)stream>>>(dlogits, k, queue, T, D, K, dq);
  return cudaGetLastError() == cudaSuccess ? COCLR_OK : COCLR_E_LAUNCH;
}

// ------------------------------------------------------------------------------------------------
// CoCLR positive mining (model/pretrain.py:392-413): mask[b, 0] = 1; mask[b, 1+j] = same video source
// (k_vsource[b] == queue_vname[j]) OR j among the top-k of kf[b] . queue_second[:, j] over the columns that are
// NOT same-source (the reference writes -inf there before torch.topk).  One CTA per row: similarities into shared
// memory, then k rounds of a block-wide arg-max (ties: lowest index).  Replaces a cuBLAS GEMM + 5 ATen kernels.
// ------------------------------------------------------------------------------------------------
namespace coclr {

__global__ void __launch_bounds__(256) mask_topk_kernel(const float* __restrict__ kf, const float* __restrict__ queue2,
                                                        const long* __restrict__ vsrc, const long* __restrict__ qvname,
                                                        int D, int K, int topk, unsigned char* __restrict__ mask) {
  extern __shared__ float sm[];
  float* sim = sm;                 // [K]
  float* sq = sm + K;              // [D]
  float* redv = sq + D;            // [8]
  int* redi = reinterpret_cast<int*>(redv + 8);   // [8]
  const int b = blockIdx.x;
  unsigned char* mrow = mask + (size_t)b * (size_t)(K + 1);
  for (int c = threadIdx.x; c < D; c += blockDim.x) sq[c] = kf[(size_t)b * D + c];
  __syncthreads();
  const long mine = vsrc[b];
  if (threadIdx.x == 0) mrow[0] = 1;
  for (int j = threadIdx.x; j < K; j += blockDim.x) {
    const bool same = qvname[j] == mine;
    float a = 0.f;
    if (topk > 0) {
#pragma unroll 8
      for (int c = 0; c < D; ++c) a = fmaf(sq[c], __ldg(queue2 + (size_t)c * K + j), a);
    }
    sim[j] = same ? -INFINITY : a;
    mrow[1 + j] = same ? 1 : 0;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int r = 0; r < topk; ++r) {
    float bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int j = threadIdx.x; j < K; j += blockDim.x) {
      const float v = sim[j];
      if (v > bv) { bv = v; bi = j; }        // ascending j per thread: the first maximum wins
    }
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    if (lane == 0) { redv[w] = bv; redi[w] = bi; }
    __syncthreads();
    if (threadIdx.x == 0) {
      float v = redv[0];
      int i = redi[0];
      for (int k = 1; k < (int)(blockDim.x >> 5); ++k)
        if (redv[k] > v || (redv[k] == v && redi[k] < i)) { v = redv[k]; i = redi[k]; }
      redi[0] = (v == -INFINITY) ? -1 : i;    // nothing but masked columns left: those are positives already
    }
    __syncthreads();
    const int sel = redi[0];
    __syncthreads();
    if (sel < 0) break;
    if (threadIdx.x == 0) {
      mrow[1 + sel] = 1;
      sim[sel] = -INFINITY;
    }
    __syncthreads();
  }
}

}  // namespace coclr

extern "C" int coclr_mask_topk(const float* kf, const float* queue_second, const long* k_vsource, const long* queue_vname,
                               int B, int D, int K, int topk, unsigned char* mask, coclr_stream_t stream) {
  if (!k_vsource || !queue_vname || !mask || B <= 0 || K <= 0 || topk < 0) return COCLR_E_ARG;
  if (topk > 0 && (!kf || !queue_second || D <= 0)) return COCLR_E_ARG;
  const size_t smem = ((size_t)K + (size_t)D + 16) * sizeof(float);
  if (smem > 200 * 1024) return COCLR_E_ARG;
  if (smem > 48 * 1024 &&
      cudaFuncSetAttribute(coclr::mask_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return COCLR_E_LAUNCH;
  coclr::mask_topk_kernel<<<B, 256, smem, (cudaStream_t)stream>>>(kf, queue_second, k_vsource, queue_vname, D, K, topk, mask);
  return cudaGetLastError() == cudaSuccess ? COCLR_OK : COCLR_E_LAUNCH;
}
