// HBM-bound kernels around the convolutions: BatchNorm finalize / apply+split / backward, max-pooling,
// global average pooling, input packing, L2-normalise, momentum (EMA) update, queue enqueue, Adam.
// Activations are channels-last rows; channel counts are multiples of 8 for the 16-bit planes and every
// kernel moves 8-16 bytes per thread with consecutive threads on consecutive addresses.
#include <stdlib.h>

#include "common.cuh"
#include "coclr_b200.h"

namespace coclr {

COCLR_DEVINL float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
COCLR_DEVINL void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

COCLR_DEVINL float h2f(uint16_t h) { return __half2float(__ushort_as_half(h)); }

// 4 consecutive channels of an fp16 hi/lo plane pair -> fp32 values (hi + lo)
COCLR_DEVINL float4 ld_pair4(const uint16_t* hi, const uint16_t* lo, size_t off) {
  const uint2 h = *reinterpret_cast<const uint2*>(hi + off);
  float4 v;
  v.x = h2f((uint16_t)(h.x & 0xffff));
  v.y = h2f((uint16_t)(h.x >> 16));
  v.z = h2f((uint16_t)(h.y & 0xffff));
  v.w = h2f((uint16_t)(h.y >> 16));
  if (lo != nullptr) {
    const uint2 l = *reinterpret_cast<const uint2*>(lo + off);
    v.x += h2f((uint16_t)(l.x & 0xffff));
    v.y += h2f((uint16_t)(l.x >> 16));
    v.z += h2f((uint16_t)(l.y & 0xffff));
    v.w += h2f((uint16_t)(l.y >> 16));
  }
  return v;
}

COCLR_DEVINL float b2f(uint16_t h) { return __uint_as_float((uint32_t)h << 16); }

// same for a run-time plane format (bf16 != 0: bf16 planes)
COCLR_DEVINL float4 ld_pair4_any(const uint16_t* hi, const uint16_t* lo, size_t off, int bf16) {
  if (!bf16) return ld_pair4(hi, lo, off);
  const uint2 h = *reinterpret_cast<const uint2*>(hi + off);
  float4 v;
  v.x = b2f((uint16_t)(h.x & 0xffff));
  v.y = b2f((uint16_t)(h.x >> 16));
  v.z = b2f((uint16_t)(h.y & 0xffff));
  v.w = b2f((uint16_t)(h.y >> 16));
  if (lo != nullptr) {
    const uint2 l = *reinterpret_cast<const uint2*>(lo + off);
    v.x += b2f((uint16_t)(l.x & 0xffff));
    v.y += b2f((uint16_t)(l.x >> 16));
    v.z += b2f((uint16_t)(l.y & 0xffff));
    v.w += b2f((uint16_t)(l.y >> 16));
  }
  return v;
}

template <bool kBf16>
COCLR_DEVINL void st_pair4(uint16_t* hi, uint16_t* lo, size_t off, float4 v) {
  uint16_t h0, h1, h2, h3, l0, l1, l2, l3;
  split2<kBf16>(v.x, h0, l0);
  split2<kBf16>(v.y, h1, l1);
  split2<kBf16>(v.z, h2, l2);
  split2<kBf16>(v.w, h3, l3);
  *reinterpret_cast<uint2*>(hi + off) =
      make_uint2((uint32_t)h0 | ((uint32_t)h1 << 16), (uint32_t)h2 | ((uint32_t)h3 << 16));
  if (lo != nullptr)
    *reinterpret_cast<uint2*>(lo + off) =
        make_uint2((uint32_t)l0 | ((uint32_t)l1 << 16), (uint32_t)l2 | ((uint32_t)l3 << 16));
}

// ------------------------------------------------------------------------------------------------
// BatchNorm finalize: per-channel sums -> (scale, shift), saved (mean, rstd), running-stat update.
// nn.BatchNorm3d train-mode semantics (backbone/s3dg.py:16,46-47): biased variance for normalisation,
// unbiased for running_var.
// ------------------------------------------------------------------------------------------------
__global__ void bn_finalize_kernel(const coclr_bn_finalize_t P) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= P.C) return;
  float mean, var;
  if (P.training) {
    const double n = (double)P.count;
    const double m = P.sum[c] / n;
    double v = P.sumsq[c] / n - m * m;
    if (v < 0.0) v = 0.0;
    mean = (float)m;
    var = (float)v;
    const float unbiased = (float)(P.count > 1 ? v * n / (n - 1.0) : v);
    P.running_mean[c] = (1.f - P.momentum) * P.running_mean[c] + P.momentum * mean;
    P.running_var[c] = (1.f - P.momentum) * P.running_var[c] + P.momentum * unbiased;
  } else {
    mean = P.running_mean[c];
    var = P.running_var[c];
  }
  const float rstd = 1.f / sqrtf(var + P.eps);
  const float sc = P.gamma[c] * rstd;
  P.scale[c] = sc;
  P.shift[c] = P.beta[c] - mean * sc;
  if (P.save_mean) P.save_mean[c] = mean;
  if (P.save_rstd) P.save_rstd[c] = rstd;
}

// ------------------------------------------------------------------------------------------------
// BatchNorm-apply + ReLU + hi/lo split: fp32 rows -> 16-bit operand planes (one read, one write)
// ------------------------------------------------------------------------------------------------
template <bool kBf16>
__global__ void __launch_bounds__(256) affine_split_kernel(const coclr_split_t P) {
  const int C4 = P.C >> 2;
  const long total = P.M * C4;
  uint16_t* hi = reinterpret_cast<uint16_t*>(P.hi);
  uint16_t* lo = reinterpret_cast<uint16_t*>(P.lo);
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long r = i / C4;
    const int c = (int)(i - r * C4) * 4;
    float4 v = ld4(P.x + r * P.ld + P.coff + c);
    if (P.scale != nullptr) {
      const float4 sc = ld4(P.scale + c), sh = ld4(P.shift + c);
      v.x = fmaf(v.x, sc.x, sh.x);
      v.y = fmaf(v.y, sc.y, sh.y);
      v.z = fmaf(v.z, sc.z, sh.z);
      v.w = fmaf(v.w, sc.w, sh.w);
    }
    if (P.res_hi != nullptr) {
      const float4 rr = ld_pair4_any(reinterpret_cast<const uint16_t*>(P.res_hi), reinterpret_cast<const uint16_t*>(P.res_lo),
                                     (size_t)(r * P.res_ld + P.res_coff + c), kBf16);
      v.x += rr.x; v.y += rr.y; v.z += rr.z; v.w += rr.w;
    }
    if (P.relu) {
      v.x = fmaxf(v.x, 0.f);
      v.y = fmaxf(v.y, 0.f);
      v.z = fmaxf(v.z, 0.f);
      v.w = fmaxf(v.w, 0.f);
    }
    st_pair4<kBf16>(hi, lo, (size_t)(r * P.out_ld + P.out_coff + c), v);
    if (P.hi2 != nullptr)
      st_pair4<true>(reinterpret_cast<uint16_t*>(P.hi2), reinterpret_cast<uint16_t*>(P.lo2),
                     (size_t)(r * P.out_ld + P.out_coff + c), v);
  }
}

// ------------------------------------------------------------------------------------------------
// column-reduce helper: thread t < A owns channel group (t % C4) and rows (t / C4) + k*(A / C4)
// ------------------------------------------------------------------------------------------------
static constexpr int kColThreads = 256;
static constexpr int kMaxBnC = 2048;   // widest BatchNorm on the path: ResNet2d3d-50 layer4 (resnet_2d3d.py:146)

// BatchNorm finalize fused with apply + ReLU + split: every block derives (scale, shift) of all channels into
// shared memory from the statistics (cheap: C <= 1024), block 0 also publishes them (backward needs
// scale/shift/mean/rstd) and updates the running statistics; then the same flat, fully coalesced pass as
// affine_split_kernel.
template <bool kBf16>
__global__ void __launch_bounds__(256) bn_apply_split_kernel(const coclr_split_t P) {
  __shared__ float s_sc[kMaxBnC], s_sh[kMaxBnC];
  const coclr_bn_finalize_t& F = P.bn;
  for (int c = threadIdx.x; c < P.C; c += blockDim.x) {
    float mean, var;
    if (F.training) {
      const double n = (double)F.count;
      const double m = F.sum[c] / n;
      double v = F.sumsq[c] / n - m * m;
      if (v < 0.0) v = 0.0;
      mean = (float)m;
      var = (float)v;
      if (blockIdx.x == 0) {
        const float unbiased = (float)(F.count > 1 ? v * n / (n - 1.0) : v);
        F.running_mean[c] = (1.f - F.momentum) * F.running_mean[c] + F.momentum * mean;
        F.running_var[c] = (1.f - F.momentum) * F.running_var[c] + F.momentum * unbiased;
      }
    } else {
      mean = F.running_mean[c];
      var = F.running_var[c];
    }
    const float rstd = 1.f / sqrtf(var + F.eps);
    const float sc = F.gamma[c] * rstd;
    const float sh = F.beta[c] - mean * sc;
    s_sc[c] = sc;
    s_sh[c] = sh;
    if (blockIdx.x == 0) {
      F.scale[c] = sc;
      F.shift[c] = sh;
      if (F.save_mean) F.save_mean[c] = mean;
      if (F.save_rstd) F.save_rstd[c] = rstd;
    }
  }
  __syncthreads();
  const int C4 = P.C >> 2;
  const long total = P.M * C4;
  uint16_t* hi = reinterpret_cast<uint16_t*>(P.hi);
  uint16_t* lo = reinterpret_cast<uint16_t*>(P.lo);
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long r = i / C4;
    const int c = (int)(i - r * C4) * 4;
    float4 v = ld4(P.x + r * P.ld + P.coff + c);
    v.x = fmaf(v.x, s_sc[c + 0], s_sh[c + 0]);
    v.y = fmaf(v.y, s_sc[c + 1], s_sh[c + 1]);
    v.z = fmaf(v.z, s_sc[c + 2], s_sh[c + 2]);
    v.w = fmaf(v.w, s_sc[c + 3], s_sh[c + 3]);
    if (P.res_hi != nullptr) {
      const float4 rr = ld_pair4_any(reinterpret_cast<const uint16_t*>(P.res_hi), reinterpret_cast<const uint16_t*>(P.res_lo),
                                     (size_t)(r * P.res_ld + P.res_coff + c), kBf16);
      v.x += rr.x; v.y += rr.y; v.z += rr.z; v.w += rr.w;
    }
    if (P.relu) {
      v.x = fmaxf(v.x, 0.f);
      v.y = fmaxf(v.y, 0.f);
      v.z = fmaxf(v.z, 0.f);
      v.w = fmaxf(v.w, 0.f);
    }
    const size_t o = (size_t)(r * P.out_ld + P.out_coff + c);
    st_pair4<kBf16>(hi, lo, o, v);
    if (P.hi2 != nullptr)
      st_pair4<true>(reinterpret_cast<uint16_t*>(P.hi2), reinterpret_cast<uint16_t*>(P.lo2), o, v);
  }
}

// BN backward.  Channel tiles of <= kBwdTileC channels on blockIdx.y (ResNet2d3d-50 has up to 2048 channels), row
// slabs on blockIdx.x.  With a residual (P.res_hi) the unit is relu(bn(y) + r): r enters the ReLU mask and dz is also
// the residual branch's gradient.
static constexpr int kBwdTileC = 1024;

struct BwdCols {
  int C4, A, R, cb;   // float4 column groups of this tile, active threads, rows per pass, first channel of the tile
};
COCLR_DEVINL BwdCols bwd_cols(const coclr_bn_bwd_t& P) {
  BwdCols k;
  k.cb = blockIdx.y * kBwdTileC;
  const int Cl = min(P.C - k.cb, kBwdTileC);
  k.C4 = Cl >> 2;
  k.A = (kColThreads / k.C4) * k.C4;
  k.R = k.A / k.C4;
  return k;
}

COCLR_DEVINL float4 bwd_dz(const coclr_bn_bwd_t& P, size_t row, int cc, const float4& y, const float4& da, const float4& sc,
                           const float4& sh) {
  if (!P.relu) return da;
  float4 z;
  z.x = fmaf(y.x, sc.x, sh.x);
  z.y = fmaf(y.y, sc.y, sh.y);
  z.z = fmaf(y.z, sc.z, sh.z);
  z.w = fmaf(y.w, sc.w, sh.w);
  if (P.res_hi != nullptr) {
    const float4 rr = ld_pair4_any(reinterpret_cast<const uint16_t*>(P.res_hi), reinterpret_cast<const uint16_t*>(P.res_lo),
                                   row * (size_t)P.res_ld + P.res_coff + cc, P.res_bf16);
    z.x += rr.x; z.y += rr.y; z.z += rr.z; z.w += rr.w;
  }
  float4 dz;
  dz.x = z.x > 0.f ? da.x : 0.f;
  dz.y = z.y > 0.f ? da.y : 0.f;
  dz.z = z.z > 0.f ? da.z : 0.f;
  dz.w = z.w > 0.f ? da.w : 0.f;
  return dz;
}

// phase 1: s1[c] = sum dz, s2[c] = sum dz * xhat, dz = dA * [scale*y+shift (+ r) > 0]
__global__ void __launch_bounds__(kColThreads) bn_bwd_reduce_kernel(const coclr_bn_bwd_t P) {
  const BwdCols K = bwd_cols(P);
  const int C4 = K.C4, A = K.A, R = K.R;
  __shared__ float red[8][kColThreads];
  const int t = threadIdx.x;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float mx[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // max |dz| and max |xhat| per channel (range of dY, see apply)
  if (t < A) {
    const int cg = t % C4, rs = t / C4;
    const int c = K.cb + cg * 4;
    const float4 sc = ld4(P.scale + c), sh = ld4(P.shift + c), mu = ld4(P.mean + c), rs4 = ld4(P.rstd + c);
    const long rows_per = ((long)P.M + gridDim.x - 1) / gridDim.x;
    const long r_begin = (long)blockIdx.x * rows_per;
    const long r_end = min((long)P.M, r_begin + rows_per);
    auto body = [&](long row, const float4& y, const float4& da) {
      const float4 dz = bwd_dz(P, (size_t)row, c, y, da, sc, sh);
      const float x0 = (y.x - mu.x) * rs4.x, x1 = (y.y - mu.y) * rs4.y, x2 = (y.z - mu.z) * rs4.z, x3 = (y.w - mu.w) * rs4.w;
      acc[0] += dz.x; acc[1] += dz.y; acc[2] += dz.z; acc[3] += dz.w;
      acc[4] += dz.x * x0;
      acc[5] += dz.y * x1;
      acc[6] += dz.z * x2;
      acc[7] += dz.w * x3;
      mx[0] = fmaxf(mx[0], fabsf(dz.x)); mx[1] = fmaxf(mx[1], fabsf(dz.y));
      mx[2] = fmaxf(mx[2], fabsf(dz.z)); mx[3] = fmaxf(mx[3], fabsf(dz.w));
      mx[4] = fmaxf(mx[4], fabsf(x0)); mx[5] = fmaxf(mx[5], fabsf(x1));
      mx[6] = fmaxf(mx[6], fabsf(x2)); mx[7] = fmaxf(mx[7], fabsf(x3));
    };
    long r = r_begin + rs;
    for (; r + 3 * R < r_end; r += 4 * R) {   // 8 independent 16-byte loads in flight per thread
      float4 y[4], da[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        y[u] = ld4(P.y + (r + u * R) * P.ld + P.coff + c);
        da[u] = ld4(P.dA + (r + u * R) * P.ld + P.coff + c);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) body(r + u * R, y[u], da[u]);
    }
    for (; r < r_end; r += R) body(r, ld4(P.y + r * P.ld + P.coff + c), ld4(P.dA + r * P.ld + P.coff + c));
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) red[j][t] = acc[j];
  __syncthreads();
  if (t < C4) {
    double s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int k = 0; k < R; ++k)
#pragma unroll
      for (int j = 0; j < 8; ++j) s[j] += (double)red[j][t + k * C4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      atomicAdd(P.sums + K.cb + t * 4 + j, s[j]);
      atomicAdd(P.sums + P.C + K.cb + t * 4 + j, s[4 + j]);
    }
  }
  if (P.amax != nullptr) {   // block-wide maxima of the two range inputs (non-negative floats order like their bit patterns)
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 8; ++j) red[j][t] = mx[j];
    __syncthreads();
    if (t < C4) {
      float m[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      for (int k = 0; k < R; ++k)
#pragma unroll
        for (int j = 0; j < 8; ++j) m[j] = fmaxf(m[j], red[j][t + k * C4]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        atomicMax(reinterpret_cast<int*>(P.amax) + K.cb + t * 4 + j, __float_as_int(m[j]));
        atomicMax(reinterpret_cast<int*>(P.amax) + P.C + K.cb + t * 4 + j, __float_as_int(m[4 + j]));
      }
    }
  }
}

// phase 2: dY = scale * (dz - s1/n - xhat * s2/n) -> bf16 hi/lo planes; dres (+)= dz; the first row slab also
// accumulates dgamma += s2, dbeta += s1.
__global__ void __launch_bounds__(kColThreads) bn_bwd_apply_kernel(const coclr_bn_bwd_t P) {
  const BwdCols K = bwd_cols(P);
  const int C4 = K.C4, A = K.A, R = K.R;
  const int t = threadIdx.x;
  const double inv_n = 1.0 / (double)P.M;
  // fp16 planes: one power-of-two scale for the whole tensor from |dY_c| <= |scale_c| (max|dz_c| + |m1_c| + max|xhat_c| |m2_c|);
  // every block derives the same value (the inputs are final after the reduce kernel)
  float dscale = 1.f;
  if (P.dy_fp16) {
    __shared__ float smax[kColThreads / 32];
    float bound = 0.f;
    for (int ch = t; ch < P.C; ch += kColThreads) {
      const float b = fabsf(P.scale[ch]) * (P.amax[ch] + fabsf((float)(P.sums[ch] * inv_n)) +
                                           P.amax[P.C + ch] * fabsf((float)(P.sums[P.C + ch] * inv_n)));
      bound = fmaxf(bound, b);
    }
    for (int o = 16; o > 0; o >>= 1) bound = fmaxf(bound, __shfl_xor_sync(0xffffffffu, bound, o));
    if ((t & 31) == 0) smax[t >> 5] = bound;
    __syncthreads();
    bound = 0.f;
    for (int k = 0; k < kColThreads / 32; ++k) bound = fmaxf(bound, smax[k]);
    if (bound > 0.f && isfinite(bound)) {
      int e;
      frexpf(bound, &e);                       // bound = f * 2^e, f in [0.5, 1)  ->  bound * 2^(14 - e) < 2^14
      dscale = ldexpf(1.f, max(-100, min(100, 14 - e)));
    }
    if (blockIdx.x == 0 && blockIdx.y == 0 && t == 0 && P.dy_scale != nullptr) {
      P.dy_scale[0] = dscale;
      P.dy_scale[1] = 1.f / dscale;
    }
  }
  if (t >= A) return;
  const int cg = t % C4, rs = t / C4;
  const int c = K.cb + cg * 4;
  const float4 sc = ld4(P.scale + c), sh = ld4(P.shift + c), mu = ld4(P.mean + c), rs4 = ld4(P.rstd + c);
  float m1[4], m2[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const double s1 = P.sums[c + j], s2 = P.sums[P.C + c + j];
    m1[j] = (float)(s1 * inv_n);
    m2[j] = (float)(s2 * inv_n);
    if (blockIdx.x == 0 && rs == 0) {
      if (P.dgamma) P.dgamma[c + j] += (float)s2;  // gradient buffers accumulate (zeroed once per step)
      if (P.dbeta) P.dbeta[c + j] += (float)s1;
    }
  }
  uint16_t* hi = reinterpret_cast<uint16_t*>(P.dy_hi);
  uint16_t* lo = reinterpret_cast<uint16_t*>(P.dy_lo);
  const long rows_per = ((long)P.M + gridDim.x - 1) / gridDim.x;
  const long r_begin = (long)blockIdx.x * rows_per;
  const long r_end = min((long)P.M, r_begin + rows_per);
  auto body = [&](long row, size_t off, const float4& y, const float4& da) {
    const float4 dz = bwd_dz(P, (size_t)row, c, y, da, sc, sh);
    float4 o;
    o.x = sc.x * (dz.x - m1[0] - ((y.x - mu.x) * rs4.x) * m2[0]);
    o.y = sc.y * (dz.y - m1[1] - ((y.y - mu.y) * rs4.y) * m2[1]);
    o.z = sc.z * (dz.z - m1[2] - ((y.z - mu.z) * rs4.z) * m2[2]);
    o.w = sc.w * (dz.w - m1[3] - ((y.w - mu.w) * rs4.w) * m2[3]);
    if (P.dy_fp16) {
      o.x *= dscale; o.y *= dscale; o.z *= dscale; o.w *= dscale;
      st_pair4<false>(hi, lo, off, o);
    } else {
      st_pair4<true>(hi, lo, off, o);
    }
    if (P.dres != nullptr) {
      float* d = P.dres + (size_t)row * P.dres_ld + P.dres_coff + c;
      float4 v = dz;
      if (P.dres_accumulate) {
        const float4 old = ld4(d);
        v.x += old.x; v.y += old.y; v.z += old.z; v.w += old.w;
      }
      st4(d, v);
    }
  };
  long r = r_begin + rs;
  for (; r + 3 * R < r_end; r += 4 * R) {
    float4 y[4], da[4];
    size_t off[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      off[u] = (size_t)((r + u * R) * P.ld + P.coff + c);
      y[u] = ld4(P.y + off[u]);
      da[u] = ld4(P.dA + off[u]);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) body(r + u * R, off[u], y[u], da[u]);
  }
  for (; r < r_end; r += R) {
    const size_t off = (size_t)(r * P.ld + P.coff + c);
    body(r, off, ld4(P.y + off), ld4(P.dA + off));
  }
}

// bias + ReLU backward for the projection head (model/pretrain.py:52-53): in place dz = dA*[h+b>0],
// dbias += sum_rows dz.  Rows are few (the batch).
__global__ void bias_relu_bwd_kernel(const float* h, const float* bias, float* dA, float* dbias, int M, int C) {
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < C; c += gridDim.x * blockDim.x) {
    float s = 0.f;
    const float b = bias[c];
    for (int r = 0; r < M; ++r) {
      const float dz = (h[(size_t)r * C + c] + b > 0.f) ? dA[(size_t)r * C + c] : 0.f;
      dA[(size_t)r * C + c] = dz;
      s += dz;
    }
    dbias[c] += s;
  }
}

// ------------------------------------------------------------------------------------------------
// MaxPool3d (nn.MaxPool3d; backbone/s3dg.py:105,151,162,173,190): -inf padding, first maximum wins.
// Input and output are fp16 hi/lo planes (the arg-max element's pair is copied, so no re-rounding).
// Compile-time window/stride for the four shapes S3D uses (0 = take the run-time value).
// ------------------------------------------------------------------------------------------------
// Comparisons stay in packed fp16: a value is the pair (hi, lo) with hi = round(value), so pairs order
// lexicographically; __h*2_mask gives a 0xffff / 0 mask per 16-bit half, i.e. two channels per instruction and
// no unpacking or conversion.
COCLR_DEVINL __half2 u2h2(uint32_t u) { return *reinterpret_cast<__half2*>(&u); }
COCLR_DEVINL uint32_t pair_gt_mask(uint32_t ah, uint32_t al, uint32_t bh, uint32_t bl) {
  return __hgt2_mask(u2h2(ah), u2h2(bh)) | (__heq2_mask(u2h2(ah), u2h2(bh)) & __hgt2_mask(u2h2(al), u2h2(bl)));
}
COCLR_DEVINL uint32_t pair_eq_mask(uint32_t ah, uint32_t al, uint32_t bh, uint32_t bl) {
  return __heq2_mask(u2h2(ah), u2h2(bh)) & __heq2_mask(u2h2(al), u2h2(bl));
}
COCLR_DEVINL uint32_t msel(uint32_t a, uint32_t b, uint32_t m) { return (a & m) | (b & ~m); }
// small non-negative integer n as an fp16 bit pattern replicated in both halves (exact for n <= 2048)
COCLR_DEVINL uint32_t int_h2(int n) {
  const uint32_t h = __half_as_ushort(__int2half_rn(n));
  return h | (h << 16);
}
COCLR_DEVINL int h_lo_int(uint32_t u) { return __half2int_rn(__ushort_as_half((uint16_t)(u & 0xffffu))); }
COCLR_DEVINL int h_hi_int(uint32_t u) { return __half2int_rn(__ushort_as_half((uint16_t)(u >> 16))); }

static constexpr uint32_t kNegInf2 = 0xfc00fc00u;  // (-inf, -inf) in fp16

template <int KT, int KH, int KW, int ST, int SH, int SW>
__global__ void __launch_bounds__(256) maxpool_fwd_kernel(const coclr_pool_t P) {
  const int kt = KT ? KT : P.g.kt, kh = KH ? KH : P.g.kh, kw = KW ? KW : P.g.kw;
  const int st = ST ? ST : P.g.st, sh = SH ? SH : P.g.sh, sw = SW ? SW : P.g.sw;
  const int C4 = P.C >> 2;
  const long total = (long)P.B * P.To * P.Ho * P.Wo * C4;
  const uint16_t* xh = reinterpret_cast<const uint16_t*>(P.x_hi);
  const uint16_t* xl = reinterpret_cast<const uint16_t*>(P.x_lo);
  uint16_t* yh = reinterpret_cast<uint16_t*>(P.y_hi);
  uint16_t* yl = reinterpret_cast<uint16_t*>(P.y_lo);
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int cg = (int)(i % C4);
    long r = i / C4;
    const int xo = (int)(r % P.Wo); r /= P.Wo;
    const int yo = (int)(r % P.Ho); r /= P.Ho;
    const int to = (int)(r % P.To);
    const int b = (int)(r / P.To);
    const int c = cg * 4;
    uint32_t bh[2] = {kNegInf2, kNegInf2}, bl[2] = {0u, 0u}, bt[2] = {0u, 0u};  // best hi / lo / tap (2 ch per word)
#pragma unroll
    for (int a = 0; a < kt; ++a) {
      const int ti = to * st - P.g.pt + a;
      if ((unsigned)ti >= (unsigned)P.Ti) continue;
#pragma unroll
      for (int bb = 0; bb < kh; ++bb) {
        const int yi = yo * sh - P.g.ph + bb;
        if ((unsigned)yi >= (unsigned)P.Hi) continue;
#pragma unroll
        for (int cc = 0; cc < kw; ++cc) {
          const int xi = xo * sw - P.g.pw + cc;
          if ((unsigned)xi >= (unsigned)P.Wi) continue;
          const uint32_t tap2 = int_h2((a * kh + bb) * kw + cc);
          const size_t off = ((((size_t)b * P.Ti + ti) * P.Hi + yi) * P.Wi + xi) * P.ldx + P.x_coff + c;
          const uint2 h = *reinterpret_cast<const uint2*>(xh + off);
          uint2 l = make_uint2(0u, 0u);
          if (xl != nullptr) l = *reinterpret_cast<const uint2*>(xl + off);
          const uint32_t hw[2] = {h.x, h.y}, lw[2] = {l.x, l.y};
#pragma unroll
          for (int p = 0; p < 2; ++p) {
            const uint32_t m = pair_gt_mask(hw[p], lw[p], bh[p], bl[p]);   // strictly greater: first max wins
            bh[p] = msel(hw[p], bh[p], m);
            bl[p] = msel(lw[p], bl[p], m);
            bt[p] = msel(tap2, bt[p], m);
          }
        }
      }
    }
    const size_t o = ((((size_t)b * P.To + to) * P.Ho + yo) * P.Wo + xo);
    const size_t oo = o * P.ldy + P.y_coff + c;
    *reinterpret_cast<uint2*>(yh + oo) = make_uint2(bh[0], bh[1]);
    if (yl != nullptr) *reinterpret_cast<uint2*>(yl + oo) = make_uint2(bl[0], bl[1]);
    if (P.y2_hi != nullptr)
      st_pair4<true>(reinterpret_cast<uint16_t*>(P.y2_hi), reinterpret_cast<uint16_t*>(P.y2_lo), oo,
                     make_float4(h2f((uint16_t)(bh[0] & 0xffff)) + h2f((uint16_t)(bl[0] & 0xffff)),
                                 h2f((uint16_t)(bh[0] >> 16)) + h2f((uint16_t)(bl[0] >> 16)),
                                 h2f((uint16_t)(bh[1] & 0xffff)) + h2f((uint16_t)(bl[1] & 0xffff)),
                                 h2f((uint16_t)(bh[1] >> 16)) + h2f((uint16_t)(bl[1] >> 16))));
    if (P.idx)
      *reinterpret_cast<uchar4*>(P.idx + o * P.C + c) =
          make_uchar4((unsigned char)h_lo_int(bt[0]), (unsigned char)h_hi_int(bt[0]), (unsigned char)h_lo_int(bt[1]),
                      (unsigned char)h_hi_int(bt[1]));
  }
}

// 3x3x3 / stride 1 / pad 1 (the Inception branch-3 pool, 18 of the 26 pool launches of a step): each thread
// produces 4 consecutive outputs along x for 4 channels and shares the loaded columns between them: first the
// maximum over the 9 (t,y) taps of each of the 6 input columns, then 3 columns per output.  Ties resolve to the
// first tap in (t,y,x) scan order like nn.MaxPool3d.
__global__ void __launch_bounds__(256) maxpool333_fwd_kernel(const coclr_pool_t P) {
  const int C4 = P.C >> 2;
  const int XG = P.Wo >> 2;  // Wo % 4 == 0 checked by the launcher
  const long total = (long)P.B * P.To * P.Ho * XG * C4;
  const uint16_t* xh = reinterpret_cast<const uint16_t*>(P.x_hi);
  const uint16_t* xl = reinterpret_cast<const uint16_t*>(P.x_lo);
  uint16_t* yh = reinterpret_cast<uint16_t*>(P.y_hi);
  uint16_t* yl = reinterpret_cast<uint16_t*>(P.y_lo);
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int cg = (int)(i % C4);
    long r = i / C4;
    const int xg = (int)(r % XG); r /= XG;
    const int yo = (int)(r % P.Ho); r /= P.Ho;
    const int to = (int)(r % P.To);
    const int b = (int)(r / P.To);
    const int c = cg * 4;
    const int x0 = xg * 4 - 1;  // first input column
    uint32_t ch[6][2], cl[6][2], cab[6][2];  // per column: best hi / lo / (t,y) tap, 2 channels per word
#pragma unroll
    for (int j = 0; j < 6; ++j)
#pragma unroll
      for (int p = 0; p < 2; ++p) { ch[j][p] = kNegInf2; cl[j][p] = 0u; cab[j][p] = 0u; }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const int ti = to - 1 + a;
      if ((unsigned)ti >= (unsigned)P.Ti) continue;
#pragma unroll
      for (int bb = 0; bb < 3; ++bb) {
        const int yi = yo - 1 + bb;
        if ((unsigned)yi >= (unsigned)P.Hi) continue;
        const uint32_t ab2 = int_h2(a * 3 + bb);
        const size_t rowoff = (((size_t)b * P.Ti + ti) * P.Hi + yi) * P.Wi;
#pragma unroll
        for (int j = 0; j < 6; ++j) {
          const int xi = x0 + j;
          if ((unsigned)xi >= (unsigned)P.Wi) continue;
          const size_t off = (rowoff + xi) * P.ldx + P.x_coff + c;
          const uint2 h = *reinterpret_cast<const uint2*>(xh + off);
          uint2 l = make_uint2(0u, 0u);
          if (xl != nullptr) l = *reinterpret_cast<const uint2*>(xl + off);
          const uint32_t hw[2] = {h.x, h.y}, lw[2] = {l.x, l.y};
#pragma unroll
          for (int p = 0; p < 2; ++p) {
            const uint32_t m = pair_gt_mask(hw[p], lw[p], ch[j][p], cl[j][p]);
            ch[j][p] = msel(hw[p], ch[j][p], m);
            cl[j][p] = msel(lw[p], cl[j][p], m);
            cab[j][p] = msel(ab2, cab[j][p], m);
          }
        }
      }
    }
#pragma unroll
    for (int o4 = 0; o4 < 4; ++o4) {
      uint32_t bh[2], bl[2], bab[2], bcc[2];
#pragma unroll
      for (int p = 0; p < 2; ++p) { bh[p] = ch[o4][p]; bl[p] = cl[o4][p]; bab[p] = cab[o4][p]; bcc[p] = 0u; }
#pragma unroll
      for (int cc = 1; cc < 3; ++cc) {
        const uint32_t cc2 = int_h2(cc);
#pragma unroll
        for (int p = 0; p < 2; ++p) {
          const uint32_t vh = ch[o4 + cc][p], vl = cl[o4 + cc][p], ab = cab[o4 + cc][p];
          // greater, or equal with an earlier (t,y) tap (same (t,y): the smaller x stays)
          const uint32_t m = pair_gt_mask(vh, vl, bh[p], bl[p]) |
                             (pair_eq_mask(vh, vl, bh[p], bl[p]) & __hlt2_mask(u2h2(ab), u2h2(bab[p])));
          bh[p] = msel(vh, bh[p], m);
          bl[p] = msel(vl, bl[p], m);
          bab[p] = msel(ab, bab[p], m);
          bcc[p] = msel(cc2, bcc[p], m);
        }
      }
      const size_t o = ((((size_t)b * P.To + to) * P.Ho + yo) * P.Wo + xg * 4 + o4);
      const size_t oo = o * P.ldy + P.y_coff + c;
      *reinterpret_cast<uint2*>(yh + oo) = make_uint2(bh[0], bh[1]);
      if (yl != nullptr) *reinterpret_cast<uint2*>(yl + oo) = make_uint2(bl[0], bl[1]);
      if (P.y2_hi != nullptr)
        st_pair4<true>(reinterpret_cast<uint16_t*>(P.y2_hi), reinterpret_cast<uint16_t*>(P.y2_lo), oo,
                       make_float4(h2f((uint16_t)(bh[0] & 0xffff)) + h2f((uint16_t)(bl[0] & 0xffff)),
                                   h2f((uint16_t)(bh[0] >> 16)) + h2f((uint16_t)(bl[0] >> 16)),
                                   h2f((uint16_t)(bh[1] & 0xffff)) + h2f((uint16_t)(bl[1] & 0xffff)),
                                   h2f((uint16_t)(bh[1] >> 16)) + h2f((uint16_t)(bl[1] >> 16))));
      if (P.idx)
        *reinterpret_cast<uchar4*>(P.idx + o * P.C + c) =
            make_uchar4((unsigned char)(h_lo_int(bab[0]) * 3 + h_lo_int(bcc[0])),
                        (unsigned char)(h_hi_int(bab[0]) * 3 + h_hi_int(bcc[0])),
                        (unsigned char)(h_lo_int(bab[1]) * 3 + h_lo_int(bcc[1])),
                        (unsigned char)(h_hi_int(bab[1]) * 3 + h_hi_int(bcc[1])));
    }
  }
}

// 3x3x3 / stride 1 / pad 1 through shared memory (the form the launcher uses when W >= 8): a CTA owns (clip, 8 output
// rows, all W columns, 16 channels) and walks along t.  Every input frame tile (10 x (W+2) pixels, -inf outside the
// image) is staged ONCE with 16-byte cp.async copies -- the next frame's copies are in flight while the current one is
// reduced -- so an input element leaves L2 1.25 times instead of 13.5 times (the register-only kernel above re-reads its
// 54 neighbours per 4 outputs through L1/L2, which is what bounds it: 14 % of the HBM roofline).  Per frame a thread
// (row, column, 8 channels) reduces the 9 taps of that frame to the plane maximum of ITS output position, keeps the
// plane maxima of the last two frames in registers and emits output t-1 as the maximum of three plane maxima.  Compares
// run on the exact fp32 sums hi + lo; ties resolve to the first tap in (t, y, x) scan order like nn.MaxPool3d; the
// output planes are the re-split of the winning value (same represented value).
static constexpr int kPoolTY = 8;
__global__ void __launch_bounds__(256) maxpool333_smem_kernel(const coclr_pool_t P) {
  extern __shared__ __align__(16) uint8_t pool_smem[];
  const int W = P.Wi, H = P.Hi, T = P.Ti;
  const int WP = W + 2;                                   // padded tile width
  const int plane_px = (kPoolTY + 2) * WP;                // pixels of one frame tile
  const uint32_t frame_bytes = (uint32_t)plane_px * 64u;  // hi (32 B / pixel) then lo
  const int ytiles = (H + kPoolTY - 1) / kPoolTY;
  const int cslices = P.C >> 4;
  int blk = blockIdx.x;
  const int cs = blk % cslices; blk /= cslices;
  const int yt = blk % ytiles;
  const int b = blk / ytiles;
  const int c0 = cs * 16, y0 = yt * kPoolTY;
  const int tid = threadIdx.x;
  const int cq = tid & 1, x = (tid >> 1) % W, y = (tid >> 1) / W;     // blockDim = 2 * W * kPoolTY
  const uint16_t* xh = reinterpret_cast<const uint16_t*>(P.x_hi);
  const uint16_t* xl = reinterpret_cast<const uint16_t*>(P.x_lo);
  uint16_t* yh = reinterpret_cast<uint16_t*>(P.y_hi);
  uint16_t* yl = reinterpret_cast<uint16_t*>(P.y_lo);
  const uint32_t sbase = smem_u32(pool_smem);
  // -inf (hi) / 0 (lo) everywhere once: the halo outside the image is never overwritten
  for (uint32_t i = tid; i < 3u * frame_bytes / 16u; i += blockDim.x) {
    const uint32_t within = (i * 16u) % frame_bytes;
    const uint32_t v = within < (uint32_t)plane_px * 32u ? kNegInf2 : 0u;
    *reinterpret_cast<uint4*>(pool_smem + (size_t)i * 16) = make_uint4(v, v, v, v);
  }
  __syncthreads();
  auto issue_frame = [&](int f) {      // copies of frame f's tile into ring slot f % 3 (in-image pixels only)
    const uint32_t slot = sbase + (uint32_t)(f % 3) * frame_bytes;
    const int nchunk = (kPoolTY + 2) * W * 4;          // 16-byte chunks: rows x in-image columns x (hi0, hi1, lo0, lo1)
    for (int i = tid; i < nchunk; i += blockDim.x) {
      const int part = i & 3, px = (i >> 2) % W, ry = (i >> 2) / W;
      const int yi = y0 - 1 + ry;
      if ((unsigned)yi >= (unsigned)H) continue;
      const size_t goff = ((((size_t)b * T + f) * H + yi) * W + px) * P.ldx + P.x_coff + c0 + (part & 1) * 8;
      const uint32_t dst = slot + (part >> 1) * (uint32_t)plane_px * 32u + (uint32_t)(ry * WP + px + 1) * 32u + (part & 1) * 16u;
      const uint16_t* src = (part >> 1) ? xl : xh;
      if (src != nullptr) cp_async16(dst, src + goff, 16u);
    }
    cp_async_commit();
  };
  float v2[8], v1[8];
  int i2[8], i1[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) { v2[k] = v1[k] = -INFINITY; i2[k] = i1[k] = 0; }
  const bool active = (y0 + y) < H;
  issue_frame(0);
  for (int f = 0; f <= T; ++f) {
    if (f + 1 < T) issue_frame(f + 1); else cp_async_commit();    // keep the group count uniform
    cp_async_wait<1>();
    __syncthreads();
    float v0[8];
    int i0[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) { v0[k] = -INFINITY; i0[k] = 0; }
    if (f < T) {
      const uint8_t* slot = pool_smem + (size_t)(f % 3) * frame_bytes;
#pragma unroll
      for (int bb = 0; bb < 3; ++bb) {
#pragma unroll
        for (int cc = 0; cc < 3; ++cc) {
          const uint32_t px = (uint32_t)((y + bb) * WP + x + cc);
          const uint4 h = *reinterpret_cast<const uint4*>(slot + px * 32u + cq * 16u);
          const uint4 l = *reinterpret_cast<const uint4*>(slot + (size_t)plane_px * 32u + px * 32u + cq * 16u);
          const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float a0 = h2f((uint16_t)(hw[k] & 0xffff)) + h2f((uint16_t)(lw[k] & 0xffff));
            const float a1 = h2f((uint16_t)(hw[k] >> 16)) + h2f((uint16_t)(lw[k] >> 16));
            if (a0 > v0[2 * k]) { v0[2 * k] = a0; i0[2 * k] = bb * 3 + cc; }            // ascending (y, x): first max wins
            if (a1 > v0[2 * k + 1]) { v0[2 * k + 1] = a1; i0[2 * k + 1] = bb * 3 + cc; }
          }
        }
      }
    }
    if (f >= 1 && active) {
      const int to = f - 1;
      float bv[8];
      int bt[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        bv[k] = v2[k]; bt[k] = i2[k];                                       // frame to - 1
        if (v1[k] > bv[k]) { bv[k] = v1[k]; bt[k] = 9 + i1[k]; }            // frame to
        if (v0[k] > bv[k]) { bv[k] = v0[k]; bt[k] = 18 + i0[k]; }           // frame to + 1
      }
      const size_t op = ((((size_t)b * P.To + to) * P.Ho + y0 + y) * P.Wo + x);
      const size_t oo = op * P.ldy + P.y_coff + c0 + cq * 8;
      st_pair4<false>(yh, yl, oo, make_float4(bv[0], bv[1], bv[2], bv[3]));
      st_pair4<false>(yh, yl, oo + 4, make_float4(bv[4], bv[5], bv[6], bv[7]));
      if (P.y2_hi != nullptr) {
        st_pair4<true>(reinterpret_cast<uint16_t*>(P.y2_hi), reinterpret_cast<uint16_t*>(P.y2_lo), oo,
                       make_float4(bv[0], bv[1], bv[2], bv[3]));
        st_pair4<true>(reinterpret_cast<uint16_t*>(P.y2_hi), reinterpret_cast<uint16_t*>(P.y2_lo), oo + 4,
                       make_float4(bv[4], bv[5], bv[6], bv[7]));
      }
      if (P.idx) {
        uchar4* ip = reinterpret_cast<uchar4*>(P.idx + op * P.C + c0 + cq * 8);
        ip[0] = make_uchar4((unsigned char)bt[0], (unsigned char)bt[1], (unsigned char)bt[2], (unsigned char)bt[3]);
        ip[1] = make_uchar4((unsigned char)bt[4], (unsigned char)bt[5], (unsigned char)bt[6], (unsigned char)bt[7]);
      }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) { v2[k] = v1[k]; i2[k] = i1[k]; v1[k] = v0[k]; i1[k] = i0[k]; }
    __syncthreads();     // everyone is done with slot f % 3's neighbours before frame f + 2 lands in slot (f + 2) % 3
  }
}

// (1,3,3) / stride (1,2,2) / pad (0,1,1) through shared memory (MaxPool_2a on 64-channel 64x64 frames, MaxPool_3a on
// 192-channel 32x32 frames): a CTA owns (clip, frame, kPool133TY output rows, all Wo columns, 16 channels); the
// (2*TY+1) x (W+1) input pixels it needs are staged once with 16-byte cp.async copies (-inf outside the image), then
// every thread (output row, output column, 8 channels) reduces its 9 taps from shared memory.  An input element leaves
// L2 ~1.1 times instead of 2.25 times, in 16-byte instead of 8-byte requests.
static constexpr int kPool133TY = 4;
__global__ void __launch_bounds__(256) maxpool133s2_smem_kernel(const coclr_pool_t P) {
  extern __shared__ __align__(16) uint8_t pool_smem[];
  const int W = P.Wi, H = P.Hi, Wo = P.Wo, Ho = P.Ho;
  const int WP = W + 1;                                   // column 0 = image column -1
  const int rows = 2 * kPool133TY + 1;
  const int plane_px = rows * WP;
  const int ytiles = (Ho + kPool133TY - 1) / kPool133TY;
  const int cslices = P.C >> 4;
  int blk = blockIdx.x;
  const int cs = blk % cslices; blk /= cslices;
  const int yt = blk % ytiles; blk /= ytiles;
  const int t = blk % P.Ti;
  const int b = blk / P.Ti;
  const int c0 = cs * 16, yo0 = yt * kPool133TY;
  const int yi0 = 2 * yo0 - 1;                             // first staged image row
  const int tid = threadIdx.x;
  const uint16_t* xh = reinterpret_cast<const uint16_t*>(P.x_hi);
  const uint16_t* xl = reinterpret_cast<const uint16_t*>(P.x_lo);
  uint16_t* yh = reinterpret_cast<uint16_t*>(P.y_hi);
  uint16_t* yl = reinterpret_cast<uint16_t*>(P.y_lo);
  const uint32_t sbase = smem_u32(pool_smem);
  // halo column and out-of-image rows: -inf (hi) / 0 (lo)
  for (int i = tid; i < rows * 2; i += blockDim.x) {       // column 0 of every row, both 16-byte halves
    const int ry = i >> 1, part = i & 1;
    *reinterpret_cast<uint4*>(pool_smem + (size_t)(ry * WP) * 32 + part * 16) = make_uint4(kNegInf2, kNegInf2, kNegInf2, kNegInf2);
    *reinterpret_cast<uint4*>(pool_smem + (size_t)plane_px * 32 + (size_t)(ry * WP) * 32 + part * 16) = make_uint4(0u, 0u, 0u, 0u);
  }
  const int nchunk = rows * W * 4;                          // rows x image columns x (hi0, hi1, lo0, lo1)
  for (int i = tid; i < nchunk; i += blockDim.x) {
    const int part = i & 3, px = (i >> 2) % W, ry = (i >> 2) / W;
    const int yi = yi0 + ry;
    const uint32_t dst = (part >> 1) * (uint32_t)plane_px * 32u + (uint32_t)(ry * WP + px + 1) * 32u + (part & 1) * 16u;
    const uint16_t* src = (part >> 1) ? xl : xh;
    if ((unsigned)yi < (unsigned)H && src != nullptr) {
      const size_t goff = ((((size_t)b * P.Ti + t) * H + yi) * W + px) * P.ldx + P.x_coff + c0 + (part & 1) * 8;
      cp_async16(sbase + dst, src + goff, 16u);
    } else {
      const uint32_t v = (part >> 1) ? 0u : kNegInf2;
      *reinterpret_cast<uint4*>(pool_smem + dst) = make_uint4(v, v, v, v);
    }
  }
  cp_async_commit();
  cp_async_wait<0>();
  __syncthreads();
  const int cq = tid & 1, xo = (tid >> 1) % Wo, yl_ = (tid >> 1) / Wo;     // blockDim = 2 * Wo * kPool133TY
  const int yo = yo0 + yl_;
  if (yo >= Ho) return;
  float bv[8];
  int bt[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) { bv[k] = -INFINITY; bt[k] = 0; }
#pragma unroll
  for (int bb = 0; bb < 3; ++bb) {
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) {
      const uint32_t px = (uint32_t)((2 * yl_ + bb) * WP + 2 * xo + cc);
      const uint4 h = *reinterpret_cast<const uint4*>(pool_smem + (size_t)px * 32 + cq * 16);
      const uint4 l = *reinterpret_cast<const uint4*>(pool_smem + (size_t)plane_px * 32 + (size_t)px * 32 + cq * 16);
      const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float a0 = h2f((uint16_t)(hw[k] & 0xffff)) + h2f((uint16_t)(lw[k] & 0xffff));
        const float a1 = h2f((uint16_t)(hw[k] >> 16)) + h2f((uint16_t)(lw[k] >> 16));
        if (a0 > bv[2 * k]) { bv[2 * k] = a0; bt[2 * k] = bb * 3 + cc; }
        if (a1 > bv[2 * k + 1]) { bv[2 * k + 1] = a1; bt[2 * k + 1] = bb * 3 + cc; }
      }
    }
  }
  const size_t op = ((((size_t)b * P.To + t) * Ho + yo) * Wo + xo);
  const size_t oo = op * P.ldy + P.y_coff + c0 + cq * 8;
  st_pair4<false>(yh, yl, oo, make_float4(bv[0], bv[1], bv[2], bv[3]));
  st_pair4<false>(yh, yl, oo + 4, make_float4(bv[4], bv[5], bv[6], bv[7]));
  if (P.y2_hi != nullptr) {
    st_pair4<true>(reinterpret_cast<uint16_t*>(P.y2_hi), reinterpret_cast<uint16_t*>(P.y2_lo), oo,
                   make_float4(bv[0], bv[1], bv[2], bv[3]));
    st_pair4<true>(reinterpret_cast<uint16_t*>(P.y2_hi), reinterpret_cast<uint16_t*>(P.y2_lo), oo + 4,
                   make_float4(bv[4], bv[5], bv[6], bv[7]));
  }
  if (P.idx) {
    uchar4* ip = reinterpret_cast<uchar4*>(P.idx + op * P.C + c0 + cq * 8);
    ip[0] = make_uchar4((unsigned char)bt[0], (unsigned char)bt[1], (unsigned char)bt[2], (unsigned char)bt[3]);
    ip[1] = make_uchar4((unsigned char)bt[4], (unsigned char)bt[5], (unsigned char)bt[6], (unsigned char)bt[7]);
  }
}

// scatter form of the backward: every output element adds its gradient to the one input element that won.  Used only
// for pools whose windows do not overlap, where every input receives at most one addend and the result does not
// depend on the order of the fp32 reductions in L2.
__global__ void __launch_bounds__(256) maxpool_bwd_scatter_kernel(const coclr_pool_t P) {
  const int C4 = P.C >> 2;
  const int khw = P.g.kh * P.g.kw;
  const long total = (long)P.B * P.To * P.Ho * P.Wo * C4;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int cg = (int)(i % C4);
    long r = i / C4;
    const int xo = (int)(r % P.Wo); r /= P.Wo;
    const int yo = (int)(r % P.Ho); r /= P.Ho;
    const int to = (int)(r % P.To);
    const int b = (int)(r / P.To);
    const int c = cg * 4;
    const size_t o = ((((size_t)b * P.To + to) * P.Ho + yo) * P.Wo + xo);
    const uchar4 id = *reinterpret_cast<const uchar4*>(P.idx + o * P.C + c);
    const float4 d = ld4(P.dy + o * P.C + c);
    const unsigned char taps[4] = {id.x, id.y, id.z, id.w};
    const float dv[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int tap = taps[k];
      const int a = tap / khw, rem = tap - a * khw;
      const int bb = rem / P.g.kw, cc = rem - bb * P.g.kw;
      const int ti = to * P.g.st - P.g.pt + a, yi = yo * P.g.sh - P.g.ph + bb, xi = xo * P.g.sw - P.g.pw + cc;
      atomicAdd(P.dx + ((((size_t)b * P.Ti + ti) * P.Hi + yi) * P.Wi + xi) * P.ldx + P.x_coff + c + k, dv[k]);
    }
  }
}

// gather form for the (3,3,3)/1 pool with padding 1 and equal input / output shapes (the SepInception branch-3 pools),
// four inputs along x per thread: the 3 x 3 x 6 windows that can hold their maxima are read once for all four instead
// of 27 times per input.  Each input's sum runs in a fixed window order.
__global__ void __launch_bounds__(256) maxpool333_bwd_gather4_kernel(const coclr_pool_t P) {
  const int C4 = P.C >> 2, W4 = P.Wi >> 2;
  const long total = (long)P.B * P.Ti * P.Hi * W4 * C4;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int cg = (int)(i % C4);
    long r = i / C4;
    const int x0 = (int)(r % W4) * 4; r /= W4;
    const int yi = (int)(r % P.Hi); r /= P.Hi;
    const int ti = (int)(r % P.Ti);
    const int b = (int)(r / P.Ti);
    const int c = cg * 4;
    float acc[4][4];
#pragma unroll
    for (int k = 0; k < 4; ++k) acc[k][0] = acc[k][1] = acc[k][2] = acc[k][3] = 0.f;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const int nt = ti + 1 - a;
      if (nt < 0 || nt >= P.To) continue;
#pragma unroll
      for (int bb = 0; bb < 3; ++bb) {
        const int ny = yi + 1 - bb;
        if (ny < 0 || ny >= P.Ho) continue;
        const size_t orow = (((size_t)b * P.To + nt) * P.Ho + ny) * P.Wo;
#pragma unroll
        for (int q = 0; q < 6; ++q) {
          const int nx = x0 - 1 + q;
          if (nx < 0 || nx >= P.Wo) continue;
          const uchar4 id = *reinterpret_cast<const uchar4*>(P.idx + (orow + nx) * P.C + c);
          const unsigned char taps[4] = {id.x, id.y, id.z, id.w};
          // input x0 + k lies in column cc = k - q + 2 of window nx
          bool hit = false;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int cc = k - q + 2;
            if (cc < 0 || cc > 2) continue;
            const int tap = (a * 3 + bb) * 3 + cc;
#pragma unroll
            for (int j = 0; j < 4; ++j) hit |= taps[j] == tap;
          }
          if (!hit) continue;
          const float4 d = ld4(P.dy + (orow + nx) * P.C + c);
          const float dv[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int cc = k - q + 2;
            if (cc < 0 || cc > 2) continue;
            const int tap = (a * 3 + bb) * 3 + cc;
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (taps[j] == tap) acc[k][j] += dv[j];
          }
        }
      }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float* dp = P.dx + ((((size_t)b * P.Ti + ti) * P.Hi + yi) * P.Wi + x0 + k) * P.ldx + P.x_coff + c;
      float4 v = make_float4(acc[k][0], acc[k][1], acc[k][2], acc[k][3]);
      if (P.accumulate) {
        const float4 old = ld4(dp);
        v.x += old.x; v.y += old.y; v.z += old.z; v.w += old.w;
      }
      st4(dp, v);
    }
  }
}

// gather form of the backward: dX[in] (+)= sum over windows whose arg-max is `in` of dY[out]
template <int KT, int KH, int KW, int ST, int SH, int SW>
__global__ void __launch_bounds__(256) maxpool_bwd_kernel(const coclr_pool_t P) {
  const int kt = KT ? KT : P.g.kt, kh = KH ? KH : P.g.kh, kw = KW ? KW : P.g.kw;
  const int st = ST ? ST : P.g.st, sh = SH ? SH : P.g.sh, sw = SW ? SW : P.g.sw;
  const int C4 = P.C >> 2;
  const long total = (long)P.B * P.Ti * P.Hi * P.Wi * C4;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int cg = (int)(i % C4);
    long r = i / C4;
    const int xi = (int)(r % P.Wi); r /= P.Wi;
    const int yi = (int)(r % P.Hi); r /= P.Hi;
    const int ti = (int)(r % P.Ti);
    const int b = (int)(r / P.Ti);
    const int c = cg * 4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int a = 0; a < kt; ++a) {
      int nt = ti + P.g.pt - a;
      if (nt < 0 || (nt % st) != 0) continue;
      nt /= st;
      if (nt >= P.To) continue;
#pragma unroll
      for (int bb = 0; bb < kh; ++bb) {
        int ny = yi + P.g.ph - bb;
        if (ny < 0 || (ny % sh) != 0) continue;
        ny /= sh;
        if (ny >= P.Ho) continue;
#pragma unroll
        for (int cc = 0; cc < kw; ++cc) {
          int nx = xi + P.g.pw - cc;
          if (nx < 0 || (nx % sw) != 0) continue;
          nx /= sw;
          if (nx >= P.Wo) continue;
          const int tap = (a * kh + bb) * kw + cc;
          const size_t o = ((((size_t)b * P.To + nt) * P.Ho + ny) * P.Wo + nx);
          const uchar4 id = *reinterpret_cast<const uchar4*>(P.idx + o * P.C + c);
          if (id.x == tap || id.y == tap || id.z == tap || id.w == tap) {
            const float4 d = ld4(P.dy + o * P.C + c);
            if (id.x == tap) acc.x += d.x;
            if (id.y == tap) acc.y += d.y;
            if (id.z == tap) acc.z += d.z;
            if (id.w == tap) acc.w += d.w;
          }
        }
      }
    }
    float* dp = P.dx + ((((size_t)b * P.Ti + ti) * P.Hi + yi) * P.Wi + xi) * P.ldx + P.x_coff + c;
    if (P.accumulate) {
      const float4 old = ld4(dp);
      acc.x += old.x; acc.y += old.y; acc.z += old.z; acc.w += old.w;
    }
    st4(dp, acc);
  }
}

// ------------------------------------------------------------------------------------------------
// AdaptiveAvgPool3d((1,1,1)) (model/pretrain.py:51) over fp16 hi/lo planes, and its backward
// ------------------------------------------------------------------------------------------------
__global__ void avgpool_fwd_kernel(const uint16_t* xh, const uint16_t* xl, int bf16, int ld, int coff, float* out, int B,
                                   int Pn, int C) {
  const int C4 = C >> 2;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * C4) return;
  const int cg = i % C4, b = i / C4;
  const int c = cg * 4;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int p = 0; p < Pn; ++p) {
    const float4 v = ld_pair4_any(xh, xl, ((size_t)b * Pn + p) * ld + coff + c, bf16);
    s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
  }
  const float inv = 1.f / (float)Pn;
  st4(out + (size_t)b * C + c, make_float4(s.x * inv, s.y * inv, s.z * inv, s.w * inv));
}
__global__ void avgpool_bwd_kernel(const float* dfeat, float* dA, int ld, int coff, int B, int Pn, int C) {
  const int C4 = C >> 2;
  const long total = (long)B * Pn * C4;
  const float inv = 1.f / (float)Pn;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int cg = (int)(i % C4);
    const long r = i / C4;
    const int b = (int)(r / Pn);
    const float4 d = ld4(dfeat + (long)b * C + cg * 4);
    st4(dA + r * ld + coff + cg * 4, make_float4(d.x * inv, d.y * inv, d.z * inv, d.w * inv));
  }
}

// ------------------------------------------------------------------------------------------------
// clip packing: x[b, c, t, h, w] (c < Cin <= 8, arbitrary batch stride: the reference's block[:, i]
// .contiguous() copies, model/pretrain.py:149-150, are folded in) -> fp16 hi/lo planes [b, thw, 8]
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pack_input_kernel(const float* x, long batch_stride, long chan_stride, int Cin,
                                                         uint16_t* out_hi, uint16_t* out_lo, uint16_t* out2_hi,
                                                         uint16_t* out2_lo, int B, long thw,
                                                         const long* __restrict__ batch_index,
                                                         const float* const* __restrict__ peer_x, int cpp,
                                                         const float* __restrict__ nmean,
                                                         const float* __restrict__ nstd) {
  const long total = (long)B * thw;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long b = i / thw, p = i - b * thw;
    const long sb = batch_index ? batch_index[b] : b;  // shuffle-BN gather folded in (pretrain.py:124)
    const float* s = (peer_x ? peer_x[sb / cpp] + (sb % cpp) * batch_stride : x + sb * batch_stride) + p;
    uint16_t h[8], l[8];
    float vv[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      vv[j] = j < Cin ? s[(long)j * chan_stride] : 0.f;
      // T.Normalize of the reference's GPU-side `tr` (main_nce.py:207-209, utils/transforms.py:57-63): (x - mean) / std
      if (nmean != nullptr && j < Cin) vv[j] = __fdiv_rn(__fsub_rn(vv[j], nmean[j]), nstd[j]);
      split2<false>(vv[j], h[j], l[j]);
    }
    if (out2_hi != nullptr) {
      st_pair4<true>(out2_hi, out2_lo, (size_t)i * 8, make_float4(vv[0], vv[1], vv[2], vv[3]));
      st_pair4<true>(out2_hi, out2_lo, (size_t)i * 8 + 4, make_float4(vv[4], vv[5], vv[6], vv[7]));
    }
    *reinterpret_cast<uint4*>(out_hi + i * 8) =
        make_uint4((uint32_t)h[0] | ((uint32_t)h[1] << 16), (uint32_t)h[2] | ((uint32_t)h[3] << 16),
                   (uint32_t)h[4] | ((uint32_t)h[5] << 16), (uint32_t)h[6] | ((uint32_t)h[7] << 16));
    if (out_lo != nullptr)
      *reinterpret_cast<uint4*>(out_lo + i * 8) =
          make_uint4((uint32_t)l[0] | ((uint32_t)l[1] << 16), (uint32_t)l[2] | ((uint32_t)l[3] << 16),
                     (uint32_t)l[4] | ((uint32_t)l[5] << 16), (uint32_t)l[6] | ((uint32_t)l[7] << 16));
  }
}

// Space-to-depth variant for the stride-2 7x7 stem (backbone/s3dg.py:145): out[b, t, Y, X, (dy*2+dx)*Cin + c] =
// x[b, c, t, 2Y+dy, 2X+dx], 16 channels per pixel (4*Cin = 12 real + zeros).  The stem then is a stride-1
// 4x4 convolution over 16-channel pixels: 32-byte gather granules and 16 instead of 49 taps.
template <int Cin>
__global__ void __launch_bounds__(256) pack_input_s2d_kernel(const float* x, long batch_stride, long chan_stride,
                                                             uint16_t* out_hi, uint16_t* out_lo,
                                                             uint16_t* out2_hi, uint16_t* out2_lo, int B, int T, int H,
                                                             int W, int pad_x, const long* __restrict__ batch_index,
                                                             const float* const* __restrict__ peer_x, int cpp,
                                                             const float* __restrict__ nmean,
                                                             const float* __restrict__ nstd) {
  const int H2 = H >> 1, W2 = W >> 1;
  const long total = (long)B * T * H2 * W2;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int X = (int)(i % W2);
    long r = i / W2;
    const int Y = (int)(r % H2); r /= H2;
    const int t = (int)(r % T);
    const long b = r / T;
    const long sb = batch_index ? batch_index[b] : b;
    const float* base = peer_x ? peer_x[sb / cpp] + (sb % cpp) * batch_stride : x + sb * batch_stride;
    const float* s = base + ((long)t * H + 2 * Y) * W + 2 * X;
    float vv[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) vv[j] = 0.f;
    // (dx = 0, 1) are adjacent floats at an even offset: one 8-byte load per (channel, dy)
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
      for (int c = 0; c < Cin; ++c) {
        float2 p2 = *reinterpret_cast<const float2*>(s + (long)c * chan_stride + dy * W);
        if (nmean != nullptr) {   // fused T.Normalize, see pack_input_kernel
          p2.x = __fdiv_rn(__fsub_rn(p2.x, nmean[c]), nstd[c]);
          p2.y = __fdiv_rn(__fsub_rn(p2.y, nmean[c]), nstd[c]);
        }
        vv[(dy * 2 + 0) * Cin + c] = p2.x;
        vv[(dy * 2 + 1) * Cin + c] = p2.y;
      }
    uint32_t hw[8], lw[8], h2[8], l2[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      uint16_t a, b, c2, d;
      split2<false>(vv[2 * j], a, b);
      split2<false>(vv[2 * j + 1], c2, d);
      hw[j] = (uint32_t)a | ((uint32_t)c2 << 16);
      lw[j] = (uint32_t)b | ((uint32_t)d << 16);
      if (out2_hi != nullptr) {
        split2<true>(vv[2 * j], a, b);
        split2<true>(vv[2 * j + 1], c2, d);
        h2[j] = (uint32_t)a | ((uint32_t)c2 << 16);
        l2[j] = (uint32_t)b | ((uint32_t)d << 16);
      }
    }
    // output rows are W2 + 2*pad_x pixels wide; the pad pixels are never written (the caller zeroes them once)
    const size_t o = ((size_t)(i / W2) * (size_t)(W2 + 2 * pad_x) + (size_t)(X + pad_x)) * 16;
    auto st32 = [](uint16_t* p, size_t off, const uint32_t* w) {
      uint4* q = reinterpret_cast<uint4*>(p + off);
      q[0] = make_uint4(w[0], w[1], w[2], w[3]);
      q[1] = make_uint4(w[4], w[5], w[6], w[7]);
    };
    st32(out_hi, o, hw);
    if (out_lo != nullptr) st32(out_lo, o, lw);
    if (out2_hi != nullptr) {
      st32(out2_hi, o, h2);
      if (out2_lo != nullptr) st32(out2_lo, o, l2);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// F.normalize(z + bias, dim=1) (model/pretrain.py:154,167) and backward; one warp per row
// ------------------------------------------------------------------------------------------------
__global__ void l2norm_fwd_kernel(const float* z, const float* bias, float* q, float* inv_norm, int B, int D) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= B) return;
  float ss = 0.f;
  for (int c = lane; c < D; c += 32) {
    const float v = z[(long)row * D + c] + (bias ? bias[c] : 0.f);
    ss += v * v;
  }
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const float inv = 1.f / fmaxf(sqrtf(ss), 1e-12f);
  for (int c = lane; c < D; c += 32) q[(long)row * D + c] = (z[(long)row * D + c] + (bias ? bias[c] : 0.f)) * inv;
  if (lane == 0 && inv_norm) inv_norm[row] = inv;
}
// dz = (dq - q * <q, dq>) * inv_norm
__global__ void l2norm_bwd_kernel(const float* q, const float* dq, const float* inv_norm, float* dz, int B, int D) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= B) return;
  float dot = 0.f;
  for (int c = lane; c < D; c += 32) dot += q[(long)row * D + c] * dq[(long)row * D + c];
  for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
  const float inv = inv_norm[row];
  for (int c = lane; c < D; c += 32)
    dz[(long)row * D + c] = (dq[(long)row * D + c] - q[(long)row * D + c] * dot) * inv;
}
__global__ void colsum_small_kernel(const float* x, float* out, int M, int C) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float s = 0.f;
  for (int r = 0; r < M; ++r) s += x[(long)r * C + c];
  out[c] += s;
}

// ------------------------------------------------------------------------------------------------
// momentum update of the key encoder: k = k*m + q*(1-m) (model/pretrain.py:76-80), bit-exact
// with the reference's two roundings (no FMA contraction), one launch for all parameters
// ------------------------------------------------------------------------------------------------
__global__ void ema_kernel(float* __restrict__ k, const float* __restrict__ q, float m, float one_minus_m, long n) {
  const long n4 = n >> 2;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    float4 a = reinterpret_cast<float4*>(k)[i];
    const float4 b = reinterpret_cast<const float4*>(q)[i];
    a.x = __fadd_rn(__fmul_rn(a.x, m), __fmul_rn(b.x, one_minus_m));
    a.y = __fadd_rn(__fmul_rn(a.y, m), __fmul_rn(b.y, one_minus_m));
    a.z = __fadd_rn(__fmul_rn(a.z, m), __fmul_rn(b.z, one_minus_m));
    a.w = __fadd_rn(__fmul_rn(a.w, m), __fmul_rn(b.w, one_minus_m));
    reinterpret_cast<float4*>(k)[i] = a;
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
    const long i = (n4 << 2) + threadIdx.x;
    k[i] = __fadd_rn(__fmul_rn(k[i], m), __fmul_rn(q[i], one_minus_m));
  }
}

// queue[:, ptr:ptr+n] = keys^T (model/pretrain.py:82-96); consecutive threads write consecutive columns
__global__ void enqueue_kernel(float* queue, const float* keys, int dim, int K, int ptr, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= dim * n) return;
  const int c = i / n, j = i - c * n;
  queue[(long)c * K + ptr + j] = keys[(long)j * dim + c];
}

// torch.optim.Adam with coupled L2 weight decay (main_nce.py:190-200) over one flat buffer
__global__ void adam_kernel(const coclr_adam_t P) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < P.n; i += (long)gridDim.x * blockDim.x) {
    const float p = P.param[i];
    float g = P.grad[i] * P.grad_scale;
    g = g + P.weight_decay * p;
    float m = P.exp_avg[i];
    float v = P.exp_avg_sq[i];
    m = m + (1.f - P.beta1) * (g - m);
    v = v * P.beta2 + (1.f - P.beta2) * g * g;
    const float denom = sqrtf(v) / P.bc2_sqrt + P.eps;
    P.param[i] = p - P.step_size * (m / denom);
    P.exp_avg[i] = m;
    P.exp_avg_sq[i] = v;
  }
}

static inline int grid_for(long total, int threads, int cap) {
  long g = (total + threads - 1) / threads;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace coclr

using namespace coclr;
#define LAUNCH_OK() (cudaGetLastError() == cudaSuccess ? COCLR_OK : COCLR_E_LAUNCH)

extern "C" int coclr_bn_finalize(const coclr_bn_finalize_t* p, coclr_stream_t stream) {
  if (!p || !p->scale || !p->shift || !p->gamma || !p->beta || p->C <= 0) return COCLR_E_ARG;
  if (p->training && (!p->sum || !p->sumsq || p->count <= 0)) return COCLR_E_ARG;
  bn_finalize_kernel<<<(p->C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*p);
  return LAUNCH_OK();
}

extern "C" int coclr_affine_split(const coclr_split_t* p, int num_sms, coclr_stream_t stream) {
  if (!p || !p->x || !p->hi || p->C % 4 || p->ld % 4 || p->coff % 4 || p->out_ld % 4 || p->out_coff % 4)
    return COCLR_E_ARG;
  if (p->res_hi && (p->res_ld % 4 || p->res_coff % 4)) return COCLR_E_ARG;
  const long total = p->M * (p->C / 4);
  if (p->bn.scale != nullptr) {  // fused BatchNorm finalize
    const coclr_bn_finalize_t& f = p->bn;
    if (!f.shift || !f.gamma || !f.beta || !f.running_mean || !f.running_var || p->C > kMaxBnC) return COCLR_E_ARG;
    if (f.training && (!f.sum || !f.sumsq || f.count <= 0)) return COCLR_E_ARG;
    const int grid = grid_for(total, 256, num_sms * 16);
    if (p->bf16)
      bn_apply_split_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(*p);
    else
      bn_apply_split_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(*p);
    return LAUNCH_OK();
  }
  const int grid = grid_for(total, 256, num_sms * 16);
  if (p->bf16)
    affine_split_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(*p);
  else
    affine_split_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(*p);
  return LAUNCH_OK();
}

extern "C" int coclr_bn_bwd(const coclr_bn_bwd_t* p, int num_sms, coclr_stream_t stream) {
  if (!p || !p->y || !p->dA || !p->sums || !p->dy_hi || p->C % 4 || p->ld % 4 || p->coff % 4) return COCLR_E_ARG;
  if (p->res_hi && (p->res_ld % 4 || p->res_coff % 4 || !p->relu)) return COCLR_E_ARG;
  if (p->dres && (p->dres_ld % 4 || p->dres_coff % 4)) return COCLR_E_ARG;
  const int ctiles = (p->C + kBwdTileC - 1) / kBwdTileC;
  if (ctiles > 1 && p->C % kBwdTileC) return COCLR_E_ARG;   // wide tensors: whole tiles only
  const int C4 = (ctiles > 1 ? kBwdTileC : p->C) / 4;
  const int R = kColThreads / C4;
  long slabs = ((long)p->M + (long)R * 16 - 1) / ((long)R * 16);
  const long cap = (long)num_sms * 8 / ctiles;
  int gx = (int)(slabs < cap ? slabs : cap);
  if (gx < 1) gx = 1;
  const dim3 grid(gx, ctiles);
  cudaStream_t s = (cudaStream_t)stream;
  if (cudaMemsetAsync(p->sums, 0, sizeof(double) * 2 * p->C, s) != cudaSuccess) return COCLR_E_LAUNCH;
  if (p->dy_fp16 && (!p->amax || !p->dy_scale)) return COCLR_E_ARG;
  if (p->amax && cudaMemsetAsync(p->amax, 0, sizeof(float) * 2 * p->C, s) != cudaSuccess) return COCLR_E_LAUNCH;
  bn_bwd_reduce_kernel<<<grid, kColThreads, 0, s>>>(*p);
  bn_bwd_apply_kernel<<<grid, kColThreads, 0, s>>>(*p);
  return LAUNCH_OK();
}

extern "C" int coclr_bias_relu_bwd(const float* h, const float* bias, float* dA, float* dbias, int M, int C,
                                   coclr_stream_t stream) {
  if (!h || !bias || !dA || !dbias) return COCLR_E_ARG;
  bias_relu_bwd_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h, bias, dA, dbias, M, C);
  return LAUNCH_OK();
}

template <bool kBwd>
static void launch_pool(const coclr_pool_t& p, long total, cudaStream_t s) {
  const int grid = grid_for(total, 256, 148 * 32);
  const coclr_geom_t& g = p.g;
#define POOL_CASE(KT, KH, KW, ST, SH, SW)                                                 \
  if (g.kt == KT && g.kh == KH && g.kw == KW && g.st == ST && g.sh == SH && g.sw == SW) { \
    if (kBwd)                                                                             \
      maxpool_bwd_kernel<KT, KH, KW, ST, SH, SW><<<grid, 256, 0, s>>>(p);                 \
    else                                                                                  \
      maxpool_fwd_kernel<KT, KH, KW, ST, SH, SW><<<grid, 256, 0, s>>>(p);                 \
    return;                                                                               \
  }
  POOL_CASE(1, 3, 3, 1, 2, 2)
  POOL_CASE(3, 3, 3, 1, 1, 1)
  POOL_CASE(3, 3, 3, 2, 2, 2)
  POOL_CASE(2, 2, 2, 2, 2, 2)
#undef POOL_CASE
  if (kBwd)
    maxpool_bwd_kernel<0, 0, 0, 0, 0, 0><<<grid, 256, 0, s>>>(p);
  else
    maxpool_fwd_kernel<0, 0, 0, 0, 0, 0><<<grid, 256, 0, s>>>(p);
}

extern "C" int coclr_maxpool_fwd(const coclr_pool_t* p, coclr_stream_t stream) {
  if (!p || !p->x_hi || !p->y_hi || p->C % 4 || p->ldx % 4 || p->ldy % 4 || p->x_coff % 4 || p->y_coff % 4)
    return COCLR_E_ARG;
  if (p->g.kt * p->g.kh * p->g.kw > 255) return COCLR_E_ARG;
  const long total = (long)p->B * p->To * p->Ho * p->Wo * (p->C / 4);
  const coclr_geom_t& g = p->g;
  if (g.kt == 3 && g.kh == 3 && g.kw == 3 && g.st == 1 && g.sh == 1 && g.sw == 1 && g.pt == 1 && g.ph == 1 &&
      g.pw == 1 && (p->Wo % 4) == 0 && p->Wo == p->Wi && p->Ho == p->Hi && p->To == p->Ti) {
    static const bool reg_form = getenv("COCLR_POOL333_REG") != nullptr;   // A/B timing: the register-only kernel
    const int threads = 2 * p->Wi * kPoolTY;
    if (!reg_form && p->Wi >= 8 && threads <= 256 && p->C % 16 == 0 && p->x_coff % 8 == 0 && p->y_coff % 8 == 0 &&
        p->ldx % 8 == 0 && p->ldy % 8 == 0) {
      const size_t smem = (size_t)3 * (kPoolTY + 2) * (p->Wi + 2) * 64;
      const int grid = p->B * ((p->Hi + kPoolTY - 1) / kPoolTY) * (p->C / 16);
      maxpool333_smem_kernel<<<grid, threads, smem, (cudaStream_t)stream>>>(*p);
      return LAUNCH_OK();
    }
    maxpool333_fwd_kernel<<<grid_for(total / 4, 256, 148 * 32), 256, 0, (cudaStream_t)stream>>>(*p);
    return LAUNCH_OK();
  }
  if (g.kt == 1 && g.kh == 3 && g.kw == 3 && g.st == 1 && g.sh == 2 && g.sw == 2 && g.pt == 0 && g.ph == 1 && g.pw == 1 &&
      getenv("COCLR_POOL133_REG") == nullptr && p->To == p->Ti && 2 * p->Ho == p->Hi && 2 * p->Wo == p->Wi &&
      2 * p->Wo * kPool133TY <= 256 && p->C % 16 == 0 && p->x_coff % 8 == 0 && p->y_coff % 8 == 0 && p->ldx % 8 == 0 &&
      p->ldy % 8 == 0) {
    const size_t smem = (size_t)(2 * kPool133TY + 1) * (p->Wi + 1) * 64;
    const int grid = p->B * p->Ti * ((p->Ho + kPool133TY - 1) / kPool133TY) * (p->C / 16);
    maxpool133s2_smem_kernel<<<grid, 2 * p->Wo * kPool133TY, smem, (cudaStream_t)stream>>>(*p);
    return LAUNCH_OK();
  }
  launch_pool<false>(*p, total, (cudaStream_t)stream);
  return LAUNCH_OK();
}
extern "C" int coclr_maxpool_bwd(const coclr_pool_t* p, coclr_stream_t stream) {
  if (!p || !p->dx || !p->dy || !p->idx || p->C % 4) return COCLR_E_ARG;
  // scatter form when the windows do not overlap, so that every input element receives at most one addend, and the
  // destination can be zero-initialised with one memset (or already holds the other consumers' contributions).
  // Overlapping windows go to the gather kernel, which sums each input's windows in a fixed order: fp32 atomics from
  // several windows would make the gradient, and every training step after it, differ from run to run.
  const bool disjoint = p->g.kt <= p->g.st && p->g.kh <= p->g.sh && p->g.kw <= p->g.sw;
  if (disjoint && (p->accumulate || (p->ldx == p->C && p->x_coff == 0))) {
    cudaStream_t s = (cudaStream_t)stream;
    if (!p->accumulate) {
      const size_t bytes = (size_t)p->B * p->Ti * p->Hi * p->Wi * p->C * sizeof(float);
      if (cudaMemsetAsync(p->dx, 0, bytes, s) != cudaSuccess) return COCLR_E_LAUNCH;
    }
    const long tot_o = (long)p->B * p->To * p->Ho * p->Wo * (p->C / 4);
    maxpool_bwd_scatter_kernel<<<grid_for(tot_o, 256, 148 * 32), 256, 0, s>>>(*p);
    return LAUNCH_OK();
  }
  const coclr_geom_t& g = p->g;
  if (g.kt == 3 && g.kh == 3 && g.kw == 3 && g.st == 1 && g.sh == 1 && g.sw == 1 && g.pt == 1 && g.ph == 1 &&
      g.pw == 1 && p->Wi % 4 == 0 && p->Wo == p->Wi && p->Ho == p->Hi && p->To == p->Ti) {
    const long total4 = (long)p->B * p->Ti * p->Hi * (p->Wi / 4) * (p->C / 4);
    maxpool333_bwd_gather4_kernel<<<grid_for(total4, 256, 148 * 32), 256, 0, (cudaStream_t)stream>>>(*p);
    return LAUNCH_OK();
  }
  const long total = (long)p->B * p->Ti * p->Hi * p->Wi * (p->C / 4);
  launch_pool<true>(*p, total, (cudaStream_t)stream);
  return LAUNCH_OK();
}

extern "C" int coclr_avgpool_fwd(const void* x_hi, const void* x_lo, int bf16, int ld, int coff, float* out, int B, int Pn,
                                 int C, coclr_stream_t stream) {
  if (!x_hi || !out || C % 4) return COCLR_E_ARG;
  avgpool_fwd_kernel<<<(B * (C / 4) + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const uint16_t*>(x_hi), reinterpret_cast<const uint16_t*>(x_lo), bf16, ld, coff, out, B, Pn, C);
  return LAUNCH_OK();
}
extern "C" int coclr_avgpool_bwd(const float* dfeat, float* dA, int ld, int coff, int B, int Pn, int C,
                                 coclr_stream_t stream) {
  if (!dfeat || !dA || C % 4) return COCLR_E_ARG;
  const long total = (long)B * Pn * (C / 4);
  avgpool_bwd_kernel<<<grid_for(total, 256, 148 * 8), 256, 0, (cudaStream_t)stream>>>(dfeat, dA, ld, coff, B, Pn, C);
  return LAUNCH_OK();
}

extern "C" int coclr_pack_input(const float* x, long batch_stride, long chan_stride, int Cin, void* out_hi, void* out_lo,
                                void* out2_hi, void* out2_lo, int B, long thw, const long* batch_index,
                                const void* const* peer_x, int clips_per_peer, const float* norm_mean,
                                const float* norm_std, coclr_stream_t stream) {
  if ((!x && !peer_x) || !out_hi || Cin < 1 || Cin > 8 || (!norm_mean != !norm_std)) return COCLR_E_ARG;
  if (peer_x && (!batch_index || clips_per_peer < 1)) return COCLR_E_ARG;
  pack_input_kernel<<<grid_for((long)B * thw, 256, 148 * 16), 256, 0, (cudaStream_t)stream>>>(
      x, batch_stride, chan_stride, Cin, reinterpret_cast<uint16_t*>(out_hi), reinterpret_cast<uint16_t*>(out_lo),
      reinterpret_cast<uint16_t*>(out2_hi), reinterpret_cast<uint16_t*>(out2_lo), B, thw, batch_index,
      reinterpret_cast<const float* const*>(peer_x), clips_per_peer, norm_mean, norm_std);
  return LAUNCH_OK();
}

extern "C" int coclr_pack_input_s2d(const float* x, long batch_stride, long chan_stride, int Cin, void* out_hi,
                                    void* out_lo, void* out2_hi, void* out2_lo, int B, int T, int H, int W, int pad_x,
                                    const long* batch_index, const void* const* peer_x, int clips_per_peer,
                                    const float* norm_mean, const float* norm_std, coclr_stream_t stream) {
  if ((!x && !peer_x) || !out_hi || Cin < 1 || Cin > 4 || (H & 1) || (W & 1) || (!norm_mean != !norm_std) || pad_x < 0)
    return COCLR_E_ARG;
  if (peer_x && (!batch_index || clips_per_peer < 1)) return COCLR_E_ARG;
  const long total = (long)B * T * (H / 2) * (W / 2);
  if ((batch_stride | chan_stride) & 1) return COCLR_E_ARG;  // 8-byte loads of (x, x+1) pairs
#define COCLR_PACK_S2D(CIN)                                                                                         \
  pack_input_s2d_kernel<CIN><<<grid_for(total, 256, 148 * 16), 256, 0, (cudaStream_t)stream>>>(                    \
      x, batch_stride, chan_stride, reinterpret_cast<uint16_t*>(out_hi), reinterpret_cast<uint16_t*>(out_lo),       \
      reinterpret_cast<uint16_t*>(out2_hi), reinterpret_cast<uint16_t*>(out2_lo), B, T, H, W, pad_x, batch_index,   \
      reinterpret_cast<const float* const*>(peer_x), clips_per_peer, norm_mean, norm_std)
  switch (Cin) {
    case 1: COCLR_PACK_S2D(1); break;
    case 2: COCLR_PACK_S2D(2); break;
    case 3: COCLR_PACK_S2D(3); break;
    default: COCLR_PACK_S2D(4); break;
  }
#undef COCLR_PACK_S2D
  return LAUNCH_OK();
}

extern "C" int coclr_l2norm_fwd(const float* z, const float* bias, float* q, float* inv_norm, int B, int D,
                                coclr_stream_t stream) {
  if (!z || !q) return COCLR_E_ARG;
  l2norm_fwd_kernel<<<(B + 3) / 4, 128, 0, (cudaStream_t)stream>>>(z, bias, q, inv_norm, B, D);
  return LAUNCH_OK();
}
extern "C" int coclr_l2norm_bwd(const float* q, const float* dq, const float* inv_norm, float* dz, float* dbias, int B,
                                int D, coclr_stream_t stream) {
  if (!q || !dq || !inv_norm || !dz) return COCLR_E_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  l2norm_bwd_kernel<<<(B + 3) / 4, 128, 0, s>>>(q, dq, inv_norm, dz, B, D);
  if (dbias) colsum_small_kernel<<<(D + 127) / 128, 128, 0, s>>>(dz, dbias, B, D);
  return LAUNCH_OK();
}

extern "C" int coclr_ema_update(float* k, const float* q, float m, float one_minus_m, long n, int num_sms,
                                coclr_stream_t stream) {
  if (!k || !q || n < 0) return COCLR_E_ARG;
  if (((uintptr_t)k | (uintptr_t)q) & 15) return COCLR_E_ARG;
  ema_kernel<<<grid_for(n / 4 + 1, 256, num_sms * 8), 256, 0, (cudaStream_t)stream>>>(k, q, m, one_minus_m, n);
  return LAUNCH_OK();
}

extern "C" int coclr_queue_enqueue(float* queue, const float* keys, int dim, int K, int ptr, int n,
                                   coclr_stream_t stream) {
  if (!queue || !keys || ptr < 0 || ptr + n > K) return COCLR_E_ARG;
  enqueue_kernel<<<(dim * n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(queue, keys, dim, K, ptr, n);
  return LAUNCH_OK();
}

extern "C" int coclr_adam_step(const coclr_adam_t* p, int num_sms, coclr_stream_t stream) {
  if (!p || !p->param || !p->grad || !p->exp_avg || !p->exp_avg_sq) return COCLR_E_ARG;
  adam_kernel<<<grid_for(p->n, 256, num_sms * 8), 256, 0, (cudaStream_t)stream>>>(*p);
  return LAUNCH_OK();
}
