// HBM-bound row kernels of the CDML hot path: gather, normalise+cast, hinge loss fwd/bwd, bias-gradient
// column sums, split-K reduction, TF1 Adam, pair distances.  One warp per row wherever a row is the unit.
#include <algorithm>
#include "../../include/cdml.h"
#include "ctx.cuh"

namespace cdml {

constexpr int kWarpsPerBlock = 8;
constexpr int kRowThreads = kWarpsPerBlock * 32;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

static inline int row_grid(cdml_ctx* ctx, int64_t rows) {
  const int64_t blocks = (rows + kWarpsPerBlock - 1) / kWarpsPerBlock;
  const int64_t cap = static_cast<int64_t>(ctx->num_sms) * 8;  // 8 resident 256-thread CTAs per SM
  return static_cast<int>(blocks < cap ? (blocks > 0 ? blocks : 1) : cap);
}

// ------------------------------------------------------------------------------------------------
// K1 gather: out[i,:] = table[idx[i],:]   (inputs.py:158)
// ------------------------------------------------------------------------------------------------
template <typename IdxT, typename VecT>
__global__ void __launch_bounds__(kRowThreads)
gather_rows_kernel(const uint8_t* __restrict__ table, int64_t num_rows, int64_t row_bytes, int64_t pitch,
                   const IdxT* __restrict__ idx, int64_t n, uint8_t* __restrict__ out, int64_t out_pitch,
                   int32_t* flags) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t nvec = row_bytes / static_cast<int64_t>(sizeof(VecT));
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * kWarpsPerBlock + warp; r < n;
       r += static_cast<int64_t>(gridDim.x) * kWarpsPerBlock) {
    int64_t g = static_cast<int64_t>(idx[r]);
    if (g < 0) g += num_rows;  // numpy wrap-around
    VecT* dst = reinterpret_cast<VecT*>(out + r * out_pitch);
    if (g < 0 || g >= num_rows) {
      if (lane == 0) atomicOr(flags, 1);
      VecT z;
      memset(&z, 0, sizeof(VecT));
      for (int64_t v = lane; v < nvec; v += 32) dst[v] = z;
      continue;
    }
    const VecT* src = reinterpret_cast<const VecT*>(table + g * pitch);
    int64_t v = lane;
    for (; v + 96 < nvec; v += 128) {  // 4 independent loads in flight per lane
      const VecT t0 = __ldg(src + v), t1 = __ldg(src + v + 32), t2 = __ldg(src + v + 64), t3 = __ldg(src + v + 96);
      dst[v] = t0, dst[v + 32] = t1, dst[v + 64] = t2, dst[v + 96] = t3;
    }
    for (; v < nvec; v += 32) dst[v] = __ldg(src + v);
  }
}

// ------------------------------------------------------------------------------------------------
// K2 normalise + cast
// ------------------------------------------------------------------------------------------------
template <int kBf16>
__global__ void __launch_bounds__(kRowThreads)
rows_normalize_cast_kernel(const float* __restrict__ in, int64_t n, int64_t F, int64_t ld_in, int normalize, float eps,
                           uint16_t* __restrict__ out16, int64_t ld_out, float* __restrict__ out32, int64_t ld_out32,
                           float* __restrict__ sumsq) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * kWarpsPerBlock + warp; r < n;
       r += static_cast<int64_t>(gridDim.x) * kWarpsPerBlock) {
    const float* x = in + r * ld_in;
    float scale = 1.f, norm = 1.f;
    if (normalize != 0) {
      float ss = 0.f;
      for (int64_t j = lane; j < F; j += 32) {
        const float v = __ldg(x + j);
        ss = fmaf(v, v, ss);
      }
      ss = warp_sum(ss);
      scale = rsqrtf(fmaxf(ss, eps));  // TF: x * rsqrt(max(sum x^2, eps))
      norm = sqrtf(ss);                // numpy: x / ||x||
    }
    float ss16 = 0.f;
    uint16_t* o = out16 != nullptr ? out16 + r * ld_out : nullptr;
    float* o32 = out32 != nullptr ? out32 + r * ld_out32 : nullptr;
    const int64_t width = o != nullptr ? ld_out : F;
    for (int64_t j = 2 * lane; j < width; j += 64) {
      float v0 = 0.f, v1 = 0.f;
      if (j < F) v0 = normalize == 2 ? __ldg(x + j) / norm : __ldg(x + j) * scale;
      if (j + 1 < F) v1 = normalize == 2 ? __ldg(x + j + 1) / norm : __ldg(x + j + 1) * scale;
      if (o32 != nullptr) {
        if (j < F) o32[j] = v0;
        if (j + 1 < F) o32[j + 1] = v1;
      }
      if (o != nullptr) {
        const uint32_t pk = pack2<kBf16>(v0, v1);
        const float2 back = unpack2<kBf16>(pk);
        ss16 = fmaf(back.x, back.x, ss16);
        ss16 = fmaf(back.y, back.y, ss16);
        if (j + 1 < ld_out) *reinterpret_cast<uint32_t*>(o + j) = pk;
        else o[j] = static_cast<uint16_t>(pk);
      }
    }
    if (sumsq != nullptr) {
      ss16 = warp_sum(ss16);
      if (lane == 0) sumsq[r] = ss16;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// K5 hinge loss (losses.py:33-38) + gradient
// ------------------------------------------------------------------------------------------------
// With mined negatives (kMined) several triplets may pick the same negative row, whose gradient is then a sum over those
// triplets.  Float atomics would make that sum depend on the order the triplets arrive in, so a training step would not
// be reproducible.  Instead each row's sum of (a - n) is accumulated in 64-bit fixed point -- integer adds are
// associative -- and added to the row once:
//   hinge_triplet_kernel<true>  plain stores of the anchor / positive rows (each owned by one triplet), zero rows 3i+2;
//                               per active triplet: claim the lowest triplet index as the negative row's accumulator
//                               slot, and the row's largest |a - n| (it fixes the row's fixed-point scale)
//   hinge_neg_accum_kernel      integer atomics of round((a - n) * 2^k) into the slot's D accumulators
//   hinge_neg_apply_kernel      per slot: G[n] += s * sum * 2^-k
// k is chosen per row so that at most 2^log2B terms of magnitude <= the row's largest |a - n| stay below 2^62.
// Non-finite inputs: a triplet whose distances are NaN has h = fmaxf(NaN, 0) = 0, is inactive and adds nothing to its
// negative row (its own anchor / positive rows still get 0 * NaN = NaN).  A row that receives a non-finite a - n from an
// active triplet becomes NaN in every element, where a float sum would give +-inf or NaN in the affected elements only.
// Either way the optimizer step that follows turns those weights into NaN.
struct MinedScratch {
  uint32_t* slot_inv;      // [3B] ~(lowest active triplet that picked the row); 0 = none
  uint32_t* row_max;       // [3B] bits of the row's largest |a - n| (non-negative floats order as integers; NaN wins)
  long long* acc;          // [B, D] fixed-point sums, indexed by slot
};

__device__ __forceinline__ int mined_scale(float m, int log2B) {
  int e;
  frexpf(m, &e);           // m < 2^e
  return 62 - log2B - e;
}

template <bool kMined>
__global__ void __launch_bounds__(kRowThreads)
hinge_triplet_kernel(const float* __restrict__ E, int64_t B, int D, int64_t ld, const int32_t* __restrict__ neg_row,
                     float margin, float gscale, float* __restrict__ pos_dist, float* __restrict__ neg_dist,
                     float* __restrict__ hinge, float* __restrict__ G, MinedScratch ms) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * kWarpsPerBlock + warp; i < B;
       i += static_cast<int64_t>(gridDim.x) * kWarpsPerBlock) {
    const int64_t ra = 3 * i, rp = 3 * i + 1;
    const int64_t rn = neg_row != nullptr ? static_cast<int64_t>(neg_row[i]) : 3 * i + 2;
    const float* a = E + ra * ld;
    const float* p = E + rp * ld;
    const float* ng = E + rn * ld;
    float sp = 0.f, sn = 0.f;
    for (int j = lane; j < D; j += 32) {
      const float av = a[j], dp = av - p[j], dn = av - ng[j];
      sp = fmaf(dp, dp, sp);
      sn = fmaf(dn, dn, sn);
    }
    sp = warp_sum(sp);
    sn = warp_sum(sn);
    const float h = fmaxf(sp - sn + margin, 0.f);
    if (lane == 0) {
      if (pos_dist != nullptr) pos_dist[i] = sp;
      if (neg_dist != nullptr) neg_dist[i] = sn;
      hinge[i] = h;
    }
    if (G != nullptr) {
      const float s = h > 0.f ? 2.f * gscale : 0.f;
      if (kMined) {
        uint32_t mx = 0u;
        for (int j = lane; j < static_cast<int>(ld); j += 32) {
          float ga = 0.f, gp = 0.f;
          if (j < D) {
            const float av = a[j], pv = p[j], nv = ng[j];
            ga = s * (nv - pv), gp = s * (pv - av);
            mx = max(mx, __float_as_uint(fabsf(av - nv)));
          }
          G[ra * ld + j] = ga, G[rp * ld + j] = gp, G[(3 * i + 2) * ld + j] = 0.f;
        }
        mx = __reduce_max_sync(0xffffffffu, mx);
        if (h > 0.f) {
          long long* acc = ms.acc + i * D;
          for (int j = lane; j < D; j += 32) acc[j] = 0;
          if (lane == 0) {
            atomicMax(ms.slot_inv + rn, ~static_cast<uint32_t>(i));
            atomicMax(ms.row_max + rn, mx);
          }
        }
      } else {
        for (int j = lane; j < D; j += 32) {
          const float av = a[j], pv = p[j], nv = ng[j];
          G[ra * ld + j] = s * (nv - pv), G[rp * ld + j] = s * (pv - av), G[rn * ld + j] = s * (av - nv);
        }
      }
    }
  }
}

__global__ void __launch_bounds__(kRowThreads)
hinge_neg_accum_kernel(const float* __restrict__ E, int64_t B, int D, int64_t ld, const int32_t* __restrict__ neg_row,
                       const float* __restrict__ hinge, MinedScratch ms, int log2B) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * kWarpsPerBlock + warp; i < B;
       i += static_cast<int64_t>(gridDim.x) * kWarpsPerBlock) {
    if (!(hinge[i] > 0.f)) continue;
    const int64_t rn = neg_row[i];
    const float m = __uint_as_float(ms.row_max[rn]);
    if (!(m > 0.f) || !isfinite(m)) continue;              // all zero: nothing to add; not finite: the apply pass writes NaN
    const int k = mined_scale(m, log2B);
    unsigned long long* acc = reinterpret_cast<unsigned long long*>(ms.acc + static_cast<int64_t>(~ms.slot_inv[rn]) * D);
    const float* a = E + 3 * i * ld;
    const float* ng = E + rn * ld;
    for (int j = lane; j < D; j += 32)
      atomicAdd(acc + j, static_cast<unsigned long long>(__float2ll_rn(scalbnf(a[j] - ng[j], k))));
  }
}

__global__ void __launch_bounds__(kRowThreads)
hinge_neg_apply_kernel(int64_t B, int D, int64_t ld, const int32_t* __restrict__ neg_row, const float* __restrict__ hinge,
                       float gscale, MinedScratch ms, int log2B, float* __restrict__ G) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * kWarpsPerBlock + warp; i < B;
       i += static_cast<int64_t>(gridDim.x) * kWarpsPerBlock) {
    if (!(hinge[i] > 0.f)) continue;
    const int64_t rn = neg_row[i];
    if (~ms.slot_inv[rn] != static_cast<uint32_t>(i)) continue;    // one triplet per negative row applies the sum
    const float m = __uint_as_float(ms.row_max[rn]);
    if (m == 0.f) continue;
    const float s = 2.f * gscale;
    float* g = G + rn * ld;
    if (!isfinite(m)) {
      for (int j = lane; j < D; j += 32) g[j] += s * __int_as_float(0x7fc00000);
      continue;
    }
    const int k = mined_scale(m, log2B);
    const long long* acc = ms.acc + i * D;
    for (int j = lane; j < D; j += 32) g[j] += s * scalbnf(__ll2float_rn(acc[j]), -k);
  }
}

// dz = (g - e (e.g)) * rinv * leaky'(e): backward of the output L2-norm and the last leaky-ReLU, per row.
template <int kBf16>
__global__ void __launch_bounds__(kRowThreads)
l2norm_leaky_bwd_kernel(const float* __restrict__ E, const float* __restrict__ G, int64_t R, int D, int64_t ld,
                        const float* __restrict__ rinv, float alpha, uint16_t* __restrict__ dz, int64_t ld_dz) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * kWarpsPerBlock + warp; r < R;
       r += static_cast<int64_t>(gridDim.x) * kWarpsPerBlock) {
    const float* e = E + r * ld;
    const float* g = G + r * ld;
    float dot = 0.f;
    for (int j = lane; j < D; j += 32) dot = fmaf(e[j], g[j], dot);
    dot = warp_sum(dot);
    const float ri = rinv[r];
    uint16_t* o = dz + r * ld_dz;
    for (int j = 2 * lane; j < D; j += 64) {
      const float e0 = e[j], v0 = (g[j] - e0 * dot) * ri * (e0 > 0.f ? 1.f : alpha);
      float v1 = 0.f;
      if (j + 1 < D) {
        const float e1 = e[j + 1];
        v1 = (g[j + 1] - e1 * dot) * ri * (e1 > 0.f ? 1.f : alpha);
      }
      const uint32_t pk = pack2<kBf16>(v0, v1);
      if (j + 1 < D) *reinterpret_cast<uint32_t*>(o + j) = pk;
      else o[j] = static_cast<uint16_t>(pk);
    }
  }
}

// Deterministic single-block reduction: stats = {mean hinge, mean pos, mean neg, #active}.
__global__ void __launch_bounds__(1024)
hinge_stats_kernel(const float* __restrict__ hinge, const float* __restrict__ pos, const float* __restrict__ neg,
                   int64_t B, float* __restrict__ stats) {
  __shared__ float sh[4][32];
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  for (int64_t i = threadIdx.x; i < B; i += blockDim.x) {
    const float h = hinge[i];
    s0 += h;
    s3 += h > 0.f ? 1.f : 0.f;
    if (pos != nullptr) s1 += pos[i];
    if (neg != nullptr) s2 += neg[i];
  }
  s0 = warp_sum(s0), s1 = warp_sum(s1), s2 = warp_sum(s2), s3 = warp_sum(s3);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) sh[0][warp] = s0, sh[1][warp] = s1, sh[2][warp] = s2, sh[3][warp] = s3;
  __syncthreads();
  if (warp == 0) {
    float t0 = sh[0][lane], t1 = sh[1][lane], t2 = sh[2][lane], t3 = sh[3][lane];
    t0 = warp_sum(t0), t1 = warp_sum(t1), t2 = warp_sum(t2), t3 = warp_sum(t3);
    if (lane == 0) {
      const float inv = 1.0f / static_cast<float>(B);
      stats[0] = t0 * inv, stats[1] = t1 * inv, stats[2] = t2 * inv, stats[3] = t3;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// bias gradient: column sums of a 16-bit matrix, two fixed-order stages
// ------------------------------------------------------------------------------------------------
constexpr int kColStrip = 64;
template <int kBf16>
__global__ void __launch_bounds__(kRowThreads)
colsum16_stage1(const uint16_t* __restrict__ X, int64_t R, int64_t N, int64_t ld, int64_t rows_per_chunk,
                float* __restrict__ partial) {
  __shared__ float sh[kWarpsPerBlock][kColStrip];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t c0 = static_cast<int64_t>(blockIdx.x) * kColStrip + 2 * lane;
  const int64_t r0 = static_cast<int64_t>(blockIdx.y) * rows_per_chunk;
  const int64_t r1 = r0 + rows_per_chunk < R ? r0 + rows_per_chunk : R;
  float a0 = 0.f, a1 = 0.f;
  if (c0 < N) {
    const bool pair = c0 + 1 < N;
    for (int64_t r = r0 + warp; r < r1; r += kWarpsPerBlock) {
      const uint16_t* p = X + r * ld + c0;
      if (pair) {
        const float2 f = unpack2<kBf16>(*reinterpret_cast<const uint32_t*>(p));
        a0 += f.x, a1 += f.y;
      } else {
        a0 += unpack2<kBf16>(static_cast<uint32_t>(*p)).x;
      }
    }
  }
  sh[warp][2 * lane] = a0, sh[warp][2 * lane + 1] = a1;
  __syncthreads();
  if (threadIdx.x < kColStrip) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kWarpsPerBlock; ++w) t += sh[w][threadIdx.x];
    const int64_t c = static_cast<int64_t>(blockIdx.x) * kColStrip + threadIdx.x;
    if (c < N) partial[static_cast<int64_t>(blockIdx.y) * N + c] = t;
  }
}

// Vectorised variant: each lane owns 8 consecutive columns (one 16-byte load per row), a warp covers 256 columns,
// the 8 warps of the block stride the rows of the chunk.  Needs ld % 8 == 0 and a 16-byte aligned base.
constexpr int kColStripV = 256;
template <int kBf16>
__global__ void __launch_bounds__(kRowThreads)
colsum16_stage1_vec(const uint16_t* __restrict__ X, int64_t R, int64_t N, int64_t ld, int64_t rows_per_chunk,
                    float* __restrict__ partial) {
  __shared__ float sh[kWarpsPerBlock][kColStripV];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t c0 = static_cast<int64_t>(blockIdx.x) * kColStripV + 8 * lane;
  const int64_t r0 = static_cast<int64_t>(blockIdx.y) * rows_per_chunk;
  const int64_t r1 = r0 + rows_per_chunk < R ? r0 + rows_per_chunk : R;
  float a[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) a[j] = 0.f;
  if (c0 + 8 <= N) {
    int64_t r = r0 + warp;
    for (; r + 3 * kWarpsPerBlock < r1; r += 4 * kWarpsPerBlock) {   // 4 independent 16-byte loads in flight
      uint4 t[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) t[u] = __ldg(reinterpret_cast<const uint4*>(X + (r + u * kWarpsPerBlock) * ld + c0));
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float2 f0 = unpack2<kBf16>(t[u].x), f1 = unpack2<kBf16>(t[u].y), f2 = unpack2<kBf16>(t[u].z),
                     f3 = unpack2<kBf16>(t[u].w);
        a[0] += f0.x, a[1] += f0.y, a[2] += f1.x, a[3] += f1.y, a[4] += f2.x, a[5] += f2.y, a[6] += f3.x, a[7] += f3.y;
      }
    }
    for (; r < r1; r += kWarpsPerBlock) {
      const uint4 t = __ldg(reinterpret_cast<const uint4*>(X + r * ld + c0));
      const float2 f0 = unpack2<kBf16>(t.x), f1 = unpack2<kBf16>(t.y), f2 = unpack2<kBf16>(t.z), f3 = unpack2<kBf16>(t.w);
      a[0] += f0.x, a[1] += f0.y, a[2] += f1.x, a[3] += f1.y, a[4] += f2.x, a[5] += f2.y, a[6] += f3.x, a[7] += f3.y;
    }
  } else {
    for (int j = 0; j < 8; ++j)
      if (c0 + j < N)
        for (int64_t r = r0 + warp; r < r1; r += kWarpsPerBlock) a[j] += unpack2<kBf16>(static_cast<uint32_t>(X[r * ld + c0 + j])).x;
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) sh[warp][8 * lane + j] = a[j];
  __syncthreads();
  {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kWarpsPerBlock; ++w) t += sh[w][threadIdx.x];
    const int64_t c = static_cast<int64_t>(blockIdx.x) * kColStripV + threadIdx.x;
    if (c < N) partial[static_cast<int64_t>(blockIdx.y) * N + c] = t;
  }
}

__global__ void sum_partials_kernel(const float* __restrict__ parts, int num_parts, int64_t stride, int64_t n,
                                    float scale, float* __restrict__ out) {
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float t = 0.f;
    for (int s = 0; s < num_parts; ++s) t += parts[s * stride + i];
    out[i] = t * scale;
  }
}

__global__ void sum_partials_vec4_kernel(const float4* __restrict__ parts, int num_parts, int64_t stride4, int64_t n4,
                                         float scale, float4* __restrict__ out) {
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int s = 0; s < num_parts; ++s) {
      const float4 v = __ldg(parts + s * stride4 + i);
      t.x += v.x, t.y += v.y, t.z += v.z, t.w += v.w;
    }
    out[i] = make_float4(t.x * scale, t.y * scale, t.z * scale, t.w * scale);
  }
}

// ------------------------------------------------------------------------------------------------
// K8 TF1 Adam
// ------------------------------------------------------------------------------------------------
__global__ void adam_prepare_kernel(int64_t* step, float base_lr, float decay_steps, float decay_rate, int staircase,
                                    float beta1, float beta2, float* scalars) {
  const int64_t gs = *step;  // global_step before this update (train.py:108-113 reads it pre-increment)
  const double t = static_cast<double>(gs + 1);
  double p = static_cast<double>(gs) / static_cast<double>(decay_steps);
  if (staircase) p = floor(p);
  const double lr = static_cast<double>(base_lr) * pow(static_cast<double>(decay_rate), p);
  const double lr_t = lr * sqrt(1.0 - pow(static_cast<double>(beta2), t)) / (1.0 - pow(static_cast<double>(beta1), t));
  scalars[0] = static_cast<float>(lr_t);
  scalars[1] = static_cast<float>(lr);
  scalars[2] = static_cast<float>(t);
  scalars[3] = 0.f;
  *step = gs + 1;
}

template <int kBf16>
__global__ void adam_apply_kernel(float* __restrict__ w, float* __restrict__ m, float* __restrict__ v,
                                  const float* __restrict__ g, int64_t n, const float* __restrict__ scalars,
                                  float beta1, float beta2, float eps, float gscale, uint16_t* __restrict__ w16) {
  const float lr_t = scalars[0];
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const float gi = g[i] * gscale;
    const float mi = beta1 * m[i] + (1.f - beta1) * gi;
    const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;
    const float wi = w[i] - lr_t * mi / (sqrtf(vi) + eps);
    m[i] = mi, v[i] = vi, w[i] = wi;
    if (w16 != nullptr) w16[i] = static_cast<uint16_t>(pack2<kBf16>(wi, 0.f));
  }
}

__global__ void fill_column16_kernel(uint16_t* __restrict__ X, int64_t rows, int64_t ld, int64_t col, uint16_t bits) {
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < rows;
       r += static_cast<int64_t>(gridDim.x) * blockDim.x)
    X[r * ld + col] = bits;
}

template <int kBf16>
__global__ void cast16_kernel(const float* __restrict__ in, int64_t n, uint16_t* __restrict__ out) {
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x)
    out[i] = static_cast<uint16_t>(pack2<kBf16>(in[i], 0.f));
}

// ------------------------------------------------------------------------------------------------
// evaluate.mean_dist
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kRowThreads)
pair_dist_kernel(const float* __restrict__ V, int64_t ld, int D, const int64_t* __restrict__ pairs, int64_t P,
                 float* __restrict__ dist) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * kWarpsPerBlock + warp; i < P;
       i += static_cast<int64_t>(gridDim.x) * kWarpsPerBlock) {
    const float* a = V + pairs[2 * i] * ld;
    const float* b = V + pairs[2 * i + 1] * ld;
    float s = 0.f;
    for (int j = lane; j < D; j += 32) {
      const float d = a[j] - b[j];
      s = fmaf(d, d, s);
    }
    s = warp_sum(s);
    if (lane == 0) dist[i] = s;
  }
}

// ------------------------------------------------------------------------------------------------
// Gradient post-processing + the other optimizers of build_graph (train.py:115-146):
//   g_eff = grad_scale * g + wd_reg * w                      (mean gradient + regularization_penalty * d reg / dw)
//   clip_by_norm per variable (train.py:47-64):  g_eff *= clip / max(||g_eff||, clip)
//   kind 0 Adam | 1 Momentum(0.9, nesterov) (train.py:115-116) | 2 LARS (tf.contrib.opt.LARSOptimizer, train.py:354)
//        | 3 plain gradient descent
// Norms come from opt_sumsq (fixed-order two-stage reduction -> deterministic).
// ------------------------------------------------------------------------------------------------
constexpr int kSumsqBlocks = 592;   // 148 SMs x 4

__global__ void __launch_bounds__(256)
opt_sumsq_stage1_kernel(const float* __restrict__ g, const float* __restrict__ w, int64_t n, float gscale, float wd_reg,
                        float* __restrict__ partial) {
  __shared__ float sh[2][8];
  float a = 0.f, b = 0.f;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const float wi = w[i];
    const float ge = fmaf(wd_reg, wi, g[i] * gscale);
    a = fmaf(ge, ge, a), b = fmaf(wi, wi, b);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o), b += __shfl_xor_sync(0xffffffffu, b, o);
  if ((threadIdx.x & 31) == 0) sh[0][threadIdx.x >> 5] = a, sh[1][threadIdx.x >> 5] = b;
  __syncthreads();
  if (threadIdx.x == 0) {
    float ta = 0.f, tb = 0.f;
    for (int i = 0; i < 8; ++i) ta += sh[0][i], tb += sh[1][i];
    partial[2 * blockIdx.x] = ta, partial[2 * blockIdx.x + 1] = tb;
  }
}

__global__ void opt_sumsq_stage2_kernel(const float* __restrict__ partial, int nblocks, float* __restrict__ out2) {
  if (threadIdx.x < 2) {
    double t = 0.0;
    for (int i = 0; i < nblocks; ++i) t += static_cast<double>(partial[2 * i + threadIdx.x]);
    out2[threadIdx.x] = static_cast<float>(t);
  }
}

template <int kBf16>
__global__ void opt_apply_kernel(int kind, float* __restrict__ w, float* __restrict__ m, float* __restrict__ v,
                                 const float* __restrict__ g, int64_t n, const float* __restrict__ scalars,
                                 const float* __restrict__ norms, float beta1, float beta2, float eps, float gscale,
                                 float wd_reg, float clip, float momentum, float lars_wd, float lars_eeta,
                                 uint16_t* __restrict__ w16) {
  const float lr_t = scalars[0], lr = scalars[1];
  float coef = 1.f, trust = 1.f;
  if (clip > 0.f) coef = clip / fmaxf(sqrtf(norms[0]), clip);
  if (kind == 2) {
    const float wn = sqrtf(norms[1]);
    const float gn = sqrtf(norms[0]) * coef;          // norm of the (clipped) gradient handed to the optimizer
    trust = (wn > 0.f && gn > 0.f) ? lars_eeta * wn / (gn + lars_wd * wn + eps) : 1.f;
  }
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float wi = w[i];
    const float gi = fmaf(wd_reg, wi, g[i] * gscale) * coef;
    if (kind == 0) {
      const float mi = beta1 * m[i] + (1.f - beta1) * gi;
      const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;
      wi -= lr_t * mi / (sqrtf(vi) + eps);
      m[i] = mi, v[i] = vi;
    } else if (kind == 1) {                              // ApplyMomentum, use_nesterov
      const float acc = momentum * m[i] + gi;
      wi -= lr * gi + lr * momentum * acc;
      m[i] = acc;
    } else if (kind == 2) {   // LARS as of TF r1.13 (_apply_dense -> apply_momentum(var, mom, lr*trust, grad, momentum)): weight
      const float acc = momentum * m[i] + gi;   // decay enters the trust ratio ONLY; the later "grad + wd*var" form is not 1.13's
      wi -= lr * trust * acc;
      m[i] = acc;
    } else {
      wi -= lr * gi;
    }
    w[i] = wi;
    if (w16 != nullptr) w16[i] = static_cast<uint16_t>(pack2<kBf16>(wi, 0.f));
  }
}

// ------------------------------------------------------------------------------------------------
// Fusion towers (models.py:65-157): 256-wide elementwise joins of 16-bit activations and the output L2-norm of a
// tensor that is not a GEMM output.  op: 0 a*b | 1 a+b | 2 a*b+a+b | 3 a*leaky'(b) | 4 a*b+a | 5 a*b+c | 6 (a*b+a)*leaky'(c)
// | 7 a*b*leaky'(c);  leaky'(t) = t > 0 ? 1 : alpha.  fp32 math, 16-bit in / out.
// ------------------------------------------------------------------------------------------------
template <int kOp>
__device__ __forceinline__ float ew_apply(float x, float y, float z, float alpha) {
  if constexpr (kOp == 0) return x * y;
  else if constexpr (kOp == 1) return x + y;
  else if constexpr (kOp == 2) return fmaf(x, y, x + y);
  else if constexpr (kOp == 3) return x * (y > 0.f ? 1.f : alpha);
  else if constexpr (kOp == 4) return fmaf(x, y, x);
  else if constexpr (kOp == 5) return fmaf(x, y, z);
  else if constexpr (kOp == 6) return fmaf(x, y, x) * (z > 0.f ? 1.f : alpha);
  else return x * y * (z > 0.f ? 1.f : alpha);
}

// kVec = 8: one 16-byte piece per operand per thread (cols, pitches multiples of 8, 16-byte aligned bases); kVec = 2 otherwise.
template <int kBf16, int kOp, int kVec>
__global__ void __launch_bounds__(256)
ew16_kernel(const uint16_t* __restrict__ a, int64_t lda, const uint16_t* __restrict__ b, int64_t ldb,
            const uint16_t* __restrict__ c, int64_t ldc, uint16_t* __restrict__ out, int64_t ldo, int64_t rows, int cols,
            float alpha) {
  constexpr int kWords = kVec / 2;
  const int per_row = cols / kVec;
  const int64_t total = rows * per_row;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t r = i / per_row;
    const int j = static_cast<int>(i - r * per_row) * kVec;
    uint32_t xa[kWords], xb[kWords], xc[kWords], xo[kWords];
    if constexpr (kVec == 8) {
      const uint4 va = *reinterpret_cast<const uint4*>(a + r * lda + j);
      const uint4 vb = *reinterpret_cast<const uint4*>(b + r * ldb + j);
      xa[0] = va.x, xa[1] = va.y, xa[2] = va.z, xa[3] = va.w;
      xb[0] = vb.x, xb[1] = vb.y, xb[2] = vb.z, xb[3] = vb.w;
      if constexpr (kOp >= 5) {
        const uint4 vc = *reinterpret_cast<const uint4*>(c + r * ldc + j);
        xc[0] = vc.x, xc[1] = vc.y, xc[2] = vc.z, xc[3] = vc.w;
      }
    } else {
      xa[0] = *reinterpret_cast<const uint32_t*>(a + r * lda + j);
      xb[0] = *reinterpret_cast<const uint32_t*>(b + r * ldb + j);
      if constexpr (kOp >= 5) xc[0] = *reinterpret_cast<const uint32_t*>(c + r * ldc + j);
    }
#pragma unroll
    for (int w = 0; w < kWords; ++w) {
      const float2 x = unpack2<kBf16>(xa[w]), y = unpack2<kBf16>(xb[w]);
      float2 z = make_float2(0.f, 0.f);
      if constexpr (kOp >= 5) z = unpack2<kBf16>(xc[w]);
      xo[w] = pack2<kBf16>(ew_apply<kOp>(x.x, y.x, z.x, alpha), ew_apply<kOp>(x.y, y.y, z.y, alpha));
    }
    if constexpr (kVec == 8) *reinterpret_cast<uint4*>(out + r * ldo + j) = make_uint4(xo[0], xo[1], xo[2], xo[3]);
    else *reinterpret_cast<uint32_t*>(out + r * ldo + j) = xo[0];
  }
}

// e = y * rsqrt(max(sum y^2, eps)) for 16-bit rows y (tf.nn.l2_normalize, models.py:90/:121/:156): fp32 e, rinv, 16-bit e.
template <int kBf16>
__global__ void __launch_bounds__(kRowThreads)
rows_l2norm16_kernel(const uint16_t* __restrict__ y, int64_t n, int D, int64_t ld_y, float eps, float* __restrict__ e,
                     int64_t ld_e, float* __restrict__ rinv, uint16_t* __restrict__ e16, int64_t ld_e16) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * kWarpsPerBlock + warp; r < n;
       r += static_cast<int64_t>(gridDim.x) * kWarpsPerBlock) {
    const uint16_t* yr = y + r * ld_y;
    float ss = 0.f;
    for (int j = 2 * lane; j < D; j += 64) {
      const float2 v = unpack2<kBf16>(*reinterpret_cast<const uint32_t*>(yr + j));
      ss = fmaf(v.x, v.x, fmaf(v.y, v.y, ss));
    }
    ss = warp_sum(ss);
    const float s = rsqrtf(fmaxf(ss, eps));
    if (lane == 0 && rinv != nullptr) rinv[r] = s;
    for (int j = 2 * lane; j < D; j += 64) {
      const float2 v = unpack2<kBf16>(*reinterpret_cast<const uint32_t*>(yr + j));
      *reinterpret_cast<float2*>(e + r * ld_e + j) = make_float2(v.x * s, v.y * s);
      if (e16 != nullptr) *reinterpret_cast<uint32_t*>(e16 + r * ld_e16 + j) = pack2<kBf16>(v.x * s, v.y * s);
    }
  }
}

static inline int flat_grid(cdml_ctx* ctx, int64_t n, int threads) {
  const int64_t blocks = (n + threads - 1) / threads;
  const int64_t cap = static_cast<int64_t>(ctx->num_sms) * 8;
  return static_cast<int>(blocks < cap ? (blocks > 0 ? blocks : 1) : cap);
}

}  // namespace cdml

using namespace cdml;

extern "C" {

int cdml_gather_rows(cdml_ctx* ctx, const void* table, int64_t num_rows, int64_t row_bytes, int64_t table_pitch_bytes,
                     const void* idx, int idx_is_64, int64_t n_idx, void* out, int64_t out_pitch_bytes, void* stream) {
  CDML_REQUIRE(ctx && table && idx && out, "cdml_gather_rows: NULL argument");
  CDML_REQUIRE(num_rows > 0 && row_bytes > 0 && table_pitch_bytes >= row_bytes && out_pitch_bytes >= row_bytes,
               "cdml_gather_rows: bad geometry");
  if (n_idx == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = row_grid(ctx, n_idx);
  const uint8_t* t = static_cast<const uint8_t*>(table);
  uint8_t* o = static_cast<uint8_t*>(out);
  const uintptr_t align = reinterpret_cast<uintptr_t>(t) | reinterpret_cast<uintptr_t>(o) |
                          static_cast<uintptr_t>(row_bytes) | static_cast<uintptr_t>(table_pitch_bytes) |
                          static_cast<uintptr_t>(out_pitch_bytes);
#define CDML_GATHER(IDX, VEC)                                                                                      \
  gather_rows_kernel<IDX, VEC><<<grid, kRowThreads, 0, st>>>(t, num_rows, row_bytes, table_pitch_bytes,            \
                                                             static_cast<const IDX*>(idx), n_idx, o, out_pitch_bytes, \
                                                             ctx->dev_flags)
  if ((align & 15) == 0) {
    if (idx_is_64) CDML_GATHER(int64_t, uint4); else CDML_GATHER(int32_t, uint4);
  } else if ((align & 3) == 0) {
    if (idx_is_64) CDML_GATHER(int64_t, uint32_t); else CDML_GATHER(int32_t, uint32_t);
  } else {
    if (idx_is_64) CDML_GATHER(int64_t, uint8_t); else CDML_GATHER(int32_t, uint8_t);
  }
#undef CDML_GATHER
  CDML_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int cdml_rows_normalize_cast(cdml_ctx* ctx, const float* in, int64_t n, int64_t F, int64_t ld_in, int normalize,
                             float eps, void* out16, int64_t ld_out, int dtype16, float* out32, int64_t ld_out32,
                             float* sumsq, void* stream) {
  CDML_REQUIRE(ctx && in && (out16 || out32), "cdml_rows_normalize_cast: NULL argument");
  CDML_REQUIRE(F > 0 && ld_in >= F && (!out16 || (ld_out >= F && ld_out % 2 == 0)) && (!out32 || ld_out32 >= F),
               "cdml_rows_normalize_cast: bad geometry (F=%lld ld_in=%lld ld_out=%lld)", (long long)F, (long long)ld_in,
               (long long)ld_out);
  if (n == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = row_grid(ctx, n);
  if (dtype16 == CDML_BF16)
    rows_normalize_cast_kernel<1><<<grid, kRowThreads, 0, st>>>(in, n, F, ld_in, normalize, eps,
                                                                static_cast<uint16_t*>(out16), ld_out, out32, ld_out32, sumsq);
  else
    rows_normalize_cast_kernel<0><<<grid, kRowThreads, 0, st>>>(in, n, F, ld_in, normalize, eps,
                                                                static_cast<uint16_t*>(out16), ld_out, out32, ld_out32, sumsq);
  CDML_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int cdml_triplet_hinge(cdml_ctx* ctx, const float* E, int64_t B, int D, int64_t ld_e, const int32_t* neg_row,
                       float margin, float grad_scale, const float* rinv, float leaky_alpha, float* pos_dist,
                       float* neg_dist, float* hinge_dist, float* stats, float* dE, void* dz16, int64_t ld_dz,
                       int dtype16, float* workspace, void* stream) {
  CDML_REQUIRE(ctx && E && hinge_dist && stats, "cdml_triplet_hinge: E, hinge_dist and stats are required");
  CDML_REQUIRE(B > 0 && D > 0 && ld_e >= D, "cdml_triplet_hinge: bad geometry");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* G = dE;
  if (G == nullptr && dz16 != nullptr) {
    CDML_REQUIRE(workspace != nullptr, "cdml_triplet_hinge: workspace needed when dz16 is requested without dE");
    G = workspace;
  }
  CDML_REQUIRE(dz16 == nullptr || (rinv != nullptr && ld_dz >= D && ld_dz % 2 == 0),
               "cdml_triplet_hinge: dz16 needs rinv and an even ld_dz >= D");
  const int grid = row_grid(ctx, B);
  if (neg_row != nullptr && G != nullptr) {
    CDML_REQUIRE(3 * B < (1ll << 31), "cdml_triplet_hinge: B=%lld too large for mined negatives", (long long)B);
    // scratch: slot_inv [3B] u32 | row_max [3B] u32 | acc [B, D] i64 (the first two zeroed by one memset)
    const size_t head = sizeof(uint32_t) * 6 * B;
    uint8_t* ws = static_cast<uint8_t*>(ctx_scratch(ctx, head + sizeof(long long) * B * D));
    if (ws == nullptr) return -2;
    MinedScratch ms{reinterpret_cast<uint32_t*>(ws), reinterpret_cast<uint32_t*>(ws) + 3 * B,
                    reinterpret_cast<long long*>(ws + head)};
    int log2B = 0;
    while ((1ll << log2B) < B) ++log2B;
    CDML_CHECK_CUDA(cudaMemsetAsync(ws, 0, head, st));
    hinge_triplet_kernel<true><<<grid, kRowThreads, 0, st>>>(E, B, D, ld_e, neg_row, margin, grad_scale, pos_dist,
                                                            neg_dist, hinge_dist, G, ms);
    CDML_CHECK_CUDA(cudaGetLastError());
    hinge_neg_accum_kernel<<<grid, kRowThreads, 0, st>>>(E, B, D, ld_e, neg_row, hinge_dist, ms, log2B);
    CDML_CHECK_CUDA(cudaGetLastError());
    hinge_neg_apply_kernel<<<grid, kRowThreads, 0, st>>>(B, D, ld_e, neg_row, hinge_dist, grad_scale, ms, log2B, G);
  } else {
    hinge_triplet_kernel<false><<<grid, kRowThreads, 0, st>>>(E, B, D, ld_e, neg_row, margin, grad_scale, pos_dist,
                                                             neg_dist, hinge_dist, G, MinedScratch{});
  }
  CDML_CHECK_CUDA(cudaGetLastError());
  hinge_stats_kernel<<<1, 1024, 0, st>>>(hinge_dist, pos_dist, neg_dist, B, stats);
  CDML_CHECK_CUDA(cudaGetLastError());
  if (dz16 != nullptr) {
    const int grid2 = row_grid(ctx, 3 * B);
    if (dtype16 == CDML_BF16)
      l2norm_leaky_bwd_kernel<1><<<grid2, kRowThreads, 0, st>>>(E, G, 3 * B, D, ld_e, rinv, leaky_alpha,
                                                               static_cast<uint16_t*>(dz16), ld_dz);
    else
      l2norm_leaky_bwd_kernel<0><<<grid2, kRowThreads, 0, st>>>(E, G, 3 * B, D, ld_e, rinv, leaky_alpha,
                                                               static_cast<uint16_t*>(dz16), ld_dz);
    CDML_CHECK_CUDA(cudaGetLastError());
  }
  return 0;
}

int64_t cdml_colsum_workspace_floats(int64_t R, int64_t N) {
  int64_t chunks = (R + 255) / 256;
  if (chunks > 128) chunks = 128;
  if (chunks < 1) chunks = 1;
  return chunks * N;
}

int cdml_colsum16(cdml_ctx* ctx, const void* X, int64_t R, int64_t N, int64_t ld, int dtype16, float* workspace,
                  float* out, void* stream) {
  CDML_REQUIRE(ctx && X && workspace && out, "cdml_colsum16: NULL argument");
  CDML_REQUIRE(R > 0 && N > 0 && ld >= N && ld % 2 == 0, "cdml_colsum16: bad geometry");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t chunks = cdml_colsum_workspace_floats(R, N) / N;
  const int64_t rows_per_chunk = (R + chunks - 1) / chunks;
  const uint16_t* x = static_cast<const uint16_t*>(X);
  if (ld % 8 == 0 && (reinterpret_cast<uintptr_t>(X) & 15) == 0) {
    dim3 grid(static_cast<unsigned>((N + kColStripV - 1) / kColStripV), static_cast<unsigned>(chunks));
    if (dtype16 == CDML_BF16) colsum16_stage1_vec<1><<<grid, kRowThreads, 0, st>>>(x, R, N, ld, rows_per_chunk, workspace);
    else colsum16_stage1_vec<0><<<grid, kRowThreads, 0, st>>>(x, R, N, ld, rows_per_chunk, workspace);
  } else {
    dim3 grid(static_cast<unsigned>((N + kColStrip - 1) / kColStrip), static_cast<unsigned>(chunks));
    if (dtype16 == CDML_BF16) colsum16_stage1<1><<<grid, kRowThreads, 0, st>>>(x, R, N, ld, rows_per_chunk, workspace);
    else colsum16_stage1<0><<<grid, kRowThreads, 0, st>>>(x, R, N, ld, rows_per_chunk, workspace);
  }
  CDML_CHECK_CUDA(cudaGetLastError());
  return cdml_sum_partials(ctx, workspace, static_cast<int>(chunks), N, N, 1.0f, out, stream);
}

int cdml_sum_partials(cdml_ctx* ctx, const float* parts, int num_parts, int64_t stride, int64_t n, float scale,
                      float* out, void* stream) {
  CDML_REQUIRE(ctx && parts && out && num_parts >= 1 && n >= 0, "cdml_sum_partials: bad argument");
  if (n == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool vec = ((reinterpret_cast<uintptr_t>(parts) | reinterpret_cast<uintptr_t>(out)) & 15) == 0 && stride % 4 == 0 &&
                   n % 4 == 0;
  if (vec)
    sum_partials_vec4_kernel<<<flat_grid(ctx, n / 4, 256), 256, 0, st>>>(reinterpret_cast<const float4*>(parts), num_parts,
                                                                         stride / 4, n / 4, scale,
                                                                         reinterpret_cast<float4*>(out));
  else
    sum_partials_kernel<<<flat_grid(ctx, n, 256), 256, 0, st>>>(parts, num_parts, stride, n, scale, out);
  CDML_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int cdml_adam_prepare(cdml_ctx* ctx, int64_t* step_counter, float base_lr, float decay_steps, float decay_rate,
                      int staircase, float beta1, float beta2, float* scalars, void* stream) {
  CDML_REQUIRE(ctx && step_counter && scalars, "cdml_adam_prepare: NULL argument");
  adam_prepare_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(step_counter, base_lr, decay_steps, decay_rate,
                                                                      staircase, beta1, beta2, scalars);
  CDML_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int cdml_adam_apply(cdml_ctx* ctx, float* w, float* m, float* v, const float* g, int64_t n, const float* scalars,
                    float beta1, float beta2, float eps, float grad_scale, void* w16, int dtype16, void* stream) {
  CDML_REQUIRE(ctx && w && m && v && g && scalars, "cdml_adam_apply: NULL argument");
  if (n == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = flat_grid(ctx, n, 256);
  if (dtype16 == CDML_BF16)
    adam_apply_kernel<1><<<grid, 256, 0, st>>>(w, m, v, g, n, scalars, beta1, beta2, eps, grad_scale,
                                               static_cast<uint16_t*>(w16));
  else
    adam_apply_kernel<0><<<grid, 256, 0, st>>>(w, m, v, g, n, scalars, beta1, beta2, eps, grad_scale,
                                               static_cast<uint16_t*>(w16));
  CDML_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int64_t cdml_opt_workspace_floats(void) { return 2 * kSumsqBlocks + 2; }

int cdml_opt_sumsq(cdml_ctx* ctx, const float* g, const float* w, int64_t n, float grad_scale, float wd_reg,
                   float* workspace, float* out2, void* stream) {
  CDML_REQUIRE(ctx && g && w && workspace && out2 && n >= 0, "cdml_opt_sumsq: bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int blocks = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, kSumsqBlocks)));
  opt_sumsq_stage1_kernel<<<blocks, 256, 0, st>>>(g, w, n, grad_scale, wd_reg, workspace);
  opt_sumsq_stage2_kernel<<<1, 32, 0, st>>>(workspace, blocks, out2);
  CDML_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int cdml_opt_apply(cdml_ctx* ctx, int kind, float* w, float* m, float* v, const float* g, int64_t n, const float* scalars,
                   const float* norms, float beta1, float beta2, float eps, float grad_scale, float wd_reg, float clip_norm,
                   float momentum, float lars_weight_decay, float lars_eeta, void* w16, int dtype16, void* stream) {
  CDML_REQUIRE(ctx && w && g && scalars && kind >= 0 && kind <= 3, "cdml_opt_apply: bad argument");
  CDML_REQUIRE(kind != 0 || (m && v), "cdml_opt_apply: Adam needs m and v");
  CDML_REQUIRE((kind != 1 && kind != 2) || m, "cdml_opt_apply: momentum optimizers need the accumulator m");
  CDML_REQUIRE((clip_norm <= 0.f && kind != 2) || norms, "cdml_opt_apply: clipping / LARS need the norms of cdml_opt_sumsq");
  if (n == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = flat_grid(ctx, n, 256);
  if (dtype16 == CDML_BF16)
    opt_apply_kernel<1><<<grid, 256, 0, st>>>(kind, w, m, v, g, n, scalars, norms, beta1, beta2, eps, grad_scale, wd_reg,
                                              clip_norm, momentum, lars_weight_decay, lars_eeta, static_cast<uint16_t*>(w16));
  else
    opt_apply_kernel<0><<<grid, 256, 0, st>>>(kind, w, m, v, g, n, scalars, norms, beta1, beta2, eps, grad_scale, wd_reg,
                                              clip_norm, momentum, lars_weight_decay, lars_eeta, static_cast<uint16_t*>(w16));
  CDML_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int cdml_ew16(cdml_ctx* ctx, int op, const void* a, int64_t lda, const void* b, int64_t ldb, const void* c, int64_t ldc,
              void* out, int64_t ldo, int64_t rows, int cols, float alpha, int dtype16, void* stream) {
  CDML_REQUIRE(ctx && a && b && out && rows >= 0 && cols > 0 && cols % 2 == 0, "cdml_ew16: bad argument");
  CDML_REQUIRE(op >= 0 && op <= 7, "cdml_ew16: unknown op %d", op);
  CDML_REQUIRE(op < 5 || c != nullptr, "cdml_ew16: op %d needs the third operand", op);
  CDML_REQUIRE(lda % 2 == 0 && ldb % 2 == 0 && ldo % 2 == 0 && (c == nullptr || ldc % 2 == 0), "cdml_ew16: odd row pitch");
  if (rows == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const uint16_t* pa = static_cast<const uint16_t*>(a);
  const uint16_t* pb = static_cast<const uint16_t*>(b);
  const uint16_t* pc = static_cast<const uint16_t*>(c);
  uint16_t* po = static_cast<uint16_t*>(out);
  const bool vec = cols % 8 == 0 && lda % 8 == 0 && ldb % 8 == 0 && ldo % 8 == 0 && (c == nullptr || ldc % 8 == 0) &&
                   ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(c) |
                     reinterpret_cast<uintptr_t>(out)) & 15) == 0;
  const int grid = flat_grid(ctx, rows * (cols / (vec ? 8 : 2)), 256);
#define CDML_EW_LAUNCH(BF, OP)                                                                                       \
  do {                                                                                                               \
    if (vec) ew16_kernel<BF, OP, 8><<<grid, 256, 0, st>>>(pa, lda, pb, ldb, pc, ldc, po, ldo, rows, cols, alpha);       \
    else ew16_kernel<BF, OP, 2><<<grid, 256, 0, st>>>(pa, lda, pb, ldb, pc, ldc, po, ldo, rows, cols, alpha);           \
  } while (0)
#define CDML_EW_OPS(BF)                                                                                              \
  switch (op) {                                                                                                      \
    case 0: CDML_EW_LAUNCH(BF, 0); break;                                                                            \
    case 1: CDML_EW_LAUNCH(BF, 1); break;                                                                            \
    case 2: CDML_EW_LAUNCH(BF, 2); break;                                                                            \
    case 3: CDML_EW_LAUNCH(BF, 3); break;                                                                            \
    case 4: CDML_EW_LAUNCH(BF, 4); break;                                                                            \
    case 5: CDML_EW_LAUNCH(BF, 5); break;                                                                            \
    case 6: CDML_EW_LAUNCH(BF, 6); break;                                                                            \
    default: CDML_EW_LAUNCH(BF, 7); break;                                                                           \
  }
  if (dtype16 == CDML_BF16) { CDML_EW_OPS(1) } else { CDML_EW_OPS(0) }
#undef CDML_EW_OPS
#undef CDML_EW_LAUNCH
  CDML_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int cdml_rows_l2norm16(cdml_ctx* ctx, const void* y16, int64_t n, int D, int64_t ld_y, float eps, int dtype16, float* e,
                       int64_t ld_e, float* rinv, void* e16, int64_t ld_e16, void* stream) {
  CDML_REQUIRE(ctx && y16 && e && n >= 0 && D > 0 && D % 2 == 0 && ld_y % 2 == 0 && ld_e % 2 == 0 && ld_e16 % 2 == 0,
               "cdml_rows_l2norm16: bad argument");
  if (n == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = row_grid(ctx, n);
  if (dtype16 == CDML_BF16)
    rows_l2norm16_kernel<1><<<grid, kRowThreads, 0, st>>>(static_cast<const uint16_t*>(y16), n, D, ld_y, eps, e, ld_e, rinv,
                                                          static_cast<uint16_t*>(e16), ld_e16);
  else
    rows_l2norm16_kernel<0><<<grid, kRowThreads, 0, st>>>(static_cast<const uint16_t*>(y16), n, D, ld_y, eps, e, ld_e, rinv,
                                                          static_cast<uint16_t*>(e16), ld_e16);
  CDML_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int cdml_cast16(cdml_ctx* ctx, const float* in, int64_t n, void* out16, int dtype16, void* stream) {
  CDML_REQUIRE(ctx && in && out16, "cdml_cast16: NULL argument");
  if (n == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = flat_grid(ctx, n, 256);
  if (dtype16 == CDML_BF16) cast16_kernel<1><<<grid, 256, 0, st>>>(in, n, static_cast<uint16_t*>(out16));
  else cast16_kernel<0><<<grid, 256, 0, st>>>(in, n, static_cast<uint16_t*>(out16));
  CDML_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int cdml_fill_column16(cdml_ctx* ctx, void* X16, int64_t rows, int64_t ld, int64_t col, float value, int dtype16,
                       void* stream) {
  CDML_REQUIRE(ctx && X16 && rows >= 0 && col >= 0 && col < ld, "cdml_fill_column16: bad argument");
  if (rows == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint16_t bits;
  if (dtype16 == CDML_BF16) {
    const __nv_bfloat16 b = __float2bfloat16(value);
    bits = *reinterpret_cast<const uint16_t*>(&b);
  } else {
    const __half h = __float2half(value);
    bits = *reinterpret_cast<const uint16_t*>(&h);
  }
  fill_column16_kernel<<<flat_grid(ctx, rows, 256), 256, 0, st>>>(static_cast<uint16_t*>(X16), rows, ld, col, bits);
  CDML_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int cdml_mean_pair_dist(cdml_ctx* ctx, const float* V, int64_t ld, int D, const int64_t* pairs, int64_t P,
                        float* out_mean, void* stream) {
  CDML_REQUIRE(ctx && V && pairs && out_mean && P > 0 && D > 0, "cdml_mean_pair_dist: bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* dist = nullptr;
  CDML_CHECK_CUDA(cudaMallocAsync(&dist, sizeof(float) * (P + 4), st));
  pair_dist_kernel<<<row_grid(ctx, P), kRowThreads, 0, st>>>(V, ld, D, pairs, P, dist);
  hinge_stats_kernel<<<1, 1024, 0, st>>>(dist, nullptr, nullptr, P, dist + P);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(out_mean, dist + P, sizeof(float), cudaMemcpyDeviceToDevice, st);
  cudaFreeAsync(dist, st);
  CDML_CHECK_CUDA(e);
  return 0;
}

}  // extern "C"
