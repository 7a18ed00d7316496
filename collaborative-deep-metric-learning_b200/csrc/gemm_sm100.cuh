// Persistent, warp-specialised tcgen05 GEMM core for sm_100a.
//
//   D[M,N] (fp32 accumulators in TMEM) = A[M,K] * B[N,K]^T     16-bit operands (fp16 | bf16)
//
// Operands may be K-major (row-major [rows,K]) or MN-major (row-major [K,rows]) independently, so the
// tower's forward (x @ W), data-gradient (dz @ W^T) and weight-gradient (x^T @ dz) all run on this one
// kernel without transposed copies.  TMA stages 128-byte-swizzled tiles into a kStages ring, a single
// thread issues tcgen05.mma (M=128, N=BN, K=16), the accumulator is double-buffered in TMEM so the
// epilogue warps (tcgen05.ld -> fused bias / leaky-ReLU / L2-norm / mask -> global) overlap the next
// tile's main loop.  Optional split-K writes fp32 partials that a separate kernel reduces in fixed order.
//
// Warp roles (384 threads): w0 TMA producer, w1 MMA issuer, w2 TMEM allocator, w3 spare, w4..11 epilogue.  Two
// epilogue warps share each TMEM lane quarter and split the tile's columns, so every SM sub-partition has two
// epilogue warps to hide TMEM / global-memory latency behind each other.
#pragma once
#include "common.cuh"

namespace cdml {

constexpr int kBM = 128;  // tile rows   (TMEM lanes)
constexpr int kBK = 64;   // 16-bit elements per k-block = one 128 B swizzle span
constexpr int kUK = 16;   // K per tcgen05.mma (kind::f16)
constexpr uint32_t kEpiStageBytes = 16384;  // per-warp transposition buffers that make the epilogue's global stores coalesced
constexpr int kGemmThreads = 384;  // 4 control warps + 8 epilogue warps (two per TMEM lane quarter)

struct GemmShape {
  int M, N, K;
  int m_tiles, n_tiles;
  int num_kb;        // ceil(K / 64)
  int kb_per_split;  // k-blocks handled by one split
  int num_splits;    // every split owns >= 1 k-block
  int m_fastest;     // tile order inside a split: 1 = consecutive CTAs walk down M (share the B panel), 0 = along N
  uint32_t idesc;
};

template <int BN, int kStages>
struct GemmSmem {
  static constexpr uint32_t kABytes = kBM * kBK * 2;  // 16 KB
  static constexpr uint32_t kBBytes = BN * kBK * 2;
  static constexpr uint32_t kEpiOff = kStages * (kABytes + kBBytes);   // epilogue staging: 8 warps x 2 KB
  static constexpr uint32_t kBarOff = kEpiOff + kEpiStageBytes;
  static constexpr uint32_t kNumBars = 2 * kStages + 4;
  static constexpr uint32_t kTotal = kBarOff + kNumBars * 8 + 16 + 1024;  // +1024: manual 1 KB alignment
};

// ------------------------------------------------------------------------------------------------
// Epilogues.  run() is executed by the epilogue warps; thread <-> one output row, 32-column chunks [c0,c1) of the tile.
//   taddr : TMEM address of (lane quarter, first accumulator column of this tile)
//   row   : global output row of this thread;  n0 : first global column of the tile
//   kSplitColumns: the two warps of a lane quarter each take half of the chunks; otherwise one warp takes all.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float leaky(float v, float alpha) { return v > 0.f ? v : alpha * v; }
// Bias of the 32 columns starting at nb: one coalesced load (lane j <-> column nb+j), handed to every thread's
// column loop by shuffle.  (A per-column uniform __ldg serialises on load latency inside the unrolled loop.)
__device__ __forceinline__ float chunk_bias(const float* bias, int nb, int N) {
  const int col = nb + static_cast<int>(threadIdx.x & 31);
  return (bias != nullptr && col < N) ? __ldg(bias + col) : 0.f;
}

// Coalesced store of one 32-row x 32-column 16-bit chunk held one row per thread (pk = this thread's 32 packed values):
// transposed through the warp's 2 KB staging buffer (XOR-swizzled 16-byte slots, conflict-free both ways) so that each
// store instruction writes 8 rows x 64 contiguous bytes instead of 32 rows x 16 bytes.
__device__ __forceinline__ void store_chunk16(uint16_t* out, int64_t ld, int row_base, int nb, int M, int N, uint32_t stg,
                                              const uint32_t (&pk)[16]) {
  const int lane = threadIdx.x & 31;
  __syncwarp();
#pragma unroll
  for (int j = 0; j < 4; ++j)
    sts128(stg + lane * 64 + ((j ^ ((lane >> 1) & 3)) << 4), pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
  __syncwarp();
  const int cch = lane & 3;
  const int col = nb + 8 * cch;
  const bool vec = (ld & 7) == 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = 8 * i + (lane >> 2);
    const uint4 v = lds128(stg + r * 64 + ((cch ^ ((r >> 1) & 3)) << 4));
    const int grow = row_base + r;
    if (grow < M) {
      uint16_t* p = out + static_cast<int64_t>(grow) * ld + col;
      if (vec && col + 8 <= N) {
        *reinterpret_cast<uint4*>(p) = v;
      } else {
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int e = 0; e < 8; ++e)
          if (col + e < N) p[e] = static_cast<uint16_t>(w[e >> 1] >> ((e & 1) * 16));
      }
    }
  }
}

// Same for a 32 x 32 fp32 chunk (4 KB staging buffer): each store instruction writes 4 rows x 128 contiguous bytes.
__device__ __forceinline__ void store_chunk32(float* out, int64_t ld, int row_base, int nb, int M, int N, uint32_t stg,
                                              const float (&f)[32]) {
  const int lane = threadIdx.x & 31;
  __syncwarp();
#pragma unroll
  for (int j = 0; j < 8; ++j)
    sts128(stg + lane * 128 + ((j ^ (lane & 7)) << 4), __float_as_uint(f[4 * j]), __float_as_uint(f[4 * j + 1]),
           __float_as_uint(f[4 * j + 2]), __float_as_uint(f[4 * j + 3]));
  __syncwarp();
  const int cch = lane & 7;
  const int col = nb + 4 * cch;
  const bool vec = (ld & 3) == 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = 4 * i + (lane >> 3);
    const uint4 v = lds128(stg + r * 128 + ((cch ^ (r & 7)) << 4));
    const int grow = row_base + r;
    if (grow < M) {
      float* p = out + static_cast<int64_t>(grow) * ld + col;
      if (vec && col + 4 <= N) {
        *reinterpret_cast<uint4*>(p) = v;
      } else {
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (col + e < N) p[e] = __uint_as_float(w[e]);
      }
    }
  }
}

// Per-warp cache of the 128 per-column 32-bit constants of the warp's four chunks (KNN bounds / half norms, mining
// candidate guids) in its 2 KB staging slice, tagged with the column block: the resident-B kernel sweeps hundreds of
// row tiles against one column block, and per-chunk global loads of these constants were measured to cost ~25% of
// the KNN scan.  Slice layout: [0,128) scratch of the epilogue's rare path | [128,640) constants | [640] tag = n0+1.
constexpr uint32_t kColCacheOff = 128, kColTagOff = 640, kWarpSliceBytes = 2048;
__device__ __forceinline__ void col_cache_reset(uint32_t epi_smem) {   // one thread, before the CTA-wide barrier
  for (int w = 0; w < 8; ++w)
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(epi_smem + w * kWarpSliceBytes + kColTagOff), "r"(0u) : "memory");
}
template <class Fetch>
__device__ __forceinline__ void col_cache_fill(uint32_t stg, int n0, int c0, Fetch&& fetch) {   // whole warp
  uint32_t tag;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tag) : "r"(stg + kColTagOff) : "memory");
  if (tag == static_cast<uint32_t>(n0 + 1)) return;   // warp-uniform
  const int lane = threadIdx.x & 31;
  __syncwarp();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const uint32_t v = fetch(n0 + (c0 + i) * 32 + lane);
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(stg + kColCacheOff + 4 * (32 * i + lane)), "r"(v) : "memory");
  }
  if (lane == 0) asm volatile("st.shared.b32 [%0], %1;" ::"r"(stg + kColTagOff), "r"(n0 + 1) : "memory");
  __syncwarp();
}

// fp32 store (optionally bias + leaky).  Split-K partials land at out + split * split_stride.
template <int BN>
struct EpiStoreF32 {
  static constexpr bool kSplitColumns = true;
  struct State {};
  __device__ __forceinline__ void pre(State&, int, int, const GemmShape&, int, int, uint32_t) const {}
  static constexpr bool kPrefetchNext = false;
  static constexpr bool kEarlyRelease = false;
  static constexpr bool kTmaStore = false;
  __device__ __forceinline__ void cols(int, const GemmShape&, int, int, uint32_t) const {}
  __device__ __forceinline__ void block_begin(uint32_t) const {}
  __device__ __forceinline__ void block_end(uint32_t) const {}
  float* out;
  int64_t ld;
  int64_t split_stride;
  const float* bias;  // nullable
  float alpha;        // 1.0f = identity
  __device__ __forceinline__ void run(uint32_t taddr, int row, int n0, int split, const GemmShape& s, int c0, int c1, uint32_t stg, State& st) const {
    float* orow = out + static_cast<int64_t>(split) * split_stride + static_cast<int64_t>(row) * ld;
    const bool row_ok = row < s.M;
#pragma unroll 1
    for (int c = c0; c < c1; ++c) {
      const int nb = n0 + c * 32;
      if (nb >= s.N) break;
      uint32_t v[32];
      tmem_ld_32x32(taddr + c * 32, v);
      const float b_lane = chunk_bias(bias, nb, s.N);
      tmem_ld_wait();
      float f[32];
#pragma unroll
      for (int j = 0; j < 32; ++j)
        f[j] = leaky(__uint_as_float(v[j]) + __shfl_sync(0xffffffffu, b_lane, j), alpha);
      if (row_ok) {
        if (nb + 32 <= s.N && (ld & 3) == 0) {
          float4* p = reinterpret_cast<float4*>(orow + nb);
#pragma unroll
          for (int j = 0; j < 8; ++j) p[j] = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (nb + j < s.N) orow[nb + j] = f[j];
        }
      }
    }
  }
};

// 16-bit store of leaky(acc + bias): the hidden-layer forward epilogue (models.py:19-30).
template <int BN, int kBf16>
struct EpiStore16 {
  static constexpr bool kSplitColumns = true;
  struct State {};
  __device__ __forceinline__ void pre(State&, int, int, const GemmShape&, int, int, uint32_t) const {}
  static constexpr bool kPrefetchNext = false;
  static constexpr bool kEarlyRelease = false;
  static constexpr bool kTmaStore = false;
  __device__ __forceinline__ void cols(int, const GemmShape&, int, int, uint32_t) const {}
  __device__ __forceinline__ void block_begin(uint32_t) const {}
  __device__ __forceinline__ void block_end(uint32_t) const {}
  uint16_t* out;
  int64_t ld;
  const float* bias;  // nullable
  float alpha;
  // Optional packed SIGN MASK of the output (1 bit per element; chunk-major: word [nb/32][row], pitch ld_mask words >= M,
  // bit j <-> column nb + j, set iff the pre-activation is > 0).  It is all the data-gradient GEMM of the backward pass
  // needs of this activation (leaky' = 1 | alpha): 1/16 of the bytes of the activation itself, and every warp access is
  // one coalesced 128-byte line (lane <-> row) here and in EpiMaskBits.
  uint32_t* mask_out;  // nullable
  int64_t ld_mask;
  __device__ __forceinline__ void run(uint32_t taddr, int row, int n0, int /*split*/, const GemmShape& s, int c0, int c1, uint32_t stg, State& st) const {
#pragma unroll 1
    for (int c = c0; c < c1; ++c) {
      const int nb = n0 + c * 32;
      if (nb >= s.N) break;
      uint32_t v[32];
      tmem_ld_32x32(taddr + c * 32, v);
      const float b_lane = chunk_bias(bias, nb, s.N);
      tmem_ld_wait();
      uint32_t pk[16];
      uint32_t bits = 0u;
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const float x0 = __uint_as_float(v[2 * j]) + __shfl_sync(0xffffffffu, b_lane, 2 * j);
        const float x1 = __uint_as_float(v[2 * j + 1]) + __shfl_sync(0xffffffffu, b_lane, 2 * j + 1);
        bits |= (x0 > 0.f ? 1u : 0u) << (2 * j);
        bits |= (x1 > 0.f ? 1u : 0u) << (2 * j + 1);
        pk[j] = pack2<kBf16>(leaky(x0, alpha), leaky(x1, alpha));
      }
      if (mask_out != nullptr && row < s.M) mask_out[static_cast<int64_t>(nb >> 5) * ld_mask + row] = bits;
      store_chunk16(out, ld, row - static_cast<int>(threadIdx.x & 31), nb, s.M, s.N, stg, pk);
    }
  }
};

// Last layer: y = leaky(acc + bias); e = y * rsqrt(max(sum y^2, 1e-12))  (models.py:60-61).
// Requires the whole row in one tile (N <= BN).  Writes e (fp32), rinv[row], optional 16-bit e.
template <int BN, int kBf16>
struct EpiL2Norm {
  static constexpr bool kSplitColumns = false;  // the row norm needs every column of the row in one thread
  struct State {};
  __device__ __forceinline__ void pre(State&, int, int, const GemmShape&, int, int, uint32_t) const {}
  static constexpr bool kPrefetchNext = false;
  static constexpr bool kEarlyRelease = false;
  static constexpr bool kTmaStore = false;
  __device__ __forceinline__ void cols(int, const GemmShape&, int, int, uint32_t) const {}
  __device__ __forceinline__ void block_begin(uint32_t) const {}
  __device__ __forceinline__ void block_end(uint32_t) const {}
  float* out;  // [M, ld] fp32 embedding
  int64_t ld;
  const float* bias;
  float alpha;
  float* rinv;      // [M] nullable
  uint16_t* out16;  // [M, ld16] nullable
  int64_t ld16;
  __device__ __forceinline__ void run(uint32_t taddr, int row, int n0, int /*split*/, const GemmShape& s, int c0, int c1, uint32_t stg, State& st) const {
    const bool row_ok = row < s.M;
    float ss = 0.f;
#pragma unroll 1
    for (int c = c0; c < c1; ++c) {
      const int nb = n0 + c * 32;
      if (nb >= s.N) break;
      uint32_t v[32];
      tmem_ld_32x32(taddr + c * 32, v);
      const float b_lane = chunk_bias(bias, nb, s.N);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        // columns beyond N hold exact zeros (TMA zero fill) and a zero bias: they add nothing
        const float x = leaky(__uint_as_float(v[j]) + __shfl_sync(0xffffffffu, b_lane, j), alpha);
        ss = fmaf(x, x, ss);
      }
    }
    const float r = rsqrtf(fmaxf(ss, 1e-12f));
    if (row_ok && rinv != nullptr) rinv[row] = r;
#pragma unroll 1
    for (int c = c0; c < c1; ++c) {
      const int nb = n0 + c * 32;
      if (nb >= s.N) break;
      uint32_t v[32];
      tmem_ld_32x32(taddr + c * 32, v);
      const float b_lane = chunk_bias(bias, nb, s.N);
      tmem_ld_wait();
      float f[32];
#pragma unroll
      for (int j = 0; j < 32; ++j)
        f[j] = leaky(__uint_as_float(v[j]) + __shfl_sync(0xffffffffu, b_lane, j), alpha) * r;
      store_chunk32(out, ld, row - static_cast<int>(threadIdx.x & 31), nb, s.M, s.N, stg, f);
      if (out16 != nullptr) {   // warp-uniform.  The 16-bit copy (mining / KNN operand) goes through the same staging
        uint32_t pk[16];        // transpose as the hidden layers: 8 rows x 64 bytes per store instead of 32 x 2 bytes
#pragma unroll
        for (int j = 0; j < 16; ++j) pk[j] = pack2<kBf16>(f[2 * j], f[2 * j + 1]);
        store_chunk16(out16, ld16, row - static_cast<int>(threadIdx.x & 31), nb, s.M, s.N, stg, pk);
      }
    }
  }
};

// Data-gradient epilogue: out = acc * (mask > 0 ? 1 : alpha), mask = the layer's own (post-leaky)
// forward output -- sign(leaky(z)) == sign(z), so no pre-activation stash is needed.
template <int BN, int kBf16>
struct EpiMaskLeaky {
  static constexpr bool kSplitColumns = true;
  struct State {
    uint4 raw[4][4];   // the four 32x32 mask chunks of this warp's half-tile, in the coalesced fetch layout
  };
  static constexpr bool kPrefetchNext = false;
  static constexpr bool kEarlyRelease = false;
  static constexpr bool kTmaStore = false;
  __device__ __forceinline__ void cols(int, const GemmShape&, int, int, uint32_t) const {}
  __device__ __forceinline__ void block_begin(uint32_t) const {}
  __device__ __forceinline__ void block_end(uint32_t) const {}
  uint16_t* out;
  int64_t ld;
  const uint16_t* mask;
  int64_t ld_mask;
  float alpha;
  // Coalesced fetch of a 32-row x 32-column mask chunk: lane l reads 16 bytes of row 8i + l/4 (i = 0..3), so one load
  // instruction covers 8 rows x 64 contiguous bytes.  Zeros outside the matrix.
  __device__ __forceinline__ void fetch_mask(int row_base, int nb, int M, int N, bool active, uint4 (&raw)[4]) const {
    const int lane = threadIdx.x & 31;
    const int col = nb + 8 * (lane & 3);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int grow = row_base + 8 * i + (lane >> 2);
      raw[i] = make_uint4(0u, 0u, 0u, 0u);
      if (active && grow < M) {
        const uint16_t* p = mask + static_cast<int64_t>(grow) * ld_mask + col;
        if ((ld_mask & 7) == 0 && col + 8 <= N) {
          raw[i] = __ldg(reinterpret_cast<const uint4*>(p));
        } else {
          uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
          for (int e = 0; e < 8; ++e)
            if (col + e < N) w[e >> 1] |= static_cast<uint32_t>(p[e]) << ((e & 1) * 16);
          raw[i] = make_uint4(w[0], w[1], w[2], w[3]);
        }
      }
    }
  }
  // Through the warp's staging buffer: every thread ends up with the 32 mask values of ITS row.
  __device__ __forceinline__ void transpose_mask(uint32_t stg, const uint4 (&raw)[4], uint32_t (&mk)[16]) const {
    const int lane = threadIdx.x & 31;
    const int cch = lane & 3;
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = 8 * i + (lane >> 2);
      sts128(stg + r * 64 + ((cch ^ ((r >> 1) & 3)) << 4), raw[i].x, raw[i].y, raw[i].z, raw[i].w);
    }
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint4 t = lds128(stg + lane * 64 + ((j ^ ((lane >> 1) & 3)) << 4));
      mk[4 * j] = t.x, mk[4 * j + 1] = t.y, mk[4 * j + 2] = t.z, mk[4 * j + 3] = t.w;
    }
  }
  // Requested BEFORE the accumulator is waited for: all four mask chunks of this warp's half-tile (64 registers).  The
  // epilogue is bound by HBM latency x bytes in flight; the fetch overlaps the tile's MMAs instead of following them.
  __device__ __forceinline__ void pre(State& st, int row, int n0, const GemmShape& s, int c0, int c1, uint32_t /*stg*/) const {
    static_assert(BN == 256, "a warp owns 4 chunks of the tile");
    const int row_base = row - static_cast<int>(threadIdx.x & 31);
#pragma unroll
    for (int cc = 0; cc < 4; ++cc)
      fetch_mask(row_base, n0 + (c0 + cc) * 32, s.M, s.N, c0 + cc < c1 && n0 + (c0 + cc) * 32 < s.N, st.raw[cc]);
  }
  __device__ __forceinline__ void run(uint32_t taddr, int row, int n0, int /*split*/, const GemmShape& s, int c0, int c1,
                                      uint32_t stg, State& st) const {
    const int row_base = row - static_cast<int>(threadIdx.x & 31);
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
      const int c = c0 + cc;
      const int nb = n0 + c * 32;
      if (c < c1 && nb < s.N) {   // warp-uniform
        uint32_t v[32];
        tmem_ld_32x32(taddr + c * 32, v);
        uint32_t mk[16];
        transpose_mask(stg, st.raw[cc], mk);
        tmem_ld_wait();
        uint32_t pk[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float2 m = unpack2<kBf16>(mk[j]);
          const float x0 = __uint_as_float(v[2 * j]) * (m.x > 0.f ? 1.f : alpha);
          const float x1 = __uint_as_float(v[2 * j + 1]) * (m.y > 0.f ? 1.f : alpha);
          pk[j] = pack2<kBf16>(x0, x1);
        }
        store_chunk16(out, ld, row_base, nb, s.M, s.N, stg, pk);
      }
    }
  }
};

// Data-gradient epilogue on the packed sign mask EpiStore16 wrote in the forward pass: out = acc * (bit ? 1 : alpha).
// The mask of a thread's four chunks is four registers (the 16-bit activation it replaces was 64), so the loads of the
// NEXT tile are issued before the current tile is processed (kPrefetchNext) and the TMEM reads are double-buffered: the
// kernel is bound by its 16-bit output stream (M*N*2 bytes), not by a second M*N*2-byte mask read.
template <int BN, int kBf16>
struct EpiMaskBits {
  static constexpr bool kSplitColumns = true;
  struct State {
    uint32_t bits[4];
  };
  static constexpr bool kPrefetchNext = true;
  static constexpr bool kEarlyRelease = false;
  static constexpr bool kTmaStore = false;
  __device__ __forceinline__ void cols(int, const GemmShape&, int, int, uint32_t) const {}
  __device__ __forceinline__ void block_begin(uint32_t) const {}
  __device__ __forceinline__ void block_end(uint32_t) const {}
  uint16_t* out;
  int64_t ld;
  const uint32_t* mask;   // [ceil(N/32)][ld_mask] words, lane <-> row
  int64_t ld_mask;
  float alpha;
  __device__ __forceinline__ void pre(State& st, int row, int n0, const GemmShape& s, int c0, int c1, uint32_t /*stg*/) const {
    static_assert(BN == 256, "a warp owns 4 chunks of the tile");
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
      const int nb = n0 + (c0 + cc) * 32;
      st.bits[cc] = (c0 + cc < c1 && nb < s.N && row < s.M) ? __ldg(mask + static_cast<int64_t>(nb >> 5) * ld_mask + row) : 0u;
    }
  }
  __device__ __forceinline__ void run(uint32_t taddr, int row, int n0, int /*split*/, const GemmShape& s, int c0, int c1,
                                      uint32_t stg, State& st) const {
    const int row_base = row - static_cast<int>(threadIdx.x & 31);
    auto ok = [&](int cc) { return c0 + cc < c1 && n0 + (c0 + cc) * 32 < s.N; };   // warp-uniform
    auto chunk = [&](const uint32_t (&v)[32], int cc) {
      const uint32_t b = st.bits[cc];
      uint32_t pk[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const float x0 = __uint_as_float(v[2 * j]) * ((b >> (2 * j)) & 1u ? 1.f : alpha);
        const float x1 = __uint_as_float(v[2 * j + 1]) * ((b >> (2 * j + 1)) & 1u ? 1.f : alpha);
        pk[j] = pack2<kBf16>(x0, x1);
      }
      store_chunk16(out, ld, row_base, n0 + (c0 + cc) * 32, s.M, s.N, stg, pk);
    };
    uint32_t va[32], vb[32];
    if (ok(0)) tmem_ld_32x32(taddr + c0 * 32, va);
#pragma unroll
    for (int cc = 0; cc < 4; cc += 2) {
      tmem_ld_wait();
      if (ok(cc + 1)) tmem_ld_32x32(taddr + (c0 + cc + 1) * 32, vb);
      if (ok(cc)) chunk(va, cc);
      tmem_ld_wait();
      if (cc + 2 < 4 && ok(cc + 2)) tmem_ld_32x32(taddr + (c0 + cc + 2) * 32, va);
      if (ok(cc + 1)) chunk(vb, cc + 1);
    }
  }
};

// The same epilogue with TMA stores (resident-B kernel only: the tensor map lives in the kernel's __grid_constant__
// parameter).  A warp writes its 32 x 32 chunk into its staging slice exactly as store_chunk16 does -- that XOR pattern IS
// the 64-byte TMA swizzle of a [32 rows x 64 bytes] box -- and one lane hands the box to the TMA engine instead of the warp
// reading it back and issuing 4 x 32 sixteen-byte global stores: half the shared-memory traffic and a quarter of the LSU
// instructions of the staged path, full 64-byte row pieces, M / N tails clipped by the tensor map.
//
// Slice reuse.  A box is staged after `wait_group.read 1` (every committed box except the newest has left shared memory),
// which is safe only if the newest box came from the OTHER slice.  Invariant: every tile's last box comes from slice 1.
// So a tile of n boxes (the ok() chunks are a prefix: cc = 0 .. n-1) stages box cc in slice (cc + n) & 1.  With n even
// the first box takes slice 0 and `read 1` suffices; with n odd (the last column block when N mod 256 lies in (0,32],
// (64,96], (128,160] or (192,224]) the first box takes slice 1, where the previous tile's last box may still be read,
// and waits with `read 0` -- for a box committed before the previous tile's epilogue ended, not for the one just issued.
template <int BN, int kBf16>
struct EpiMaskBitsTma {
  static constexpr bool kSplitColumns = true;
  struct State {
    uint32_t bits[4];
    uint32_t release_bar;   // the accumulator buffer's "empty" barrier (kEarlyRelease)
  };
  static constexpr bool kPrefetchNext = true;
  static constexpr bool kEarlyRelease = true;
  static constexpr bool kTmaStore = true;    // two 2 KB staging slices per warp: a box is written while the previous one drains
  __device__ __forceinline__ void cols(int, const GemmShape&, int, int, uint32_t) const {}
  __device__ __forceinline__ void block_begin(uint32_t) const {}
  __device__ __forceinline__ void block_end(uint32_t) const {}
  CUtensorMap out_map;    // [M rows, N cols] 16-bit, box 32 x 32, SWIZZLE_64B
  const uint32_t* mask;   // [ceil(N/32)][ld_mask] words, lane <-> row
  int64_t ld_mask;
  float alpha;
  __device__ __forceinline__ void pre(State& st, int row, int n0, const GemmShape& s, int c0, int c1, uint32_t /*stg*/) const {
    static_assert(BN == 256, "a warp owns 4 chunks of the tile");
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
      const int nb = n0 + (c0 + cc) * 32;
      st.bits[cc] = (c0 + cc < c1 && nb < s.N && row < s.M) ? __ldg(mask + static_cast<int64_t>(nb >> 5) * ld_mask + row) : 0u;
    }
    st.release_bar = 0u;
  }
  __device__ __forceinline__ void run(uint32_t taddr, int row, int n0, int /*split*/, const GemmShape& s, int c0, int c1,
                                      uint32_t stg0, State& st) const {
    const int lane = threadIdx.x & 31;
    const int row_base = row - lane;
    auto ok = [&](int cc) { return c0 + cc < c1 && n0 + (c0 + cc) * 32 < s.N; };   // warp-uniform
    const int boxes = ok(0) + ok(1) + ok(2) + ok(3);
    auto chunk = [&](const uint32_t (&v)[32], int cc) {
      const uint32_t b = st.bits[cc];
      uint32_t pk[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const float x0 = __uint_as_float(v[2 * j]) * ((b >> (2 * j)) & 1u ? 1.f : alpha);
        const float x1 = __uint_as_float(v[2 * j + 1]) * ((b >> (2 * j + 1)) & 1u ? 1.f : alpha);
        pk[j] = pack2<kBf16>(x0, x1);
      }
      const uint32_t stg = stg0 + ((cc + boxes) & 1) * 2048u;
      if (lane == 0) {
        if (cc == 0 && (boxes & 1)) bulk_wait_read0();   // slice 1 may hold the previous tile's last box
        else bulk_wait_read1();                          // the newest box came from the other slice
      }
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 4; ++j)
        sts128(stg + lane * 64 + ((j ^ ((lane >> 1) & 3)) << 4), pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) {
        tma_store_2d(&out_map, stg, n0 + (c0 + cc) * 32, row_base);
        bulk_commit();
      }
    };
    uint32_t va[32], vb[32];
    if (ok(0)) tmem_ld_32x32(taddr + c0 * 32, va);
#pragma unroll
    for (int cc = 0; cc < 4; cc += 2) {
      tmem_ld_wait();
      if (ok(cc + 1)) tmem_ld_32x32(taddr + (c0 + cc + 1) * 32, vb);
      if (ok(cc)) chunk(va, cc);
      tmem_ld_wait();
      if (cc + 2 < 4 && ok(cc + 2)) tmem_ld_32x32(taddr + (c0 + cc + 2) * 32, va);
      if (cc + 2 >= 4 && st.release_bar != 0u) {   // last TMEM read of this warp has landed: hand the buffer back
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(st.release_bar);
      }
      if (ok(cc + 1)) chunk(vb, cc + 1);
    }
  }
};

// Measurement aid (epilogue codes 100/101 of cdml_gemm16): no epilogue work at all / TMEM reads only.  Separates the
// main-loop rate from the TMEM-read and store costs when tuning.
template <int BN, int kReadTmem>
struct EpiNull {
  static constexpr bool kSplitColumns = true;
  struct State {};
  __device__ __forceinline__ void pre(State&, int, int, const GemmShape&, int, int, uint32_t) const {}
  static constexpr bool kPrefetchNext = false;
  static constexpr bool kEarlyRelease = false;
  static constexpr bool kTmaStore = false;
  __device__ __forceinline__ void cols(int, const GemmShape&, int, int, uint32_t) const {}
  __device__ __forceinline__ void block_begin(uint32_t) const {}
  __device__ __forceinline__ void block_end(uint32_t) const {}
  float* out;
  __device__ __forceinline__ void run(uint32_t taddr, int row, int n0, int /*split*/, const GemmShape& s, int c0, int c1, uint32_t stg, State& st) const {
    if (kReadTmem) {
      uint32_t acc = 0u;
#pragma unroll 1
      for (int c = c0; c < c1; ++c) {
        uint32_t v[32];
        tmem_ld_32x32(taddr + c * 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) acc ^= v[j];
      }
      if (acc == 0x7fc12345u && row == s.M + 7) out[0] = 1.f;   // never true; keeps the loads alive
    }
  }
};

// ------------------------------------------------------------------------------------------------
// The kernel
// ------------------------------------------------------------------------------------------------
template <int kAMajorMN, int kBMajorMN, int BN, int kStages, class Epi>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                    const GemmShape s, const Epi epi) {
  using L = GemmSmem<BN, kStages>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_u32 = smem_u32(smem_raw);
  const uint32_t base = (raw_u32 + 1023u) & ~1023u;
  const uint32_t bar0 = base + L::kBarOff;
  auto a_smem = [&](int st) { return base + st * L::kABytes; };
  auto b_smem = [&](int st) { return base + kStages * L::kABytes + st * L::kBBytes; };
  auto full_bar = [&](int st) { return bar0 + 8u * st; };
  auto empty_bar = [&](int st) { return bar0 + 8u * (kStages + st); };
  auto tfull_bar = [&](int i) { return bar0 + 8u * (2 * kStages + i); };
  auto tempty_bar = [&](int i) { return bar0 + 8u * (2 * kStages + 2 + i); };
  const uint32_t tmem_slot = bar0 + 8u * L::kNumBars;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw_u32));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr uint32_t kTmemCols = (2 * BN <= 32) ? 32 : (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;
  static_assert(2 * BN <= 512, "two accumulator stages must fit TMEM");

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kStages; ++i) {
      mbar_init(full_bar(i), 1);
      mbar_init(empty_bar(i), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(tfull_bar(i), 1);
      mbar_init(tempty_bar(i), 8);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  if (threadIdx.x == 96) epi.block_begin(base + L::kEpiOff);  // warp 3: per-CTA epilogue state (e.g. the KNN candidate log cursor)
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  const int tiles = s.m_tiles * s.n_tiles;
  const int units = tiles * s.num_splits;

  if (warp == 0 && lane == 0) {
    // ===================== TMA producer =====================
    int stage = 0;
    uint32_t phase = 0;
    for (int u = blockIdx.x; u < units; u += gridDim.x) {
      const int split = u / tiles, t = u - split * tiles;
      const int m0 = (s.m_fastest ? t % s.m_tiles : t / s.n_tiles) * kBM;
      const int n0 = (s.m_fastest ? t / s.m_tiles : t % s.n_tiles) * BN;
      const int kb0 = split * s.kb_per_split;
      const int kb1 = min(s.num_kb, kb0 + s.kb_per_split);
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(empty_bar(stage), phase ^ 1, 100 + stage);
        mbar_arrive_expect_tx(full_bar(stage), L::kABytes + L::kBBytes);
        const int k0 = kb * kBK;
        if constexpr (kAMajorMN == 0) {
          tma_load_2d(a_smem(stage), &tma_a, full_bar(stage), k0, m0);
        } else {
#pragma unroll
          for (int i = 0; i < kBM / 64; ++i)
            tma_load_2d(a_smem(stage) + i * (kBK * 128), &tma_a, full_bar(stage), m0 + i * 64, k0);
        }
        if constexpr (kBMajorMN == 0) {
          tma_load_2d(b_smem(stage), &tma_b, full_bar(stage), k0, n0);
        } else {
#pragma unroll
          for (int i = 0; i < BN / 64; ++i)
            tma_load_2d(b_smem(stage) + i * (kBK * 128), &tma_b, full_bar(stage), n0 + i * 64, k0);
        }
        if (++stage == kStages) stage = 0, phase ^= 1;
      }
    }
  } else if (warp == 1 && lane == 0) {
    // ===================== MMA issuer =====================
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    // K-major: +32 B per UMMA_K inside the 128 B swizzle span; MN-major: +16 K-rows * 128 B.
    constexpr uint32_t kAStep = kAMajorMN ? (kUK * 128) : (kUK * 2);
    constexpr uint32_t kBStep = kBMajorMN ? (kUK * 128) : (kUK * 2);
    constexpr uint32_t kALbo = kAMajorMN ? (kBK * 128) : 16;
    constexpr uint32_t kBLbo = kBMajorMN ? (kBK * 128) : 16;
    for (int u = blockIdx.x; u < units; u += gridDim.x, ++it) {
      const int split = u / tiles;
      const int kb0 = split * s.kb_per_split;
      const int kb1 = min(s.num_kb, kb0 + s.kb_per_split);
      const int as = it & 1;
      const uint32_t ap = (it >> 1) & 1;
      mbar_wait(tempty_bar(as), ap ^ 1, 200 + as);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + as * BN;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(full_bar(stage), phase, 300 + stage);
        tc_fence_after();
#pragma unroll
        for (int k = 0; k < kBK / kUK; ++k) {
          const uint64_t ad = make_smem_desc(a_smem(stage) + k * kAStep, kALbo, 1024);
          const uint64_t bd = make_smem_desc(b_smem(stage) + k * kBStep, kBLbo, 1024);
          umma_f16(tmem_d, ad, bd, s.idesc, (kb > kb0 || k > 0) ? 1u : 0u);
        }
        tc_commit(empty_bar(stage));  // frees the smem slot once these MMAs retire
        if (kb == kb1 - 1) tc_commit(tfull_bar(as));
        if (++stage == kStages) stage = 0, phase ^= 1;
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue =====================
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    const int half = (warp - 4) >> 2;
    const uint32_t stg = base + L::kEpiOff + (warp - 4) * (Epi::kSplitColumns ? 2048u : 4096u);
    int it = 0;
    for (int u = blockIdx.x; u < units; u += gridDim.x, ++it) {
      const int split = u / tiles, t = u - split * tiles;
      const int m0 = (s.m_fastest ? t % s.m_tiles : t / s.n_tiles) * kBM;
      const int n0 = (s.m_fastest ? t / s.m_tiles : t % s.n_tiles) * BN;
      const int as = it & 1;
      const uint32_t ap = (it >> 1) & 1;
      const int ec0 = Epi::kSplitColumns ? half * (BN / 64) : 0, ec1 = Epi::kSplitColumns ? (half + 1) * (BN / 64) : BN / 32;
      typename Epi::State est;
      if (Epi::kSplitColumns || half == 0) {
        epi.cols(n0, s, ec0, ec1, stg);                           // per-column constants cached in the warp's staging slice
        epi.pre(est, m0 + q * 32 + lane, n0, s, ec0, ec1, stg);  // loads that do not need the accumulator
      }
      mbar_wait(tfull_bar(as), ap, 400 + as);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * BN;
      if (Epi::kSplitColumns || half == 0) epi.run(taddr, m0 + q * 32 + lane, n0, split, s, ec0, ec1, stg, est);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(as));
    }
  }

  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 96) epi.block_end(base + L::kEpiOff);
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------------
// Resident-B variant for short K (K <= 256: the data-gradient, mining and KNN scans).
//
// With only 4 k-blocks per tile the generic kernel re-streams 128 KB of B per 128x256 tile and is bound by L2->SM
// bandwidth, not by the tensor pipe.  Here a CTA owns one 256-wide column block (B panel: <=4 x 32 KB, loaded once)
// and sweeps a contiguous range of row tiles, streaming only A (16 KB per k-block): 3x less L2 traffic per tile.
// Both operands K-major.  Work unit = (column block, chunk of row tiles).
// ------------------------------------------------------------------------------------------------
struct ResBShape {
  int M, N, K;
  int m_tiles, n_tiles, num_kb;
  int m_chunks;         // row-tile chunks per column block
  int tiles_per_chunk;  // ceil(m_tiles / m_chunks)
  int n_fastest;        // unit order: 1 = column block fastest (concurrent CTAs share A rows), 0 = row chunk fastest
  uint32_t idesc;
};

// kStageSlices: 2 KB staging slices per epilogue warp (two for Epi::kTmaStore: a box is written while the previous drains).
template <int BN, int kAStages, int kStageSlices = 1>
struct ResBSmem {
  static constexpr uint32_t kABytes = kBM * kBK * 2;
  static constexpr uint32_t kBPanel = BN * kBK * 2;
  static constexpr uint32_t kMaxKb = 4;
  static constexpr uint32_t kEpiOff = kMaxKb * kBPanel + kAStages * kABytes;
  static constexpr uint32_t kEpiBytes = 8 * 2048 * kStageSlices;
  static constexpr uint32_t kBarOff = kEpiOff + kEpiBytes;
  static constexpr uint32_t kNumBars = 2 * kAStages + 2 + 4;
  static constexpr uint32_t kTotal = kBarOff + kNumBars * 8 + 16 + 1024;
};

template <int BN, int kAStages, class Epi>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_resb_tcgen05_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                         const ResBShape s, const __grid_constant__ Epi epi) {
  using L = ResBSmem<BN, kAStages, Epi::kTmaStore ? 2 : 1>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_u32 = smem_u32(smem_raw);
  const uint32_t base = (raw_u32 + 1023u) & ~1023u;
  const uint32_t bar0 = base + L::kBarOff;
  auto b_panel = [&](int kb) { return base + kb * L::kBPanel; };
  auto a_smem = [&](int st) { return base + L::kMaxKb * L::kBPanel + st * L::kABytes; };
  auto a_full = [&](int st) { return bar0 + 8u * st; };
  auto a_empty = [&](int st) { return bar0 + 8u * (kAStages + st); };
  const uint32_t b_full = bar0 + 8u * (2 * kAStages);
  const uint32_t b_empty = bar0 + 8u * (2 * kAStages + 1);
  auto tfull_bar = [&](int i) { return bar0 + 8u * (2 * kAStages + 2 + i); };
  auto tempty_bar = [&](int i) { return bar0 + 8u * (2 * kAStages + 4 + i); };
  const uint32_t tmem_slot = bar0 + 8u * L::kNumBars;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw_u32));
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr uint32_t kTmemCols = 512;
  static_assert(2 * BN <= 512, "two accumulator stages must fit TMEM");

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kAStages; ++i) {
      mbar_init(a_full(i), 1);
      mbar_init(a_empty(i), 1);
    }
    mbar_init(b_full, 1);
    mbar_init(b_empty, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(tfull_bar(i), 1);
      mbar_init(tempty_bar(i), 8);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  if (threadIdx.x == 96) epi.block_begin(base + L::kEpiOff);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  const int units = s.n_tiles * s.m_chunks;
  // unit u -> (column block, row tiles [chunk*tpc, min(m_tiles, (chunk+1)*tpc))).  n_fastest = 1: column block fastest,
  // the CTAs that run concurrently sweep the SAME rows of A against different resident panels (an A tile comes from HBM
  // once and from L2 for the other column blocks -- the KNN index scan streams 512 MB of rows per 256 queries).
  // n_fastest = 0: row chunk fastest, concurrent CTAs visit DIFFERENT rows (mining: the per-anchor running bound that
  // prunes its epilogue has been tightened by earlier visits instead of 148 CTAs meeting the anchor cold at once).
  if (warp == 0 && lane == 0) {
    // ===================== TMA producer =====================
    int stage = 0;
    uint32_t phase = 0, bphase = 0;
    for (int u = blockIdx.x; u < units; u += gridDim.x) {
      const int chunk = s.n_fastest ? u / s.n_tiles : u % s.m_chunks, nblk = s.n_fastest ? u % s.n_tiles : u / s.m_chunks;
      const int t0 = chunk * s.tiles_per_chunk, t1 = min(s.m_tiles, t0 + s.tiles_per_chunk);
      if (t0 >= t1) continue;
      mbar_wait(b_empty, bphase ^ 1, 500);
      mbar_arrive_expect_tx(b_full, s.num_kb * L::kBPanel);
      for (int kb = 0; kb < s.num_kb; ++kb) tma_load_2d(b_panel(kb), &tma_b, b_full, kb * kBK, nblk * BN);
      bphase ^= 1;
      for (int t = t0; t < t1; ++t) {
        for (int kb = 0; kb < s.num_kb; ++kb) {
          mbar_wait(a_empty(stage), phase ^ 1, 100 + stage);
          mbar_arrive_expect_tx(a_full(stage), L::kABytes);
          tma_load_2d(a_smem(stage), &tma_a, a_full(stage), kb * kBK, t * kBM);
          if (++stage == kAStages) stage = 0, phase ^= 1;
        }
      }
    }
  } else if (warp == 1 && lane == 0) {
    // ===================== MMA issuer =====================
    int stage = 0, it = 0;
    uint32_t phase = 0, bphase = 0;
    for (int u = blockIdx.x; u < units; u += gridDim.x) {
      const int chunk = s.n_fastest ? u / s.n_tiles : u % s.m_chunks, nblk = s.n_fastest ? u % s.n_tiles : u / s.m_chunks;
      const int t0 = chunk * s.tiles_per_chunk, t1 = min(s.m_tiles, t0 + s.tiles_per_chunk);
      if (t0 >= t1) continue;
      mbar_wait(b_full, bphase, 600);
      bphase ^= 1;
      tc_fence_after();
      for (int t = t0; t < t1; ++t, ++it) {
        const int as = it & 1;
        const uint32_t ap = (it >> 1) & 1;
        mbar_wait(tempty_bar(as), ap ^ 1, 200 + as);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + as * BN;
        for (int kb = 0; kb < s.num_kb; ++kb) {
          mbar_wait(a_full(stage), phase, 300 + stage);
          tc_fence_after();
#pragma unroll
          for (int k = 0; k < kBK / kUK; ++k) {
            const uint64_t ad = make_smem_desc(a_smem(stage) + k * (kUK * 2), 16, 1024);
            const uint64_t bd = make_smem_desc(b_panel(kb) + k * (kUK * 2), 16, 1024);
            umma_f16(tmem_d, ad, bd, s.idesc, (kb > 0 || k > 0) ? 1u : 0u);
          }
          tc_commit(a_empty(stage));
          if (kb == s.num_kb - 1) tc_commit(tfull_bar(as));
          if (++stage == kAStages) stage = 0, phase ^= 1;
        }
      }
      tc_commit(b_empty);  // the panel may be overwritten once every MMA of this unit has retired
    }
  } else if (warp >= 4) {
    // ===================== epilogue =====================
    const int q = warp & 3;
    const int half = (warp - 4) >> 2;         // which half of the tile's columns
    const uint32_t stg = base + L::kEpiOff + (warp - 4) * (Epi::kSplitColumns && !Epi::kTmaStore ? 2048u : 4096u);
    int it = 0;
    GemmShape gs;
    gs.M = s.M, gs.N = s.N, gs.K = s.K, gs.m_tiles = s.m_tiles, gs.n_tiles = s.n_tiles, gs.num_kb = s.num_kb;
    gs.kb_per_split = s.num_kb, gs.num_splits = 1, gs.m_fastest = 0, gs.idesc = s.idesc;
    // (unit, row tile) iterator; `nxt` runs one tile ahead so that an epilogue with kPrefetchNext can issue the next
    // tile's accumulator-independent loads (row constants) BEFORE it processes the current tile: when the epilogue is
    // the bottleneck the accumulator is already complete at the wait and those loads would sit on the critical path.
    struct TileIter {
      int u, t, t1, nblk;
      bool valid;
    };
    auto seek = [&](TileIter& ti) {   // first non-empty unit at or after ti.u
      ti.valid = false;
      for (; ti.u < units; ti.u += gridDim.x) {
        const int chunk = s.n_fastest ? ti.u / s.n_tiles : ti.u % s.m_chunks;
        const int t0 = chunk * s.tiles_per_chunk, t1 = min(s.m_tiles, t0 + s.tiles_per_chunk);
        if (t0 < t1) {
          ti.t = t0, ti.t1 = t1, ti.nblk = s.n_fastest ? ti.u % s.n_tiles : ti.u / s.m_chunks, ti.valid = true;
          return;
        }
      }
    };
    const bool active = Epi::kSplitColumns || half == 0;
    const int ec0 = Epi::kSplitColumns ? half * (BN / 64) : 0, ec1 = Epi::kSplitColumns ? (half + 1) * (BN / 64) : BN / 32;
    TileIter cur;
    cur.u = blockIdx.x;
    seek(cur);
    typename Epi::State est;
    if (cur.valid && active) {
      epi.cols(cur.nblk * BN, gs, ec0, ec1, stg);
      epi.pre(est, cur.t * kBM + q * 32 + lane, cur.nblk * BN, gs, ec0, ec1, stg);
    }
    while (cur.valid) {
      TileIter nxt = cur;
      if (++nxt.t >= nxt.t1) {
        nxt.u += gridDim.x;
        seek(nxt);
      }
      const int as = it & 1;
      const uint32_t ap = (it >> 1) & 1;
      typename Epi::State est_next;
      mbar_wait(tfull_bar(as), ap, 400 + as);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * BN;
      if (active) {
        if (Epi::kPrefetchNext && nxt.valid) epi.pre(est_next, nxt.t * kBM + q * 32 + lane, nxt.nblk * BN, gs, ec0, ec1, stg);
        // kEarlyRelease: the epilogue hands the accumulator buffer back itself, right after its LAST TMEM read (it still
        // has that chunk to process from registers): the MMA of the tile after next starts that much earlier
        if constexpr (Epi::kEarlyRelease) est.release_bar = tempty_bar(as);
        epi.run(taddr, cur.t * kBM + q * 32 + lane, cur.nblk * BN, 0, gs, ec0, ec1, stg, est);
      }
      if (!(Epi::kEarlyRelease && active)) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(as));
      }
      if (active && nxt.valid) {
        epi.cols(nxt.nblk * BN, gs, ec0, ec1, stg);   // the previous tile no longer reads the column cache
        if (!Epi::kPrefetchNext) epi.pre(est_next, nxt.t * kBM + q * 32 + lane, nxt.nblk * BN, gs, ec0, ec1, stg);
      }
      est = est_next;
      cur = nxt;
      ++it;
    }
    if constexpr (Epi::kTmaStore) {
      if (lane == 0) bulk_wait_all();    // this warp's last boxes are in global memory before the CTA retires
    }
  }

  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 96) epi.block_end(base + L::kEpiOff);
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

}  // namespace cdml
