// Exact flat KNN (IndexFlatL2 / IndexFlatIP semantics, faiss_knn.py:116-128) on the tcgen05 GEMM core.
//
// The nq x N score matrix never reaches HBM.  Per query chunk:
//   pass A  (sample)   S = Q16 . Xs16^T  over ~N/8 evenly spaced index rows; the epilogue keeps, per query, the best
//                      score of every 32-row group.  The k-th best group score is a LOWER bound of the k-th best score
//                      over the whole index (k distinct rows reach it).
//   pass B  (collect)  S = X16 . Q16^T   over the whole index; the epilogue appends (row, score) to the query's
//                      candidate list when score > bound - 2*eps, eps = a rigorous bound of the fp16 rounding error,
//                      so every true top-k row is nominated.  Warp-uniform ballot per column: no divergence.
//   refine             per query: prune by approximate score (again with the 2*eps guard), recompute the survivors in
//                      exact fp32 (||q||^2 + ||x||^2 - 2 q.x, clamped at 0 like faiss), sort by (distance, id), emit k.
// Queries whose list overflows (mass duplicates) take an exact fp32 brute-force path.
// score s = q.x - ||x||^2/2 (L2; ranking by s descending == distance ascending) or q.x (IP).
#include <math.h>
#include <string.h>

#include <algorithm>

#include <vector>

#include "gemm_launch.cuh"

namespace cdml {

constexpr int kCandCap = 2048;   // candidate list capacity per query
constexpr int kKeepCap = 2048;   // survivors of the approximate prune that get an exact re-rank
constexpr int kMaxGroups = 4096; // sample groups per query (sample <= 131072 rows)
constexpr int kRefineThreads = 256;

__device__ __forceinline__ float neg_inf() { return __int_as_float(0xff800000); }
__device__ __forceinline__ float pos_inf() { return __int_as_float(0x7f800000); }

// Four consecutive per-column constants (thresholds / half norms) as one uniform 16-byte load; columns beyond N
// read a sentinel so the unrolled loops need no branches.
__device__ __forceinline__ float4 ld4_or(const float* p, int col, int N, float fill) {
  if (col + 4 <= N) return __ldg(reinterpret_cast<const float4*>(p + col));
  float4 r;
  r.x = col < N ? __ldg(p + col) : fill;
  r.y = col + 1 < N ? __ldg(p + col + 1) : fill;
  r.z = col + 2 < N ? __ldg(p + col + 2) : fill;
  r.w = col + 3 < N ? __ldg(p + col + 3) : fill;
  return r;
}

// ---- pass A epilogue: thread <-> query row; best score of each 32-column (index-row) group ----
template <int BN>
struct EpiKnnGroupMax {
  static constexpr bool kSplitColumns = true;
  static constexpr bool kPrefetchNext = false;
  static constexpr bool kEarlyRelease = false;
  static constexpr bool kTmaStore = false;
  struct State {};
  __device__ __forceinline__ void pre(State&, int, int, const GemmShape&, int, int, uint32_t) const {}
  __device__ __forceinline__ void block_begin(uint32_t epi_smem) const { col_cache_reset(epi_smem); }
  __device__ __forceinline__ void block_end(uint32_t) const {}
  const float* h;  // [Ns] ||x||^2/2 of the sampled rows (zeros for IP)
  float* gmax;     // [nq, ldg]
  int64_t ldg;
  int wide;        // 0: one maximum per 32 sampled rows; 1: per 128 (4x less k-th selection work; needs Ns/128 >= 2k)
  // half norms of the warp's 128 columns (sample rows), once per column block; beyond N: +inf -> score -inf
  __device__ __forceinline__ void cols(int n0, const GemmShape& s, int c0, int /*c1*/, uint32_t stg) const {
    static_assert(BN == 256, "a warp owns 4 chunks (128 columns) of the tile");
    col_cache_fill(stg, n0, c0, [&](int col) { return __float_as_uint(col < s.N ? __ldg(h + col) : pos_inf()); });
  }
  __device__ __forceinline__ void run(uint32_t taddr, int row, int n0, int /*split*/, const GemmShape& s, int c0,
                                      int /*c1*/, uint32_t stg, State& /*st*/) const {
    float g[4];   // this warp's half of the tile: 4 groups of 32 columns
    uint32_t va[32], vb[32];
    // packed subtract + 3-input max: one instruction per accumulator element; next chunk's TMEM read in flight
    auto group = [&](const uint32_t (&v)[32], int cc) {
      const uint32_t hbase = stg + kColCacheOff + 128 * cc;
      float b0 = neg_inf(), b1 = neg_inf();
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const uint4 t = lds128(hbase + 16 * j);   // broadcast read
        const float2 lo = sub2(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(t.x), __uint_as_float(t.y));
        const float2 hi = sub2(__uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]), __uint_as_float(t.z), __uint_as_float(t.w));
        b0 = fmax3(b0, lo.x, lo.y);
        b1 = fmax3(b1, hi.x, hi.y);
      }
      return fmaxf(b0, b1);
    };
    auto ok = [&](int cc) { return n0 + (c0 + cc) * 32 < s.N; };   // warp-uniform
    tmem_ld_32x32(taddr + c0 * 32, va);
#pragma unroll
    for (int cc = 0; cc < 4; cc += 2) {
      tmem_ld_wait();
      if (ok(cc + 1)) tmem_ld_32x32(taddr + (c0 + cc + 1) * 32, vb);
      g[cc] = ok(cc) ? group(va, cc) : neg_inf();
      tmem_ld_wait();
      if (cc + 2 < 4 && ok(cc + 2)) tmem_ld_32x32(taddr + (c0 + cc + 2) * 32, va);
      g[cc + 1] = ok(cc + 1) ? group(vb, cc + 1) : neg_inf();
    }
    if (row < s.M) {
      if (wide) gmax[static_cast<int64_t>(row) * ldg + n0 / 128 + c0 / 4] = fmaxf(fmaxf(g[0], g[1]), fmaxf(g[2], g[3]));
      else *reinterpret_cast<float4*>(gmax + static_cast<int64_t>(row) * ldg + n0 / 32 + c0) = make_float4(g[0], g[1], g[2], g[3]);
    }
  }
};

// ---- pass B epilogue: thread <-> index row, column <-> query ----
// Survivors go to WARP-private logs (cursor and bounds cached in the warp's slice of the epilogue staging memory, no
// atomics, fire-and-forget 16-byte stores); knn_bin_kernel later files the log entries under their queries.  Measured
// on B200 (N=1M, 32768 queries, k=100; scan alone 12.9 ms): per-chunk global loads of the bounds cost +3 ms, a
// CTA-wide shared-atomic cursor with its round trip per hit +6.5 ms -- hence the cached bounds and private cursors.
// Staging layout per warp (2 KB): [0,128) row hand-over of the hit path | [128,640) the 128 bounds of this warp's
// columns | [640] tag = n0+1 of the cached bounds | [644] log cursor.
constexpr uint32_t kKnnWarpStage = kWarpSliceBytes;
constexpr uint32_t kKnnThrOff = kColCacheOff, kKnnCurOff = 644;
constexpr int kKnnLogsPerCta = 8;   // one per epilogue warp

template <int BN>
struct EpiKnnCollect {
  static constexpr bool kSplitColumns = true;
  const float* h;    // [N] ||x||^2/2 (zeros for IP)
  const float* thr;  // [nq] score bound per query
  uint4* log;        // [gridDim.x * 8, warp_cap] entries (query, row, score bits, 0)
  int32_t* log_count;  // [gridDim.x * 8]
  int32_t* log_overflow;
  unsigned int warp_cap;
  struct State {
    float hr;
    uint32_t release_bar;   // resident-B kernel: the accumulator buffer's "empty" barrier (0: the kernel arrives itself)
  };
  static constexpr bool kPrefetchNext = true;   // pre() only loads a row constant into registers
  static constexpr bool kEarlyRelease = true;
  static constexpr bool kTmaStore = false;
  __device__ __forceinline__ void block_begin(uint32_t epi_smem) const {
    col_cache_reset(epi_smem);
    for (int w = 0; w < kKnnLogsPerCta; ++w)
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(epi_smem + w * kKnnWarpStage + kKnnCurOff), "r"(0u) : "memory");
  }
  __device__ __forceinline__ void block_end(uint32_t epi_smem) const {
    for (int w = 0; w < kKnnLogsPerCta; ++w) {
      unsigned int n;
      asm volatile("ld.shared.b32 %0, [%1];" : "=r"(n) : "r"(epi_smem + w * kKnnWarpStage + kKnnCurOff) : "memory");
      log_count[blockIdx.x * kKnnLogsPerCta + w] = static_cast<int32_t>(n < warp_cap ? n : warp_cap);
      if (n > warp_cap) atomicOr(log_overflow, 1);
    }
  }
  // the row's half norm does not depend on the accumulator (issued one tile ahead by the resident-B kernel)
  __device__ __forceinline__ void pre(State& st, int row, int, const GemmShape& s, int, int, uint32_t) const {
    st.hr = row < s.M ? __ldg(h + row) : pos_inf();   // rows beyond M: score -inf, never pass
    st.release_bar = 0u;
  }
  // the bounds of the warp's 128 columns (queries), once per column block; beyond N: +inf, never pass
  __device__ __forceinline__ void cols(int n0, const GemmShape& s, int c0, int /*c1*/, uint32_t stg) const {
    static_assert(BN == 256, "a warp owns 4 chunks (128 columns) of the tile");
    col_cache_fill(stg, n0, c0, [&](int col) { return __float_as_uint(col < s.N ? __ldg(thr + col) : pos_inf()); });
  }
  __device__ __forceinline__ void run(uint32_t taddr, int row, int n0, int /*split*/, const GemmShape& s, int c0,
                                      int c1, uint32_t stg, State& st) const {
    const float hr = st.hr;
    const int lane = threadIdx.x & 31;
    const int warp_slot = (threadIdx.x >> 5) - 4;
    uint4* my_log = log + (static_cast<size_t>(blockIdx.x) * kKnnLogsPerCta + warp_slot) * warp_cap;
    unsigned int cursor;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(cursor) : "r"(stg + kKnnCurOff) : "memory");
    uint32_t va[32], vb[32];
    tmem_ld_32x32(taddr + c0 * 32, va);
    // one chunk: bounds from the staging slice, detection, hit path; the NEXT chunk's TMEM read is already in flight
    auto chunk = [&](const uint32_t (&v)[32], int cc) {
      const int nb = n0 + (c0 + cc) * 32;
      const uint32_t tbase = stg + kKnnThrOff + 128 * cc;
      // Detection -- one instruction per accumulator element: max over the row's 32 columns of (acc - bound[col]) in
      // packed fp32x2 subtracts and 3-input maxima; the row holds a survivor iff that maximum exceeds ||x_row||^2/2.
      float m0 = neg_inf(), m1 = neg_inf();
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const uint4 t = lds128(tbase + 16 * j);   // broadcast read
        const float2 lo = sub2(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(t.x), __uint_as_float(t.y));
        const float2 hi = sub2(__uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]), __uint_as_float(t.z), __uint_as_float(t.w));
        m0 = fmax3(m0, lo.x, lo.y);
        m1 = fmax3(m1, hi.x, hi.y);
      }
      unsigned int hits = __ballot_sync(0xffffffffu, fmaxf(m0, m1) > hr);
      // Hit path (about one row per 32x32 chunk at k=100): the row's 32 accumulators go through the staging slice so
      // that lane j re-tests column j with the SAME arithmetic; survivors are appended at the warp's own cursor.
      if (hits != 0u) {
        float thr_lane;
        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(thr_lane) : "r"(tbase + 4 * lane) : "memory");
        do {
          const int src = __ffs(hits) - 1;
          hits &= hits - 1u;
          __syncwarp();
          if (lane == src) {
#pragma unroll
            for (int j = 0; j < 8; ++j) sts128(stg + 16 * j, v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          }
          __syncwarp();
          float val;
          asm volatile("ld.shared.f32 %0, [%1];" : "=f"(val) : "r"(stg + 4 * lane) : "memory");
          const float hr_src = __shfl_sync(0xffffffffu, hr, src);
          const bool pass = val - thr_lane > hr_src;
          const unsigned int pm = __ballot_sync(0xffffffffu, pass);
          const unsigned int pos = cursor + static_cast<unsigned int>(__popc(pm & ((1u << lane) - 1u)));
          if (pass && pos < warp_cap)
            my_log[pos] = make_uint4(static_cast<uint32_t>(nb + lane), static_cast<uint32_t>(row - lane + src),
                                     __float_as_uint(val - hr_src), 0u);
          cursor += static_cast<unsigned int>(__popc(pm));
        } while (hits != 0u);
      }
    };
#pragma unroll
    for (int cc = 0; cc < 4; cc += 2) {
      const bool ok0 = c0 + cc < c1 && n0 + (c0 + cc) * 32 < s.N;          // warp-uniform
      const bool ok1 = c0 + cc + 1 < c1 && n0 + (c0 + cc + 1) * 32 < s.N;
      const bool ok2 = cc + 2 < 4 && c0 + cc + 2 < c1 && n0 + (c0 + cc + 2) * 32 < s.N;
      tmem_ld_wait();
      if (ok1) tmem_ld_32x32(taddr + (c0 + cc + 1) * 32, vb);
      if (ok0) chunk(va, cc);
      tmem_ld_wait();
      if (ok2) tmem_ld_32x32(taddr + (c0 + cc + 2) * 32, va);
      if (cc + 2 >= 4 && st.release_bar != 0u) {   // the last TMEM read of this warp has landed: hand the buffer back now
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(st.release_bar);
      }
      if (ok1) chunk(vb, cc + 1);
    }
    __syncwarp();
    if (lane == 0) asm volatile("st.shared.b32 [%0], %1;" ::"r"(stg + kKnnCurOff), "r"(cursor) : "memory");
  }
};

// File the CTA logs under their queries: cand[q][atomicAdd(cnt[q])] = (row, score).
__global__ void __launch_bounds__(256)
knn_bin_kernel(const uint4* __restrict__ log, const int32_t* __restrict__ log_count, unsigned int log_cap,
               int32_t* __restrict__ cand_idx, float* __restrict__ cand_val, int32_t* __restrict__ cnt, int cap) {
  const int n = log_count[blockIdx.y];
  const uint4* my = log + static_cast<size_t>(blockIdx.y) * log_cap;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint4 e = my[i];
    const int pos = atomicAdd(cnt + e.x, 1);
    if (pos < cap) {
      cand_idx[static_cast<int64_t>(e.x) * cap + pos] = static_cast<int32_t>(e.y);
      cand_val[static_cast<int64_t>(e.x) * cap + pos] = __uint_as_float(e.z);
    }
  }
}

// ---- small helpers -----------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
row_sumsq32_kernel(const float* __restrict__ X, int64_t n, int d, int64_t ld, float* __restrict__ ss, float half_scale,
                   float* __restrict__ half_out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * 8 + warp; r < n; r += static_cast<int64_t>(gridDim.x) * 8) {
    const float* x = X + r * ld;
    float a = 0.f;
    for (int j = lane; j < d; j += 32) a = fmaf(x[j], x[j], a);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) {
      ss[r] = a;
      if (half_out != nullptr) half_out[r] = a * half_scale;
    }
  }
}

__global__ void max_reduce_kernel(const float* __restrict__ x, int64_t n, float* __restrict__ out) {
  __shared__ float sh[32];
  float m = 0.f;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) m = fmaxf(m, x[i]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x < 32) {
    m = threadIdx.x < (blockDim.x >> 5) ? sh[threadIdx.x] : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (threadIdx.x == 0) *out = m;
  }
}

__global__ void fill_f32_kernel(float* p, int64_t n, float v) {
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x)
    p[i] = v;
}

// block-wide sum of an int (all threads get the result)
__device__ __forceinline__ int block_sum(int v, int* sh) {
  v = __reduce_add_sync(0xffffffffu, v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  int t = 0;
  for (int w = 0; w < (blockDim.x >> 5); ++w) t += sh[w];
  return t;
}

// k-th best sampled group score per query -> collection bound  thr = kth - slack(q).
// Bitwise bisection over the order-preserving key, stopped after the top kSelectBits bits: the result is the true
// k-th key rounded DOWN (a bound may always be lower), at 2^-12 relative precision -- far inside the slack.
constexpr int kSelectBits = 20;
// Both selections of one launch share the loaded keys and the block reductions (the two counts travel in one int).
template <int kPer, bool kDual>
__global__ void __launch_bounds__(kRefineThreads)
knn_kth_kernel(const float* __restrict__ gmax, int64_t ldg, int G, int k, int k2, const float* __restrict__ qss,
               float slack_scale, float slack_abs, float* __restrict__ thr, float* __restrict__ thr2, float sign2) {
  __shared__ int sh[kRefineThreads / 32];
  const int q = blockIdx.x;
  const float* g = gmax + static_cast<int64_t>(q) * ldg;
  uint32_t keys[kPer];
#pragma unroll
  for (int i = 0; i < kPer; ++i) {
    const int j = threadIdx.x + i * kRefineThreads;
    keys[i] = j < G ? f2key(g[j]) : 0u;
  }
  uint32_t T = 0, T2 = 0;   // k-th and k2-th best key (k2 only when thr2 != nullptr); counts fit 16 bits (G <= 4096)
  for (int bit = 31; bit >= 32 - kSelectBits; --bit) {
    const uint32_t cand = T | (1u << bit), cand2 = T2 | (1u << bit);
    int c = 0;
#pragma unroll
    for (int i = 0; i < kPer; ++i) c += (keys[i] >= cand ? 1 : 0) + (kDual && keys[i] >= cand2 ? 65536 : 0);
    c = block_sum(c, sh);
    if ((c & 0xffff) >= k) T = cand;
    if (kDual && (c >> 16) >= k2) T2 = cand2;
  }
  if (threadIdx.x == 0) {
    const float slack = slack_scale * sqrtf(qss[q]) + slack_abs;
    thr[q] = T > f2key(neg_inf()) ? key2f(T) - slack : neg_inf();
    if (kDual) thr2[q] = sign2 * (T2 > f2key(neg_inf()) ? key2f(T2) - slack : neg_inf());
  }
}

// Same selection, one WARP per query (G <= 1024 group maxima: 32 keys per lane in registers, counts by one
// __reduce_add_sync per bit).  A block per query spends its time in 2 x 20 __syncthreads for a few hundred keys: on an
// 8-way sharded 1M index (488 groups per query) the block version took 1.02 ms per 65536 queries, 12% of the shard's time.
template <bool kDual>
__global__ void __launch_bounds__(256)
knn_kth_warp_kernel(const float* __restrict__ gmax, int64_t ldg, int G, int k, int k2, const float* __restrict__ qss,
                    int64_t nq, float slack_scale, float slack_abs, float* __restrict__ thr, float* __restrict__ thr2,
                    float sign2) {
  const int lane = threadIdx.x & 31;
  const int64_t q = static_cast<int64_t>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (q >= nq) return;
  const float* g = gmax + q * ldg;
  uint32_t keys[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const int j = lane + 32 * i;
    keys[i] = j < G ? f2key(g[j]) : 0u;
  }
  uint32_t T = 0, T2 = 0;
  for (int bit = 31; bit >= 32 - kSelectBits; --bit) {
    const uint32_t cand = T | (1u << bit), cand2 = T2 | (1u << bit);
    int c = 0;
#pragma unroll
    for (int i = 0; i < 32; ++i) c += (keys[i] >= cand ? 1 : 0) + (kDual && keys[i] >= cand2 ? 65536 : 0);
    c = __reduce_add_sync(0xffffffffu, c);
    if ((c & 0xffff) >= k) T = cand;
    if (kDual && (c >> 16) >= k2) T2 = cand2;
  }
  if (lane == 0) {
    const float slack = slack_scale * sqrtf(qss[q]) + slack_abs;
    thr[q] = T > f2key(neg_inf()) ? key2f(T) - slack : neg_inf();
    if (kDual) thr2[q] = sign2 * (T2 > f2key(neg_inf()) ? key2f(T2) - slack : neg_inf());
  }
}

// Row-sharded index, after the collect pass: per query the k-th and the k_part-th best APPROXIMATE score among this
// shard's nominees (truncated bisection like above; a bound may always be lower).  pair[0][q] = k-th (-inf when the
// shard nominated fewer than k), pair[1][q] = -(k_part-th) (+inf when fewer than k_part): ONE all-reduce(MAX) of the pair
// over the shards then yields max_s(k-th) and min_s(k_part-th), both lower bounds of the GLOBAL k-th best approximate
// score (k_part = ceil(k / shards): if every shard holds k_part nominees above t, the index holds k).  The refine pass
// prunes against that global bound instead of its local k-th: 8 shards then re-rank ~25 rows per query each, not ~105.
__global__ void __launch_bounds__(256)
knn_nominee_kth_kernel(const float* __restrict__ cand_val, const int32_t* __restrict__ cnt, int cap, int k, int k2,
                       int64_t nq, float* __restrict__ pair) {
  const int lane = threadIdx.x & 31;
  const int64_t q = static_cast<int64_t>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (q >= nq) return;
  const int n = cnt[q];
  float a = neg_inf(), b = neg_inf();
  if (n <= cap && n >= min(k, k2)) {
    const float* v = cand_val + q * cap;
    uint32_t keys[8];
    const bool in_regs = n <= 256;
#pragma unroll
    for (int i = 0; i < 8; ++i) keys[i] = (in_regs && lane + 32 * i < n) ? f2key(v[lane + 32 * i]) : 0u;
    uint32_t T = 0, T2 = 0;
    for (int bit = 31; bit >= 32 - kSelectBits; --bit) {
      const uint32_t cand = T | (1u << bit), cand2 = T2 | (1u << bit);
      int c = 0;
      if (in_regs) {
#pragma unroll
        for (int i = 0; i < 8; ++i) c += (keys[i] >= cand ? 1 : 0) + (keys[i] >= cand2 ? 65536 : 0);
      } else {
        for (int i = lane; i < n; i += 32) {
          const uint32_t key = f2key(v[i]);
          c += (key >= cand ? 1 : 0) + (key >= cand2 ? 65536 : 0);
        }
      }
      c = __reduce_add_sync(0xffffffffu, c);
      if ((c & 0xffff) >= k) T = cand;
      if ((c >> 16) >= k2) T2 = cand2;
    }
    if (n >= k && T > f2key(neg_inf())) a = key2f(T);
    if (n >= k2 && T2 > f2key(neg_inf())) b = key2f(T2);
  }
  if (lane == 0) pair[q] = a, pair[nq + q] = -b;
}

// Collection bound from bounds agreed across index shards: thr = max(full, part) - slack(q)  (-inf when no shard had one)
__global__ void knn_thr_combine_kernel(const float* __restrict__ full, const float* __restrict__ part,
                                       const float* __restrict__ qss, int64_t n, float slack_scale, float slack_abs,
                                       float* __restrict__ thr, float part_sign) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float b = fmaxf(full[i], part_sign * part[i]);
  thr[i] = b > neg_inf() ? b - (slack_scale * sqrtf(qss[i]) + slack_abs) : neg_inf();
}

// Per query: approximate prune -> exact fp32 re-rank -> (distance,id) sort -> top-k.
__global__ void __launch_bounds__(kRefineThreads)
knn_refine_kernel(const float* __restrict__ Q, int64_t ldq, int d, const float* __restrict__ qss,
                  const float* __restrict__ X, int64_t ldx, const float* __restrict__ xss,
                  const int32_t* __restrict__ cand_idx, const float* __restrict__ cand_val,
                  const int32_t* __restrict__ cnt, int cap, int k, int metric, float slack_scale, float slack_abs,
                  int64_t id_offset, float* __restrict__ D, int64_t* __restrict__ I, int64_t out_ld,
                  int32_t* __restrict__ overflow, int n_all, const float* __restrict__ prune_pair, int64_t prune_ld,
                  const int32_t* __restrict__ handled) {
  __shared__ unsigned long long kept[kKeepCap];
  __shared__ int sh[kRefineThreads / 32];
  __shared__ uint32_t shu[2 * (kRefineThreads / 32)];
  __shared__ int n_keep;
  const int q = blockIdx.x;
  const int tid = threadIdx.x;
  if (handled != nullptr && handled[q] != 0) return;   // knn_refine_warp_kernel already wrote this query's list
  const int n = n_all > 0 ? 0 : cnt[q];   // n_all > 0: tiny database, every row is re-ranked exactly (no scan, no prune)
  if (n > cap) {  // too many nominees (mass ties): exact fallback handles this query
    if (tid == 0) overflow[q] = 1;
    return;
  }
  // the nominees stay in registers: kCandCap / kRefineThreads per thread
  constexpr int kPer = kCandCap / kRefineThreads;
  uint32_t keys[kPer];
  int32_t idxs[kPer];
  uint32_t kmax = 0u, kmin = 0xffffffffu;
#pragma unroll
  for (int t = 0; t < kPer; ++t) {
    const int i = tid + t * kRefineThreads;
    keys[t] = 0u, idxs[t] = 0;
    if (i < n) {
      keys[t] = f2key(cand_val[static_cast<int64_t>(q) * cap + i]);
      idxs[t] = cand_idx[static_cast<int64_t>(q) * cap + i];
      kmax = max(kmax, keys[t]), kmin = min(kmin, keys[t]);
    }
  }
  if (tid == 0) n_keep = 0;
  // k-th best approximate score among the nominees: bitwise bisection, skipping the bits every key shares (nominees
  // all lie between the collection bound and the best score: the top ~10 bits of the 20 examined are common)
  uint32_t T = 0;
  if (n > k) {
    kmax = __reduce_max_sync(0xffffffffu, kmax), kmin = __reduce_min_sync(0xffffffffu, kmin);
    if ((tid & 31) == 0) shu[tid >> 5] = kmax, shu[kRefineThreads / 32 + (tid >> 5)] = kmin;
    __syncthreads();
#pragma unroll
    for (int w = 0; w < kRefineThreads / 32; ++w) kmax = max(kmax, shu[w]), kmin = min(kmin, shu[kRefineThreads / 32 + w]);
    const uint32_t diff = kmax ^ kmin;
    const int top = diff == 0u ? -1 : 31 - __clz(diff);          // highest bit in which two keys differ
    T = top >= 31 ? 0u : (kmax >> (top + 1)) << (top + 1);      // the shared prefix
    for (int bit = top; bit >= 32 - kSelectBits; --bit) {       // k-th key rounded down: a prune bound may always be lower
      const uint32_t cand = T | (1u << bit);
      int c = 0;
#pragma unroll
      for (int t = 0; t < kPer; ++t) c += keys[t] >= cand ? 1 : 0;   // empty slots hold key 0 < cand
      if (block_sum(c, sh) >= k) T = cand;
    }
  } else {
    __syncthreads();
  }
  const float slack = slack_scale * sqrtf(qss[q]) + slack_abs;
  uint32_t keep_key = n > k ? f2key(key2f(T) - slack) : 0u;
  if (prune_pair != nullptr) {
    // row-sharded index: lower bound of the GLOBAL k-th best approximate score agreed across the shards (max_s of the
    // shards' k-th best nominee, min_s of their ceil(k/W)-th best) -- a row of the true top-k scores within 2*eps of it
    const float tg = fmaxf(prune_pair[q], -prune_pair[prune_ld + q]);
    if (tg > neg_inf()) keep_key = max(keep_key, f2key(tg - slack));
  }
#pragma unroll
  for (int t = 0; t < kPer; ++t) {
    if (tid + t * kRefineThreads < n && keys[t] >= keep_key) {
      const int pos = atomicAdd(&n_keep, 1);
      if (pos < kKeepCap) kept[pos] = static_cast<unsigned long long>(static_cast<uint32_t>(idxs[t]));
    }
  }
  if (n_all > 0) {
    for (int i = tid; i < n_all; i += kRefineThreads) kept[i] = static_cast<unsigned long long>(i);
    if (tid == 0) n_keep = n_all;
  }
  __syncthreads();
  const int nk = n_keep;
  if (nk > kKeepCap) {
    if (tid == 0) overflow[q] = 1;
    return;
  }
  // exact fp32 scores of the survivors: each warp takes four candidates at a time so that their row fetches (1 KB each
  // at d=256, scattered over the index) are all in flight together -- the re-rank is bound by HBM latency, not bytes
  const int warp = tid >> 5, lane = tid & 31;
  const float* qv = Q + static_cast<int64_t>(q) * ldq;
  const float qn = qss[q];
  const bool vec = (d & 3) == 0 && (ldx & 3) == 0 && (ldq & 3) == 0 &&
                   ((reinterpret_cast<uintptr_t>(X) | reinterpret_cast<uintptr_t>(Q)) & 15) == 0;
  for (int i0 = warp * 4; i0 < nk; i0 += (kRefineThreads / 32) * 4) {
    uint32_t id[4];
    float dot[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int c = 0; c < 4; ++c) id[c] = static_cast<uint32_t>(kept[min(i0 + c, nk - 1)]);
    if (vec) {
      for (int j = lane * 4; j < d; j += 128) {
        const float4 qq = __ldg(reinterpret_cast<const float4*>(qv + j));
        float4 xx[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) xx[c] = __ldg(reinterpret_cast<const float4*>(X + static_cast<int64_t>(id[c]) * ldx + j));
#pragma unroll
        for (int c = 0; c < 4; ++c)
          dot[c] = fmaf(qq.x, xx[c].x, fmaf(qq.y, xx[c].y, fmaf(qq.z, xx[c].z, fmaf(qq.w, xx[c].w, dot[c]))));
      }
    } else {
      for (int j = lane; j < d; j += 32) {
        const float qj = qv[j];
#pragma unroll
        for (int c = 0; c < 4; ++c) dot[c] = fmaf(qj, X[static_cast<int64_t>(id[c]) * ldx + j], dot[c]);
      }
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) dot[c] += __shfl_xor_sync(0xffffffffu, dot[c], o);
    }
    __syncwarp();
    if (lane < 4 && i0 + lane < nk) {
      const float dsel = lane == 0 ? dot[0] : lane == 1 ? dot[1] : lane == 2 ? dot[2] : dot[3];
      const uint32_t isel = lane == 0 ? id[0] : lane == 1 ? id[1] : lane == 2 ? id[2] : id[3];
      const float key = metric == 0 ? fmaxf(qn + xss[isel] - 2.f * dsel, 0.f) : -dsel;
      kept[i0 + lane] = (static_cast<unsigned long long>(f2key(key)) << 32) | isel;
    }
  }
  __syncthreads();
  const auto emit = [&](int i, unsigned long long e) {
    const float key = key2f(static_cast<uint32_t>(e >> 32));
    D[static_cast<int64_t>(q) * out_ld + i] = metric == 0 ? key : -key;
    I[static_cast<int64_t>(q) * out_ld + i] = static_cast<int64_t>(static_cast<uint32_t>(e)) + id_offset;
  };
  if (nk <= 2 * kRefineThreads) {
    // few survivors (the usual ~1.2 k): rank sort -- every element counts the (distance,id) keys below it (they are
    // distinct) and goes straight to its output slot; broadcast shared-memory reads, no barriers
    for (int i = tid; i < nk; i += kRefineThreads) {
      const unsigned long long e = kept[i];
      int rank = 0;
      for (int j = 0; j < nk; ++j) rank += kept[j] < e ? 1 : 0;
      if (rank < k) emit(rank, e);
    }
  } else {
    int P = 2;
    while (P < nk) P <<= 1;
    for (int i = nk + tid; i < P; i += kRefineThreads) kept[i] = ~0ull;
    __syncthreads();
    // bitonic sort ascending on (distance key, id)
    for (int size = 2; size <= P; size <<= 1) {
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        for (int t = tid; t < (P >> 1); t += kRefineThreads) {
          const int lo = ((t / stride) * (stride << 1)) + (t % stride);
          const int hi = lo + stride;
          const bool up = (lo & size) == 0;
          const unsigned long long a = kept[lo], b = kept[hi];
          if ((a > b) == up) kept[lo] = b, kept[hi] = a;
        }
        __syncthreads();
      }
    }
    for (int i = tid; i < k && i < nk; i += kRefineThreads) emit(i, kept[i]);
  }
  for (int i = nk + tid; i < k; i += kRefineThreads) {   // fewer than k database rows: faiss pads with inf / -1
    D[static_cast<int64_t>(q) * out_ld + i] = metric == 0 ? pos_inf() : neg_inf();
    I[static_cast<int64_t>(q) * out_ld + i] = -1;
  }
}

// Row-sharded index: a shard's query usually has a few hundred nominees of which a few dozen survive the GLOBAL prune bound.
// One warp per query then does what the block kernel above does with 256 threads and ~40 block barriers: nominees in
// registers (8 per lane), survivors compacted by ballot, exact fp32 re-rank four rows at a time, rank sort, emit.  Queries
// it does not take (no global bound, > 256 nominees, > kWarpKeep survivors) are left to the block kernel via handled[q] = 0.
constexpr int kWarpNom = 256;
constexpr int kWarpKeep = 96;
__global__ void __launch_bounds__(256)
knn_refine_warp_kernel(const float* __restrict__ Q, int64_t ldq, int d, const float* __restrict__ qss,
                       const float* __restrict__ X, int64_t ldx, const float* __restrict__ xss,
                       const int32_t* __restrict__ cand_idx, const float* __restrict__ cand_val,
                       const int32_t* __restrict__ cnt, int cap, int k, int metric, float slack_scale, float slack_abs,
                       int64_t id_offset, float* __restrict__ D, int64_t* __restrict__ I, int64_t out_ld,
                       const float* __restrict__ prune_pair, int64_t prune_ld, int64_t nq, int32_t* __restrict__ handled) {
  __shared__ unsigned long long kept_all[8][kWarpKeep];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t q = static_cast<int64_t>(blockIdx.x) * 8 + warp;
  if (q >= nq) return;
  unsigned long long* kept = kept_all[warp];
  const int n = cnt[q];
  const float tg = fmaxf(prune_pair[q], -prune_pair[prune_ld + q]);
  if (n > kWarpNom || n > cap || !(tg > neg_inf())) {
    if (lane == 0) handled[q] = 0;
    return;
  }
  const float slack = slack_scale * sqrtf(qss[q]) + slack_abs;
  const uint32_t keep_key = f2key(tg - slack);
  int nk = 0;
#pragma unroll
  for (int t = 0; t < kWarpNom / 32; ++t) {
    const int i = lane + 32 * t;
    const bool pass = i < n && f2key(cand_val[q * cap + i]) >= keep_key;
    const unsigned int m = __ballot_sync(0xffffffffu, pass);
    const int pos = nk + __popc(m & ((1u << lane) - 1u));
    if (pass && pos < kWarpKeep) kept[pos] = static_cast<unsigned long long>(static_cast<uint32_t>(cand_idx[q * cap + i]));
    nk += __popc(m);
  }
  if (nk > kWarpKeep) {
    if (lane == 0) handled[q] = 0;
    return;
  }
  __syncwarp();
  const float* qv = Q + q * ldq;
  const float qn = qss[q];
  const bool vec = (d & 3) == 0 && (ldx & 3) == 0 && (ldq & 3) == 0 &&
                   ((reinterpret_cast<uintptr_t>(X) | reinterpret_cast<uintptr_t>(Q)) & 15) == 0;
  for (int i0 = 0; i0 < nk; i0 += 4) {
    uint32_t id[4];
    float dot[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int c = 0; c < 4; ++c) id[c] = static_cast<uint32_t>(kept[min(i0 + c, nk - 1)]);
    if (vec) {
      for (int j = lane * 4; j < d; j += 128) {
        const float4 qq = __ldg(reinterpret_cast<const float4*>(qv + j));
        float4 xx[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) xx[c] = __ldg(reinterpret_cast<const float4*>(X + static_cast<int64_t>(id[c]) * ldx + j));
#pragma unroll
        for (int c = 0; c < 4; ++c)
          dot[c] = fmaf(qq.x, xx[c].x, fmaf(qq.y, xx[c].y, fmaf(qq.z, xx[c].z, fmaf(qq.w, xx[c].w, dot[c]))));
      }
    } else {
      for (int j = lane; j < d; j += 32) {
        const float qj = qv[j];
#pragma unroll
        for (int c = 0; c < 4; ++c) dot[c] = fmaf(qj, X[static_cast<int64_t>(id[c]) * ldx + j], dot[c]);
      }
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) dot[c] += __shfl_xor_sync(0xffffffffu, dot[c], o);
    }
    __syncwarp();
    if (lane < 4 && i0 + lane < nk) {
      const float dsel = lane == 0 ? dot[0] : lane == 1 ? dot[1] : lane == 2 ? dot[2] : dot[3];
      const uint32_t isel = lane == 0 ? id[0] : lane == 1 ? id[1] : lane == 2 ? id[2] : id[3];
      const float key = metric == 0 ? fmaxf(qn + xss[isel] - 2.f * dsel, 0.f) : -dsel;
      kept[i0 + lane] = (static_cast<unsigned long long>(f2key(key)) << 32) | isel;
    }
    __syncwarp();
  }
  for (int i = lane; i < nk; i += 32) {      // rank sort on (distance key, id): the keys are distinct
    const unsigned long long e = kept[i];
    int rank = 0;
    for (int j = 0; j < nk; ++j) rank += kept[j] < e ? 1 : 0;
    if (rank < k) {
      const float key = key2f(static_cast<uint32_t>(e >> 32));
      D[q * out_ld + rank] = metric == 0 ? key : -key;
      I[q * out_ld + rank] = static_cast<int64_t>(static_cast<uint32_t>(e)) + id_offset;
    }
  }
  for (int i = nk + lane; i < k; i += 32) {
    D[q * out_ld + i] = metric == 0 ? pos_inf() : neg_inf();
    I[q * out_ld + i] = -1;
  }
  if (lane == 0) handled[q] = 1;
}

// ---- exact fallback: queries whose candidate list overflowed (dense near-tie bands, e.g. tight clusters) ----
// One CTA takes up to kFbQueries such queries and streams the whole index once in fp32 (every row fetch is shared by
// the CTA's queries); per query a shared-memory buffer of 2*kcap (distance,id) keys collects the rows that beat the
// running k-th best and is compacted (bitonic sort, keep k) whenever it may overflow in the next round.  All overflow
// queries of a search run in ONE launch with no host round trips (the former per-query scan + select took ~2 ms each).
constexpr int kFbQueries = 8;
constexpr int kFbThreads = 256;
constexpr int kFbRound = (kFbThreads / 32) * 32;   // rows examined between two block barriers

__global__ void __launch_bounds__(kFbThreads)
knn_exact_batch_kernel(const int32_t* __restrict__ qlist, int nlist, const float* __restrict__ Q, int64_t ldq, int d,
                       const float* __restrict__ X, int64_t N, int64_t ldx, const float* __restrict__ xss, int metric,
                       int k, int kcap, int64_t id_offset, float* __restrict__ D, int64_t* __restrict__ I, int compact_out) {
  // gridDim.y row splits: this CTA scans rows [row_lo, row_hi); with compact_out the lists go to [split, list slot, k]
  // (merged afterwards by knn_merge_kernel), otherwise straight to the queries' rows of D / I
  extern __shared__ unsigned long long fb_smem[];
  unsigned long long* buf = fb_smem;                                   // [kFbQueries][2*kcap]
  float* qs = reinterpret_cast<float*>(buf + kFbQueries * 2 * kcap);   // [kFbQueries][d]
  __shared__ uint32_t thr_key[kFbQueries];                             // key of the running k-th best distance
  __shared__ int cnt[kFbQueries];
  __shared__ float qnorm[kFbQueries];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q0 = blockIdx.x * kFbQueries;
  const int nqs = min(kFbQueries, nlist - q0);
  const int cap = 2 * kcap;
  for (int i = tid; i < kFbQueries * d; i += kFbThreads) {
    const int j = i / d;
    qs[i] = j < nqs ? Q[static_cast<int64_t>(qlist[q0 + j]) * ldq + (i - j * d)] : 0.f;
  }
  if (tid < kFbQueries) thr_key[tid] = 0xffffffffu, cnt[tid] = 0;
  __syncthreads();
  if (warp < kFbQueries) {
    float a = 0.f;
    for (int c = lane; c < d; c += 32) a = fmaf(qs[warp * d + c], qs[warp * d + c], a);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) qnorm[warp] = a;
  }
  __syncthreads();
  auto compact = [&](int j) {   // block-wide: keep the k smallest keys of query j's buffer
    const int n = min(cnt[j], cap);
    unsigned long long* b = buf + static_cast<size_t>(j) * cap;
    int P = 2;
    while (P < n) P <<= 1;
    for (int i = n + tid; i < P; i += kFbThreads) b[i] = ~0ull;
    __syncthreads();
    for (int size = 2; size <= P; size <<= 1)
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        for (int t = tid; t < (P >> 1); t += kFbThreads) {
          const int lo = ((t / stride) * (stride << 1)) + (t % stride), hi = lo + stride;
          const bool up = (lo & size) == 0;
          const unsigned long long x = b[lo], y = b[hi];
          if ((x > y) == up) b[lo] = y, b[hi] = x;
        }
        __syncthreads();
      }
    if (tid == 0) {
      const int keep = min(n, k);
      cnt[j] = keep;
      if (keep == k) thr_key[j] = static_cast<uint32_t>(b[k - 1] >> 32);
    }
    __syncthreads();
  };
  const int64_t row_lo = N * blockIdx.y / gridDim.y, row_hi = N * (blockIdx.y + 1) / gridDim.y;
  float qreg[kFbQueries][8];   // this lane's columns (lane + 32p) of the CTA's queries, d <= 256
#pragma unroll
  for (int j = 0; j < kFbQueries; ++j)
#pragma unroll
    for (int p = 0; p < 8; ++p) qreg[j][p] = (d <= 256 && lane + 32 * p < d) ? qs[j * d + lane + 32 * p] : 0.f;
  for (int64_t r0 = row_lo; r0 < row_hi; r0 += kFbRound) {
    // each warp: 32 consecutive rows of the round, lane <-> columns.  d <= 256: the queries' pieces live in registers
    // (qreg, loaded once) and four rows are fetched together -- the scan is bound by row-fetch latency otherwise.
    auto offer = [&](int64_t r, const float (&dot)[kFbQueries]) {
      if (lane < nqs) {
        float dsel = dot[0];
#pragma unroll
        for (int j = 1; j < kFbQueries; ++j) dsel = lane == j ? dot[j] : dsel;
        const float key = metric == 0 ? fmaxf(qnorm[lane] + xss[r] - 2.f * dsel, 0.f) : -dsel;
        const uint32_t kk = f2key(key);
        if (kk <= thr_key[lane]) {   // ties with the running k-th best stay candidates: (distance,id) decides later
          const int pos = atomicAdd(&cnt[lane], 1);
          if (pos < cap) buf[static_cast<size_t>(lane) * cap + pos] = (static_cast<unsigned long long>(kk) << 32) | static_cast<uint32_t>(r);
        }
      }
    };
    if (d <= 256) {
      for (int rr = 0; rr < 32; rr += 4) {
        const int64_t rb = r0 + warp * 32 + rr;
        if (rb >= row_hi) break;
        float x[4][8];
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          const float* xv = X + min(rb + a, row_hi - 1) * ldx;
#pragma unroll
          for (int p = 0; p < 8; ++p) x[a][p] = lane + 32 * p < d ? __ldg(xv + lane + 32 * p) : 0.f;
        }
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          float dot[kFbQueries];
#pragma unroll
          for (int j = 0; j < kFbQueries; ++j) {
            float t = 0.f;
#pragma unroll
            for (int p = 0; p < 8; ++p) t = fmaf(x[a][p], qreg[j][p], t);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
            dot[j] = t;
          }
          if (rb + a < row_hi) offer(rb + a, dot);
        }
      }
    } else {
      for (int rr = 0; rr < 32; ++rr) {
        const int64_t r = r0 + warp * 32 + rr;
        if (r >= row_hi) break;
        const float* xv = X + r * ldx;
        float dot[kFbQueries];
#pragma unroll
        for (int j = 0; j < kFbQueries; ++j) dot[j] = 0.f;
        for (int c = lane; c < d; c += 32) {
          const float x = __ldg(xv + c);
#pragma unroll
          for (int j = 0; j < kFbQueries; ++j) dot[j] = fmaf(x, qs[j * d + c], dot[j]);
        }
#pragma unroll
        for (int j = 0; j < kFbQueries; ++j) {
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) dot[j] += __shfl_xor_sync(0xffffffffu, dot[j], o);
        }
        offer(r, dot);
      }
    }
    __syncthreads();
    unsigned int need = 0u;   // latched by every thread BEFORE anyone appends again: the decision must be block-uniform
    for (int j = 0; j < nqs; ++j) need |= (cnt[j] + kFbRound > cap ? 1u : 0u) << j;
    __syncthreads();
    for (int j = 0; j < nqs; ++j)
      if ((need >> j) & 1u) compact(j);
  }
  for (int j = 0; j < nqs; ++j) {
    compact(j);
    const int64_t q = compact_out ? static_cast<int64_t>(blockIdx.y) * nlist + q0 + j : qlist[q0 + j];
    const int have = cnt[j];
    for (int i = tid; i < k; i += kFbThreads) {
      if (i < have) {
        const unsigned long long e = buf[static_cast<size_t>(j) * cap + i];
        const float key = key2f(static_cast<uint32_t>(e >> 32));
        D[q * k + i] = metric == 0 ? key : -key;
        I[q * k + i] = static_cast<int64_t>(static_cast<uint32_t>(e)) + id_offset;
      } else {
        D[q * k + i] = metric == 0 ? pos_inf() : neg_inf();
        I[q * k + i] = -1;
      }
    }
    __syncthreads();
  }
}

__global__ void knn_scatter_rows_kernel(const int32_t* __restrict__ qlist, int nlist, int k, const float* __restrict__ Dm,
                                        const int64_t* __restrict__ Im, float* __restrict__ D, int64_t* __restrict__ I) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<int64_t>(nlist) * k) return;
  const int64_t q = qlist[i / k];
  D[q * k + i % k] = Dm[i], I[q * k + i % k] = Im[i];
}

// ---- sharded merge: [G, nq, k] -> top-k by (distance, id) ----
__global__ void __launch_bounds__(256)
knn_merge_kernel(const float* __restrict__ Dg, const int64_t* __restrict__ Ig, int G, int64_t nq, int k, int metric,
                 float* __restrict__ D, int64_t* __restrict__ I) {
  extern __shared__ unsigned long long mk[];  // P composite keys + P payload slots
  const int64_t q = blockIdx.x;
  const int tid = threadIdx.x;
  const int n = G * k;
  int P = 2;
  while (P < n) P <<= 1;
  unsigned long long* key = mk;
  int* src = reinterpret_cast<int*>(mk + P);
  for (int i = tid; i < P; i += 256) {
    if (i < n) {
      const int g = i / k, j = i % k;
      const int64_t off = (static_cast<int64_t>(g) * nq + q) * k + j;
      const int64_t id = Ig[off];
      const float dv = Dg[off];
      // rank by (distance, id); ids fit 32 bits per shard set of < 2^32 rows
      key[i] = id < 0 ? ~0ull : ((static_cast<unsigned long long>(f2key(metric == 0 ? dv : -dv)) << 32) |
                                 static_cast<uint32_t>(id));
    } else {
      key[i] = ~0ull;
    }
    src[i] = i;
  }
  __syncthreads();
  for (int size = 2; size <= P; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = tid; t < (P >> 1); t += 256) {
        const int lo = ((t / stride) * (stride << 1)) + (t % stride);
        const int hi = lo + stride;
        const bool up = (lo & size) == 0;
        const unsigned long long a = key[lo], b = key[hi];
        if ((a > b) == up) {
          key[lo] = b, key[hi] = a;
          const int s = src[lo];
          src[lo] = src[hi], src[hi] = s;
        }
      }
      __syncthreads();
    }
  }
  for (int i = tid; i < k; i += 256) {
    const int s = src[i];
    if (key[i] != ~0ull && s < n) {
      const int g = s / k, j = s % k;
      const int64_t off = (static_cast<int64_t>(g) * nq + q) * k + j;
      D[q * k + i] = Dg[off];
      I[q * k + i] = Ig[off];
    } else {
      D[q * k + i] = metric == 0 ? pos_inf() : neg_inf();
      I[q * k + i] = -1;
    }
  }
}

__global__ void knn_any_overflow_kernel(const int32_t* __restrict__ overflow, int64_t n, const int32_t* __restrict__ log_overflow,
                                        int32_t* __restrict__ flag) {
  int any = (threadIdx.x == 0 && *log_overflow != 0) ? 1 : 0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) any |= overflow[i] != 0 ? 1 : 0;
  if (__syncthreads_or(any) && threadIdx.x == 0) *flag = 1;
}

// (D, I) lists -> one sortable 64-bit record per entry: (order-preserving distance key << 32) | global id; padding
// (id < 0) -> ~0.  One record array makes the shard exchange ONE all-to-all of 8 bytes per entry instead of two of 4 + 8.
__global__ void knn_pack_kernel(const float* __restrict__ D, const int64_t* __restrict__ I, int64_t n, int metric,
                                unsigned long long* __restrict__ rec) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t id = I[i];
  const float dv = D[i];
  rec[i] = id < 0 ? ~0ull : ((static_cast<unsigned long long>(f2key(metric == 0 ? dv : -dv)) << 32) | static_cast<uint32_t>(id));
}

__global__ void knn_unpack_kernel(const unsigned long long* __restrict__ rec, int64_t n, int metric, float* __restrict__ D,
                                  int64_t* __restrict__ I) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long e = rec[i];
  if (e == ~0ull) {
    D[i] = metric == 0 ? pos_inf() : neg_inf();
    I[i] = -1;
  } else {
    const float key = key2f(static_cast<uint32_t>(e >> 32));
    D[i] = metric == 0 ? key : -key;
    I[i] = static_cast<int64_t>(static_cast<uint32_t>(e));
  }
}

// k-way merge of G sorted record lists per query, one WARP per query: the lists are staged in shared memory with
// coalesced loads, lane g holds the head of list g, every round takes the warp-minimum head (records are distinct: the
// id is part of the key) and advances that list.  G <= 32.  [G, nq, k] records -> D, I [nq, k].
__global__ void __launch_bounds__(256)
knn_merge_packed_kernel(const unsigned long long* __restrict__ rec, int G, int64_t nq, int k, int metric, int warps,
                        float* __restrict__ D, int64_t* __restrict__ I, unsigned long long* __restrict__ rec_out) {
  extern __shared__ unsigned long long ms[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp >= warps) return;
  const int64_t q = static_cast<int64_t>(blockIdx.x) * warps + warp;
  if (q >= nq) return;
  unsigned long long* mine = ms + static_cast<size_t>(warp) * G * k;
  for (int g = 0; g < G; ++g)
    for (int j = lane; j < k; j += 32) mine[g * k + j] = rec[(static_cast<int64_t>(g) * nq + q) * k + j];
  __syncwarp();
  int pos = 0;
  unsigned long long head = lane < G ? mine[lane * k] : ~0ull;
  for (int i = 0; i < k; ++i) {
    const uint32_t hi = static_cast<uint32_t>(head >> 32);
    const uint32_t mhi = __reduce_min_sync(0xffffffffu, hi);
    const uint32_t lo = hi == mhi ? static_cast<uint32_t>(head) : 0xffffffffu;
    const uint32_t mlo = __reduce_min_sync(0xffffffffu, lo);
    const bool win = hi == mhi && static_cast<uint32_t>(head) == mlo && head != ~0ull;
    const unsigned int who = __ballot_sync(0xffffffffu, win);
    if (who == 0u) {          // every list exhausted: pad like faiss
      if (lane == 0) {
        if (rec_out != nullptr) {
          rec_out[q * k + i] = ~0ull;
        } else {
          D[q * k + i] = metric == 0 ? pos_inf() : neg_inf();
          I[q * k + i] = -1;
        }
      }
      continue;
    }
    if (lane == __ffs(who) - 1) {
      if (rec_out != nullptr) {   // merged list stays packed (one all-gather of 8-byte records instead of two of 4 + 8)
        rec_out[q * k + i] = head;
      } else {
        const float key = key2f(mhi);
        D[q * k + i] = metric == 0 ? key : -key;
        I[q * k + i] = static_cast<int64_t>(mlo);
      }
      ++pos;
      head = pos < k ? mine[lane * k + pos] : ~0ull;
    }
  }
}

template <typename T>
static int dev_alloc(T** p, size_t n) {
  CDML_CHECK_CUDA(cudaMalloc(reinterpret_cast<void**>(p), n * sizeof(T)));
  return 0;
}

}  // namespace cdml

using namespace cdml;

struct cdml_index {
  cdml_ctx* ctx;
  int64_t N;
  int d, dpad, metric;
  float* x32;      // [N, d] copy of the database
  float* xss;      // [N] exact ||x||^2
  float* h;        // [N] ||x||^2/2 (L2) or 0 (IP)
  uint16_t* x16;   // [N, dpad] fp16 operand
  int64_t Ns;      // sampled rows (0 = collect everything)
  uint16_t* xs16;  // [Ns, dpad]
  float* hs;       // [Ns]
  float xmaxnorm;
  // per-chunk workspace
  int64_t qc;
  uint16_t* q16;
  float *qss, *gmax, *thr, *cand_val;
  int32_t *cand_idx, *cnt, *overflow, *handled;
  uint4* log;          // [num_sms * 8, log_cap] warp-private candidate logs of pass B
  int32_t* log_count;  // [num_sms * 8] + 1 overflow word
  unsigned int log_cap;
  // pinned host mirrors of the per-query counters (one stream synchronisation per search, not per chunk)
  int32_t *h_cnt, *h_ovf, *h_logovf;
  float* h_qss;
  int64_t h_cap;
  int64_t ldg;
  int64_t stats[2];
  // row-sharded protocol: (D, I) of one chunk before they are packed into records
  float* Dtmp;
  int64_t* Itmp;
  int64_t tmp_cap;
};

static void index_free(cdml_index* ix) {
  if (ix == nullptr) return;
  cudaFree(ix->x32), cudaFree(ix->xss), cudaFree(ix->h), cudaFree(ix->x16), cudaFree(ix->xs16), cudaFree(ix->hs);
  cudaFree(ix->q16), cudaFree(ix->qss), cudaFree(ix->gmax), cudaFree(ix->thr), cudaFree(ix->cand_val);
  cudaFree(ix->cand_idx), cudaFree(ix->cnt), cudaFree(ix->overflow), cudaFree(ix->handled);
  cudaFree(ix->log), cudaFree(ix->log_count);
  cudaFree(ix->Dtmp), cudaFree(ix->Itmp);
  cudaFreeHost(ix->h_cnt), cudaFreeHost(ix->h_ovf), cudaFreeHost(ix->h_qss), cudaFreeHost(ix->h_logovf);
  delete ix;
}

extern "C" {

int cdml_knn_index_build(cdml_ctx* ctx, const float* X, int64_t N, int d, int64_t ldx, int metric, void* stream,
                         cdml_index** out) {
  CDML_REQUIRE(ctx && X && out, "cdml_knn_index_build: NULL argument");
  CDML_REQUIRE(N > 0 && N < (1ll << 31) && d > 0 && ldx >= d && (metric == 0 || metric == 1),
               "cdml_knn_index_build: bad geometry N=%lld d=%d", (long long)N, d);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cdml_index* ix = new cdml_index();
  memset(ix, 0, sizeof(*ix));
  ix->ctx = ctx, ix->N = N, ix->d = d, ix->dpad = (d + 7) / 8 * 8, ix->metric = metric;
  *out = nullptr;
  int rc = 0;
  rc |= dev_alloc(&ix->x32, static_cast<size_t>(N) * d);
  rc |= dev_alloc(&ix->xss, N + 1);
  rc |= dev_alloc(&ix->h, N);
  rc |= dev_alloc(&ix->x16, static_cast<size_t>(N) * ix->dpad);
  if (rc) { index_free(ix); return -2; }
  cudaError_t e = cudaMemcpy2DAsync(ix->x32, sizeof(float) * d, X, sizeof(float) * ldx, sizeof(float) * d, N,
                                    cudaMemcpyDeviceToDevice, st);
  if (e != cudaSuccess) { index_free(ix); set_error("index build copy failed: %s", cudaGetErrorString(e)); return -2; }
  const int grid = static_cast<int>(std::min<int64_t>((N + 7) / 8, ctx->num_sms * 8));
  row_sumsq32_kernel<<<grid, 256, 0, st>>>(ix->x32, N, d, d, ix->xss, metric == 0 ? 0.5f : 0.f, ix->h);
  max_reduce_kernel<<<1, 1024, 0, st>>>(ix->xss, N, ix->xss + N);
  rc = cdml_rows_normalize_cast(ctx, ix->x32, N, d, d, 0, 0.f, ix->x16, ix->dpad, CDML_F16, nullptr, 0, nullptr, stream);
  if (rc) { index_free(ix); return rc; }
  float maxss = 0.f;
  e = cudaMemcpyAsync(&maxss, ix->xss + N, sizeof(float), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) { index_free(ix); set_error("index build failed: %s", cudaGetErrorString(e)); return -2; }
  ix->xmaxnorm = sqrtf(maxss);
  // evenly spaced row sample for the bound pass (robust to any ordering of the database)
  if (N > kCandCap) {
    int64_t ns = std::max<int64_t>(N / 8, 4096);
    ns = std::min<int64_t>(std::min<int64_t>(ns, N), static_cast<int64_t>(kMaxGroups) * 32);
    ns = ns / 32 * 32;
    ix->Ns = ns;
    std::vector<int32_t> rows(ns);
    for (int64_t i = 0; i < ns; ++i) rows[i] = static_cast<int32_t>(i * N / ns);
    int32_t* drows = nullptr;
    rc |= dev_alloc(&drows, ns);
    rc |= dev_alloc(&ix->xs16, static_cast<size_t>(ns) * ix->dpad);
    rc |= dev_alloc(&ix->hs, ns);
    if (rc) { cudaFree(drows); index_free(ix); return -2; }
    cudaMemcpyAsync(drows, rows.data(), sizeof(int32_t) * ns, cudaMemcpyHostToDevice, st);
    rc = cdml_gather_rows(ctx, ix->x16, N, ix->dpad * 2, ix->dpad * 2, drows, 0, ns, ix->xs16, ix->dpad * 2, stream);
    if (!rc) rc = cdml_gather_rows(ctx, ix->h, N, 4, 4, drows, 0, ns, ix->hs, 4, stream);
    cudaStreamSynchronize(st);
    cudaFree(drows);
    if (rc) { index_free(ix); return rc; }
  }
  *out = ix;
  return 0;
}

int cdml_knn_index_destroy(cdml_index* index) {
  index_free(index);
  return 0;
}

int cdml_knn_last_stats(cdml_index* index, int64_t* stats) {
  CDML_REQUIRE(index && stats, "cdml_knn_last_stats: NULL argument");
  stats[0] = index->stats[0], stats[1] = index->stats[1];
  return 0;
}

static int ensure_workspace(cdml_index* ix, int64_t qc) {
  if (ix->qc >= qc) return 0;
  cudaFree(ix->q16), cudaFree(ix->qss), cudaFree(ix->gmax), cudaFree(ix->thr), cudaFree(ix->cand_val);
  cudaFree(ix->cand_idx), cudaFree(ix->cnt), cudaFree(ix->overflow), cudaFree(ix->log), cudaFree(ix->log_count);
  cudaFree(ix->handled);
  ix->handled = nullptr;
  ix->log = nullptr, ix->log_count = nullptr;
  ix->q16 = nullptr, ix->qss = ix->gmax = ix->thr = ix->cand_val = nullptr, ix->cand_idx = ix->cnt = ix->overflow = nullptr;
  ix->qc = 0;
  ix->ldg = ix->Ns > 0 ? ((ix->Ns / 32 + 7) / 8 * 8) : 8;
  int rc = 0;
  rc |= dev_alloc(&ix->q16, static_cast<size_t>(qc) * ix->dpad);
  rc |= dev_alloc(&ix->qss, qc);
  rc |= dev_alloc(&ix->gmax, static_cast<size_t>(qc) * ix->ldg);
  rc |= dev_alloc(&ix->thr, qc);
  rc |= dev_alloc(&ix->cand_val, static_cast<size_t>(qc) * kCandCap);
  rc |= dev_alloc(&ix->cand_idx, static_cast<size_t>(qc) * kCandCap);
  rc |= dev_alloc(&ix->cnt, qc);
  rc |= dev_alloc(&ix->overflow, qc);
  rc |= dev_alloc(&ix->handled, qc);
  // log capacity: 2048 nominees per query on average, never less than 16K entries per epilogue warp
  const int sms = ix->ctx->num_sms;
  ix->log_cap = static_cast<unsigned int>(std::max<int64_t>(qc * 2048 / (sms * kKnnLogsPerCta), 16384));
  rc |= dev_alloc(&ix->log, static_cast<size_t>(sms) * kKnnLogsPerCta * ix->log_cap);
  rc |= dev_alloc(&ix->log_count, sms * kKnnLogsPerCta + 1);
  if (rc) return -2;
  ix->qc = qc;
  return 0;
}

// One implementation, three uses:
//   search          (ext_full == nullptr, out_full == nullptr): bound pass + collect + refine, self-contained;
//   bounds only     (out_full != nullptr): bound pass; writes the raw k_full-th / k_part-th best sampled scores per query;
//   bounded search  (ext_full != nullptr): skips the bound pass, collects above max(ext_full, ext_part) - slack.
//   row-sharded protocol (one chunk of <= 65536 queries per call, the workspace carries the nominees between the calls;
//   a larger chunk than the self-contained search's 32768 because every chunk costs the shards two all-reduces):
//     phase 1 = cast + [bounded] collect + bin, then the nominee selection into nom_pair;  phase 2 = refine only, pruning
//     against prune_pair (the all-reduced nom_pair).  part_sign = -1: the `part` bounds travel negated (packed MAX all-reduce).
static int knn_run(cdml_ctx* ctx, cdml_index* ix, const float* Q, int64_t nq, int64_t ldq, int k, float* D, int64_t* I,
                   int64_t id_offset, void* stream, const float* ext_full, const float* ext_part, int k_part,
                   float* out_full, float* out_part, int phase = 0, float part_sign = 1.f, float* nom_pair = nullptr,
                   const float* prune_pair = nullptr, int32_t* defer_flag = nullptr) {
  const bool bounds_only = out_full != nullptr;
  CDML_REQUIRE((phase == 0 && !(bounds_only && part_sign < 0.f)) || nq <= 65536,
               "cdml_knn_shard_*: one chunk of at most 65536 queries per call (got %lld)", (long long)nq);
  CDML_REQUIRE(ctx && ix && Q && (bounds_only || phase == 1 || (D && I)), "cdml_knn_search: NULL argument");
  CDML_REQUIRE(nq >= 0 && ldq >= ix->d && k >= 1 && k <= 1024, "cdml_knn_search: bad arguments (k=%d, supported 1..1024)", k);
  CDML_REQUIRE(k <= kKeepCap / 2, "cdml_knn_search: k=%d exceeds the re-rank capacity %d", k, kKeepCap / 2);
  if (nq == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t chunk = std::min<int64_t>(nq, (phase != 0 || (bounds_only && part_sign < 0.f)) ? 65536 : 32768);
  int rc = ensure_workspace(ix, chunk);
  if (rc) { set_error("cdml_knn_search: workspace allocation failed"); return rc; }
  if (phase != 2) ix->stats[0] = ix->stats[1] = 0;
  const int d = ix->d;
  // rigorous bound of |fp16 tensor-core score - exact score| <= (2u+u^2)|q||x| + accumulation; u = 2^-11
  const float rel = 1.5f * 0.0009765625f + 1.2e-7f * d;            // operand rounding + fp32 accumulation
  const float slack_scale = 2.f * rel * ix->xmaxnorm;               // times |q|
  const float slack_abs = 2.f * 1e-6f * (1.f + ix->xmaxnorm);       // fp16 subnormal floor
  if (ix->h_cap < nq) {
    cudaFreeHost(ix->h_cnt), cudaFreeHost(ix->h_ovf), cudaFreeHost(ix->h_qss), cudaFreeHost(ix->h_logovf);
    ix->h_cnt = ix->h_ovf = ix->h_logovf = nullptr, ix->h_qss = nullptr, ix->h_cap = 0;
    CDML_CHECK_CUDA(cudaMallocHost(reinterpret_cast<void**>(&ix->h_cnt), sizeof(int32_t) * nq));
    CDML_CHECK_CUDA(cudaMallocHost(reinterpret_cast<void**>(&ix->h_ovf), sizeof(int32_t) * nq));
    CDML_CHECK_CUDA(cudaMallocHost(reinterpret_cast<void**>(&ix->h_qss), sizeof(float) * nq));
    CDML_CHECK_CUDA(cudaMallocHost(reinterpret_cast<void**>(&ix->h_logovf), sizeof(int32_t) * (nq / chunk + 2)));
    ix->h_cap = nq;
  }
  for (int64_t q0 = 0; q0 < nq; q0 += chunk) {
    const int64_t qc = std::min<int64_t>(chunk, nq - q0);
    const float* Qc = Q + q0 * ldq;
    const bool tiny = ix->N <= kKeepCap;   // tiny database: exact re-rank of every row, no tensor-core scan
    if (phase != 2) {
    rc = cdml_rows_normalize_cast(ctx, Qc, qc, d, ldq, 0, 0.f, ix->q16, ix->dpad, CDML_F16, nullptr, 0, nullptr, stream);
    if (rc) return rc;
    const int grid = static_cast<int>(std::min<int64_t>((qc + 7) / 8, ctx->num_sms * 8));
    row_sumsq32_kernel<<<grid, 256, 0, st>>>(Qc, qc, d, ldq, ix->qss, 0.f, nullptr);
    CDML_CHECK_CUDA(cudaMemsetAsync(ix->cnt, 0, sizeof(int32_t) * qc, st));
    CDML_CHECK_CUDA(cudaMemsetAsync(ix->overflow, 0, sizeof(int32_t) * qc, st));
    CDML_CHECK_CUDA(cudaMemsetAsync(ix->log_count, 0, sizeof(int32_t) * (ctx->num_sms * kKnnLogsPerCta + 1), st));
    if (bounds_only && (tiny || !(ix->Ns > 0 && ix->Ns / 32 >= k))) {   // no usable sample: no bound from this shard
      fill_f32_kernel<<<64, 256, 0, st>>>(out_full + q0, qc, -INFINITY);
      fill_f32_kernel<<<64, 256, 0, st>>>(out_part + q0, qc, -INFINITY * part_sign);
      continue;
    }
    }
    if (!tiny) {
     if (phase != 2) {
      if (ext_full != nullptr) {
        knn_thr_combine_kernel<<<static_cast<int>((qc + 255) / 256), 256, 0, st>>>(ext_full + q0, ext_part + q0, ix->qss, qc,
                                                                                slack_scale, slack_abs, ix->thr, part_sign);
      } else if (ix->Ns > 0 && ix->Ns / 32 >= k) {
        const int wide = (ix->Ns / 128 >= 2 * static_cast<int64_t>(k)) ? 1 : 0;
        const int groups = wide ? static_cast<int>((ix->Ns + 255) / 256 * 2) : static_cast<int>(ix->Ns / 32);
        EpiKnnGroupMax<kBN> ea{ix->hs, ix->gmax, ix->ldg, wide};
        if (resb_applicable(ix->dpad) && qc >= 8 * kBM)
          rc = launch_gemm_resb(ctx, ix->q16, ix->dpad, ix->xs16, ix->dpad, qc, ix->Ns, ix->dpad, CDML_F16, ea, st);
        else
          rc = launch_gemm<0, 0>(ctx, ix->q16, ix->dpad, ix->xs16, ix->dpad, qc, ix->Ns, ix->dpad, CDML_F16, 1, ea, st);
        if (rc < 0) return rc;
        auto kth = [&](int kk, int kk2, float sc, float ab, float* out, float* out2) {
          const int grid = static_cast<int>(qc);
          if (groups <= 1024) {          // one warp per query
            const int wgrid = static_cast<int>((qc + 7) / 8);
            if (out2) knn_kth_warp_kernel<true><<<wgrid, 256, 0, st>>>(ix->gmax, ix->ldg, groups, kk, kk2, ix->qss, qc, sc, ab, out, out2, part_sign);
            else knn_kth_warp_kernel<false><<<wgrid, 256, 0, st>>>(ix->gmax, ix->ldg, groups, kk, kk2, ix->qss, qc, sc, ab, out, out2, part_sign);
          } else if (groups <= 4 * kRefineThreads) {
            if (out2) knn_kth_kernel<4, true><<<grid, kRefineThreads, 0, st>>>(ix->gmax, ix->ldg, groups, kk, kk2, ix->qss, sc, ab, out, out2, part_sign);
            else knn_kth_kernel<4, false><<<grid, kRefineThreads, 0, st>>>(ix->gmax, ix->ldg, groups, kk, kk2, ix->qss, sc, ab, out, out2, part_sign);
          } else {
            constexpr int kP = kMaxGroups / kRefineThreads;
            if (out2) knn_kth_kernel<kP, true><<<grid, kRefineThreads, 0, st>>>(ix->gmax, ix->ldg, groups, kk, kk2, ix->qss, sc, ab, out, out2, part_sign);
            else knn_kth_kernel<kP, false><<<grid, kRefineThreads, 0, st>>>(ix->gmax, ix->ldg, groups, kk, kk2, ix->qss, sc, ab, out, out2, part_sign);
          }
        };
        if (bounds_only) {   // raw scores: the caller combines them across shards
          kth(k, std::max(1, std::min(k_part, k)), 0.f, 0.f, out_full + q0, out_part + q0);
          CDML_CHECK_CUDA(cudaGetLastError());
          continue;
        }
        kth(k, k, slack_scale, slack_abs, ix->thr, nullptr);
      } else {
        fill_f32_kernel<<<64, 256, 0, st>>>(ix->thr, qc, -INFINITY);
      }
      EpiKnnCollect<kBN> eb{ix->h, ix->thr, ix->log, ix->log_count, ix->log_count + ctx->num_sms * kKnnLogsPerCta, ix->log_cap};
      if (resb_applicable(ix->dpad) && ix->N >= 8 * kBM)
        rc = launch_gemm_resb(ctx, ix->x16, ix->dpad, ix->q16, ix->dpad, ix->N, qc, ix->dpad, CDML_F16, eb, st, 1);   // column block fastest: 14.4 vs 16.2 ms
      else
        rc = launch_gemm<0, 0>(ctx, ix->x16, ix->dpad, ix->q16, ix->dpad, ix->N, qc, ix->dpad, CDML_F16, 1, eb, st);
      if (rc < 0) return rc;
      knn_bin_kernel<<<dim3(4, ctx->num_sms * kKnnLogsPerCta), 256, 0, st>>>(ix->log, ix->log_count, ix->log_cap, ix->cand_idx, ix->cand_val,
                                                            ix->cnt, kCandCap);
     }
      if (phase == 1) {   // nominees stay in the workspace; their k-th / k_part-th best scores go to the caller's all-reduce
        knn_nominee_kth_kernel<<<static_cast<int>((qc + 7) / 8), 256, 0, st>>>(ix->cand_val, ix->cnt, kCandCap, k,
                                                                              std::max(1, std::min(k_part, k)), qc, nom_pair);
        CDML_CHECK_CUDA(cudaGetLastError());
        continue;
      }
      if (prune_pair != nullptr)    // the common case of a shard: few nominees, a global bound -> one warp per query
        knn_refine_warp_kernel<<<static_cast<int>((qc + 7) / 8), 256, 0, st>>>(
            Qc, ldq, d, ix->qss, ix->x32, d, ix->xss, ix->cand_idx, ix->cand_val, ix->cnt, kCandCap, k, ix->metric,
            slack_scale, slack_abs, id_offset, D + q0 * k, I + q0 * k, k, prune_pair, qc, qc, ix->handled);
      knn_refine_kernel<<<static_cast<int>(qc), kRefineThreads, 0, st>>>(
          Qc, ldq, d, ix->qss, ix->x32, d, ix->xss, ix->cand_idx, ix->cand_val, ix->cnt, kCandCap, k, ix->metric,
          slack_scale, slack_abs, id_offset, D + q0 * k, I + q0 * k, k, ix->overflow, 0, prune_pair, qc,
          prune_pair != nullptr ? ix->handled : nullptr);
    } else {
      if (phase == 1) {   // tiny shard: every row is re-ranked exactly in phase 2, no bound to contribute
        fill_f32_kernel<<<64, 256, 0, st>>>(nom_pair, qc, -INFINITY);
        fill_f32_kernel<<<64, 256, 0, st>>>(nom_pair + qc, qc, INFINITY);
        CDML_CHECK_CUDA(cudaGetLastError());
        continue;
      }
      knn_refine_kernel<<<static_cast<int>(qc), kRefineThreads, 0, st>>>(
          Qc, ldq, d, ix->qss, ix->x32, d, ix->xss, ix->cand_idx, ix->cand_val, ix->cnt, kCandCap, k, ix->metric,
          slack_scale, slack_abs, id_offset, D + q0 * k, I + q0 * k, k, ix->overflow, static_cast<int>(ix->N), nullptr, 0, nullptr);
      ix->stats[0] += ix->N * qc;
    }
    CDML_CHECK_CUDA(cudaGetLastError());
    // counters of this chunk -> pinned host memory, stream-ordered before the next chunk reuses the workspace
    CDML_CHECK_CUDA(cudaMemcpyAsync(ix->h_cnt + q0, ix->cnt, sizeof(int32_t) * qc, cudaMemcpyDeviceToHost, st));
    CDML_CHECK_CUDA(cudaMemcpyAsync(ix->h_ovf + q0, ix->overflow, sizeof(int32_t) * qc, cudaMemcpyDeviceToHost, st));
    CDML_CHECK_CUDA(cudaMemcpyAsync(ix->h_qss + q0, ix->qss, sizeof(float) * qc, cudaMemcpyDeviceToHost, st));
    CDML_CHECK_CUDA(cudaMemcpyAsync(ix->h_logovf + q0 / chunk, ix->log_count + ctx->num_sms * kKnnLogsPerCta, sizeof(int32_t),
                                    cudaMemcpyDeviceToHost, st));
  }
  if (bounds_only || phase == 1) return 0;
  if (defer_flag != nullptr) {
    // deferred check (row-sharded protocol): no host synchronisation here.  Whether ANY query of this call overflowed its
    // candidate list or a warp log goes into the caller's device word; the caller looks at it once, after the exchange
    // that follows, and only then repeats the search synchronously (exact fallback) -- the common case never stalls.
    knn_any_overflow_kernel<<<1, 1024, 0, st>>>(ix->overflow, nq, ix->log_count + ctx->num_sms * kKnnLogsPerCta, defer_flag);
    CDML_CHECK_CUDA(cudaGetLastError());
    return 0;
  }
  CDML_CHECK_CUDA(cudaStreamSynchronize(st));
  // queries whose candidate list (or whose chunk's warp log) overflowed are redone exactly in fp32, all in one launch
  std::vector<int32_t> redo;
  for (int64_t i = 0; i < nq; ++i) {
    ix->stats[0] += ix->N <= kKeepCap ? 0 : ix->h_cnt[i];
    if (ix->h_ovf[i] || ix->h_logovf[i / chunk]) redo.push_back(static_cast<int32_t>(i));   // a full warp log may have dropped nominees of any query
  }
  ix->stats[1] = static_cast<int64_t>(redo.size());
  if (!redo.empty()) {
    int kcap = 64;
    while (kcap < k) kcap <<= 1;
    kcap = std::max(kcap, kFbRound);      // a round may append up to kFbRound rows per query before the next compaction
    const size_t smem = static_cast<size_t>(kFbQueries) * 2 * kcap * sizeof(unsigned long long) + static_cast<size_t>(kFbQueries) * d * sizeof(float);
    CDML_REQUIRE(smem <= 200 * 1024, "cdml_knn_search: exact fallback needs %zu bytes of shared memory (k=%d, d=%d)", smem, k, d);
    CDML_CHECK_CUDA(cudaFuncSetAttribute(knn_exact_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    int32_t* dlist = nullptr;
    if (dev_alloc(&dlist, redo.size())) return -2;
    CDML_CHECK_CUDA(cudaMemcpyAsync(dlist, redo.data(), sizeof(int32_t) * redo.size(), cudaMemcpyHostToDevice, st));
    const int nlist = static_cast<int>(redo.size());
    const int blocks = (nlist + kFbQueries - 1) / kFbQueries;
    // few overflow queries: split the index rows over several CTAs per query group so that the whole GPU scans
    int splits = std::max(1, std::min(16, (2 * ctx->num_sms + blocks - 1) / blocks));
    if (ix->N < 64 * 1024) splits = 1;
    float* Dp = nullptr;
    int64_t* Ip = nullptr;
    if (splits > 1 && (dev_alloc(&Dp, static_cast<size_t>(splits + 1) * nlist * k) || dev_alloc(&Ip, static_cast<size_t>(splits + 1) * nlist * k))) {
      cudaFree(dlist), cudaFree(Dp);
      return -2;
    }
    knn_exact_batch_kernel<<<dim3(blocks, splits), kFbThreads, smem, st>>>(dlist, nlist, Q, ldq, d, ix->x32, ix->N, d, ix->xss,
                                                                          ix->metric, k, kcap, id_offset, splits > 1 ? Dp : D,
                                                                          splits > 1 ? Ip : I, splits > 1 ? 1 : 0);
    CDML_CHECK_CUDA(cudaGetLastError());
    if (splits > 1) {   // per-split lists -> top-k (same merge kernel as the sharded index) -> the queries' rows
      float* Dm = Dp + static_cast<size_t>(splits) * nlist * k;
      int64_t* Im = Ip + static_cast<size_t>(splits) * nlist * k;
      int rcm = cdml_knn_merge(ctx, Dp, Ip, splits, nlist, k, ix->metric, Dm, Im, stream);
      if (rcm) { cudaFree(dlist), cudaFree(Dp), cudaFree(Ip); return rcm; }
      const int64_t tot = static_cast<int64_t>(nlist) * k;
      knn_scatter_rows_kernel<<<static_cast<int>((tot + 255) / 256), 256, 0, st>>>(dlist, nlist, k, Dm, Im, D, I);
      CDML_CHECK_CUDA(cudaGetLastError());
    }
    CDML_CHECK_CUDA(cudaStreamSynchronize(st));   // `redo` (pageable) and the scratch buffers must outlive the kernels
    cudaFree(dlist), cudaFree(Dp), cudaFree(Ip);
  }
  return 0;
}

int cdml_knn_search(cdml_ctx* ctx, cdml_index* ix, const float* Q, int64_t nq, int64_t ldq, int k, float* D,
                    int64_t* I, int64_t id_offset, void* stream) {
  return knn_run(ctx, ix, Q, nq, ldq, k, D, I, id_offset, stream, nullptr, nullptr, k, nullptr, nullptr);
}

int cdml_knn_bounds(cdml_ctx* ctx, cdml_index* ix, const float* Q, int64_t nq, int64_t ldq, int k_full, int k_part,
                    float* bound_full, float* bound_part, void* stream) {
  CDML_REQUIRE(bound_full && bound_part && k_part >= 1, "cdml_knn_bounds: NULL / bad argument");
  return knn_run(ctx, ix, Q, nq, ldq, k_full, nullptr, nullptr, 0, stream, nullptr, nullptr, k_part, bound_full, bound_part);
}

int cdml_knn_search_bounded(cdml_ctx* ctx, cdml_index* ix, const float* Q, int64_t nq, int64_t ldq, int k,
                            const float* bound_full, const float* bound_part, float* D, int64_t* I, int64_t id_offset,
                            void* stream) {
  CDML_REQUIRE(bound_full && bound_part, "cdml_knn_search_bounded: NULL bounds");
  return knn_run(ctx, ix, Q, nq, ldq, k, D, I, id_offset, stream, bound_full, bound_part, k, nullptr, nullptr);
}

// ---- row-sharded protocol, one chunk (<= 65536 queries) per call -------------------------------------------------
int cdml_knn_shard_bounds(cdml_ctx* ctx, cdml_index* ix, const float* Q, int64_t nq, int64_t ldq, int k, int k_part,
                          float* pair, void* stream) {
  CDML_REQUIRE(pair && k_part >= 1, "cdml_knn_shard_bounds: NULL / bad argument");
  return knn_run(ctx, ix, Q, nq, ldq, k, nullptr, nullptr, 0, stream, nullptr, nullptr, k_part, pair, pair + nq, 0, -1.f);
}

int cdml_knn_shard_collect(cdml_ctx* ctx, cdml_index* ix, const float* Q, int64_t nq, int64_t ldq, int k, int k_part,
                           const float* pair, float* nom_pair, void* stream) {
  CDML_REQUIRE(pair && nom_pair && k_part >= 1, "cdml_knn_shard_collect: NULL / bad argument");
  return knn_run(ctx, ix, Q, nq, ldq, k, nullptr, nullptr, 0, stream, pair, pair + nq, k_part, nullptr, nullptr, 1, -1.f,
                 nom_pair);
}

int cdml_knn_shard_refine(cdml_ctx* ctx, cdml_index* ix, const float* Q, int64_t nq, int64_t ldq, int k,
                          const float* nom_pair, unsigned long long* rec, int64_t id_offset, int32_t* overflow_flag,
                          void* stream) {
  CDML_REQUIRE(ix && rec, "cdml_knn_shard_refine: NULL argument");
  CDML_REQUIRE(id_offset >= 0 && id_offset + ix->N <= (1ll << 32) - 1, "cdml_knn_shard_refine: global ids must fit 32 bits");
  if (ix->tmp_cap < nq * k) {
    cudaFree(ix->Dtmp), cudaFree(ix->Itmp);
    ix->Dtmp = nullptr, ix->Itmp = nullptr, ix->tmp_cap = 0;
    if (dev_alloc(&ix->Dtmp, static_cast<size_t>(nq) * k) || dev_alloc(&ix->Itmp, static_cast<size_t>(nq) * k)) return -2;
    ix->tmp_cap = nq * k;
  }
  int rc = knn_run(ctx, ix, Q, nq, ldq, k, ix->Dtmp, ix->Itmp, id_offset, stream, nullptr, nullptr, k, nullptr, nullptr, 2, -1.f,
                   nullptr, nom_pair, overflow_flag);
  if (rc) return rc;
  const int64_t n = nq * k;
  knn_pack_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(ix->Dtmp, ix->Itmp, n, ix->metric, rec);
  CDML_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int cdml_knn_unpack_records(cdml_ctx* ctx, const unsigned long long* rec, int64_t n, int metric, float* D, int64_t* I,
                            void* stream) {
  CDML_REQUIRE(ctx && rec && D && I && n >= 0, "cdml_knn_unpack_records: bad argument");
  if (n == 0) return 0;
  knn_unpack_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(rec, n, metric, D, I);
  CDML_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int cdml_knn_merge_packed(cdml_ctx* ctx, const unsigned long long* rec, int G, int64_t nq, int k, int metric, float* D,
                          int64_t* I, unsigned long long* rec_out, void* stream) {
  CDML_REQUIRE(ctx && rec && ((D && I) || rec_out) && G >= 1 && G <= 32 && k >= 1 && nq >= 0,
               "cdml_knn_merge_packed: bad argument (1 <= G <= 32)");
  if (nq == 0) return 0;
  const size_t per = static_cast<size_t>(G) * k * sizeof(unsigned long long);
  CDML_REQUIRE(per <= 200 * 1024, "cdml_knn_merge_packed: G*k=%d too large for one warp's staging", G * k);
  const int warps = static_cast<int>(std::max<size_t>(1, std::min<size_t>(8, (96 * 1024) / per)));
  const size_t smem = per * warps;
  if (smem > 48 * 1024)
    CDML_CHECK_CUDA(cudaFuncSetAttribute(knn_merge_packed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  knn_merge_packed_kernel<<<static_cast<unsigned>((nq + warps - 1) / warps), 256, smem, static_cast<cudaStream_t>(stream)>>>(
      rec, G, nq, k, metric, warps, D, I, rec_out);
  CDML_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int cdml_knn_merge(cdml_ctx* ctx, const float* Dg, const int64_t* Ig, int G, int64_t nq, int k, int metric, float* D,
                   int64_t* I, void* stream) {
  CDML_REQUIRE(ctx && Dg && Ig && D && I && G >= 1 && k >= 1 && nq >= 0, "cdml_knn_merge: bad argument");
  if (nq == 0) return 0;
  int P = 2;
  while (P < G * k) P <<= 1;
  const size_t smem = static_cast<size_t>(P) * (sizeof(unsigned long long) + sizeof(int));
  CDML_REQUIRE(smem <= 200 * 1024, "cdml_knn_merge: G*k=%d too large for one block", G * k);
  if (smem > 48 * 1024)
    CDML_CHECK_CUDA(cudaFuncSetAttribute(knn_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  knn_merge_kernel<<<static_cast<unsigned>(nq), 256, smem, static_cast<cudaStream_t>(stream)>>>(Dg, Ig, G, nq, k, metric, D, I);
  CDML_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"
