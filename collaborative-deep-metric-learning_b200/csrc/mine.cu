// In-batch semi-hard negative mining (SURVEY.md 8a row M; build-defined, the reference draws negatives at random).
//
// For triplet i with dp = |a_i - p_i|^2, over the candidate rows r = 3j+1, 3j+2 (positives and negatives of the
// batch) whose guid is neither a_i nor p_i:
//   (1) argmin d(a_i, r) with dp < d < dp + margin, else (2) argmin d with d >= dp + margin, else (3) keep row 3i+2.
// The B x 2B distance matrix is a tcgen05 GEMM (anchors x candidates, fp16 operands) whose epilogue keeps a running
// (distance,row) minimum per anchor and folds it into a global 64-bit key with atomicMin, so the matrix
// never reaches HBM.  d = 2 - 2 a.c (unit-norm embeddings).  Ties -> lowest row.
#include <algorithm>

#include "gemm_launch.cuh"

namespace cdml {

constexpr unsigned long long kNoCand = ~0ull;
constexpr int kMassHits = 4;   // rows of a warp hitting in one chunk from which the per-thread re-scan takes over

// epilogue warps of the mining scans: 8 (two per TMEM lane quarter).  CDML_MINE_EPI_WARPS=16 selects four per quarter (A/B
// measurement aid): measured on B200 it is SLOWER (4.28 vs 4.02 ms structureless, 4.24 vs 3.94 ms clustered for both scans) --
// the epilogue is not short of warps; see DESIGN.md section 4.4
static int epi_warps() {
  static int w = -1;
  if (w < 0) {
    const char* e = getenv("CDML_MINE_EPI_WARPS");
    w = (e != nullptr && e[0] == '1') ? 16 : 8;
  }
  return w;
}

// (1)/(2) collapse into ONE criterion: the chosen row is argmin d over valid candidates with d > dp -- if that minimum
// is below dp+margin it is the semi-hard pick, otherwise it is exactly the closest beyond-margin pick.
// Common path per score: d = 2-2s, keep min over (d > dp).  Only when a 32-column chunk can beat the anchor's current
// best (a bound read from the global key at tile start; rare after the first tiles) are guids checked and the row
// recorded.  Result: 64-bit key (float bits of d << 32 | row) folded with atomicMin -> ties go to the lowest row.
template <int BN, int kVariant = 0>
struct EpiMine {
  static constexpr bool kSplitColumns = true;
  static constexpr bool kPrefetchNext = (kVariant & 1) == 0;   // pre() only loads the anchor's constants into registers
  // resident-B kernel: the anchor's four constants arrive through shared memory, fetched one tile ahead by the spare
  // control warp (row_consts / load_state); the generic kernel (small batches) still calls pre()
  static constexpr bool kRowConsts = (kVariant & 4) != 0;   // measured on B200: no gain (3.93 vs 3.89 ms clustered) and the
                                                             // two-tile-old bound costs re-scans (5.0 vs 4.3 ms structureless)
  struct State {
    float dpi, bound_d;
    int ga, gp;
    uint32_t bound_row;   // row of the anchor's best candidate so far (ties -> lowest row)
    uint32_t release_bar; // resident-B kernel: the accumulator buffer's "empty" barrier (0: the kernel arrives itself)
  };
  static constexpr bool kEarlyRelease = true;
  static constexpr bool kTmaStore = false;
  const float* dp;        // [B] exact |a-p|^2
  const int32_t* guid;    // [B,3] int32 guids
  unsigned long long* best;  // [B] (float bits of d) << 32 | row
  int cand;  // 1: columns are the positives' rows 3j+1, 2: the negatives' rows 3j+2
  unsigned long long* stats;   // [0] += re-scanned (anchor, 32-column chunk) pairs
  __device__ __forceinline__ void row_consts(int row, const GemmShape& s, uint32_t dst) const {
    const bool row_ok = row < s.M;
    const uint32_t inf = 0x7f800000u;
    const uint32_t dpi = row_ok ? __float_as_uint(__ldg(dp + row)) : inf;
    const uint32_t ga = row_ok ? static_cast<uint32_t>(__ldg(guid + 3 * row)) : 0u;
    const uint32_t gp = row_ok ? static_cast<uint32_t>(__ldg(guid + 3 * row + 1)) : 0u;
    const unsigned long long key = row_ok ? *(reinterpret_cast<volatile unsigned long long*>(best) + row) : ~0ull;
    sts128(dst, dpi, ga, gp, static_cast<uint32_t>(key >> 32));
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(dst + 16), "r"(static_cast<uint32_t>(key)) : "memory");
  }
  __device__ __forceinline__ void load_state(State& st, uint32_t src) const {
    const uint4 v = lds128(src);
    st.dpi = __uint_as_float(v.x), st.ga = static_cast<int>(v.y), st.gp = static_cast<int>(v.z), st.bound_d = __uint_as_float(v.w);
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(st.bound_row) : "r"(src + 16) : "memory");
    st.release_bar = 0u;
  }
  // the anchor's constants do not depend on the accumulator: the resident-B kernel issues them one tile ahead
  __device__ __forceinline__ void pre(State& st, int row, int /*n0*/, const GemmShape& s, int, int, uint32_t) const {
    const bool row_ok = row < s.M;
    const float inf = __int_as_float(0x7f800000);
    st.dpi = row_ok ? __ldg(dp + row) : inf;
    st.ga = row_ok ? __ldg(guid + 3 * row) : 0;
    st.gp = row_ok ? __ldg(guid + 3 * row + 1) : 0;
    const unsigned long long key = row_ok ? best[row] : ~0ull;
    st.bound_d = __uint_as_float(static_cast<uint32_t>(key >> 32));   // empty key reads as NaN
    st.bound_row = static_cast<uint32_t>(key);
    st.release_bar = 0u;
  }
  // candidate guids of the warp's 128 columns, once per column block (-1 beyond N: the re-scan skips them)
  __device__ __forceinline__ void cols(int n0, const GemmShape& s, int c0, int /*c1*/, uint32_t stg) const {
    static_assert(BN == 256, "a warp owns 4 chunks (128 columns) of the tile");
    col_cache_fill(stg, n0, c0, [&](int col) { return static_cast<uint32_t>(col < s.N ? __ldg(guid + 3 * col + cand) : -1); });
  }
  __device__ __forceinline__ void block_begin(uint32_t epi_smem) const { col_cache_reset(epi_smem); }
  __device__ __forceinline__ void block_end(uint32_t) const {}
  // Works in score space: d = 2 - 2s, so "d > dp" is "s < s_hi" and the closest candidate is the LARGEST such score.
  __device__ __forceinline__ void run(uint32_t taddr, int row, int n0, int /*split*/, const GemmShape& s, int c0,
                                      int c1, uint32_t stg, State& st) const {
    const int lane = threadIdx.x & 31;
    const bool row_ok = row < s.M;
    const float inf = __int_as_float(0x7f800000);
    const float dpi = st.dpi;
    const float s_hi = row_ok ? 1.f - 0.5f * dpi : -inf;      // scores must stay BELOW this (rows beyond M: nothing does)
    const int ga = st.ga, gp = st.gp;
    float bound_d = st.bound_d;                                // best distance known for this anchor (any tile)
    if (!(bound_d == bound_d)) bound_d = inf;                  // empty key reads as NaN
    float s_lo = 1.f - 0.5f * bound_d;                         // a chunk matters only if it holds a score >= this
    uint32_t brow = st.bound_row;                              // ... and a score EQUAL to it only in a row below this one
    float bd = inf;
    int br = -1;
    uint32_t va[32], vb[32];
    auto chunk = [&](const uint32_t (&v)[32], int cc) {
      const int nb = n0 + (c0 + cc) * 32;
      // Hot loop, one instruction per score: t = s_hi - score in packed fp32x2 subtracts, then a 3-input UNSIGNED
      // minimum over the raw bits.  Positive floats order like their bit patterns and every negative float is
      // >= 0x80000000, so the minimum is the smallest t > 0 (the closest candidate with d > dp) whenever one exists.
      uint32_t u0 = 0xffffffffu, u1 = 0xffffffffu;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float2 lo = sub2(s_hi, s_hi, __uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]));
        const float2 hi = sub2(s_hi, s_hi, __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
        u0 = umin3(u0, __float_as_uint(lo.x), __float_as_uint(lo.y));
        u1 = umin3(u1, __float_as_uint(hi.x), __float_as_uint(hi.y));
      }
      // the chunk matters only if it holds a score in [s_lo, s_hi), i.e. 0 <= t <= s_hi - s_lo (monotone in fp32;
      // t == +0 is a harmless false alarm: the re-scan below applies the exact conditions).  A score that merely TIES
      // the bound wins only with a lower row (the result is the minimum over (distance, row)): chunks whose first row lies
      // beyond the bound's row skip the re-scan -- on near-degenerate batches (an untrained tower: every candidate within
      // 1e-3 of the anchor, fp32 scores 6e-8 apart) ties were 3/4 of all re-scans.
      const uint32_t mu = min(u0, u1), thr = __float_as_uint(s_hi - s_lo);
      unsigned int hits = __ballot_sync(0xffffffffu, mu < thr || (mu == thr && static_cast<uint32_t>(3 * nb + cand) < brow));
      // Re-scan (rare once the anchors' bounds have tightened): the triggering row's 32 scores go through the warp's
      // staging slice so that lane j examines column j -- compact code (the former per-thread unrolled scan made the
      // kernel 70 KB of SASS and the epilogue instruction-cache bound), same selection: minimum d, ties -> lowest row.
      if (hits != 0u && __popc(hits) >= kMassHits) {
        // Many rows of the warp hit at once -- the first visits of a scan, when the anchors' bounds are still loose (all
        // 32 rows on the very first): one cooperative re-scan per row would serialise up to 32 x ~70 warp instructions.
        // Here every hitting THREAD scans its own 32 scores in registers, all rows in parallel, with exactly the same
        // conditions and tie rule (minimum d, lowest column).  The guids of the 32 columns are broadcast reads of the
        // column cache.  Used only above kMassHits rows, so the unrolled code stays off the common path's instruction stream.
        if (lane == 0) atomicAdd(stats, static_cast<unsigned long long>(__popc(hits)));
        if ((hits >> lane) & 1u) {
          uint32_t kbest = 0xffffffffu;
          int cbest = -1;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            int g;
            asm volatile("ld.shared.b32 %0, [%1];" : "=r"(g) : "r"(stg + kColCacheOff + 128 * cc + 4 * j) : "memory");
            const float sc = __uint_as_float(v[j]);
            const float d = fmaxf(fmaf(-2.f, sc, 2.f), 0.f);
            const bool pass = sc < s_hi && sc >= s_lo && d > dpi && d < bd && g != ga && g != gp && g >= 0;
            if (pass && __float_as_uint(d) < kbest) kbest = __float_as_uint(d), cbest = j;
          }
          if (cbest >= 0) {
            bd = __uint_as_float(kbest), br = 3 * (nb + cbest) + cand;
            const float s_new = 1.f - 0.5f * bd;
            if (s_new > s_lo || (s_new == s_lo && static_cast<uint32_t>(br) < brow)) brow = static_cast<uint32_t>(br);
            s_lo = fmaxf(s_lo, s_new);
          }
        }
        __syncwarp();
      } else if (hits != 0u) {
        if (lane == 0) atomicAdd(stats, static_cast<unsigned long long>(__popc(hits)));
        int g_lane;   // candidate guid of column nb + lane (column cache)
        asm volatile("ld.shared.b32 %0, [%1];" : "=r"(g_lane) : "r"(stg + kColCacheOff + 128 * cc + 4 * lane) : "memory");
        do {
          const int src = __ffs(hits) - 1;
          hits &= hits - 1u;
          __syncwarp();
          if (lane == src) {
#pragma unroll
            for (int j = 0; j < 8; ++j) sts128(stg + 16 * j, v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          }
          __syncwarp();
          float sc;
          asm volatile("ld.shared.f32 %0, [%1];" : "=f"(sc) : "r"(stg + 4 * lane) : "memory");
          const float hi_s = __shfl_sync(0xffffffffu, s_hi, src), lo_s = __shfl_sync(0xffffffffu, s_lo, src);
          const float dp_s = __shfl_sync(0xffffffffu, dpi, src), bd_s = __shfl_sync(0xffffffffu, bd, src);
          const int ga_s = __shfl_sync(0xffffffffu, ga, src), gp_s = __shfl_sync(0xffffffffu, gp, src);
          const float d = fmaxf(fmaf(-2.f, sc, 2.f), 0.f);
          const bool pass = sc < hi_s && sc >= lo_s && d > dp_s && d < bd_s && g_lane != ga_s && g_lane != gp_s && g_lane >= 0;
          const uint32_t kmin = __reduce_min_sync(0xffffffffu, pass ? __float_as_uint(d) : 0xffffffffu);   // d >= 0: bits order
          if (kmin != 0xffffffffu) {   // warp-uniform
            const int col = __ffs(__ballot_sync(0xffffffffu, pass && __float_as_uint(d) == kmin)) - 1;
            if (lane == src) {
              bd = __uint_as_float(kmin), br = 3 * (nb + col) + cand;
              const float s_new = 1.f - 0.5f * bd;
              if (s_new > s_lo || (s_new == s_lo && static_cast<uint32_t>(br) < brow)) brow = static_cast<uint32_t>(br);
              s_lo = fmaxf(s_lo, s_new);
            }
          }
        } while (hits != 0u);
      }
    };
    auto ok = [&](int cc) { return c0 + cc < c1 && n0 + (c0 + cc) * 32 < s.N; };   // warp-uniform
    if constexpr ((kVariant & 2) == 0) {
      tmem_ld_32x32(taddr + c0 * 32, va);
#pragma unroll
      for (int cc = 0; cc < 4; cc += 2) {
        tmem_ld_wait();
        if (ok(cc + 1)) tmem_ld_32x32(taddr + (c0 + cc + 1) * 32, vb);
        if (ok(cc)) chunk(va, cc);
        tmem_ld_wait();
        if (cc + 2 < 4 && ok(cc + 2)) tmem_ld_32x32(taddr + (c0 + cc + 2) * 32, va);
        if (cc + 2 >= 4 && st.release_bar != 0u) {   // every TMEM read of this warp has landed: release the buffer now
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(st.release_bar);
        }
        if (ok(cc + 1)) chunk(vb, cc + 1);
      }
    } else {
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) {
        if (ok(cc)) {
          tmem_ld_32x32(taddr + (c0 + cc) * 32, va);
          tmem_ld_wait();
          chunk(va, cc);
        }
      }
      if (st.release_bar != 0u) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(st.release_bar);
      }
    }
    if (br >= 0)
      atomicMin(best + row, (static_cast<unsigned long long>(__float_as_uint(bd)) << 32) | static_cast<uint32_t>(br));
  }
};

// Distance-weighted negative sampling (Wu et al. 2017, "Sampling Matters in Deep Embedding Learning"), the second mining
// mode.  Same candidates as EpiMine.  With delta = max(2 - 2s, dmin) (dmin = cutoff^2), a candidate is eligible iff
// delta < dp + margin, and the pick is argmin over eligible candidates of key = ln E - log w(delta), E ~ Exp(1) iid per
// (anchor, candidate): an exponential race, P(pick j) = w_j / sum w.  log w is the inverse density of squared distances
// between uniform points of the unit sphere in D dimensions:
//   log w(delta) = -((D-2)/2) ln delta - ((D-3)/2) ln max(1 - delta/4, kDwOneMinusMin).
// Draws, per 32-column chunk of a launch (chunk id = 2 * (column / 32) + cand - 1), from Philox4x32-10 with key = seed and
// counter = (anchor, chunk id, step lo, (step hi << 4) | w); a word x maps to U = ((x >> 9) + 0.5) 2^-23, Exp(1) = -ln U.
//   w = 0: M = Exp(1) / 32 from word 0 (the chunk's minimum, Exp(32)), K = word 1 >> 27 (its column),
//   w = 1..8: word t gives X_j for column j = 4 (w - 1) + t;  E_j = M for j = K, M + X_j otherwise.
// By memorylessness and symmetry the E_j are 32 iid Exp(1), and every E_j >= M.  Common path per chunk: the score range
// (packed sub + 3-input min/max over t = 2 - s > 0, as EpiMine) bounds delta to [dlo, dhi]; log w is U-shaped (minimum
// at delta = 4(D-2)/(2D-5)), so L = max(log w(dlo), log w(dhi)) bounds it over the chunk, and ln M - L bounds every key.
// Only a chunk whose bound beats the anchor's best key draws the other 31 E_j and evaluates the exact keys (re-scan).
// Result: 64-bit key (f2key(key) << 32 | row) folded with atomicMin -> ties go to the lowest row.
constexpr float kDwOneMinusMin = 1e-6f;
constexpr float kDwLnMFloor = -20.5f;   // ln M >= ln(-ln(1 - 2^-24) / 32) = -20.1 for every draw: skips the Philox call

__device__ __forceinline__ float dw_exp1(uint32_t x) {   // accurate log: relative precision of E near 0 matters
  return -logf((static_cast<float>(x >> 9) + 0.5f) * 0x1p-23f);
}

template <int BN>
struct EpiMineDW {
  static constexpr bool kSplitColumns = true;
  static constexpr bool kPrefetchNext = false;
  static constexpr bool kRowConsts = false;
  static constexpr bool kEarlyRelease = true;
  static constexpr bool kTmaStore = false;
  struct State {
    float dpm;            // dp + margin: eligible iff delta < dpm
    int ga, gp;
    uint32_t bkey, brow;  // the anchor's best (key, row) so far, from the global key at tile start
    uint32_t release_bar;
  };
  const float* dp;
  const int32_t* guid;
  unsigned long long* best;  // [B] f2key(key) << 32 | row
  int cand;
  unsigned long long* stats;
  float margin, dmin, ha, hb;   // dmin = cutoff^2, ha = (D-2)/2, hb = (D-3)/2
  uint32_t seed_lo, seed_hi;
  const int64_t* step;          // device step counter (nullptr: 0), read at every launch so graph replays draw anew
  __device__ __forceinline__ float logw(float delta) const {
    return -(ha * __logf(delta) + hb * __logf(fmaxf(fmaf(-0.25f, delta, 1.f), kDwOneMinusMin)));
  }
  __device__ __forceinline__ void pre(State& st, int row, int /*n0*/, const GemmShape& s, int, int, uint32_t) const {
    const bool row_ok = row < s.M;
    st.dpm = row_ok ? __ldg(dp + row) + margin : -__int_as_float(0x7f800000);   // rows beyond M: nothing eligible
    st.ga = row_ok ? __ldg(guid + 3 * row) : 0;
    st.gp = row_ok ? __ldg(guid + 3 * row + 1) : 0;
    const unsigned long long key = row_ok ? best[row] : ~0ull;
    st.bkey = static_cast<uint32_t>(key >> 32), st.brow = static_cast<uint32_t>(key);
    st.release_bar = 0u;
  }
  __device__ __forceinline__ void cols(int n0, const GemmShape& s, int c0, int /*c1*/, uint32_t stg) const {
    static_assert(BN == 256, "a warp owns 4 chunks (128 columns) of the tile");
    col_cache_fill(stg, n0, c0, [&](int col) { return static_cast<uint32_t>(col < s.N ? __ldg(guid + 3 * col + cand) : -1); });
  }
  __device__ __forceinline__ void block_begin(uint32_t epi_smem) const { col_cache_reset(epi_smem); }
  __device__ __forceinline__ void block_end(uint32_t) const {}
  __device__ __forceinline__ void run(uint32_t taddr, int row, int n0, int /*split*/, const GemmShape& s, int c0,
                                      int c1, uint32_t stg, State& st) const {
    const int lane = threadIdx.x & 31;
    const float inf = __int_as_float(0x7f800000);
    const float dpm = st.dpm;
    const int ga = st.ga, gp = st.gp;
    uint32_t bkey = st.bkey, brow = st.brow;
    float bf = key2f(bkey);
    if (!(bf == bf)) bf = inf;   // empty key reads as NaN
    bool found = false;
    const uint64_t stp = step != nullptr ? static_cast<uint64_t>(__ldg(step)) : 0ull;
    const uint32_t ctr2 = static_cast<uint32_t>(stp), ctr3 = static_cast<uint32_t>(stp >> 32) << 4;
    uint32_t va[32], vb[32];
    // exact key of column j's score sc given its draw word x (unused for j == K); +inf when not eligible
    auto key_of = [&](float sc, int j, uint32_t x, float M, uint32_t K, float dpm_, int g, int ga_, int gp_) {
      const float delta = fmaxf(fmaf(-2.f, sc, 2.f), dmin);
      const float E = static_cast<uint32_t>(j) == K ? M : M + dw_exp1(x);
      const bool pass = delta < dpm_ && g != ga_ && g != gp_ && g >= 0;
      return pass ? f2key(__logf(E) - logw(delta)) : 0xffffffffu;
    };
    auto chunk = [&](const uint32_t (&v)[32], int cc) {
      const int nb = n0 + (c0 + cc) * 32;
      const uint32_t cid = 2u * static_cast<uint32_t>(nb >> 5) + static_cast<uint32_t>(cand - 1);
      // t = 2 - s > 0 for every score, so the raw bits order like the values: min/max of t = the chunk's score range
      uint32_t u0 = 0xffffffffu, u1 = 0xffffffffu, w0 = 0u, w1 = 0u;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float2 lo = sub2(2.f, 2.f, __uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]));
        const float2 hi = sub2(2.f, 2.f, __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
        u0 = umin3(u0, __float_as_uint(lo.x), __float_as_uint(lo.y));
        u1 = umin3(u1, __float_as_uint(hi.x), __float_as_uint(hi.y));
        w0 = umax3(w0, __float_as_uint(lo.x), __float_as_uint(lo.y));
        w1 = umax3(w1, __float_as_uint(hi.x), __float_as_uint(hi.y));
      }
      const float dlo = fmaxf(fmaf(2.f, __uint_as_float(min(u0, u1)), -2.f), dmin);
      const float dhi = fminf(fmaxf(fmaf(2.f, __uint_as_float(max(w0, w1)), -2.f), dmin), dpm);
      float L = fmaxf(logw(dlo), logw(dhi));
      L += 1e-3f + 1e-4f * fabsf(L);   // covers the rounding of t, delta and the approximate logs
      float M = 0.f;
      uint32_t K = 0u;
      bool hit = dlo < dpm && kDwLnMFloor - L < bf;
      if (hit) {
        const uint4 x = philox4x32_10(static_cast<uint32_t>(row), cid, ctr2, ctr3, seed_lo, seed_hi);
        M = dw_exp1(x.x) * (1.f / 32.f), K = x.y >> 27;
        hit = __logf(M) - L < bf;
      }
      unsigned int hits = __ballot_sync(0xffffffffu, hit);
      if (hits == 0u) return;
      if (lane == 0) atomicAdd(stats, static_cast<unsigned long long>(__popc(hits)));
      if (__popc(hits) >= kMassHits) {
        // many rows at once (first visits, while the bounds are loose): every hitting thread scans its own 32 columns
        if (hit) {
          uint32_t kbest = 0xffffffffu;
          int cbest = -1;
#pragma unroll
          for (int w = 0; w < 8; ++w) {
            const uint4 x = philox4x32_10(static_cast<uint32_t>(row), cid, ctr2, ctr3 | (w + 1), seed_lo, seed_hi);
            const uint32_t xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              const int j = 4 * w + t;
              int g;
              asm volatile("ld.shared.b32 %0, [%1];" : "=r"(g) : "r"(stg + kColCacheOff + 128 * cc + 4 * j) : "memory");
              const uint32_t k = key_of(__uint_as_float(v[j]), j, xs[t], M, K, dpm, g, ga, gp);
              if (k < kbest) kbest = k, cbest = j;
            }
          }
          const uint32_t r = static_cast<uint32_t>(3 * (nb + cbest) + cand);
          if (cbest >= 0 && (kbest < bkey || (kbest == bkey && r < brow))) bkey = kbest, brow = r, bf = key2f(kbest), found = true;
        }
        __syncwarp();
      } else {
        int g_lane;   // candidate guid of column nb + lane (column cache)
        asm volatile("ld.shared.b32 %0, [%1];" : "=r"(g_lane) : "r"(stg + kColCacheOff + 128 * cc + 4 * lane) : "memory");
        do {   // one hitting row at a time: lane j evaluates column j (its draw is word j % 4 of call 1 + j / 4)
          const int src = __ffs(hits) - 1;
          hits &= hits - 1u;
          __syncwarp();
          if (lane == src) {
#pragma unroll
            for (int j = 0; j < 8; ++j) sts128(stg + 16 * j, v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          }
          __syncwarp();
          float sc;
          asm volatile("ld.shared.f32 %0, [%1];" : "=f"(sc) : "r"(stg + 4 * lane) : "memory");
          const int row_s = __shfl_sync(0xffffffffu, row, src);
          const float M_s = __shfl_sync(0xffffffffu, M, src), dpm_s = __shfl_sync(0xffffffffu, dpm, src);
          const uint32_t K_s = __shfl_sync(0xffffffffu, K, src);
          const int ga_s = __shfl_sync(0xffffffffu, ga, src), gp_s = __shfl_sync(0xffffffffu, gp, src);
          const uint4 x = philox4x32_10(static_cast<uint32_t>(row_s), cid, ctr2, ctr3 | (1 + (lane >> 2)), seed_lo, seed_hi);
          const int t = lane & 3;
          const uint32_t xw = t == 0 ? x.x : t == 1 ? x.y : t == 2 ? x.z : x.w;
          const uint32_t k = key_of(sc, lane, xw, M_s, K_s, dpm_s, g_lane, ga_s, gp_s);
          const uint32_t kmin = __reduce_min_sync(0xffffffffu, k);
          if (kmin != 0xffffffffu) {   // warp-uniform
            const int col = __ffs(__ballot_sync(0xffffffffu, k == kmin)) - 1;
            const uint32_t r = static_cast<uint32_t>(3 * (nb + col) + cand);
            if (lane == src && (kmin < bkey || (kmin == bkey && r < brow))) bkey = kmin, brow = r, bf = key2f(kmin), found = true;
          }
        } while (hits != 0u);
      }
    };
    auto ok = [&](int cc) { return c0 + cc < c1 && n0 + (c0 + cc) * 32 < s.N; };   // warp-uniform
    tmem_ld_32x32(taddr + c0 * 32, va);
#pragma unroll
    for (int cc = 0; cc < 4; cc += 2) {
      tmem_ld_wait();
      if (ok(cc + 1)) tmem_ld_32x32(taddr + (c0 + cc + 1) * 32, vb);
      if (ok(cc)) chunk(va, cc);
      tmem_ld_wait();
      if (cc + 2 < 4 && ok(cc + 2)) tmem_ld_32x32(taddr + (c0 + cc + 2) * 32, va);
      if (cc + 2 >= 4 && st.release_bar != 0u) {   // every TMEM read of this warp has landed: release the buffer now
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(st.release_bar);
      }
      if (ok(cc + 1)) chunk(vb, cc + 1);
    }
    if (found) atomicMin(best + row, (static_cast<unsigned long long>(bkey) << 32) | brow);
  }
};

__global__ void mine_prepare_kernel(const float* __restrict__ E, int64_t ld, int D, const int64_t* __restrict__ guid64,
                                    int64_t B, float* __restrict__ dp, int32_t* __restrict__ guid32,
                                    unsigned long long* __restrict__ best, unsigned long long* __restrict__ stats) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (blockIdx.x == 0 && threadIdx.x < 2) stats[threadIdx.x] = 0ull;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * 8 + warp; i < B; i += static_cast<int64_t>(gridDim.x) * 8) {
    const float* a = E + 3 * i * ld;
    const float* p = a + ld;
    float s = 0.f;
    for (int j = lane; j < D; j += 32) {
      const float t = a[j] - p[j];
      s = fmaf(t, t, s);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) dp[i] = s, best[i] = kNoCand;
    if (lane < 3) guid32[3 * i + lane] = static_cast<int32_t>(guid64[3 * i + lane]);
  }
}

__global__ void mine_finalize_kernel(const float* __restrict__ E, int64_t ld, int D,
                                     const unsigned long long* __restrict__ best, int64_t B,
                                     int32_t* __restrict__ neg_row, float* __restrict__ d_an,
                                     unsigned long long* __restrict__ stats) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned int mined = 0;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * 8 + warp; i < B; i += static_cast<int64_t>(gridDim.x) * 8) {
    const unsigned long long kb = best[i];
    const int r = kb != kNoCand ? static_cast<int>(static_cast<uint32_t>(kb)) : static_cast<int>(3 * i + 2);
    mined += kb != kNoCand ? 1u : 0u;
    if (lane == 0) neg_row[i] = r;
    if (d_an != nullptr) {  // exact fp32 distance of the chosen negative
      const float* a = E + 3 * i * ld;
      const float* n = E + static_cast<int64_t>(r) * ld;
      float s = 0.f;
      for (int j = lane; j < D; j += 32) {
        const float t = a[j] - n[j];
        s = fmaf(t, t, s);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) d_an[i] = s;
    }
  }
  if (lane == 0 && mined != 0u) atomicAdd(stats + 1, static_cast<unsigned long long>(mined));
}

}  // namespace cdml

using namespace cdml;

extern "C" int cdml_mine_semihard(cdml_ctx* ctx, const void* E16, int64_t ld16, int dtype16, const float* E32,
                                  int64_t ld32, const int64_t* guid, int64_t B, int D, float margin, int32_t* neg_row,
                                  float* d_an, void* stream) {
  CDML_REQUIRE(ctx && E16 && E32 && guid && neg_row, "cdml_mine_semihard: NULL argument");
  CDML_REQUIRE(B > 0 && 3 * B < (1ll << 31) && D > 0 && D % 8 == 0 && ld16 >= D && ld32 >= D,
               "cdml_mine_semihard: bad geometry B=%lld D=%d", (long long)B, D);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // scratch: best [B] u64 | dp [B] f32 | guid32 [3B] i32
  const size_t bytes = static_cast<size_t>(B) * (8 + 4 + 12) + 64;
  uint8_t* ws = static_cast<uint8_t*>(ctx_scratch(ctx, bytes));
  if (ws == nullptr) return -2;
  if (ctx->mine_stats == nullptr) CDML_CHECK_CUDA(cudaMalloc(&ctx->mine_stats, 2 * sizeof(unsigned long long)));
  unsigned long long* stats = ctx->mine_stats;
  unsigned long long* best = reinterpret_cast<unsigned long long*>(ws);
  float* dp = reinterpret_cast<float*>(best + B);
  int32_t* guid32 = reinterpret_cast<int32_t*>(dp + B);
  const int grid = static_cast<int>(std::min<int64_t>((B + 7) / 8, ctx->num_sms * 8));
  mine_prepare_kernel<<<grid, 256, 0, st>>>(E32, ld32, D, guid, B, dp, guid32, best, stats);
  int rc = 0;
  const uint16_t* e16 = static_cast<const uint16_t*>(E16);
  for (int cand = 1; cand <= 2 && rc >= 0; ++cand) {
    // A: anchors = rows 0,3,6,.. (pitch 3*ld16); B: candidates = rows cand, cand+3, .. ; both K-major, K = D.
    // Variant 1 (measured best of the four on B200: 3.79 ms vs 4.17-4.25): pipelined TMEM reads, anchor constants
    // fetched after the previous tile is released (a one-tile-ahead fetch of the running bound makes it staler).
    EpiMine<kBN, 1> epi{dp, guid32, best, cand, stats};
    static int rowc = -1;   // CDML_MINE_ROWCONSTS=1: anchor constants through the spare warp's shared-memory slots (A/B aid)
    if (rowc < 0) rowc = getenv("CDML_MINE_ROWCONSTS") != nullptr ? 1 : 0;
    if (resb_applicable(D) && B >= 8 * kBM && rowc) {
      EpiMine<kBN, 5> epi5{dp, guid32, best, cand, stats};
      rc = launch_gemm_resb(ctx, e16, 3 * ld16, e16 + cand * ld16, 3 * ld16, B, B, D, dtype16, epi5, st);
    } else if (resb_applicable(D) && B >= 8 * kBM && epi_warps() == 16)
      rc = launch_gemm_resb<EpiMine<kBN, 1>, 16>(ctx, e16, 3 * ld16, e16 + cand * ld16, 3 * ld16, B, B, D, dtype16, epi, st);
    else if (resb_applicable(D) && B >= 8 * kBM)
      rc = launch_gemm_resb(ctx, e16, 3 * ld16, e16 + cand * ld16, 3 * ld16, B, B, D, dtype16, epi, st);
    else
      rc = launch_gemm<0, 0>(ctx, e16, 3 * ld16, e16 + cand * ld16, 3 * ld16, B, B, D, dtype16, 1, epi, st);
  }
  if (rc >= 0) {
    mine_finalize_kernel<<<grid, 256, 0, st>>>(E32, ld32, D, best, B, neg_row, d_an, stats);
    rc = cudaGetLastError() == cudaSuccess ? 0 : -2;
  }
  return rc < 0 ? rc : 0;
}

extern "C" int cdml_mine_distance_weighted(cdml_ctx* ctx, const void* E16, int64_t ld16, int dtype16, const float* E32,
                                           int64_t ld32, const int64_t* guid, int64_t B, int D, float margin, float cutoff,
                                           uint64_t seed, const int64_t* step, int32_t* neg_row, float* d_an,
                                           void* stream) {
  CDML_REQUIRE(ctx && E16 && E32 && guid && neg_row, "cdml_mine_distance_weighted: NULL argument");
  CDML_REQUIRE(B > 0 && 3 * B < (1ll << 31) && D >= 8 && D % 8 == 0 && ld16 >= D && ld32 >= D,
               "cdml_mine_distance_weighted: bad geometry B=%lld D=%d", (long long)B, D);
  CDML_REQUIRE(cutoff > 0.f && cutoff < 2.f && margin == margin, "cdml_mine_distance_weighted: cutoff %g not in (0, 2)",
               (double)cutoff);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t bytes = static_cast<size_t>(B) * (8 + 4 + 12) + 64;   // as cdml_mine_semihard
  uint8_t* ws = static_cast<uint8_t*>(ctx_scratch(ctx, bytes));
  if (ws == nullptr) return -2;
  if (ctx->mine_stats == nullptr) CDML_CHECK_CUDA(cudaMalloc(&ctx->mine_stats, 2 * sizeof(unsigned long long)));
  unsigned long long* stats = ctx->mine_stats;
  unsigned long long* best = reinterpret_cast<unsigned long long*>(ws);
  float* dp = reinterpret_cast<float*>(best + B);
  int32_t* guid32 = reinterpret_cast<int32_t*>(dp + B);
  const int grid = static_cast<int>(std::min<int64_t>((B + 7) / 8, ctx->num_sms * 8));
  mine_prepare_kernel<<<grid, 256, 0, st>>>(E32, ld32, D, guid, B, dp, guid32, best, stats);
  int rc = 0;
  const uint16_t* e16 = static_cast<const uint16_t*>(E16);
  for (int cand = 1; cand <= 2 && rc >= 0; ++cand) {
    EpiMineDW<kBN> epi{dp, guid32, best, cand, stats, margin, cutoff * cutoff, 0.5f * (D - 2), 0.5f * (D - 3),
                       static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32), step};
    if (resb_applicable(D) && B >= 8 * kBM)
      rc = launch_gemm_resb(ctx, e16, 3 * ld16, e16 + cand * ld16, 3 * ld16, B, B, D, dtype16, epi, st);
    else
      rc = launch_gemm<0, 0>(ctx, e16, 3 * ld16, e16 + cand * ld16, 3 * ld16, B, B, D, dtype16, 1, epi, st);
  }
  if (rc >= 0) {
    mine_finalize_kernel<<<grid, 256, 0, st>>>(E32, ld32, D, best, B, neg_row, d_an, stats);
    rc = cudaGetLastError() == cudaSuccess ? 0 : -2;
  }
  return rc < 0 ? rc : 0;
}

extern "C" int cdml_mine_last_stats(cdml_ctx* ctx, int64_t* out2, void* stream) {
  CDML_REQUIRE(ctx && out2, "cdml_mine_last_stats: NULL argument");
  out2[0] = out2[1] = 0;
  if (ctx->mine_stats == nullptr) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned long long h[2];
  CDML_CHECK_CUDA(cudaMemcpyAsync(h, ctx->mine_stats, sizeof(h), cudaMemcpyDeviceToHost, st));
  CDML_CHECK_CUDA(cudaStreamSynchronize(st));
  out2[0] = static_cast<int64_t>(h[0]), out2[1] = static_cast<int64_t>(h[1]);
  return 0;
}
