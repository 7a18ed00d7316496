// On-device triplet reader (SURVEY 8f row 3; inputs.py:102-142 + parse_data.py:292-298): the co-watch pairs of a *.train
// file stay resident in HBM and a batch of [B,3] index triplets is produced where it is consumed -- no per-line Python,
// no Manager queue, no H2D copy per step.
//
//   out[i] = (a, p, n)   with (a, p) = pairs[(start + i) % n_pairs]           (the file wraps num_epochs times, :114-122)
//                        and n ~ U{0..G-1}, re-drawn while n in {a, p}        (:123-129)
//
// The reference draws n from numpy's global Mersenne Twister in an unseeded forked worker (SURVEY Q10); there is no
// stream to reproduce, only the distribution.  Here every stream position (start + i) owns a counter-based generator:
// Philox4x32-10 (Salmon et al., SC'11; pinned in tests to the Random123 known-answer vectors) with key = seed and
// counter = (position lo, position hi, attempt, 0).  A draw is word 0 mapped to [0,G) by Lemire's multiply-shift WITH its
// rejection step, so the result is exactly uniform; a rejected or excluded draw moves on to attempt + 1.
#include "../../include/cdml.h"
#include "ctx.cuh"

namespace cdml {

__device__ __forceinline__ uint32_t philox4x32_10_word0(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                                        uint32_t k1) {
  return philox4x32_10(c0, c1, c2, c3, k0, k1).x;
}

__global__ void __launch_bounds__(256)
sample_triplets_kernel(const int64_t* __restrict__ pairs, int64_t n_pairs, int64_t start, int64_t B, uint32_t G,
                       uint32_t seed_lo, uint32_t seed_hi, int64_t* __restrict__ out) {
  const uint32_t threshold = (0u - G) % G;                    // 2^32 mod G
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < B;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const uint64_t pos = static_cast<uint64_t>(start + i);
    const int64_t row = static_cast<int64_t>(pos % static_cast<uint64_t>(n_pairs));
    const int64_t a = pairs[2 * row], p = pairs[2 * row + 1];
    int64_t neg = -1;
    for (uint32_t attempt = 0; neg < 0; ++attempt) {
      const uint32_t x = philox4x32_10_word0(static_cast<uint32_t>(pos), static_cast<uint32_t>(pos >> 32), attempt, 0u,
                                             seed_lo, seed_hi);
      const uint64_t m = static_cast<uint64_t>(x) * G;
      if (static_cast<uint32_t>(m) < threshold) continue;       // Lemire's rejection: exact uniformity
      const int64_t cand = static_cast<int64_t>(m >> 32);
      if (cand != a && cand != p) neg = cand;
    }
    out[3 * i] = a, out[3 * i + 1] = p, out[3 * i + 2] = neg;
  }
}

}  // namespace cdml

extern "C" int cdml_sample_triplets(cdml_ctx* ctx, const int64_t* pairs, int64_t n_pairs, int64_t start, int64_t B,
                                    int64_t num_guid, uint64_t seed, int64_t* out, void* stream) {
  using namespace cdml;
  CDML_REQUIRE(ctx && pairs && out, "cdml_sample_triplets: NULL argument");
  CDML_REQUIRE(n_pairs > 0 && start >= 0 && B >= 0, "cdml_sample_triplets: bad geometry");
  CDML_REQUIRE(num_guid >= 3 && num_guid < (1ll << 32), "cdml_sample_triplets: num_guid must be in [3, 2^32) (got %lld)",
               (long long)num_guid);
  if (B == 0) return 0;
  const int64_t blocks = (B + 255) / 256, cap = static_cast<int64_t>(ctx->num_sms) * 8;
  sample_triplets_kernel<<<static_cast<int>(blocks < cap ? blocks : cap), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      pairs, n_pairs, start, B, static_cast<uint32_t>(num_guid), static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32),
      out);
  CDML_CHECK_CUDA(cudaGetLastError());
  return 0;
}
