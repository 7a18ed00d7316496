// Host launchers + C ABI for the tcgen05 GEMM family (cdml_gemm16).
#include "gemm_launch.cuh"

namespace cdml {

// K-major x K-major with K <= 256 -> resident-B kernel (3x less L2 operand traffic); everything else -> generic.
template <int AMN, int BMN, class Epi>
static int launch_any(cdml_ctx* ctx, const void* A, int64_t lda, const void* B, int64_t ldb, int64_t M, int64_t N, int64_t K,
                      int dtype16, int num_splits, const Epi& epi, cudaStream_t stream) {
  if constexpr (AMN == 0 && BMN == 0) {
    if (num_splits <= 1 && resb_applicable(K) && M >= 8 * kBM)
      return launch_gemm_resb(ctx, A, lda, B, ldb, M, N, K, dtype16, epi, stream, 1);
  }
  return launch_gemm<AMN, BMN>(ctx, A, lda, B, ldb, M, N, K, dtype16, num_splits, epi, stream);
}

template <int AMN, int BMN>
static int dispatch_epilogue(cdml_ctx* ctx, const void* A, int64_t lda, const void* B, int64_t ldb, int64_t M, int64_t N,
                             int64_t K, int dtype16, int epilogue, void* out, int64_t ld_out, const float* bias,
                             float alpha, void* aux0, void* aux1, int64_t ld_aux1, int num_splits, int64_t split_stride,
                             cudaStream_t stream) {
  const bool bf = dtype16 == CDML_BF16;
  switch (epilogue) {
    case 0: {
      EpiStoreF32<kBN> e{static_cast<float*>(out), ld_out, split_stride, bias, alpha};
      return launch_any<AMN, BMN>(ctx, A, lda, B, ldb, M, N, K, dtype16, num_splits, e, stream);
    }
    case 1: {
      CDML_REQUIRE(aux0 == nullptr || ld_aux1 >= M, "STORE_16: the sign-mask pitch (ld_aux1, words) must be >= M");
      if (bf) {
        EpiStore16<kBN, 1> e{static_cast<uint16_t*>(out), ld_out, bias, alpha, static_cast<uint32_t*>(aux0), ld_aux1};
        return launch_any<AMN, BMN>(ctx, A, lda, B, ldb, M, N, K, dtype16, 1, e, stream);
      }
      EpiStore16<kBN, 0> e{static_cast<uint16_t*>(out), ld_out, bias, alpha, static_cast<uint32_t*>(aux0), ld_aux1};
      return launch_any<AMN, BMN>(ctx, A, lda, B, ldb, M, N, K, dtype16, 1, e, stream);
    }
    case 2: {
      CDML_REQUIRE(N <= kBN, "L2NORM epilogue needs the whole row in one tile (N=%lld > %d)", (long long)N, kBN);
      if (bf) {
        EpiL2Norm<kBN, 1> e{static_cast<float*>(out), ld_out, bias, alpha, static_cast<float*>(aux0),
                            static_cast<uint16_t*>(aux1), ld_aux1};
        return launch_any<AMN, BMN>(ctx, A, lda, B, ldb, M, N, K, dtype16, 1, e, stream);
      }
      EpiL2Norm<kBN, 0> e{static_cast<float*>(out), ld_out, bias, alpha, static_cast<float*>(aux0),
                          static_cast<uint16_t*>(aux1), ld_aux1};
      return launch_any<AMN, BMN>(ctx, A, lda, B, ldb, M, N, K, dtype16, 1, e, stream);
    }
    case 3: {
      CDML_REQUIRE(aux1 != nullptr, "MASK_LEAKY epilogue needs aux1 (the forward activation)");
      if (bf) {
        EpiMaskLeaky<kBN, 1> e{static_cast<uint16_t*>(out), ld_out, static_cast<const uint16_t*>(aux1), ld_aux1, alpha};
        return launch_any<AMN, BMN>(ctx, A, lda, B, ldb, M, N, K, dtype16, 1, e, stream);
      }
      EpiMaskLeaky<kBN, 0> e{static_cast<uint16_t*>(out), ld_out, static_cast<const uint16_t*>(aux1), ld_aux1, alpha};
      return launch_any<AMN, BMN>(ctx, A, lda, B, ldb, M, N, K, dtype16, 1, e, stream);
    }
    case 4: {
      CDML_REQUIRE(aux1 != nullptr && ld_aux1 >= M, "MASK_BITS epilogue needs aux1 (packed sign mask) with a pitch of >= M words");
      if constexpr (AMN == 0 && BMN == 0) {
        // resident-B kernel with TMA stores of the output (CDML_TMA_STORE=0: the staged global stores, A/B aid)
        static int tma_on = -1;
        if (tma_on < 0) {
          const char* e = getenv("CDML_TMA_STORE");
          tma_on = (e != nullptr && e[0] == '0') ? 0 : 1;
        }
        // N % 8 == 0 as well: a box that crosses the tensor map's inner bound inside a 16-byte piece was found (B200) to
        // write zeros past column N-1, into the caller's pitch padding or neighbouring columns
        // (profiles/r03_gemm_exact_on_parent.log; tests/test_gemm_exact.py checks the padding of every output)
        if (tma_on && num_splits <= 1 && resb_applicable(K) && M >= 8 * kBM && (ld_out * 2) % 16 == 0 && N % 8 == 0) {
          CUtensorMap om;
          int rc = make_tmap_2d(ctx, &om, out, dtype16, N, M, ld_out, 32, 32, 64);
          if (rc) return rc;
          if (bf) {
            EpiMaskBitsTma<kBN, 1> e{om, static_cast<const uint32_t*>(aux1), ld_aux1, alpha};
            return launch_gemm_resb(ctx, A, lda, B, ldb, M, N, K, dtype16, e, stream, 1);
          }
          EpiMaskBitsTma<kBN, 0> e{om, static_cast<const uint32_t*>(aux1), ld_aux1, alpha};
          return launch_gemm_resb(ctx, A, lda, B, ldb, M, N, K, dtype16, e, stream, 1);
        }
      }
      if (bf) {
        EpiMaskBits<kBN, 1> e{static_cast<uint16_t*>(out), ld_out, static_cast<const uint32_t*>(aux1), ld_aux1, alpha};
        return launch_any<AMN, BMN>(ctx, A, lda, B, ldb, M, N, K, dtype16, 1, e, stream);
      }
      EpiMaskBits<kBN, 0> e{static_cast<uint16_t*>(out), ld_out, static_cast<const uint32_t*>(aux1), ld_aux1, alpha};
      return launch_any<AMN, BMN>(ctx, A, lda, B, ldb, M, N, K, dtype16, 1, e, stream);
    }
    case 100: {
      EpiNull<kBN, 0> e{static_cast<float*>(out)};
      return launch_any<AMN, BMN>(ctx, A, lda, B, ldb, M, N, K, dtype16, 1, e, stream);
    }
    case 101: {
      EpiNull<kBN, 1> e{static_cast<float*>(out)};
      return launch_any<AMN, BMN>(ctx, A, lda, B, ldb, M, N, K, dtype16, 1, e, stream);
    }
    default:
      set_error("cdml_gemm16: unknown epilogue %d", epilogue);
      return -1;
  }
}

}  // namespace cdml

extern "C" {

int cdml_gemm16_auto_splits(cdml_ctx* ctx, int64_t M, int64_t N, int64_t K) {
  if (ctx == nullptr || M <= 0 || N <= 0 || K <= 0) return 1;
  const int tiles = static_cast<int>(((M + cdml::kBM - 1) / cdml::kBM) * ((N + cdml::kBN - 1) / cdml::kBN));
  return cdml::pick_splits(ctx->num_sms, tiles, static_cast<int>((K + cdml::kBK - 1) / cdml::kBK));
}

int cdml_gemm16(cdml_ctx* ctx, const void* A, int a_mn_major, int64_t lda, const void* B, int b_mn_major, int64_t ldb,
                int64_t M, int64_t N, int64_t K, int dtype16, int epilogue, void* out, int64_t ld_out,
                const float* bias, float alpha, void* aux0, void* aux1, int64_t ld_aux1, int num_splits,
                int64_t split_stride, int* splits_used, void* stream) {
  using namespace cdml;
  CDML_REQUIRE(ctx != nullptr && A != nullptr && B != nullptr && out != nullptr, "cdml_gemm16: NULL argument");
  CDML_REQUIRE(M > 0 && N > 0 && K > 0 && M < (1ll << 31) && N < (1ll << 31) && K < (1ll << 31),
               "cdml_gemm16: bad shape M=%lld N=%lld K=%lld", (long long)M, (long long)N, (long long)K);
  CDML_REQUIRE(dtype16 == CDML_F16 || dtype16 == CDML_BF16, "cdml_gemm16: dtype16 must be 0 (fp16) or 1 (bf16)");
  CDML_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0, "cdml_gemm16: out is not 16-byte aligned");
  if (epilogue == 0) {
    if (num_splits <= 0) num_splits = cdml_gemm16_auto_splits(ctx, M, N, K);
    CDML_REQUIRE(num_splits == 1 || (bias == nullptr && alpha == 1.0f),
                 "cdml_gemm16: split-K partials cannot carry bias/activation");
    CDML_REQUIRE(num_splits == 1 || split_stride >= M * ld_out, "cdml_gemm16: split_stride too small");
  } else {
    num_splits = 1;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc;
  if (a_mn_major == 0 && b_mn_major == 1)
    rc = dispatch_epilogue<0, 1>(ctx, A, lda, B, ldb, M, N, K, dtype16, epilogue, out, ld_out, bias, alpha, aux0, aux1,
                                 ld_aux1, num_splits, split_stride, st);
  else if (a_mn_major == 0 && b_mn_major == 0)
    rc = dispatch_epilogue<0, 0>(ctx, A, lda, B, ldb, M, N, K, dtype16, epilogue, out, ld_out, bias, alpha, aux0, aux1,
                                 ld_aux1, num_splits, split_stride, st);
  else if (a_mn_major == 1 && b_mn_major == 1)
    rc = dispatch_epilogue<1, 1>(ctx, A, lda, B, ldb, M, N, K, dtype16, epilogue, out, ld_out, bias, alpha, aux0, aux1,
                                 ld_aux1, num_splits, split_stride, st);
  else {
    set_error("cdml_gemm16: operand layout (a_mn_major=%d, b_mn_major=%d) is not instantiated", a_mn_major, b_mn_major);
    return -1;
  }
  if (rc < 0) return rc;
  if (splits_used != nullptr) *splits_used = rc;
  return 0;
}

}  // extern "C"
