// Host-side launcher of gemm_tcgen05_kernel, shared by the translation units that instantiate epilogues.
#pragma once
#include "../../include/cdml.h"
#include "ctx.cuh"
#include "gemm_sm100.cuh"
#include "gemm2_sm100.cuh"

#include <stdlib.h>

namespace cdml {

// CDML_TRACE=1: announce every tensor-core launch on stderr and synchronise after it (bring-up aid).
inline bool trace_on() {
  static int on = -1;
  if (on < 0) on = getenv("CDML_TRACE") != nullptr ? 1 : 0;
  return on == 1;
}
inline int trace_sync(const char* what, long M, long N, long K, int grid, cudaStream_t st) {
  if (!trace_on()) return 0;
  fprintf(stderr, "[cdml] %s M=%ld N=%ld K=%ld grid=%d ... ", what, M, N, K, grid);
  fflush(stderr);
  cudaError_t e = cudaStreamSynchronize(st);
  fprintf(stderr, "%s\n", cudaGetErrorString(e));
  fflush(stderr);
  return e == cudaSuccess ? 0 : -2;
}

constexpr int kBN = 256;
constexpr int kStages = 4;

inline int pick_splits(int num_sms, int tiles, int num_kb) {
  // Few output tiles but a long K (weight gradients): split K so that tiles*S fills whole waves of SMs.
  if (tiles >= 2 * num_sms || num_kb < 16) return 1;
  const int smax = max(1, min(64, num_kb / 8));
  int best = 1;
  double best_eff = -1.0;
  for (int s = 1; s <= smax; ++s) {
    const int per = (num_kb + s - 1) / s;
    const int seff = (num_kb + per - 1) / per;
    if (seff != s) continue;
    const long units = static_cast<long>(tiles) * s;
    const long waves = (units + num_sms - 1) / num_sms;
    double eff = static_cast<double>(units) / static_cast<double>(waves * num_sms);
    if (units < num_sms) eff *= 0.5;          // leaves SMs idle
    eff -= 0.002 * s;                          // partial-buffer traffic: prefer fewer splits on ties
    if (eff > best_eff) best_eff = eff, best = s;
  }
  return best;
}

// CDML_2CTA=0 disables the CTA-pair kernel (A/B measurement aid); it is used for tiles of >= 8 k-blocks.
inline bool two_cta_enabled() {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("CDML_2CTA");
    on = (e != nullptr && e[0] == '0') ? 0 : 1;
  }
  return on == 1;
}

template <int AMN, int BMN, class Epi>
static int launch_gemm2(cdml_ctx* ctx, const void* A, int64_t lda, const void* B, int64_t ldb, int64_t M, int64_t N,
                        int64_t K, int dtype16, int num_splits, const Epi& epi, cudaStream_t stream) {
  using L = Gemm2Smem;
  CUtensorMap ta, tb;
  int rc;
  if (AMN == 0) rc = make_tmap_2d(ctx, &ta, A, dtype16, K, M, lda, kBK, kBM);
  else rc = make_tmap_2d(ctx, &ta, A, dtype16, M, K, lda, 64, kBK);
  if (rc) return rc;
  if (BMN == 0) rc = make_tmap_2d(ctx, &tb, B, dtype16, K, N, ldb, kBK, kBN2 / 2);
  else rc = make_tmap_2d(ctx, &tb, B, dtype16, N, K, ldb, 64, kBK);
  if (rc) return rc;
  GemmShape s;
  s.M = static_cast<int>(M), s.N = static_cast<int>(N), s.K = static_cast<int>(K);
  s.m_tiles = (s.M + 2 * kBM - 1) / (2 * kBM);   // 256-row pair tiles
  s.n_tiles = (s.N + kBN2 - 1) / kBN2;
  s.num_kb = (s.K + kBK - 1) / kBK;
  num_splits = max(1, min(num_splits, s.num_kb));
  s.kb_per_split = (s.num_kb + num_splits - 1) / num_splits;
  s.num_splits = (s.num_kb + s.kb_per_split - 1) / s.kb_per_split;
  s.idesc = make_idesc_f16(dtype16 == CDML_BF16 ? 1 : 0, AMN, BMN, 2 * kBM, kBN2);
  s.m_fastest = (s.num_splits > 1 && N >= M) ? 1 : 0;
  auto kern = gemm2_tcgen05_kernel<AMN, BMN, Epi>;
  static bool attr_set = false;
  if (!attr_set) {
    CDML_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kTotal));
    attr_set = true;
  }
  const long units = static_cast<long>(s.m_tiles) * s.n_tiles * s.num_splits;
  const int clusters = static_cast<int>(units < ctx->num_sms / 2 ? units : ctx->num_sms / 2);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * clusters);
  cfg.blockDim = dim3(kGemmThreads);
  cfg.dynamicSmemBytes = L::kTotal;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2, attr[0].val.clusterDim.y = 1, attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  CDML_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, ta, tb, s, epi));
  if (trace_sync("gemm2_tcgen05", M, N, K, 2 * clusters, stream)) return -2;
  return s.num_splits;
}

template <int AMN, int BMN, class Epi>
static int launch_gemm(cdml_ctx* ctx, const void* A, int64_t lda, const void* B, int64_t ldb, int64_t M, int64_t N,
                       int64_t K, int dtype16, int num_splits, const Epi& epi, cudaStream_t stream) {
  {
    const int64_t kb_per = ((K + kBK - 1) / kBK + max(num_splits, 1) - 1) / max(num_splits, 1);
    if (two_cta_enabled() && M >= 2 * kBM && kb_per >= 8)
      return launch_gemm2<AMN, BMN>(ctx, A, lda, B, ldb, M, N, K, dtype16, num_splits, epi, stream);
  }
  using L = GemmSmem<kBN, kStages>;
  CUtensorMap ta, tb;
  int rc;
  if (AMN == 0) rc = make_tmap_2d(ctx, &ta, A, dtype16, K, M, lda, kBK, kBM);
  else rc = make_tmap_2d(ctx, &ta, A, dtype16, M, K, lda, 64, kBK);
  if (rc) return rc;
  if (BMN == 0) rc = make_tmap_2d(ctx, &tb, B, dtype16, K, N, ldb, kBK, kBN);
  else rc = make_tmap_2d(ctx, &tb, B, dtype16, N, K, ldb, 64, kBK);
  if (rc) return rc;

  GemmShape s;
  s.M = static_cast<int>(M), s.N = static_cast<int>(N), s.K = static_cast<int>(K);
  s.m_tiles = (s.M + kBM - 1) / kBM;
  s.n_tiles = (s.N + kBN - 1) / kBN;
  s.num_kb = (s.K + kBK - 1) / kBK;
  num_splits = max(1, min(num_splits, s.num_kb));
  s.kb_per_split = (s.num_kb + num_splits - 1) / num_splits;
  s.num_splits = (s.num_kb + s.kb_per_split - 1) / s.kb_per_split;
  s.idesc = make_idesc_f16(dtype16 == CDML_BF16 ? 1 : 0, AMN, BMN, kBM, kBN);
  // Split-K (weight gradients): every k-block of the larger operand should be shared by ALL tiles that run
  // concurrently, so that it is fetched from HBM once per split.
  s.m_fastest = (s.num_splits > 1 && N >= M) ? 1 : 0;

  auto kern = gemm_tcgen05_kernel<AMN, BMN, kBN, kStages, Epi>;
  static bool attr_set = false;  // per template instantiation
  if (!attr_set) {
    CDML_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kTotal));
    attr_set = true;
  }
  const long units = static_cast<long>(s.m_tiles) * s.n_tiles * s.num_splits;
  const int grid = static_cast<int>(units < ctx->num_sms ? units : ctx->num_sms);
  kern<<<grid, kGemmThreads, L::kTotal, stream>>>(ta, tb, s, epi);
  CDML_CHECK_CUDA(cudaGetLastError());
  if (trace_sync("gemm_tcgen05", M, N, K, grid, stream)) return -2;
  return s.num_splits;
}

// Resident-B launch (K <= 256, both operands K-major).  Chooses the row-tile chunking so that units fill whole waves.
constexpr int kResBStages = 4;  // 6 stages (224 KB) leave no L1 for the epilogue's global loads and measured slower
inline bool resb_applicable(int64_t K) {
  static int off = -1;   // CDML_NO_RESB=1 forces the generic kernel (A/B measurement aid)
  if (off < 0) off = getenv("CDML_NO_RESB") != nullptr ? 1 : 0;
  return off == 0 && K <= 4 * kBK;
}

template <class Epi, int kEpiWarps = 8>
static int launch_gemm_resb(cdml_ctx* ctx, const void* A, int64_t lda, const void* B, int64_t ldb, int64_t M, int64_t N,
                            int64_t K, int dtype16, const Epi& epi, cudaStream_t stream, int n_fastest = 0) {
  using L = ResBSmem<kBN, kResBStages, kEpiWarps, Epi::kRowConsts, Epi::kTmaStore ? 2 : 1>;
  static_assert(L::kTotal <= 232448, "resident-B kernel: shared memory over the 227 KB limit");
  CUtensorMap ta, tb;
  int rc = make_tmap_2d(ctx, &ta, A, dtype16, K, M, lda, kBK, kBM);
  if (rc) return rc;
  rc = make_tmap_2d(ctx, &tb, B, dtype16, K, N, ldb, kBK, kBN);
  if (rc) return rc;
  ResBShape s;
  s.M = static_cast<int>(M), s.N = static_cast<int>(N), s.K = static_cast<int>(K);
  s.m_tiles = (s.M + kBM - 1) / kBM;
  s.n_tiles = (s.N + kBN - 1) / kBN;
  s.num_kb = (s.K + kBK - 1) / kBK;
  // chunks per column block: whole waves of SMs, >= 8 row tiles per unit when possible
  int best = 1;
  double best_eff = -1.0;
  const int cmax = max(1, min(s.m_tiles / 8, 4 * ctx->num_sms));
  for (int c = 1; c <= cmax; ++c) {
    const int tpc = (s.m_tiles + c - 1) / c;
    const int ceff = (s.m_tiles + tpc - 1) / tpc;
    if (ceff != c) continue;
    const long units = static_cast<long>(s.n_tiles) * c;
    const long waves = (units + ctx->num_sms - 1) / ctx->num_sms;
    double eff = static_cast<double>(units) / static_cast<double>(waves * ctx->num_sms);
    eff -= 0.15 / tpc;   // panel reload bubble per unit
    if (eff > best_eff) best_eff = eff, best = c;
  }
  s.m_chunks = best;
  s.tiles_per_chunk = (s.m_tiles + best - 1) / best;
  s.n_fastest = n_fastest;
  s.idesc = make_idesc_f16(dtype16 == CDML_BF16 ? 1 : 0, 0, 0, kBM, kBN);
  auto kern = gemm_resb_tcgen05_kernel<kBN, kResBStages, Epi, kEpiWarps>;
  static bool attr_set = false;
  if (!attr_set) {
    CDML_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kTotal));
    attr_set = true;
  }
  const long units = static_cast<long>(s.n_tiles) * s.m_chunks;
  const int grid = static_cast<int>(units < ctx->num_sms ? units : ctx->num_sms);
  kern<<<grid, 128 + 32 * kEpiWarps, L::kTotal, stream>>>(ta, tb, s, epi);
  CDML_CHECK_CUDA(cudaGetLastError());
  if (trace_sync(Epi::kTmaStore ? "gemm_resb[tma]" : "gemm_resb", M, N, K, grid, stream)) return -2;
  return 1;
}

}  // namespace cdml
