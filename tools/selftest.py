"""GPU bring-up checks for libcdml kernels against torch (checker only).  Each group runs in its own process
(tools/run_selftest.sh) so a trapped kernel cannot poison the rest.   python tools/selftest.py <group>"""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import cdml_b200  # noqa: F401
from cdml_b200 import ops
from cdml_b200._lib import BF16, EPI_L2NORM, EPI_MASK_LEAKY, EPI_STORE_16, EPI_STORE_F32, F16

dev = torch.device("cuda:0")
torch.manual_seed(0)


def report(name, got, ref, tol):
  got, ref = got.float(), ref.float()
  err = (got - ref).abs()
  denom = ref.abs().max().item() + 1e-30
  rel = err.max().item() / denom
  ok = rel <= tol and torch.isfinite(got).all().item()
  print("%-58s max_abs=%.3e rel=%.3e tol=%.1e %s" % (name, err.max().item(), rel, tol, "OK" if ok else "FAIL"), flush=True)
  if not ok:
    bad = (err > tol * denom)
    rows = bad.any(1).nonzero().flatten()
    cols = bad.any(0).nonzero().flatten()
    print("   bad rows: n=%d first=%s | bad cols: n=%d first=%s" % (rows.numel(), rows[:12].tolist(), cols.numel(), cols[:12].tolist()))
    print("   got[0,:8]=%s\n   ref[0,:8]=%s" % (got[0, :8].tolist(), ref[0, :8].tolist()))
  return ok


def mk(shape, dt, scale=1.0):
  return (torch.randn(shape, device=dev) * scale).to(dt)


def gemm_case(M, N, K, amn, bmn, dt=torch.float16, splits=1, tag=""):
  p8 = lambda n: (n + 7) // 8 * 8
  A = mk((K, p8(M)) if amn else (M, p8(K)), dt)
  B = mk((K, p8(N)) if bmn else (N, p8(K)), dt)
  Af = A.float()[:, :M].t() if amn else A.float()[:, :K]
  Bf = B.float()[:, :N] if bmn else B.float()[:, :K].t()
  ref = Af @ Bf
  if splits == 1:
    out = torch.full((M, N), float("nan"), device=dev)
    ops.gemm16(A, B, M, N, K, amn, bmn, EPI_STORE_F32, out)
  else:
    if splits <= 0:
      splits = max(ops.auto_splits(A, M, N, K), 1)
    parts = torch.full((splits, M, N), float("nan"), device=dev)
    used = ops.gemm16(A, B, M, N, K, amn, bmn, EPI_STORE_F32, parts, num_splits=splits, split_stride=M * N)
    out = torch.empty((M, N), device=dev)
    ops.sum_partials(parts, used, M * N, M * N, out)
    tag += " used=%d" % used
  torch.cuda.synchronize()
  return report("gemm M=%d N=%d K=%d A%s B%s %s%s" % (M, N, K, "mn" if amn else "k", "mn" if bmn else "k",
                                                      str(dt).split(".")[-1], tag), out, ref, 2e-3 if dt == torch.float16 else 2e-2)


def group_rowops():
  G, F = 1000, 1500
  table = torch.rand((G, F), device=dev)
  idx = torch.randint(0, G, (257, 3), device=dev)
  out = ops.gather_rows(table, idx)
  print("gather fp32 int64 bit-exact:", torch.equal(out, table[idx.reshape(-1)]))
  out = ops.gather_rows(table, idx.to(torch.int32))
  print("gather fp32 int32 bit-exact:", torch.equal(out, table[idx.reshape(-1)]))
  t16 = torch.rand((G, 1504), device=dev).half()
  print("gather fp16 bit-exact:", torch.equal(ops.gather_rows(t16, idx), t16[idx.reshape(-1)]))
  todd = torch.rand((G, 13), device=dev)
  print("gather odd width bit-exact:", torch.equal(ops.gather_rows(todd, idx), todd[idx.reshape(-1)]))
  neg = torch.tensor([-1, 0, G - 1, G], device=dev)
  o = ops.gather_rows(table, neg)
  print("gather wrap/oob: wrap", torch.equal(o[0], table[-1]), "oob zero", bool((o[3] == 0).all()), "flag", ops.poll_errors(table))
  x16, x32, ss = ops.rows_normalize_cast(table, F16, 1, want_fp32=True, want_sumsq=True)
  ref = table / table.norm(dim=1, keepdim=True)
  report("normalize fp32", x32, ref, 1e-6)
  report("normalize fp16", x16[:, :F], ref, 1e-3)
  print("normalize pad zero:", bool((x16[:, F:] == 0).all()), "sumsq~1:", float((ss - 1).abs().max()))
  # hinge
  B, D = 1000, 256
  E = torch.nn.functional.normalize(torch.randn((3 * B, D), device=dev), dim=1)
  Et = E.view(B, 3, D)
  pos = ((Et[:, 0] - Et[:, 1]) ** 2).sum(-1)
  negd = ((Et[:, 0] - Et[:, 2]) ** 2).sum(-1)
  hin = (pos - negd + 0.8).clamp(min=0)
  rinv = torch.rand((3 * B,), device=dev) + 0.5
  dz = torch.empty((3 * B, D), device=dev, dtype=torch.float16)
  r = ops.triplet_hinge(E, B, 0.8, grad_scale=1.0, rinv=rinv, want_dE=True, dz16=dz)
  report("hinge pos", r["pos_dist"][None], pos[None], 1e-5)
  report("hinge hinge", r["hinge_dist"][None], hin[None], 1e-5)
  print("stats", r["stats"].tolist(), "ref", [hin.mean().item(), pos.mean().item(), negd.mean().item(), (hin > 0).sum().item()])
  act = (hin > 0).float()[:, None]
  g = torch.stack([2 * (Et[:, 2] - Et[:, 1]) * act, 2 * (Et[:, 1] - Et[:, 0]) * act, 2 * (Et[:, 0] - Et[:, 2]) * act], 1).view(3 * B, D)
  report("hinge dE", r["dE"], g, 1e-5)
  dzr = (g - E * (E * g).sum(-1, keepdim=True)) * rinv[:, None] * torch.where(E > 0, 1.0, 0.2)
  report("hinge dz16", dz, dzr, 2e-3)
  nr = torch.randint(0, 3 * B, (B,), device=dev, dtype=torch.int32)
  r2 = ops.triplet_hinge(E, B, 0.8, neg_row=nr, grad_scale=1.0, rinv=rinv, want_dE=True, dz16=dz)
  En = E[nr.long()]
  negd2 = ((Et[:, 0] - En) ** 2).sum(-1)
  hin2 = (pos - negd2 + 0.8).clamp(min=0)
  act2 = (hin2 > 0).float()[:, None]
  g2 = torch.zeros_like(E)
  g2.index_add_(0, torch.arange(0, 3 * B, 3, device=dev), 2 * (En - Et[:, 1]) * act2)
  g2.index_add_(0, torch.arange(1, 3 * B, 3, device=dev), 2 * (Et[:, 1] - Et[:, 0]) * act2)
  g2.index_add_(0, nr.long(), 2 * (Et[:, 0] - En) * act2)
  report("hinge mined dE", r2["dE"], g2, 1e-5)
  # colsum / adam / cast
  X = mk((3000, 5000), torch.float16)
  cs = torch.empty((5000,), device=dev)
  ops.colsum16(X, 3000, 5000, cs)
  report("colsum16", cs[None], X.float().sum(0)[None], 1e-5)
  n = 100003
  w = torch.randn(n, device=dev); m = torch.zeros(n, device=dev); v = torch.zeros(n, device=dev); g = torch.randn(n, device=dev)
  w0 = w.clone()
  step = torch.zeros(1, dtype=torch.int64, device=dev); sc = torch.zeros(4, device=dev)
  w16 = torch.empty(n, device=dev, dtype=torch.float16)
  for t in range(1, 4):
    ops.adam_prepare(step, sc, 1e-3)
    ops.adam_apply(w, m, v, g, sc, grad_scale=0.5, w16=w16)
  mr = torch.zeros(n, device=dev, dtype=torch.float64); vr = mr.clone(); wr = w0.double()
  for t in range(1, 4):
    gg = g.double() * 0.5
    lr_t = 1e-3 * (1 - 0.999 ** t) ** 0.5 / (1 - 0.9 ** t)
    mr = 0.9 * mr + 0.1 * gg; vr = 0.999 * vr + 0.001 * gg * gg
    wr = wr - lr_t * mr / (vr.sqrt() + 1e-8)
  report("adam w (3 steps)", w[None], wr[None], 1e-6)
  report("adam w16", w16[None], wr[None], 1e-3)
  print("step counter", step.item())
  V = torch.randn((500, 256), device=dev); pairs = torch.randint(0, 500, (300, 2), device=dev)
  md = ops.mean_pair_dist(V, pairs)
  print("mean_pair_dist", md.item(), ((V[pairs[:, 0]] - V[pairs[:, 1]]) ** 2).sum(-1).mean().item())


def group_gemm_basic():
  gemm_case(128, 256, 64, 0, 0)
  gemm_case(128, 256, 256, 0, 0)
  gemm_case(128, 256, 64, 0, 0, torch.bfloat16)
  gemm_case(256, 512, 512, 0, 0)
  gemm_case(300, 700, 200, 0, 0)
  gemm_case(4096, 5000, 256, 0, 0)


def group_gemm_kslices():
  # isolate each UMMA k-step of the K-major path
  M, N, K = 128, 256, 64
  for j in range(4):
    A = torch.zeros((M, K), device=dev, dtype=torch.float16)
    A[:, 16 * j:16 * j + 16] = mk((M, 16), torch.float16)
    B = mk((N, K), torch.float16)
    out = torch.full((M, N), float("nan"), device=dev)
    ops.gemm16(A, B, M, N, K, 0, 0, EPI_STORE_F32, out)
    torch.cuda.synchronize()
    report("k-slice %d (AK,BK)" % j, out, A.float() @ B.float().t(), 2e-3)


def group_gemm_bmn():
  gemm_case(128, 256, 64, 0, 1)
  gemm_case(128, 256, 256, 0, 1)
  gemm_case(384, 512, 320, 0, 1, torch.bfloat16)
  gemm_case(300, 5000, 1500, 0, 1)
  gemm_case(3072, 256, 5000, 0, 1)


def group_gemm_mnmn():
  gemm_case(128, 256, 64, 1, 1)
  gemm_case(128, 256, 256, 1, 1)
  gemm_case(1500, 5000, 3072, 1, 1)
  gemm_case(5000, 256, 3072, 1, 1)
  gemm_case(1500, 5000, 3072, 1, 1, splits=4)
  gemm_case(5000, 256, 6144, 1, 1, splits=0, tag=" auto")


def group_gemm_epilogues():
  M, N, K = 1000, 5000, 1500
  A = mk((M, 1504), torch.float16, 0.05)
  W = mk((K, N), torch.float16, 0.05)
  bias = torch.randn(N, device=dev) * 0.1
  ref = torch.nn.functional.leaky_relu(A[:, :K].float() @ W.float() + bias, 0.2)
  out16 = torch.empty((M, N), device=dev, dtype=torch.float16)
  ops.gemm16(A, W, M, N, K, 0, 1, EPI_STORE_16, out16, bias=bias, alpha=0.2)
  report("epi STORE_16 bias+leaky", out16, ref, 2e-3)
  out32 = torch.empty((M, N), device=dev)
  ops.gemm16(A, W, M, N, K, 0, 1, EPI_STORE_F32, out32, bias=bias, alpha=0.2)
  report("epi STORE_F32 bias+leaky", out32, ref, 2e-3)
  # L2NORM
  H, D = 5000, 256
  Hh = mk((M, H), torch.float16, 0.1)
  W2 = mk((H, D), torch.float16, 0.03)
  b2 = torch.randn(D, device=dev) * 0.01
  y = torch.nn.functional.leaky_relu(Hh.float() @ W2.float() + b2, 0.2)
  ss = (y * y).sum(-1, keepdim=True).clamp(min=1e-12)
  e_ref = y * ss.rsqrt()
  e = torch.empty((M, D), device=dev); rinv = torch.empty((M,), device=dev); e16 = torch.empty((M, D), device=dev, dtype=torch.float16)
  ops.gemm16(Hh, W2, M, D, H, 0, 1, EPI_L2NORM, e, bias=b2, alpha=0.2, aux0=rinv, aux1=e16)
  report("epi L2NORM e", e, e_ref, 2e-3)
  report("epi L2NORM rinv", rinv[None], ss.rsqrt().flatten()[None], 2e-3)
  report("epi L2NORM e16", e16, e_ref, 3e-3)
  # MASK_LEAKY (dgrad)
  dz = mk((M, D), torch.float16)
  mask = mk((M, H), torch.float16)
  ref = (dz.float() @ W2.float().t()) * torch.where(mask.float() > 0, 1.0, 0.2)
  o = torch.empty((M, H), device=dev, dtype=torch.float16)
  ops.gemm16(dz, W2, M, H, D, 0, 0, EPI_MASK_LEAKY, o, alpha=0.2, aux1=mask)
  report("epi MASK_LEAKY", o, ref, 2e-3)


def group_gemm_resb():
  # K <= 256, K-major x K-major, M >= 1024 -> resident-B kernel
  gemm_case(4096, 5000, 256, 0, 0)
  gemm_case(3000, 700, 200, 0, 0)
  gemm_case(1024, 256, 64, 0, 0, torch.bfloat16)
  gemm_case(20000, 1000, 256, 0, 0)
  gemm_case(1300, 70000, 256, 0, 0)
  M, H, D = 4000, 5000, 256
  W2 = mk((H, D), torch.float16, 0.03)
  dz = mk((M, D), torch.float16)
  mask = mk((M, H), torch.float16)
  ref = (dz.float() @ W2.float().t()) * torch.where(mask.float() > 0, 1.0, 0.2)
  o = torch.empty((M, H), device=dev, dtype=torch.float16)
  ops.gemm16(dz, W2, M, H, D, 0, 0, EPI_MASK_LEAKY, o, alpha=0.2, aux1=mask)
  report("resb epi MASK_LEAKY", o, ref, 2e-3)


def group_gemm_perf():
  for (M, N, K, amn, bmn) in [(196608, 5000, 1500, 0, 1), (196608, 256, 5000, 0, 1), (196608, 5000, 256, 0, 0),
                              (1500, 5000, 196608, 1, 1), (5000, 256, 196608, 1, 1), (8192, 8192, 8192, 0, 0)]:
    A = mk((K, (M + 7) // 8 * 8) if amn else (M, (K + 7) // 8 * 8), torch.float16, 0.05)
    B = mk((K, N) if bmn else (N, (K + 7) // 8 * 8), torch.float16, 0.05)
    splits = ops.auto_splits(A, M, N, K)
    if splits > 1:
      out = torch.empty((splits, M, N), device=dev)
    else:
      out = torch.empty((M, N), device=dev, dtype=torch.float16)
    def run():
      if splits > 1:
        ops.gemm16(A, B, M, N, K, amn, bmn, EPI_STORE_F32, out, num_splits=splits, split_stride=M * N)
      else:
        ops.gemm16(A, B, M, N, K, amn, bmn, EPI_STORE_16, out)
    for _ in range(2):
      run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
      run()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    print("perf M=%d N=%d K=%d A%s B%s splits=%d: %.3f ms  %.1f TFLOP/s" % (M, N, K, "mn" if amn else "k", "mn" if bmn else "k",
                                                                           splits, ms, 2.0 * M * N * K / ms / 1e9), flush=True)




def group_gemm_null():
  """main loop only (epi 100) / + TMEM reads (epi 101) / + fp16 stores (epi 1), each shape timed 3x in one process"""
  shapes = [(196608, 5000, 256, 0, 0), (65536, 65536, 256, 0, 0), (196608, 5000, 1500, 0, 1), (8192, 8192, 8192, 0, 0)]
  for (M, N, K, amn, bmn) in shapes:
    A = mk((K, (M + 7) // 8 * 8) if amn else (M, (K + 7) // 8 * 8), torch.float16, 0.05)
    B = mk((K, N) if bmn else (N, (K + 7) // 8 * 8), torch.float16, 0.05)
    out = torch.empty((M, N), device=dev, dtype=torch.float16) if M * N <= 2 ** 31 else torch.empty((16,), device=dev)
    for epi in (100, 101, 1):
      if epi == 1 and out.dim() == 1:
        continue
      res = []
      for rep in range(3):
        for _ in range(2):
          ops.gemm16(A, B, M, N, K, amn, bmn, epi, out, ld_out=N)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
          ops.gemm16(A, B, M, N, K, amn, bmn, epi, out, ld_out=N)
        e1.record()
        torch.cuda.synchronize()
        res.append(e0.elapsed_time(e1) / 5)
      ms = min(res)
      print("null M=%d N=%d K=%d epi=%d resb=%s: %.3f ms (runs %s)  %.1f TFLOP/s" %
            (M, N, K, epi, "on" if (not amn and not bmn and K <= 256 and M >= 1024) else "off", ms, ["%.3f" % r for r in res], 2.0 * M * N * K / ms / 1e9), flush=True)


if __name__ == "__main__":
  t0 = time.time()
  globals()["group_" + sys.argv[1]]()
  torch.cuda.synchronize()
  print("[group %s done in %.1fs]" % (sys.argv[1], time.time() - t0), flush=True)
