"""Epilogue cost decomposition of the resident-B tcgen05 kernel (K = 256 scans): main loop alone (epilogue 100), main loop
+ TMEM reads (101), the mining scans in two regimes, and the data-gradient GEMM with the 16-bit mask vs the sign-bit mask.

  python tools/epi_diag.py [--batch 65536] [--reps 5]
"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import cdml_b200  # noqa: F401
from cdml_b200 import ops
from cdml_b200._lib import EPI_MASK_BITS, EPI_MASK_LEAKY, EPI_STORE_16

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=65536)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--only", default="", help="comma list of sections: scan, mine-structureless, mine-clustered, mine-random-sphere, dgrad")
ap.add_argument("--dgrad-n", type=int, default=5000, help="output columns of the dgrad section (5000: VNet, 1500: fusion towers)")
ap.add_argument("--no-warm", action="store_true", help="no untimed warm-up call (ncu captures: one launch per kernel)")
args = ap.parse_args()
only = set(x for x in args.only.split(",") if x)
want = lambda name: not only or name in only
dev = torch.device("cuda:0")
torch.cuda.set_device(0)
gen = torch.Generator(device=dev)
gen.manual_seed(1)
B, D = args.batch, 256


def timed(fn, reps=args.reps):
  if not args.no_warm:
    fn()
  torch.cuda.synchronize()
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  a.record()
  for _ in range(reps):
    fn()
  b.record()
  torch.cuda.synchronize()
  return a.elapsed_time(b) / reps


X = torch.nn.functional.normalize(torch.randn((B, D), generator=gen, device=dev), dim=1).half()
Y = torch.nn.functional.normalize(torch.randn((B, D), generator=gen, device=dev), dim=1).half()
sink = torch.zeros((16,), dtype=torch.float32, device=dev)
flop = 2.0 * B * B * D
for epi, name in ((100, "main loop only (no epilogue)"), (101, "main loop + TMEM reads")):
  if not want("scan"):
    continue
  ms = timed(lambda: ops.gemm16(X, Y, B, B, D, 0, 0, epi, sink))
  print("scan %dx%dx%d %-32s %.3f ms  %.0f TFLOP/s" % (B, B, D, name, ms, flop / ms / 1e9))

# mining in two regimes: structureless (all embeddings nearly parallel, like an untrained tower on uniform features) and
# clustered (1000 clusters, anchor/positive from the same cluster)
idx = torch.randint(0, 1000000, (B, 3), generator=gen, device=dev)
for regime in ("structureless", "clustered", "random-sphere"):
  if not want("mine-" + regime):
    continue
  if regime == "structureless":
    base = torch.randn((1, D), generator=gen, device=dev)
    E = torch.nn.functional.normalize(base + 0.02 * torch.randn((3 * B, D), generator=gen, device=dev), dim=1)
  elif regime == "clustered":
    centres = torch.randn((1000, D), generator=gen, device=dev)
    c = torch.randint(0, 1000, (B,), generator=gen, device=dev)
    cn = torch.randint(0, 1000, (B,), generator=gen, device=dev)
    cl = torch.stack([c, c, cn], 1).reshape(-1)
    E = torch.nn.functional.normalize(centres[cl] + 0.5 * torch.randn((3 * B, D), generator=gen, device=dev), dim=1)
  else:
    E = torch.nn.functional.normalize(torch.randn((3 * B, D), generator=gen, device=dev), dim=1)
  E16 = E.half()
  ms = timed(lambda: ops.mine_semihard(E16, E, idx, B, 0.8, want_dist=False))
  neg, _ = ops.mine_semihard(E16, E, idx, B, 0.8, want_dist=True)
  mined = float((neg.long() != 3 * torch.arange(B, device=dev) + 2).float().mean().item())
  print("mining %-14s %.3f ms for both scans + prepare/finalize (%.0f TFLOP/s), mined fraction %.3f" % (regime, ms, 2 * flop / ms / 1e9, mined))

# data gradient: dz2 [R,256] x W2 [N,256]^T -> [R,N] masked by the sign of h1 (N = 5000: VNet's layer 1)
R, N = 3 * B, args.dgrad_n
pad = lambda n: (n + 63) // 64 * 64
dz = (torch.randn((R, D), generator=gen, device=dev) * 0.1).half()
W = (torch.randn((N, D), generator=gen, device=dev) * 0.1).half()
H = torch.randn((R, pad(N + 1)), generator=gen, device=dev).half()[:, :N]
out = torch.empty((R, pad(N)), dtype=torch.float16, device=dev)[:, :N]
mask = ops.sign_mask_buffer(R, N, dev)
mask.random_(generator=gen)
for epi, name, aux in () if not want("dgrad") else ((EPI_MASK_LEAKY, "16-bit activation as mask", H), (EPI_MASK_BITS, "packed sign-bit mask", mask),
                       (EPI_STORE_16, "no mask (store only)", None)):
  ms = timed(lambda: ops.gemm16(dz, W, R, N, D, 0, 0, epi, out, alpha=0.2, aux1=aux))
  byt = R * N * 2 + R * D * 2 + (R * N * 2 if epi == EPI_MASK_LEAKY else R * N / 8 if epi == EPI_MASK_BITS else 0)
  print("dgrad %dx%dx%d %-28s %.3f ms  %.0f TFLOP/s  %.2f TB/s algorithmic" % (R, N, D, name, ms, 2.0 * R * N * D / ms / 1e9, byt / ms / 1e9))
