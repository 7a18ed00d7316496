"""Cost of distance-weighted negative sampling next to semi-hard mining at the bench batch: both scans alone (prepare +
two resident-B scans + finalize) in three regimes, with re-scanned (anchor, 32-candidate chunk) pairs per anchor, and the
CUDA-graph training step of the bench tower with each mode.  The modes are timed alternately, `--rounds` times; the
output is the median (min-max) over the rounds.

  python tools/mine_dw_diag.py [--batch 65536] [--rounds 5] [--reps 5] [--no-step]
"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import cdml_b200  # noqa: F401
from cdml_b200 import engine, ops

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=65536)
ap.add_argument("--rounds", type=int, default=5)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--steps", type=int, default=10, help="graph replays per timed round of the training step")
ap.add_argument("--no-step", action="store_true")
args = ap.parse_args()
dev = torch.device("cuda:0")
torch.cuda.set_device(0)
try:
  print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip())
except OSError:
  print("nvidia-smi not found: GPU name and power limit unknown")
gen = torch.Generator(device=dev)
gen.manual_seed(1)
B, D = args.batch, 256


def timed(fn, reps):
  fn()
  torch.cuda.synchronize()
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  a.record()
  for _ in range(reps):
    fn()
  b.record()
  torch.cuda.synchronize()
  return a.elapsed_time(b) / reps


def summary(xs):
  return "%.3f ms (%.3f-%.3f)" % (np.median(xs), min(xs), max(xs))


step = torch.zeros(1, dtype=torch.int64, device=dev)
modes = {"semihard": lambda E16, E, idx: ops.mine_semihard(E16, E, idx, B, 0.8, want_dist=False),
         "distance_weighted": lambda E16, E, idx: ops.mine_distance_weighted(E16, E, idx, B, 0.8, 0.5, 1, step, want_dist=False)}
# regimes: uniform (random points of the sphere), clustered (1000 clusters, anchor and positive from one cluster) and
# contracted (every embedding within ~0.02 of one direction, as after the semi-hard collapse or an untrained tower)
idx = torch.randint(0, 1000000, (B, 3), generator=gen, device=dev)
for regime in ("uniform", "clustered", "contracted"):
  if regime == "uniform":
    E = torch.nn.functional.normalize(torch.randn((3 * B, D), generator=gen, device=dev), dim=1)
  elif regime == "clustered":
    centres = torch.randn((1000, D), generator=gen, device=dev)
    c = torch.randint(0, 1000, (B,), generator=gen, device=dev)
    cn = torch.randint(0, 1000, (B,), generator=gen, device=dev)
    cl = torch.stack([c, c, cn], 1).reshape(-1)
    E = torch.nn.functional.normalize(centres[cl] + 0.5 * torch.randn((3 * B, D), generator=gen, device=dev), dim=1)
  else:
    base = torch.randn((1, D), generator=gen, device=dev)
    E = torch.nn.functional.normalize(base + 0.02 * torch.randn((3 * B, D), generator=gen, device=dev), dim=1)
  E16 = E.half()
  times = {m: [] for m in modes}
  for _ in range(args.rounds):
    for m, fn in modes.items():
      times[m].append(timed(lambda: fn(E16, E, idx), args.reps))
  for m, fn in modes.items():
    rescans = []
    for t in range(3):                        # distance-weighted: three draws
      step.fill_(t)
      neg, _ = fn(E16, E, idx)
      rescans.append(ops.mine_stats(E)["rescans"] / B)
    mined = float((neg.long() != 3 * torch.arange(B, device=dev) + 2).float().mean().item())
    print("scan %-10s %-17s %s  re-scans/anchor %.2f (%s)  mined %.3f" % (
        regime, m, summary(times[m]), np.mean(rescans), " ".join("%.2f" % r for r in rescans), mined))
  print("scan %-10s ratio distance_weighted / semihard (median) %.2f" % (regime, np.median(times["distance_weighted"]) /
                                                                          np.median(times["semihard"])))

if not args.no_step:
  # the bench workload's tower (VNet [1500, 5000, 256]) on uniform features, one CUDA-graph replay per step
  G, F = 1000000, 1500
  feats = torch.rand((G, F), generator=gen, device=dev)
  eng = {}
  replay = {}
  for m in ("semihard", "distance_weighted"):
    eng[m] = engine.TowerEngine([F, 5000, 256], device=dev, base_lr=1e-4, margin=0.8, seed=2)
    table16 = eng[m].prepare_table(feats)
    replay[m] = eng[m].capture_step(table16, B, mine=True if m == "semihard" else m)
  del feats
  batches = [torch.randint(0, G, (B, 3), generator=gen, device=dev) for _ in range(args.steps)]
  times = {m: [] for m in replay}
  for _ in range(args.rounds):
    for m, r in replay.items():
      times[m].append(timed(lambda: [r(b) for b in batches], 1) / len(batches))
  for m in replay:
    print("step B=%d %-17s %s per graph-replayed step" % (B, m, summary(times[m])))
