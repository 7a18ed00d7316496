"""Local, HDFS-free composition of the reference's serving cycle (cdml_run.sh:73-150; BASELINE configs[4]) through the
public API: train (train.Trainer on *.train index triplets) -> embed every guid (predict.Prediction.run_features) ->
exact top-k KNN (faiss_knn.calc_knn semantics, device resident) -> raw-feature KNN + de-similarity filter
(faiss_knn.py:376-378, iter_desim_mp) -> knn_split* files (faiss_knn.write_knn, native formatter).

  python tools/cycle.py [--guids G] [--triplets T] [--batch B] [--knn-k K] [--write-rows R] [--out DIR]

Defaults are a 1/10-scale cycle (1M guids, 5M triplets, 1M x 1M KNN) that finishes in about a minute on one B200;
--guids 10000000 --triplets 50000000 is configs[4] itself.  Features and cowatch pairs are synthetic and generated on
the device (a 10M x 1500 float32 feature file would be 60 GB of host I/O that has nothing to do with the path)."""
import argparse
import json
import os
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import cdml_b200  # noqa: F401
from cdml_b200 import engine, faiss_knn, ops, predict

ap = argparse.ArgumentParser()
ap.add_argument("--guids", type=int, default=1000000)
ap.add_argument("--triplets", type=int, default=5000000)
ap.add_argument("--batch", type=int, default=65536)
ap.add_argument("--knn-k", type=int, default=100)
ap.add_argument("--write-rows", type=int, default=100000, help="rows of the KNN result formatted into knn_split* files")
ap.add_argument("--out", default="")
ap.add_argument("--lr", type=float, default=1e-4, help="Adam base learning rate (1e-3 collapses this synthetic set within 76 steps)")
ap.add_argument("--no-desim", action="store_true", help="skip the raw-feature KNN + de-similarity stage")
ap.add_argument("--feat-k", type=int, default=26, help="desim_nearest_num (faiss_knn.py:46)")
ap.add_argument("--mine", action="store_true", help="in-batch semi-hard mining (default: the reference's random negatives)")
ap.add_argument("--mine-dw", action="store_true", help="in-batch distance-weighted negative sampling (not with --mine)")
ap.add_argument("--dw-cutoff", type=float, default=0.5, help="distance cutoff of --mine-dw")
ap.add_argument("--centre-weight", type=float, default=1.0, help="weight of the cluster centre in a feature row (row = signal * centre + "
                "noise_weight * U[0,1)); 1.0 / 0.25 = the well-separated default, 0.3 / 1.0 = clusters the tower has to learn")
ap.add_argument("--noise-weight", type=float, default=0.25)
ap.add_argument("--clusters", type=int, default=1000)
ap.add_argument("--knn-block", type=int, default=262144, help="queries per sharded search call")
args = ap.parse_args()
# one process per GPU under torchrun: the feature table is replicated (every rank generates the same rows from the same
# seed), every rank trains its own batches (NCCL all-reduce inside the captured step), embeds its slice of the guids,
# holds its row shard of the index and ends up with the KNN lists of its slice of the queries (written as its own files)
world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
dev = torch.device("cuda:%d" % local)
torch.cuda.set_device(local)
pg = None
if world > 1:
  torch.distributed.init_process_group("nccl", device_id=dev)
  pg = torch.distributed.group.WORLD
G, F, B = args.guids, 1500, args.batch
gen = torch.Generator(device=dev)
gen.manual_seed(11)
t = {}


def tick(name, t0):
  torch.cuda.synchronize()
  if world > 1:
    torch.distributed.barrier()
  t[name] = time.time() - t0


# ---- stage 0: resident feature table (normalised 16-bit, built slab by slab) + guid clusters so that there is a signal
t0 = time.time()
eng = engine.TowerEngine([F, 5000, 256], device=dev, base_lr=args.lr, margin=0.8, process_group=pg)
table16 = torch.empty((G, eng.F_pad), dtype=eng.t16, device=dev)
feats32 = None if args.no_desim else torch.empty((G, F), dtype=torch.float32, device=dev)   # features.npy of predict.py:150
NC = args.clusters
centres = torch.rand((NC, F), generator=gen, device=dev)
cluster = torch.randint(0, NC, (G,), generator=gen, device=dev)
for s in range(0, G, 65536):
  rows = min(65536, G - s)
  slab = args.centre_weight * centres[cluster[s:s + rows]] + args.noise_weight * torch.rand((rows, F), generator=gen, device=dev)
  eng.prepare_table(slab, out=table16[s:s + rows])
  if feats32 is not None:
    feats32[s:s + rows] = slab
tick("build_feature_table_s", t0)

# ---- stage 1: one training epoch over `triplets` cowatch pairs (anchor/positive from the same cluster, random negative)
t0 = time.time()
steps = max(1, args.triplets // B)
if args.mine and args.mine_dw:
  raise SystemExit("--mine and --mine-dw exclude each other")
mine = "distance_weighted" if args.mine_dw else args.mine
eng.dw_cutoff = args.dw_cutoff
replay = eng.capture_step(table16, B, mine=mine)
order = torch.argsort(cluster)
start = torch.searchsorted(cluster[order], torch.arange(NC + 1, device=dev))
losses = []
steps = max(1, steps // world)             # `triplets` is the size of the epoch: the ranks share it
gen.manual_seed(1000 + rank)               # from here on every rank draws its own cowatch pairs


def same_cluster_pairs(n):
  a = torch.randint(0, G, (n,), generator=gen, device=dev)
  c = cluster[a]
  span = (start[c + 1] - start[c]).clamp(min=1)
  return a, order[start[c] + (torch.rand((n,), generator=gen, device=dev) * span).long() % span]


def eval_dists():
  """Evaluation.mean_dist (evaluate.py:57-73) of 20 000 held-out cowatch pairs next to 20 000 random pairs: training must
  shrink the first relative to the second (a collapse shrinks both)."""
  a, p = same_cluster_pairs(20000)
  r = torch.randint(0, G, (20000,), generator=gen, device=dev)
  rows = torch.cat([a, p, r])
  e = eng.forward_rows(table16[rows], rows.numel())["e"]
  pairs_pos = torch.stack([torch.arange(20000, device=dev), torch.arange(20000, 40000, device=dev)], 1)
  pairs_rnd = torch.stack([torch.arange(20000, device=dev), torch.arange(40000, 60000, device=dev)], 1)
  return float(ops.mean_pair_dist(e, pairs_pos).item()), float(ops.mean_pair_dist(e, pairs_rnd).item())


eval_before = eval_dists()
for i in range(steps):
  a = torch.randint(0, G, (B,), generator=gen, device=dev)
  c = cluster[a]
  span = (start[c + 1] - start[c]).clamp(min=1)
  p = order[start[c] + (torch.rand((B,), generator=gen, device=dev) * span).long() % span]
  n = torch.randint(0, G, (B,), generator=gen, device=dev)
  st = replay(torch.stack([a, p, n], 1))
  if i % 16 == 0 or i == steps - 1:
    losses.append(float(st[0].item()))
tick("train_s", t0)
eval_after = eval_dists()

# ---- stage 2: embed every guid (Prediction.run_features on the live engine, batches of 100 000 like predict.py:42); with
#      N ranks every rank embeds its contiguous slice of the rows and one all-gather completes the query set everywhere
t0 = time.time()
pred = predict.Prediction(sess=eng)
glo, ghi = rank * G // world, (rank + 1) * G // world
emb = torch.empty((G, 256), dtype=torch.float32, device=dev)
for s in range(glo, ghi, 100000):
  rows = min(100000, ghi - s)
  x16 = table16[s:s + rows]                                   # already normalised 16-bit rows: forward only
  emb[s:s + rows].copy_(eng.forward_rows(x16, rows)["e"])
if world > 1:
  per = (G + world - 1) // world
  assert G % world == 0, "--guids must be a multiple of the world size"
  torch.distributed.all_gather_into_tensor(emb, emb[glo:ghi].clone(), group=pg)
tick("embed_s", t0)
if world > 1:
  del replay
  eng._graph_keepalive = None               # the captured step holds NCCL kernels: release it before the KNN collectives

# ---- stage 3: exact top-k over all embeddings, queries = the index itself (faiss_knn.py:105-106).  N ranks: the index is
#      row-sharded (rank r holds rows [r*G/N, (r+1)*G/N)), every block of queries goes through faiss_knn.sharded_search and
#      leaves rank r with the lists of ITS slice of the block
t0 = time.time()
index = ops.FlatIndex(emb[glo:ghi].contiguous() if world > 1 else emb, "L2")
blk = args.knn_block if world > 1 else 262144
nblocks = (G + blk - 1) // blk
mine_rows = []                              # global query ids of the lists this rank ends up with
Dl, Il = [], []
for s in range(0, G, blk):
  rows = min(blk, G - s)
  d_, i_ = faiss_knn.sharded_search(index, emb[s:s + rows], args.knn_k, glo, "L2", pg, gather=False)
  if world > 1:
    per = -(-rows // world)
    mine_rows.append(torch.arange(s + rank * per, s + min((rank + 1) * per, rows), device=dev))
  else:
    mine_rows.append(torch.arange(s, s + rows, device=dev))
  Dl.append(d_), Il.append(i_)
  if os.environ.get("CYCLE_DEBUG"):
    print("block %d: stats %s, ids out of range %d, emb finite %s, loss %s" % (s, index.last_stats(), int(((i_ < -1) | (i_ >= G)).sum().item()),
          bool(torch.isfinite(emb[s:s + rows]).all().item()), losses[-3:]), file=sys.stderr, flush=True)
D, I, qrows = torch.cat(Dl), torch.cat(Il), torch.cat(mine_rows)
del Dl, Il
stats = index.last_stats()
tick("knn_s", t0)
same_cluster = (cluster[I[:, 1:6]] == cluster[qrows][:, None]).float().mean()
self_first = (I[:, 0] == qrows).float().mean()
if world > 1:
  both = torch.stack([same_cluster, self_first]) / world
  torch.distributed.all_reduce(both, group=pg)
  same_cluster, self_first = both[0], both[1]
same_cluster, self_first = float(same_cluster.item()), float(self_first.item())

# ---- stage 3b: raw-feature KNN (faiss_knn.py:378) and the de-similarity filter of the embedding lists (iter_desim_mp)
desim_info = None
if not args.no_desim and world == 1:
  t0 = time.time()
  index.close()
  torch.nn.functional.normalize(feats32, dim=1, out=feats32)            # calc_knn(l2_norm=True): plumbing-level normalisation of the synthetic rows
  findex = ops.FlatIndex(feats32, "L2")
  fD = torch.empty((G, args.feat_k), dtype=torch.float32, device=dev)
  fI = torch.empty((G, args.feat_k), dtype=torch.int64, device=dev)
  for s in range(0, G, 131072):
    rows = min(131072, G - s)
    fD[s:s + rows], fI[s:s + rows] = findex.search(feats32[s:s + rows], args.feat_k)
  fstats = findex.last_stats()
  findex.close()
  tick("feature_knn_s", t0)
  t0 = time.time()
  I_desim = ops.desim(I, fI, fD, 1.4, 31)
  tick("desim_s", t0)
  desim_info = {"feature_knn_queries_per_s": G / t["feature_knn_s"], "desim_rows_per_s": G / t["desim_s"],
                "dropped_fraction": float((I_desim < 0).float().mean().item()),
                "feature_knn_fallback_queries_last_block": fstats["fallback_queries"]}
  I = I_desim

# ---- stage 4: knn_split* files (write_knn format) for the first `write_rows` queries this rank holds
t0 = time.time()
out_dir = args.out or tempfile.mkdtemp(prefix="cdml_cycle_")
R = min(args.write_rows, int(qrows.numel()))
if R:
  q0 = int(qrows[0].item())
  assert bool((qrows[:R] == torch.arange(q0, q0 + R, device=dev)).all().item()) or world > 1
  dm = {i: "g%08d" % i for i in range(G)} if world == 1 else None
  if world == 1:
    faiss_knn.write_knn(out_dir, split_num=10, D=D[:R].cpu().numpy(), I=I[:R].cpu().numpy(), prefix="knn_split", decode_map=dm)
  else:       # every rank writes its own split file of the rows it holds (consecutive global query ids within a block)
    table = faiss_knn.GuidTable({i: "g%08d" % i for i in range(G)})
    os.makedirs(out_dir, exist_ok=True)
    first_block = min(R, int((qrows[:R] - qrows[0] == torch.arange(R, device=dev)).sum().item()))
    faiss_knn.write_process(out_dir, rank, q0, D[:first_block].cpu().numpy(), I[:first_block].cpu().numpy(), "knn_split", decode_map=table)
    R = first_block
tick("write_s", t0)
if rank == 0:
  print(json.dumps({"guids": G, "triplets": steps * B * world, "steps_per_rank": steps, "n_gpus": world, "knn_k": args.knn_k, "seconds": t,
                  "train_triplets_per_s": steps * B * world / t["train_s"], "embed_rows_per_s": G / t["embed_s"],
                  "knn_queries_per_s": G / t["knn_s"], "loss_first_last": [losses[0], losses[-1]], "loss_curve": [round(x, 5) for x in losses],
                  "eval_cowatch_vs_random_pair_dist_before": eval_before, "eval_cowatch_vs_random_pair_dist_after": eval_after,
                  "features": {"signal": args.centre_weight, "noise": args.noise_weight, "clusters": NC, "lr": args.lr},
                  "top5_same_cluster": same_cluster, "self_is_first_neighbour": self_first,
                  "knn_fallback_queries_last_block": stats["fallback_queries"], "mining": bool(mine),
                  "mining_mode": "distance_weighted" if args.mine_dw else "semihard" if args.mine else None,
                  "dw_cutoff": args.dw_cutoff if args.mine_dw else None, "desim": desim_info,
                  "write_rows_per_rank": R, "write_rows_per_s": R / t["write_s"] if R else None, "out_dir": out_dir}))
if world > 1:
  torch.distributed.barrier()
  torch.distributed.destroy_process_group()
