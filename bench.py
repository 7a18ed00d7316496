#!/usr/bin/env python
"""bench.py -- headline benchmark of the CDML hot path on B200 (one JSON line on stdout).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--no-mine] [--no-knn]

Metric (BASELINE.json): train triplets/sec.  Workload at N=1: configs[1] -- the default models.py tower
(VNet 1500->5000->256) at batch 65536 with in-batch semi-hard negative mining, feature table of 1M guids resident in
HBM.  A step = gather -> tower fwd -> mining -> hinge loss -> bwd -> Adam (+ NCCL all-reduce of the flat gradient
buffer when N>1; weak scaling: every rank keeps batch 65536).  `value` is timed with CUDA events with the index
triplets already on the device; `e2e` times the same step through the public API from pinned HOST index buffers with
the H2D copy and the D2H read of the loss inside the timed region.  The second BASELINE metric (KNN top-100
queries/sec on a 1M-item index) is reported in `knn_summary` (scalars, early in the line) and the `knn` object.
Further keys: `roofline` / `roofline_summary`, `cpu_baseline`, `clocks`, `get_batch_e2e` (host float features in),
`config0_batch1024`, `mining_regimes` (N=1), `weights_identical_across_ranks`, `strong_scaling` (N>1), `desim`.
  --tower vnet|wide|resnet   --dtype fp16|bf16   --features uniform|clustered   --scaling weak|strong   --no-extras
  --dump-outputs DIR   after the run, write what the timed paths computed as DIR/<name>.npy (see dump_outputs)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TOWERS = {"vnet": ([1500, 5000, 256], "fp16"),                      # configs[1]: the default models.py tower
          "wide": ([2048, 2048, 2048, 2048, 256], "bf16"),          # configs[2]: 2048-d input, 3 x 2048 hidden, bf16
          "resnet": ([1628, 256], "fp16")}                          # SURVEY 8f row 1: the fusion tower of train.py main()
DIMS = TOWERS["vnet"][0]


def flop_per_triplet(dims):
  """3 rows x (forward 2*in*out + weight gradient 2*in*out per layer, + data gradient 2*in*out for every layer but the
  first).  VNet: 3*(4FH + 6HD) = 113.04 MFLOP (SURVEY 8d); wide tower: 210.76 MFLOP."""
  return 3 * sum((4 if l == 0 else 6) * dims[l] * dims[l + 1] for l in range(len(dims) - 1))


FLOP_PER_TRIPLET = flop_per_triplet(DIMS)


def flop_per_triplet_graph(spec, widths):
  """Same count over the op list of a fusion tower: forward + weight gradient for every fc, data gradient unless the fc
  reads an input slice.  ResNet (models.py:125-157): 3 * (4*1500*5000 + 6*5000*256 + 4*128*400 + 6*400*256 + 2*6*256*256)."""
  return 3 * sum((4 if spec[e["src"]]["op"] == "input" else 6) * widths[e["src"]] * e["out"] for e in spec if e["op"] == "fc")


def peaks():
  p = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}
  path = os.path.join(ROOT, "MEASURED_PEAKS.json")
  if os.path.exists(path):
    with open(path) as f:
      m = json.load(f)
    p.update({k: m[k] for k in ("hbm_gbs", "bf16_tflops", "bf16_tflops_sustained") if k in m})
    p["source"] = "measured"
  return p


DUMP_SAMPLE_ROWS = 4096             # queries of the KNN result / rows of the de-similarity output
DUMP_SAMPLE_WEIGHTS = 1 << 22       # elements of the flat weight buffer (VNet has 8.8M, the wide tower 13.1M)
# the most --dump-outputs writes: the weight sample (fp32), the KNN sample at k=100 (fp32 distances + float64 ids), the
# de-similarity sample at 81 neighbours (float64) and the 4 training stats -- about 24 MB, fixed by the sizes above
DUMP_MAX_BYTES = 4 * DUMP_SAMPLE_WEIGHTS + DUMP_SAMPLE_ROWS * (100 * (4 + 8) + 81 * 8) + 4 * 4
assert DUMP_MAX_BYTES <= 64 << 20


def sample_index(n, k, seed=0):
  """Ascending indices of a fixed, seeded sample of k of n rows (all n when n <= k): the same rows on every run."""
  if n <= k:
    return np.arange(n)
  return np.sort(np.random.RandomState(seed).choice(n, k, replace=False))


def sample_rows(t, k):
  import torch
  return t[torch.as_tensor(sample_index(t.shape[0], k), device=t.device)].cpu().numpy()


def dump_outputs(out_dir, arrays):
  """What the timed paths computed, one float32 / float64 .npy per array, so that two builds run with the same arguments
  (hence the same seeded inputs) can be compared output for output:
    train_stats    [4] stats the last timed training step returned (loss first)
    train_weights  seeded sample of the flat fp32 weight buffer right after that step
    knn_distances, knn_ids   seeded sample of query rows of the last timed KNN search (ids as float64, exact)
    desim_out      seeded sample of rows of the last timed de-similarity filter call (-1 = dropped; float64)
  The inputs are seeded, so they are the same on every run.  Two runs of one build wrote identical arrays (measured on a
  B200 at 1000 W).  Across builds the kernels may round differently: compare train_stats, train_weights and knn_distances
  with a tolerance, the ids and desim_out exactly up to ties."""
  os.makedirs(out_dir, exist_ok=True)
  for name, a in arrays.items():
    assert a.dtype in (np.float32, np.float64), (name, a.dtype)
    np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler(object):
  """nvidia-smi clocks + throttle reasons sampled every 200 ms while the timed region runs."""
  Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
       "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

  def __init__(self, index):
    self.index, self.proc, self.lines = index, None, []

  def start(self):
    try:
      self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                    "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE, text=True)
      self.thread = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
      self.thread.start()
    except Exception:
      self.proc = None

  def stop(self):
    if self.proc is None:
      return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    time.sleep(0.25)
    self.proc.terminate()
    self.thread.join(timeout=2)
    sm, mx, reasons = [], [], set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for ln in self.lines:
      parts = [p.strip() for p in ln.split(",")]
      if len(parts) < 6:
        continue
      try:
        sm.append(float(parts[0])), mx.append(float(parts[1]))
      except ValueError:
        continue
      for n, v in zip(names, parts[2:6]):
        if v.lower().startswith("active"):
          reasons.add(n)
    return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
            "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference path on the host cores
# --------------------------------------------------------------------------------------------------
def use_all_host_threads():
  """torchrun exports OMP_NUM_THREADS=1 to every rank, which pins numpy's BLAS to one thread for the whole process: the
  CPU legs would then run 3-4x slower at N>1 than at N=1 (round-1 SCALE records).  Lift the limit at run time."""
  n = os.cpu_count() or 1
  try:
    from threadpoolctl import threadpool_limits
    threadpool_limits(limits=n)
  except Exception:
    pass
  try:
    import torch
    torch.set_num_threads(n)
  except Exception:
    pass
  return n


def blas_threads():
  try:
    from threadpoolctl import threadpool_info
    return max([int(i.get("num_threads", 1)) for i in threadpool_info() if i.get("user_api") == "blas"] or [1])
  except Exception:
    return None


def cpu_train_baseline(budget_s=12.0, batch=1024, G=10000):
  from oracle import cdml_oracle as O
  use_all_host_threads()
  feats = O.synth_features(G, DIMS[0], 0)
  params = O.init_tower(DIMS, seed=2)
  tr = O.OracleTrainer(params, lr=1e-3, margin=0.8, dtype=np.float32)
  trip = O.synth_triplets(batch, G, 1)
  tr.step(O.flatten_triplets(O.gather_rows(feats, trip)))                 # warm-up (BLAS threads, page faults)
  n, t0 = 0, time.time()
  while time.time() - t0 < budget_s or n < 2:
    trip = O.synth_triplets(batch, G, 2 + n)
    tr.step(O.flatten_triplets(O.gather_rows(feats, trip)))               # numpy gather exactly as inputs.py:158
    n += 1
  dt = time.time() - t0
  return {"value": n * batch / dt, "unit": "triplets/s", "cores": blas_threads() or os.cpu_count(), "kind": "port",
          "host_cpus": os.cpu_count(), "batch": batch, "guids": G,
          "sample": "%d steps of batch %d (VNet 1500-5000-256, fp32 numpy/BLAS oracle, G=%d, random negatives) in %.1f s" % (n, batch, G, dt)}


def cpu_knn_baseline(budget_s=10.0, N=1000000, d=256, k=100, nq_block=1024):
  from oracle import cdml_oracle as O
  use_all_host_threads()
  X = O.knn_normalize(np.random.RandomState(4).standard_normal((N, d)).astype(np.float32))
  n, t0 = 0, time.time()
  while time.time() - t0 < budget_s or n < 1:
    O.flat_knn(X, X[n * nq_block:(n + 1) * nq_block], k=k, l2_norm=False, block=nq_block)
    n += 1
  dt = time.time() - t0
  return {"value": n * nq_block / dt, "unit": "queries/s", "cores": blas_threads() or os.cpu_count(), "kind": "port",
          "sample": "%d queries against N=%d d=%d k=%d (blocked sgemm + argpartition oracle) in %.1f s" % (n * nq_block, N, d, k, dt)}


def _desim_inputs(rng_or_gen, n, ke, kf, torch=None, dev=None):
  """KNN-shaped synthetic lists: row r starts with r, the rest are uniform ids (worst case for the filter: hardly any
  overlap, so every entry stays a pivot and gathers its feature-neighbour row); distances ascending in [0, 2)."""
  if torch is None:
    eI = rng_or_gen.randint(0, n, (n, ke)).astype(np.int64)
    fI = rng_or_gen.randint(0, n, (n, kf)).astype(np.int64)
    eI[:, 0] = fI[:, 0] = np.arange(n)
    fD = np.sort(rng_or_gen.rand(n, kf).astype(np.float32) * 2.0, axis=1)
    return eI, fI, fD
  eI = torch.randint(0, n, (n, ke), generator=rng_or_gen, device=dev, dtype=torch.int64)
  fI = torch.randint(0, n, (n, kf), generator=rng_or_gen, device=dev, dtype=torch.int64)
  eI[:, 0] = fI[:, 0] = torch.arange(n, device=dev)
  fD = torch.sort(torch.rand((n, kf), generator=rng_or_gen, device=dev) * 2.0, dim=1).values
  return eI, fI, fD


def cpu_desim_baseline(budget_s=8.0, n=20000, ke=81, kf=26):
  from oracle import cdml_oracle as O
  eI, fI, fD = _desim_inputs(np.random.RandomState(6), n, ke, kf)
  rows, t0 = 0, time.time()
  while time.time() - t0 < budget_s and rows < n:
    O.iter_desim(eI[rows:rows + 500], fI, fD, 1.4, 31)          # rows are independent: any slice is a valid sample
    rows += 500
  dt = time.time() - t0
  return {"value": rows / dt, "unit": "rows/s", "cores": 1, "kind": "port",
          "sample": "%d rows of %d neighbours against a %d x %d feature-KNN table (row-wise numpy restatement of "
                    "iter_desim_mp; the reference itself spawns 81 x Pool(22) numpy passes) in %.1f s" % (rows, ke, n, kf, dt)}


def bench_desim(torch, ops, dev, n, world, rank, barrier, dist, pk, ke=81, kf=26, reps=5, dump=None):
  gen = torch.Generator(device=dev)
  gen.manual_seed(6 + rank)
  eI, fI, fD = _desim_inputs(gen, n, ke, kf, torch, dev)
  out = torch.empty_like(eI)
  ops.desim(eI, fI, fD, 1.4, 31, out=out)                        # warm-up
  barrier()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(reps):
    ops.desim(eI, fI, fD, 1.4, 31, out=out)
  e1.record()
  barrier()
  if dump is not None:
    dump["desim_out"] = sample_rows(out, DUMP_SAMPLE_ROWS).astype(np.float64)
  t = torch.tensor([e0.elapsed_time(e1) / reps], device=dev, dtype=torch.float64)
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  ms = float(t.item())
  # end to end through faiss_knn.iter_desim_mp: host numpy lists -> H2D -> kernels -> D2H
  from cdml_b200 import faiss_knn
  survivors = int((out >= 0).sum().item())
  e2e = None
  if rank == 0:                       # rank 0 alone: 6.4 GB of pageable host arrays per rank are not worth repeating N times
    eh, fh, dh = eI.cpu().numpy(), fI.cpu().numpy(), fD.cpu().numpy()
    t0 = time.time()
    res = faiss_knn.iter_desim_mp(eh, fh, dh)
    e2e_s = time.time() - t0
    e2e = {"value": n / e2e_s, "unit": "rows/s (one GPU, host numpy lists in and out)", "h2d_bytes": n * (ke * 8 + kf * 12),
           "d2h_bytes": n * ke * 8, "rows_equal_device_run": bool((torch.as_tensor(res) == out.cpu()).all().item())}
    del eh, fh, dh, res
  barrier()
  fw_pad = 32
  # algorithmic bytes: prepare pass (read fI int64 + fD fp32, write the int32 table) + eI in/out + one table row per
  # alive pivot (= the survivors plus the row's own id)
  alg = n * kf * 12 + n * fw_pad * 4 + 2 * n * ke * 8 + (survivors + n) * fw_pad * 4
  # DRAM bytes per call from the committed ncu --set full capture of the same workload (4M rows), if present
  traffic, traffic_src = None, None
  prof = os.path.join(ROOT, "profiles", "r01_ncu_desim_summary.json")
  if os.path.exists(prof) and n == 4000000 and ke == 81 and kf == 26:
    try:
      ks = json.load(open(prof))["kernels"]
      traffic = sum((k["dram_read_GB"] + k["dram_write_GB"]) * 1e9 for k in ks)
      traffic_src = "profiles/r01_ncu_desim_summary.json: desim_prepare_kernel + desim_rows_kernel"
    except Exception:
      traffic = None
  return {"metric": "desim_rows_per_sec", "value": world * n / (ms / 1e3), "unit": "rows/s", "scaling": "weak",
          "config": {"workload": "iter_desim_mp (faiss_knn.py:187-244): %d rows x %d neighbours per GPU against a %d x %d "
                                 "feature-KNN table, fD_threshold 1.4, fI_end 31, uniform ids (every entry stays a pivot)"
                                 % (n, ke, n, kf)},
          "ms": ms, "dtype": "int64 ids / int32 table", "dropped_fraction": 1.0 - survivors / float(n * ke),
          "e2e": e2e,
          "roofline": {"bound": "hbm", "achieved": alg / (ms / 1e3) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                       "frac": alg / (ms / 1e3) / 1e9 / pk["hbm_gbs"], "traffic": traffic, "traffic_source": traffic_src,
                       "algorithmic_bytes": alg}}


def run_reference(args):
  """--impl reference: the reference's CPU implementation of the path on the host cores.  TensorFlow 1.13 / faiss cannot be
  installed offline, so this times the oracle port (numpy/BLAS, every host thread).  The line's `config` describes what
  this arm ACTUALLY ran -- a bounded sample of the workload: the same tower, batches of 2048 triplets (CPU throughput is
  flat in the batch size beyond that; one batch of 65536 is ~25 s of host BLAS), a 10 000-guid table, random negatives
  (the reference has no in-batch mining, SURVEY Q4) -- next to the GPU arm's workload it stands in for."""
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return
  threads = use_all_host_threads()
  steps = max(args.steps, 1)
  per_step = max(2.0, min(20.0, 90.0 / (steps + args.warmup)))
  batch = 2048 if args.batch >= 2048 else args.batch
  base = cpu_train_baseline(budget_s=per_step * steps, batch=batch)
  cfg = workload_config(args, mine=False)
  cfg.update({"workload": "bounded CPU sample of configs[1]: tower 1500-5000-256 (fp32), batch %d triplets, random negatives "
                          "(the reference has no in-batch mining), feature table %d guids in host memory"
                          % (batch, base["guids"]),
              "batch_per_gpu": batch, "guids": base["guids"], "mining": False, "cuda_graph": False,
              "parallelism": "host threads x%d" % threads, "l2_policy": "n/a (CPU)",
              "stands_in_for": workload_config(args, mine=not args.no_mine)["workload"]})
  line = {"impl": "reference", "metric": "train_triplets_per_sec", "value": base["value"], "unit": "triplets/s",
          "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": None, "higher_is_better": True,
          "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
          "config": cfg, "cpu_baseline": base,
          "e2e": {"value": base["value"], "unit": "triplets/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
          "note": "TensorFlow 1.13 / faiss are not installable offline; this arm times the oracle port of the reference "
                  "path (numpy/BLAS, all host threads; OMP_NUM_THREADS=1 from torchrun is lifted at run time) on the bounded "
                  "sample named in config.workload"}
  emit(line)


def workload_config(args, mine):
  dims, dt = TOWERS[getattr(args, "tower", "vnet")]
  dt = getattr(args, "dtype", "") or dt
  label = {"vnet": "configs[1]: tower", "wide": "configs[2]: tower",
           "resnet": "SURVEY 8f row 1: fusion tower ResNet (models.py:125-157; visual 1500-5000-256 x doc 128-400-256, two "
                     "residual 256-256 layers), feature width"}[getattr(args, "tower", "vnet")]
  world = max(int(os.environ.get("WORLD_SIZE", "1")), 1)
  b_local = args.batch // world if getattr(args, "scaling", "weak") == "strong" else args.batch
  return {"workload": "%s %s (%s operands), batch %d triplets/GPU, in-batch semi-hard mining %s, "
                      "feature table %d guids resident in HBM, %s features" % (label, "-".join(map(str, dims)), dt,
                                                                  b_local, "on" if mine else "off", args.guids,
                                                                  getattr(args, "features", "uniform")),
          "tower": dims, "batch_per_gpu": b_local, "guids": args.guids, "mining": bool(mine), "margin": 0.8,
          "features": getattr(args, "features", "uniform"),
          "optimizer": "adam(tf1) lr=1e-3", "parallelism": "dp%d" % args.gpus,
          "cuda_graph": bool(not getattr(args, "no_graph", False)),
          "l2_policy": "inputs_exceed_l2 (table+activations per step >> 126 MB)"}


# --------------------------------------------------------------------------------------------------
def emit(line):
  """The one JSON line goes to the REAL stdout; everything else this process prints (NCCL banners, library chatter)
  was redirected to stderr at start-up."""
  os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=20)
  ap.add_argument("--warmup", type=int, default=3)
  ap.add_argument("--impl", default="ours")
  ap.add_argument("--batch", type=int, default=65536)
  ap.add_argument("--guids", type=int, default=1000000)
  ap.add_argument("--no-mine", action="store_true")
  ap.add_argument("--no-knn", action="store_true")
  ap.add_argument("--no-cpu", action="store_true")
  ap.add_argument("--no-graph", action="store_true")
  ap.add_argument("--tower", default="vnet", choices=sorted(TOWERS),
                  help="vnet = configs[1] (default), wide = configs[2], resnet = the fusion tower of train.py main()")
  ap.add_argument("--no-desim", action="store_true")
  ap.add_argument("--desim-n", type=int, default=4000000)
  ap.add_argument("--knn-n", type=int, default=1000000)
  ap.add_argument("--knn-queries", type=int, default=65536)
  ap.add_argument("--dtype", default="", choices=["", "fp16", "bf16"], help="override the tower's operand type")
  ap.add_argument("--features", default="uniform", choices=["uniform", "clustered"],
                  help="uniform = imitation_data.gen_features (configs[1]); clustered = 1000 guid clusters, cowatch pairs from "
                       "the same cluster (a regime in which mining has something to find)")
  ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                  help="weak: --batch triplets per GPU; strong: --batch triplets per step split over the GPUs")
  ap.add_argument("--no-extras", action="store_true", help="skip the secondary measurements (regimes, configs[0], strong scaling)")
  ap.add_argument("--dump-outputs", metavar="DIR", default="",
                  help="write what the timed steps computed (last training step, KNN search, de-similarity filter) as "
                       "DIR/<name>.npy, about 24 MB in all")
  args = ap.parse_args()
  args.warmup = max(args.warmup, 3)
  if args.dump_outputs and args.impl == "reference":
    ap.error("--dump-outputs applies to --impl ours")
  if args.impl == "reference":
    return run_reference(args)

  import torch
  import torch.distributed as dist
  import __graft_entry__ as graft
  graft.build()
  from cdml_b200 import _lib, engine, ops

  world = int(os.environ.get("WORLD_SIZE", "1"))
  rank = int(os.environ.get("RANK", "0"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  torch.cuda.set_device(local)
  dev = torch.device("cuda:%d" % local)
  pg = None
  if world > 1:
    dist.init_process_group("nccl", device_id=dev)
    pg = dist.group.WORLD
  mine = not args.no_mine
  dims, dt16 = TOWERS[args.tower]
  dt16 = args.dtype or dt16
  flop_triplet = flop_per_triplet(dims)
  B, G, F = args.batch, args.guids, dims[0]
  if args.scaling == "strong":
    B = args.batch // world
  graph = None
  if args.tower == "resnet":
    from cdml_b200 import fusion, models
    graph = models.compile_graph(models.ResNet().create_model(models.placeholder(F))["l2_norm"])

  # ---- synthetic inputs (seeded; uniform [0,1) features like imitation_data.gen_features) generated on the device
  gen = torch.Generator(device=dev)
  gen.manual_seed(1234)
  if graph is not None:
    eng = fusion.GraphEngine(graph["spec"], feature_size=F, device=dev, base_lr=1e-3, margin=0.8, seed=2, process_group=pg)
    flop_triplet = flop_per_triplet_graph(eng.spec, eng.widths)
    table16 = tuple(torch.empty((G, engine._pad64(eng.widths[i] + 1)), dtype=eng.t16, device=dev) for i in eng.inputs)
  else:
    eng = engine.TowerEngine(dims, device=dev, base_lr=1e-3, margin=0.8, seed=2, process_group=pg,
                             dtype16=_lib.BF16 if dt16 == "bf16" else _lib.F16)
    table16 = torch.empty((G, eng.F_pad), dtype=eng.t16, device=dev)
  def fill_table(e, tables, features, g):
    """Seeded synthetic features, generated on the device slab by slab and folded into the resident 16-bit table (K2).
    uniform: imitation_data.gen_features' U[0,1) rows.  clustered: 1000 guid clusters, row = centre + 0.25 U[0,1)."""
    g.manual_seed(1234)
    cluster = None
    if features == "clustered":
      centres = torch.rand((1000, F), generator=g, device=dev)
      cluster = torch.randint(0, 1000, (G,), generator=g, device=dev)
    for s0 in range(0, G, 65536):
      rows = min(65536, G - s0)
      slab = torch.rand((rows, F), generator=g, device=dev, dtype=torch.float32)
      if cluster is not None:
        slab = centres[cluster[s0:s0 + rows]] + 0.25 * slab
      e.prepare_table(slab, out=[t[s0:s0 + rows] for t in tables] if isinstance(tables, tuple) else tables[s0:s0 + rows])
    return cluster

  def make_triplets(n, b, g, cluster):
    """[n,b,3] int64 index triplets: negative not in {a,p} (inputs.py:123-129); clustered: positive from the anchor's cluster."""
    idx = torch.randint(0, G, (n, b, 3), generator=g, device=dev, dtype=torch.int64)
    if cluster is None:
      idx[:, :, 1] = (idx[:, :, 0] + 1 + idx[:, :, 1] % (G - 1)) % G        # positive != anchor
    else:
      order = torch.argsort(cluster)
      start = torch.searchsorted(cluster[order], torch.arange(1001, device=dev))
      c = cluster[idx[:, :, 0]]
      span = (start[c + 1] - start[c]).clamp(min=1)
      k = idx[:, :, 1] % span
      p_ = order[start[c] + k]
      idx[:, :, 1] = torch.where(p_ == idx[:, :, 0], order[start[c] + (k + 1) % span], p_)     # positive != anchor
    idx[:, :, 2] = (idx[:, :, 1] + 1 + idx[:, :, 2] % (G - 2)) % G
    clash = (idx[:, :, 2] == idx[:, :, 0]) | (idx[:, :, 2] == idx[:, :, 1])
    idx[:, :, 2][clash] = (idx[:, :, 2][clash] + 1) % G
    clash = (idx[:, :, 2] == idx[:, :, 0]) | (idx[:, :, 2] == idx[:, :, 1])
    idx[:, :, 2][clash] = (idx[:, :, 2][clash] + 1) % G                      # negative not in {a,p}
    return idx

  cluster = fill_table(eng, table16, args.features, gen)
  gen.manual_seed(100 + rank)
  nbatch = args.steps + args.warmup
  idx_all = make_triplets(nbatch, B, gen, cluster)
  idx_host = idx_all.cpu().pin_memory()

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  # The whole step is one CUDA-graph launch (the product's fast path); with N>1 the NCCL all-reduce is captured inside.
  replay = eng.capture_step(table16, B, mine=mine) if not args.no_graph else None

  def step(i, idx_any):
    if replay is not None:
      return replay(idx_any)
    return eng.train_step_indices(table16, idx_any, mine=mine)

  # ---- value: device-resident indices, CUDA events, max over ranks
  for i in range(args.warmup):
    step(i, idx_all[i])
  barrier()
  sampler = ClockSampler(local)
  if rank == 0:
    sampler.start()
  launches0 = ops.launch_count()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for i in range(args.steps):
    stats = step(i, idx_all[args.warmup + i])
  e1.record()
  barrier()
  ms = e0.elapsed_time(e1)
  launches = ops.launch_count() - launches0
  clocks = sampler.stop() if rank == 0 else None
  loss_last = float(stats[0].item())
  dump = {} if args.dump_outputs else None
  if dump is not None:                # before the e2e steps below train on
    dump["train_stats"] = stats.cpu().numpy().astype(np.float32)
    dump["train_weights"] = sample_rows(eng.w, DUMP_SAMPLE_WEIGHTS)
  t = torch.tensor([ms], device=dev, dtype=torch.float64)
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  ms = float(t.item())
  value = world * B * args.steps / (ms / 1e3)

  # ---- e2e: pinned host indices -> H2D -> step -> D2H loss, every step
  barrier()
  stats_host = torch.empty(4, dtype=torch.float32).pin_memory()
  idx_dev = torch.empty((B, 3), dtype=torch.int64, device=dev)
  e0.record()
  for i in range(args.steps):
    if replay is not None:
      st = step(i, idx_host[args.warmup + i])                             # pinned host -> static device buffer -> graph
    else:
      idx_dev.copy_(idx_host[args.warmup + i], non_blocking=True)
      st = step(i, idx_dev)
    stats_host.copy_(st, non_blocking=True)
    torch.cuda.current_stream().synchronize()                             # the host reads the loss every step
  e1.record()
  barrier()
  t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  e2e_value = world * B * args.steps / (float(t.item()) / 1e3)

  # ---- per-kernel timing of one step (CUDA events around every tensor-core GEMM launch) for the roofline entry
  timings = {}
  orig = ops.gemm16

  def timed_gemm16(A, Bm, M, N, K, amn, bmn, epi, out, **kw):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    r = orig(A, Bm, M, N, K, amn, bmn, epi, out, **kw)
    b.record()
    timings.setdefault((M, N, K, amn, bmn, epi), []).append((a, b))
    return r

  mine_orig = ops.mine_semihard
  mine_ev = []

  def timed_mine(*a, **kw):
    x, y = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    x.record()
    r = mine_orig(*a, **kw)
    y.record()
    mine_ev.append((x, y))
    return r

  ops.gemm16 = timed_gemm16
  engine.ops.gemm16 = timed_gemm16
  ops.mine_semihard = timed_mine
  reps = min(5, args.steps)
  for i in range(reps):
    eng.train_step_indices(table16, idx_all[i], mine=mine)                # eager: events around every launch
  torch.cuda.synchronize()
  ops.gemm16 = orig
  engine.ops.gemm16 = orig
  ops.mine_semihard = mine_orig
  kern = []
  if mine_ev:
    avg = float(np.mean([a.elapsed_time(b) for a, b in mine_ev]))
    kern.append({"gemm": "mining scan M=%d N=%d K=256 Ak Bk, selection epilogue (per launch; 2 launches/step, time incl. prepare/finalize)" % (B, B),
                 "key": (0, 0, 99), "ms": avg / 2, "tflops": 2.0 * B * B * 256 / (avg / 2) / 1e9, "bytes": 2 * (2 * B * 256)})
  for (M, N, K, amn, bmn, epi), evs in timings.items():
    avg = float(np.mean([a.elapsed_time(b) for a, b in evs]))
    out_bytes = M * N * (4 if epi in (0, 2) else 2) * (2 if epi == 3 else 1)      # MASK_LEAKY also reads the 16-bit mask
    if epi == 4:
      out_bytes += M * N // 8                                                       # MASK_BITS reads 1 bit per element
    kern.append({"gemm": "M=%d N=%d K=%d A%s B%s epi=%d" % (M, N, K, "mn" if amn else "k", "mn" if bmn else "k", epi),
                 "key": (int(amn), int(bmn), int(epi)), "ms": avg, "tflops": 2.0 * M * N * K / avg / 1e9,
                 "bytes": 2 * (M * K + N * K) + out_bytes})
  kern.sort(key=lambda r: -r["ms"])
  pk = peaks()
  top = kern[0]
  # DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture (profiles/).  The summary
  # carries the digest of the kernel sources it was captured from; a capture of OTHER kernel code is refused (null +
  # the reason) instead of being quoted as if it described this build.
  traffic, traffic_src = None, None
  prof = os.path.join(ROOT, "profiles", "r02_ncu_step_gemms_summary.json")
  if os.path.exists(prof) and args.batch == 65536:
    pj = json.load(open(prof))
    here = graft.source_digest()
    if pj.get("csrc_digest") != here:
      traffic_src = "stale: profiles/r02_ncu_step_gemms_summary.json was captured from csrc digest %s, this build is %s" % (
          str(pj.get("csrc_digest"))[:12], here[:12])
    else:
      want = {(0, 1, 1): "EpiStore16", (0, 1, 2): "EpiL2Norm", (1, 1, 0): "EpiStoreF32", (0, 0, 3): "EpiMaskLeaky",
              (0, 0, 4): "EpiMaskBits", (0, 0, 99): "EpiMine"}.get(top["key"])
      cands = [k for k in pj["kernels"] if want and want in k["kernel"]]
      if cands:
        best = max(cands, key=lambda k: k["duration_ms"])
        traffic = (best["dram_read_GB"] + best["dram_write_GB"]) * 1e9
        traffic_src = "profiles/r02_ncu_step_gemms_summary.json: " + best["kernel"]
  kern_all = kern
  roofline = {"bound": "tensor", "kernel": "cdml gemm tcgen05 " + top["gemm"], "achieved": top["tflops"],
              "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s", "frac": top["tflops"] / pk["bf16_tflops_sustained"],
              "traffic": traffic, "traffic_source": traffic_src,
              "algorithmic_bytes": top["bytes"],
              "peak_source": "%s bf16_tflops_sustained (kernel timed inside the step)" % pk["source"],
              "step_tensor_frac": (flop_triplet * value / world / 1e12) / pk["bf16_tflops_sustained"],
              "gemms": [{k: v for k, v in g.items() if k != "key"} for g in kern]}

  line = {"metric": "train_triplets_per_sec", "value": value, "unit": "triplets/s", "n_gpus": world, "steps": args.steps,
          "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
          "vs_baseline": None, "dtype": "%s operands / fp32 accumulate (tcgen05 kind::f16), fp32 master weights" % dt16,
          "data": "synthetic", "config": workload_config(args, mine),
          "e2e": {"value": e2e_value, "unit": "triplets/s", "h2d_bytes_per_step": B * 3 * 8, "d2h_bytes_per_step": 16,
                  "note": "host INDEX triplets in, loss out; the feature table stays resident in HBM (SURVEY 8b). The drop-in "
                          "get_batch() float path (host features in) is timed separately: key get_batch_e2e"},
          "gpu_launches": int(launches), "clocks": clocks, "loss_last_step": loss_last,
          "tflops_per_gpu": flop_triplet * value / world / 1e12,
          "knn_summary": None,       # second BASELINE metric: filled below, kept EARLY in the line (record tails are truncated)
          "roofline_summary": {"kernel": roofline["kernel"], "frac": roofline["frac"], "achieved": roofline["achieved"],
                               "peak": roofline["peak"], "unit": roofline["unit"], "step_tensor_frac": roofline["step_tensor_frac"]}}

  # ---- N>1: what the ranks computed, not only how fast (weights bit-identical after the timed steps)
  if world > 1:
    w0 = eng.w.clone()
    dist.broadcast(w0, src=0)
    differ = torch.tensor([float((w0 != eng.w).any().item())], device=dev)
    dist.all_reduce(differ, op=dist.ReduceOp.MAX)
    line["weights_identical_across_ranks"] = bool(differ.item() == 0.0)

  extras = not args.no_extras and args.tower == "vnet"
  # ---- N>1, weak run: the strong-scaling figure beside it (SURVEY 8d C2 "report both"): the same global batch of
  #      --batch triplets per step split over the ranks
  if extras and world > 1 and args.scaling == "weak" and B % world == 0 and replay is not None:
    Bs = B // world
    replay_s = eng.capture_step(table16, Bs, mine=mine)
    for i in range(args.warmup):
      replay_s(idx_all[i, :Bs])
    barrier()
    e0.record()
    for i in range(args.steps):
      replay_s(idx_all[args.warmup + i, :Bs])
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    line["strong_scaling"] = {"value": world * Bs * args.steps / (float(t.item()) / 1e3), "unit": "triplets/s",
                              "ms_per_step": float(t.item()) / args.steps, "global_batch": B, "batch_per_gpu": Bs,
                              "scaling": "strong"}
    del replay_s

  # ---- N=1 secondary measurements
  if extras and world == 1 and replay is not None:
    # (1) the drop-in get_batch() path (inputs.py:144-166 -> train.py:313-318): HOST fp32 feature rows in, every step
    #     (pinned staging, H2D of B*3*F floats, normalise+cast on the device, then the same step)
    xb = min(B, 16384)
    xh = torch.empty((3 * xb, F), dtype=torch.float32).pin_memory()
    xh.uniform_(0, 1)
    xd = torch.empty((3 * xb, F), dtype=torch.float32, device=dev)
    st_h = torch.empty(4, dtype=torch.float32).pin_memory()
    def float_step():
      xd.copy_(xh, non_blocking=True)
      x16 = eng.prepare_table(xd)
      st = eng.train_step_rows(x16, xb, mine=False, input_ones=True)
      st_h.copy_(st, non_blocking=True)
      torch.cuda.current_stream().synchronize()
    for _ in range(2):
      float_step()
    e0.record()
    for _ in range(5):
      float_step()
    e1.record()
    torch.cuda.synchronize()
    line["get_batch_e2e"] = {"value": xb * 5 / (e0.elapsed_time(e1) / 1e3), "unit": "triplets/s", "batch": xb, "mining": False,
                             "h2d_bytes_per_step": 3 * xb * F * 4, "d2h_bytes_per_step": 16,
                             "note": "host float features in (the reference's feed_dict path): PCIe-bound"}
    # (2) configs[0]: batch 1024, 10 000 guids, no mining (the case the CPU baseline runs) as one CUDA graph per step
    e_small = engine.TowerEngine(dims, device=dev, base_lr=1e-3, margin=0.8, seed=2, dtype16=_lib.BF16 if dt16 == "bf16" else _lib.F16)
    G0 = 10000
    replay0 = e_small.capture_step(table16[:G0], 1024, mine=False)
    idx0 = torch.randint(0, G0, (64, 1024, 3), generator=gen, device=dev, dtype=torch.int64)
    for i in range(8):
      replay0(idx0[i])
    e0.record()
    for i in range(200):
      replay0(idx0[i % 64])
    e1.record()
    torch.cuda.synchronize()
    line["config0_batch1024"] = {"value": 1024 * 200 / (e0.elapsed_time(e1) / 1e3), "unit": "triplets/s",
                                 "ms_per_step": e0.elapsed_time(e1) / 200, "config": {"workload": "configs[0]: tower %s, batch 1024, "
                                 "%d guids, random negatives, one CUDA graph per step" % ("-".join(map(str, dims)), G0)}}
    del replay0, e_small, idx0
    # (3) mining on trial in a regime with structure: clustered features, cowatch pairs from the same cluster, lr 1e-4,
    #     fresh weights; the loss trajectory with mining ON, the scan time and the re-scan rate next to the uniform case
    if mine and args.features == "uniform":
      uniform_stats = ops.mine_stats(eng.w)
      cl = fill_table(eng, table16, "clustered", gen)
      e_cl = engine.TowerEngine(dims, device=dev, base_lr=1e-4, margin=0.8, seed=2, dtype16=_lib.BF16 if dt16 == "bf16" else _lib.F16)
      replay_c = e_cl.capture_step(table16, B, mine=True)
      gen.manual_seed(77)
      n_c = 24
      idx_c = make_triplets(n_c, B, gen, cl)
      traj = []
      for i in range(3):
        replay_c(idx_c[i])                   # these steps train too: the trajectory below starts at step 3
      torch.cuda.synchronize()
      e0.record()
      for i in range(3, n_c):
        st = replay_c(idx_c[i])
        traj.append(st.clone())
      e1.record()
      torch.cuda.synchronize()
      ms_c = e0.elapsed_time(e1) / (n_c - 3)
      traj = [[round(float(v), 5) for v in t_.tolist()[:3]] for t_ in traj]
      # scan time alone, on the embeddings of the last batch
      buf = e_cl._buffers(3 * B, True)
      e16 = e_cl._ws[("e16", 3 * B)]
      ops.mine_semihard(e16, buf["e"], idx_c[-1], B, 0.8, want_dist=False)
      e0.record()
      for _ in range(3):
        neg_c, _ = ops.mine_semihard(e16, buf["e"], idx_c[-1], B, 0.8, want_dist=False)
      e1.record()
      torch.cuda.synchronize()
      cst = ops.mine_stats(eng.w)
      line["mining_regimes"] = {
          "uniform": {"mining_ms_per_step": [g["ms"] * 2 for g in kern if g["key"] == (0, 0, 99)][0], "loss_last_step": loss_last,
                      "rescans_per_anchor_per_step": uniform_stats["rescans"] / float(B), "mined_fraction": uniform_stats["mined"] / float(B)},
          "clustered": {"mining_ms_per_step": e0.elapsed_time(e1) / 3, "ms_per_step": ms_c, "triplets_per_s": B / (ms_c / 1e3),
                        "rescans_per_anchor_per_step": cst["rescans"] / float(B), "mined_fraction": cst["mined"] / float(B),
                        "loss_pos_neg_trajectory_mining_on": traj[::3] + [traj[-1]], "lr": 1e-4,
                        "workload": "1000 guid clusters (centre + 0.25 U[0,1)), positives from the anchor's cluster, batch %d, "
                                    "fresh Xavier weights, %d steps" % (B, n_c)}}
      del replay_c, e_cl, idx_c
  # ---- second BASELINE metric: exact KNN top-100 queries/sec on a 1M-item index.  N>1: the index is row-sharded over
  # the ranks (strong scaling: same 1M rows, same queries).  The training engine -- and with it the captured CUDA graph,
  # which holds NCCL kernels when N>1 -- is released before anything else runs and long before the process group is torn
  # down (a live NCCL graph at teardown was seen to hang the exit of a 2-GPU run after the line had been printed)
  del table16, idx_all, eng, replay
  import gc
  gc.collect()
  torch.cuda.synchronize()
  torch.cuda.empty_cache()
  if not args.no_knn:
    from cdml_b200 import faiss_knn
    N, nq, k, d = args.knn_n, args.knn_queries, 100, 256
    gen.manual_seed(4)
    X = torch.nn.functional.normalize(torch.randn((N, d), generator=gen, device=dev), dim=1)   # same on every rank
    lo, hi = rank * N // world, (rank + 1) * N // world
    Q = X[:nq].clone()
    index = ops.FlatIndex(X[lo:hi].contiguous(), "L2")
    if world > 1:
      del X
    faiss_knn.sharded_search(index, Q, k, lo, "L2", pg)                   # warm-up at full size (workspace, L2, NCCL)

    def timed_search(reps, **kw):
      """`reps` searches, each timed on the device and taken as the MAX over ranks; the MEDIAN is reported (a search is a
      few milliseconds and, at N>1, a chain of rendezvous between N Python processes: single shots scatter by 30 %)."""
      out, times = None, []
      for _ in range(reps):
        barrier()
        e0.record()
        out = faiss_knn.sharded_search(index, Q, k, lo, "L2", pg, **kw)
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
          dist.all_reduce(t, op=dist.ReduceOp.MAX)
        times.append(float(t.item()))
      return out, float(np.median(times)), times

    (D, I), kms, kms_all = timed_search(5)
    if dump is not None:
      dump["knn_distances"] = sample_rows(D, DUMP_SAMPLE_ROWS)
      dump["knn_ids"] = sample_rows(I, DUMP_SAMPLE_ROWS).astype(np.float64)
    kms_slice, kms_slice_all = None, None
    if world > 1:       # the same search leaving every rank with ITS slice of the queries (no final all-gather)
      _, kms_slice, kms_slice_all = timed_search(5, gather=False)
    self_first = float((I[:, 0] == torch.arange(nq, device=dev)).float().mean().item())
    Xh = Q.cpu().pin_memory()
    Dh, Ih = torch.empty((nq, k)).pin_memory(), torch.empty((nq, k), dtype=torch.int64).pin_memory()
    barrier()
    t0 = time.time()
    D2, I2 = faiss_knn.sharded_search(index, Xh.to(dev, non_blocking=True), k, lo, "L2", pg)
    Dh.copy_(D2, non_blocking=True), Ih.copy_(I2, non_blocking=True)
    barrier()
    t = torch.tensor([time.time() - t0], device=dev, dtype=torch.float64)
    if world > 1:
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ke2e = nq / float(t.item())
    st = index.last_stats()
    # what the shards computed, not only how fast: 256 sampled queries against an exact fp32 search of ALL rows
    # (every rank scores its own rows with a plain fp32 matmul -- the checker, not the product -- top-k per rank, gathered
    # and merged; ids must equal the sharded product's except inside fp32-noise ties)
    sq = torch.arange(0, nq, max(nq // 256, 1), device=dev)[:256]
    dq = (Q[sq] ** 2).sum(1, keepdim=True) + (index._ref ** 2).sum(1)[None, :] - 2.0 * Q[sq] @ index._ref.T
    dloc, iloc = torch.topk(dq, min(k, hi - lo), dim=1, largest=False)
    iloc = iloc + lo
    if world > 1:
      dl = [torch.empty_like(dloc) for _ in range(world)]
      il = [torch.empty_like(iloc) for _ in range(world)]
      dist.all_gather(dl, dloc.contiguous()), dist.all_gather(il, iloc.contiguous())
      dloc, iloc = torch.cat(dl, 1), torch.cat(il, 1)
    order = torch.argsort(dloc, dim=1, stable=True)[:, :k]
    want_ids = torch.gather(iloc, 1, order)
    got_ids = I[sq]
    row_equal = (want_ids == got_ids).all(dim=1)
    set_equal = torch.tensor([set(a.tolist()) == set(b.tolist()) for a, b in zip(want_ids.cpu(), got_ids.cpu())])
    knn_ids_ok = bool(set_equal.float().mean().item() >= 0.99)
    line["knn_summary"] = {"queries_per_s": nq / (kms / 1e3), "ms": kms, "n_gpus": world, "N": N, "nq": nq, "k": k,
                           "ms_all_runs": [round(x, 3) for x in kms_all], "timing": "median of 5 searches, each the max over ranks",
                           "ms_result_left_sharded_by_query": kms_slice,
                           "ms_result_left_sharded_all_runs": [round(x, 3) for x in kms_slice_all] if kms_slice_all else None,
                           "tflops_per_gpu": 2.0 * nq * N * d / kms / 1e9 / world,
                           "frac_of_sustained_peak_per_gpu": 2.0 * nq * N * d / kms / 1e9 / world / pk["bf16_tflops_sustained"],
                           "sharded_knn_ids_equal_unsharded_sample": knn_ids_ok,
                           "sample_rows_identical": float(row_equal.float().mean().item()),
                           "sample_sets_identical": float(set_equal.float().mean().item())}
    del dq
    line["knn"] = {"metric": "knn_top100_queries_per_sec", "value": nq / (kms / 1e3), "unit": "queries/s",
                   "scaling": "strong",
                   "config": {"workload": "configs[3]: exact flat L2 top-100, N=%d d=%d row-sharded over %d GPU(s), %d queries "
                                          "(rows of the index)" % (N, d, world, nq)},
                   "ms": kms, "tflops": 2.0 * nq * N * d / kms / 1e9, "e2e": {"value": ke2e, "unit": "queries/s",
                   "h2d_bytes": nq * d * 4, "d2h_bytes": nq * k * 12},
                   # (N>1: the shard protocol defers its overflow check and keeps no host-side counters)
                   "candidates_per_query_rank0": st["candidates"] / nq if world == 1 else None,
                   "fallback_queries_rank0": st["fallback_queries"] if world == 1 else None,
                   "self_is_first_neighbour": self_first,
                   "roofline": {"bound": "tensor", "achieved": 2.0 * nq * N * d / kms / 1e9 / world,
                                "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s (per GPU)",
                                "frac": 2.0 * nq * N * d / kms / 1e9 / world / pk["bf16_tflops_sustained"]}}
    index.close()
  # ---- SURVEY 8f row 2: de-similarity filter of the KNN lists (integer work, HBM-bound; rows are independent -> each
  # rank filters its own slice of the rows, no collective: weak scaling)
  if not args.no_desim:
    line["desim"] = bench_desim(torch, ops, dev, args.desim_n, world, rank, barrier, dist, pk, dump=dump)
  line["roofline"] = roofline          # last: its per-GEMM list is the long tail of the line
  if world > 1:                       # a teardown that does not finish within a minute must not hold the job
    t = threading.Timer(60.0, os._exit, (0,))
    t.daemon = True
    t.start()
  if rank != 0:
    if world > 1:
      dist.barrier()
      dist.destroy_process_group()
    return
  if dump is not None:                # rank 0: the weights are identical on every rank
    dump_outputs(args.dump_outputs, dump)
  if not args.no_cpu and world == 1:
    if not args.no_desim:
      line["desim"]["cpu_baseline"] = cpu_desim_baseline()
    line["cpu_baseline"] = cpu_train_baseline()
    if not args.no_knn:
      line["knn"]["cpu_baseline"] = cpu_knn_baseline(N=min(args.knn_n, 1000000))
  emit(line)
  if world > 1:
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
  main()
