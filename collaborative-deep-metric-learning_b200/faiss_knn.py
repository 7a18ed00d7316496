"""KNN retrieval + result files -- host-side mirror of the reference's faiss_knn.py: `calc_knn` (faiss_knn.py:82-131),
`write_process` / `write_knn` (:267-305), loaders (:52-66) and `main` (:359-402), same names / arguments / flags /
file formats.  `faiss.Index*.add/search` is replaced by libcdml's exact flat index (tensor-core candidate pass +
fp32 re-rank); with WORLD_SIZE>1 the index is row-sharded over the ranks and the per-shard top-k are all-gathered
and merged on the GPU.  The de-similarity post-filter (`desim`, `fliter_fI`, `iter_desim_mp`, faiss_knn.py:134-244) runs as
libcdml's cdml_desim kernels; `strict_knn` / `cross_knn` (faiss_knn.py:308-351) compose them with calc_knn."""
import json
from multiprocessing.pool import ThreadPool
import os
import shutil
import time
import traceback

import numpy as np
import torch
from absl import app, flags

from . import ops

FLAGS = flags.FLAGS
if "embedding_file" not in FLAGS:
  flags.DEFINE_string("embedding_file", "serving_dir/predict_result/output.npy", "embeddings to index / query")
  flags.DEFINE_string("decode_map_file", "serving_dir/predict_result/decode_map.json", "row index -> guid")
  flags.DEFINE_string("pred_feature_file", "serving_dir/predict_result/features.npy", "raw feature vectors")
  flags.DEFINE_string("pred_feature_info", "serving_dir/dataset/feature.info", "feature info file")
  flags.DEFINE_integer("nearest_num", 81, "neighbours per embedding (incl. the query itself)")
  flags.DEFINE_integer("desim_nearest_num", 26, "neighbours per raw feature vector (de-similarity)")
  flags.DEFINE_string("knn_result", "serving_dir/knn_result/newresult", "where knn results are written")
  flags.DEFINE_string("knn_mode", "knn", "knn: calc_knn + knn_split* files (what cdml_run.sh:147 uploads) | strict: "
                      "+ de-similarity against the raw-feature KNN (strict_knn, faiss_knn.py:308-322) | cross: video<->doc "
                      "cross search + de-similarity (cross_knn, faiss_knn.py:325-351; the reference's main at HEAD)")
  flags.DEFINE_integer("doc_location", 343455, "first doc row of the embeddings (hard-coded in the reference, faiss_knn.py:389)")

DECODE_MAP = {}


def load_decode_map(filename):
  """json {"0": guid, ...} -> ({int: guid}, {guid: int}) (faiss_knn.py:52-61)."""
  with open(filename, "r") as f:
    index2guid_str = json.load(f)
  decode_map = {int(k): v for k, v in index2guid_str.items()}
  encode_map = {v: int(k) for k, v in index2guid_str.items()}
  return decode_map, encode_map


def load_embedding(filename):
  return np.load(filename)


def _device():
  if not torch.cuda.is_available():
    raise RuntimeError("calc_knn runs on the CUDA device only (libcdml has no CPU path)")
  return torch.device("cuda:%d" % torch.cuda.current_device())


def sharded_search(index, xq, k, id_offset=0, metric="L2", process_group=None, merge_fn=None, gather=True,
                   merge_packed_fn=None, _sync_refine=False):
  """Top-k of the (replicated) queries `xq` over a row-sharded index; device tensors in and out.

  Per chunk of <= 65536 queries, one collective per phase (each an all-reduce MAX of a [2,n] fp32 pair):
    1. bound pass on every shard -> all-reduce: max over shards of their k-th best sampled score / min of their
       ceil(k/W)-th best -- one collection bound per query, so that together the shards nominate about as many candidates
       as one unsharded index would instead of W times as many;
    2. collect on every shard, k-th / ceil(k/W)-th best APPROXIMATE score among its nominees -> all-reduce: a lower bound of
       the global k-th best approximate score;
    3. exact fp32 re-rank of the nominees within 2 eps of that global bound only (~k rows per query over all shards, not W*k)
       -> sorted local list as 64-bit records (distance key | global id).
  Then ONE all-to-all: rank r receives every shard's lists for ITS slice of the queries and merges them on the GPU
  (cdml_knn_merge_packed, ties -> lower id).  gather=True completes the result on every rank with one all-gather;
  gather=False returns (D, I) of this rank's query slice [r*nq/W, (r+1)*nq/W) only -- what a caller that writes its own
  knn_split files needs.
  The whole protocol is enqueued without a host round trip: a query whose candidate list overflows (dense near-tie bands)
  only sets a device flag, the ranks agree on it with one 4-byte all-reduce after the exchange, and in that rare case the
  search is repeated with the synchronous refine that redoes such queries exactly."""
  world = torch.distributed.get_world_size(process_group) if process_group is not None else 1
  if world == 1:
    return index.search(xq, k, id_offset=id_offset)
  if not hasattr(index, "shard_bounds"):
    return _sharded_search_lists(index, xq, k, id_offset, metric, process_group, merge_fn)
  deferred = merge_packed_fn is None and not _sync_refine       # (the CPU stand-in of the gloo test has no deferred mode)
  out, flag = _run_sharded(index, xq, k, id_offset, metric, process_group, gather, deferred, merge_packed_fn)
  if flag is not None and int(flag.item()) != 0:             # some shard overflowed somewhere: redo with the exact fallback (rare)
    return sharded_search(index, xq, k, id_offset, metric, process_group, merge_fn, gather, merge_packed_fn, _sync_refine=True)
  return out


def _run_sharded(index, xq, k, id_offset, metric, process_group, gather, deferred, merge_packed_fn=None):
  """One pass of the record protocol, enqueued on the current stream without a host round trip when `deferred`.  Returns
  ((D, I), flag): flag is the device word agreed over the ranks (None in the synchronous form)."""
  dist = torch.distributed
  world = dist.get_world_size(process_group)
  nq = xq.shape[0]
  k_part = -(-k // world)
  pad = (-nq) % world                      # the all-to-all needs equal slices: pad with copies of the last query
  if pad:
    xq = torch.cat([xq, xq[-1:].expand(pad, -1)], 0)
  nqp = nq + pad
  rec = torch.empty((nqp, k), dtype=torch.int64, device=xq.device)
  flag = torch.zeros((1,), dtype=torch.int32, device=xq.device) if deferred else None
  for s in range(0, nqp, index.CHUNK):
    q = xq[s:s + index.CHUNK]
    pair = index.shard_bounds(q, k, k_part)
    dist.all_reduce(pair, op=dist.ReduceOp.MAX, group=process_group)
    nom = index.shard_collect(q, k, k_part, pair)
    dist.all_reduce(nom, op=dist.ReduceOp.MAX, group=process_group)
    if deferred:
      index.shard_refine(q, k, nom, rec[s:s + index.CHUNK], id_offset=id_offset, overflow_flag=flag)
    else:
      index.shard_refine(q, k, nom, rec[s:s + index.CHUNK], id_offset=id_offset)
  got = torch.empty_like(rec)                # [W, nqp/W, k]: every shard's lists for my query slice
  dist.all_to_all_single(got, rec, group=process_group)
  got = got.view(world, nqp // world, k)
  if merge_packed_fn is not None:           # CPU stand-in of the gloo test (no records output: gather the two arrays)
    Dm, Im = merge_packed_fn(got, metric)
    if not gather:
      rank = dist.get_rank(process_group)
      lo, hi = rank * (nqp // world), min((rank + 1) * (nqp // world), nq)
      return (Dm[:max(hi - lo, 0)], Im[:max(hi - lo, 0)]), None
    D = torch.empty((nqp, k), dtype=Dm.dtype, device=Dm.device)
    I = torch.empty((nqp, k), dtype=Im.dtype, device=Im.device)
    dist.all_gather_into_tensor(D, Dm, group=process_group)
    dist.all_gather_into_tensor(I, Im, group=process_group)
    return (D[:nq], I[:nq]), None
  out = _finish_sharded(got, nq, nqp, k, world, metric, process_group, gather, xq.device)
  if flag is not None:
    dist.all_reduce(flag, op=dist.ReduceOp.MAX, group=process_group)
  return out, flag


def _finish_sharded(got, nq, nqp, k, world, metric, process_group, gather, device):
  """Merge of the received record lists (+ all-gather and unpack when every rank wants the whole result)."""
  dist = torch.distributed
  if not gather:
    Dm, Im = ops.knn_merge_packed(got, metric)
    rank = dist.get_rank(process_group)
    lo, hi = rank * (nqp // world), min((rank + 1) * (nqp // world), nq)
    return Dm[:max(hi - lo, 0)], Im[:max(hi - lo, 0)]
  mine = ops.knn_merge_packed(got, metric, as_records=True)         # merged slice stays packed: ONE all-gather of 8 B / entry
  allr = torch.empty((nqp, k), dtype=torch.int64, device=device)
  dist.all_gather_into_tensor(allr, mine, group=process_group)
  D, I = ops.knn_unpack_records(allr, metric)
  return D[:nq], I[:nq]


def _sharded_search_lists(index, xq, k, id_offset=0, metric="L2", process_group=None, merge_fn=None):
  """The same search with (D, I) lists instead of packed records and local pruning only (an index object that offers
  bounds / search_bounded but not the shard_* calls: the CPU stand-in of the gloo protocol test)."""
  world = torch.distributed.get_world_size(process_group)
  merge_fn = merge_fn or ops.knn_merge
  bf, bp = index.bounds(xq, k, -(-k // world))
  torch.distributed.all_reduce(bf, op=torch.distributed.ReduceOp.MAX, group=process_group)
  torch.distributed.all_reduce(bp, op=torch.distributed.ReduceOp.MIN, group=process_group)
  D, I = index.search_bounded(xq, k, bf, bp, id_offset=id_offset)
  nq = xq.shape[0]
  if nq % world == 0 and nq >= world:
    Dg, Ig = torch.empty_like(D), torch.empty_like(I)           # [W, nq/W, k]: every shard's lists for my query slice
    torch.distributed.all_to_all_single(Dg, D, group=process_group)
    torch.distributed.all_to_all_single(Ig, I, group=process_group)
    Dm, Im = merge_fn(Dg.view(world, nq // world, k), Ig.view(world, nq // world, k), metric)
    D, I = torch.empty_like(D), torch.empty_like(I)
    torch.distributed.all_gather_into_tensor(D, Dm, group=process_group)
    torch.distributed.all_gather_into_tensor(I, Im, group=process_group)
    return D, I
  Dg = torch.empty((world * nq, k), dtype=D.dtype, device=D.device)
  Ig = torch.empty((world * nq, k), dtype=I.dtype, device=I.device)
  torch.distributed.all_gather_into_tensor(Dg, D, group=process_group)
  torch.distributed.all_gather_into_tensor(Ig, I, group=process_group)
  return merge_fn(Dg.view(world, nq, k), Ig.view(world, nq, k), metric)


def calc_knn(embeddings, q_embeddings=None, nearest_num=51, l2_norm=True, M=80, efConstruction=64, efSearch=32,
             metric="L2", process_group=None):
  """Exact KNN of q_embeddings (default: the embeddings themselves) in embeddings.
  Returns D [nq,k] float32 squared-L2 ascending, I [nq,k] int64.  The HNSW arguments of the reference signature are
  accepted and ignored: the flat index is exact (docstring faiss_knn.py:86-89).  As in the reference, rows are
  L2-normalised first when l2_norm (queries in place, faiss_knn.py:99-104)."""
  begin = time.time()
  dev = _device()
  embeddings = embeddings.astype(np.float32)
  if l2_norm:
    embeddings /= np.linalg.norm(embeddings, axis=1, keepdims=True)
    if q_embeddings is not None:
      q_embeddings /= np.linalg.norm(q_embeddings, axis=1, keepdims=True)
    else:
      q_embeddings = embeddings
  elif q_embeddings is None:
    q_embeddings = embeddings
  xq = torch.as_tensor(np.ascontiguousarray(q_embeddings, np.float32)).to(dev)
  world = torch.distributed.get_world_size(process_group) if process_group is not None else 1
  rank = torch.distributed.get_rank(process_group) if process_group is not None else 0
  N = embeddings.shape[0]
  lo, hi = rank * N // world, (rank + 1) * N // world          # row shard of this rank
  xb = torch.as_tensor(np.ascontiguousarray(embeddings[lo:hi])).to(dev)
  index = ops.FlatIndex(xb, metric)
  print('create index time cost:', time.time() - begin)
  end = time.time()
  D, I = sharded_search(index, xq, nearest_num, lo, metric, process_group)
  D, I = D.cpu().numpy(), I.cpu().numpy()
  index.close()
  print('whole set query time cost:', time.time() - end)
  return D, I


# ============================ de-similarity  ============================
def desim(eI, fI):
  """eI[i, j] = -1 wherever eI[i, j] occurs in row i of fI (faiss_knn.py:134-143); returns the filtered copy."""
  dev = _device()
  e = torch.as_tensor(np.ascontiguousarray(eI, np.int64)).to(dev)
  f = torch.as_tensor(np.ascontiguousarray(fI, np.int64)).to(dev)
  return ops.desim_simple(e, f).cpu().numpy()


def fliter_fI(fI, fD, fD_threshold):
  """Feature neighbours farther than fD_threshold, and the row itself, become -1 (faiss_knn.py:146-155).  iter_desim_mp
  applies this inside its own kernel; this entry point filters a table on its own (desim of an empty eI column)."""
  dev = _device()
  f = torch.as_tensor(np.ascontiguousarray(fI, np.int64)).to(dev)
  d = torch.as_tensor(np.ascontiguousarray(fD, np.float32)).to(dev)
  return ops.filter_fI(f, d, fD_threshold).cpu().numpy().astype(np.int64)


def sharded_desim(eI, fI, fD, fD_threshold=1.4, fI_end=31, process_group=None, desim_fn=None):
  """De-similarity filter with the ROWS of eI split over the ranks (rows are independent: no exchange on the data path);
  every rank holds the whole feature-KNN table (its rows are gathered at random) and the filtered slices are joined by one
  all-gather.  Device tensors in and out, identical on every rank.  `desim_fn` lets the CPU tests drive this protocol
  over gloo with an oracle-backed stand-in for cdml_desim."""
  desim_fn = desim_fn or ops.desim
  world = torch.distributed.get_world_size(process_group) if process_group is not None else 1
  if world == 1:
    return desim_fn(eI, fI, fD, fD_threshold, fI_end)
  rank = torch.distributed.get_rank(process_group)
  n = eI.shape[0]
  per = -(-n // world)                                   # equal slices (the last ones padded with -1 rows) for all_gather
  lo, hi = min(rank * per, n), min((rank + 1) * per, n)
  mine = torch.full((per, eI.shape[1]), -1, dtype=eI.dtype, device=eI.device)
  if hi > lo:
    # the filter drops a row's own id: slice rows keep their GLOBAL row number through the row offset argument
    mine[:hi - lo] = desim_fn(eI[lo:hi].contiguous(), fI, fD, fD_threshold, fI_end, row_offset=lo)
  out = torch.empty((world * per, eI.shape[1]), dtype=eI.dtype, device=eI.device)
  torch.distributed.all_gather_into_tensor(out, mine, group=process_group)
  return out[:n]


def iter_desim_mp(eI, fI, fD, fD_threshold=1.4, fI_end=31, process_num=22, as_device=False, process_group=None):
  """Greedy de-similarity of the KNN lists eI against the raw-feature KNN (fI, fD) (faiss_knn.py:187-244): per row, left
  to right, a surviving entry removes every later entry that is one of its first fI_end near feature neighbours; the
  row's own id is removed last.  Returns int64 [n,ke] with removed entries -1.  `process_num` is accepted and ignored
  (one warp per row on the GPU instead of a process pool); unlike the reference, the inputs are not shifted in place
  (faiss_knn.py:161-162, SURVEY Q6)."""
  begin = time.time()
  dev = _device()
  to_dev = lambda a, dt: a.to(dev) if torch.is_tensor(a) else torch.as_tensor(np.ascontiguousarray(a, dt)).to(dev)
  out = sharded_desim(to_dev(eI, np.int64), to_dev(fI, np.int64), to_dev(fD, np.float32), fD_threshold, fI_end, process_group)
  if ops.poll_errors(out) & 2:
    raise IndexError("iter_desim_mp: eI holds ids beyond the feature KNN table (%d rows)" % fI.shape[0])
  if not as_device:
    out = out.cpu().numpy()
  print('faiss_knn iter_desim_mp cost: ', time.time() - begin)
  return out


def strict_knn(embeddings, fI, fD, knn_result=None, nearest_num=None, decode_map=None, process_group=None):
  """KNN of the embeddings, de-similarised against the raw-feature KNN, written as `strict_knn*` (faiss_knn.py:308-322)."""
  knn_result = FLAGS.knn_result if knn_result is None else knn_result
  nearest_num = FLAGS.nearest_num if nearest_num is None else nearest_num
  strictD, strictI = calc_knn(embeddings, nearest_num=nearest_num, process_group=process_group)
  strictI_desim = iter_desim_mp(strictI, fI, fD, process_group=process_group)
  if process_group is None or torch.distributed.get_rank(process_group) == 0:
    np.save(knn_result + '/strictD.npy', strictD)
    np.save(knn_result + '/strictI.npy', strictI)
    np.save(knn_result + '/strictI_desim.npy', strictI_desim)
    write_knn(knn_result, split_num=10, D=strictD, I=strictI_desim, prefix='strict_knn', decode_map=decode_map)
  return strictD, strictI_desim


def cross_knn(embeddings, doc_location, fI, fD, knn_result=None, nearest_num=None, decode_map=None, process_group=None):
  """Video rows [0, doc_location) search the doc rows and vice versa; the joined lists are de-similarised and written as
  `cross_knn*` (faiss_knn.py:325-351).  The reference at HEAD writes the un-filtered, +1-shifted crossI (SURVEY Q6, its
  own TODO at faiss_knn.py:349); this writes crossI_desim, which is what it saves as crossI_desim.npy."""
  knn_result = FLAGS.knn_result if knn_result is None else knn_result
  nearest_num = FLAGS.nearest_num if nearest_num is None else nearest_num
  video_vec = embeddings[:doc_location]
  doc_vec = embeddings[doc_location:]
  vdD, vdI = calc_knn(doc_vec, video_vec, nearest_num=nearest_num, process_group=process_group)
  vdI = np.where(vdI >= 0, vdI + doc_location, vdI)
  dvD, dvI = calc_knn(video_vec, doc_vec, nearest_num=nearest_num, process_group=process_group)
  crossI = np.concatenate((vdI, dvI), axis=0)
  crossD = np.concatenate((vdD, dvD), axis=0)
  crossI_desim = iter_desim_mp(crossI, fI, fD, process_group=process_group)
  if process_group is None or torch.distributed.get_rank(process_group) == 0:
    np.save(knn_result + '/crossD.npy', crossD)
    np.save(knn_result + '/crossI.npy', crossI)
    np.save(knn_result + '/crossI_desim.npy', crossI_desim)
    write_knn(knn_result, split_num=10, D=crossD, I=crossI_desim, prefix='cross_knn', decode_map=decode_map)
  return crossD, crossI, crossI_desim


# ============================ write result ============================
def format_rows(begin_index, D, I, decode_map):
  """Lines '<query_guid>,<nbr_guid>#<dist><...' ; column 0 skipped; a neighbour is kept iff idx > 0 and
  0.0 < dist < 1.4; dist printed as str(np.float32) (faiss_knn.py:272-280)."""
  lines = []
  for i in range(I.shape[0]):
    parts = [decode_map[begin_index + i], ","]
    for idx, dist in zip(I[i][1:], D[i][1:]):
      if idx > 0 and dist > 0.0 and dist < 1.4:
        parts += [decode_map[idx], "#", str(dist), "<"]
    parts.append("\n")
    lines.append("".join(parts))
  return lines


class GuidTable(object):
  """The decode map {0: guid, ..., n-1: guid} as one UTF-8 blob + offsets: what cdml_format_knn_rows indexes."""

  def __init__(self, decode_map):
    n = len(decode_map)
    try:
      guids = [decode_map[i].encode("utf-8") for i in range(n)]
    except KeyError:
      raise KeyError("the decode map must hold every row index 0..%d" % (n - 1))
    self.n = n
    self.max_len = max((len(g) for g in guids), default=0)
    self.offsets = np.zeros(n + 1, np.int64)
    np.cumsum([len(g) for g in guids], out=self.offsets[1:])
    self.blob = np.frombuffer(b"".join(guids) + b"\0", np.uint8)


def format_rows_bytes(begin_index, D, I, table):
  """The bytes of `format_rows` for a block of rows, produced by libcdml (cdml_format_knn_rows, host code)."""
  from . import _lib
  D = np.ascontiguousarray(D, np.float32)
  I = np.ascontiguousarray(I, np.int64)
  nq, k = I.shape
  out = np.empty(nq * (table.max_len + 2 + (k - 1) * (table.max_len + 42)) + 64, np.uint8)
  n = _lib.load().cdml_format_knn_rows(D.ctypes.data, I.ctypes.data, nq, k, k, int(begin_index), table.blob.ctypes.data,
                                       table.offsets.ctypes.data, table.n, out.ctypes.data, out.size)
  if n < 0:
    _lib.check(-1)
  return out[:n].tobytes()


def write_process(path, index, begin_index, D, I, prefix='knn_split', decode_map=None):
  """One shard file `<path>/<prefix><index>` (faiss_knn.py:267-283)."""
  decode_map = DECODE_MAP if decode_map is None else decode_map
  table = decode_map if isinstance(decode_map, GuidTable) else GuidTable(decode_map)
  try:
    with open(os.path.join(path, prefix + str(index)), 'wb') as fp:
      for lo in range(0, I.shape[0], 65536):                         # bounded scratch: 64k rows at a time
        fp.write(format_rows_bytes(begin_index + lo, D[lo:lo + 65536], I[lo:lo + 65536], table))
  except Exception:
    print(traceback.format_exc())
    raise


def write_knn(knn_result, split_num=10, D=None, I=None, prefix='knn_result', decode_map=None):
  """split_num contiguous patches, the last takes the remainder, one process each (faiss_knn.py:285-305)."""
  os.makedirs(knn_result, exist_ok=True)
  decode_map = DECODE_MAP if decode_map is None else decode_map
  table = GuidTable(decode_map)
  total_num = D.shape[0]
  patch_num = total_num // split_num
  begin = time.time()
  jobs = []
  for i in range(split_num):
    lo = i * patch_num
    hi = (i + 1) * patch_num if i < split_num - 1 else total_num
    jobs.append((knn_result, i, lo, D[lo:hi], I[lo:hi], prefix, table))
  # the formatter is native code called through ctypes (GIL released): threads replace the reference's process pool
  with ThreadPool(processes=min(split_num, os.cpu_count() or 1)) as pool:
    pool.starmap(write_process, jobs)
  print('write_knn cost: %fs' % (time.time() - begin))


def main(args):
  global DECODE_MAP
  try:
    global_begin = time.time()
    DECODE_MAP, _ = load_decode_map(FLAGS.decode_map_file)
    os.makedirs(FLAGS.knn_result, exist_ok=True)
    pg = None
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
      torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
      torch.distributed.init_process_group("nccl")
      pg = torch.distributed.group.WORLD
    embeddings = load_embedding(FLAGS.embedding_file)
    print("faiss_knn embedding_file shape", embeddings.shape)
    if FLAGS.knn_mode in ("strict", "cross"):
      features = load_embedding(FLAGS.pred_feature_file)
      desim_nearest_num = min(FLAGS.desim_nearest_num, FLAGS.nearest_num)                    # faiss_knn.py:376
      fD, fI = calc_knn(features, nearest_num=desim_nearest_num, l2_norm=True, process_group=pg)
      if pg is None or torch.distributed.get_rank() == 0:
        np.save(FLAGS.knn_result + '/fD.npy', fD)
        np.save(FLAGS.knn_result + '/fI.npy', fI)
      if FLAGS.knn_mode == "cross":
        if not 0 < FLAGS.doc_location < embeddings.shape[0]:                                 # faiss_knn.py:390
          raise ValueError("doc_location %d outside (0, %d)" % (FLAGS.doc_location, embeddings.shape[0]))
        cross_knn(embeddings, FLAGS.doc_location, fI, fD, process_group=pg)
      else:
        strict_knn(embeddings, fI, fD, process_group=pg)
      if pg is None or torch.distributed.get_rank() == 0:
        shutil.copyfile(FLAGS.decode_map_file, FLAGS.knn_result + '/decode_map.json')
      print("faiss_knn cost: %fs" % (time.time() - global_begin))
      return
    D, I = calc_knn(embeddings, nearest_num=FLAGS.nearest_num, process_group=pg)
    if pg is None or torch.distributed.get_rank() == 0:
      np.save(FLAGS.knn_result + '/strictD.npy', D)
      np.save(FLAGS.knn_result + '/strictI.npy', I)
      write_knn(FLAGS.knn_result, split_num=10, D=D, I=I, prefix='knn_split')   # cdml_run.sh:147 uploads knn_split*
      shutil.copyfile(FLAGS.decode_map_file, FLAGS.knn_result + '/decode_map.json')
    print("faiss_knn cost: %fs" % (time.time() - global_begin))
  except Exception:
    print(traceback.format_exc())
    raise


if __name__ == '__main__':
  app.run(main)
