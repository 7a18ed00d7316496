"""Thin tensor-level wrappers over the C ABI (one function per libcdml entry point).

All tensors are CUDA tensors on the current device; outputs are allocated here with torch (plumbing) and filled by
the hand-written kernels.  Nothing in this module computes on the host or with torch ops."""
import ctypes

import torch

from . import _lib
from ._lib import BF16, EPI_L2NORM, EPI_MASK_BITS, EPI_MASK_LEAKY, EPI_STORE_16, EPI_STORE_F32, F16, check, ptr, stream_ptr

TORCH16 = {F16: torch.float16, BF16: torch.bfloat16}

_LAUNCHES = 0   # kernels of libcdml launched through this module (bench.py reports it as gpu_launches)


def _count(n):
  global _LAUNCHES
  _LAUNCHES += n


def launch_count():
  return _LAUNCHES


def _ctx(t):
  return _lib.context(t.device.index if t.device.index is not None else torch.cuda.current_device())


def dtype16_of(t):
  if t.dtype == torch.float16:
    return F16
  if t.dtype == torch.bfloat16:
    return BF16
  raise TypeError("expected a float16/bfloat16 tensor, got %s" % t.dtype)


def _row_major_2d(t, name):
  if t.dim() != 2 or t.stride(1) != 1:
    raise ValueError("%s must be a 2-D tensor with unit inner stride" % name)
  return t.stride(0)


def poll_errors(device_tensor):
  flags = ctypes.c_int32(0)
  check(_lib.load().cdml_ctx_poll_errors(_ctx(device_tensor), stream_ptr(), ctypes.byref(flags)))
  return flags.value


def gather_rows(table, idx, out=None):
  """out[i] = table[idx[i]]  (inputs.py:158).  table [G,W] any dtype, idx int32/int64 (any shape) -> [*idx.shape, W]."""
  pitch = _row_major_2d(table, "table") * table.element_size()
  flat = idx.reshape(-1)
  if flat.dtype not in (torch.int32, torch.int64):
    raise TypeError("idx must be int32 or int64")
  flat = flat.contiguous()
  row_bytes = table.shape[1] * table.element_size()
  if out is None:
    out = torch.empty((flat.numel(), table.shape[1]), dtype=table.dtype, device=table.device)
  if flat.numel() == 0:
    return out
  out_pitch = _row_major_2d(out, "out") * out.element_size()
  _count(1)
  check(_lib.load().cdml_gather_rows(_ctx(table), ptr(table), table.shape[0], row_bytes, pitch, ptr(flat),
                                     int(flat.dtype == torch.int64), flat.numel(), ptr(out), out_pitch, stream_ptr()))
  return out


def rows_normalize_cast(x, dtype16=F16, normalize=1, eps=1e-12, ld_out=None, want_fp32=False, want_sumsq=False,
                        out16=None):
  """fp32 [n,F] -> 16-bit [n,ld_out] rows, optionally L2-normalised (1: TF semantics, 2: numpy x/||x||)."""
  ld_in = _row_major_2d(x, "x")
  n, F = x.shape
  if ld_out is None:
    ld_out = (F + 7) // 8 * 8
  if out16 is None:
    out16 = torch.empty((n, ld_out), dtype=TORCH16[dtype16], device=x.device)
  out32 = torch.empty((n, F), dtype=torch.float32, device=x.device) if want_fp32 else None
  sumsq = torch.empty((n,), dtype=torch.float32, device=x.device) if want_sumsq else None
  _count(1)
  check(_lib.load().cdml_rows_normalize_cast(_ctx(x), ptr(x), n, F, ld_in, normalize, eps, ptr(out16), out16.stride(0),
                                             dtype16, ptr(out32), F, ptr(sumsq), stream_ptr()))
  return out16, out32, sumsq


def gemm16(A, B, M, N, K, a_mn_major, b_mn_major, epilogue, out, bias=None, alpha=1.0, aux0=None, aux1=None,
           num_splits=1, split_stride=0, ld_out=None):
  """Raw cdml_gemm16 call.  A/B are 16-bit 2-D tensors; shapes are passed explicitly (logical M,N,K)."""
  lda, ldb = _row_major_2d(A, "A"), _row_major_2d(B, "B")
  used = ctypes.c_int(0)
  if ld_out is None:
    ld_out = out.stride(-2) if out.dim() >= 2 else N
  # ld_aux1: row pitch of aux1, or -- STORE_16 with a sign-mask output in aux0 -- the mask's pitch in words
  ld_aux1 = aux1.stride(0) if aux1 is not None else (aux0.stride(0) if (epilogue == EPI_STORE_16 and aux0 is not None) else 0)
  _count(1)
  check(_lib.load().cdml_gemm16(_ctx(A), ptr(A), int(a_mn_major), lda, ptr(B), int(b_mn_major), ldb, M, N, K,
                                dtype16_of(A), epilogue, ptr(out), ld_out, ptr(bias), float(alpha), ptr(aux0),
                                ptr(aux1), ld_aux1, num_splits, split_stride,
                                ctypes.byref(used), stream_ptr()))
  return used.value


def sign_mask_buffer(rows, cols, device):
  """Packed sign mask of a [rows, cols] activation (STORE_16's aux0 / MASK_BITS' aux1): int32 [ceil(cols/32), rows]."""
  return torch.empty(((cols + 31) // 32, rows), dtype=torch.int32, device=device)


def auto_splits(ref, M, N, K):
  return _lib.load().cdml_gemm16_auto_splits(_ctx(ref), M, N, K)


def sum_partials(parts, num_parts, stride, n, out, scale=1.0):
  _count(1)
  check(_lib.load().cdml_sum_partials(_ctx(parts), ptr(parts), num_parts, stride, n, float(scale), ptr(out), stream_ptr()))
  return out


def colsum16(X, R, N, out, workspace=None):
  need = _lib.load().cdml_colsum_workspace_floats(R, N)
  if workspace is None or workspace.numel() < need:
    workspace = torch.empty((need,), dtype=torch.float32, device=X.device)
  _count(2)
  check(_lib.load().cdml_colsum16(_ctx(X), ptr(X), R, N, X.stride(0), dtype16_of(X), ptr(workspace), ptr(out), stream_ptr()))
  return out


def colsum_workspace_floats(R, N):
  return _lib.load().cdml_colsum_workspace_floats(R, N)


def triplet_hinge(E, B, margin, neg_row=None, grad_scale=1.0, rinv=None, leaky_alpha=0.2, want_dE=False, dz16=None,
                  workspace=None, out=None):
  """HingeLoss forward (+ optional backward).  E fp32 [3B,D].  Returns dict of device tensors."""
  D = E.shape[1]
  dev = E.device
  out = out or {}
  pos = out.get("pos_dist") if "pos_dist" in out else torch.empty((B,), dtype=torch.float32, device=dev)
  neg = out.get("neg_dist") if "neg_dist" in out else torch.empty((B,), dtype=torch.float32, device=dev)
  hin = out.get("hinge_dist") if "hinge_dist" in out else torch.empty((B,), dtype=torch.float32, device=dev)
  stats = out.get("stats") if "stats" in out else torch.empty((4,), dtype=torch.float32, device=dev)
  dE = None
  if want_dE:
    dE = out.get("dE") if "dE" in out else torch.empty_like(E)
  if dz16 is not None and dE is None and workspace is None:
    workspace = torch.empty((3 * B * E.stride(0),), dtype=torch.float32, device=dev)
  mined_grad = neg_row is not None and (dE is not None or dz16 is not None)     # + the two fixed-point passes
  _count(2 + (2 if mined_grad else 0) + (1 if dz16 is not None else 0))
  check(_lib.load().cdml_triplet_hinge(_ctx(E), ptr(E), B, D, E.stride(0), ptr(neg_row), float(margin), float(grad_scale),
                                       ptr(rinv), float(leaky_alpha), ptr(pos), ptr(neg), ptr(hin), ptr(stats), ptr(dE),
                                       ptr(dz16), dz16.stride(0) if dz16 is not None else 0,
                                       dtype16_of(dz16) if dz16 is not None else F16, ptr(workspace), stream_ptr()))
  return {"pos_dist": pos, "neg_dist": neg, "hinge_dist": hin, "stats": stats, "dE": dE, "dz16": dz16}


def adam_prepare(step_counter, scalars, base_lr, decay_steps=1e6, decay_rate=0.96, staircase=True, beta1=0.9,
                 beta2=0.999):
  _count(1)
  check(_lib.load().cdml_adam_prepare(_ctx(scalars), ptr(step_counter), float(base_lr), float(decay_steps),
                                      float(decay_rate), int(staircase), float(beta1), float(beta2), ptr(scalars),
                                      stream_ptr()))


def adam_apply(w, m, v, g, scalars, beta1=0.9, beta2=0.999, eps=1e-8, grad_scale=1.0, w16=None):
  _count(1)
  check(_lib.load().cdml_adam_apply(_ctx(w), ptr(w), ptr(m), ptr(v), ptr(g), w.numel(), ptr(scalars), float(beta1),
                                    float(beta2), float(eps), float(grad_scale), ptr(w16),
                                    dtype16_of(w16) if w16 is not None else F16, stream_ptr()))


OPT_ADAM, OPT_MOMENTUM, OPT_LARS, OPT_SGD = 0, 1, 2, 3


def opt_workspace_floats():
  return int(_lib.load().cdml_opt_workspace_floats())


def opt_sumsq(g, w, out2, workspace, grad_scale=1.0, wd_reg=0.0):
  """out2 = {sum (grad_scale*g + wd_reg*w)^2, sum w^2} of one variable (device fp32 [2])."""
  _count(2)
  check(_lib.load().cdml_opt_sumsq(_ctx(w), ptr(g), ptr(w), w.numel(), float(grad_scale), float(wd_reg), ptr(workspace),
                                   ptr(out2), stream_ptr()))
  return out2


def opt_apply(kind, w, m, v, g, scalars, norms=None, beta1=0.9, beta2=0.999, eps=1e-8, grad_scale=1.0, wd_reg=0.0,
              clip_norm=0.0, momentum=0.9, lars_weight_decay=1e-4, lars_eeta=1e-3, w16=None):
  _count(1)
  check(_lib.load().cdml_opt_apply(_ctx(w), int(kind), ptr(w), ptr(m), ptr(v), ptr(g), w.numel(), ptr(scalars), ptr(norms),
                                   float(beta1), float(beta2), float(eps), float(grad_scale), float(wd_reg), float(clip_norm),
                                   float(momentum), float(lars_weight_decay), float(lars_eeta), ptr(w16),
                                   dtype16_of(w16) if w16 is not None else F16, stream_ptr()))


EW_MUL, EW_ADD, EW_MUL_ADD_BOTH, EW_MASK, EW_MUL_ADD, EW_FMA, EW_MUL_ADD_MASK, EW_MUL_MASK = 0, 1, 2, 3, 4, 5, 6, 7


def ew16(op, a, b, out, c=None, alpha=0.2):
  """Elementwise join of 16-bit [rows, cols] matrices (cdml_ew16); `out` may alias an input."""
  rows, cols = out.shape
  _count(1)
  check(_lib.load().cdml_ew16(_ctx(out), int(op), ptr(a), a.stride(0), ptr(b), b.stride(0), ptr(c),
                              c.stride(0) if c is not None else 0, ptr(out), out.stride(0), rows, cols, float(alpha),
                              dtype16_of(out), stream_ptr()))
  return out


def rows_l2norm16(y16, e, rinv=None, e16=None, eps=1e-12):
  """tf.nn.l2_normalize of 16-bit rows -> fp32 e (+ rinv, + 16-bit copy)."""
  n, D = y16.shape
  _count(1)
  check(_lib.load().cdml_rows_l2norm16(_ctx(y16), ptr(y16), n, D, y16.stride(0), float(eps), dtype16_of(y16), ptr(e),
                                       e.stride(0), ptr(rinv), ptr(e16), e16.stride(0) if e16 is not None else 0,
                                       stream_ptr()))
  return e


def cast16(x, out16):
  _count(1)
  check(_lib.load().cdml_cast16(_ctx(x), ptr(x), x.numel(), ptr(out16), dtype16_of(out16), stream_ptr()))
  return out16


def fill_column16(X16, col, value):
  """X16[:, col] = value for a 16-bit matrix whose pitch exceeds its logical width (padding columns)."""
  if X16.dim() != 2 or X16.stride(1) != 1 or not (0 <= col < X16.stride(0)):
    raise ValueError("fill_column16: column %d outside the row pitch" % col)
  _count(1)
  check(_lib.load().cdml_fill_column16(_ctx(X16), ptr(X16), X16.shape[0], X16.stride(0), int(col), float(value),
                                       dtype16_of(X16), stream_ptr()))


def sample_triplets(pairs, start, B, num_guid, seed, out=None):
  """[B,3] int64 (anchor, positive, negative) index triplets from device-resident pairs [n,2] (cdml_sample_triplets)."""
  if pairs.dtype != torch.int64 or pairs.dim() != 2 or pairs.shape[1] != 2 or not pairs.is_contiguous():
    raise TypeError("pairs must be a contiguous int64 [n,2] tensor")
  if out is None:
    out = torch.empty((B, 3), dtype=torch.int64, device=pairs.device)
  if B == 0:
    return out
  _count(1)
  check(_lib.load().cdml_sample_triplets(_ctx(pairs), ptr(pairs), pairs.shape[0], int(start), int(B), int(num_guid),
                                         int(seed) & 0xFFFFFFFFFFFFFFFF, ptr(out), stream_ptr()))
  return out


def desim(eI, fI, fD=None, fD_threshold=1.4, f_end=31, out=None, row_offset=0):
  """De-similarity filter of KNN lists (cdml_desim; faiss_knn.py:187-244).  eI [n,ke] int64, fI [nf,kf] int64, fD [nf,kf]
  fp32 device tensors -> int64 [n,ke] with dropped entries -1."""
  if eI.dtype != torch.int64 or fI.dtype != torch.int64 or (fD is not None and fD.dtype != torch.float32):
    raise TypeError("desim: eI / fI must be int64, fD float32")
  n, ke = eI.shape
  nf, kf = fI.shape
  lib = _lib.load()
  ws = torch.empty((max(int(lib.cdml_desim_workspace_bytes(nf, kf, int(f_end))), 4),), dtype=torch.uint8, device=eI.device)
  if out is None:
    out = torch.empty_like(eI)
  if n == 0:
    return out
  _count(2)
  check(lib.cdml_desim(_ctx(eI), ptr(eI), n, ke, _row_major_2d(eI, "eI"), ptr(fI), ptr(fD), nf, kf, _row_major_2d(fI, "fI"),
                       _row_major_2d(fD, "fD") if fD is not None else 0, float(fD_threshold), int(f_end), ptr(ws), ptr(out),
                       _row_major_2d(out, "out"), int(row_offset), stream_ptr()))
  return out


def filter_fI(fI, fD, fD_threshold=1.4):
  """fliter_fI (faiss_knn.py:146-155) on its own: the int32 table cdml_desim gathers from ([nf,kf] view)."""
  nf, kf = fI.shape
  probe = torch.full((1, 1), -1, dtype=torch.int64, device=fI.device)          # a row without pivots: only `prepare` matters
  lib = _lib.load()
  ws = torch.empty((int(lib.cdml_desim_workspace_bytes(nf, kf, kf)),), dtype=torch.uint8, device=fI.device)
  _count(2)
  check(lib.cdml_desim(_ctx(fI), ptr(probe), 1, 1, 1, ptr(fI), ptr(fD), nf, kf, _row_major_2d(fI, "fI"),
                       _row_major_2d(fD, "fD"), float(fD_threshold), kf, ptr(ws), ptr(probe), 1, 0, stream_ptr()))
  return ws.view(torch.int32).view(nf, -1)[:, :kf]          # int32 ids, -1 = filtered


def desim_simple(eI, fI, out=None):
  """out[i,j] = -1 where eI[i,j] occurs in fI[i,:] (cdml_desim_simple; faiss_knn.py:134-143)."""
  n, ke = eI.shape
  if out is None:
    out = torch.empty_like(eI)
  _count(1)
  check(_lib.load().cdml_desim_simple(_ctx(eI), ptr(eI), n, ke, _row_major_2d(eI, "eI"), ptr(fI), fI.shape[1],
                                      _row_major_2d(fI, "fI"), ptr(out), _row_major_2d(out, "out"), stream_ptr()))
  return out


def mean_pair_dist(V, pairs):
  out = torch.empty((1,), dtype=torch.float32, device=V.device)
  pairs = pairs.to(torch.int64).contiguous()
  _count(2)
  check(_lib.load().cdml_mean_pair_dist(_ctx(V), ptr(V), V.stride(0), V.shape[1], ptr(pairs), pairs.shape[0], ptr(out),
                                        stream_ptr()))
  return out


def mine_semihard(E16, E32, guid, B, margin, want_dist=True):
  D = E32.shape[1]
  neg_row = torch.empty((B,), dtype=torch.int32, device=E32.device)
  d_an = torch.empty((B,), dtype=torch.float32, device=E32.device) if want_dist else None
  guid = guid.to(torch.int64).contiguous()
  _count(4)
  check(_lib.load().cdml_mine_semihard(_ctx(E32), ptr(E16), E16.stride(0), dtype16_of(E16), ptr(E32), E32.stride(0),
                                       ptr(guid), B, D, float(margin), ptr(neg_row), ptr(d_an), stream_ptr()))
  return neg_row, d_an


def mine_distance_weighted(E16, E32, guid, B, margin, cutoff=0.5, seed=0, step=None, want_dist=True):
  """Distance-weighted negative sampling (Wu et al. 2017): neg_row [B] int32 sampled among the candidates with
  max(d, cutoff^2) < |a-p|^2 + margin with probability ~ 1/q(d), q the density of distances on the unit sphere; d_an the
  exact fp32 distance of the pick (want_dist).  step: a one-element int64 device tensor read by the kernel (the engine's
  step counter, so that graph replays draw afresh), or None for step 0."""
  D = E32.shape[1]
  if step is not None and (step.dtype != torch.int64 or step.device != E32.device or step.numel() < 1):
    raise ValueError("mine_distance_weighted: step must be an int64 tensor on %s" % E32.device)
  neg_row = torch.empty((B,), dtype=torch.int32, device=E32.device)
  d_an = torch.empty((B,), dtype=torch.float32, device=E32.device) if want_dist else None
  guid = guid.to(torch.int64).contiguous()
  _count(4)
  check(_lib.load().cdml_mine_distance_weighted(_ctx(E32), ptr(E16), E16.stride(0), dtype16_of(E16), ptr(E32),
                                                E32.stride(0), ptr(guid), B, D, float(margin), float(cutoff),
                                                int(seed) & 0xFFFFFFFFFFFFFFFF, ptr(step), ptr(neg_row), ptr(d_an),
                                                stream_ptr()))
  return neg_row, d_an


def mine_stats(ref):
  """Diagnostics of the last mine_semihard or mine_distance_weighted on ref's device: {"rescans": re-scanned (anchor, 32-candidate chunk) pairs,
  "mined": anchors that received a mined negative}.  Synchronises the current stream."""
  out = (ctypes.c_int64 * 2)()
  check(_lib.load().cdml_mine_last_stats(_ctx(ref), out, stream_ptr()))
  return {"rescans": int(out[0]), "mined": int(out[1])}


class FlatIndex(object):
  """Exact flat index resident on one GPU (IndexFlatL2 / IndexFlatIP semantics; faiss_knn.py:116-128)."""

  def __init__(self, xb, metric="L2"):
    if xb.dtype != torch.float32 or xb.dim() != 2 or not xb.is_cuda:
      raise TypeError("FlatIndex needs a CUDA float32 [N,d] tensor")
    self.metric = {"L2": _lib.METRIC_L2, "IP": _lib.METRIC_IP}[metric]
    self.n, self.d = xb.shape
    self._ref = xb
    self._h = ctypes.c_void_p()
    _count(5)
    check(_lib.load().cdml_knn_index_build(_ctx(xb), ptr(xb), self.n, self.d, _row_major_2d(xb, "xb"), self.metric,
                                           stream_ptr(), ctypes.byref(self._h)))

  def search(self, xq, k, id_offset=0):
    if xq.dtype != torch.float32 or xq.dim() != 2 or xq.shape[1] != self.d:
      raise TypeError("queries must be float32 [nq,%d]" % self.d)
    nq = xq.shape[0]
    D = torch.empty((nq, k), dtype=torch.float32, device=xq.device)
    I = torch.empty((nq, k), dtype=torch.int64, device=xq.device)
    _count(6 * ((nq + 32767) // 32768))
    check(_lib.load().cdml_knn_search(_ctx(xq), self._h, ptr(xq), nq, _row_major_2d(xq, "xq"), k, ptr(D), ptr(I),
                                      int(id_offset), stream_ptr()))
    return D, I

  def bounds(self, xq, k_full, k_part):
    """Bound pass only: per query the raw k_full-th and k_part-th best sampled scores of this shard (device fp32 [nq])."""
    nq = xq.shape[0]
    bf = torch.empty((nq,), dtype=torch.float32, device=xq.device)
    bp = torch.empty((nq,), dtype=torch.float32, device=xq.device)
    _count(4 * ((nq + 32767) // 32768))
    check(_lib.load().cdml_knn_bounds(_ctx(xq), self._h, ptr(xq), nq, _row_major_2d(xq, "xq"), int(k_full), int(k_part),
                                      ptr(bf), ptr(bp), stream_ptr()))
    return bf, bp

  def search_bounded(self, xq, k, bound_full, bound_part, id_offset=0):
    """Collect + refine above max(bound_full, bound_part) - slack (bounds agreed across shards by the caller)."""
    nq = xq.shape[0]
    D = torch.empty((nq, k), dtype=torch.float32, device=xq.device)
    I = torch.empty((nq, k), dtype=torch.int64, device=xq.device)
    _count(5 * ((nq + 32767) // 32768))
    check(_lib.load().cdml_knn_search_bounded(_ctx(xq), self._h, ptr(xq), nq, _row_major_2d(xq, "xq"), k, ptr(bound_full),
                                              ptr(bound_part), ptr(D), ptr(I), int(id_offset), stream_ptr()))
    return D, I

  # ---- row-sharded protocol, one chunk (<= 65536 queries) per call; see include/cdml.h
  CHUNK = 65536

  def shard_bounds(self, xq, k, k_part, pair=None):
    nq = xq.shape[0]
    if pair is None:
      pair = torch.empty((2, nq), dtype=torch.float32, device=xq.device)
    _count(4)
    check(_lib.load().cdml_knn_shard_bounds(_ctx(xq), self._h, ptr(xq), nq, _row_major_2d(xq, "xq"), int(k), int(k_part),
                                            ptr(pair), stream_ptr()))
    return pair

  def shard_collect(self, xq, k, k_part, pair, nom_pair=None):
    nq = xq.shape[0]
    if nom_pair is None:
      nom_pair = torch.empty((2, nq), dtype=torch.float32, device=xq.device)
    _count(6)
    check(_lib.load().cdml_knn_shard_collect(_ctx(xq), self._h, ptr(xq), nq, _row_major_2d(xq, "xq"), int(k), int(k_part),
                                             ptr(pair), ptr(nom_pair), stream_ptr()))
    return nom_pair

  def shard_refine(self, xq, k, nom_pair, rec, id_offset=0, overflow_flag=None):
    """rec: int64 [nq,k] slice receiving the packed records of this chunk.  overflow_flag (device int32 [1]): deferred
    overflow check -- no host synchronisation; the word becomes 1 if a query overflowed (the caller then repeats the
    search without the flag)."""
    nq = xq.shape[0]
    _count(3)
    check(_lib.load().cdml_knn_shard_refine(_ctx(xq), self._h, ptr(xq), nq, _row_major_2d(xq, "xq"), int(k), ptr(nom_pair),
                                            ptr(rec), int(id_offset), ptr(overflow_flag), stream_ptr()))
    return rec

  def last_stats(self):
    s = (ctypes.c_int64 * 2)()
    check(_lib.load().cdml_knn_last_stats(self._h, s))
    return {"candidates": int(s[0]), "fallback_queries": int(s[1])}

  def close(self):
    if self._h:
      _lib.load().cdml_knn_index_destroy(self._h)
      self._h = ctypes.c_void_p()

  def __del__(self):
    try:
      self.close()
    except Exception:
      pass


def knn_merge_packed(rec, metric="L2", as_records=False):
  """[G,nq,k] int64 packed records (FlatIndex.shard_refine) -> global top-k D fp32 / I int64 [nq,k] (ties -> lower id), or
  (as_records) the merged lists as int64 records [nq,k]."""
  G, nq, k = rec.shape
  rec = rec.contiguous()
  m = {"L2": 0, "IP": 1}[metric]
  _count(1)
  if as_records:
    out = torch.empty((nq, k), dtype=torch.int64, device=rec.device)
    check(_lib.load().cdml_knn_merge_packed(_ctx(rec), ptr(rec), G, nq, k, m, None, None, ptr(out), stream_ptr()))
    return out
  D = torch.empty((nq, k), dtype=torch.float32, device=rec.device)
  I = torch.empty((nq, k), dtype=torch.int64, device=rec.device)
  check(_lib.load().cdml_knn_merge_packed(_ctx(rec), ptr(rec), G, nq, k, m, ptr(D), ptr(I), None, stream_ptr()))
  return D, I


def knn_unpack_records(rec, metric="L2"):
  """int64 records [nq,k] -> D fp32, I int64 (padding -> inf / -1)."""
  rec = rec.contiguous()
  D = torch.empty(rec.shape, dtype=torch.float32, device=rec.device)
  I = torch.empty(rec.shape, dtype=torch.int64, device=rec.device)
  _count(1)
  check(_lib.load().cdml_knn_unpack_records(_ctx(rec), ptr(rec), rec.numel(), {"L2": 0, "IP": 1}[metric], ptr(D), ptr(I),
                                            stream_ptr()))
  return D, I


def knn_merge(Dg, Ig, metric="L2"):
  """[G,nq,k] per-shard results -> global top-k (ties -> lower id)."""
  G, nq, k = Dg.shape
  Dg, Ig = Dg.contiguous(), Ig.contiguous()
  D = torch.empty((nq, k), dtype=torch.float32, device=Dg.device)
  I = torch.empty((nq, k), dtype=torch.int64, device=Dg.device)
  _count(1)
  check(_lib.load().cdml_knn_merge(_ctx(Dg), ptr(Dg), ptr(Ig), G, nq, k, {"L2": 0, "IP": 1}[metric], ptr(D), ptr(I),
                                   stream_ptr()))
  return D, I
