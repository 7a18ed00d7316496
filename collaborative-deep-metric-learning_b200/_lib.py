"""ctypes binding of libcdml.so (include/cdml.h).  PyTorch tensors only carry device memory: every call passes
``tensor.data_ptr()`` + geometry + the current CUDA stream.  There is no CPU fallback: a missing library raises."""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcdml.so")

F16, BF16 = 0, 1
EPI_STORE_F32, EPI_STORE_16, EPI_L2NORM, EPI_MASK_LEAKY, EPI_MASK_BITS = 0, 1, 2, 3, 4
METRIC_L2, METRIC_IP = 0, 1

_P = c_void_p
_SIGNATURES = {
  "cdml_ctx_create": (c_int, [c_int, POINTER(c_void_p)]),
  "cdml_ctx_destroy": (c_int, [_P]),
  "cdml_last_error": (c_char_p, []),
  "cdml_version": (c_int, []),
  "cdml_ctx_poll_errors": (c_int, [_P, _P, POINTER(c_int32)]),
  "cdml_gather_rows": (c_int, [_P, _P, c_int64, c_int64, c_int64, _P, c_int, c_int64, _P, c_int64, _P]),
  "cdml_rows_normalize_cast": (c_int, [_P, _P, c_int64, c_int64, c_int64, c_int, c_float, _P, c_int64, c_int, _P,
                                       c_int64, _P, _P]),
  "cdml_gemm16": (c_int, [_P, _P, c_int, c_int64, _P, c_int, c_int64, c_int64, c_int64, c_int64, c_int, c_int, _P,
                          c_int64, _P, c_float, _P, _P, c_int64, c_int, c_int64, POINTER(c_int), _P]),
  "cdml_gemm16_auto_splits": (c_int, [_P, c_int64, c_int64, c_int64]),
  "cdml_sum_partials": (c_int, [_P, _P, c_int, c_int64, c_int64, c_float, _P, _P]),
  "cdml_colsum_workspace_floats": (c_int64, [c_int64, c_int64]),
  "cdml_colsum16": (c_int, [_P, _P, c_int64, c_int64, c_int64, c_int, _P, _P, _P]),
  "cdml_triplet_hinge": (c_int, [_P, _P, c_int64, c_int, c_int64, _P, c_float, c_float, _P, c_float, _P, _P, _P, _P,
                                 _P, _P, c_int64, c_int, _P, _P]),
  "cdml_adam_prepare": (c_int, [_P, _P, c_float, c_float, c_float, c_int, c_float, c_float, _P, _P]),
  "cdml_adam_apply": (c_int, [_P, _P, _P, _P, _P, c_int64, _P, c_float, c_float, c_float, c_float, _P, c_int, _P]),
  "cdml_opt_workspace_floats": (c_int64, []),
  "cdml_opt_sumsq": (c_int, [_P, _P, _P, c_int64, c_float, c_float, _P, _P, _P]),
  "cdml_opt_apply": (c_int, [_P, c_int, _P, _P, _P, _P, c_int64, _P, _P, c_float, c_float, c_float, c_float, c_float,
                             c_float, c_float, c_float, c_float, _P, c_int, _P]),
  "cdml_ew16": (c_int, [_P, c_int, _P, c_int64, _P, c_int64, _P, c_int64, _P, c_int64, c_int64, c_int, c_float, c_int, _P]),
  "cdml_rows_l2norm16": (c_int, [_P, _P, c_int64, c_int, c_int64, c_float, c_int, _P, c_int64, _P, _P, c_int64, _P]),
  "cdml_desim_workspace_bytes": (c_int64, [c_int64, c_int, c_int]),
  "cdml_desim": (c_int, [_P, _P, c_int64, c_int, c_int64, _P, _P, c_int64, c_int, c_int64, c_int64, c_float, c_int, _P, _P,
                         c_int64, c_int64, _P]),
  "cdml_desim_simple": (c_int, [_P, _P, c_int64, c_int, c_int64, _P, c_int, c_int64, _P, c_int64, _P]),
  "cdml_sample_triplets": (c_int, [_P, _P, c_int64, c_int64, c_int64, c_int64, ctypes.c_uint64, _P, _P]),
  "cdml_format_knn_rows": (c_int64, [_P, _P, c_int64, c_int, c_int64, c_int64, _P, _P, c_int64, _P, c_int64]),
  "cdml_format_f32": (c_int64, [_P, c_int64, _P, c_int64]),
  "cdml_parse_features_txt": (c_int64, [_P, c_int64, c_int, _P, c_int64, _P, _P, c_int]),
  "cdml_cast16": (c_int, [_P, _P, c_int64, _P, c_int, _P]),
  "cdml_fill_column16": (c_int, [_P, _P, c_int64, c_int64, c_int64, c_float, c_int, _P]),
  "cdml_mine_semihard": (c_int, [_P, _P, c_int64, c_int, _P, c_int64, _P, c_int64, c_int, c_float, _P, _P, _P]),
  "cdml_mine_distance_weighted": (c_int, [_P, _P, c_int64, c_int, _P, c_int64, _P, c_int64, c_int, c_float, c_float,
                                          ctypes.c_uint64, _P, _P, _P, _P]),
  "cdml_mine_last_stats": (c_int, [_P, _P, _P]),
  "cdml_knn_index_build": (c_int, [_P, _P, c_int64, c_int, c_int64, c_int, _P, POINTER(c_void_p)]),
  "cdml_knn_index_destroy": (c_int, [_P]),
  "cdml_knn_search": (c_int, [_P, _P, _P, c_int64, c_int64, c_int, _P, _P, c_int64, _P]),
  "cdml_knn_bounds": (c_int, [_P, _P, _P, c_int64, c_int64, c_int, c_int, _P, _P, _P]),
  "cdml_knn_search_bounded": (c_int, [_P, _P, _P, c_int64, c_int64, c_int, _P, _P, _P, _P, c_int64, _P]),
  "cdml_knn_last_stats": (c_int, [_P, POINTER(c_int64)]),
  "cdml_knn_merge": (c_int, [_P, _P, _P, c_int, c_int64, c_int, c_int, _P, _P, _P]),
  "cdml_knn_shard_bounds": (c_int, [_P, _P, _P, c_int64, c_int64, c_int, c_int, _P, _P]),
  "cdml_knn_shard_collect": (c_int, [_P, _P, _P, c_int64, c_int64, c_int, c_int, _P, _P, _P]),
  "cdml_knn_shard_refine": (c_int, [_P, _P, _P, c_int64, c_int64, c_int, _P, _P, c_int64, _P, _P]),
  "cdml_knn_merge_packed": (c_int, [_P, _P, c_int, c_int64, c_int, c_int, _P, _P, _P, _P]),
  "cdml_knn_unpack_records": (c_int, [_P, _P, c_int64, c_int, _P, _P, _P]),
  "cdml_mean_pair_dist": (c_int, [_P, _P, c_int64, c_int, _P, c_int64, _P, _P]),
}

_lib = None


class CdmlError(RuntimeError):
  pass


def load():
  """dlopen libcdml.so and attach prototypes.  Raises if the extension has not been built."""
  global _lib
  if _lib is not None:
    return _lib
  if not os.path.exists(LIB_PATH):
    raise CdmlError("libcdml.so is missing at %s -- run `python -c 'import __graft_entry__ as g; g.build()'`. "
                    "There is no CPU fallback for the CDML hot path." % LIB_PATH)
  lib = ctypes.CDLL(LIB_PATH)
  for name, (res, args) in _SIGNATURES.items():
    fn = getattr(lib, name)
    fn.restype = res
    fn.argtypes = args
  _lib = lib
  return lib


def exported_symbols():
  return sorted(_SIGNATURES)


def check(rc):
  if rc != 0:
    msg = load().cdml_last_error()
    raise CdmlError("libcdml call failed (%d): %s" % (rc, msg.decode() if msg else "?"))


_contexts = {}


def context(device_index):
  """One cdml_ctx per (process, device)."""
  ctx = _contexts.get(device_index)
  if ctx is None:
    lib = load()
    h = c_void_p()
    check(lib.cdml_ctx_create(int(device_index), ctypes.byref(h)))
    ctx = _contexts[device_index] = h
  return ctx


def ptr(t):
  """Device pointer of a torch tensor (None -> NULL)."""
  return None if t is None else c_void_p(t.data_ptr())


def stream_ptr():
  import torch
  return c_void_p(torch.cuda.current_stream().cuda_stream)
