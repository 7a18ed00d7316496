"""CPU oracle of in-batch distance-weighted negative sampling -- TEST INFRASTRUCTURE ONLY.

Wu, Manmatha, Smola, Kraehenbuehl: "Sampling Matters in Deep Embedding Learning" (ICCV 2017), build-defined here as the
second mining mode next to cdml_oracle.mine_semihard.  Two statements: the float64 definition
(mine_distance_weighted) and the precision model of the kernel (mine_distance_weighted_emulated16).  The draws use
cdml_oracle.philox4x32_10, pinned to the Random123 known-answer vectors.
"""
from __future__ import annotations

import numpy as np

from .cdml_oracle import philox4x32_10, round16

DW_ONE_MINUS_MIN = 1e-6   # 1 - delta/4 is clamped to this before its log


def dw_log_weight(delta, D):
  """log w(delta) = -((D-2)/2) ln delta - ((D-3)/2) ln max(1 - delta/4, DW_ONE_MINUS_MIN): the inverse of the density
  q(d) ~ d^(D-2) (1 - d^2/4)^((D-3)/2) of distances between uniform points of the unit sphere, written in delta = d^2.
  U-shaped in delta with its minimum at 4(D-2)/(2D-5)."""
  delta = np.asarray(delta, np.float64)
  return -0.5 * (D - 2) * np.log(delta) - 0.5 * (D - 3) * np.log(np.maximum(1.0 - delta / 4.0, DW_ONE_MINUS_MIN))


def dw_unit(x):
  """Philox word -> U = ((x >> 9) + 0.5) 2^-23 in (0, 1), exact in float32."""
  return ((np.asarray(x, np.uint64) >> np.uint64(9)).astype(np.float64) + 0.5) * 2.0 ** -23


def dw_chunk_draws(seed, step, anchor, cid, dtype=np.float64):
  """The 32 Exp(1) draws of each chunk (anchor[k], cid[k]) -> (E [n, 32], M [n], K [n]) (csrc/mine.cu EpiMineDW).
  Philox4x32-10 with key = seed and counter = (anchor, cid, step lo, (step hi << 4) | w):
    w = 0: M = -ln U(word 0) / 32 (the chunk's minimum, Exp(32)), K = word 1 >> 27 (its column);
    w = 1..8: word t -> X_j = -ln U(word t) for column j = 4 (w-1) + t;  E_j = M for j = K, else M + X_j.
  cid = 2 * (column // 32) + cand - 1 for the candidate row 3 * column + cand.  dtype=np.float32 computes M, X and E
  with the kernel's fp32 roundings."""
  anchor = np.asarray(anchor, np.uint64)
  cid = np.asarray(cid, np.uint64)
  n = len(anchor)
  key = (int(seed) & 0xFFFFFFFF, (int(seed) >> 32) & 0xFFFFFFFF)
  c2 = np.full(n, int(step) & 0xFFFFFFFF, np.uint64)
  hi = ((int(step) >> 32) << 4) & 0xFFFFFFFF

  def call(w):
    return philox4x32_10((anchor, cid, c2, np.full(n, hi | w, np.uint64)), key)
  x = call(0)
  M = (-np.log(dw_unit(x[0]).astype(dtype))).astype(dtype) * dtype(1.0 / 32.0)
  K = (x[1] >> np.uint64(27)).astype(np.int64)
  X = np.empty((n, 32), dtype)
  for w in range(1, 9):
    x = call(w)
    for t in range(4):
      X[:, 4 * (w - 1) + t] = -np.log(dw_unit(x[t]).astype(dtype))
  E = (M[:, None] + X).astype(dtype)
  E[np.arange(n), K] = M
  return E, M, K


def dw_draws(seed, step, anchors, B, dtype=np.float64):
  """Draws E [len(anchors), 2B] of every (anchor, candidate) pair, candidates in the order of cand_rows(B)."""
  anchors = np.asarray(anchors, np.int64)
  nq = (B + 31) // 32
  cid = np.arange(2 * nq, dtype=np.uint64)                  # cid = 2 q + cand - 1
  E, _, _ = dw_chunk_draws(seed, step, np.repeat(anchors, 2 * nq), np.tile(cid, len(anchors)), dtype)
  E = E.reshape(len(anchors), nq, 2, 32).transpose(0, 2, 1, 3).reshape(len(anchors), 2, nq * 32)[:, :, :B]
  return E.reshape(len(anchors), 2 * B)


def cand_rows(B):
  """Candidate rows in draw order: the positives' rows 3n+1, then the negatives' rows 3n+2."""
  n = np.arange(B)
  return np.concatenate([3 * n + 1, 3 * n + 2])


def _pick(keys, rows):
  """argmin over (key, row) per anchor; -1 where no key is finite.  Also the gap between the best two keys."""
  order = np.lexsort((np.broadcast_to(rows, keys.shape), keys), axis=1)
  k0 = np.take_along_axis(keys, order[:, :1], 1)[:, 0]
  k1 = np.take_along_axis(keys, order[:, 1:2], 1)[:, 0] if keys.shape[1] > 1 else np.full(len(keys), np.inf)
  pick = np.where(np.isfinite(k0), rows[order[:, 0]], -1)
  return pick, k0, k1 - k0


def mine_distance_weighted(E, guid_triplets, margin, cutoff=0.5, seed=0, step=0, anchors=None):
  """Distance-weighted negative sampling, float64.

  E [3B,D] unit-norm embeddings (rows a0,p0,n0,...), guid_triplets [B,3].  Candidates for triplet i: the rows 3j+1,
  3j+2 whose guid is not a_i or p_i (as mine_semihard).  With s = a_i . c, delta = max(2 - 2s, cutoff^2) and
  dp = |a_i - p_i|^2, a candidate is eligible iff delta < dp + margin (the hinge is active; hard negatives included).
  The pick is argmin over eligible candidates of  ln E_c - dw_log_weight(delta_c, D),  E_c ~ Exp(1) from dw_draws
  (an exponential race: P(c) = w_c / sum w); ties -> lowest row.  No eligible candidate: row 3i+2.
  anchors: optional subset of triplet indices.  Returns (neg_row int32, d_an = |a - E[neg_row]|^2) for those anchors."""
  E = np.asarray(E, np.float64)
  g = np.asarray(guid_triplets)
  B, D = g.shape[0], E.shape[1]
  anchors = np.arange(B) if anchors is None else np.asarray(anchors, np.int64)
  rows = cand_rows(B)
  cg = np.concatenate([g[:, 1], g[:, 2]])
  C = E[rows]
  neg_row = np.empty(len(anchors), np.int32)
  d_an = np.empty(len(anchors))
  for s0 in range(0, len(anchors), 128):
    a = anchors[s0:s0 + 128]
    A = E[3 * a]
    dp = np.sum((A - E[3 * a + 1]) ** 2, -1)
    delta = np.maximum(2.0 - 2.0 * (A @ C.T), cutoff * cutoff)
    ok = (delta < (dp + margin)[:, None]) & (cg[None, :] != g[a, 0:1]) & (cg[None, :] != g[a, 1:2])
    keys = np.where(ok, np.log(dw_draws(seed, step, a, B)) - dw_log_weight(delta, D), np.inf)
    pick, _, _ = _pick(keys, rows)
    pick = np.where(pick < 0, 3 * a + 2, pick)
    neg_row[s0:s0 + 128] = pick
    d_an[s0:s0 + 128] = np.sum((A - E[pick]) ** 2, -1)
  return neg_row, d_an


def mine_distance_weighted_emulated16(E, guid_triplets, margin, cutoff=0.5, seed=0, step=0, kind="fp16", anchors=None):
  """PRECISION MODEL of cdml_mine_distance_weighted (test infrastructure): the definition of mine_distance_weighted with
  the kernel's selection arithmetic -- scores s = a16 . c16 on operands rounded to 16 bits (accumulated in float64,
  rounded once to fp32), dp = |a-p|^2 from the fp32 embeddings, delta = max(fma(-2, s, 2), cutoff^2) and dp + margin in
  fp32, the draws with their fp32 roundings; keys in float64.  Returns (neg_row int32, best key, gap to the runner-up
  key: picks whose gap is at fp32 accumulation noise may legitimately differ, delta of the pick) for `anchors`."""
  E32 = np.asarray(E, np.float32)
  g = np.asarray(guid_triplets)
  B, D = g.shape[0], E32.shape[1]
  anchors = np.arange(B) if anchors is None else np.asarray(anchors, np.int64)
  E16 = round16(E32, kind)
  rows = cand_rows(B)
  cg = np.concatenate([g[:, 1], g[:, 2]])
  C16 = E16[rows]
  dmin = np.float32(cutoff) * np.float32(cutoff)
  n = len(anchors)
  neg_row, key, gap, dsel = np.empty(n, np.int32), np.full(n, np.inf), np.full(n, np.inf), np.full(n, np.nan)
  for s0 in range(0, n, 128):
    a = anchors[s0:s0 + 128]
    dpf = np.sum((E32[3 * a] - E32[3 * a + 1]) ** 2, -1, dtype=np.float32)
    dpm = (dpf + np.float32(margin)).astype(np.float32)
    S = (E16[3 * a] @ C16.T).astype(np.float32)
    delta = np.maximum((np.float32(2.0) - np.float32(2.0) * S).astype(np.float32), dmin)
    ok = (delta < dpm[:, None]) & (cg[None, :] != g[a, 0:1]) & (cg[None, :] != g[a, 1:2])
    Edraw = dw_draws(seed, step, a, B, np.float32).astype(np.float64)
    keys = np.where(ok, np.log(Edraw) - dw_log_weight(delta.astype(np.float64), D), np.inf)
    pick, k0, gp = _pick(keys, rows)
    col = np.where(pick % 3 == 1, (pick - 1) // 3, B + (pick - 2) // 3)     # column of the pick in cand_rows
    neg_row[s0:s0 + 128] = np.where(pick < 0, 3 * a + 2, pick)
    key[s0:s0 + 128], gap[s0:s0 + 128] = k0, gp
    dsel[s0:s0 + 128] = np.where(pick < 0, np.nan, delta[np.arange(len(a)), np.maximum(col, 0)])
  return neg_row, key, gap, dsel
