"""Graph engine for the visual+doc fusion towers (models.py:65-243: MultiplyNet, MlpNet, ResNet -- the tower of train.py
main(), train.py:363 -- and ResNetV2).  Executes the op list `models.compile_graph` produces:

  input(lo,hi)  l2-normalised column slice of the raw features (visual 0:1500, doc 1500:1628; models.py:80-86)
  fc            leaky(x.W + b)                      tcgen05 GEMM, STORE_16 epilogue (L2NORM epilogue when it feeds the output)
  mul / add     elementwise joins of 256-wide rows  cdml_ew16
  l2norm        the model output                    cdml_rows_l2norm16 (fp32 e, rinv, 16-bit e for mining)

and its reverse sweep (gradients of the SUM of hinges, 16-bit, like the chain engine): every node collects the
contributions of its consumers -- `direct` (adds, data-gradient GEMMs) or `prod` (multiply: g * other operand) -- and
materialises them with cdml_ew16 (first contribution: alias or MUL, later ones: ADD / FMA) when the sweep reaches it.
A data-gradient GEMM whose target is a single-use fc output applies leaky' in its epilogue (MASK_LEAKY) and writes dz
directly, so the 5000-wide visual layer never sees an elementwise pass.  Parameters, optimizers, the all-reduce and CUDA
graph capture are inherited from TowerEngine; each input slice has its own normalised 16-bit table with the ones column
of [x | 1] behind it (bias gradient = extra row of the weight-gradient GEMM).
"""
import json

import torch

from . import ops
from ._lib import EPI_L2NORM, EPI_MASK_BITS, EPI_MASK_LEAKY, EPI_STORE_16, F16
from .engine import LEAKY_ALPHA, TowerEngine, _pad64


def _widths(spec):
  w = []
  for e in spec:
    if e["op"] == "input":
      w.append(int(e["hi"]) - int(e["lo"]))
    elif e["op"] == "fc":
      w.append(int(e["out"]))
    elif e["op"] in ("mul", "add"):
      w.append(w[e["src"][0]])
    else:
      w.append(w[e["src"]])
  return w


class GraphEngine(TowerEngine):

  def __init__(self, spec, feature_size=None, device=None, dtype16=F16, seed=2, init_params=None, loss_scale=256.0, **kw):
    spec = [dict(e) for e in spec]
    if not spec or spec[-1]["op"] != "l2norm" or any(e["op"] == "l2norm" for e in spec[:-1]):
      raise ValueError("the op list must end with its only l2norm (the model output)")
    self.spec = spec
    self.widths = _widths(spec)
    for i, e in enumerate(spec):
      srcs = e["src"] if isinstance(e.get("src"), list) else [e["src"]] if "src" in e else []
      if any(not (0 <= s < i) for s in srcs):
        raise ValueError("op %d consumes a later op" % i)
      if any(spec[s]["op"] == "input" for s in srcs) and e["op"] != "fc":
        raise NotImplementedError("input slices feed fully_connected layers only")
      if e["op"] in ("mul", "add") and len({self.widths[s] for s in srcs}) != 1:
        raise ValueError("op %d joins tensors of different widths" % i)
      if e["op"] == "mul" and len(srcs) != 2:
        raise ValueError("mul takes two operands")
    self.inputs = [i for i, e in enumerate(spec) if e["op"] == "input"]
    self.fcs = [i for i, e in enumerate(spec) if e["op"] == "fc"]
    self.layer_of = {i: l for l, i in enumerate(self.fcs)}
    self.consumers = {i: [] for i in range(len(spec))}
    for i, e in enumerate(spec):
      for s in (e["src"] if isinstance(e.get("src"), list) else [e["src"]] if "src" in e else []):
        self.consumers[s].append(i)
    dead = [i for i in range(len(spec) - 1) if not self.consumers[i]]
    if dead:
      raise ValueError("ops %s do not reach the model output" % dead)
    F = int(feature_size) if feature_size is not None else max(int(spec[i]["hi"]) for i in self.inputs)
    D = self.widths[-1]
    if D % 2:
      raise ValueError("output width must be even")
    alphas = {float(spec[i].get("alpha", LEAKY_ALPHA)) for i in self.fcs}
    if len(alphas) != 1:
      raise NotImplementedError("all layers must share one leaky slope")
    kw.setdefault("alpha", alphas.pop())
    kw.setdefault("bias_init", [float(spec[i].get("bias_init", 0.1)) for i in self.fcs])
    # an fc whose only consumer is the output l2norm runs the fused L2NORM epilogue (MlpNet; VNet as a graph)
    last = spec[-1]["src"]
    self.fused_out = last if (spec[last]["op"] == "fc" and len(self.consumers[last]) == 1 and D <= 256) else None
    super().__init__([F, D], device=device, dtype16=dtype16, seed=seed, init_params=init_params,
                     layer_shapes=[(self.widths[spec[i]["src"]], self.widths[i]) for i in self.fcs], **kw)
    # The residual sums make |y| of the output large (rinv ~ 0.08 on an untrained ResNet), so the backward signal of the
    # sum of hinges sits at 1e-4..1e-3 -- around fp16's smallest normal 6.1e-5.  A power-of-two loss scale lifts it into the
    # normal range (headroom: |g| <= 4, rinv of order 1 -> <= ~1e4 of 65504); the optimizer kernel divides it out again.
    self.loss_scale = float(loss_scale)
    self.names = [spec[i].get("name") or ("fully_connected" if l == 0 else "fully_connected_%d" % l)
                  for l, i in enumerate(self.fcs)]

  # ------------------------------------------------------------------ parameters
  def state_dict(self):
    sd = super().state_dict()
    sd["spec"] = json.dumps(self.spec)
    return sd

  # ------------------------------------------------------------------ inputs: one normalised 16-bit table per slice
  def _table_rows(self, tables):
    return tables[0].shape[0]

  def prepare_table(self, features, out=None):
    """fp32 [G,F] -> tuple of L2-normalised 16-bit tables, one per input slice, each with the ones column behind it."""
    segs = []
    for k, i in enumerate(self.inputs):
      lo, hi = int(self.spec[i]["lo"]), int(self.spec[i]["hi"])
      x16, _, _ = ops.rows_normalize_cast(features[:, lo:hi], self.dtype16, 1, float(self.spec[i].get("eps", 1e-12)),
                                          ld_out=_pad64(hi - lo + 1), out16=None if out is None else out[k])
      ops.fill_column16(x16, hi - lo, 1.0)
      segs.append(x16)
    return tuple(segs)

  def _input_has_ones(self, tables):
    return all(TowerEngine._input_has_ones(_Seg(self, w), t) for t, w in zip(tables, (self.widths[i] for i in self.inputs)))

  # ------------------------------------------------------------------ buffers
  def _buffers(self, R, train):
    key = (R, train)
    buf = self._bufs.get(key)
    if buf is not None:
      if key not in self._pinned_bufs:
        self._bufs[key] = self._bufs.pop(key)      # most recently used goes last (TowerEngine._store_buffers)
      return buf
    dev, t16, spec, D = self.device, self.t16, self.spec, self.widths[-1]

    def mat16(cols, ones):
      m = torch.empty((R, _pad64(cols + 1)), dtype=t16, device=dev)
      if ones:
        ops.fill_column16(m, cols, 1.0)
      return m[:, :cols]

    buf = {"val": {}, "e": torch.empty((R, D), dtype=torch.float32, device=dev),
           "rinv": torch.empty((R,), dtype=torch.float32, device=dev)}
    for i, e in enumerate(spec[:-1]):
      if e["op"] != "input" and i != self.fused_out:
        feeds_fc = any(spec[c]["op"] == "fc" for c in self.consumers[i])
        buf["val"][i] = mat16(self.widths[i], train and feeds_fc)
    if train:
      B = R // 3
      # single-use fc outputs that feed an fc: their data gradient applies leaky' in the GEMM epilogue and needs only the
      # SIGN of the activation -- one bit per element, written by the forward epilogue (TowerEngine does the same)
      buf["mask"] = {s: ops.sign_mask_buffer(R, self.widths[s], dev) for s in self._masked_nodes()}
      buf["dz"] = {i: mat16(self.widths[i], False) for i in self.fcs}
      buf["grad"] = {}     # materialised node gradients / data-gradient temporaries, allocated on first use
      buf["dzo"] = mat16(D, False)
      buf["G"] = torch.empty((R, D), dtype=torch.float32, device=dev)
      buf["loss"] = {k: torch.empty((B,), dtype=torch.float32, device=dev) for k in ("pos_dist", "neg_dist", "hinge_dist")}
      buf["loss"]["stats"] = torch.empty((4,), dtype=torch.float32, device=dev)
      buf["wrows"] = [fi + 1 for fi, _ in self.shapes]      # every fc input here carries the ones column
      buf["splits"] = [ops.auto_splits(self.w, buf["wrows"][l], fo, R) for l, (_, fo) in enumerate(self.shapes)]
      part = max(s * buf["wrows"][l] * self.shapes[l][1] if s > 1 else 0 for l, s in enumerate(buf["splits"]))
      buf["partials"] = torch.empty((max(part, 1),), dtype=torch.float32, device=dev)
      buf["colsum_ws"] = torch.empty((max(ops.colsum_workspace_floats(R, fo) for _, fo in self.shapes),),
                                     dtype=torch.float32, device=dev)
    self._store_buffers(key, buf)
    return buf

  def _masked_nodes(self):
    """fc outputs whose only consumer is an fc: the targets of the MASK_BITS data-gradient epilogue (backward_rows)."""
    spec = self.spec
    return [e["src"] for i, e in enumerate(spec) if e["op"] == "fc" and spec[e["src"]]["op"] == "fc"
            and len(self.consumers[e["src"]]) == 1 and e["src"] != self.fused_out]

  def _scratch(self, buf, key, cols):
    m = buf["grad"].get(key)
    if m is None:
      R = buf["e"].shape[0]
      m = buf["grad"][key] = torch.empty((R, _pad64(cols + 1)), dtype=self.t16, device=self.device)[:, :cols]
    return m

  # ------------------------------------------------------------------ forward
  def forward_rows(self, xsegs, R, train=False, want_e16=None):
    buf = self._buffers(R, train)
    val = dict(buf["val"])
    for k, i in enumerate(self.inputs):
      val[i] = xsegs[k][:, :self.widths[i]]
    for i, e in enumerate(self.spec):
      op = e["op"]
      if op == "fc":
        l = self.layer_of[i]
        K, N = self.shapes[l]
        if i == self.fused_out:
          ops.gemm16(val[e["src"]], self.W16[l], R, N, K, 0, 1, EPI_L2NORM, buf["e"], bias=self.b[l], alpha=self.alpha,
                     aux0=buf["rinv"], aux1=want_e16)
        else:
          ops.gemm16(val[e["src"]], self.W16[l], R, N, K, 0, 1, EPI_STORE_16, val[i], bias=self.b[l], alpha=self.alpha,
                     aux0=buf["mask"].get(i) if train else None)
      elif op == "mul":
        ops.ew16(ops.EW_MUL, val[e["src"][0]], val[e["src"][1]], val[i])
      elif op == "add":
        acc = val[e["src"][0]]
        for s in e["src"][1:]:
          acc = ops.ew16(ops.EW_ADD, acc, val[s], val[i])
      elif op == "l2norm" and e["src"] != self.fused_out:
        ops.rows_l2norm16(val[e["src"]], buf["e"], rinv=buf["rinv"], e16=want_e16, eps=float(e.get("eps", 1e-12)))
    buf["vals"] = val
    return buf

  def embed(self, x, batch_rows=None):
    """Prediction.predict (predict.py:67-69): fp32 [n,F] raw features -> fp32 [n,D] embeddings (device tensor)."""
    n = x.shape[0]
    segs = []
    for i in self.inputs:
      lo, hi = int(self.spec[i]["lo"]), int(self.spec[i]["hi"])
      segs.append(ops.rows_normalize_cast(x[:, lo:hi], self.dtype16, 1, float(self.spec[i].get("eps", 1e-12)),
                                          ld_out=_pad64(hi - lo + 1))[0])
    return self.forward_rows(tuple(segs), n, train=False)["e"]

  # ------------------------------------------------------------------ training
  def train_step_indices(self, tables, idx, mine=False, guid=None):
    B = idx.shape[0]
    xsegs = []
    for k, t in enumerate(tables):
      x16 = self._ws.get(("x16", k, B))
      if x16 is None:
        x16 = self._ws[("x16", k, B)] = torch.empty((3 * B, t.stride(0)), dtype=self.t16, device=self.device)
      ops.gather_rows(t, idx, out=x16)
      xsegs.append(x16)
    return self.train_step_rows(tuple(xsegs), B, mine=mine, guid=idx if guid is None else guid,
                                input_ones=self._input_has_ones(tables))

  def train_step_rows(self, xsegs, B, mine=False, guid=None, input_ones=None):
    R = 3 * B
    if input_ones is None:
      input_ones = self._input_has_ones(xsegs)
    e16 = None
    if mine:
      e16 = self._ws.get(("e16", R))
      if e16 is None:
        e16 = self._ws[("e16", R)] = torch.empty((R, self.widths[-1]), dtype=self.t16, device=self.device)
    buf = self.forward_rows(xsegs, R, train=True, want_e16=e16)
    neg_row = self._mine_negatives(e16, buf["e"], guid, B, mine) if mine else None
    # loss + backward through the output L2-norm (and the last leaky when the output fc is fused)
    ops.triplet_hinge(buf["e"], B, self.margin, neg_row=neg_row, grad_scale=self.loss_scale, rinv=buf["rinv"],
                      leaky_alpha=self.alpha if self.fused_out is not None else 1.0, dz16=buf["dzo"],
                      workspace=buf["G"], out=buf["loss"])
    self.backward_rows(xsegs, R, buf, input_ones)
    self.apply_gradients(B)
    return buf["loss"]["stats"]

  def _materialise(self, i, contrib, buf):
    """Sum of the gradient contributions of node i (16-bit [R,w])."""
    terms = contrib.pop(i, [])
    if not terms:
      raise RuntimeError("op %d received no gradient" % i)
    if len(terms) == 1 and terms[0][0] == "direct":
      return terms[0][1]
    acc = None
    out = self._scratch(buf, ("g", i), self.widths[i])
    for t in terms:
      if t[0] == "direct":
        if acc is None:
          acc = t[1]
          continue
        ops.ew16(ops.EW_ADD, acc, t[1], out)
      elif acc is None:
        ops.ew16(ops.EW_MUL, t[1], t[2], out)
      else:
        ops.ew16(ops.EW_FMA, t[1], t[2], out, c=acc)
      acc = out
    return acc

  def backward_rows(self, xsegs, R, buf, input_ones=False):
    spec, val = self.spec, buf["vals"]
    contrib, dz = {}, {}
    last = spec[-1]["src"]
    if last == self.fused_out:
      dz[last] = buf["dzo"]
    else:
      contrib.setdefault(last, []).append(("direct", buf["dzo"]))
    for i in range(len(spec) - 2, -1, -1):
      e = spec[i]
      op = e["op"]
      if op == "input":
        continue
      if op == "fc":
        l = self.layer_of[i]
        K_in, N_out = self.shapes[l]
        s = e["src"]
        if i not in dz:
          dz[i] = ops.ew16(ops.EW_MASK, self._materialise(i, contrib, buf), val[i], buf["dz"][i], alpha=self.alpha)
        from_input = spec[s]["op"] == "input"
        inp = xsegs[self.inputs.index(s)] if from_input else val[s]
        self._weight_gradient(l, inp, dz[i], R, buf, with_bias_row=(input_ones or not from_input))
        if from_input:
          continue
        if spec[s]["op"] == "fc" and len(self.consumers[s]) == 1:
          # data gradient + leaky' of the producing layer in one epilogue: dz[s] = (dz[i] . W^T) * leaky'(h_s)
          ops.gemm16(dz[i], self.W16[l], R, K_in, N_out, 0, 0, EPI_MASK_BITS, buf["dz"][s], alpha=self.alpha, aux1=buf["mask"][s])
          dz[s] = buf["dz"][s]
        else:
          tmp = self._scratch(buf, ("d", i), K_in)
          ops.gemm16(dz[i], self.W16[l], R, K_in, N_out, 0, 0, EPI_STORE_16, tmp, alpha=1.0)
          contrib.setdefault(s, []).append(("direct", tmp))
      elif op == "mul":
        g = self._materialise(i, contrib, buf)
        a, b = e["src"]
        contrib.setdefault(a, []).append(("prod", g, val[b]))
        contrib.setdefault(b, []).append(("prod", g, val[a]))
      else:  # add
        g = self._materialise(i, contrib, buf)
        for s in e["src"]:
          contrib.setdefault(s, []).append(("direct", g))

  def loss_rows(self, xsegs, B):
    buf = self.forward_rows(xsegs, 3 * B, train=True)
    ops.triplet_hinge(buf["e"], B, self.margin, out=buf["loss"])
    return buf


class _Seg:
  """Adapter that lets TowerEngine._input_has_ones inspect one input slice's table."""

  def __init__(self, eng, width):
    self.F, self._ones_checked, self.fused_bias_grad = width, eng._ones_checked, eng.fused_bias_grad

  def _bias_row_ok(self, width, pitch):
    return self.fused_bias_grad and pitch > width
