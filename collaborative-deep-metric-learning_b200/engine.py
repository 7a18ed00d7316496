"""Tower engine: the reference's `build_graph` (train.py:74-175) + `Prediction.predict` (predict.py:67-69) executed by
libcdml kernels.  Owns the fp32 master weights / Adam state (one flat buffer each, so the data-parallel gradient
exchange is a single all-reduce), the 16-bit shadow weights the tensor cores read, and the per-batch activation
buffers.  Every arithmetic step is a C-ABI call; torch only allocates memory and (for N>1 ranks) runs the NCCL
all-reduce of the flat gradient buffer.

Forward (models.py:46-62 and `fully_connected` models.py:19-30), per row of the [3B,F] batch:
  xhat = l2norm(x) -> h_l = leaky(h_{l-1} W_l + b_l) for every layer (also the last) -> e = l2norm(h_L)
Backward = the written-out autodiff of train.py:141-142 (see oracle/cdml_oracle.py::tower_backward).
"""
import math
import os
import weakref

import numpy as np
import torch

from . import ops
from ._lib import BF16, EPI_L2NORM, EPI_MASK_BITS, EPI_MASK_LEAKY, EPI_STORE_16, EPI_STORE_F32, F16

LEAKY_ALPHA = 0.2


def _pad8(n):
  return (n + 7) // 8 * 8


def _pad64(n):
  """Row pitch of 16-bit activation matrices: a multiple of 64 elements = 128 bytes, so that every row starts on a
  cache line and the epilogues' 64-byte row pieces never straddle 32-byte sectors (1.3x DRAM over-fetch otherwise)."""
  return (n + 63) // 64 * 64


class TowerEngine:
  """Stack of `fully_connected` layers with input/output L2-normalisation (VNet: dims=[1500,5000,256])."""

  def __init__(self, dims, device=None, dtype16=F16, seed=2, bias_init=0.0, base_lr=1e-3, margin=0.8,
               lr_decay_steps=1000000, lr_decay=0.96, beta1=0.9, beta2=0.999, eps=1e-8, alpha=LEAKY_ALPHA,
               process_group=None, init_params=None, optimizer="adam", clip_norm=0.0, reg_penalty=0.0, l2_penalty=1e-8,
               momentum=0.9, lars_weight_decay=1e-4, lars_eeta=1e-3, layer_shapes=None):
    """`layer_shapes` ([(in,out)] per fully_connected layer; `bias_init` may then be a list): parameter layout of a tower
    that is not a plain chain (fusion.GraphEngine); default = consecutive `dims`."""
    if not torch.cuda.is_available():
      raise RuntimeError("TowerEngine needs a CUDA device (sm_100a); there is no CPU path")
    self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
    self.dims = [int(d) for d in dims]
    if self.dims[-1] > 256:
      raise ValueError("output_size must be <= 256 (the L2-norm epilogue holds the whole row in one tile)")
    for d in self.dims[1:]:
      if d % 8:
        raise ValueError("layer widths must be multiples of 8 (16-byte row pitch for TMA); got %d" % d)
    self.shapes = [(int(a), int(b)) for a, b in (layer_shapes if layer_shapes is not None else zip(self.dims[:-1], self.dims[1:]))]
    for _, d in self.shapes:
      if d % 8:
        raise ValueError("layer widths must be multiples of 8 (16-byte row pitch for TMA); got %d" % d)
    self.L = len(self.shapes)
    self.dtype16 = dtype16
    self.t16 = ops.TORCH16[dtype16]
    self.alpha = float(alpha)
    self.margin = float(margin)
    self.base_lr, self.lr_decay_steps, self.lr_decay = float(base_lr), float(lr_decay_steps), float(lr_decay)
    self.beta1, self.beta2, self.eps = beta1, beta2, eps
    # build_graph's gradient path (train.py:133-146): final_loss = reg_penalty * sum(l2_penalty * |W|^2 / 2) + loss, optional
    # per-variable clip_by_norm, then the optimizer: adam | momentum (nesterov) | lars | sgd
    self.opt_kind = {"adam": ops.OPT_ADAM, "momentum": ops.OPT_MOMENTUM, "lars": ops.OPT_LARS, "sgd": ops.OPT_SGD}[optimizer]
    self.clip_norm, self.wd_reg = float(clip_norm), float(reg_penalty) * float(l2_penalty)
    self.momentum, self.lars_wd, self.lars_eeta = float(momentum), float(lars_weight_decay), float(lars_eeta)
    self.pg = process_group
    self.world = torch.distributed.get_world_size(process_group) if process_group is not None else 1
    self.F = self.dims[0]
    self.F_pad = _pad64(self.F + 1)     # always one spare column: it carries the ones of [x | 1] (bias gradient row)
    self.loss_scale = 1.0          # multiplies the 16-bit backward signal; divided out inside the optimizer kernel's grad_scale
    self.fused_bias_grad = True    # bias gradients as an extra row of the weight-gradient GEMMs (no colsum kernels)
    self.ddp_buckets = os.environ.get("CDML_DDP_BUCKETS", "0") == "1"
    self._ones_checked = {}

    # ---- flat fp32 parameter / gradient / Adam buffers; per-tensor views ----
    sizes = []
    for fi, fo in self.shapes:
      sizes += [fi * fo, fo]
    self.offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    # keep every tensor 16-byte aligned inside the flat buffer
    self.offsets = np.concatenate([[0], np.cumsum([_pad8(s) for s in sizes])]).astype(np.int64)
    total = int(self.offsets[-1])
    dev = self.device
    self.w = torch.zeros(total, dtype=torch.float32, device=dev)
    self.m = torch.zeros(total, dtype=torch.float32, device=dev)
    self.v = torch.zeros(total, dtype=torch.float32, device=dev)
    self.g = torch.zeros(total, dtype=torch.float32, device=dev)
    self.sizes = sizes
    self.W = [self._view(self.w, 2 * l).view(*self.shapes[l]) for l in range(self.L)]
    self.b = [self._view(self.w, 2 * l + 1) for l in range(self.L)]
    self.gW = [self._view(self.g, 2 * l).view(*self.shapes[l]) for l in range(self.L)]
    self.gb = [self._view(self.g, 2 * l + 1) for l in range(self.L)]
    self.W16 = [torch.zeros(self.shapes[l], dtype=self.t16, device=dev) for l in range(self.L)]
    self.step_counter = torch.zeros(1, dtype=torch.int64, device=dev)
    # distance-weighted mining (mine="distance_weighted"): distance cutoff and the seed of its draws; the draws of a step
    # are also keyed by step_counter, which the kernel reads from device memory (a replayed graph draws afresh)
    self.dw_cutoff, self.dw_seed = 0.5, int(seed)
    self.scalars = torch.zeros(4, dtype=torch.float32, device=dev)
    self.norms = torch.zeros((2 * self.L, 2), dtype=torch.float32, device=dev)       # per variable: {sum g_eff^2, sum w^2}
    self.opt_ws = torch.empty((ops.opt_workspace_floats(),), dtype=torch.float32, device=dev)
    self._bufs = {}
    self._pinned_bufs = set()      # keys of self._bufs whose pointers are baked into a captured CUDA graph
    self._ws = {}

    if init_params is None:
      rng = np.random.RandomState(seed)
      init_params = []
      biases = list(bias_init) if isinstance(bias_init, (list, tuple)) else [bias_init] * self.L
      for (fi, fo), b0 in zip(self.shapes, biases):
        lim = math.sqrt(6.0 / (fi + fo))  # slim xavier_initializer (uniform)
        init_params.append((rng.uniform(-lim, lim, size=(fi, fo)).astype(np.float32), np.full((fo,), b0, np.float32)))
    self.load_params(init_params)

  # ------------------------------------------------------------------ parameters
  def _view(self, flat, i):
    o = int(self.offsets[i])
    return flat[o:o + self.sizes[i]]

  def load_params(self, params):
    """params: [(W [in,out], b [out])] numpy / torch, e.g. from a checkpoint or the oracle's init."""
    for l, (W, b) in enumerate(params):
      self.W[l].copy_(torch.as_tensor(np.asarray(W), dtype=torch.float32))
      self.b[l].copy_(torch.as_tensor(np.asarray(b), dtype=torch.float32))
    self.refresh_shadows()

  def refresh_shadows(self):
    for l in range(self.L):
      ops.cast16(self.W[l], self.W16[l])

  def get_params(self):
    return [(self.W[l].detach().cpu().numpy().copy(), self.b[l].detach().cpu().numpy().copy()) for l in range(self.L)]

  OPT_NAMES = {ops.OPT_ADAM: "adam", ops.OPT_MOMENTUM: "momentum", ops.OPT_LARS: "lars", ops.OPT_SGD: "sgd"}

  def hyper(self):
    """Everything besides the tensors that a served / resumed tower must agree on (saved with every checkpoint): the
    operand type the tower was TRAINED in, the activation slope, which optimizer the m / v slots belong to."""
    return {"dtype16": int(self.dtype16), "alpha": self.alpha, "optimizer": self.OPT_NAMES[self.opt_kind],
            "loss_scale": self.loss_scale, "margin": self.margin, "base_lr": self.base_lr,
            "lr_decay_steps": self.lr_decay_steps, "lr_decay": self.lr_decay, "beta1": self.beta1, "beta2": self.beta2,
            "eps": self.eps, "clip_norm": self.clip_norm, "wd_reg": self.wd_reg, "momentum": self.momentum,
            "lars_weight_decay": self.lars_wd, "lars_eeta": self.lars_eeta}

  def state_dict(self):
    return {"dims": self.dims, "w": self.w.cpu().numpy(), "m": self.m.cpu().numpy(), "v": self.v.cpu().numpy(),
            "step": int(self.step_counter.item()), "hyper": self.hyper()}

  def load_state_dict(self, sd):
    have = sd.get("hyper")
    if have is not None and have.get("optimizer", self.OPT_NAMES[self.opt_kind]) != self.OPT_NAMES[self.opt_kind]:
      # the m / v slots of another optimizer mean something else (Momentum / LARS accumulators are not Adam moments)
      raise ValueError("checkpoint optimizer state is %s, this engine runs %s" % (have["optimizer"], self.OPT_NAMES[self.opt_kind]))
    self.w.copy_(torch.as_tensor(sd["w"]))
    self.m.copy_(torch.as_tensor(sd["m"]))
    self.v.copy_(torch.as_tensor(sd["v"]))
    self.step_counter.fill_(int(sd["step"]))
    self.refresh_shadows()

  @property
  def global_step(self):
    return int(self.step_counter.item())

  # ------------------------------------------------------------------ buffers
  def _buffers(self, R, train):
    key = (R, train)
    buf = self._bufs.get(key)
    if buf is not None:
      if key not in self._pinned_bufs:
        self._bufs[key] = self._bufs.pop(key)      # most recently used goes last
      return buf
    dev, t16 = self.device, self.t16
    D = self.dims[-1]
    def mat16(cols, spare=0):
      return torch.empty((R, _pad64(cols + spare)), dtype=t16, device=dev)[:, :cols]

    def act16(cols):
      # hidden activations feed the next layer's weight-gradient GEMM as [h | 1]: the spare pitch column `cols` holds 1.0
      # (written once; the forward epilogue only writes columns < cols, the forward GEMM of the next layer reads K = cols)
      m = mat16(cols, 1 if train else 0)
      if train and self._bias_row_ok(cols, m.stride(0)):
        ops.fill_column16(m, cols, 1.0)
      return m

    buf = {"acts": [act16(self.dims[l + 1]) for l in range(self.L - 1)],
           "e": torch.empty((R, D), dtype=torch.float32, device=dev),
           "rinv": torch.empty((R,), dtype=torch.float32, device=dev)}
    if train:
      B = R // 3
      buf["dz"] = [mat16(self.dims[l + 1]) for l in range(self.L)]
      # 1 bit per hidden activation: written by the forward epilogue, read by the data-gradient epilogue (leaky')
      buf["mask"] = [ops.sign_mask_buffer(R, self.dims[l + 1], dev) for l in range(self.L - 1)]
      buf["G"] = torch.empty((R, D), dtype=torch.float32, device=dev)
      buf["loss"] = {k: torch.empty((B,), dtype=torch.float32, device=dev) for k in ("pos_dist", "neg_dist", "hinge_dist")}
      buf["loss"]["stats"] = torch.empty((4,), dtype=torch.float32, device=dev)
      # rows of the weight-gradient GEMM: in (+1 when the bias gradient rides along as the row of the ones column)
      in_pitch = [self.F_pad] + [a.stride(0) for a in buf["acts"]]
      buf["wrows"] = [self.dims[l] + (1 if self._bias_row_ok(self.dims[l], in_pitch[l]) else 0) for l in range(self.L)]
      buf["splits"] = [ops.auto_splits(self.w, buf["wrows"][l], self.dims[l + 1], R) for l in range(self.L)]
      part = max(s * buf["wrows"][l] * self.dims[l + 1] if s > 1 else 0 for l, s in enumerate(buf["splits"]))
      buf["partials"] = torch.empty((max(part, 1),), dtype=torch.float32, device=dev)
      buf["colsum_ws"] = torch.empty((max(ops.colsum_workspace_floats(R, d) for d in self.dims[1:]),),
                                     dtype=torch.float32, device=dev)
    self._store_buffers(key, buf)
    return buf

  def _store_buffers(self, key, buf):
    """Cache policy: a captured CUDA graph holds the raw pointers of its (R, train=True) buffers, so those are pinned for
    the life of the engine (`_pinned_bufs`); everything else is an LRU of 4 entries (eval batch, eval tail, predict
    batch, predict tail come and go with different row counts and must not push the training buffers out)."""
    self._bufs[key] = buf
    loose = [k for k in self._bufs if k not in self._pinned_bufs]
    for k in loose[:max(0, len(loose) - 4)]:       # dict order = insertion order; hits are re-inserted by _buffers
      del self._bufs[k]

  def _bias_row_ok(self, width, pitch):
    """[x | 1]^T . dz = [dW ; db]: possible when the input matrix has a spare pitch column for the ones and the bias
    gradient directly follows the weight gradient in the flat buffer (true whenever in*out is a multiple of 8)."""
    return self.fused_bias_grad and pitch > width

  # ------------------------------------------------------------------ forward
  def forward_rows(self, x16, R, train=False, want_e16=None):
    """x16: 16-bit [R, >=F] already-normalised input rows.  Returns the buffer dict (e, rinv, acts)."""
    buf = self._buffers(R, train)
    h = x16
    for l in range(self.L):
      K, N = self.dims[l], self.dims[l + 1]
      if l < self.L - 1:
        ops.gemm16(h, self.W16[l], R, N, K, 0, 1, EPI_STORE_16, buf["acts"][l], bias=self.b[l], alpha=self.alpha,
                   aux0=buf["mask"][l] if train else None)
        h = buf["acts"][l]
      else:
        ops.gemm16(h, self.W16[l], R, N, K, 0, 1, EPI_L2NORM, buf["e"], bias=self.b[l], alpha=self.alpha,
                   aux0=buf["rinv"], aux1=want_e16)
    return buf

  def embed(self, x, batch_rows=None):
    """Prediction.predict (predict.py:67-69): fp32 [n,F] raw features -> fp32 [n,D] embeddings (device tensor)."""
    n = x.shape[0]
    x16, _, _ = ops.rows_normalize_cast(x, self.dtype16, 1, 1e-12, ld_out=self.F_pad)
    buf = self.forward_rows(x16, n, train=False)
    return buf["e"]

  # ------------------------------------------------------------------ training
  def prepare_table(self, features, out=None):
    """K2 folded into a one-off table transform: fp32 [G,F] -> L2-normalised 16-bit [G,F_pad] resident in HBM."""
    x16, _, _ = ops.rows_normalize_cast(features, self.dtype16, 1, 1e-12, ld_out=self.F_pad, out16=out)
    if self._bias_row_ok(self.F, x16.stride(0)):
      ops.fill_column16(x16, self.F, 1.0)     # the ones column of [x | 1] (first padding column; never read by the forward GEMM)
    return x16

  def _table_rows(self, table16):
    return table16.shape[0]

  def _input_has_ones(self, x16):
    """First use of an input matrix: does its padding column F hold the ones `prepare_table` plants?  (One 2-byte
    read per distinct buffer; a table built by other means silently falls back to the column-sum kernel.)"""
    key = (x16.data_ptr(), x16.stride(0), x16.shape[0])
    hit = self._ones_checked.get(key)
    # the verdict is tied to the tensor's STORAGE (weak reference): an address the allocator hands out again after the
    # checked buffer was freed must be looked at again
    if hit is not None and hit[1]() is not None and hit[1]()._cdata == x16.untyped_storage()._cdata:
      return hit[0]
    ok = bool(self._bias_row_ok(self.F, x16.stride(0)) and float(x16[0, :self.F + 1][-1].item()) == 1.0
              and float(x16[x16.shape[0] - 1, :self.F + 1][-1].item()) == 1.0) if x16.shape[0] else False
    if len(self._ones_checked) > 64:
      self._ones_checked.clear()
    self._ones_checked[key] = (ok, weakref.ref(x16.untyped_storage()))
    return ok

  def train_step_indices(self, table16, idx, mine=False, guid=None):
    """One optimisation step from guid index triplets [B,3] (device int32/int64): gather -> fwd -> loss -> bwd -> Adam."""
    B = idx.shape[0]
    x16 = self._ws.get(("x16", B))
    if x16 is None:
      x16 = self._ws[("x16", B)] = torch.empty((3 * B, self.F_pad), dtype=self.t16, device=self.device)
    ops.gather_rows(table16, idx, out=x16)
    return self.train_step_rows(x16, B, mine=mine, guid=idx if guid is None else guid,
                                input_ones=self._input_has_ones(table16))

  def train_step_rows(self, x16, B, mine=False, guid=None, input_ones=None):
    R = 3 * B
    if input_ones is None:
      input_ones = self._input_has_ones(x16)
    D = self.dims[-1]
    e16 = None
    if mine:
      e16 = self._ws.get(("e16", R))
      if e16 is None:
        e16 = self._ws[("e16", R)] = torch.empty((R, D), dtype=self.t16, device=self.device)
    buf = self.forward_rows(x16, R, train=True, want_e16=e16)
    neg_row = self._mine_negatives(e16, buf["e"], guid, B, mine) if mine else None
    dz = buf["dz"]
    # loss + backward through the output L2-norm and last leaky (gradients of the SUM of hinges; 1/B goes into Adam)
    ops.triplet_hinge(buf["e"], B, self.margin, neg_row=neg_row, grad_scale=1.0, rinv=buf["rinv"],
                      leaky_alpha=self.alpha, dz16=dz[self.L - 1], workspace=buf["G"], out=buf["loss"])
    self.backward_rows(x16, R, buf, input_ones)
    self.apply_gradients(B)
    return buf["loss"]["stats"]

  def _mine_negatives(self, e16, e, guid, B, mine):
    """In-batch negatives of a training step.  mine: True or "semihard" -> semi-hard mining; "distance_weighted" ->
    distance-weighted sampling with (dw_cutoff, dw_seed) at the current step_counter."""
    if mine is True or mine == "semihard":
      return ops.mine_semihard(e16, e, guid, B, self.margin, want_dist=False)[0]
    if mine == "distance_weighted":
      return ops.mine_distance_weighted(e16, e, guid, B, self.margin, self.dw_cutoff, self.dw_seed, self.step_counter,
                                        want_dist=False)[0]
    raise ValueError("mine must be False, True, 'semihard' or 'distance_weighted' (got %r)" % (mine,))

  def backward_rows(self, x16, R, buf, input_ones=False):
    dz = buf["dz"]
    self._pending = []
    for l in range(self.L - 1, -1, -1):
      K_in, N_out = self.dims[l], self.dims[l + 1]
      inp = x16 if l == 0 else buf["acts"][l - 1]
      self._weight_gradient(l, inp, dz[l], R, buf, with_bias_row=(l > 0 or input_ones))
      if self.world > 1 and self.ddp_buckets and l > 0:
        # bucketed exchange: [dW_l ; db_l] is complete -- its all-reduce may run (on NCCL's stream) under the data-gradient
        # and weight-gradient GEMMs of the layers below.  Off by default: the GEMMs are persistent kernels that own every
        # SM (one CTA of ~215 KB shared memory and ~56K registers per SM), so a concurrent NCCL kernel only gets SMs
        # when a GEMM CTA retires -- measured no gain (DESIGN.md section 5)
        o0, o1 = int(self.offsets[2 * l]), int(self.offsets[2 * l + 2])
        self._pending.append(torch.distributed.all_reduce(self.g[o0:o1], group=self.pg, async_op=True))
      if l > 0:
        # data gradient + leaky' of the previous layer: dz[l-1] = (dz[l] . W_l^T) * leaky'(h_{l-1})
        ops.gemm16(dz[l], self.W16[l], R, K_in, N_out, 0, 0, EPI_MASK_BITS, dz[l - 1], alpha=self.alpha,
                   aux1=buf["mask"][l - 1])

  def _weight_gradient(self, l, inp, dz, R, buf, with_bias_row):
    """dW[in,out] = inp^T[in,R] . dz[R,out]   (both operands MN-major, K = R).  With the ones column the GEMM has in+1
    rows and its last row IS the bias gradient; [dW ; db] is one contiguous block of the flat buffer."""
    K_in, N_out = self.shapes[l]
    s = buf["splits"][l]
    rows = buf["wrows"][l] if with_bias_row else K_in
    o = int(self.offsets[2 * l])
    gWb = self.g[o:o + rows * N_out]
    if s > 1:
      used = ops.gemm16(inp, dz, rows, N_out, R, 1, 1, EPI_STORE_F32, buf["partials"], num_splits=s,
                        split_stride=rows * N_out, ld_out=N_out)
      ops.sum_partials(buf["partials"], used, rows * N_out, rows * N_out, gWb)
    else:
      ops.gemm16(inp, dz, rows, N_out, R, 1, 1, EPI_STORE_F32, gWb, ld_out=N_out)
    if rows == K_in:
      ops.colsum16(dz, R, N_out, self.gb[l], buf["colsum_ws"])

  def apply_gradients(self, B_local):
    if self.world > 1:
      pending = getattr(self, "_pending", [])
      if pending:                      # layers >= 1 are already in flight; layer 0's block follows and all are awaited
        torch.distributed.all_reduce(self.g[:int(self.offsets[2])], group=self.pg)
        for w in pending:
          w.wait()
        self._pending = []
      else:
        torch.distributed.all_reduce(self.g, group=self.pg)  # NCCL sum over ranks, one flat buffer
    ops.adam_prepare(self.step_counter, self.scalars, self.base_lr, self.lr_decay_steps, self.lr_decay, True,
                     self.beta1, self.beta2)
    scale = 1.0 / (B_local * self.world * self.loss_scale)
    plain_adam = self.opt_kind == ops.OPT_ADAM and self.clip_norm <= 0 and self.wd_reg == 0
    for l in range(self.L):
      for i, (w, g, w16, wd) in enumerate(((self.W[l], self.gW[l], self.W16[l], self.wd_reg), (self.b[l], self.gb[l], None, 0.0))):
        m, v = self._view(self.m, 2 * l + i), self._view(self.v, 2 * l + i)
        if plain_adam:
          ops.adam_apply(w, m, v, g, self.scalars, self.beta1, self.beta2, self.eps, scale, w16=w16)
          continue
        norms = None
        if self.clip_norm > 0 or self.opt_kind == ops.OPT_LARS:
          norms = ops.opt_sumsq(g, w, self.norms[2 * l + i], self.opt_ws, grad_scale=scale, wd_reg=wd)
        ops.opt_apply(self.opt_kind, w, m, v, g, self.scalars, norms, self.beta1, self.beta2,
                      0.0 if self.opt_kind == ops.OPT_LARS else self.eps, scale, wd, self.clip_norm, self.momentum,
                      self.lars_wd, self.lars_eeta, w16=w16)

  def reg_loss(self):
    """sum_l l2_penalty * |W_l|^2 / 2 scaled by nothing (the summary `reg_loss`, train.py:133-136); host-side read."""
    tot = 0.0
    for l in range(self.L):
      ops.opt_sumsq(self.gW[l], self.W[l], self.norms[2 * l], self.opt_ws)
      tot += 0.5 * float(self.norms[2 * l][1].item())
    return tot * (self.wd_reg if self.wd_reg else 0.0)

  # ------------------------------------------------------------------ CUDA graph
  def capture_step(self, table16, B, mine=False):
    """Capture one full optimisation step (gather -> fwd -> [mining] -> loss -> bwd -> [all-reduce] -> Adam) in a CUDA
    graph and return `replay(idx) -> stats`: `idx` [B,3] int64 (device or pinned host) is copied into the graph's static
    index buffer, then ONE graph launch replaces the ~30 kernel launches of the step (the host launch phase, ~0.35 ms,
    is what bounds small batches such as config 1's B=1024).  With N>1 ranks the NCCL all-reduce of the flat gradient
    buffer is captured inside the graph (every rank must call capture_step / replay the same number of times);
    CDML_DDP_GRAPH=0 keeps data-parallel steps eager."""
    if self.world > 1 and os.environ.get("CDML_DDP_GRAPH", "1") == "0":
      raise RuntimeError("capture_step disabled for data-parallel runs (CDML_DDP_GRAPH=0)")
    # warm-up triplets with distinct guids per row: a degenerate batch (one guid everywhere) drives the mining
    # epilogue through its re-scan on every chunk (measured 21 ms per scan instead of 2)
    G = self._table_rows(table16)
    ar = torch.arange(B, dtype=torch.int64, device=self.device)
    static_idx = torch.stack([(3 * ar) % G, (3 * ar + 1) % G, (3 * ar + 2) % G], dim=1).contiguous()
    snap = (self.w.clone(), self.m.clone(), self.v.clone(), self.step_counter.clone())   # warm-up must not train
    side = torch.cuda.Stream(device=self.device)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                      # warm-up on the capture stream: buffers, scratch, smem attributes
      for _ in range(2):
        self.train_step_indices(table16, static_idx, mine=mine)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    if self.world > 1:
      torch.distributed.barrier(group=self.pg)
    graph = torch.cuda.CUDAGraph()
    launches0 = ops.launch_count()
    # thread_local: NCCL's watchdog thread may touch the CUDA API while this thread captures
    with torch.cuda.graph(graph, capture_error_mode="thread_local" if self.world > 1 else "global"):
      stats = self.train_step_indices(table16, static_idx, mine=mine)
    launches_per_step = ops.launch_count() - launches0
    ops._count(-launches_per_step)                     # nothing ran during capture
    self.w.copy_(snap[0]), self.m.copy_(snap[1]), self.v.copy_(snap[2]), self.step_counter.copy_(snap[3])
    self.refresh_shadows()
    torch.cuda.synchronize()
    # the graph replays raw pointers: pin the training buffers (activations, dz, G, partials, loss) and the workspaces
    self._pinned_bufs.add((3 * B, True))
    self._graph_keepalive = (graph, static_idx, stats, self._bufs[(3 * B, True)])

    def replay(idx):
      static_idx.copy_(idx, non_blocking=True)
      graph.replay()
      ops._count(launches_per_step)                    # kernels of libcdml inside one replay
      return stats
    replay.launches_per_step = launches_per_step
    return replay

  # loss only (no update) -- used by tests and by the summaries of train.py
  def loss_rows(self, x16, B):
    buf = self.forward_rows(x16, 3 * B, train=True)
    ops.triplet_hinge(buf["e"], B, self.margin, out=buf["loss"])
    return buf
