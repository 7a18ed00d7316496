"""Bit-exact tests of the tcgen05 GEMM family (cdml_gemm16) on every dispatch route, and of its row helpers
(cdml_sum_partials, cdml_colsum16).

Method: 16-bit operands are small integers, |a|, |b| <= r.  Every product is exact in fp32, and r is chosen per case so
that K * r^2 < 2^21: every partial sum is an integer the fp32 accumulator holds exactly.  The accumulator must then
equal the float64 product bit for bit, whatever the split, the k-block order or the TMA zero fill of a tail.  The
epilogues are single IEEE operations in float32 -- x = f32(acc) + bias, x > 0 ? x : alpha * x, a round-to-nearest cast to
fp16 / bf16, acc * (bit ? 1 : alpha) -- and the reference applies the same operations with torch, so every output element
is compared bit for bit, with the production alpha = 0.2.  Only the sign of an exact-zero accumulator is left open
where no bias is added (the tensor core does not promise IEEE signed-zero rules): there +0 and -0 compare equal.
L2NORM uses rsqrtf: e and rinv are held to 4 fp32 ulp of the float64 value and the 16-bit copy to 1 ulp of the
round-to-nearest of the float64 e.  Those cases use alpha = 0.25 and sparse ternary operands, so that y^2 is exact and
the row sum of squares is nearly always exact too (|y| is a few tens, the sum stays far below 2^20 in units of 1/16);
the 4-ulp bound does not rely on it.

Every case also poisons what the kernels must not read and guards what they must not write:
  * the pitch padding of A and B and the rows past their logical extent hold NaN, so a tensor map that reads past its
    extent turns results into NaN.  The forward cases with K = 1500 have NaN in column F = 1500, where the training
    table keeps its ones column (DESIGN section 3); the forward's tensor map must not reach it.
  * outputs have extra rows, pitch padding, extra mask words (pitch > M) and unused split-K partial slots, all holding a
    sentinel that must survive.  The bias vector is followed by NaN.
  * acc + bias holds exact zeros (a zero row of A against zero bias columns) and exact cancellations (the bias of some
    columns is minus the accumulator of the last row): leaky(+0) = +0 and the sign-mask bit there is 0.
  * mask bits of columns >= N in the last word are 0.
  * a second call gives bit-identical buffers (the split-K reduction has a fixed order).

The sign-mask contract (include/cdml.h): a bit is set iff acc + bias > 0 in fp32.  MASK_LEAKY instead tests the stored
16-bit activation, and the two differ in one band: pre-activations in (0, 2^-25] round to +0 in fp16 (in bf16 the band
is (0, 2^-134], fp32 subnormals).  There the bit is 1, so MASK_BITS multiplies the data gradient by 1 where MASK_LEAKY
multiplies it by alpha.  test_sign_mask_band_between_mask_bits_and_mask_leaky pins both.

Cases with M or K = 196 608 draw their rows from a pool of a few thousand distinct rows, so the float64 reference is a
product of the pool; the kernels cannot know that rows repeat.

route() restates the dispatch rules of gemm_ops.cu / gemm_launch.cuh, and test_routes_match_the_dispatcher checks each
case's kernel, and for resident-B MASK_BITS its store path ("gemm_resb[tma]"), against the CDML_TRACE log of a child
process:
  resident-B (gemm_resb)    layout (0,0), one split, K <= 256, M >= 1024; MASK_BITS stores through TMA iff
                            ld_out % 8 == 0 and N % 8 == 0, else staged
  CTA pair (gemm2_tcgen05)  otherwise, if M >= 256 and a split has >= 8 k-blocks
  generic (gemm_tcgen05)    everything else
"""
import math
import os
import re
import subprocess
import sys
import zlib
from dataclasses import dataclass

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

STORE_F32, STORE_16, L2NORM, MASK_LEAKY, MASK_BITS = 0, 1, 2, 3, 4
KBM, KBK = 128, 64
ALPHA = 0.2
T16 = {"f16": torch.float16, "bf16": torch.bfloat16}
SENT16, SENT32 = 0x7E5A, 0x7FC5A5A5   # NaN payloads no kernel writes
CHUNK = 32768                         # rows per step of the large reference computations


@pytest.fixture(scope="module")
def cd():
  import __graft_entry__ as graft
  graft.build()
  return _env()


def _env():
  import cdml_b200  # noqa: F401
  from cdml_b200 import ops
  torch.cuda.set_device(0)

  class NS:
    pass
  ns = NS()
  ns.ops = ops
  ns.dev = torch.device("cuda:0")
  return ns


def cdiv(a, b):
  return -(-a // b)


# ---------------------------------------------------------------- the dispatch rules
def route(layout, M, N, K, splits=1, epilogue=STORE_F32):
  """Kernel that cdml_gemm16 launches (splits: the resolved request; epilogues other than STORE_F32 never split)."""
  if epilogue != STORE_F32:
    splits = 1
  if tuple(layout) == (0, 0) and splits <= 1 and K <= 4 * KBK and M >= 8 * KBM:
    return "gemm_resb"
  kb_per = cdiv(cdiv(K, KBK), max(splits, 1))
  if M >= 2 * KBM and kb_per >= 8:
    return "gemm2_tcgen05"
  return "gemm_tcgen05"


def traced_name(c, splits):
  """The CDML_TRACE name of case c's launch: the kernel, with "[tma]" when MASK_BITS stores through TMA."""
  k = route(c.layout, c.M, c.N, c.K, splits, c.epilogue)
  tma = k == "gemm_resb" and c.epilogue == MASK_BITS and c.out_ld() % 8 == 0 and c.N % 8 == 0
  return k + ("[tma]" if tma else "")


def splits_used(kernel, K, splits):
  """Split count the launcher reports: the request clamped to [1, k-blocks], then every split owns >= 1 k-block."""
  if kernel == "gemm_resb":
    return 1
  nkb = cdiv(K, KBK)
  per = cdiv(nkb, max(1, min(splits, nkb)))
  return cdiv(nkb, per)


# ---------------------------------------------------------------- the case table
@dataclass
class Case:
  kind: str            # fwd16 | fwd32 | l2norm | dgrad | wgrad
  M: int
  N: int
  K: int
  dt: str = "f16"
  epi: int = STORE_16
  mask: bool = False   # fwd16: write the packed sign mask
  bias: bool = True
  ld: str = "pad"      # output pitch: "pad" (multiple of 8 elements, + 8) or "odd" (N + 1 or N + 3: no vector / TMA stores)
  splits: int = 1      # wgrad: requested splits, 0 = automatic
  pool: int = 0        # rows of A (fwd / dgrad) or K rows (wgrad) drawn from this many distinct rows
  sub: bool = False    # A = integers * 2^-24: fp16 subnormal operands

  @property
  def layout(self):
    return {"fwd16": (0, 1), "fwd32": (0, 1), "l2norm": (0, 1), "dgrad": (0, 0), "wgrad": (1, 1)}[self.kind]

  @property
  def epilogue(self):
    return {"fwd16": STORE_16, "fwd32": STORE_F32, "l2norm": L2NORM, "wgrad": STORE_F32}.get(self.kind, self.epi)

  @property
  def id(self):
    epi = {STORE_16: "store16", MASK_LEAKY: "leaky", MASK_BITS: "bits"}[self.epi] if self.kind == "dgrad" else ""
    tags = [self.kind + ("_" + epi if epi else ""), "%dx%dx%d" % (self.M, self.N, self.K), self.dt]
    tags += (["mask"] if self.mask else []) + ([] if self.bias else ["nobias"]) + (["ld_odd"] if self.ld == "odd" else [])
    tags += (["S%d" % self.splits] if self.kind == "wgrad" else []) + (["sub"] if self.sub else [])
    return "-".join(tags)

  def out_ld(self):
    if self.ld == "odd":
      return self.N + 1 if (self.N + 1) % 8 else self.N + 3
    return cdiv(self.N, 8) * 8 + 8


C = Case
CASES = [
    # forward, layout (0,1): STORE_16 (+ sign mask) on generic and CTA-pair; the production layer 1 once
    C("fwd16", 196608, 5000, 1500, mask=True, pool=2048),
    C("fwd16", 1, 8, 8, mask=True),
    C("fwd16", 31, 200, 100, ld="odd"),
    C("fwd16", 255, 257, 1500, mask=True),
    C("fwd16", 257, 257, 1500, mask=True),
    C("fwd16", 513, 5000, 1500, mask=True),          # the last pair tile has one row
    C("fwd16", 513, 200, 100),
    C("fwd16", 257, 8, 1500, ld="odd"),
    C("fwd16", 1041, 257, 8, mask=True),
    C("fwd16", 513, 257, 1500, dt="bf16", mask=True),
    C("fwd16", 255, 200, 100, dt="bf16", mask=True),
    # STORE_F32 with bias and alpha, no split; fp16 subnormal operands
    C("fwd32", 257, 200, 1500),
    C("fwd32", 100, 257, 100, ld="odd"),
    C("fwd32", 513, 256, 640, dt="bf16"),
    C("fwd32", 60, 100, 64, dt="bf16"),
    C("fwd32", 257, 200, 1500, bias=False, sub=True),
    C("fwd32", 100, 257, 100, bias=False, sub=True),
    # L2NORM: CTA pair (K = 5000) and generic; without bias rows 0 and M-1 are zero rows
    C("l2norm", 513, 256, 5000),
    C("l2norm", 300, 200, 5000, bias=False, ld="odd"),
    C("l2norm", 257, 128, 100),
    C("l2norm", 100, 256, 1500, bias=False),
    C("l2norm", 513, 200, 5000, dt="bf16"),
    C("l2norm", 100, 128, 64, dt="bf16", bias=False, ld="odd"),
    # data gradient, layout (0,0), MASK_BITS: resident-B with TMA stores on the ragged N that give a warp an odd number
    # of boxes in the last column block (N mod 256 = 136, 24, 80, 200) and even ones (128), many row tiles per CTA.
    # N % 8 != 0 (785, 1500: the fusion towers) takes the staged stores.
    C("dgrad", 196608, 5000, 256, epi=MASK_BITS, pool=4096),
    C("dgrad", 196608, 1500, 256, epi=MASK_BITS, pool=4096),
    C("dgrad", 5137, 280, 256, epi=MASK_BITS),
    C("dgrad", 5137, 785, 200, epi=MASK_BITS),
    C("dgrad", 9233, 592, 64, epi=MASK_BITS),
    C("dgrad", 5137, 392, 256, epi=MASK_BITS),
    C("dgrad", 5137, 1224, 200, epi=MASK_BITS),
    C("dgrad", 5137, 128, 64, epi=MASK_BITS),
    # ... resident-B with staged stores, generic (M < 1024), CTA pair (K = 2048, the wide tower)
    C("dgrad", 5137, 392, 200, epi=MASK_BITS, ld="odd"),
    C("dgrad", 20497, 5000, 256, epi=MASK_BITS, ld="odd", pool=4096),
    C("dgrad", 1000, 392, 256, epi=MASK_BITS),
    C("dgrad", 255, 200, 64, epi=MASK_BITS),
    C("dgrad", 1, 17, 8, epi=MASK_BITS),
    C("dgrad", 1537, 2048, 2048, epi=MASK_BITS),
    C("dgrad", 513, 1500, 2048, epi=MASK_BITS),
    C("dgrad", 5137, 1224, 256, dt="bf16", epi=MASK_BITS),
    C("dgrad", 5137, 392, 200, dt="bf16", epi=MASK_BITS, ld="odd"),
    C("dgrad", 1000, 200, 256, dt="bf16", epi=MASK_BITS),
    C("dgrad", 513, 1500, 2048, dt="bf16", epi=MASK_BITS),
    C("dgrad", 5137, 392, 256, epi=MASK_BITS, sub=True),
    # MASK_LEAKY and the unmasked STORE_16 data gradient of the fusion towers
    C("dgrad", 5137, 392, 200, epi=MASK_LEAKY),
    C("dgrad", 1000, 200, 256, epi=MASK_LEAKY),
    C("dgrad", 513, 1500, 2048, epi=MASK_LEAKY),
    C("dgrad", 5137, 1224, 256, dt="bf16", epi=MASK_LEAKY),
    C("dgrad", 5137, 1500, 256, epi=STORE_16, bias=False),
    C("dgrad", 300, 200, 256, epi=STORE_16, bias=False, ld="odd"),
    C("dgrad", 513, 1500, 1024, epi=STORE_16, bias=False),
    C("dgrad", 5137, 785, 200, dt="bf16", epi=STORE_16, bias=False),
    # weight gradient, layout (1,1): STORE_F32 split-K partials, then sum_partials
    C("wgrad", 1501, 5000, 196608, splits=0, pool=512),
    C("wgrad", 257, 256, 196608, splits=0, pool=512),
    C("wgrad", 2049, 2048, 768, splits=0),
    C("wgrad", 65, 256, 1536, splits=0),
    C("wgrad", 300, 256, 640, splits=6),               # 10 k-blocks, 6 requested -> 5
    C("wgrad", 300, 256, 640, splits=1),
    C("wgrad", 65, 100, 200, splits=9),                # more splits than k-blocks -> 4
    C("wgrad", 300, 256, 4096, dt="bf16", splits=4),
    C("wgrad", 65, 256, 1536, dt="bf16", splits=3),
]


# ---------------------------------------------------------------- operands, outputs, references
class Opnd:
  """A 16-bit operand view [rows, cols] of a NaN-filled buffer with extra rows and pitch padding, and the exact values
  it holds: float64 `vals` [P, cols], row i of the view = vals[idx[i]] (idx None: vals itself)."""

  def __init__(self, rows, cols, t16, gen, dev, r=1, pool=0, idx=None, density=1.0, scale=1.0, vals=None):
    pitch = cdiv(cols, 8) * 8 + 8
    self.buf = torch.full((rows + 3, pitch), float("nan"), dtype=t16, device=dev)
    P = pool if (pool or idx is not None) else rows
    if vals is None:
      vals = torch.randint(-r, r + 1, (P, cols), generator=gen, device=dev).double()
      if density < 1.0:
        vals = torch.where(torch.rand((P, cols), generator=gen, device=dev) < density, vals, torch.zeros_like(vals))
      vals = vals * scale
    if idx is None and pool:
      idx = torch.randint(0, P, (rows,), generator=gen, device=dev)
    self.vals, self.idx = vals, idx
    for r0 in range(0, rows, CHUNK):
      r1 = min(rows, r0 + CHUNK)
      self.buf[r0:r1, :cols] = (vals[r0:r1] if idx is None else vals[idx[r0:r1]]).to(t16)
    self.t = self.buf[:rows, :cols]

  def zero_row(self, i):
    """Make logical row i all zeros (a pooled operand points it at a zeroed pool row)."""
    if self.idx is None:
      self.vals[i] = 0
    else:
      self.vals[0] = 0
      self.idx[i] = 0
      self.buf[(self.idx == 0).nonzero().flatten(), :self.t.shape[1]] = 0
    self.buf[i, :self.t.shape[1]] = 0

  def full(self):
    return self.vals if self.idx is None else self.vals[self.idx]


def bits(t):
  return t.view(torch.int16) if t.element_size() == 2 else t.view(torch.int32)


def sentinel_buf(shape, dtype, dev):
  b = torch.empty(shape, dtype=dtype, device=dev)
  bits(b).fill_(SENT16 if b.element_size() == 2 else SENT32)
  return b


def canon(b):
  """Bit patterns with -0 mapped to +0."""
  neg0 = -32768 if b.dtype == torch.int16 else -2 ** 31
  return torch.where(b == neg0, torch.zeros_like(b), b)


def assert_bits_equal(got, want, what, zero_sign=True):
  g, w = bits(got), bits(want)
  if not zero_sign:
    g, w = canon(g), canon(w)
  if torch.equal(g, w):
    return
  bad = (g != w).nonzero()
  i = tuple(bad[0].tolist())
  raise AssertionError("%s: %d of %d elements differ; first at %s: got %r (0x%x) want %r (0x%x)" % (
      what, bad.shape[0], g.numel(), i, float(got[i]), int(g[i]) & 0xFFFFFFFF, float(want[i]), int(w[i]) & 0xFFFFFFFF))


def assert_untouched(buf, M, N, what):
  """Everything outside [:M, :N] of a 2-D output still holds the sentinel."""
  b = bits(buf)
  s = SENT16 if b.dtype == torch.int16 else SENT32
  assert bool((b[:M, N:] == s).all()), "%s: written in the pitch padding (columns >= N)" % what
  assert bool((b[M:] == s).all()), "%s: written below row M" % what


def leaky32(x, alpha):
  return torch.where(x > 0, x, x * torch.tensor(alpha, dtype=torch.float32, device=x.device))


def gathered(rows_val, idx):
  return rows_val if idx is None else rows_val[idx]


def pack_bits(pos):
  """bool [M, N] -> int32 words [ceil(N/32), M], bit j of word [c][m] <-> column 32c + j (the STORE_16 sign mask)."""
  M, N = pos.shape
  nw = cdiv(N, 32)
  out = torch.empty((nw, M), dtype=torch.int32, device=pos.device)
  sh = torch.arange(32, dtype=torch.int64, device=pos.device)
  for r0 in range(0, M, CHUNK):
    p = torch.zeros((min(M, r0 + CHUNK) - r0, nw * 32), dtype=torch.int64, device=pos.device)
    p[:, :N] = pos[r0:r0 + CHUNK]
    w = (p.view(-1, nw, 32) << sh).sum(-1)
    out[:, r0:r0 + CHUNK] = torch.where(w >= 2 ** 31, w - 2 ** 32, w).to(torch.int32).T
  return out


def unpack_bits(words, M, N):
  """int32 words [>= ceil(N/32), >= M] -> bool [M, N]."""
  nw = cdiv(N, 32)
  out = torch.empty((M, N), dtype=torch.bool, device=words.device)
  sh = torch.arange(32, dtype=torch.int32, device=words.device)
  for r0 in range(0, M, CHUNK):
    w = words[:nw, r0:min(M, r0 + CHUNK)].T
    out[r0:r0 + CHUNK] = ((w.unsqueeze(-1) >> sh) & 1).reshape(w.shape[0], -1)[:, :N].bool()
  return out


def rmax(K, out16):
  """Operand bound r: |acc| <= K r^2 stays below 2^21 (exact fp32 partial sums) or, for 16-bit outputs, 2^15."""
  return max(1, min(8, math.isqrt((2 ** 15 if out16 else 2 ** 21) // K)))


def ulp32(v):
  """fp32 ulp at |v| (v float64), as float64."""
  a = v.abs().float()
  return (torch.nextafter(a, torch.full_like(a, float("inf"))) - a).double()


def ordered16(b):
  """16-bit patterns -> integers that are consecutive for adjacent values (+0 and -0 both 0)."""
  b = b.to(torch.int32)
  return torch.where(b < 0, -(b & 0x7FFF), b)


# ---------------------------------------------------------------- one case: build, launch, check
def prepare(cd, c, seed_extra=0):
  dev, t16 = cd.dev, T16[c.dt]
  gen = torch.Generator(device=dev)
  gen.manual_seed(zlib.crc32(c.id.encode()) + seed_extra)
  st = {}
  M, N, K = c.M, c.N, c.K
  out16 = c.kind in ("fwd16", "dgrad")
  r = rmax(K, out16)
  if c.kind == "wgrad":
    idx = torch.randint(0, c.pool, (K,), generator=gen, device=dev) if c.pool else None
    st["A"] = Opnd(K, M, t16, gen, dev, r=r, pool=c.pool, idx=idx)         # [K, M]: MN-major A
    st["B"] = Opnd(K, N, t16, gen, dev, r=r, pool=c.pool, idx=idx)         # [K, N]: MN-major B
    S = c.splits if c.splits > 0 else cd.ops.auto_splits(st["A"].t, M, N, K)
    st["S"] = S
    ld = c.out_ld()
    st["parts"] = sentinel_buf((S + 1, M + 2, ld), torch.float32, dev)
    st["final"] = sentinel_buf((M * ld + 8,), torch.float32, dev)
    return st
  if c.kind == "l2norm":
    st["A"] = Opnd(M, K, t16, gen, dev, r=1, density=0.5)
    st["B"] = Opnd(K, N, t16, gen, dev, r=1, density=0.5)
    st["A"].zero_row(0)
    st["A"].zero_row(M - 1)
  else:
    scale = 2.0 ** -24 if c.sub else 1.0
    st["A"] = Opnd(M, K, t16, gen, dev, r=r, pool=c.pool, scale=scale)    # [M, K]: K-major A
    shape_b = (K, N) if c.layout[1] == 1 else (N, K)
    st["B"] = Opnd(*shape_b, t16, gen, dev, r=r)
    if M > 1 and not c.sub:
      st["A"].zero_row(1)
  # accumulator of the distinct rows of A (pool rows or all rows): exact in float64
  Bnk = st["B"].vals if c.layout[1] == 0 else st["B"].vals.T                  # [N, K]
  st["acc_rows"] = st["A"].vals @ Bnk.T
  if c.kind in ("fwd16", "fwd32", "l2norm"):
    bias_buf = torch.full((N + 32,), float("nan"), dtype=torch.float32, device=dev)
    if c.bias:
      rb = 4 if c.kind == "l2norm" else 8
      b = torch.randint(-rb, rb + 1, (N,), generator=gen, device=dev).double()
      j = torch.arange(N, device=dev)
      b[j % 5 == 0] = 0.0                                                    # with the zero row: acc + bias = +0
      if M > 2 and c.kind != "l2norm":
        last = st["A"].idx[M - 1] if st["A"].idx is not None else M - 1
        b = torch.where(j % 5 == 1, -st["acc_rows"][last] + 0.0, b)          # exact cancellation in row M-1 (+0, not -0)
      bias_buf[:N] = b.float()
      st["bias"] = bias_buf[:N]
    else:
      st["bias"] = None
  ld = c.out_ld()
  if c.kind == "fwd16":
    st["out"] = sentinel_buf((M + 3, ld), t16, dev)
    st["mask"] = sentinel_buf((cdiv(N, 32) + 1, M + 5), torch.int32, dev) if c.mask else None
  elif c.kind == "fwd32":
    st["out"] = sentinel_buf((M + 3, ld), torch.float32, dev)
  elif c.kind == "l2norm":
    st["out"] = sentinel_buf((M + 3, ld), torch.float32, dev)
    st["rinv"] = sentinel_buf((M + 8,), torch.float32, dev)
    st["e16"] = sentinel_buf((M + 3, ld if c.ld == "pad" else ld + 2), t16, dev)
  else:
    st["out"] = sentinel_buf((M + 3, ld), t16, dev)
    if c.epi == MASK_BITS:
      st["aux"] = torch.randint(-2 ** 31, 2 ** 31, (cdiv(N, 32) + 1, M + 5), generator=gen, device=dev,
                                dtype=torch.int64).to(torch.int32)            # bits past N and past M are garbage
    elif c.epi == MASK_LEAKY:
      H = torch.full((M + 3, cdiv(N, 8) * 8 + 8), float("nan"), dtype=t16, device=dev)
      choice = torch.tensor([-2.0, -0.0, 0.0, 1.0, 2.0 ** -24, -(2.0 ** -24), 0.5], device=dev).to(t16)
      H[:M, :N] = choice[torch.randint(0, choice.numel(), (M, N), generator=gen, device=dev)]
      st["aux"] = H
  return st


def launch(cd, c, st):
  ops = cd.ops
  A, B, M, N, K = st["A"].t, st["B"].t, c.M, c.N, c.K
  if c.kind == "wgrad":
    parts = st["parts"]
    return ops.gemm16(A, B, M, N, K, 1, 1, STORE_F32, parts[0], num_splits=c.splits,
                      split_stride=parts.stride(0), ld_out=parts.stride(1))
  if c.kind == "fwd16":
    return ops.gemm16(A, B, M, N, K, 0, 1, STORE_16, st["out"], bias=st["bias"], alpha=ALPHA, aux0=st["mask"])
  if c.kind == "fwd32":
    return ops.gemm16(A, B, M, N, K, 0, 1, STORE_F32, st["out"], bias=st["bias"], alpha=1.0 if c.sub else ALPHA)
  if c.kind == "l2norm":
    return ops.gemm16(A, B, M, N, K, 0, 1, L2NORM, st["out"], bias=st["bias"], alpha=0.25, aux0=st["rinv"],
                      aux1=st["e16"])
  if c.epi == STORE_16:
    return ops.gemm16(A, B, M, N, K, 0, 0, STORE_16, st["out"], alpha=1.0)
  return ops.gemm16(A, B, M, N, K, 0, 0, c.epi, st["out"], alpha=ALPHA, aux1=st["aux"])


def snapshot(c, st):
  keys = {"wgrad": ("parts", "final")}.get(c.kind, ("out", "mask", "rinv", "e16"))
  return {k: bits(st[k]).clone() for k in keys if st.get(k) is not None}


def check_wgrad(cd, c, st, used):
  M, N, K = c.M, c.N, c.K
  A, B = st["A"], st["B"]
  nkb = cdiv(K, KBK)
  per = cdiv(nkb, max(1, min(st["S"], nkb))) * KBK     # the launcher's k-blocks per split
  parts = st["parts"]
  for s in range(parts.shape[0]):
    what = "%s partial %d" % (c.id, s)
    if s >= used:
      assert bool((bits(parts[s]) == SENT32).all()), what + ": an unused partial slot was written"
      continue
    k0, k1 = s * per, min(K, (s + 1) * per)
    if A.idx is None:
      want = A.vals[k0:k1].T @ B.vals[k0:k1]
    else:
      cnt = torch.bincount(A.idx[k0:k1], minlength=A.vals.shape[0]).double()
      want = (A.vals * cnt[:, None]).T @ B.vals
    assert_bits_equal(parts[s, :M, :N], want.float(), what, zero_sign=False)
    assert_untouched(parts[s], M, N, what)
  ld = parts.stride(1)
  cd.ops.sum_partials(parts, used, parts.stride(0), M * ld, st["final"])
  torch.cuda.synchronize()
  if A.idx is None:
    want = A.vals.T @ B.vals
  else:
    want = (A.vals * torch.bincount(A.idx, minlength=A.vals.shape[0]).double()[:, None]).T @ B.vals
  assert_bits_equal(st["final"][:M * ld].view(M, ld)[:, :N], want.float(), c.id + " summed", zero_sign=False)
  assert bool((bits(st["final"][M * ld:]) == SENT32).all()), c.id + ": sum_partials wrote past n"


def check(cd, c, st, used):
  M, N = c.M, c.N
  kernel = route(c.layout, M, N, c.K, st.get("S", 1), c.epilogue)
  assert used == splits_used(kernel, c.K, st.get("S", 1)), "%s: splits_used %d" % (c.id, used)
  if c.kind == "wgrad":
    check_wgrad(cd, c, st, used)
    return
  t16 = T16[c.dt]
  idx = st["A"].idx
  acc_rows = st["acc_rows"].float()        # exact: |acc| < 2^21
  out = st["out"]
  if c.kind in ("fwd16", "fwd32"):
    x_rows = acc_rows + (st["bias"] if st["bias"] is not None else torch.zeros((N,), device=cd.dev))[None, :]
    y_rows = leaky32(x_rows, 1.0 if c.sub else ALPHA)
    want = gathered(y_rows.to(t16) if c.kind == "fwd16" else y_rows, idx)
    assert_bits_equal(out[:M, :N], want, c.id)
    assert_untouched(out, M, N, c.id)
    if c.kind == "fwd16" and st["mask"] is not None:
      nw = cdiv(N, 32)
      wm = pack_bits(gathered(x_rows > 0, idx))
      assert_bits_equal(st["mask"][:nw, :M], wm, c.id + " sign mask")        # includes: bits of columns >= N are 0
      assert bool((st["mask"][:nw, M:] == SENT32).all()), c.id + ": sign mask written past M"
      assert bool((st["mask"][nw:] == SENT32).all()), c.id + ": sign mask written past its last word"
    return
  if c.kind == "l2norm":
    bias = st["bias"] if st["bias"] is not None else torch.zeros((N,), device=cd.dev)
    y = leaky32(acc_rows + bias[None, :], 0.25).double()                     # exact: multiples of 1/4
    ss = (y * y).sum(1)                                                      # exact (< 2^20 in units of 1/16)
    rinv = 1.0 / torch.sqrt(torch.clamp(ss, min=float(torch.tensor(1e-12, dtype=torch.float32))))
    e = y * rinv[:, None]
    got_r = st["rinv"][:M].double()
    assert bool(((got_r - rinv).abs() <= 4 * ulp32(rinv)).all()), c.id + ": rinv beyond 4 ulp"
    assert bool((bits(st["rinv"][M:]) == SENT32).all()), c.id + ": rinv written past M"
    got_e = out[:M, :N].double()
    assert bool(((got_e - e).abs() <= 4 * ulp32(e)).all()), c.id + ": e beyond 4 ulp"
    assert bool((got_e[e == 0] == 0).all()), c.id + ": e of a zero activation is not 0"
    if not c.bias:
      assert bool((out[0, :N] == 0).all() and (out[M - 1, :N] == 0).all()), c.id + ": zero row"
    assert_untouched(out, M, N, c.id)
    d = (ordered16(bits(st["e16"][:M, :N])) - ordered16(bits(e.float().to(t16)))).abs()
    assert int(d.max()) <= 1, c.id + ": 16-bit e beyond 1 ulp of RN(e)"
    assert_untouched(st["e16"], M, N, c.id + " 16-bit e")
    return
  # data gradient
  acc = gathered(acc_rows, idx)
  if c.epi == STORE_16:
    want = acc.to(t16)
  else:
    pos = unpack_bits(st["aux"], M, N) if c.epi == MASK_BITS else st["aux"][:M, :N] > 0
    one = torch.ones((), dtype=torch.float32, device=cd.dev)
    want = (acc * torch.where(pos, one, torch.tensor(ALPHA, dtype=torch.float32, device=cd.dev))).to(t16)
  assert_bits_equal(out[:M, :N], want, c.id, zero_sign=False)
  assert_untouched(out, M, N, c.id)


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=[c.id for c in CASES])
def test_gemm16_bit_exact(cd, c):
  st = prepare(cd, c)
  used = launch(cd, c, st)
  torch.cuda.synchronize()
  check(cd, c, st, used)
  first = snapshot(c, st)
  assert launch(cd, c, st) == used
  if c.kind == "wgrad":
    cd.ops.sum_partials(st["parts"], used, st["parts"].stride(0), c.M * st["parts"].stride(1), st["final"])
  torch.cuda.synchronize()
  for k, v in snapshot(c, st).items():
    assert torch.equal(v, first[k]), "%s: a second call changed %s" % (c.id, k)


def test_case_table_covers_every_route_layout_and_epilogue():
  """Every route x layout x epilogue cell has an fp16 case and at least one bf16 case (automatic split counts depend
  on the SM count and are left out here; test_routes_match_the_dispatcher checks them)."""
  cells = set()
  for c in CASES:
    if c.kind == "wgrad" and c.splits == 0:
      continue
    k = route(c.layout, c.M, c.N, c.K, c.splits, c.epilogue)
    cells.add((k, c.layout, c.epilogue, c.dt))
    if c.epilogue == MASK_BITS and k == "gemm_resb":
      cells.add(("tma" if traced_name(c, 1).endswith("[tma]") else "staged", c.dt))
  for layout, epis in (((0, 1), (STORE_16, STORE_F32, L2NORM)), ((0, 0), (MASK_BITS, MASK_LEAKY, STORE_16)),
                       ((1, 1), (STORE_F32,))):
    for e in epis:
      kernels = ("gemm_tcgen05", "gemm2_tcgen05") + (("gemm_resb",) if layout == (0, 0) else ())
      for k in kernels:
        assert (k, layout, e, "f16") in cells, (k, layout, e)
      assert any((k, layout, e, "bf16") in cells for k in kernels), (layout, e)
  for dt in ("f16", "bf16"):
    assert ("tma", dt) in cells and ("staged", dt) in cells
  assert any(c.sub for c in CASES)


# ---------------------------------------------------------------- the dispatcher agrees with route()
def _trace_routes():
  """Child-process body: launch every case once with CDML_TRACE=1 and mark each case on stderr."""
  cd = _env()
  for c in CASES:
    st = prepare(cd, c)
    sys.stderr.write("CASE %s\n" % c.id)
    sys.stderr.flush()
    launch(cd, c, st)
    torch.cuda.synchronize()
    del st
  sys.stderr.write("DONE\n")


@pytest.mark.gpu
def test_routes_match_the_dispatcher(cd):
  env = dict(os.environ, CDML_TRACE="1")
  r = subprocess.run([sys.executable, os.path.abspath(__file__), "--trace-routes"], env=env, cwd=ROOT,
                     capture_output=True, text=True, timeout=900)
  assert r.returncode == 0 and "DONE" in r.stderr, r.stderr[-4000:]
  seen, cur = {}, None
  for line in r.stderr.splitlines():
    if line.startswith("CASE "):
      cur = line[5:].strip()
      seen[cur] = []
    m = re.match(r"\[cdml\] (\S+) M=(\d+) N=(\d+) K=(\d+) .*no error", line)
    if m and cur is not None:
      seen[cur].append((m.group(1), int(m.group(2)), int(m.group(3)), int(m.group(4))))
  ref = torch.empty((1,), device=cd.dev)
  for c in CASES:
    S = c.splits if c.splits > 0 else cd.ops.auto_splits(ref, c.M, c.N, c.K)
    want = traced_name(c, S)
    got = seen.get(c.id)
    assert got and len(got) == 1, "%s: traced launches %r" % (c.id, got)
    assert got[0] == (want, c.M, c.N, c.K), "%s: dispatched to %r, the table says %s" % (c.id, got[0], want)


# ---------------------------------------------------------------- the sign-mask band
@pytest.mark.gpu
def test_sign_mask_band_between_mask_bits_and_mask_leaky(cd):
  """z = acc + bias in (0, 2^-25]: the fp16 activation is +0 but the mask bit is 1."""
  ops, dev = cd.ops, cd.dev
  gen = torch.Generator(device=dev)
  gen.manual_seed(25)
  M, N, K, K2 = 1100, 70, 64, 64
  X = Opnd(M, K, torch.float16, gen, dev, r=3)
  W = Opnd(K, N, torch.float16, gen, dev, r=3)
  X.zero_row(0)
  band = torch.arange(N, device=dev) % 4 == 0
  bias = torch.where(band, torch.tensor(2.0 ** -26, device=dev), torch.tensor(-1.0, device=dev)).float()
  H = sentinel_buf((M, N + 2), torch.float16, dev)[:, :N]
  mask = sentinel_buf((cdiv(N, 32), M), torch.int32, dev)
  ops.gemm16(X.t, W.t, M, N, K, 0, 1, STORE_16, H, bias=bias, alpha=ALPHA, aux0=mask)
  torch.cuda.synchronize()
  bit0 = unpack_bits(mask, M, N)[0]
  assert bool((bits(H[0, band]) == 0).all()), "z = 2^-26 must store as +0 in fp16"
  assert bool(bit0[band].all()) and not bool(bit0[~band].any()), "mask bit = (acc + bias > 0) in fp32"
  # data gradient of the same layer: MASK_BITS scales by 1 there, MASK_LEAKY (reading H = +0) by alpha
  dz = Opnd(M, K2, torch.float16, gen, dev, r=3)
  Wb = Opnd(N, K2, torch.float16, gen, dev, r=3)
  acc0 = (dz.vals[0] @ Wb.vals.T).float()
  out_b = sentinel_buf((M, N + 2), torch.float16, dev)
  out_l = sentinel_buf((M, N + 2), torch.float16, dev)
  ops.gemm16(dz.t, Wb.t, M, N, K2, 0, 0, MASK_BITS, out_b, alpha=ALPHA, aux1=mask)
  ops.gemm16(dz.t, Wb.t, M, N, K2, 0, 0, MASK_LEAKY, out_l, alpha=ALPHA, aux1=H)
  torch.cuda.synchronize()
  a = torch.tensor(ALPHA, dtype=torch.float32, device=dev)
  assert_bits_equal(out_b[0, :N][band], acc0[band].half(), "MASK_BITS in the band", zero_sign=False)
  assert_bits_equal(out_l[0, :N][band], (acc0[band] * a).half(), "MASK_LEAKY in the band", zero_sign=False)
  assert_bits_equal(out_b[0, :N][~band], out_l[0, :N][~band], "outside the band", zero_sign=False)
  assert bool((out_b[0, :N][band] != out_l[0, :N][band]).any())


# ---------------------------------------------------------------- row helpers of the same path
@pytest.mark.gpu
@pytest.mark.parametrize("dt", ["f16", "bf16"])
@pytest.mark.parametrize("R,N,ld", [(1, 5000, "vec"), (3001, 257, "vec"), (3001, 67, "scalar"), (196608, 5000, "vec"),
                                    (196608, 1500, "scalar"), (3001, 1, "scalar")])
def test_colsum16_bit_exact(cd, dt, R, N, ld):
  ops, dev, t16 = cd.ops, cd.dev, T16[dt]
  gen = torch.Generator(device=dev)
  gen.manual_seed(R * 7 + N)
  pitch = cdiv(N, 8) * 8 + 8 if ld == "vec" else cdiv(N, 2) * 2 + 2      # scalar branch: even, not a multiple of 8
  pitch += 2 if ld == "scalar" and pitch % 8 == 0 else 0
  buf = torch.full((R + 2, pitch), float("nan"), dtype=t16, device=dev)
  vals = torch.randint(-8, 9, (R, N), generator=gen, device=dev)
  buf[:R, :N] = vals.to(t16)
  out = sentinel_buf((N + 8,), torch.float32, dev)
  ops.colsum16(buf[:R, :N], R, N, out)
  torch.cuda.synchronize()
  assert_bits_equal(out[:N], vals.sum(0).float(), "colsum16")                 # |sum| <= 8 R < 2^24: exact
  assert bool((bits(out[N:]) == SENT32).all()), "colsum16 wrote past N"


@pytest.mark.gpu
@pytest.mark.parametrize("dt", ["f16", "bf16"])
def test_colsum16_equals_the_ones_row_of_the_weight_gradient(cd, dt):
  """The bias gradient two ways: colsum16(dz) and row `in` of [x | 1]^T dz (the ones column of DESIGN section 3)."""
  ops, dev, t16 = cd.ops, cd.dev, T16[dt]
  gen = torch.Generator(device=dev)
  gen.manual_seed(3001)
  R, n_in, N = 3001, 100, 1500
  X = Opnd(R, n_in + 1, t16, gen, dev, r=4)
  X.buf[:R, n_in] = 1
  X.vals[:, n_in] = 1
  dz = Opnd(R, N, t16, gen, dev, r=4)
  S = ops.auto_splits(X.t, n_in + 1, N, R)
  parts = sentinel_buf((S, n_in + 1, N), torch.float32, dev)
  used = ops.gemm16(X.t, dz.t, n_in + 1, N, R, 1, 1, STORE_F32, parts[0], num_splits=S,
                    split_stride=parts.stride(0), ld_out=N)
  gW = torch.empty(((n_in + 1) * N,), dtype=torch.float32, device=dev)
  ops.sum_partials(parts, used, parts.stride(0), (n_in + 1) * N, gW)
  gb = torch.empty((N,), dtype=torch.float32, device=dev)
  ops.colsum16(dz.t, R, N, gb)
  torch.cuda.synchronize()
  assert_bits_equal(gW.view(n_in + 1, N)[n_in], gb, "ones row vs colsum16", zero_sign=False)
  assert_bits_equal(gb, dz.vals.sum(0).float(), "colsum16", zero_sign=False)


@pytest.mark.gpu
@pytest.mark.parametrize("branch,n,stride,offset", [("vec4", 4096, 4100, 0), ("vec4", 1_000_000, 1_000_000, 0),
                                                     ("scalar", 4097, 4100, 0), ("scalar", 4096, 4098, 0),
                                                     ("scalar", 4096, 4100, 1)])
@pytest.mark.parametrize("parts_n", [1, 3, 7])
@pytest.mark.parametrize("scale", [1.0, 0.2])
def test_sum_partials_fixed_order_and_scale(cd, branch, n, stride, offset, parts_n, scale):
  ops, dev = cd.ops, cd.dev
  gen = torch.Generator(device=dev)
  gen.manual_seed(n + stride + parts_n)
  base = sentinel_buf((offset + parts_n * stride + 8,), torch.float32, dev)
  vals = torch.randint(-1000, 1001, (parts_n, n), generator=gen, device=dev)
  view = base[offset:offset + parts_n * stride].view(parts_n, stride)
  view[:, :n] = vals.float()
  obuf = sentinel_buf((offset + n + 8,), torch.float32, dev)
  out = obuf[offset:offset + n]
  ops.sum_partials(view, parts_n, stride, n, out, scale=scale)
  torch.cuda.synchronize()
  want = vals.sum(0).float() * torch.tensor(scale, dtype=torch.float32, device=dev)   # exact sum, one rounding
  assert_bits_equal(out, want, "sum_partials %s" % branch)
  assert bool((bits(obuf[:offset]) == SENT32).all() and (bits(obuf[offset + n:]) == SENT32).all())


if __name__ == "__main__":
  if "--trace-routes" in sys.argv:
    _trace_routes()
