"""GPU parity tests: every kernel family called through the C ABI (ctypes) and compared with the CPU oracle on the
same seeded inputs.  Tolerances (north_star): gather / ids bit-exact (ids: except exact or sub-ulp distance ties);
embeddings and loss <= 1e-3 relative with fp16 operands + fp32 accumulation."""
import json
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import cdml_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cd():
  import __graft_entry__ as graft
  graft.build()
  import cdml_b200  # noqa: F401
  from cdml_b200 import engine, faiss_knn, inputs, losses, models, ops, predict, train
  torch.cuda.set_device(0)

  class NS:
    pass
  ns = NS()
  ns.engine, ns.faiss_knn, ns.inputs, ns.losses, ns.models, ns.ops, ns.predict, ns.train = \
      engine, faiss_knn, inputs, losses, models, ops, predict, train
  ns.dev = torch.device("cuda:0")
  return ns


def dev_t(cd, a):
  return torch.as_tensor(np.ascontiguousarray(a)).to(cd.dev)


def rel_rows(got, ref):
  return np.linalg.norm(got - ref, axis=1) / np.maximum(np.linalg.norm(ref, axis=1), 1e-30)


# ---------------------------------------------------------------- K1 gather
def test_gather_bit_exact_golden_and_random(cd, golden):
  out = cd.ops.gather_rows(dev_t(cd, golden["gather_features"]), dev_t(cd, golden["sampler_seed99_triplets"]))
  assert np.array_equal(out.cpu().numpy().reshape(8, 3, 12), golden["gather_out"])
  feats = O.synth_features(3000, 1500, 0)
  trip = O.synth_triplets(1024, 3000, 1)
  want = O.flatten_triplets(O.gather_rows(feats, trip))
  for idx in (trip, trip.astype(np.int32)):
    got = cd.ops.gather_rows(dev_t(cd, feats), dev_t(cd, idx))
    assert got.dtype == torch.float32 and np.array_equal(got.cpu().numpy(), want)
  # ragged widths, empty index, numpy-style negative wrap, out-of-range flag
  odd = O.synth_features(100, 7, 3)
  ii = np.array([-1, 0, 99, 5], np.int64)
  assert np.array_equal(cd.ops.gather_rows(dev_t(cd, odd), dev_t(cd, ii)).cpu().numpy(), odd[ii])
  assert cd.ops.gather_rows(dev_t(cd, odd), dev_t(cd, np.zeros((0,), np.int64))).shape == (0, 7)
  assert cd.ops.poll_errors(dev_t(cd, odd)) == 0
  cd.ops.gather_rows(dev_t(cd, odd), dev_t(cd, np.array([100], np.int64)))
  assert cd.ops.poll_errors(dev_t(cd, odd)) == 1


def test_mptripletpipe_get_batch_matches_numpy(cd, tmp_path):
  feats = O.synth_features(400, 1500, 0)
  np.save(tmp_path / "features.npy", feats)
  pairs = O.synth_pairs(300, 400, seed=9)
  with open(tmp_path / "a.train", "w") as f:
    f.writelines("%d,%d\n" % (a, p) for a, p in pairs)
  pipe = cd.inputs.MPTripletPipe(str(tmp_path / "*.train"), str(tmp_path / "features.npy"), seed=1)
  pipe.create_pipe(1, 128)
  ref = cd.inputs.MPTripletPipe(str(tmp_path / "*.train"), str(tmp_path / "features.npy"), seed=1)
  ref.create_pipe(1, 128)
  n = 0
  while True:
    batch = pipe.get_batch()
    idx = ref.get_batch_indices()
    if batch is None:
      assert idx is None
      break
    assert batch.shape == (128, 3, 1500) and batch.dtype == np.float32
    assert np.array_equal(batch, feats[idx])                       # FEATURES[np.asarray(guid_triplets)]
    n += 1
  assert n == 2


# ---------------------------------------------------------------- K5 loss
def test_hinge_loss_fixture_and_random(cd):
  fx = json.load(open(os.path.join(GOLDEN, "loss_fixture.json")))
  r = cd.losses.HingeLoss().calculate_loss(np.asarray(fx["triplets"], np.float32), margin=0.1)
  assert r["pos_dist"].shape == (5, 1) and r["anchors"].shape == (5, 1, 2)
  assert np.allclose(r["pos_dist"][:, 0], fx["pos_dist"]) and np.allclose(r["hinge_dist"][:, 0], fx["hinge_dist@0.1"])
  assert abs(float(r["hinge_loss"]) - 18.06) < 1e-5
  assert abs(float(cd.losses.HingeLoss().calculate_loss(np.asarray(fx["triplets"], np.float32), margin=0.8)["hinge_loss"]) - 18.48) < 1e-5
  E = O.l2_normalize(np.random.RandomState(0).standard_normal((4096, 3, 256))).astype(np.float32)
  want = O.hinge_loss(E, 0.8)
  got = cd.losses.HingeLoss().calculate_loss(dev_t(cd, E), margin=0.8)
  assert abs(float(got["hinge_loss"]) / want["hinge_loss"] - 1) < 1e-5
  assert np.allclose(got["hinge_dist"].cpu().numpy(), want["hinge_dist"], atol=1e-5)
  # gradient of the fused kernel == oracle gradient (mean reduction -> grad_scale 1/B)
  r = cd.ops.triplet_hinge(dev_t(cd, E.reshape(-1, 256)), 4096, 0.8, grad_scale=1.0 / 4096, want_dE=True)
  assert np.allclose(r["dE"].cpu().numpy(), O.hinge_loss_grad(E, 0.8).reshape(-1, 256), atol=1e-9)


@pytest.mark.parametrize("B", [4096, 3001])
def test_hinge_gradient_with_mined_negatives_is_exact_and_reproducible(cd, B):
  """Mined negatives alias rows: several triplets pick the same row, here up to 512 of them, on a row 3i+2 (no gradient of
  its own) and on a positive row.  The gradient equals the float64 sum, and is bit-identical from call to call (the sum
  over the triplets that picked a row must not depend on the order they are processed in) -- returned as dE, and in the
  training form, where it lands in the caller's workspace and only the fp16 dz of the L2-norm / leaky backward is kept."""
  D, margin, alpha = 256, 0.1, 0.2
  rs = np.random.RandomState(11)
  E = O.l2_normalize(rs.standard_normal((3 * B, D))).astype(np.float32)
  neg = (3 * rs.randint(0, B, B) + rs.randint(1, 3, B)).astype(np.int32)        # positives / negatives, as the miner picks
  neg[:512], neg[512:800] = 5, 7
  rinv = rs.uniform(0.5, 2.0, 3 * B).astype(np.float32)
  a, p, n = E[0::3].astype(np.float64), E[1::3].astype(np.float64), E[neg].astype(np.float64)
  h = np.maximum(((a - p) ** 2).sum(1) - ((a - n) ** 2).sum(1) + margin, 0.0)
  s = np.where(h > 0, 2.0, 0.0)[:, None]
  want = np.zeros((3 * B, D))
  want[0::3], want[1::3] = s * (n - p), s * (p - a)
  bound = np.abs(want)
  np.add.at(want, neg, s * (a - n))
  np.add.at(bound, neg, np.abs(s * (a - n)))
  E64 = E.astype(np.float64)
  want_dz = (want - E64 * (E64 * want).sum(1, keepdims=True)) * rinv[:, None] * np.where(E64 > 0, 1.0, alpha)
  Ed, nd, rd = dev_t(cd, E), dev_t(cd, neg), dev_t(cd, rinv)
  got = [cd.ops.triplet_hinge(Ed, B, margin, neg_row=nd, want_dE=True)["dE"].cpu().numpy() for _ in range(3)]
  assert 0.3 < (h > 0).mean() < 0.9                                                 # active and inactive triplets
  assert np.all(np.abs(got[0] - want) <= 1e-6 * bound + 1e-7)
  assert np.array_equal(got[0], got[1]) and np.array_equal(got[0], got[2])
  dz = []
  for _ in range(2):
    ws = torch.full((3 * B * D,), float("nan"), dtype=torch.float32, device=cd.dev)
    dz16 = torch.empty((3 * B, D), dtype=torch.float16, device=cd.dev)
    cd.ops.triplet_hinge(Ed, B, margin, neg_row=nd, rinv=rd, leaky_alpha=alpha, dz16=dz16, workspace=ws)
    assert np.array_equal(ws.view(3 * B, D).cpu().numpy(), got[0])
    dz.append(dz16.float().cpu().numpy())
  assert np.array_equal(dz[0], dz[1])
  live = np.abs(want_dz).sum(1) > 0
  assert rel_rows(dz[0][live], want_dz[live]).max() < 2e-3                           # fp16 output


# ---------------------------------------------------------------- K2-K4 forward
@pytest.mark.parametrize("dims,rows", [([1500, 5000, 256], 3 * 171), ([64, 128, 256], 3 * 50), ([2048, 2048, 2048, 2048, 256], 3 * 64)])
def test_tower_forward_embeddings_within_1e3(cd, dims, rows):
  feats = O.synth_features(rows, dims[0], 7)
  params = O.init_tower(dims, seed=2)
  eng = cd.engine.TowerEngine(dims, device=cd.dev, init_params=params)
  e = eng.embed(dev_t(cd, feats)).cpu().numpy()
  want = O.tower_forward(feats, params)["l2_norm"]
  assert e.shape == (rows, dims[-1])
  assert np.allclose(np.linalg.norm(e, axis=1), 1.0, atol=1e-5)
  assert rel_rows(e, want).max() < 1e-3                          # fp16 operands, fp32 accumulate: stated tolerance 1e-3


@pytest.mark.parametrize("t16", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("R,N,K", [(1200, 5000, 256), (300, 200, 256), (2100, 333 * 8, 128)])
def test_sign_mask_forward_and_mask_bits_data_gradient(cd, t16, R, N, K):
  """The packed sign mask (STORE_16 aux0) is exactly `activation > 0`, bit for bit, and the MASK_BITS data gradient equals
  the MASK_LEAKY one (which reads the 16-bit activation) bit for bit -- on the resident-B kernel (R >= 1024) and the
  generic one, ragged N, both operand types.  (mask == (H > 0) only outside the band where a positive pre-activation rounds
  to a 16-bit +0, (0, 2^-25] in fp16; these random inputs do not reach it, test_gemm_exact.py covers it.)"""
  from cdml_b200._lib import EPI_MASK_BITS, EPI_MASK_LEAKY, EPI_STORE_16
  gen = torch.Generator(device=cd.dev)
  gen.manual_seed(R + N)
  pad = lambda n: (n + 63) // 64 * 64
  X = (torch.randn((R, pad(K)), generator=gen, device=cd.dev) * 0.3).to(t16)[:, :K]
  W = (torch.randn((K, pad(N)), generator=gen, device=cd.dev) * 0.2).to(t16)[:, :N]          # [K,N]: MN-major B of the forward
  bias = torch.randn((N,), generator=gen, device=cd.dev) * 0.1
  H = torch.zeros((R, pad(N)), dtype=t16, device=cd.dev)[:, :N]
  mask = cd.ops.sign_mask_buffer(R, N, cd.dev)
  mask.fill_(-1)
  cd.ops.gemm16(X, W, R, N, K, 0, 1, EPI_STORE_16, H, bias=bias, alpha=0.2, aux0=mask)
  bits = (H > 0).cpu().numpy()
  want = np.zeros(((N + 31) // 32, R), np.uint32)
  for j in range(N):
    want[j // 32] |= bits[:, j].astype(np.uint32) << np.uint32(j % 32)
  got = mask.cpu().numpy().view(np.uint32)
  tail = N % 32
  if tail:                                                 # bits beyond N in the last word: columns that do not exist
    got[-1] &= np.uint32((1 << tail) - 1)
  assert np.array_equal(got, want)
  # backward: dY [R,N] . W2^T with W2 = [N2,N] K-major... here: dz [R,K2] x Wb [N,K2]^T -> [R,N], masked by H's sign
  K2 = 256
  dz = (torch.randn((R, K2), generator=gen, device=cd.dev) * 0.1).to(t16)
  Wb = (torch.randn((N, K2), generator=gen, device=cd.dev) * 0.1).to(t16)
  out_a = torch.zeros((R, pad(N)), dtype=t16, device=cd.dev)[:, :N]
  out_b = torch.zeros((R, pad(N)), dtype=t16, device=cd.dev)[:, :N]
  cd.ops.gemm16(dz, Wb, R, N, K2, 0, 0, EPI_MASK_LEAKY, out_a, alpha=0.2, aux1=H)
  cd.ops.gemm16(dz, Wb, R, N, K2, 0, 0, EPI_MASK_BITS, out_b, alpha=0.2, aux1=mask)
  assert torch.equal(out_a, out_b)
  ref = (dz.double() @ Wb.double().T) * torch.where(H > 0, 1.0, 0.2)
  assert float((out_b.double() - ref).abs().max().item()) < 2e-2 * float(ref.abs().max().item())


# bf16 operands (configs[2]; `--compute_dtype bf16`).  Stated tolerances, measured on B200 (profiles/r02_pytest_gpu.log):
#   * against the bf16 PRECISION MODEL (float64 arithmetic, operands rounded to bf16 exactly where the kernels store them --
#     "the reference computing in bf16"): median row error ~3e-5, worst row 1.0e-3 (VNet) / 1.5e-3 (4-layer wide tower).
#     The worst rows are rounding-boundary flips: a stored activation the model rounds up and the fp32-accumulating tensor
#     core rounds down differs by one bf16 ulp = 3.9e-3 of its value.  Gate: median <= 3e-4, max <= 2.5e-3.
#   * bf16 itself against the unrounded float64 oracle is an 8-bit-significand property (2^-9 per operand, ~sqrt(layers)
#     growth): measured 3.0-3.9e-3, gate 8e-3 -- OUTSIDE north_star's 1e-3, which bf16 operands cannot meet on this tower.
#     fp16 operands (the default; TF32's significand) meet 1e-3 against float64 directly at the same tensor-core rate.
BF16_VS_F64 = 8e-3
BF16_VS_MODEL_MAX, BF16_VS_MODEL_MEDIAN = 2.5e-3, 3e-4


@pytest.mark.parametrize("dims,rows", [([1500, 5000, 256], 3 * 171), ([2048, 2048, 2048, 2048, 256], 3 * 64)])
def test_tower_forward_bf16_matches_precision_model(cd, dims, rows):
  from cdml_b200 import _lib
  feats = O.synth_features(rows, dims[0], 7)
  params = O.init_tower(dims, seed=2, bias_init=0.1 if len(dims) > 3 else 0.0)
  eng = cd.engine.TowerEngine(dims, device=cd.dev, init_params=params, dtype16=_lib.BF16)
  e = eng.embed(dev_t(cd, feats)).cpu().numpy()
  model = O.tower_grads_emulated16(feats, params, 0.8, "bf16")["l2_norm"]
  want = O.tower_forward(feats, params)["l2_norm"]
  assert np.allclose(np.linalg.norm(e, axis=1), 1.0, atol=1e-5)
  print("bf16 forward %s: vs model %.2e, vs float64 %.2e" % (dims, rel_rows(e, model).max(), rel_rows(e, want).max()))
  assert rel_rows(e, model).max() < BF16_VS_MODEL_MAX and np.median(rel_rows(e, model)) < BF16_VS_MODEL_MEDIAN
  assert rel_rows(e, want).max() < BF16_VS_F64


@pytest.mark.parametrize("dims,G,B", [([1500, 5000, 256], 2000, 512), ([2048, 2048, 2048, 2048, 256], 1500, 256)])
def test_training_step_bf16_loss_gradients_and_adam(cd, dims, G, B):
  """One optimisation step + a 6-step loss curve in bf16 against the bf16 precision model (and float64 at the stated
  bf16 tolerance): the wide tower of configs[2] and the default tower with `dtype16=BF16`."""
  from cdml_b200 import _lib
  F, L = dims[0], len(dims) - 1
  feats = O.synth_features(G, F, 0)
  trip = O.synth_triplets(B, G, 1)
  params = O.init_tower(dims, seed=2, bias_init=0.1 if L > 2 else 0.0)
  eng = cd.engine.TowerEngine(dims, device=cd.dev, base_lr=1e-3, margin=0.8, init_params=params, dtype16=_lib.BF16)
  table16 = eng.prepare_table(dev_t(cd, feats))
  assert table16.dtype == torch.bfloat16
  x = O.flatten_triplets(O.gather_rows(feats, trip))
  tr16 = O.OracleTrainer(params, lr=1e-3, margin=0.8, emulate16="bf16")
  tr64 = O.OracleTrainer(params, lr=1e-3, margin=0.8)
  _, loss16, grads16 = tr16.loss_and_grads(x)
  _, loss64, grads64 = tr64.loss_and_grads(x)
  s = eng.train_step_indices(table16, dev_t(cd, trip)).cpu().numpy()
  print("bf16 step %s: loss gpu %.6f model %.6f f64 %.6f" % (dims, s[0], loss16["hinge_loss"], loss64["hinge_loss"]))
  assert abs(s[0] / loss16["hinge_loss"] - 1) < 1e-3
  assert abs(s[0] / loss64["hinge_loss"] - 1) < BF16_VS_F64
  for l in range(L):
    gW, gb = eng.gW[l].cpu().numpy() / B, eng.gb[l].cpu().numpy() / B
    rW, rb = _grad_rel(gW, grads16[l][0]), _grad_rel(gb, grads16[l][1])
    dW_model, db_model = _grad_rel(grads16[l][0], grads64[l][0]), _grad_rel(grads16[l][1], grads64[l][1])
    print("  layer %d: dW vs model %.2e, db vs model %.2e   (bf16 model vs float64: dW %.2e, db %.2e)" % (l, rW, rb, dW_model, db_model))
    # rounding-boundary flips of stored activations / dz (a value the model rounds up and the kernel down, one bf16 ulp
    # apart) are amplified like every forward error by the differences of nearly equal embeddings; the kernels are another
    # realisation of the same rounding, gated (like the fusion towers) at 1e-2 + the model's own distance from float64
    assert rW < 1e-2 + dW_model and rb < 1e-2 + db_model, (l, rW, rb, dW_model, db_model)
  tr16.step(x)
  lg, lm = [], []
  for t in range(2, 7):
    trip_t = O.synth_triplets(B, G, t)
    lg.append(float(eng.train_step_indices(table16, dev_t(cd, trip_t))[0].item()))
    lm.append(tr16.step(O.flatten_triplets(O.gather_rows(feats, trip_t)))[0])
  print("  loss curve gpu", lg, "model", lm)
  assert np.max(np.abs(np.array(lg) / np.array(lm) - 1)) < 2e-3
  assert bool(torch.isfinite(eng.w).all().item())


def test_adam_trajectory_matches_the_16bit_precision_model(cd):
  """Ten Adam steps against the fp16 PRECISION MODEL's trajectory (same rounding points, float64 arithmetic): replaces the
  former `max |W - W_oracle| < 2.5e-2` bound, which was the maximum possible travel.  Adam's update is sign-like, so a
  weight whose gradient is at the noise floor may step the other way; against the precision model that floor is fp32
  accumulation order + rounding-boundary flips, orders of magnitude below the float64-vs-fp16 distance."""
  G, F, B = 1500, 1500, 384
  dims = [F, 5000, 256]
  feats = O.synth_features(G, F, 0)
  params = O.init_tower(dims, seed=2)
  eng = cd.engine.TowerEngine(dims, device=cd.dev, base_lr=1e-3, margin=0.8, init_params=params)
  table16 = eng.prepare_table(dev_t(cd, feats))
  tr = O.OracleTrainer(params, lr=1e-3, margin=0.8, emulate16="fp16")
  for t in range(10):
    trip = O.synth_triplets(B, G, 20 + t)
    lg = float(eng.train_step_indices(table16, dev_t(cd, trip))[0].item())
    lm = tr.step(O.flatten_triplets(O.gather_rows(feats, trip)))[0]
    assert abs(lg / lm - 1) < 1e-3, (t, lg, lm)
  for l, (W, b) in enumerate(eng.get_params()):
    travel = tr.params[l][0] - params[l][0]
    diff = W - tr.params[l][0]
    rel = np.linalg.norm(diff) / np.linalg.norm(travel)
    frac_off = float((np.abs(diff) > 1e-3).mean())                # more than ONE lr step apart after ten
    print("adam trajectory layer %d: |dW| rel to travel %.3e, max %.3e, frac > 1 lr step %.2e" % (l, rel, np.abs(diff).max(), frac_off))
    assert rel < 1e-1 and frac_off < 2e-2          # measured 1.9e-2 / 5.6e-4 (layer 1) and 5.4e-2 / 7.6e-3 (layer 2)
    db_ = b - tr.params[l][1]
    rel_b = np.linalg.norm(db_) / np.linalg.norm(tr.params[l][1] - params[l][1])
    print("  bias: rel to travel %.3e, max %.3e, frac > 1 lr step %.2e" % (rel_b, np.abs(db_).max(), float((np.abs(db_) > 1e-3).mean())))
    assert rel_b < 1.5e-1 and float((np.abs(db_) > 1e-3).mean()) < 2e-2


def test_flat_knn_ids_equal_the_reference_show_knn_golden(cd, knn_golden):
  """Ids pinned to the reference's OWN brute force (show_knn.calc_nn run by tests/golden/make_knn_golden.py): IndexFlatIP
  and, the rows being unit vectors, IndexFlatL2 must return exactly those ids except inside fp32-noise ties."""
  for name, (seed, N, d, nq, k, clustered) in knn_golden["cases"].items():
    X = knn_golden["rows"](seed, N, d, clustered)
    q = knn_golden["ids"][name + "_queries"]
    want, gap = knn_golden["ids"][name + "_ids"], knn_golden["ids"][name + "_gap"]
    clear = gap > 2e-6
    for metric in ("IP", "L2"):
      index = cd.ops.FlatIndex(dev_t(cd, X), metric)
      D, I = index.search(dev_t(cd, X[q]), k)
      I = I.cpu().numpy()
      assert np.array_equal(I[clear], want[clear]), (name, metric, int((I[clear] != want[clear]).sum()))
      assert all(set(I[i]) == set(want[i]) for i in np.flatnonzero(~clear) if gap[i] > 0), (name, metric)
      index.close()


def test_prediction_run_features_batches_and_tail(cd, tmp_path):
  dims = [1500, 5000, 256]
  params = O.init_tower(dims, seed=2)
  eng = cd.engine.TowerEngine(dims, device=cd.dev, init_params=params)
  feats = O.synth_features(250, 1500, 8)
  pred = cd.predict.Prediction(sess=eng)
  out = pred.run_features(feats, batch_size=100, output_dir=str(tmp_path), suffix="_x")
  assert out.dtype == np.float32 and out.shape == (250, 256)
  assert np.array_equal(np.load(tmp_path / "output_x.npy"), out)
  want = O.tower_forward(feats, params)["l2_norm"]
  assert rel_rows(out, want).max() < 1e-3
  assert np.allclose(pred.predict(feats[:7]), out[:7], atol=1e-6)


# ---------------------------------------------------------------- K5-K8 training step
def _grad_rel(got, want):
  return np.linalg.norm(got - want) / np.linalg.norm(want)


def test_training_step_gradients_loss_and_adam(cd):
  G, F, B = 2000, 1500, 512
  dims = [F, 5000, 256]
  feats = O.synth_features(G, F, 0)
  trip = O.synth_triplets(B, G, 1)
  params = O.init_tower(dims, seed=2)
  eng = cd.engine.TowerEngine(dims, device=cd.dev, base_lr=1e-3, margin=0.8, init_params=params)
  table16 = eng.prepare_table(dev_t(cd, feats))
  x = O.flatten_triplets(O.gather_rows(feats, trip))
  tr = O.OracleTrainer(params, lr=1e-3, margin=0.8)
  _, loss0, grads = tr.loss_and_grads(x)
  stats = eng.train_step_indices(table16, dev_t(cd, trip))
  torch.cuda.synchronize()
  s = stats.cpu().numpy()
  assert abs(s[0] / loss0["hinge_loss"] - 1) < 1e-3
  assert abs(s[1] / loss0["pos_dist"].mean() - 1) < 1e-3 and abs(s[2] / loss0["neg_dist"].mean() - 1) < 1e-3
  # gradient buffers hold SUM-gradients; the oracle's are means over B.
  # (1) against the 16-bit precision model of the same step the kernels must agree tightly;
  # (2) against the unrounded float64 oracle the distance is the inherent price of 16-bit operands: the loss
  #     gradient is built from DIFFERENCES of nearly equal embeddings, which amplifies their ~5e-4 error to 1-2e-2
  #     (the numpy model shows the same figure), so the stated tolerance there is 4e-2.
  model = O.tower_grads_emulated16(x, params, 0.8, "fp16")
  for l in range(2):
    gW, gb = eng.gW[l].cpu().numpy() / B, eng.gb[l].cpu().numpy() / B
    assert _grad_rel(gW, model["grads"][l][0]) < 1e-2 and _grad_rel(gb, model["grads"][l][1]) < 1e-2, l   # + tensor-core accumulation noise, amplified the same way
    assert _grad_rel(gW, grads[l][0]) < 4e-2 and _grad_rel(gb, grads[l][1]) < 4e-2, l
  # 10 optimisation steps on fresh batches: loss curve within 1e-3, weights drift << one lr step
  tr.step(x)
  losses_g, losses_c = [], []
  for t in range(2, 11):
    trip_t = O.synth_triplets(B, G, t)
    losses_g.append(float(eng.train_step_indices(table16, dev_t(cd, trip_t))[0].item()))
    losses_c.append(tr.step(O.flatten_triplets(O.gather_rows(feats, trip_t)))[0])
  assert eng.global_step == 10 and tr.global_step == 10
  assert np.max(np.abs(np.array(losses_g) / np.array(losses_c) - 1)) < 1e-3
  for l, (W, b) in enumerate(eng.get_params()):
    # Adam's update is sign-like (|step| ~ lr whatever the gradient's size), so a weight whose gradient is at the
    # 1-2 % noise floor of the 16-bit operands may travel the other way: bound the worst case by the 10-step travel
    # (2 * 10 * lr) and require the overall travel to agree.
    assert np.abs(W - tr.params[l][0]).max() < 2.5e-2 and _grad_rel(W - params[l][0], tr.params[l][0] - params[l][0]) < 0.2
    assert np.abs(b - tr.params[l][1]).max() < 2.5e-2


@pytest.mark.parametrize("kind,clip,wd", [("adam", 1.0, 1e-3), ("momentum", 0.0, 0.0), ("momentum", 0.7, 1e-3), ("lars", 0.0, 0.0),
                                          ("lars", 0.5, 1e-3), ("sgd", 2.0, 0.0)])
def test_optimizer_kernels_match_oracle_on_identical_gradients(cd, kind, clip, wd):
  """cdml_opt_sumsq + cdml_opt_apply against the oracle's statements of clip_by_norm / regularizer / Momentum / LARS /
  Adam, fed the SAME gradients (fp32 kernels vs float64 oracle: 1e-5 relative)."""
  rng = np.random.RandomState(9)
  n, B = 100003, 64.0
  w = rng.standard_normal(n).astype(np.float32) * 0.05
  kinds = {"adam": cd.ops.OPT_ADAM, "momentum": cd.ops.OPT_MOMENTUM, "lars": cd.ops.OPT_LARS, "sgd": cd.ops.OPT_SGD}
  wd_t, md, vd = dev_t(cd, w), torch.zeros(n, device=cd.dev), torch.zeros(n, device=cd.dev)
  w16 = torch.zeros(n, dtype=torch.float16, device=cd.dev)
  wo, mo, vo = w.astype(np.float64), np.zeros(n), np.zeros(n)
  step = torch.zeros(1, dtype=torch.int64, device=cd.dev)
  scalars = torch.zeros(4, device=cd.dev)
  norms = torch.zeros(2, device=cd.dev)
  ws = torch.empty(cd.ops.opt_workspace_floats(), device=cd.dev)
  lr = 0.05 if kind != "lars" else 1.0
  for t in range(1, 5):
    gsum = (rng.standard_normal(n) * (3.0 if t % 2 else 0.01)).astype(np.float32) * B      # SUM gradient; 1/B folded in
    cd.ops.adam_prepare(step, scalars, lr, 2, 0.5, True)                                    # lr halves every 2 steps
    nz = cd.ops.opt_sumsq(dev_t(cd, gsum), wd_t, norms, ws, grad_scale=1 / B, wd_reg=wd) if (clip > 0 or kind == "lars") else None
    cd.ops.opt_apply(kinds[kind], wd_t, md, vd, dev_t(cd, gsum), scalars, nz, eps=0.0 if kind == "lars" else 1e-8,
                     grad_scale=1 / B, wd_reg=wd, clip_norm=clip, w16=w16)
    g = gsum.astype(np.float64) / B + wd * wo
    if clip > 0:
      g = O.clip_by_norm(g, clip)
    lr_t = O.exponential_decay(lr, t - 1, 2, 0.5)
    if kind == "adam":
      wo, mo, vo = O.adam_step_tf1(wo, mo, vo, g, lr_t, t)
    elif kind == "momentum":
      wo, mo = O.momentum_step_tf1(wo, mo, g, lr_t)
    elif kind == "lars":
      wo, mo = O.lars_step_tf1(wo, mo, g, lr_t)
    else:
      wo = wo - lr_t * g
    got = wd_t.cpu().numpy()
    assert np.abs(got - wo).max() < 1e-5 * max(1.0, np.abs(wo).max()), (kind, t, np.abs(got - wo).max())
  assert np.abs(w16.float().cpu().numpy() - got).max() < 1e-3            # 16-bit shadow weights follow


@pytest.mark.parametrize("optimizer_name,lr", [("LARSOptimizer", 1.0), ("MomentumOptimizer", 0.05)])
def test_build_graph_with_reference_defaults_clip_and_regularizer(cd, optimizer_name, lr):
  """build_graph with ITS OWN defaults (clip_gradient_norm=1.0, regularization_penalty=1; train.py:83-84) and the
  optimizer of main() (LARS, train.py:354) tracks the oracle: loss curve within 1e-3, same weight travel."""
  G, F, B = 1500, 1500, 256
  feats = O.synth_features(G, F, 0)
  params = O.init_tower([F, 5000, 256], seed=2)
  g = cd.train.build_graph(cd.models.placeholder(F), cd.models.VNet(), base_learning_rate=lr, margin=0.8,
                           optimizer_class=getattr(cd.train, optimizer_name), init_params=params)
  eng = g.engine
  kind = {"LARSOptimizer": "lars", "MomentumOptimizer": "momentum"}[optimizer_name]
  tr = O.OracleTrainer(params, lr=lr, margin=0.8, decay_steps=100000, optimizer=kind, clip_norm=1.0, reg_penalty=1.0, l2_penalty=1e-8)
  table16 = eng.prepare_table(dev_t(cd, feats))
  lg, lc = [], []
  for t in range(6):
    trip = O.synth_triplets(B, G, 70 + t)
    lg.append(float(eng.train_step_indices(table16, dev_t(cd, trip))[0].item()))
    lc.append(tr.step(O.flatten_triplets(O.gather_rows(feats, trip)))[0])
  assert np.max(np.abs(np.array(lg) / np.array(lc) - 1)) < 1e-3, (lg, lc)
  for l, (W, b) in enumerate(eng.get_params()):
    assert _grad_rel(W - params[l][0], tr.params[l][0] - params[l][0]) < 0.2, l    # 16-bit gradient noise (1-2 %), compounded by momentum


def test_cuda_graph_step_equals_eager_step(cd):
  G, F, B = 1500, 1500, 256
  dims = [F, 5000, 256]
  feats = O.synth_features(G, F, 0)
  params = O.init_tower(dims, seed=2)
  trips = [O.synth_triplets(B, G, 40 + t) for t in range(4)]
  runs = []
  for use_graph in (False, True):
    eng = cd.engine.TowerEngine(dims, device=cd.dev, base_lr=1e-3, margin=0.8, init_params=params)
    table16 = eng.prepare_table(dev_t(cd, feats))
    replay = eng.capture_step(table16, B, mine=True) if use_graph else None
    assert eng.global_step == 0                                  # capture warm-up must not train
    losses = []
    for t in trips:
      idx = dev_t(cd, t)
      st = replay(idx) if use_graph else eng.train_step_indices(table16, idx, mine=True)
      losses.append(float(st[0].item()))
    runs.append((losses, eng.get_params(), eng.global_step))
  assert runs[0][2] == runs[1][2] == 4
  # step 1 starts from identical weights -> identical loss; later steps inherit the fp32 atomicAdd ordering noise of the
  # mined-negative gradient scatter, which can flip a few fp16-ranked selections (1e-4-level loss differences)
  assert np.allclose(runs[0][0][0], runs[1][0][0], rtol=1e-6), (runs[0][0], runs[1][0])
  assert np.allclose(runs[0][0], runs[1][0], rtol=1e-3), (runs[0][0], runs[1][0])
  for (W0, b0), (W1, b1) in zip(runs[0][1], runs[1][1]):
    assert np.abs(W0 - W1).max() < 5e-3 and np.abs(b0 - b1).max() < 5e-3     # same kernels; atomics order in mined dE only


def test_trainer_end_to_end_small(cd, tmp_path):
  G, F = 600, 1500
  feats = O.synth_features(G, F, 0)
  np.save(tmp_path / "features.npy", feats)
  for i in range(2):
    with open(tmp_path / ("c%d.train" % i), "w") as f:
      f.writelines("%d,%d\n" % (a, p) for a, p in O.synth_pairs(1024, G, seed=20 + i))
  for name, seed in (("cowatches.eval", 30), ("cowatches.test", 31)):
    with open(tmp_path / name, "w") as f:
      f.writelines("%d,%d\n" % (a, p) for a, p in O.synth_pairs(64, G, seed=seed))
  from cdml_b200.online_data import load_cowatches
  pipe = cd.inputs.MPTripletPipe(str(tmp_path / "*.train"), str(tmp_path / "features.npy"), seed=1)
  trainer = cd.train.Trainer(pipe=pipe, num_epochs=2, batch_size=256, model=cd.models.VNet(), loss_fn=cd.losses.HingeLoss(),
                             learning_rate=1e-3, margin=0.8, checkpoint_dir=str(tmp_path / "ckpt"),
                             optimizer_class=cd.train.AdamOptimizer, config=None,
                             eval_cowatches=load_cowatches(str(tmp_path / "cowatches.eval")),
                             test_cowatches=load_cowatches(str(tmp_path / "cowatches.test")),
                             check_stop_epoch=0, best_eval_dist=10.0, eval_per_epoch=2, require_improve_num=100)
  eng = trainer.run()
  assert eng.global_step == 16                                   # 2 files x (2048 lines / 256) batches
  assert trainer.total_eval_num >= 3 and np.isfinite(trainer.eval_dist) and trainer.best_eval_dist < 10.0
  ckpt = cd.predict.latest_checkpoint(str(tmp_path / "ckpt"))
  assert ckpt is not None and os.path.exists(ckpt + ".npz")
  z = np.load(ckpt + ".npz")
  assert z["fully_connected/weights"].shape == (1500, 5000) and z["fully_connected_1/biases"].shape == (256,)
  pred = cd.predict.Prediction(ckpt=ckpt)
  e = pred.run_features(feats[:50], batch_size=32)
  assert e.shape == (50, 256) and np.allclose(np.linalg.norm(e, axis=1), 1, atol=1e-5)


# ---------------------------------------------------------------- K11-K13 KNN
def assert_knn_matches(D, I, Dw, Iw, metric="L2", X=None, Q=None, noise=3e-6):
  """ids identical to the fp32 flat oracle except inside runs of distances that tie within fp32 summation noise.
  With X/Q given, near-ties are adjudicated by float64 distances: every row strictly closer than the k-th (by more
  than `noise`) must be present, nothing farther than the k-th (by more than `noise`) may be, and the reported
  distances must equal the float64 ones to fp32 accuracy."""
  assert D.shape == Dw.shape and I.shape == Iw.shape
  finite = np.isfinite(Dw)
  assert np.array_equal(np.isfinite(D), finite) and np.array_equal(I < 0, Iw < 0)
  assert np.allclose(D[finite], Dw[finite], atol=2e-5, rtol=1e-5)
  sign = 1.0 if metric == "L2" else -1.0
  with np.errstate(invalid="ignore"):
    steps = np.diff(np.where(finite, sign * D, np.inf), axis=1)
  assert (steps[finite[:, 1:]] >= -1e-7).all()                                        # sorted best-first
  diff_rows = np.unique(np.nonzero(I != Iw)[0])
  if len(diff_rows) and X is not None:
    X64, Q64 = X.astype(np.float64), Q.astype(np.float64)
    for r in diff_rows:
      if metric == "L2":
        d64 = np.maximum((Q64[r] ** 2).sum() + (X64 ** 2).sum(1) - 2.0 * (X64 @ Q64[r]), 0)
      else:
        d64 = -(X64 @ Q64[r])
      k = int(finite[r].sum())
      kth = np.partition(d64, k - 1)[k - 1]
      got = I[r, :k]
      assert len(set(got.tolist())) == k
      must = np.nonzero(d64 < kth - noise)[0]
      assert set(must.tolist()) <= set(got.tolist()), (r, "missing a strictly closer row")
      assert (d64[got] <= kth + noise).all(), (r, "reported a strictly farther row")
      assert np.allclose(sign * D[r, :k], d64[got], atol=2e-6 + 1e-5 * np.abs(d64[got]))
  elif len(diff_rows):
    for r in diff_rows:
      for c in np.nonzero(I[r] != Iw[r])[0]:
        near = np.abs(Dw[r] - Dw[r, c]) <= noise
        assert near.sum() >= 2 or c == Dw.shape[1] - 1, (r, c)
  return len(diff_rows) / max(D.shape[0], 1)


@pytest.mark.parametrize("N,nq,k,metric", [(20000, 1000, 100, "L2"), (5000, 300, 10, "IP"), (1500, 200, 51, "L2"),
                                           (60, 60, 100, "L2"), (33000, 257, 81, "L2")])
def test_flat_knn_ids_match_oracle(cd, N, nq, k, metric):
  rng = np.random.RandomState(4)
  X = O.knn_normalize(rng.standard_normal((N, 256)).astype(np.float32))
  if metric == "IP":
    X = (X * rng.uniform(0.5, 2.0, size=(N, 1))).astype(np.float32)
  Q = X[:nq] if nq <= N else X
  index = cd.ops.FlatIndex(dev_t(cd, X), metric)
  D, I = index.search(dev_t(cd, Q), k)
  Dw, Iw = O.flat_knn(X, Q, k=k, l2_norm=False, metric=metric)
  frac = assert_knn_matches(D.cpu().numpy(), I.cpu().numpy(), Dw, Iw, metric, X, Q)
  assert frac < 0.02                                              # random data: essentially every row bit-identical
  st = index.last_stats()
  assert st["fallback_queries"] == 0 and st["candidates"] >= min(k, N) * Q.shape[0]
  if metric == "L2" and N >= k:
    assert (I[:, 0].cpu().numpy() == np.arange(Q.shape[0])).all()         # self query first, distance ~0


def test_flat_knn_clustered_duplicates_and_separate_queries(cd):
  rng = np.random.RandomState(5)
  centres = rng.standard_normal((50, 256)).astype(np.float32)
  X = centres[rng.randint(0, 50, 12000)] + 0.05 * rng.standard_normal((12000, 256)).astype(np.float32)
  X[rng.randint(0, 12000, 120)] = X[rng.randint(0, 12000, 120)]             # ~1% exact duplicate rows -> exact ties
  X = O.knn_normalize(X)
  Q = O.knn_normalize(centres + 0.05 * rng.standard_normal((50, 256)).astype(np.float32))
  index = cd.ops.FlatIndex(dev_t(cd, X), "L2")
  D, I = index.search(dev_t(cd, Q), 100)
  Dw, Iw = O.flat_knn(X, Q, k=100, l2_norm=False)
  assert_knn_matches(D.cpu().numpy(), I.cpu().numpy(), Dw, Iw, "L2", X, Q)
  D2, I2 = index.search(dev_t(cd, X[:500]), 100)
  assert_knn_matches(D2.cpu().numpy(), I2.cpu().numpy(), *O.flat_knn(X, X[:500], k=100, l2_norm=False), "L2", X, X[:500])
  # a database made of ONE repeated row overflows every candidate list -> exact fallback, ties -> lowest ids
  Xd = np.tile(X[:1], (5000, 1))
  idx2 = cd.ops.FlatIndex(dev_t(cd, Xd), "L2")
  D3, I3 = idx2.search(dev_t(cd, X[:3]), 7)
  assert np.array_equal(I3.cpu().numpy(), np.tile(np.arange(7), (3, 1)))
  assert idx2.last_stats()["fallback_queries"] == 3


def test_calc_knn_api_and_sharded_merge(cd, tmp_path):
  rng = np.random.RandomState(6)
  emb = rng.standard_normal((3000, 256)).astype(np.float32)
  D, I = cd.faiss_knn.calc_knn(emb, nearest_num=51)
  Dw, Iw = O.flat_knn(emb, k=51)
  assert D.dtype == np.float32 and I.dtype == np.int64
  Xn = O.knn_normalize(emb)
  assert_knn_matches(D, I, Dw, Iw, 'L2', Xn, Xn)
  assert np.abs(np.linalg.norm(emb, axis=1) - 1).max() > 0.1          # caller's index array is not mutated (astype copy)
  q = emb[:40].copy()
  cd.faiss_knn.calc_knn(emb, q, nearest_num=5)
  assert np.allclose(np.linalg.norm(q, axis=1), 1, atol=1e-6)         # queries ARE normalised in place (faiss_knn.py:103-104)
  # row-sharded search on one GPU (4 shards) + merge kernel == unsharded
  Xn = O.knn_normalize(emb)
  parts = []
  for s in range(4):
    lo, hi = s * 3000 // 4, (s + 1) * 3000 // 4
    ix = cd.ops.FlatIndex(dev_t(cd, Xn[lo:hi]), "L2")
    parts.append(ix.search(dev_t(cd, Xn), 51, id_offset=lo))
  Dm, Im = cd.ops.knn_merge(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]), "L2")
  assert_knn_matches(Dm.cpu().numpy(), Im.cpu().numpy(), Dw, Iw, 'L2', Xn, Xn)
  # merge kernel alone against the oracle merge (bit-exact: same inputs, (distance,id) order)
  Dg = np.stack([p[0].cpu().numpy() for p in parts]); Ig = np.stack([p[1].cpu().numpy() for p in parts])
  Do, Io = O.knn_merge(list(Dg), list(Ig), 51)
  assert np.array_equal(Im.cpu().numpy(), Io) and np.array_equal(Dm.cpu().numpy(), Do)
  # result files
  dm = {i: "g%04d" % i for i in range(3000)}
  cd.faiss_knn.write_knn(str(tmp_path / "res"), split_num=10, D=D, I=I, prefix="knn_split", decode_map=dm)
  txt = "".join(open(tmp_path / "res" / ("knn_split%d" % j)).read() for j in range(10))
  assert txt == "".join(O.format_knn_rows(0, D, I, dm))


def test_sharded_two_phase_search_with_agreed_bounds(cd):
  """Row-sharded index, bound exchange emulated on one GPU: per-shard cdml_knn_bounds, MAX / MIN across the shards (what
  the NCCL all-reduces do), cdml_knn_search_bounded per shard (lists may be SHORTER than k: -1 / inf padded), merge."""
  rng = np.random.RandomState(11)
  N, nq, k, W = 40000, 512, 100, 4
  X = O.knn_normalize(rng.standard_normal((N, 256)).astype(np.float32))
  Q = X[rng.choice(N, nq, replace=False)]
  Dw, Iw = O.flat_knn(X, Q, k=k, l2_norm=False)
  xq = dev_t(cd, Q)
  shards = [(s * N // W, (s + 1) * N // W) for s in range(W)]
  idx = [cd.ops.FlatIndex(dev_t(cd, X[lo:hi]), "L2") for lo, hi in shards]
  b = [ix.bounds(xq, k, -(-k // W)) for ix in idx]
  bf = torch.stack([x[0] for x in b]).max(0).values
  bp = torch.stack([x[1] for x in b]).min(0).values
  assert torch.isfinite(bf).all() and torch.isfinite(bp).all()
  parts = [ix.search_bounded(xq, k, bf, bp, id_offset=lo) for ix, (lo, hi) in zip(idx, shards)]
  total = sum(ix.last_stats()["candidates"] for ix in idx)
  single = cd.ops.FlatIndex(dev_t(cd, X), "L2")
  single.search(xq, k)
  assert total < 2.5 * single.last_stats()["candidates"]         # ~ one index's worth of nominees, not W times as many
  assert any((p[1] < 0).any().item() for p in parts)             # some shard lists really are short (padding path taken)
  Dm, Im = cd.ops.knn_merge(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]), "L2")
  assert (Im >= 0).all().item()
  assert_knn_matches(Dm.cpu().numpy(), Im.cpu().numpy(), Dw, Iw, 'L2', X, Q)


@pytest.mark.parametrize("metric,W", [("L2", 4), ("L2", 8), ("IP", 3)])
def test_sharded_record_protocol_prunes_against_the_global_bound(cd, metric, W):
  """The three-call shard protocol emulated on one GPU (the element-wise max of the [2,nq] pairs is what the NCCL all-reduce
  MAX does): bounds -> collect (+ nominee selection) -> refine against the GLOBAL bound -> packed records -> k-way merge.
  Result == flat oracle; the records and the merge are bit-identical to their oracle statements; the shards' lists are
  short (the global bound leaves ~k rows per query over all shards to re-rank, not W*k)."""
  rng = np.random.RandomState(13)
  N, nq, k = 48000, 640, 100
  X = O.knn_normalize(rng.standard_normal((N, 256)).astype(np.float32))
  if metric == "IP":
    X = (X * rng.uniform(0.5, 2.0, size=(N, 1))).astype(np.float32)
  Q = X[rng.choice(N, nq, replace=False)]
  Dw, Iw = O.flat_knn(X, Q, k=k, l2_norm=False, metric=metric)
  xq = dev_t(cd, Q)
  shards = [(s * N // W, (s + 1) * N // W) for s in range(W)]
  idx = [cd.ops.FlatIndex(dev_t(cd, X[lo:hi]), metric) for lo, hi in shards]
  k_part = -(-k // W)
  pair = torch.stack([ix.shard_bounds(xq, k, k_part) for ix in idx]).max(0).values
  nom = torch.stack([ix.shard_collect(xq, k, k_part, pair) for ix in idx]).max(0).values
  assert torch.isfinite(nom[1]).all()                                  # every shard nominated >= ceil(k/W) rows per query
  rec = torch.empty((W, nq, k), dtype=torch.int64, device=cd.dev)
  for s_, (ix, (lo, hi)) in enumerate(zip(idx, shards)):
    ix.shard_refine(xq, k, nom, rec[s_], id_offset=lo)
  filled = (rec != -1).sum().item() / float(nq)                        # -1 = all ones = padding
  assert k <= filled < 2.5 * k, filled                                 # local pruning alone would fill W*k per query
  Dm, Im = cd.ops.knn_merge_packed(rec, metric)
  assert (Im >= 0).all().item()
  assert_knn_matches(Dm.cpu().numpy(), Im.cpu().numpy(), Dw, Iw, metric, X, Q)
  # the record format and the merge against their oracle statements, bit for bit
  Do, Io = O.knn_merge_records(rec.cpu().numpy().view(np.uint64), k, metric)
  assert np.array_equal(Im.cpu().numpy(), Io) and np.array_equal(Dm.cpu().numpy(), Do)
  merged = cd.ops.knn_merge_packed(rec, metric, as_records=True)       # the form that is all-gathered, and its unpacking
  Du, Iu = cd.ops.knn_unpack_records(merged, metric)
  assert torch.equal(Du, Dm) and torch.equal(Iu, Im)
  one = idx[0].search(xq[:64], 10, id_offset=shards[0][0])
  packed = O.knn_pack_records(one[0].cpu().numpy(), one[1].cpu().numpy(), metric)
  D1, I1 = O.knn_merge_records(packed[None], 10, metric)
  assert np.array_equal(I1, one[1].cpu().numpy()) and np.array_equal(D1, one[0].cpu().numpy())
  for ix in idx:
    ix.close()


def test_sharded_refine_deferred_overflow_check(cd):
  """The deferred form of cdml_knn_shard_refine (no host synchronisation): same records as the synchronous form and a
  clear flag on ordinary data; on an index of near-identical rows (every query's candidate list overflows) the flag is
  raised -- the caller then repeats the search synchronously, which redoes those queries exactly."""
  rng = np.random.RandomState(17)
  N, nq, k = 30000, 300, 50
  X = O.knn_normalize(rng.standard_normal((N, 256)).astype(np.float32))
  xq = dev_t(cd, X[:nq])
  ix = cd.ops.FlatIndex(dev_t(cd, X), "L2")
  pair = ix.shard_bounds(xq, k, k)
  nom = ix.shard_collect(xq, k, k, pair)
  rec_sync = torch.empty((nq, k), dtype=torch.int64, device=cd.dev)
  ix.shard_refine(xq, k, nom, rec_sync)
  nom = ix.shard_collect(xq, k, k, pair)
  rec_def = torch.empty((nq, k), dtype=torch.int64, device=cd.dev)
  flag = torch.zeros((1,), dtype=torch.int32, device=cd.dev)
  ix.shard_refine(xq, k, nom, rec_def, overflow_flag=flag)
  assert int(flag.item()) == 0 and torch.equal(rec_def, rec_sync)
  Dm, Im = cd.ops.knn_merge_packed(rec_def[None], "L2")
  Dw, Iw = O.flat_knn(X, X[:nq], k=k, l2_norm=False)
  assert_knn_matches(Dm.cpu().numpy(), Im.cpu().numpy(), Dw, Iw, "L2", X, X[:nq])
  ix.close()
  # a collapsed index: 30 000 rows within 1e-4 of one direction -> every row is a nominee of every query
  base = O.knn_normalize(rng.standard_normal((1, 256)).astype(np.float32))
  Xc = O.knn_normalize((base + 1e-4 * rng.standard_normal((N, 256))).astype(np.float32))
  xqc = dev_t(cd, Xc[:64])
  ixc = cd.ops.FlatIndex(dev_t(cd, Xc), "L2")
  pair = ixc.shard_bounds(xqc, k, k)
  nom = ixc.shard_collect(xqc, k, k, pair)
  rec = torch.empty((64, k), dtype=torch.int64, device=cd.dev)
  flag.zero_()
  ixc.shard_refine(xqc, k, nom, rec, overflow_flag=flag)
  assert int(flag.item()) == 1
  nom = ixc.shard_collect(xqc, k, k, pair)
  ixc.shard_refine(xqc, k, nom, rec)                                     # synchronous form: exact fallback inside
  assert ixc.last_stats()["fallback_queries"] > 0
  Dm, Im = cd.ops.knn_merge_packed(rec[None], "L2")
  Dw, Iw = O.flat_knn(Xc, Xc[:64], k=k, l2_norm=False)
  assert np.allclose(Dm.cpu().numpy(), Dw, atol=2e-6)                    # near-ties everywhere: distances, not ids
  ixc.close()


def test_mean_dist_matches_oracle(cd, golden):
  from cdml_b200.evaluate import Evaluation
  ev = Evaluation(golden["gather_features"], golden["eval_cowatches"].tolist())
  assert np.array_equal(ev.features, golden["eval_rencoded_features"])
  assert np.array_equal(np.asarray(ev.cowatches), golden["eval_rencoded_cowatches"])
  got = ev.mean_dist(golden["eval_vectors"], golden["eval_cowatches"].tolist())
  assert abs(got - float(golden["eval_mean_dist"])) < 1e-6


# ---------------------------------------------------------------- row M: in-batch semi-hard mining
def test_semihard_mining_matches_oracle_up_to_fp16_selection_noise(cd):
  _check_semihard_mining(cd, 700)                 # generic kernel


def test_semihard_mining_resident_b_matches_oracle_up_to_fp16_selection_noise(cd):
  _check_semihard_mining(cd, 2048)                # resident-B kernel (B >= 1024)


def _check_semihard_mining(cd, B):
  rng = np.random.RandomState(11)
  D, G = 256, 4 * B // 7                        # few guids -> plenty of excluded (same-guid) candidates
  trip = O.synth_triplets(B, G, seed=3)
  base = O.l2_normalize(rng.standard_normal((G, D)))
  E = O.l2_normalize(base[trip.reshape(-1)] + 0.15 * rng.standard_normal((3 * B, D))).astype(np.float32)
  E32 = dev_t(cd, E)
  E16 = E32.half()
  margin = 0.8
  neg_row, d_an = cd.ops.mine_semihard(E16, E32, dev_t(cd, trip), B, margin)
  neg_row, d_an = neg_row.cpu().numpy(), d_an.cpu().numpy()
  want_row, want_d = O.mine_semihard(E, trip, margin)
  A, P = E[0::3].astype(np.float64), E[1::3].astype(np.float64)
  dp = ((A - P) ** 2).sum(-1)
  exact = ((A - E[neg_row].astype(np.float64)) ** 2).sum(-1)
  assert np.allclose(d_an, exact, atol=1e-5)                     # reported distance is the exact fp32 one
  # (1) against the PRECISION MODEL of the selection (same fp16-rounded operands, same d = 2 - 2s / dp / s_hi arithmetic):
  #     the picks must be the same except where the two best candidates are closer than fp32 accumulation noise
  model_row, model_d, model_gap = O.mine_semihard_emulated16(E, trip, margin, "fp16")
  same16 = neg_row == model_row
  assert same16.mean() >= 0.99, same16.mean()
  for i in np.nonzero(~same16)[0]:
    # fp32 accumulation (tensor core vs float64; ~1e-6 on a K=256 dot product near 1, doubled by d = 2 - 2s): near-ties
    # of the selection distance, or a candidate within that noise of the d > dp boundary
    sel = max(2.0 - 2.0 * float(np.dot(E16.cpu().numpy()[3 * i].astype(np.float64), E16.cpu().numpy()[neg_row[i]].astype(np.float64))), 0.0)
    assert model_gap[i] < 2e-5 or abs(sel - model_d[i]) < 2e-5 or abs(model_d[i] - dp[i]) < 2e-5 or abs(sel - dp[i]) < 2e-5, \
        (i, neg_row[i], model_row[i], sel, model_d[i], model_gap[i], dp[i])
  # (2) against the float64 definition on unrounded embeddings: a different pick is only acceptable as a near-tie of the
  #     oracle's pick within the fp16 operand rounding of the selection distances, or at a category boundary
  same = neg_row == want_row
  tol = 4e-3
  for i in np.nonzero(~same)[0]:
    r = neg_row[i]
    g = trip[r // 3, r % 3]
    assert r == 3 * i + 2 or (r % 3 != 0 and g != trip[i, 0] and g != trip[i, 1])
    near_tie = abs(exact[i] - want_d[i]) < tol
    at_boundary = min(abs(exact[i] - dp[i]), abs(exact[i] - dp[i] - margin), abs(want_d[i] - dp[i]),
                      abs(want_d[i] - dp[i] - margin)) < tol
    assert near_tie or at_boundary, (i, r, want_row[i], exact[i], want_d[i], dp[i])
  # mined training step runs and lowers/keeps a finite loss
  dims = [64, 128, 256]
  eng = cd.engine.TowerEngine(dims, device=cd.dev, init_params=O.init_tower(dims, seed=2))
  feats = O.synth_features(G, 64, 0)
  t16 = eng.prepare_table(dev_t(cd, feats))
  s = eng.train_step_indices(t16, dev_t(cd, trip), mine=True).cpu().numpy()
  assert np.isfinite(s).all() and s[3] <= B


# ---------------------------------------------------------------------------------------------------------------
# BASELINE.json's full sizes, through size-independent properties (the oracle only spot-checks a few rows there)
# ---------------------------------------------------------------------------------------------------------------
def test_full_size_knn_1m_index_properties_and_oracle_spot_check(cd):
  """configs[3]: N = 1M x 256, top-100.  Self is the first neighbour at distance ~0, rows ascending, 0 <= D <= 4,
  ids unique and in range; 24 random queries are compared with the float32 oracle over the whole index."""
  N, d, nq, k = 1000000, 256, 16384, 100
  gen = torch.Generator(device=cd.dev)
  gen.manual_seed(4)
  X = torch.nn.functional.normalize(torch.randn((N, d), generator=gen, device=cd.dev), dim=1)
  index = cd.ops.FlatIndex(X, "L2")
  qrows = torch.randperm(N, generator=gen, device=cd.dev)[:nq]
  D, I = index.search(X[qrows].contiguous(), k)
  st = index.last_stats()
  assert st["fallback_queries"] == 0
  assert bool((I[:, 0] == qrows).all().item())
  assert float(D[:, 0].abs().max().item()) < 1e-5
  assert bool((D[:, 1:] >= D[:, :-1]).all().item())
  assert float(D.min().item()) >= 0.0 and float(D.max().item()) <= 4.0
  assert int(I.min().item()) >= 0 and int(I.max().item()) < N
  srt = torch.sort(I, dim=1).values
  assert bool((srt[:, 1:] != srt[:, :-1]).all().item())
  Xh = X.cpu().numpy()
  pick = np.random.RandomState(0).choice(nq, 24, replace=False)
  Qh = Xh[qrows.cpu().numpy()[pick]]
  Dw, Iw = O.flat_knn(Xh, Qh, k=k, l2_norm=False)
  assert_knn_matches(D[pick].cpu().numpy(), I[pick].cpu().numpy(), Dw, Iw, "L2", Xh, Qh)
  index.close()


def test_full_size_training_step_batch_65536_properties(cd):
  """configs[1]: batch 65536 with in-batch mining on a 200k-guid table.  Gather bit-exact against torch indexing, unit-norm
  embeddings, loss consistent with its own per-triplet outputs, mined negatives valid (guid not in {a,p}, farther than
  the positive), every rank-free invariant of the step."""
  G, F, B = 200000, 1500, 65536
  dims = [F, 5000, 256]
  eng = cd.engine.TowerEngine(dims, device=cd.dev, base_lr=1e-3, margin=0.8, seed=2)
  eng_params0 = eng.get_params()                                    # before the step: what the forward pass used
  gen = torch.Generator(device=cd.dev)
  gen.manual_seed(7)
  table16 = torch.empty((G, eng.F_pad), dtype=torch.float16, device=cd.dev)
  for s in range(0, G, 50000):
    eng.prepare_table(torch.rand((50000, F), generator=gen, device=cd.dev), out=table16[s:s + 50000])
  idx = torch.randint(0, G, (B, 3), generator=gen, device=cd.dev)
  idx[:, 1] = (idx[:, 0] + 1 + idx[:, 1] % (G - 1)) % G
  idx[:, 2] = (idx[:, 1] + 1 + idx[:, 2] % (G - 2)) % G
  clash = idx[:, 2] == idx[:, 0]
  idx[:, 2][clash] = (idx[:, 2][clash] + 1) % G
  x16 = cd.ops.gather_rows(table16, idx)
  assert torch.equal(x16, table16[idx.reshape(-1)])                                     # bit-exact row gather at full size
  w0 = eng.w.clone()
  stats = eng.train_step_rows(x16, B, mine=True, guid=idx)
  buf = eng._buffers(3 * B, True)
  e = buf["e"]
  assert float((e.norm(dim=1) - 1).abs().max().item()) < 1e-3
  s = stats.cpu().numpy()
  pos, neg, hin = (buf["loss"][k_] for k_ in ("pos_dist", "neg_dist", "hinge_dist"))
  assert abs(s[0] - float(hin.double().mean().item())) < 1e-5 and abs(s[1] - float(pos.double().mean().item())) < 1e-5
  assert bool(torch.allclose(hin, torch.clamp(pos - neg + 0.8, min=0), atol=1e-6))
  assert 0.0 <= s[0] <= 0.8 + 4.0
  # mining: recompute with the ops-level call on the same embeddings
  e16 = eng._ws[("e16", 3 * B)]
  neg_row, d_an = cd.ops.mine_semihard(e16, e, idx, B, 0.8, want_dist=True)
  flat = idx.reshape(-1)
  g_neg = flat[neg_row.long()]
  assert bool(((g_neg != idx[:, 0]) & (g_neg != idx[:, 1])).all().item())
  assert bool((neg_row.long() % 3 != 0).all().item())                                    # candidates are positives / negatives, never anchors
  mined = neg_row.long() != 3 * torch.arange(B, device=cd.dev) + 2
  assert float(mined.float().mean().item()) > 0.9
  assert bool((d_an[mined] > pos[mined] - 2e-2).all().item())                            # d(a,n) > d(a,p) up to the fp16 selection noise
  assert bool(torch.isfinite(eng.w).all().item()) and float((eng.w - w0).abs().max().item()) <= 1.01e-3   # one Adam step
  # oracle spot check at full size (like the 1 M KNN / de-similarity tests): 256 sampled triplets -- their 768 embeddings
  # against the float64 oracle of the forward pass on the same table rows (<= 1e-3), the loss of the sample with the
  # kernel's own mined negatives, and the mined pick of those anchors against the precision model of the selection
  rs = np.random.RandomState(3)
  samp = np.sort(rs.choice(B, 256, replace=False))
  rows = (3 * samp[:, None] + np.arange(3)[None, :]).reshape(-1)
  x_s = x16[torch.as_tensor(rows, device=cd.dev)][:, :F].float().cpu().numpy().astype(np.float64)    # normalised fp16 table rows
  init = eng_params0
  fwd = O.tower_forward(x_s, init)["l2_norm"]           # the rows are unit to fp16 rounding; tower_forward re-normalises
  e_s = e[torch.as_tensor(rows, device=cd.dev)].cpu().numpy()
  assert rel_rows(e_s, fwd).max() < 1e-3
  nr = neg_row.cpu().numpy()
  E_all = e.cpu().numpy()
  a_, p_, n_ = E_all[3 * samp], E_all[3 * samp + 1], E_all[nr[samp]]
  hin_s = np.maximum(((a_ - p_) ** 2).sum(-1) - ((a_ - n_) ** 2).sum(-1) + 0.8, 0.0)
  assert np.allclose(hin.cpu().numpy()[samp], hin_s, atol=2e-5)
  fa, fp_, fn_ = fwd[0::3], fwd[1::3], O.tower_forward(x16[torch.as_tensor(nr[samp], device=cd.dev).long()][:, :F].float().cpu().numpy().astype(np.float64), init)["l2_norm"]
  loss_s = np.maximum(((fa - fp_) ** 2).sum(-1) - ((fa - fn_) ** 2).sum(-1) + 0.8, 0.0).mean()
  assert abs(hin_s.mean() / loss_s - 1) < 1e-3, (hin_s.mean(), loss_s)
  e16_np = e16.float().cpu().numpy()
  trip_np = idx.cpu().numpy()
  cand = np.concatenate([3 * np.arange(B) + 1, 3 * np.arange(B) + 2])
  cg = np.concatenate([trip_np[:, 1], trip_np[:, 2]])
  agree = 0
  C64 = e16_np[cand].astype(np.float64)
  for i in samp[:64]:
    sc = (C64 @ e16_np[3 * i].astype(np.float64)).astype(np.float32)
    dpi = np.float32(((E_all[3 * i] - E_all[3 * i + 1]) ** 2).sum(dtype=np.float32))
    d = np.maximum(np.float32(2) - np.float32(2) * sc, np.float32(0))
    ok = (sc < np.float32(1) - np.float32(0.5) * dpi) & (d > dpi) & (cg != trip_np[i, 0]) & (cg != trip_np[i, 1])
    dm = np.where(ok, d, np.inf)
    best = cand[np.flatnonzero(dm == dm.min())].min()
    # the tensor core's fp32 accumulation of a K=256 dot product near 1.0 differs from the float64 sum by up to ~1e-6
    # (d = 2 - 2s doubles it); in this structureless regime the candidates are 1e-8 apart, so the pick itself is noise --
    # what is checked is that the kernel's pick is within that accumulation noise of the model's minimum
    near = abs(float(d[np.flatnonzero(cand == nr[i])[0]]) - float(dm.min())) < 2e-5
    agree += int(best == nr[i] or near)
  assert agree == 64, agree


# ---------------------------------------------------------------- fusion towers (SURVEY 8f row 1; models.py:65-243)
def _fusion_engine(cd, name, **kw):
  model = getattr(cd.models, name)()
  g = cd.models.compile_graph(model.create_model(cd.models.placeholder(1628))["l2_norm"])
  from cdml_b200 import fusion
  spec = O.fusion_spec(name)
  params = O.init_graph(spec, seed=2)
  return fusion.GraphEngine(g["spec"], feature_size=1628, device=cd.dev, init_params=params, **kw), spec, params


def test_ew16_and_rows_l2norm16_kernels(cd):
  """cdml_ew16 (all eight joins, vector and 2-element paths, aliased output) and cdml_rows_l2norm16 against numpy."""
  rng = np.random.RandomState(5)
  for rows, cols, pitch in ((515, 256, 320), (33, 10, 14)):
    a, b, c = (rng.standard_normal((rows, cols)).astype(np.float16) for _ in range(3))
    def dev(m):
      t = torch.zeros((rows, pitch), dtype=torch.float16, device=cd.dev)[:, :cols]
      t.copy_(torch.as_tensor(m))
      return t
    A, Bm, C = a.astype(np.float64), b.astype(np.float64), c.astype(np.float64)
    lk = lambda t: np.where(t > 0, 1.0, 0.2)
    want = {cd.ops.EW_MUL: A * Bm, cd.ops.EW_ADD: A + Bm, cd.ops.EW_MUL_ADD_BOTH: A * Bm + A + Bm, cd.ops.EW_MASK: A * lk(Bm),
            cd.ops.EW_MUL_ADD: A * Bm + A, cd.ops.EW_FMA: A * Bm + C, cd.ops.EW_MUL_ADD_MASK: (A * Bm + A) * lk(C),
            cd.ops.EW_MUL_MASK: A * Bm * lk(C)}
    for op, w in want.items():
      out = cd.ops.ew16(op, dev(a), dev(b), dev(np.zeros_like(a)), c=dev(c), alpha=0.2).cpu().numpy()
      if op in (cd.ops.EW_MUL, cd.ops.EW_ADD):
        assert np.array_equal(out, w.astype(np.float16)), op                 # exact in fp32, one rounding: bit-exact
      else:                                                                  # fp32 rounding, then fp16 / fp32(0.2): 1 fp16 ulp
        assert np.allclose(out.astype(np.float64), w, rtol=1e-3, atol=1e-7), op
    x = dev(a)
    cd.ops.ew16(cd.ops.EW_ADD, x, dev(b), x)                                 # out aliases an input
    assert np.array_equal(x.cpu().numpy(), (A + Bm).astype(np.float16))
  y = (rng.standard_normal((300, 256)) * 3).astype(np.float16)
  y[7] = 0
  e = torch.empty((300, 256), dtype=torch.float32, device=cd.dev)
  rinv = torch.empty((300,), dtype=torch.float32, device=cd.dev)
  e16 = torch.empty((300, 256), dtype=torch.float16, device=cd.dev)
  cd.ops.rows_l2norm16(dev_t(cd, y), e, rinv=rinv, e16=e16)
  want = O.l2_normalize(y.astype(np.float64))
  assert np.allclose(e.cpu().numpy(), want, atol=1e-6) and np.all(e.cpu().numpy()[7] == 0)
  assert np.allclose(e16.cpu().numpy().astype(np.float64), want, atol=1e-3)
  assert np.allclose(rinv.cpu().numpy()[:7], 1 / np.linalg.norm(y[:7].astype(np.float64), axis=1), rtol=1e-5)


@pytest.mark.parametrize("name", ["MultiplyNet", "MlpNet", "ResNet", "ResNetV2"])
def test_fusion_tower_embeddings_within_1e3(cd, name):
  eng, spec, params = _fusion_engine(cd, name)
  feats = O.synth_features(3 * 130, 1628, 11)
  e = eng.embed(dev_t(cd, feats)).cpu().numpy()
  want = O.graph_forward(feats, spec, params)["l2_norm"]
  assert e.shape == (390, 256) and np.allclose(np.linalg.norm(e, axis=1), 1.0, atol=1e-5)
  assert rel_rows(e, want).max() < 1e-3                          # fp16 operands, fp32 accumulate: stated tolerance 1e-3


@pytest.mark.parametrize("name", ["MultiplyNet", "MlpNet", "ResNet", "ResNetV2"])
def test_fusion_tower_training_step_gradients_and_loss(cd, name):
  G, B = 2000, 384
  eng, spec, params = _fusion_engine(cd, name, base_lr=1e-3, margin=0.8)
  feats = O.synth_features(G, 1628, 0)
  trip = O.synth_triplets(B, G, 1)
  tables = eng.prepare_table(dev_t(cd, feats))
  x = O.flatten_triplets(O.gather_rows(feats, trip))
  tr = O.OracleTrainer(params, lr=1e-3, margin=0.8, spec=spec)
  _, loss0, grads = tr.loss_and_grads(x)
  s = eng.train_step_indices(tables, dev_t(cd, trip)).cpu().numpy()
  assert abs(s[0] / loss0["hinge_loss"] - 1) < 1e-3
  assert abs(s[1] / loss0["pos_dist"].mean() - 1) < 1e-3 and abs(s[2] / loss0["neg_dist"].mean() - 1) < 1e-3
  # Gates relative to what 16-bit storage costs on THIS tower: on an untrained fusion tower the 0.1 biases dominate, the
  # three embeddings of a triplet nearly coincide, and the loss gradient (their differences) amplifies the 2.4e-4 rounding
  # of the stored activations to 1-13 % (numpy precision model vs float64: d_model below).  The kernels are another
  # realisation of the same rounding process (fp32 accumulation order differs), so they must stay within
  # 1e-2 + d_model of the model and 1e-2 + 1.5 d_model of float64; a wrong mask or a lost contribution is off by >30 %.
  model = O.graph_grads_emulated16(x, spec, params, 0.8, "fp16", loss_scale=eng.loss_scale)
  for l in range(eng.L):
    gW, gb = eng.gW[l].cpu().numpy() / (B * eng.loss_scale), eng.gb[l].cpu().numpy() / (B * eng.loss_scale)
    for got, k in ((gW, 0), (gb, 1)):
      d_model = _grad_rel(model["grads"][l][k], grads[l][k])
      assert _grad_rel(got, model["grads"][l][k]) < 1e-2 + d_model, (name, l, k, d_model)
      assert _grad_rel(got, grads[l][k]) < 1e-2 + 1.5 * d_model, (name, l, k, d_model)


def test_resnet_lars_training_as_main_runs_it_and_checkpoint_roundtrip(cd, tmp_path):
  """train.py main(): ResNet + tf.contrib.opt.LARSOptimizer, lr 1.0, margin 0.8 (train.py:354-364) through build_graph;
  loss curve against the oracle, CUDA-graph replay == eager, checkpoint -> predict.load_engine -> same embeddings."""
  G, B = 1500, 256
  spec = O.fusion_spec("ResNet")
  params = O.init_graph(spec, seed=2)
  feats = O.synth_features(G, 1628, 0)
  def build():
    return cd.train.build_graph(cd.models.placeholder(1628), cd.models.ResNet(), base_learning_rate=1.0, margin=0.8,
                                learning_rate_decay_examples=1000000, optimizer_class=cd.train.LARSOptimizer,
                                clip_gradient_norm=0, regularization_penalty=0, init_params=params).engine
  eng, eng2 = build(), build()
  tables = eng.prepare_table(dev_t(cd, feats))
  replay = eng2.capture_step(tables, B)
  tr = O.OracleTrainer(params, lr=1.0, margin=0.8, optimizer="lars", spec=spec)
  lg, lr_, lc = [], [], []
  for t in range(1, 7):
    trip = O.synth_triplets(B, G, t)
    lg.append(float(eng.train_step_indices(tables, dev_t(cd, trip))[0].item()))
    lr_.append(float(replay(dev_t(cd, trip))[0].item()))
    lc.append(tr.step(O.flatten_triplets(O.gather_rows(feats, trip)))[0])
  assert np.max(np.abs(np.array(lg) / np.array(lc) - 1)) < 2e-3, (lg, lc)
  assert np.allclose(lg, lr_, rtol=1e-6)
  for (W, b), (W2, b2), (Wo, bo) in zip(eng.get_params(), eng2.get_params(), tr.params):
    assert np.array_equal(W, W2) and np.array_equal(b, b2)
    assert _grad_rel(W, Wo) < 3e-3                               # LARS moves |W| by ~1e-3 relative per step; 6 steps
  prefix = cd.train.save_checkpoint(eng, str(tmp_path), 6, "ResNet")
  z = np.load(prefix + ".npz")
  assert "layer_visual_1/weights" in z.files and "layer_fusion_2/biases" in z.files
  eng3 = cd.predict.load_engine(prefix)
  q = dev_t(cd, feats[:300])
  assert np.array_equal(eng3.embed(q).cpu().numpy(), eng.embed(q).cpu().numpy())


def test_fusion_tower_mined_step_matches_oracle_selection(cd):
  """ResNet step with in-batch semi-hard mining: the loss of the mined step equals the hinge of the oracle's selection on
  the oracle's embeddings (mining is tower-independent: it sees only E and the guids)."""
  eng, spec, params = _fusion_engine(cd, "ResNet", base_lr=1e-3, margin=0.8)
  G, B = 3000, 512
  feats = O.synth_features(G, 1628, 0)
  trip = O.synth_triplets(B, G, 3)
  tables = eng.prepare_table(dev_t(cd, feats))
  s = eng.train_step_indices(tables, dev_t(cd, trip), mine=True).cpu().numpy()
  E = O.graph_forward(O.flatten_triplets(O.gather_rows(feats, trip)), spec, params)["l2_norm"]
  rows, _ = O.mine_semihard(E, trip, 0.8)
  a, p, n = E[0::3], E[1::3], E[np.asarray(rows)]
  want = np.maximum(((a - p) ** 2).sum(-1) - ((a - n) ** 2).sum(-1) + 0.8, 0).mean()
  assert np.isfinite(s).all() and abs(s[0] / want - 1) < 1e-2       # a few fp16-ranked selections may differ (near ties)


# ---------------------------------------------------------------- de-similarity filter + cross_knn (SURVEY 8f row 2)
def _knn_like(rng, n, k, n_ids, holes=0.0):
  I = np.empty((n, k), np.int64)
  for r in range(n):
    ids = rng.choice(n_ids, size=k, replace=False)
    I[r] = np.concatenate(([r % n_ids], ids[ids != r % n_ids][:k - 1]))
    if holes and rng.rand() < holes:
      I[r, rng.randint(1, k):] = -1
  return I


def test_desim_kernels_bit_exact_vs_reference_golden_and_oracle(cd):
  """cdml_desim / cdml_desim_simple: bit-exact against the reference's own iter_desim_mp outputs (golden) and against the
  oracle on larger seeded cases covering every template path (1-8 entries per lane, 1-2 feature chunks)."""
  g = np.load(os.path.join(GOLDEN, "desim_golden.npz"))
  for name in "abcd":
    eI, fI, fD = g[name + "_eI"], g[name + "_fI"], g[name + "_fD"]
    got = cd.faiss_knn.iter_desim_mp(eI.copy(), fI.copy(), fD.copy(), fD_threshold=1.4, fI_end=int(g[name + "_args"][0]))
    assert got.dtype == np.int64 and np.array_equal(got, g[name + "_out"]), name
    assert np.array_equal(cd.faiss_knn.desim(eI.copy(), fI.copy()), g[name + "_simple"]), name
  gold = np.load(os.path.join(GOLDEN, "reference_golden.npz"))
  assert np.array_equal(cd.faiss_knn.fliter_fI(gold["desim_fI_in"], gold["desim_fD_in"], 1.4), gold["fliter_fI_out"])
  assert np.array_equal(cd.faiss_knn.desim(gold["desim_eI_in"], gold["desim_fI_in"]), gold["desim_out"])
  rng = np.random.RandomState(21)
  for n, ke, kf, f_end, holes in ((3000, 81, 26, 31, 0.0), (1000, 100, 26, 31, 0.1), (500, 20, 50, 40, 0.0),
                                  (300, 200, 31, 31, 0.05), (257, 33, 64, 64, 0.0), (64, 1, 3, 31, 0.0)):
    nid = max(n, ke + 2, kf + 2)
    eI = _knn_like(rng, n, ke, nid, holes)
    fI = _knn_like(rng, nid, kf, nid, holes)
    for r in range(nid):                                            # overlap the two neighbourhoods
      src = eI[r % n]
      take = min(rng.randint(0, 6), kf - 1, ke - 1)
      if take:
        fI[r, 1:1 + take] = src[1:1 + take]
    fD = np.sort(rng.rand(nid, kf).astype(np.float32) * 2.0, axis=1)
    fD[0, 1] = np.nan                                               # NaN is not > threshold: kept, as in numpy
    want = O.iter_desim(eI, fI, fD, 1.4, f_end)
    got = cd.faiss_knn.iter_desim_mp(eI.copy(), fI.copy(), fD.copy(), fI_end=f_end)
    assert np.array_equal(got, want), (n, ke, kf, f_end)
    assert (want == -1).sum() > (eI == -1).sum()
  # a slice of the rows keeps its global row numbers through row_offset (what each rank of sharded_desim filters)
  lo, hi = n // 3, n // 3 + 20
  part = cd.ops.desim(dev_t(cd, eI[lo:hi]), dev_t(cd, fI), dev_t(cd, fD), 1.4, f_end, row_offset=lo)
  assert np.array_equal(part.cpu().numpy(), want[lo:hi])
  # in place (out aliases eI), empty input, ids beyond the feature table (IndexError in the reference)
  e = dev_t(cd, eI)
  assert cd.ops.desim(e, dev_t(cd, fI), dev_t(cd, fD), 1.4, f_end, out=e) is e and np.array_equal(e.cpu().numpy(), want)
  assert cd.ops.desim(dev_t(cd, eI[:0]), dev_t(cd, fI), dev_t(cd, fD)).shape == (0, 1)
  bad = eI.copy()
  bad[3, 0] = nid + 5
  with pytest.raises(IndexError):
    cd.faiss_knn.iter_desim_mp(bad, fI, fD)


def test_strict_and_cross_knn_flows_match_oracle_composition(cd, tmp_path):
  """strict_knn / cross_knn (faiss_knn.py:308-351): KNN of embeddings, de-similarised against the raw-feature KNN, files
  written; every stage against the oracle's statement of the same composition."""
  rng = np.random.RandomState(8)
  n, doc_location, k, kf = 1200, 800, 12, 9
  emb = rng.standard_normal((n, 64)).astype(np.float32)
  feats = rng.standard_normal((n, 32)).astype(np.float32)
  feats[1::7] = feats[0::7][:len(feats[1::7])] + 0.01 * rng.standard_normal(feats[1::7].shape).astype(np.float32)  # near-duplicates
  emb[1::7] = emb[0::7][:len(emb[1::7])] + 0.05 * rng.standard_normal(emb[1::7].shape).astype(np.float32)
  decode = {i: "g%d" % i for i in range(n)}
  fD, fI = cd.faiss_knn.calc_knn(feats.copy(), nearest_num=kf, l2_norm=True)
  fn = O.knn_normalize(feats.copy())
  wD, wI = O.flat_knn(fn, None, k=kf, l2_norm=False)
  assert_knn_matches(fD, fI, wD, wI, "L2", fn, fn)
  out = str(tmp_path)
  # each KNN stage is checked tie-aware against the oracle; the (deterministic, integer) filter stage is then checked
  # bit-exact on the product's own lists, so a sub-ulp tie flip in a KNN cannot masquerade as a filter error
  sD, sI = cd.faiss_knn.strict_knn(emb.copy(), fI, fD, knn_result=out, nearest_num=k, decode_map=decode)
  en = O.knn_normalize(emb.copy())
  eD, eI = O.flat_knn(en, None, k=k, l2_norm=False)
  rawI = np.load(out + "/strictI.npy")
  assert_knn_matches(sD, rawI, eD, eI, "L2", en, en)
  want = O.iter_desim(rawI, fI, fD, 1.4, 31)
  assert np.array_equal(sI, want) and (want[:, 0] == -1).all() and (want != rawI).sum() > n
  assert np.array_equal(np.load(out + "/strictI_desim.npy"), want)
  lines = []
  for j in range(10):
    lines += open(os.path.join(out, "strict_knn%d" % j)).read().splitlines(True)
  assert lines == O.format_knn_rows(0, sD, want, decode)
  cD, cI, cI_desim = cd.faiss_knn.cross_knn(emb.copy(), doc_location, fI, fD, knn_result=out, nearest_num=k, decode_map=decode)
  vdD, vdI = O.flat_knn(en[doc_location:], en[:doc_location], k=k, l2_norm=False)
  dvD, dvI = O.flat_knn(en[:doc_location], en[doc_location:], k=k, l2_norm=False)
  assert_knn_matches(cD[:doc_location], cI[:doc_location] - doc_location, vdD, vdI, "L2", en[doc_location:], en[:doc_location])
  assert_knn_matches(cD[doc_location:], cI[doc_location:], dvD, dvI, "L2", en[:doc_location], en[doc_location:])
  assert np.array_equal(cI_desim, O.iter_desim(cI, fI, fD, 1.4, 31))
  assert np.array_equal(np.load(out + "/crossI_desim.npy"), cI_desim) and os.path.exists(os.path.join(out, "cross_knn9"))


# ---------------------------------------------------------------- on-device triplet reader (SURVEY 8f row 3)
def test_device_reader_bit_exact_vs_oracle_and_pipe_integration(cd, tmp_path):
  """cdml_sample_triplets against the oracle's statement of the same counter-based sampler (integer work: bit-exact),
  its distributional contract, and MPTripletPipe(device_reader=True) end to end."""
  rng = np.random.RandomState(2)
  for n_pairs, G, start, B, seed in ((1000, 1000, 0, 4096, 5), (77, 5000, 123456789, 1000, 2 ** 40 + 17), (1, 3, 0, 64, 1),
                                     (50000, 4000000000, 2 ** 33, 2048, 9)):
    pairs = rng.randint(0, min(G, 2 ** 31), (n_pairs, 2)).astype(np.int64)
    pairs[:, 1] = (pairs[:, 0] + 1 + pairs[:, 1] % (G - 1)) % G
    got = cd.ops.sample_triplets(dev_t(cd, pairs), start, B, G, seed).cpu().numpy()
    assert np.array_equal(got, O.sample_triplets_device(pairs, start, B, G, seed)), (n_pairs, G)
    assert ((got[:, 2] != got[:, 0]) & (got[:, 2] != got[:, 1]) & (got[:, 2] >= 0) & (got[:, 2] < G)).all()
  G = 2000
  pairs = np.stack([np.arange(G), (np.arange(G) + 7) % G], 1).astype(np.int64)
  t = cd.ops.sample_triplets(dev_t(cd, pairs), 0, 1000000, G, 3).cpu().numpy()
  h = np.bincount(t[:, 2], minlength=G)
  assert abs(h - 500.0).max() < 6 * np.sqrt(500.0)                               # uniform negatives
  assert cd.ops.sample_triplets(dev_t(cd, pairs), 0, 0, G, 3).shape == (0, 3)
  # the pipe: device batches == oracle sampler at the positions the host reader would serve; a trainer consumes them
  feats = O.synth_features(300, 1500, 0)
  np.save(tmp_path / "features.npy", feats)
  for i, n in enumerate((700, 333)):
    with open(tmp_path / ("cowatches_%d.train" % i), "w") as f:
      for a, p in O.synth_pairs(n, 300, seed=10 + i):
        f.write("%d,%d\n" % (a, p))
  pipe = cd.inputs.MPTripletPipe(str(tmp_path / "*.train"), str(tmp_path / "features.npy"), seed=4, device_reader=True)
  pipe.create_pipe(num_epochs=2, batch_size=128)
  pos = list(pipe._position_batches())
  served = 0
  while True:
    b = pipe.get_batch_indices_device()
    if b is None:
      break
    i, start = pos[served]
    assert np.array_equal(b.cpu().numpy(), O.sample_triplets_device(pipe._pairs[i], start, 128, 300, 4 + 7919 * i))
    served += 1
  assert served == len(pos) == (1400 // 128) + (666 // 128)
  pipe.create_pipe(num_epochs=2, batch_size=128)
  trainer = cd.train.Trainer(pipe=pipe, num_epochs=2, batch_size=128, model=cd.models.VNet(), loss_fn=cd.losses.HingeLoss(),
                             learning_rate=1e-3, margin=0.8, checkpoint_dir=str(tmp_path / "ckpt"),
                             optimizer_class=cd.train.AdamOptimizer, config=None, eval_cowatches=np.array([[0, 1], [2, 3]]),
                             test_cowatches=np.array([[4, 5]]), check_stop_epoch=3, max_steps=6)
  eng = trainer.run()
  assert eng.global_step == 6


@pytest.mark.parametrize("N,d,nq,k", [(6000, 1628, 700, 26), (3000, 300, 300, 26), (40000, 1500, 1200, 26), (2500, 8, 100, 5)])
def test_flat_knn_over_raw_feature_widths(cd, N, d, nq, k):
  """The raw-feature KNN of faiss_knn.main (faiss_knn.py:378: calc_knn(features, nearest_num=desim_nearest_num)) runs on
  1628- / 1500-wide rows, i.e. outside the d <= 256 resident-panel kernels: generic tcgen05 scans, long-row re-rank."""
  rng = np.random.RandomState(12)
  X = O.knn_normalize(rng.rand(N, d).astype(np.float32) + 0.05 * rng.standard_normal((N, d)).astype(np.float32))
  index = cd.ops.FlatIndex(dev_t(cd, X), "L2")
  D, I = index.search(dev_t(cd, X[:nq]), k)
  Dw, Iw = O.flat_knn(X, X[:nq], k=k, l2_norm=False)
  assert_knn_matches(D.cpu().numpy(), I.cpu().numpy(), Dw, Iw, "L2", X, X[:nq])
  assert (I[:, 0].cpu().numpy() == np.arange(nq)).all()
  index.close()


def test_full_size_desim_properties_and_oracle_spot_check(cd):
  """1M rows x 81 neighbours against a 1M x 26 feature-KNN table (the production shape of faiss_knn.main): survivors are
  a subset of the input in place, the row's own id is gone, the filter is idempotent, no survivor is a near feature
  neighbour of an earlier survivor of its row, and 300 random rows equal the oracle."""
  n, ke, kf = 1000000, 81, 26
  gen = torch.Generator(device=cd.dev)
  gen.manual_seed(21)
  eI = torch.randint(0, n, (n, ke), generator=gen, device=cd.dev, dtype=torch.int64)
  fI = torch.randint(0, n, (n, kf), generator=gen, device=cd.dev, dtype=torch.int64)
  eI[:, 0] = fI[:, 0] = torch.arange(n, device=cd.dev)
  fI[:, 1:9] = eI[:, 1:9]                                       # the query's closest neighbours are also near duplicates of it
  hop = eI[eI[:, 1], 2:6]                                       # and some entries are near duplicates of the first neighbour
  eI[:, 40:44] = hop
  fD = torch.sort(torch.rand((n, kf), generator=gen, device=cd.dev) * 2.0, dim=1).values
  out = cd.ops.desim(eI, fI, fD, 1.4, 31)
  assert cd.ops.poll_errors(out) == 0
  kept = out >= 0
  assert bool((out[kept] == eI[kept]).all().item()) and bool((out[~kept] == -1).all().item())
  assert not bool((out == torch.arange(n, device=cd.dev)[:, None]).any().item())
  frac = float((~kept).float().mean().item())
  assert 0.05 < frac < 0.5, frac
  again = cd.ops.desim(out, fI, fD, 1.4, 31)
  assert bool((again == out).all().item())                      # idempotent
  pick = np.random.RandomState(0).choice(n, 300, replace=False)
  eh, oh = eI[torch.as_tensor(pick, device=cd.dev)].cpu().numpy(), out[torch.as_tensor(pick, device=cd.dev)].cpu().numpy()
  Ff = O.filter_fI(fI.cpu().numpy(), fD.cpu().numpy(), 1.4)[:, :31]        # fliter_fI once for the whole table
  for row, got, r in zip(eh, oh, pick):
    want = row.copy()
    for c in range(ke):                                                      # oracle.iter_desim's row loop on the prepared table
      v = want[c]
      if v < 0:
        continue
      near = Ff[v][Ff[v] >= 0]
      tail = want[c + 1:]
      tail[np.isin(tail, near)] = -1
    want[want == r] = -1
    assert np.array_equal(got, want), r
  # no survivor is a near feature neighbour of an earlier survivor (checked on the sampled rows)
  for got in oh:
    alive = got[got >= 0]
    for i, v in enumerate(alive[:-1]):
      assert not np.isin(alive[i + 1:], Ff[v][Ff[v] >= 0]).any()
