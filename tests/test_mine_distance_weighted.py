"""Distance-weighted negative sampling (Wu et al. 2017), the second in-batch mining mode: the oracle's statement of the
draws and weights on the CPU, and cdml_mine_distance_weighted against the oracle's precision model on the GPU."""
import numpy as np
import pytest
from scipy import stats

from oracle import cdml_oracle as O
from oracle import mine_dw_oracle as DW

D = 256


# ---------------------------------------------------------------- CPU: the definition
def test_hierarchical_chunk_draws_are_iid_exp1():
  """M ~ Exp(32) at a uniform column K plus M + Exp(1) elsewhere: 32 iid Exp(1) per chunk."""
  n = 20000
  E, M, K = DW.dw_chunk_draws(seed=12345, step=7, anchor=np.arange(n) % 997, cid=np.arange(n) // 997)
  assert E.shape == (n, 32) and np.all(E > 0)
  assert np.array_equal(E.min(1), M) and np.array_equal(E.argmin(1), K)
  assert stats.kstest(E.reshape(-1), "expon").pvalue > 1e-3
  for j in (0, 5, 31):
    assert stats.kstest(E[:, j], "expon").pvalue > 1e-3, j
  assert stats.kstest(32.0 * M, "expon").pvalue > 1e-3
  assert stats.chisquare(np.bincount(K, minlength=32)).pvalue > 1e-3           # the minimum's column is uniform
  # K independent of M: contingency of K against the quartile of M
  q = np.searchsorted(np.quantile(M, [0.25, 0.5, 0.75]), M)
  table = np.zeros((4, 32))
  np.add.at(table, (q, K), 1)
  assert stats.chi2_contingency(table).pvalue > 1e-3
  c = np.corrcoef(E[:, :8].T)[np.triu_indices(8, 1)]
  assert np.abs(c).max() < 5.0 / np.sqrt(n)
  # keyed by every field: a different step, seed, anchor or chunk gives different draws
  for kw in ({"seed": 12346, "step": 7}, {"seed": 12345, "step": 8}, {"seed": 12345, "step": 7 + (1 << 32)}):
    E2, _, _ = DW.dw_chunk_draws(anchor=np.arange(n) % 997, cid=np.arange(n) // 997, **kw)
    assert not np.any(np.all(E2 == E, axis=1))


def test_log_weight_is_u_shaped_and_the_endpoint_bound_holds():
  grid = np.linspace(0.25, 3.999, 200001)
  lw = DW.dw_log_weight(grid, D)
  i = int(np.argmin(lw))
  assert abs(grid[i] - 4.0 * (D - 2) / (2 * D - 5)) < 1e-4
  assert np.all(np.diff(lw[:i]) < 0) and np.all(np.diff(lw[i:]) > 0)
  rng = np.random.RandomState(0)
  for _ in range(2000):
    lo, hi = np.sort(rng.uniform(0.25, 3.99, 2))
    x = np.linspace(lo, hi, 257)
    assert DW.dw_log_weight(x, D).max() <= max(DW.dw_log_weight(lo, D), DW.dw_log_weight(hi, D)) + 1e-9


def _unit(x):
  return x / np.linalg.norm(x, axis=-1, keepdims=True)


def test_oracle_exponential_race_reproduces_the_weights():
  """Over many steps the oracle's picks of one anchor follow w / sum w over its eligible candidates (chi-square)."""
  rng = np.random.RandomState(3)
  B, Dn, margin, cutoff = 6, 8, 0.8, 0.5
  E = _unit(rng.standard_normal((3 * B, Dn)))
  E[1] = _unit(E[0] + 0.9 * rng.standard_normal(Dn))          # dp around 1: a band of eligible candidates around it
  g = np.arange(3 * B).reshape(B, 3)
  steps = 4000
  picks = np.array([DW.mine_distance_weighted(E, g, margin, cutoff, seed=5, step=t, anchors=[0])[0][0] for t in range(steps)])
  rows = np.concatenate([3 * np.arange(B) + 1, 3 * np.arange(B) + 2])
  dp = np.sum((E[0] - E[1]) ** 2)
  delta = np.maximum(2 - 2 * E[rows] @ E[0], cutoff ** 2)
  ok = (delta < dp + margin) & (rows != 1)
  assert ok.sum() >= 3
  w = np.exp(DW.dw_log_weight(delta[ok], Dn) - DW.dw_log_weight(delta[ok], Dn).max())
  p = w / w.sum()
  counts = np.array([(picks == r).sum() for r in rows[ok]])
  assert counts.sum() == steps                                      # never an ineligible row
  keep = p * steps >= 5
  obs = np.append(counts[keep], counts[~keep].sum())
  exp = np.append(p[keep], p[~keep].sum()) * steps
  if exp[-1] == 0:
    obs, exp = obs[:-1], exp[:-1]
  assert stats.chisquare(obs, exp).pvalue > 1e-4, (obs, exp)


# ---------------------------------------------------------------- GPU
def _cd():
  import torch
  import __graft_entry__ as graft
  graft.build()
  from cdml_b200 import engine, models, ops
  torch.cuda.set_device(0)
  return engine, models, ops


@pytest.fixture(scope="module")
def cd():
  import torch

  class NS:
    pass
  ns = NS()
  ns.engine, ns.models, ns.ops = _cd()
  ns.dev = torch.device("cuda:0")
  ns.torch = torch
  return ns


def _batch(cd, B, G, noise, seed):
  """Clustered unit embeddings of B triplets over G guids (few guids: plenty of same-guid exclusions)."""
  torch = cd.torch
  gen = torch.Generator(device=cd.dev)
  gen.manual_seed(seed)
  trip = torch.randint(0, G, (B, 3), generator=gen, device=cd.dev)
  base = torch.nn.functional.normalize(torch.randn((G, D), generator=gen, device=cd.dev), dim=1)
  E = base[trip.reshape(-1)] + noise / np.sqrt(D) * torch.randn((3 * B, D), generator=gen, device=cd.dev)
  return torch.nn.functional.normalize(E, dim=1).contiguous(), trip.contiguous()


def _slope(delta):
  """|d log w / d delta| (the bound on how fp32 score noise moves a key)."""
  return 0.5 * (D - 2) / delta + 0.5 * (D - 3) / np.maximum(4.0 - delta, 4e-6)


# fp32 accumulation of a K=256 tensor-core dot product of unit vectors: <= K * 2^-24 in the score, doubled in delta
EPS_DELTA = 2 * D * 2.0 ** -24


def _model_key(E, trip, i, row, margin, cutoff, seed, step, kind):
  """The precision model's key of candidate `row` for anchor i (inf when not eligible there)."""
  B = trip.shape[0]
  E16 = O.round16(np.asarray(E, np.float32), kind)
  s = np.float32(E16[3 * i] @ E16[row])
  delta = max(np.float32(np.float32(2) - np.float32(2) * s), np.float32(cutoff) * np.float32(cutoff))
  dpm = np.float32(np.sum((E[3 * i] - E[3 * i + 1]) ** 2, dtype=np.float32) + np.float32(margin))
  g = trip[row // 3, row % 3]
  if not (delta < dpm and g != trip[i, 0] and g != trip[i, 1]):
    return np.inf, float(delta), float(dpm)
  col = (row - 1) // 3 if row % 3 == 1 else B + (row - 2) // 3
  e = DW.dw_draws(seed, step, [i], B, np.float32)[0, col]
  return float(np.log(np.float64(e)) - DW.dw_log_weight(float(delta), D)), float(delta), float(dpm)


@pytest.mark.gpu
@pytest.mark.parametrize("B,G,kind,n_check", [(64, 40, "fp16", None), (1000, 400, "fp16", None), (777, 300, "bf16", None),
                                              (4096, 1500, "fp16", None), (4096, 1500, "bf16", 512),
                                              (65536, 20000, "fp16", 256)])
def test_picks_match_the_precision_model(cd, B, G, kind, n_check):
  """Generic kernel (B < 1024) and resident-B kernel (B >= 1024): picks equal the precision model's except at key
  near-ties within fp32 accumulation noise x |d log w / d delta|; every pick is a valid eligible candidate and d_an is
  its exact fp32 distance."""
  torch = cd.torch
  margin, cutoff, seed, step = 0.8, 0.5, 0x1234567890AB, 3
  E32, trip_t = _batch(cd, B, G, noise=1.0, seed=B)
  E16 = E32.half() if kind == "fp16" else E32.bfloat16()
  st = torch.tensor([step], dtype=torch.int64, device=cd.dev)
  neg, d_an = cd.ops.mine_distance_weighted(E16, E32, trip_t, B, margin, cutoff, seed, st)
  neg, d_an = neg.cpu().numpy(), d_an.cpu().numpy()
  E, trip = E32.cpu().numpy(), trip_t.cpu().numpy()
  anchors = np.arange(B) if n_check is None else np.random.RandomState(1).choice(B, n_check, replace=False)
  model_row, model_key, model_gap, model_delta = DW.mine_distance_weighted_emulated16(E, trip, margin, cutoff, seed, step,
                                                                                      kind, anchors)
  got = neg[anchors]
  # invariants
  a64 = E[3 * anchors].astype(np.float64)
  exact = np.sum((a64 - E[got].astype(np.float64)) ** 2, -1)
  assert np.abs(d_an[anchors] - exact).max() < 1e-5
  dp = np.sum((a64 - E[3 * anchors + 1].astype(np.float64)) ** 2, -1)
  mined = got != 3 * anchors + 2
  assert mined.mean() > 0.5
  g = trip[got // 3, got % 3]
  assert np.all(got[mined] % 3 != 0) and np.all(g[mined] != trip[anchors[mined], 0]) and np.all(g[mined] != trip[anchors[mined], 1])
  assert np.all(np.maximum(exact[mined], cutoff ** 2) < dp[mined] + margin + 4e-3)      # fp16 rounding of the selection
  same = got == model_row
  assert same.mean() >= 0.99, same.mean()
  for k in np.nonzero(~same)[0]:
    i = anchors[k]
    kg, dg, dpm = _model_key(E, trip, i, got[k], margin, cutoff, seed, step, kind)
    at_edge = abs(dg - dpm) < 2 * EPS_DELTA or abs(model_delta[k] - dpm) < 2 * EPS_DELTA
    if not at_edge and got[k] != 3 * i + 2:
      tol = EPS_DELTA * (_slope(dg) + _slope(model_delta[k])) + 2e-4 * (1 + abs(model_key[k]))
      assert kg - model_key[k] <= tol, (i, got[k], model_row[k], kg, model_key[k], tol)
    else:
      assert at_edge, (i, got[k], model_row[k])
  print("B=%d %s: %d/%d picks differ from the model (near-ties)" % (B, kind, (~same).sum(), len(anchors)))


@pytest.mark.gpu
def test_empty_band_keeps_the_readers_negative_and_stats(cd):
  torch = cd.torch
  B = 300
  E32, trip = _batch(cd, B, 100, 1.0, 9)
  neg, d_an = cd.ops.mine_distance_weighted(E32.half(), E32, trip, B, -5.0)
  assert np.array_equal(neg.cpu().numpy(), 3 * np.arange(B) + 2)
  assert cd.ops.mine_stats(E32)["mined"] == 0
  E = E32.cpu().numpy().astype(np.float64)
  assert np.abs(d_an.cpu().numpy() - np.sum((E[0::3] - E[2::3]) ** 2, -1)).max() < 1e-5
  neg, _ = cd.ops.mine_distance_weighted(E32.half(), E32, trip, B, 0.8)
  st = cd.ops.mine_stats(E32)
  # "mined": anchors with an eligible candidate (which may be the anchor's own negative row 3i+2)
  assert B >= st["mined"] >= int((neg.cpu().numpy() != 3 * np.arange(B) + 2).sum()) > 0 and st["rescans"] > 0
  with pytest.raises(RuntimeError):
    cd.ops.mine_distance_weighted(E32.half(), E32, trip, B, 0.8, cutoff=2.5)
  with pytest.raises(ValueError):
    cd.ops.mine_distance_weighted(E32.half(), E32, trip, B, 0.8, step=torch.zeros(1, dtype=torch.int32, device=cd.dev))


def _dist_case(cd, case):
  """Small frozen batches: 'sphere' -- near-orthogonal candidates, weights within a few nats; 'cutoff' -- tight
  clusters, most eligible candidates closer than the cutoff (equal weights), a few farther ones."""
  rng = np.random.RandomState(4)
  B = 24
  if case == "sphere":
    E = _unit(rng.standard_normal((3 * B, D)))
  else:                                         # triplet i in cluster i % 3: a, p and its cluster's candidates all close
    base = _unit(rng.standard_normal((3, D)))
    grp = (np.arange(3 * B) // 3) % 3
    E = _unit(base[grp] + 0.2 * rng.standard_normal((3 * B, D)) / np.sqrt(D))
    E[5::9] = _unit(base[grp[5::9]] + 0.6 * rng.standard_normal((len(E[5::9]), D)) / np.sqrt(D))   # beyond the cutoff
  trip = np.arange(3 * B).reshape(B, 3)
  return E.astype(np.float32), trip


def _pool_cells(obs, exp, least=5.0):
  """Chi-square cells with an expected count >= least: the rarest cells are pooled in ascending order of expectation."""
  order = np.argsort(exp)
  o_out, e_out, o_acc, e_acc = [], [], 0.0, 0.0
  for k in order:
    o_acc, e_acc = o_acc + obs[k], e_acc + exp[k]
    if e_acc >= least:
      o_out.append(o_acc), e_out.append(e_acc)
      o_acc = e_acc = 0.0
  if e_out:
    o_out[-1] += o_acc
    e_out[-1] += e_acc
  else:
    o_out, e_out = [o_acc], [e_acc]
  return np.array(o_out), np.array(e_out)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["sphere", "cutoff"])
def test_pick_frequencies_follow_the_weights(cd, case):
  """Thousands of steps on a frozen batch: each anchor's pick frequencies match w_j / sum w (every cell within 5 sigma,
  pooled chi-square)."""
  torch = cd.torch
  E, trip = _dist_case(cd, case)
  B, margin, cutoff = trip.shape[0], 0.8, 0.5
  E32 = torch.as_tensor(E).to(cd.dev)
  E16, trip_t = E32.half(), torch.as_tensor(trip).to(cd.dev)
  steps = 3000
  st = torch.zeros(1, dtype=torch.int64, device=cd.dev)
  picks = torch.empty((steps, B), dtype=torch.int32, device=cd.dev)
  for t in range(steps):
    st.fill_(t)
    picks[t] = cd.ops.mine_distance_weighted(E16, E32, trip_t, B, margin, cutoff, 77, st, want_dist=False)[0]
  picks = picks.cpu().numpy()
  E16n = O.round16(E, "fp16")
  rows = np.concatenate([3 * np.arange(B) + 1, 3 * np.arange(B) + 2])
  below = 0
  obs_all, exp_all = [], []
  for i in range(B):
    s = (E16n[rows] @ E16n[3 * i]).astype(np.float32)
    delta = np.maximum(np.float32(2) - np.float32(2) * s, np.float32(cutoff * cutoff)).astype(np.float64)
    dpm = np.float32(np.sum((E[3 * i] - E[3 * i + 1]) ** 2, dtype=np.float32) + np.float32(margin))
    ok = (delta < dpm) & (rows != 3 * i + 1)
    if not ok.any():
      assert np.all(picks[:, i] == 3 * i + 2)
      continue
    below += int((delta[ok] <= cutoff * cutoff).sum())
    lw = DW.dw_log_weight(delta[ok], D)
    p = np.exp(lw - lw.max())
    p /= p.sum()
    cnt = np.array([(picks[:, i] == r).sum() for r in rows[ok]])
    assert cnt.sum() == steps, i                                    # every pick eligible
    sig = np.sqrt(steps * p * (1 - p))
    assert np.all(np.abs(cnt - steps * p) <= 5 * sig + 1), (i, cnt, steps * p)
    o, e = _pool_cells(cnt, steps * p)
    obs_all.append(o)
    exp_all.append(e)
  dof = sum(len(o) - 1 for o in obs_all)
  chi = sum(((o - e) ** 2 / e).sum() for o, e in zip(obs_all, exp_all))
  assert dof > 0 and stats.chi2.sf(chi, dof) > 1e-4, (chi, dof)
  if case == "cutoff":
    assert below > B                                               # most eligible candidates clamp to the cutoff


@pytest.mark.gpu
def test_draws_are_keyed_by_seed_and_device_step(cd):
  torch = cd.torch
  B = 1000
  E32, trip = _batch(cd, B, 400, 1.0, 21)
  E16 = E32.half()

  def run(seed, step):
    st = None if step is None else torch.tensor([step], dtype=torch.int64, device=cd.dev)
    return cd.ops.mine_distance_weighted(E16, E32, trip, B, 0.8, 0.5, seed, st)[0].cpu().numpy()
  a = run(3, 5)
  assert np.array_equal(a, run(3, 5))
  assert np.array_equal(run(3, 0), run(3, None))                  # NULL step reads as 0
  assert (a != run(3, 6)).mean() > 0.2 and (a != run(4, 5)).mean() > 0.2 and (a != run(3, 5 + (1 << 32))).mean() > 0.2


def _recording(cd, monkeypatch):
  """Wrap ops.mine_distance_weighted to keep (E16, E32, guid, B, step value, neg_row) of every call."""
  calls = []
  orig = cd.ops.mine_distance_weighted

  def rec(E16, E32, guid, B, margin, cutoff=0.5, seed=0, step=None, want_dist=True):
    out = orig(E16, E32, guid, B, margin, cutoff, seed, step, want_dist)
    calls.append({"E16": E16, "E32": E32, "guid": guid, "B": B, "margin": margin, "cutoff": cutoff, "seed": seed,
                  "step": step, "neg": out[0]})
    return out
  monkeypatch.setattr(cd.ops, "mine_distance_weighted", rec)
  return calls, orig


@pytest.mark.gpu
def test_graph_replays_advance_the_draws_and_equal_eager_mining(cd, monkeypatch):
  torch = cd.torch
  dims = [64, 128, 256]
  G, B = 400, 300
  eng = cd.engine.TowerEngine(dims, device=cd.dev, init_params=O.init_tower(dims, seed=2))
  eng.dw_seed = 99
  table16 = eng.prepare_table(torch.as_tensor(O.synth_features(G, 64, 0)).to(cd.dev))
  calls, orig = _recording(cd, monkeypatch)
  replay = eng.capture_step(table16, B, mine="distance_weighted")
  cap = calls[-1]
  assert cap["step"] is eng.step_counter and eng.global_step == 0
  picks = []
  for t in range(2):
    idx = torch.as_tensor(O.synth_triplets(B, G, 50 + t)).to(cd.dev)
    s0 = eng.global_step
    replay(idx)
    torch.cuda.synchronize()
    got = cap["neg"].cpu().numpy().copy()
    want = orig(cap["E16"], cap["E32"], cap["guid"], B, cap["margin"], cap["cutoff"], 99,
                torch.tensor([s0], dtype=torch.int64, device=cd.dev))[0].cpu().numpy()
    assert np.array_equal(got, want), t
    picks.append(got)
  assert eng.global_step == 2
  # the same batch at the next step draws differently
  idx = torch.as_tensor(O.synth_triplets(B, G, 51)).to(cd.dev)
  replay(idx)
  torch.cuda.synchronize()
  assert (cap["neg"].cpu().numpy() != picks[1]).mean() > 0.1


def _hinge(E, rows, margin):
  a, p, n = E[0::3], E[1::3], E[np.asarray(rows)]
  return np.maximum(((a - p) ** 2).sum(-1) - ((a - n) ** 2).sum(-1) + margin, 0).mean()


@pytest.mark.gpu
def test_vnet_step_matches_the_oracle_fed_the_same_negatives(cd, monkeypatch):
  torch = cd.torch
  dims = [64, 128, 256]
  G, B = 400, 700
  params = O.init_tower(dims, seed=2)
  eng = cd.engine.TowerEngine(dims, device=cd.dev, init_params=params, margin=0.8)
  feats = O.synth_features(G, 64, 0)
  trip = O.synth_triplets(B, G, seed=3)
  calls, _ = _recording(cd, monkeypatch)
  s = eng.train_step_indices(eng.prepare_table(torch.as_tensor(feats).to(cd.dev)), torch.as_tensor(trip).to(cd.dev),
                             mine="distance_weighted").cpu().numpy()
  rows = calls[-1]["neg"].cpu().numpy()
  E = O.tower_forward(O.flatten_triplets(O.gather_rows(feats, trip)), params)["l2_norm"]
  assert (rows != 3 * np.arange(B) + 2).mean() > 0.5
  assert np.isfinite(s).all() and abs(s[0] / _hinge(E, rows, 0.8) - 1) < 1e-2
  # same rows as the float64 definition on the oracle's embeddings, up to fp16 near-ties
  want, _ = DW.mine_distance_weighted(E, trip, 0.8, 0.5, eng.dw_seed, 0)
  assert (rows == want).mean() > 0.95
  assert eng.global_step == 1


@pytest.mark.gpu
def test_resnet_step_matches_the_oracle_fed_the_same_negatives(cd, monkeypatch):
  torch = cd.torch
  from cdml_b200 import fusion
  model = cd.models.ResNet()
  g = cd.models.compile_graph(model.create_model(cd.models.placeholder(1628))["l2_norm"])
  spec = O.fusion_spec("ResNet")
  params = O.init_graph(spec, seed=2)
  eng = fusion.GraphEngine(g["spec"], feature_size=1628, device=cd.dev, init_params=params, base_lr=1e-3, margin=0.8)
  G, B = 3000, 512
  feats = O.synth_features(G, 1628, 0)
  trip = O.synth_triplets(B, G, 3)
  calls, _ = _recording(cd, monkeypatch)
  s = eng.train_step_indices(eng.prepare_table(torch.as_tensor(feats).to(cd.dev)), torch.as_tensor(trip).to(cd.dev),
                             mine="distance_weighted").cpu().numpy()
  rows = calls[-1]["neg"].cpu().numpy()
  E = O.graph_forward(O.flatten_triplets(O.gather_rows(feats, trip)), spec, params)["l2_norm"]
  assert np.isfinite(s).all() and abs(s[0] / _hinge(E, rows, 0.8) - 1) < 1e-2
  with pytest.raises(ValueError):
    eng.train_step_indices(eng.prepare_table(torch.as_tensor(feats).to(cd.dev)), torch.as_tensor(trip).to(cd.dev),
                           mine="hardest")
