"""Training entry point -- host-side mirror of the reference's train.py: `build_graph` (train.py:74-175), `Trainer`
(train.py:177-336) and `main` (train.py:339-379) with the same names, arguments and flags.  The step itself
(gather -> tower fwd -> hinge loss -> bwd -> Adam [-> NCCL all-reduce]) is executed by `engine.TowerEngine` on libcdml.

One process per GPU: launched under torchrun the trainer shards every global batch across ranks and all-reduces the
flat gradient buffer (the reference is single-GPU with a distributed TODO, train.py:341-342).
"""
import json
import logging
import os
import time
import traceback

import numpy as np
import torch
from absl import app, flags

from . import inputs, losses, models
from .engine import TowerEngine
from .fusion import GraphEngine
from .evaluate import Evaluation
from .online_data import feature_size, load_cowatches
from .predict import Prediction
from .utils import find_class_by_name

FLAGS = flags.FLAGS
if "train_dir" not in FLAGS:
  flags.DEFINE_string("train_dir", "training_dir/dataset/cdml_1", "training set root: *.train, features.npy, cowatches.eval/.test")
  flags.DEFINE_string("checkpoint_dir", "training_dir/checkpoints", "where model.ckpt-<step> and summaries go")
  flags.DEFINE_string("model", "VNet", "tower class name in models.py (the reference's default 'VedeNet' does not exist, SURVEY Q1)")
  flags.DEFINE_string("optimizer", "AdamOptimizer", "AdamOptimizer (build_graph default, train.py:82) | LARSOptimizer (main(), train.py:354) | MomentumOptimizer | GradientDescentOptimizer")
  flags.DEFINE_float("learning_rate", 1e-3, "base learning rate for Adam (main() hard-codes 1.0 for LARS, train.py:363)")
  flags.DEFINE_float("margin", 0.8, "hinge margin (train.py:364)")
  flags.DEFINE_integer("num_epochs", 8, "passes over each *.train file (train.py:359)")
  flags.DEFINE_integer("batch_size", 1024, "triplets per step (train.py:360)")
  flags.DEFINE_boolean("mine_semihard", False, "in-batch semi-hard negative mining (SURVEY 8a row M)")
  flags.DEFINE_boolean("mine_distance_weighted", False, "in-batch distance-weighted negative sampling (Wu et al. 2017); "
                       "not together with --mine_semihard")
  flags.DEFINE_float("dw_cutoff", 0.5, "distance cutoff of --mine_distance_weighted: closer candidates weigh as this distance")
  flags.DEFINE_boolean("device_reader", False, "sample the index triplets on the GPU (cdml_sample_triplets; SURVEY 8f row 3)")
  flags.DEFINE_string("compute_dtype", "fp16", "tensor-core operand type: fp16 | bf16 (fp32 accumulate)")


class AdamOptimizer(object):
  """Stand-in for tf.train.AdamOptimizer as the `optimizer_class` argument (TF1 defaults b1=.9 b2=.999 eps=1e-8)."""

  def __init__(self, learning_rate, beta1=0.9, beta2=0.999, epsilon=1e-8):
    self._lr, self.beta1, self.beta2, self.epsilon = learning_rate, beta1, beta2, epsilon


class MomentumOptimizer(object):
  """tf.train.MomentumOptimizer; build_graph constructs it with momentum=0.9, use_nesterov=True (train.py:115-116)."""

  def __init__(self, learning_rate, momentum=0.9, name="Momentum", use_nesterov=True):
    if not use_nesterov:
      raise NotImplementedError("build_graph only ever asks for the Nesterov form (train.py:116)")
    self._learning_rate, self.momentum = learning_rate, momentum


class GradientDescentOptimizer(object):
  """tf.train.GradientDescentOptimizer."""

  def __init__(self, learning_rate):
    self._learning_rate = learning_rate


class LARSOptimizer(object):
  """tf.contrib.opt.LARSOptimizer with its TF-1.13 defaults (the optimizer of the reference's main(), train.py:354)."""

  def __init__(self, learning_rate, momentum=0.9, weight_decay=0.0001, eeta=0.001, epsilon=0.0):
    self._learning_rate, self.momentum, self.weight_decay, self.eeta, self.epsilon = (
        learning_rate, momentum, weight_decay, eeta, epsilon)
    if epsilon != 0.0:
      raise NotImplementedError("LARSOptimizer epsilon != 0 is not wired through")


_OPTIMIZER_KINDS = {"AdamOptimizer": "adam", "MomentumOptimizer": "momentum", "LARSOptimizer": "lars",
                    "GradientDescentOptimizer": "sgd"}


class Graph(object):
  """What `build_graph` leaves behind (the reference's TF collections, train.py:162-174)."""

  def __init__(self, engine, input_node, result, loss_fn):
    self.engine, self.input_node, self.result, self.loss_fn = engine, input_node, result, loss_fn
    self.output_name = type(result.get("__model__", None)).__name__ + "/model_output"


_DEFAULT_GRAPH = None


def get_default_graph():
  return _DEFAULT_GRAPH


def clip_gradient_norms(gradients_to_variables, max_norm):
  """Per-variable clip_by_norm (train.py:47-64) on (grad, var) torch pairs; the Trainer runs with clipping off."""
  out = []
  for grad, var in gradients_to_variables:
    if grad is not None:
      n = torch.linalg.vector_norm(grad)
      grad = grad * (max_norm / torch.clamp(n, min=max_norm))
    out.append((grad, var))
  return out


def calc_var(triplets, name=None):
  """mean((E - mean_{B,3}(E))^2) (train.py:67-71) -- a summary scalar, host-side."""
  t = np.asarray(triplets, np.float64)
  return float(np.mean((t - t.mean(axis=(0, 1))) ** 2))


def build_graph(input_batch, model, output_size=256, loss_fn=None, base_learning_rate=0.01,
                learning_rate_decay_examples=100000, learning_rate_decay=0.96, margin=0.8,
                optimizer_class=AdamOptimizer, clip_gradient_norm=1.0, regularization_penalty=1,
                dtype16="fp16", process_group=None, seed=2, init_params=None):
  """Model -> lr schedule -> optimizer -> loss -> gradients -> apply, as one TowerEngine (train.py:74-146)."""
  global _DEFAULT_GRAPH
  loss_fn = loss_fn or losses.HingeLoss()
  if not isinstance(loss_fn, losses.HingeLoss):
    raise NotImplementedError("only HingeLoss is fused into the B200 training step")
  if optimizer_class.__name__ not in _OPTIMIZER_KINDS:
    raise NotImplementedError("optimizer %s: built are %s" % (optimizer_class.__name__, sorted(_OPTIMIZER_KINDS)))
  result = model.create_model(input_batch, output_size)
  graph = None
  try:
    spec = models.compile_chain(result["l2_norm"])
  except NotImplementedError:
    # not a plain fully_connected chain: the visual+doc fusion towers (models.py:65-243) run on fusion.GraphEngine
    graph = models.compile_graph(result["l2_norm"])
    fcs = [e for e in graph["spec"] if e["op"] == "fc"]
    spec = {"l2_penalty": [e["l2_penalty"] for e in fcs], "alpha": fcs[0]["alpha"]}
  if optimizer_class.__name__ == "MomentumOptimizer":                       # train.py:115-118
    opt = optimizer_class(base_learning_rate, momentum=0.9, name='Momentum', use_nesterov=True)
  else:
    opt = optimizer_class(base_learning_rate)
  l2_penalties = set(spec["l2_penalty"])
  if regularization_penalty and len(l2_penalties) != 1:
    raise NotImplementedError("layers with different l2_penalty")
  common = dict(dtype16={"fp16": 0, "bf16": 1}[dtype16] if isinstance(dtype16, str) else dtype16, seed=seed)
  if graph is not None:
    make = lambda **kw: GraphEngine(graph["spec"], feature_size=graph["F"], **common, **kw)
  else:
    make = lambda **kw: TowerEngine(spec["dims"], bias_init=spec["bias_init"][0], **common, **kw)
  engine = make(base_lr=base_learning_rate, margin=margin,
                       lr_decay_steps=learning_rate_decay_examples, lr_decay=learning_rate_decay,
                       beta1=getattr(opt, "beta1", 0.9), beta2=getattr(opt, "beta2", 0.999), eps=getattr(opt, "epsilon", 1e-8),
                       alpha=spec["alpha"], process_group=process_group, init_params=init_params,
                       optimizer=_OPTIMIZER_KINDS[optimizer_class.__name__], clip_norm=max(float(clip_gradient_norm), 0.0),
                       reg_penalty=float(regularization_penalty), l2_penalty=l2_penalties.pop(),
                       momentum=getattr(opt, "momentum", 0.9), lars_weight_decay=getattr(opt, "weight_decay", 1e-4),
                       lars_eeta=getattr(opt, "eeta", 1e-3))
  result = dict(result)
  result["__model__"] = model
  _DEFAULT_GRAPH = Graph(engine, input_batch, result, loss_fn)
  return _DEFAULT_GRAPH


# --------------------------------------------------------------------------------------------------
# checkpoints: model.ckpt-<step>.npz + a TF-style `checkpoint` index file (train.py:240, :275; predict.py:119-132)
# --------------------------------------------------------------------------------------------------
def save_checkpoint(engine, checkpoint_dir, step, model_name):
  """tf.train.Saver(max_to_keep=1).save (train.py:240, :275): the new file is written completely (temp name + rename),
  then the `checkpoint` index is switched to it, and only then are older checkpoints removed -- a crash at any point
  leaves an index that names an existing, complete file.  Format: one .npz with the flat fp32 buffers (w, m, v), the
  per-variable arrays under their slim scope names, and `hyper` (JSON: operand dtype, leaky slope, optimizer kind, loss
  scale, margin, ...) so that predict.load_engine serves / resumes the tower as it was trained.  TensorFlow's own
  .meta/.index/.data files are a different container and are NOT read or written (INTEGRATION.md)."""
  os.makedirs(checkpoint_dir, exist_ok=True)
  name = "model.ckpt-%d" % step
  prefix = os.path.join(checkpoint_dir, name)
  sd = engine.state_dict()
  names = {}
  scopes = getattr(engine, "names", None)        # fusion towers name their layers (models.py:82-88)
  for l, (W, b) in enumerate(engine.get_params()):
    scope = scopes[l] if scopes else ("fully_connected" if l == 0 else "fully_connected_%d" % l)   # slim auto scopes
    names[scope + "/weights"], names[scope + "/biases"] = W, b
  if "spec" in sd:
    names["spec"] = np.asarray(sd["spec"])
  tmp = prefix + ".npz.tmp%d" % os.getpid()
  try:
    with open(tmp, "wb") as f:
      np.savez(f, dims=np.asarray(sd["dims"]), w=sd["w"], m=sd["m"], v=sd["v"], step=sd["step"], model=model_name,
               hyper=np.asarray(json.dumps(sd.get("hyper", {}))), **names)
      f.flush()
      os.fsync(f.fileno())
    os.replace(tmp, prefix + ".npz")
  finally:
    if os.path.exists(tmp):
      os.remove(tmp)
  index_tmp = os.path.join(checkpoint_dir, "checkpoint.tmp%d" % os.getpid())
  with open(index_tmp, "w") as f:
    f.write('model_checkpoint_path: "%s"\nall_model_checkpoint_paths: "%s"\n' % (name, name))
  os.replace(index_tmp, os.path.join(checkpoint_dir, "checkpoint"))
  for f in os.listdir(checkpoint_dir):   # max_to_keep=1: older checkpoints go last
    if f.startswith("model.ckpt-") and f.endswith(".npz") and f != name + ".npz":
      os.remove(os.path.join(checkpoint_dir, f))
  return prefix


class Trainer():

  def __init__(self, pipe, num_epochs, batch_size, model, loss_fn, learning_rate, margin,
               checkpoint_dir, optimizer_class, config, eval_cowatches, test_cowatches,
               check_stop_epoch, best_eval_dist=1.0, eval_per_epoch=100, require_improve_num=10,
               mine_semihard=False, dtype16="fp16", process_group=None, max_steps=None, mine_mode=None, dw_cutoff=0.5):
    """mine_mode: None (mine_semihard decides), "semihard" or "distance_weighted" (with dw_cutoff)."""
    if mine_mode not in (None, "semihard", "distance_weighted"):
      raise ValueError("mine_mode must be None, 'semihard' or 'distance_weighted' (got %r)" % (mine_mode,))
    if mine_mode == "distance_weighted" and mine_semihard:
      raise ValueError("mine_semihard and mine_mode='distance_weighted' exclude each other")
    self.pipe, self.num_epochs, self.batch_size = pipe, num_epochs, batch_size
    self.model, self.loss_fn = model, loss_fn
    self.learning_rate, self.margin = learning_rate, margin
    self.checkpoint_dir, self.optimizer_class, self.config = checkpoint_dir, optimizer_class, config
    self.total_eval_num = 0
    self.last_improve_num = 0
    self.check_stop_epoch = check_stop_epoch
    self.best_eval_dist = best_eval_dist
    self.eval_dist = 0.0
    self.eval_per_epoch = eval_per_epoch
    self.require_improve_num = require_improve_num
    self.evaluater = Evaluation(inputs.FEATURES, eval_cowatches)
    self.tester = Evaluation(inputs.FEATURES, test_cowatches)
    self.mine_semihard, self.dtype16, self.pg, self.max_steps = mine_semihard, dtype16, process_group, max_steps
    self.mine = mine_mode or bool(mine_semihard)      # the engines' `mine` argument
    self.dw_cutoff = float(dw_cutoff)
    self.is_master = process_group is None or torch.distributed.get_rank(process_group) == 0
    self.history = []

  def _build_model(self, input_batch):
    """Fixed hyper-parameters of the reference (train.py:210-222)."""
    return build_graph(input_batch=input_batch, model=self.model, output_size=256, loss_fn=self.loss_fn,
                       base_learning_rate=self.learning_rate, learning_rate_decay_examples=1000000,
                       learning_rate_decay=0.96, margin=self.margin, optimizer_class=self.optimizer_class,
                       clip_gradient_norm=0, regularization_penalty=0, dtype16=self.dtype16, process_group=self.pg)

  def _eval(self, predictor, engine, global_step_np, check_stop_step):
    self.total_eval_num += 1
    try:
      if self.evaluater.features is None:
        raise RuntimeError("Train.run evaluater.features is None")
      eval_embeddings = predictor.run_features(self.evaluater.features, batch_size=10000, as_device=True)
      self.eval_dist = self.evaluater.mean_dist(eval_embeddings, self.evaluater.cowatches)
      if engine.world > 1:
        # early stopping and the best-checkpoint decision hang on this number: every rank uses rank 0's value, so the
        # ranks leave the loop in the same step even if their copies ever differed in the last bit
        t = torch.tensor([float(self.eval_dist)], dtype=torch.float64, device=engine.device)
        torch.distributed.broadcast(t, src=0, group=self.pg)
        self.eval_dist = float(t.item())
      if global_step_np <= check_stop_step:
        self.last_improve_num = self.total_eval_num
      elif self.eval_dist < self.best_eval_dist:
        self.best_eval_dist = self.eval_dist
        if self.is_master:
          save_checkpoint(engine, self.checkpoint_dir, global_step_np, type(self.model).__name__)
        self.last_improve_num = self.total_eval_num
      logging.info("Eval %d | best_eval_dist: %s eval_dist: %s", self.total_eval_num, self.best_eval_dist, self.eval_dist)
      self.history.append({"step": int(global_step_np), "eval/eval_dist": self.eval_dist,
                           "eval/best_eval_dist": self.best_eval_dist})
    except Exception as e:
      logging.error("Train._eval %s", e)

  def _test(self, predictor):
    test_embeddings = predictor.run_features(self.tester.features, batch_size=50000, as_device=True)
    return self.evaluater.mean_dist(test_embeddings, self.tester.cowatches)

  def run(self):
    self.pipe.create_pipe(self.num_epochs, self.batch_size)
    F = feature_size() if not isinstance(inputs.FEATURES, np.ndarray) else inputs.FEATURES.shape[1]
    graph = self._build_model(models.placeholder(F, name="input_batch"))
    engine = graph.engine
    engine.dw_cutoff = self.dw_cutoff
    predictor = Prediction(sess=engine)
    fused = hasattr(self.pipe, "get_batch_indices")
    table16 = engine.prepare_table(self.pipe.device_features()) if fused else None
    # the whole step is one CUDA-graph launch -- with N>1 ranks the NCCL all-reduce of the gradients is captured inside it
    # (every rank captures and replays the same number of times: the reader serves whole rounds of `world` batches);
    # CDML_DDP_GRAPH=0 keeps data-parallel steps eager
    use_graph = fused and (engine.world == 1 or os.environ.get("CDML_DDP_GRAPH", "1") != "0")
    replay = engine.capture_step(table16, self.batch_size, mine=self.mine) if use_graph else None

    world = engine.world
    global_step_np = 0
    steps_total = self.pipe.cowatch_num / self.batch_size / world
    check_stop_step = int(steps_total * self.check_stop_epoch)
    step_per_epoch = max(int(steps_total), 1)
    eval_step = int(steps_total / self.eval_per_epoch)
    show_step = int(eval_step / 10)
    logging.info("check_stop_step: %d step_per_epoch: %d eval_step: %d show_step: %d", check_stop_step,
                 step_per_epoch, eval_step, show_step)

    while True:
      try:
        fetch_start_time = time.time()
        if fused and getattr(self.pipe, "device_reader", False):
          batch = self.pipe.get_batch_indices_device()            # triplets sampled on the GPU: no host work per step
        elif fused:
          idx = self.pipe.get_batch_indices()
          batch = None if idx is None else torch.as_tensor(idx).to(engine.device, non_blocking=True)
        else:
          batch = self.pipe.get_batch()
        if batch is None:
          if self.eval_dist < self.best_eval_dist and self.is_master:
            save_checkpoint(engine, self.checkpoint_dir, global_step_np, type(self.model).__name__)
          break
        if self.total_eval_num - self.last_improve_num > self.require_improve_num and global_step_np > check_stop_step:
          logging.info("total_eval_num %s. last_improve_num %s. early stop", self.total_eval_num, self.last_improve_num)
          break
        fetch_time = time.time() - fetch_start_time

        batch_start_time = time.time()
        if fused:
          stats = replay(batch) if replay is not None else engine.train_step_indices(table16, batch, mine=self.mine)
        else:
          if batch.shape[1:] != (3, F):
            continue
          x = torch.as_tensor(np.reshape(batch, (-1, F))).to(engine.device)     # 3-D to 2-D (train.py:313)
          x16 = engine.prepare_table(x)
          stats = engine.train_step_rows(x16, batch.shape[0], mine=False)
        global_step_np += 1
        if show_step > 0 and global_step_np % show_step == 0:
          loss_np = float(stats[0].item())
          train_time = time.time() - batch_start_time
          logging.debug("Epoch %d Step %d | Loss: %.8f | Time: fetch: %.4fsec train: %.4fsec",
                        int(global_step_np / step_per_epoch) + 1, global_step_np, loss_np, fetch_time, train_time)
          self.history.append({"step": global_step_np, "loss": loss_np, "mean_pos_dist": float(stats[1].item()),
                               "mean_neg_dist": float(stats[2].item())})
        if eval_step > 0 and global_step_np % eval_step == 0:
          self._eval(predictor, engine, global_step_np, check_stop_step)
        if self.max_steps is not None and global_step_np >= self.max_steps:
          break
      except Exception as e:
        logging.error("Train.run %s", e)
        raise
    if self.is_master and self.checkpoint_dir:
      os.makedirs(self.checkpoint_dir, exist_ok=True)
      with open(os.path.join(self.checkpoint_dir, "summaries.jsonl"), "w") as f:
        for h in self.history:
          f.write(json.dumps(h) + "\n")
    self.engine = engine
    logging.info("Exited training loop.")
    return engine


def main(args):
  if FLAGS.mine_semihard and FLAGS.mine_distance_weighted:
    raise app.UsageError("--mine_semihard and --mine_distance_weighted exclude each other")
  try:
    pg = None
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
      torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
      torch.distributed.init_process_group("nccl")
      pg = torch.distributed.group.WORLD
    rank = torch.distributed.get_rank() if pg is not None else 0
    world = torch.distributed.get_world_size() if pg is not None else 1
    pipe = inputs.MPTripletPipe(cowatch_file_patten=FLAGS.train_dir + "/*.train",
                                feature_file=FLAGS.train_dir + "/features.npy", wait_times=20, rank=rank, world=world,
                                device_reader=FLAGS.device_reader)
    eval_cowatches = load_cowatches(FLAGS.train_dir + "/cowatches.eval")
    test_cowatches = load_cowatches(FLAGS.train_dir + "/cowatches.test")
    model = find_class_by_name(FLAGS.model, [models])()
    loss_fn = find_class_by_name("HingeLoss", [losses])()
    optimizer_class = {"AdamOptimizer": AdamOptimizer, "LARSOptimizer": LARSOptimizer, "MomentumOptimizer": MomentumOptimizer,
                       "GradientDescentOptimizer": GradientDescentOptimizer}[FLAGS.optimizer]
    trainer = Trainer(pipe=pipe, num_epochs=FLAGS.num_epochs, batch_size=FLAGS.batch_size, model=model, loss_fn=loss_fn,
                      learning_rate=FLAGS.learning_rate, margin=FLAGS.margin, checkpoint_dir=FLAGS.checkpoint_dir,
                      optimizer_class=optimizer_class, config=None, eval_cowatches=eval_cowatches,
                      test_cowatches=test_cowatches, check_stop_epoch=3, best_eval_dist=1.0, eval_per_epoch=100,
                      require_improve_num=40, mine_semihard=FLAGS.mine_semihard, dtype16=FLAGS.compute_dtype,
                      process_group=pg, mine_mode="distance_weighted" if FLAGS.mine_distance_weighted else None,
                      dw_cutoff=FLAGS.dw_cutoff)
    trainer.run()
  except Exception:
    logging.error(traceback.format_exc())
    raise


if __name__ == "__main__":
  app.run(main)
