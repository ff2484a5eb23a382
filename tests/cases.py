# coding=utf-8
"""Seeded unit-case inputs shared by tests/golden/make_golden.py and the parity tests.

Inputs are regenerated from the seed (the 12 MB ConvLSTM kernels are not committed); every golden
file stores a checksum of the regenerated inputs so a drifting generator is detected, plus the
oracle's fp64 outputs."""
from __future__ import annotations

import math

import numpy as np

CELL_CASES = {
    # name: (ns, h, w, cx, x_scale, seed)
    "dec_cx32": (2, 6, 5, 32, 1.0, 11),
    "enc_class_cx64": (3, 5, 7, 64, 1.0, 12),
    "enc_reg_cx2": (2, 7, 4, 2, 600.0, 13),      # raw pixel offsets: large magnitude
    "tile_edge": (5, 9, 5, 32, 1.0, 14),          # 300 halo rows: crosses a 128-row M tile
}


def cell_inputs(ns, h, w, cx, seed, x_scale=1.0):
  """Seeded ConvLSTM cell inputs of any size, drawn like cell_case: Glorot-range kernel, small biases, x of the
  given scale, tanh-bounded h and unit-scale c (tests/test_cell_variants_gpu.py and its worker process)."""
  rng = np.random.default_rng(seed)
  ch = 256
  lim = math.sqrt(6.0 / (9 * (cx + ch) + 9 * 4 * ch))
  return dict(kernel=rng.uniform(-lim, lim, size=(3, 3, cx + ch, 4 * ch)).astype(np.float32),
              biases=(rng.standard_normal(4 * ch) * 0.1).astype(np.float32),
              x=(rng.standard_normal((ns, h, w, cx), dtype=np.float32) * np.float32(x_scale)),
              h=np.tanh(rng.standard_normal((ns, h, w, ch), dtype=np.float32)),
              c=rng.standard_normal((ns, h, w, ch), dtype=np.float32))


def checksum(*arrays):
  return float(sum(float(np.sum(np.asarray(a, dtype=np.float64))) for a in arrays))


def cell_case(name):
  ns, h, w, cx, xs, seed = CELL_CASES[name]
  rng = np.random.default_rng(seed)
  ch = 256
  lim = math.sqrt(6.0 / (9 * (cx + ch) + 9 * 4 * ch))
  kernel = rng.uniform(-lim, lim, size=(3, 3, cx + ch, 4 * ch)).astype(np.float32)
  biases = (rng.standard_normal(4 * ch) * 0.1).astype(np.float32)
  x = (rng.standard_normal((ns, h, w, cx)) * xs).astype(np.float32)
  hh = np.tanh(rng.standard_normal((ns, h, w, ch))).astype(np.float32)
  c = rng.standard_normal((ns, h, w, ch)).astype(np.float32)
  return dict(x=x, h=hh, c=c, kernel=kernel, biases=biases)


def gnn_case(seed=21, ns=3, h=5, w=4):
  rng = np.random.default_rng(seed)
  return dict(h=np.tanh(rng.standard_normal((ns, h, w, 256))).astype(np.float32),
              scene=np.tanh(rng.standard_normal((ns, h, w, 64))).astype(np.float32))


def head_case(seed=31, ns=3, h=6, w=5, e=32):
  rng = np.random.default_rng(seed)
  return dict(h=np.tanh(rng.standard_normal((ns, h, w, 256))).astype(np.float32),
              Wo1=(rng.standard_normal((3, 3, 256, 1)) * 0.1).astype(np.float32),
              Wo2=(rng.standard_normal((3, 3, 256, 2)) * 0.1).astype(np.float32),
              We1=(rng.standard_normal((3, 3, 1, e)) * 0.5).astype(np.float32),
              We2=(rng.standard_normal((3, 3, 2, e)) * 0.5).astype(np.float32),
              be=(rng.standard_normal(e) * 0.2).astype(np.float32))


def beam_case(seed=41, n=3, b=5, v=30):
  rng = np.random.default_rng(seed)
  logits = (rng.standard_normal((n, b, v)) * 2).astype(np.float32)
  logits[0, 1, 7] = logits[0, 1, 3]          # exact tie inside a row (rank / top-k tie-break)
  score = (-np.abs(rng.standard_normal((n, b)))).astype(np.float32)
  return dict(logits=logits, score=score)


def scene_case(seed=51, f=3, sh=12, sw=10, sc=11):
  rng = np.random.default_rng(seed)
  seg = rng.integers(0, sc, size=(f, sh, sw))
  feat = np.eye(sc, dtype=np.float32)[seg]
  return dict(scene_feat=feat,
              W1=(rng.standard_normal((3, 3, sc, 64)) * 0.2).astype(np.float32),
              b1=(rng.standard_normal(64) * 0.1).astype(np.float32),
              W2=(rng.standard_normal((3, 3, 64, 64)) * 0.1).astype(np.float32),
              b2=(rng.standard_normal(64) * 0.1).astype(np.float32),
              obs_scene=rng.integers(0, f, size=(4, 8)).astype(np.int32))


ROLLOUTS = {
    # name: config overrides (oracle.default_config), seed
    "greedy_two_scale": (dict(batch_size=2), 0),
    "beam_k20_diverse": (dict(batch_size=2, use_grids=[True, False], use_beam_search=True,
                              beam_size=20, diverse_beam=True, diverse_gamma=0.01,
                              fix_num_timestep=1), 1),
    "beam_k5_plain": (dict(batch_size=2, use_grids=[False, True], use_beam_search=True,
                           beam_size=5, diverse_beam=False, fix_num_timestep=0), 2),
    "greedy_native_18x32": (dict(batch_size=2, scene_h=36, scene_w=64, use_grids=[True, False]), 3),
}


# At-size rollouts (the shapes bench.py actually runs: CTA-pair cell kernel, x-fold + row_map, fan-out with K = 20).
# Their goldens hold REDUCED statistics of the fp64 oracle run (tests/golden/make_golden_atsize.py), not the tensors.
ROLLOUTS_ATSIZE = {
    "beam_k20_n16": (dict(batch_size=16, use_grids=[True, False], use_beam_search=True, beam_size=20,
                          diverse_beam=True, diverse_gamma=0.01, fix_num_timestep=1), 21),
    "greedy_two_scale_n64": (dict(batch_size=64), 22),
    "beam_k20_native_18x32_n4": (dict(batch_size=4, scene_h=36, scene_w=64, use_grids=[True, False],
                                      use_beam_search=True, beam_size=20, diverse_beam=True, diverse_gamma=0.01,
                                      fix_num_timestep=1), 23),
}


def rollout_stats(cfg, out):
  """Size-reduced view of a forward() result (numpy arrays shaped like the reference fetches): what the at-size
  goldens store and what the GPU run is reduced to before the comparison."""
  import numpy as np
  st = {}
  n, tp = cfg.batch_size, cfg.pred_len
  for i, (h, w) in enumerate(cfg.scene_grids):
    if not cfg.use_grids[i]:
      continue
    v = h * w
    lg = np.asarray(out["grid_pred_decoded"][i], np.float64).reshape(n, tp, v)
    reg = np.asarray(out["grid_pred_reg_decoded"][i], np.float64).reshape(n, tp, v, 2)
    am = lg.argmax(-1)
    srt = np.sort(lg, -1)
    cells = (np.arange(8) * 79 + 3) % v
    st["argmax_%d" % i] = am.astype(np.int32)
    st["margin_%d" % i] = srt[..., -1] - srt[..., -2]
    st["lg_max_%d" % i] = srt[..., -1]
    st["lg_mean_%d" % i] = lg.mean(-1)
    st["lg_at_%d" % i] = lg[..., cells]
    st["reg_at_argmax_%d" % i] = np.take_along_axis(reg, am[..., None, None], 2)[:, :, 0]
    st["reg_mean_%d" % i] = reg.mean(2)
    st["reg_at_%d" % i] = reg[:, :, cells]
  if out.get("beam_outputs") is not None:
    blg, ids, lp = out["beam_outputs"]
    blg = np.asarray(blg, np.float64)
    st["beam_ids"] = np.asarray(ids, np.int32)
    st["beam_logprobs"] = np.asarray(lp, np.float64)
    st["beam_lg_max"] = blg.max(-1)
    st["beam_lg_mean"] = blg.mean(-1)
  return st


def simaug_case():
  """Seeded inputs of the SimAug multi-view golden (tests/golden/make_golden_simaug.py): 2 samples, 3 other views,
  one scale (18x9), soft scene features in (-1, 1).  Returns (synthetic config, weights, feeds, extra-view feeds,
  spec)."""
  from multiverse_b200 import synthetic
  n, m = 2, 3
  # gnn_scene_in_greedy=False: SimAug's gnn_edge feeds the scene features to the attention only in the beam decoder
  conf = dict(batch_size=n, use_grids=[False, True], grid_loss_weight=1.0, grid_reg_loss_weight=0.1, wd=0.001,
              gnn_scene_in_greedy=False)
  cfg = synthetic.make_config(clip_gradient_norm=10.0, **conf)
  w = synthetic.make_weights(cfg, 41)
  f = synthetic.make_feeds(cfg, n, 41, with_pred=True)
  rng = np.random.default_rng(9)
  f["scene_feat"] = np.clip(f["scene_feat"] * 0.8 + rng.uniform(-0.1, 0.1, f["scene_feat"].shape), -1, 1).astype(np.float32)
  hw = 18 * 9
  extra = dict(grid_pred_labels_extra=[None, rng.integers(0, hw, size=(n, m, cfg.pred_len)).astype(np.int32)],
               grid_obs_labels_extra=[None, rng.integers(0, hw, size=(n, m, cfg.obs_len)).astype(np.int32)],
               obs_scene_extra=rng.integers(0, f["scene_feat"].shape[0], size=(n, m, cfg.obs_len)).astype(np.int32))
  return cfg, w, f, extra, dict(n=n, m=m, eps=0.1, beta_draw=0.3, config=conf)


def grad_sample_stride(size):
  """Stride of the gradient samples stored in tests/golden/simaug_multiview.npz (<= 2048 entries per variable)."""
  return max(1, -(-size // 2048))


ADV_SAMPLE_STRIDE = 7      # every 7th element of the augmented features is stored in simaug_multiview.npz


# ---- reference-execution goldens (tests/golden/make_golden_refexec.py) --------------------------------------------
REFEXEC_FORWARD = {
    # name: oracle.default_config overrides, seed
    "beam_k5_plain": ROLLOUTS["beam_k5_plain"],
    "beam_k20_diverse": (dict(batch_size=3, use_grids=[False, True], use_beam_search=True, beam_size=20,
                              diverse_beam=True, diverse_gamma=0.01, fix_num_timestep=1), 7),
    "greedy_two_scale": (dict(batch_size=2, scene_h=24, scene_w=16), 8),
    "no_gnn": (dict(batch_size=2, use_grids=[False, True], use_gnn=False), 9),
}
REFEXEC_TRAIN = (dict(batch_size=2, use_grids=[False, True]), 10,
                 dict(grid_loss_weight=1.0, grid_reg_loss_weight=0.1, wd=0.001))
SIMAUG_ATTACKS = ("fgsm", "pgd_mixup")
FEED_DICT_CONFIGS = (dict(), dict(use_grids=[True, False]))


def ref_sample(a, n=4096):
  """Every k-th element of the flattened array, k the smallest stride that leaves at most n: what the
  reference-execution goldens keep of a large output."""
  a = np.asarray(a).reshape(-1)
  return a[::max(1, -(-a.size // n))]


def simaug_attack(mode, n, pred_len, eps, hw):
  """Random target offsets and the (fgsm, step size, iterations, mixup beta) of a white_box_attack case."""
  rng = np.random.default_rng(3)
  off = rng.integers(1, hw, size=(n, pred_len)).astype(np.int32)
  fgsm = mode == "fgsm"
  step, iters, beta = (eps, 1, None) if fgsm else (0.03, 3, 0.4)
  return off, fgsm, step, iters, beta


def dropin_args(**kw):
  """(argparse-like namespace for pred_models.get_model, synthetic config) at batch 3."""
  import types
  from multiverse_b200 import synthetic
  cfg = synthetic.make_config(batch_size=3, **kw)
  a = dict(vars(cfg))
  a.update(modelname="m", runId=0, gpuid=0, use_soft_grid_class=False, soft_grid=1, use_gt_grid=False,
           mask_grid_regression=False, use_single_decoder=False, use_teacher_forcing=False,
           train_w_onehot=True, grid_loss_weight=1.0, grid_reg_loss_weight=0.1, wd=0.001, optimizer="adadelta")
  return types.SimpleNamespace(**a), cfg


def feed_digest(v):
  """sha1 of the value as contiguous float64: equal digests and shapes <=> np.array_equal after the float64 cast."""
  import hashlib
  return hashlib.sha1(np.ascontiguousarray(np.asarray(v).astype(np.float64)).tobytes()).hexdigest()


def feed_labels(model, feed):
  """Placeholder -> the Model attribute holding it ("grid_obs_labels[1]"): placeholder names repeat across scales."""
  labels = {}
  for attr, v in vars(model).items():
    for i, p in enumerate(v if isinstance(v, list) else [v]):
      labels.setdefault(id(p), "%s[%d]" % (attr, i) if isinstance(v, list) else attr)
  out = {labels[id(k)]: v for k, v in feed.items()}
  assert len(out) == len(feed)
  return out


def put_feed_digests(d, prefix, model, feed):
  feed = feed_labels(model, feed)
  d[prefix + "names"] = np.asarray(sorted(feed))
  for k, v in feed.items():
    d[prefix + k + "/shape"] = np.asarray(np.asarray(v).shape, np.int64)
    d[prefix + k + "/sha1"] = np.asarray(feed_digest(v))


def check_feed_digests(g, prefix, model, feed):
  """feed (placeholder -> value) holds, label for label, the stored values; returns the stored labels."""
  feed = feed_labels(model, feed)
  names = set(str(s) for s in g[prefix + "names"])
  for name in names:
    a = np.asarray(feed[name])
    assert a.shape == tuple(g[prefix + name + "/shape"]), name
    assert feed_digest(a) == str(g[prefix + name + "/sha1"]), name
  return names


def _dense_targets(traj, centers):
  return [(np.asarray(t, np.float64)[:, None, None, :] - centers[None]).astype(np.float32) for t in traj]


def put_batch(d, prefix, batch):
  """A pred_utils batch (data lists, shared grid centres) as arrays.  The dense offset targets are not stored when
  they equal float32(trajectory - cell centre), which load_batch then rebuilds."""
  data, shared = batch.data, batch.shared
  centers = {k: np.asarray(v) for k, v in shared.items() if k.startswith("grid_center_")}
  for k, v in centers.items():
    d[prefix + "shared/" + k] = v
  for k, v in data.items():
    if k.startswith(("obs_grid_target_all_", "pred_grid_target_all_")):
      j = k.rsplit("_", 1)[1]
      traj = data["obs_traj" if k.startswith("obs") else "pred_traj"]
      if all(np.array_equal(a, b) for a, b in zip(_dense_targets(traj, centers["grid_center_" + j]), v)):
        d[prefix + "rebuilt/" + k] = np.asarray(len(v))
        continue
    kind = "list/" if isinstance(v, list) else ("array/" if isinstance(v, np.ndarray) else "scalar/")
    d[prefix + kind + k] = np.stack([np.asarray(a) for a in v]) if kind == "list/" else np.asarray(v)


def load_batch(g, prefix):
  import types
  data, shared, rebuilt = {}, {}, []
  for key in g.files:
    if not key.startswith(prefix):
      continue
    kind, k = key[len(prefix):].split("/", 1)
    if kind == "shared":
      shared[k] = g[key]
    elif kind == "list":
      data[k] = list(g[key])
    elif kind == "array":
      data[k] = g[key]
    elif kind == "scalar":
      data[k] = g[key].item()
    elif kind == "rebuilt":
      rebuilt.append(k)
  for k in rebuilt:
    traj = data["obs_traj" if k.startswith("obs") else "pred_traj"]
    data[k] = _dense_targets(traj, shared["grid_center_" + k.rsplit("_", 1)[1]])
  return types.SimpleNamespace(data=data, shared=shared)


def multiview_feed_case(pm):
  """A multiview_train batch (3 samples, 3 extra views) and the drop-in Model it is fed to.  Returns
  (args, config, model, batch)."""
  import types
  args, cfg = dropin_args(use_grids=[False, True])
  n, m = args.batch_size, 3
  args.is_train, args.multiview_train, args.multiview_max_num, args.multiview_exp = True, True, m, 1
  model = pm.get_model(args, gpuid=0)
  rng = np.random.default_rng(5)
  t_in, t_pred = cfg.obs_len, cfg.pred_len

  def views(count):
    return [np.stack([rng.integers(0, h * w, count) for (h, w) in cfg.scene_grids]) for _ in range(m)]
  data = dict(obs_grid_class=[np.stack([rng.integers(0, h * w, t_in) for (h, w) in cfg.scene_grids]) for _ in range(n)],
              pred_grid_class=[np.stack([rng.integers(0, h * w, t_pred) for (h, w) in cfg.scene_grids]) for _ in range(n)],
              batch_scene_feat=rng.random((7, cfg.scene_h, cfg.scene_w, cfg.scene_class)).astype(np.float32),
              batch_obs_scene=rng.integers(0, 7, (n, t_in, 1)),
              batch_extra_obs_scene=rng.integers(0, 7, (n, m, t_in, 1)), extra=[])
  for j, (h, w) in enumerate(cfg.scene_grids):
    data["obs_grid_target_all_%d" % j] = [rng.standard_normal((t_in, h, w, 2)).astype(np.float32) for _ in range(n)]
    data["pred_grid_target_all_%d" % j] = [rng.standard_normal((t_pred, h, w, 2)).astype(np.float32) for _ in range(n)]
  for i in range(n):
    ex = dict(obs_grid_class=views(t_in), pred_grid_class=views(t_pred))
    for j, (h, w) in enumerate(cfg.scene_grids):
      ex["obs_grid_target_all_%d" % j] = [rng.standard_normal((t_in, h, w, 2)).astype(np.float32) for _ in range(m)]
      ex["pred_grid_target_all_%d" % j] = [rng.standard_normal((t_pred, h, w, 2)).astype(np.float32) for _ in range(m)]
    data["extra"].append(ex)
  return args, cfg, model, types.SimpleNamespace(data=data)
