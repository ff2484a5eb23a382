# coding=utf-8
"""Regenerates the reference-execution goldens: what the original project's own code returns on the seeded cases of
tests/test_reference_exec_cpu.py, tests/test_simaug_reference_cpu.py and the feed-dict tests of
tests/test_dropin_cpu.py.  Those tests compare this repository's oracle and drop-in Model against these files.

Needs a checkout of the original project (code/ and SimAug/code/ of JunweiLiang/Multiverse), named by
MVB_REFERENCE_ROOT:
    MVB_REFERENCE_ROOT=<checkout> python tests/golden/make_golden_refexec.py
Writes
  refexec_forward.npz     Model.build_forward / Trainer of code/pred_models.py on the eager TF-1.15 stand-in
                          (oracle/tf1_eager/run_reference.py), fp64; large arrays as cases.ref_sample
  refexec_simaug.npz      SimAug's multiview_augmentation and white_box_attack (oracle/tf1_eager/run_simaug.py)
  refexec_feed_dicts.npz  Model.get_feed_dict of code/pred_models.py and of SimAug/code/pred_models.py executed on
                          the drop-in Model, plus the batches the first was given (code/pred_utils.py read_data)
"""
import importlib.util
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import cases  # noqa: E402
from oracle import multiverse_ref as R  # noqa: E402
from oracle.tf1_eager import run_reference as X  # noqa: E402
from oracle.tf1_eager import run_simaug as RS  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def put(d, key, a, n=4096):
  """The array itself when small, else cases.ref_sample of it with its shape and largest magnitude."""
  a = np.asarray(a)
  d[key] = cases.ref_sample(a, n)
  d[key + "/shape"] = np.asarray(a.shape, np.int64)
  if a.dtype.kind == "f":
    d[key + "/absmax"] = np.abs(a).max()


def forward_goldens():
  d = {}
  for name, (over, seed) in cases.REFEXEC_FORWARD.items():
    cfg = R.default_config(**over)
    w, f = R.make_weights(cfg, seed), R.make_inputs(cfg, seed)
    out = X.forward(cfg, w, f)
    d[name + "/checksum"] = cases.checksum(*w.values()) + cases.checksum(f["scene_feat"], f["traj"])
    d[name + "/variables"] = np.asarray(sorted(out["variables"]))
    for i in range(len(cfg.scene_grids)):
      if not cfg.use_grids[i]:
        assert out["grid_pred_decoded"][i] == [] and out["grid_pred_reg_decoded"][i] == []
        continue
      for k in ("grid_pred_decoded", "grid_pred_reg_decoded", "scene_convs"):
        put(d, "%s/%s_%d" % (name, k, i), out[k][i])
    if cfg.use_beam_search:
      lg, ids, lp = out["beam_outputs"]
      put(d, name + "/beam_logits", lg)
      d[name + "/beam_ids"], d[name + "/beam_logprobs"] = ids, lp
    else:
      assert out["beam_outputs"] is None
  over, seed, kw = cases.REFEXEC_TRAIN
  cfg = R.default_config(**over, **kw)
  w, f = R.make_weights(cfg, seed), R.make_inputs(cfg, seed)
  got = X.train_step(cfg, w, f, **kw)
  d["train/checksum"] = cases.checksum(*w.values()) + cases.checksum(f["scene_feat"], f["traj"])
  for k in ("loss", "wd_loss", "pred_grid_loss", "global_step"):
    d["train/" + k] = np.asarray(got[k])
  for k in w:
    put(d, "train/grad/" + k, got["grads"][k], 1024)
    put(d, "train/updated/" + k, got["updated"][k], 1024)
  return d


def simaug_goldens():
  d = {}
  cfg, w, f, extra, spec = cases.simaug_case()
  rcfg = R.default_config(**spec["config"])
  for exp in (1, 4, 3):
    ref = RS.multiview(rcfg, w, f, extra, spec["m"], exp, spec["eps"], spec["beta_draw"], with_trainer=(exp == 3),
                       double_weighting=(exp == 3))
    p = "exp%d/" % exp
    put(d, p + "adv_final", ref["adv_final"], 16384)
    d[p + "beta"], d[p + "losses"] = np.asarray(ref["beta_weight"]), np.asarray(ref["losses"], np.float64)
    if exp == 3:
      d[p + "selected"], d[p + "focal"] = ref["selected_extra_indices"], ref["focal_loss_weight"]
      for k, g in ref["grads"].items():
        put(d, p + "grad/" + k, g, 1024)
  n, eps, hw = spec["n"], spec["eps"], 18 * 9
  for mode in cases.SIMAUG_ATTACKS:
    off, fgsm, step, iters, beta = cases.simaug_attack(mode, n, cfg.pred_len, eps, hw)
    ref = RS.adversarial(rcfg, w, f, eps, off, fgsm=fgsm, step_size=step, num_iter=iters, mixup_beta=beta)
    put(d, mode + "/adv_final", ref["adv_final"], 16384)
    d[mode + "/target_label"], d[mode + "/losses"] = ref["target_label"], np.asarray(ref["losses"], np.float64)
  return d


def feed_dict_goldens():
  """The reference's Model.get_feed_dict run on the drop-in Model (placeholders keyed by Model attribute, values as digests)."""
  sys.path.insert(0, os.path.join(ROOT, "multiverse_b200", "dropin"))
  import tensorflow as tf       # the drop-in shim
  import pred_models as pm
  sys.path.insert(0, os.path.join(X.REFERENCE_ROOT, "code"))
  import pred_utils
  spec = importlib.util.spec_from_file_location("ref_pred_models", os.path.join(X.REFERENCE_ROOT, "code", "pred_models.py"))
  ref = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(ref)
  d = {}
  tmp = tempfile.mkdtemp()
  for c, kw in enumerate(cases.FEED_DICT_CONFIGS):
    tf.reset_default_graph()
    args, cfg = cases.dropin_args(**kw)
    args.prepropath = tmp
    from multiverse_b200 import synthetic
    synthetic.write_npz(os.path.join(tmp, "data_test.npz"), cfg, 5, seed=3)
    data = pred_utils.read_data(args, "test")
    model = pm.get_model(args, gpuid=0)
    for b, (_, batch) in enumerate(data.get_batches(args.batch_size, full=True, shuffle=False)):
      cases.put_batch(d, "cfg%d/batch%d/" % (c, b), batch)
      for is_train in (False, True):
        theirs = ref.Model.get_feed_dict(model, batch, is_train=is_train)
        cases.put_feed_digests(d, "cfg%d/batch%d/train%d/" % (c, b, is_train), model, theirs)
  # SimAug's get_feed_dict on a multiview_train batch
  spec = importlib.util.spec_from_file_location("ref_simaug_pred_models", RS.SIMAUG_FILE)
  saved = sys.modules.get("tensorflow")
  sim = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(sim)
  if saved is not None:
    sys.modules["tensorflow"] = saved
  tf.reset_default_graph()
  args, cfg, model, batch = cases.multiview_feed_case(pm)
  cases.put_feed_digests(d, "multiview/", model, sim.Model.get_feed_dict(model, batch, is_train=True))
  return d


def save(name, d):
  np.savez_compressed(os.path.join(OUT, name + ".npz"), **d)
  print("wrote %s.npz (%d entries, %.0f kB)" % (name, len(d), os.path.getsize(os.path.join(OUT, name + ".npz")) / 1e3))


def main():
  assert X.available() and RS.available(), "set MVB_REFERENCE_ROOT to a checkout of the original project"
  save("refexec_forward", forward_goldens())
  save("refexec_simaug", simaug_goldens())
  save("refexec_feed_dicts", feed_dict_goldens())


if __name__ == "__main__":
  main()
