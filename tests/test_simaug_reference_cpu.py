# coding=utf-8
"""SURVEY.md section 8 row f-4, the pin: SimAug's multi-view augmentation as EXECUTED FROM THE REFERENCE'S OWN FILE
(the unmodified SimAug/code/pred_models.py of the original project on the eager TF-1.15 stand-in,
oracle/tf1_eager/run_simaug.py; stored by tests/golden/make_golden_refexec.py in tests/golden/refexec_simaug.npz, the
augmented features as an fp64 sample, cases.ref_sample) against the same pipeline written on the oracle
(oracle/multiverse_ref_torch.py: autograd input gradient, per-view losses, selection, mixup, mixed-label objective) -
the expectation the GPU tests of multiverse_b200/simaug.py and TrainEngine's mixup path are held to."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import cases  # noqa: E402
from oracle import multiverse_ref as R  # noqa: E402
from oracle import multiverse_ref_torch as RT  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden", "refexec_simaug.npz")


def sampled(a, g, key):
  """The stored sample's positions of a (whose shape must be the reference array's)."""
  a = np.asarray(a, np.float64)
  assert a.shape == tuple(g[key + "/shape"]), key
  return cases.ref_sample(a, 16384)


def oracle_pipeline(exp):
  """multiview_augmentation + the training objective on its output, on the oracle.  Returns what the reference run
  returns."""
  cfg, w, f, extra, spec = cases.simaug_case()
  n, m, eps = spec["n"], spec["m"], spec["eps"]
  t_obs, tp = cfg.obs_len, cfg.pred_len
  tile = lambda a: np.repeat(np.asarray(a), m, axis=0)
  clean = f["scene_feat"].astype(np.float64)[f["obs_scene"]]                  # [N,T,SH,SW,SC]
  tf_ = dict(scene_feat=tile(clean).reshape((n * m * t_obs,) + clean.shape[2:]),
             obs_scene=np.arange(n * m * t_obs, dtype=np.int32).reshape(n * m, t_obs))
  for key in ("grid_obs_labels", "grid_obs_regress", "grid_pred_labels", "grid_pred_regress"):
    tf_[key] = [None if a is None else tile(a) for a in f[key]]
  target = extra["grid_pred_labels_extra"][1].reshape(n * m, tp)
  rcfg_t = R.default_config(**dict(spec["config"], batch_size=n * m))
  g, loss = RT.scene_input_grad(rcfg_t, w, tf_, target, 1, per_sample=True)
  loss = loss.reshape(n, m)
  x = tf_["scene_feat"]
  adv = np.minimum(np.maximum(x - eps * np.sign(g), np.clip(x - eps, -1, 1)), np.clip(x + eps, -1, 1))
  adv = adv.reshape((n, m, t_obs) + clean.shape[2:])
  order = np.argsort(-loss, axis=1, kind="stable")
  rows = np.arange(n)
  beta = max(spec["beta_draw"], 1 - spec["beta_draw"])
  res = dict(beta=beta)
  if exp == 1:
    f1, f2 = adv[rows, order[:, 0]], adv[rows, order[:, 1]]
  elif exp == 4:
    f1, f2 = adv[rows, order[:, m - 1]], adv[rows, order[:, m - 2]]
  else:
    f1 = adv[rows, order[:, 0]]
    f2 = f["scene_feat"].astype(np.float64)[extra["obs_scene_extra"][rows, order[:, 0]]]
    res["selected"] = order[:, 0]
    res["focal"] = (1.0 - np.exp(-np.sort(loss, axis=1)[:, -1])) ** 2.0
  final = (f1 * beta + f2 * (1 - beta)).reshape((n * t_obs,) + clean.shape[2:])
  res["adv_final"] = final
  # the training tower on the augmented features (one private frame per (sample, step) row)
  ft = dict(f, scene_feat=final, obs_scene=np.arange(n * t_obs, dtype=np.int32).reshape(n, t_obs))
  if exp == 3:
    sel = res["selected"]
    ft["mixup"] = dict(beta=beta, obs_labels2=[None, extra["grid_obs_labels_extra"][1][rows, sel]],
                       pred_labels2=[None, extra["grid_pred_labels_extra"][1][rows, sel]], focal=res["focal"])
  rcfg = R.default_config(**spec["config"])
  _, losses, _, grads = RT.loss_and_grads(rcfg, w, ft)
  res["losses"], res["grads"] = losses, grads
  return res


@pytest.mark.parametrize("exp", [1, 4, 3])
def test_reference_execution_matches_golden_and_oracle_pipeline(exp):
  g = np.load(GOLD)
  p = "exp%d/" % exp
  o = oracle_pipeline(exp)
  assert abs(o["beta"] - float(g[p + "beta"])) < 1e-12
  d = np.abs(sampled(o["adv_final"], g, p + "adv_final") - g[p + "adv_final"])
  # both are fp64: the sign of an input-gradient entry that is ~0 is the only thing that may differ
  assert (d <= 1e-9).mean() > 0.99999 and d.max() <= 2 * cases.simaug_case()[4]["eps"] + 1e-9
  ref_losses = g[p + "losses"]
  assert np.abs(np.array(o["losses"]) - ref_losses).max() < 1e-6 * max(ref_losses)
  if exp == 3:
    assert np.array_equal(o["selected"], g[p + "selected"])
    assert np.abs(o["focal"] - g[p + "focal"]).max() < 1e-9
    worst = 0.0
    names = set(k[len(p + "grad/"):] for k in g.files
                if k.startswith(p + "grad/") and not k.endswith(("/shape", "/absmax")))
    assert names and names <= set(o["grads"])
    for k in names:
      key = p + "grad/" + k
      og = np.asarray(o["grads"][k], np.float64)
      assert og.shape == tuple(g[key + "/shape"]), k
      scale = max(float(g[key + "/absmax"]), 1e-30)
      worst = max(worst, np.abs(cases.ref_sample(og, 1024) - g[key]).max() / scale)
    print("exp 3: oracle vs reference-exec gradients, worst relative error %.2e over %d variables" % (worst, len(names)))
    assert worst < 1e-6


@pytest.mark.parametrize("mode", cases.SIMAUG_ATTACKS)
def test_white_box_attack_reference_execution_matches_oracle_pipeline(mode):
  """white_box_attack (SimAug/code/pred_models.py:60-170) as executed from the reference file - targeted FGSM, and PGD
  (tf.while_loop, 3 iterations, bounds around the clean input) followed by the mixup with the clean input - against
  the same update rule driven by the oracle's autograd input gradient: what multiverse_b200/simaug.py::
  white_box_attack and mvb_adv_step / mvb_mix implement (GPU: test_simaug_scene_input_gradient_and_attack)."""
  cfg, w, f, extra, spec = cases.simaug_case()
  rcfg = R.default_config(**spec["config"])
  g = np.load(GOLD)
  n, eps, hw = spec["n"], spec["eps"], 18 * 9
  off, fgsm, step, iters, beta = cases.simaug_attack(mode, n, cfg.pred_len, eps, hw)
  target = (f["grid_pred_labels"][1].astype(np.int64) + off) % hw                       # create_random_target
  assert np.array_equal(g[mode + "/target_label"], target) and not (target == f["grid_pred_labels"][1]).any()
  # the oracle's pipeline: one private frame per (sample, step) row, like the reference's [N*T,SH,SW,SC] input
  t_obs = cfg.obs_len
  x = f["scene_feat"].astype(np.float64)[f["obs_scene"]].reshape((n * t_obs,) + f["scene_feat"].shape[1:])
  rows = dict(f, obs_scene=np.arange(n * t_obs, dtype=np.int32).reshape(n, t_obs))
  lo, hi = np.clip(x - eps, -1, 1), np.clip(x + eps, -1, 1)
  adv = x.copy()
  for _ in range(iters):
    gr = RT.scene_input_grad(rcfg, w, dict(rows, scene_feat=adv), target, 1)
    adv = np.minimum(np.maximum(adv - step * np.sign(gr), lo), hi)
  if beta is not None:
    adv = x * beta + adv * (1 - beta)
  d = np.abs(sampled(adv, g, mode + "/adv_final") - g[mode + "/adv_final"])
  print("white_box_attack %s: %.6f of the sampled pixels equal, max diff %.3g" % (mode, (d <= 1e-9).mean(), d.max()))
  assert (d <= 1e-9).mean() > 0.9999 and d.max() <= 2 * eps + 1e-9
  # and the training tower on the attacked features: the oracle's losses on its own attacked features
  _, losses, _, _ = RT.loss_and_grads(rcfg, w, dict(rows, scene_feat=adv))
  ref_losses = g[mode + "/losses"]
  assert np.abs(np.array(losses) - ref_losses).max() < 1e-9 * max(ref_losses)
