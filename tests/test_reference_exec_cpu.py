# coding=utf-8
"""Pins the oracle on an EXECUTION of the reference's own graph code.

``oracle/tf1_eager`` imports the unmodified ``code/pred_models.py`` of the original project against an eager,
torch-fp64-backed stand-in for the TensorFlow-1.15 symbols it uses and runs ``Model.__init__ / build_forward /
build_loss`` and ``Trainer.__init__`` as written; tests/golden/make_golden_refexec.py stored what that run returned
(tests/golden/refexec_forward.npz).  These tests assert that ``oracle/multiverse_ref.py`` equals it (fp64, <=1e-12;
ids identical) - the wiring of code/pred_models.py:123-308, 311-471, 474-806, 808-909, 961-1040, 1197-1251,
1636-1717 is therefore pinned on executed reference code, not a restatement; only the per-op TF semantics underneath
stay restated (and torch-anchored in test_oracle_cpu.py).  Large outputs are compared on the stored sample
(cases.ref_sample), relative to the largest magnitude of the whole array.
"""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import cases  # noqa: E402
from oracle import multiverse_ref as R  # noqa: E402

TOL = 1e-12


@pytest.fixture(scope="module")
def gold():
  return np.load(os.path.join(ROOT, "tests", "golden", "refexec_forward.npz"))


def rel(ours, g, key):
  """max |sample(ours) - stored sample| over the reference array's largest magnitude."""
  ours = np.asarray(ours, np.float64)
  assert ours.shape == tuple(g[key + "/shape"]), key
  return float(np.abs(cases.ref_sample(ours) - g[key]).max() / max(float(g[key + "/absmax"]), 1e-300))


def check_forward(gold, name):
  over, seed = cases.REFEXEC_FORWARD[name]
  cfg = R.default_config(**over)
  w, f = R.make_weights(cfg, seed), R.make_inputs(cfg, seed)
  assert float(gold[name + "/checksum"]) == cases.checksum(*w.values()) + cases.checksum(f["scene_feat"], f["traj"])
  ref = R.forward(cfg, w, f, np.float64)
  assert set(str(v) for v in gold[name + "/variables"]) - {"global_step"} == set(w.keys())     # TF variable names, §8a
  for i in range(len(cfg.scene_grids)):
    if not cfg.use_grids[i]:
      # the reference fetches [] for an unused scale (:170-171): nothing stored
      assert not any(k.startswith("%s/grid_pred_decoded_%d" % (name, i)) for k in gold.files)
      continue
    for k in ("grid_pred_decoded", "grid_pred_reg_decoded", "scene_convs"):
      assert rel(ref[k][i], gold, "%s/%s_%d" % (name, k, i)) < TOL, (k, i)
  if cfg.use_beam_search:
    lg, ids, lp = ref["beam_outputs"]
    assert gold[name + "/beam_ids"].dtype == np.int32 and np.array_equal(ids, gold[name + "/beam_ids"])
    assert rel(lg, gold, name + "/beam_logits") < TOL
    assert np.abs(lp - gold[name + "/beam_logprobs"]).max() < 1e-11
  else:
    assert name + "/beam_ids" not in gold.files and ref["beam_outputs"] is None
  return ref


def test_reference_beam_k5_plain_equals_oracle_and_golden(gold):
  """Coarse 18x9 grid, K=5 plain beam (no penalty, fix_num_timestep=0): the reference's own
  grid_decoder_beam_search + back-trace, and the committed rollout golden made from it."""
  out = check_forward(gold, "beam_k5_plain")
  g = np.load(os.path.join(ROOT, "tests", "golden", "rollout_beam_k5_plain.npz"))
  assert str(g["source"]) == "reference_exec"
  assert np.array_equal(g["beam_ids"], out["beam_outputs"][1])
  assert np.abs(g["beam_logprobs"] - out["beam_outputs"][2]).max() < 1e-11
  assert np.abs(g["logits_1"] - out["grid_pred_decoded"][1]).max() < 1e-6     # stored as fp32


def test_reference_beam_k20_diverse_equals_oracle(gold):
  """K=20 diverse beam (gamma 0.01, first step's scores zeroed) - the multifuture_inference.py
  configuration (TESTING.md:84-93) - on the coarse grid with 3 trajectories."""
  check_forward(gold, "beam_k20_diverse")


def test_reference_greedy_two_scale_equals_oracle(gold):
  """Both scales, greedy class decoder with graph attention + regression decoder (test.py path)."""
  assert R.default_config(**cases.REFEXEC_FORWARD["greedy_two_scale"][0]).scene_grids == [(12, 8), (6, 4)]
  check_forward(gold, "greedy_two_scale")


def test_reference_ragged_pred_length_and_no_gnn(gold):
  """use_gnn off (the reference then hands the raw state to the cell)."""
  check_forward(gold, "no_gnn")


def test_reference_training_step_equals_oracle(gold):
  """Model.build_loss + Trainer.__init__ executed: total / class / Huber / wd losses, the clipped
  gradient of every trainable variable (tf.gradients -> clip_by_value +-10, :1698-1705) and one
  Adadelta train_op (:1672,:1716) against the oracle's torch-autograd restatement and the
  closed-form update the CUDA optimizer kernel implements."""
  from oracle import multiverse_ref_torch as RT
  over, seed, kw = cases.REFEXEC_TRAIN
  cfg = R.default_config(**over, **kw)
  w, f = R.make_weights(cfg, seed), R.make_inputs(cfg, seed)
  assert float(gold["train/checksum"]) == cases.checksum(*w.values()) + cases.checksum(f["scene_feat"], f["traj"])
  tot, losses, wd, grads = RT.loss_and_grads(cfg, w, f)
  assert abs(float(gold["train/loss"]) - tot) < 1e-11 * abs(tot)
  assert abs(float(gold["train/wd_loss"]) - wd) < 1e-12 * wd
  assert np.abs(gold["train/pred_grid_loss"] - np.array(losses)).max() < 1e-11
  assert set(k[len("train/grad/"):] for k in gold.files if k.startswith("train/grad/") and "/shape" not in k
             and "/absmax" not in k) == set(w.keys())
  lr = 0.2 * 1.0 * 0.95 ** 0        # init_lr * emb_lr * decay^(floor(step/decay_steps)), step 0
  for k, g in grads.items():
    gc = np.clip(g, -10.0, 10.0)
    key = "train/grad/" + k
    assert tuple(gold[key + "/shape"]) == gc.shape, k
    assert np.abs(gold[key] - cases.ref_sample(gc, 1024)).max() <= 1e-10 * max(np.abs(gc).max(), 1e-30), k
    acc = 0.05 * gc * gc                                  # rho=.95, zero slots, eps=1e-8
    upd = np.sqrt(1e-8) / np.sqrt(acc + 1e-8) * gc
    want = w[k].astype(np.float64) - lr * upd
    assert np.abs(gold["train/updated/" + k] - cases.ref_sample(want, 1024)).max() < 1e-12, k
  assert int(gold["train/global_step"]) == 1
