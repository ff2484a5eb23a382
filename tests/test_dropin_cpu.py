# coding=utf-8
"""CPU tests of the drop-in boundary (host logic only - no kernel runs here).

With multiverse_b200/dropin first on sys.path the reference's callers import OUR `pred_models`
and the `tensorflow`-named shim.  The reference's own Model.get_feed_dict results are stored in
tests/golden/refexec_feed_dicts.npz (tests/golden/make_golden_refexec.py)."""
import os
import sys
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DROPIN = os.path.join(ROOT, "multiverse_b200", "dropin")
sys.path.insert(0, os.path.join(ROOT, "tests"))
import cases  # noqa: E402
FEED_GOLD = os.path.join(ROOT, "tests", "golden", "refexec_feed_dicts.npz")


@pytest.fixture()
def dropin(monkeypatch):
  monkeypatch.syspath_prepend(DROPIN)
  for m in ("tensorflow", "tensorflow.compat", "tensorflow.compat.v1", "pred_models", "pred_utils",
            "multiverse_b200.pred_models"):
    monkeypatch.delitem(sys.modules, m, raising=False)
  import tensorflow as tf
  tf.reset_default_graph()
  import pred_models
  yield tf, pred_models
  tf.reset_default_graph()


def make_args(tmp_path, **kw):
  return cases.dropin_args(**kw)


def test_model_surface_matches_reference_names(dropin, tmp_path):
  tf, pm = dropin
  args, _ = make_args(tmp_path)
  model = pm.get_model(args, gpuid=0)
  for attr in ("obs_length", "pred_length", "is_train", "obs_scene", "obs_scene_mask", "scene_feat",
               "grid_obs_labels", "grid_obs_regress", "grid_pred_labels_T", "grid_pred_regress",
               "grid_pred_decoded", "grid_pred_reg_decoded", "beam_outputs", "global_step", "N"):
    assert hasattr(model, attr), attr
  names = [v.name for v in tf.global_variables()]
  assert "global_step:0" in names
  assert "person_pred/encoder_grid_class_0/enc_grid_0/kernel:0" in names
  assert "person_pred/decoder_grid_reg_1/decoder_rnn/grid_emb/W:0" in names
  assert "person_pred/hidden2grid_decoder_grid_class_0/out_dec_grid/W:0" in names
  shapes = {v.name: tuple(v.get_shape()) for v in tf.global_variables()}
  assert shapes["person_pred/encoder_grid_reg_0/enc_grid_regress_0/kernel:0"] == (3, 3, 258, 1024)
  assert shapes["person_pred/decoder_grid_class_0/decoder_rnn/dec_grid_0/kernel:0"] == (3, 3, 288, 1024)
  n_params = sum(int(np.prod(s)) for n, s in shapes.items() if n != "global_step:0")
  assert n_params == 21337728          # SURVEY.md §8a: two scales, emb 32
  # unused scales are fetched as [] (code/pred_models.py:170-171)
  args2, _ = make_args(tmp_path, use_grids=[True, False])
  tf.reset_default_graph()
  m2 = pm.get_model(args2, gpuid=0)
  assert m2.grid_pred_decoded[1] == [] and m2.grid_pred_reg_decoded[1] == []
  with pytest.raises(AssertionError):
    a3, _ = make_args(tmp_path, use_beam_search=True, beam_size=5)     # two scales + beam (:262)
    pm.get_model(a3, gpuid=0)


def test_saver_round_trip_and_initializer(dropin, tmp_path):
  tf, pm = dropin
  args, _ = make_args(tmp_path, use_grids=[False, True])
  model = pm.get_model(args, gpuid=0)
  tf.global_variables_initializer().run()
  w0 = {k: v.copy() for k, v in model.weights().items()}
  assert any(np.abs(v).max() > 0 for k, v in w0.items() if k.endswith("kernel"))
  assert all(np.abs(v).max() == 0 for k, v in w0.items() if k.endswith("biases"))   # TF zeros init
  saver = tf.train.Saver(max_to_keep=2)
  sess = tf.Session(config=tf.ConfigProto(allow_soft_placement=True))
  path = saver.save(sess, str(tmp_path / "save" / "save"), global_step=model.global_step)
  assert tf.train.get_checkpoint_state(str(tmp_path / "save")).model_checkpoint_path == path
  for v in tf.global_variables():
    if v.dtype == "float32":
      v.assign(np.ones(v.get_shape(), dtype=np.float32))
  restore_vars = [v for v in tf.global_variables() if "global_step" not in v.name]
  tf.train.Saver(restore_vars).restore(sess, path)
  for k, v in model.weights().items():
    assert np.array_equal(v, w0[k])


def test_saver_relative_path_round_trip(dropin, tmp_path, monkeypatch):
  """The published commands pass a RELATIVE output base (`multiverse-models`, TRAINING.md:32-39): the `checkpoint`
  index must then name the file relative to its own directory, as TF's generate_checkpoint_state_proto does, so
  that get_checkpoint_state (which joins the directory back, code/pred_utils.py:186-188) finds it - train.py
  followed by test.py --load_best, and train.py --load."""
  tf, pm = dropin
  args, _ = make_args(tmp_path, use_grids=[False, True])
  model = pm.get_model(args, gpuid=0)
  tf.global_variables_initializer().run()
  w0 = {k: v.copy() for k, v in model.weights().items()}
  monkeypatch.chdir(tmp_path)
  sess = tf.Session()
  rel = os.path.join("out", "model", "00", "save", "save")
  path = tf.train.Saver().save(sess, rel, global_step=7)
  assert path == rel + "-7"
  state = tf.train.get_checkpoint_state(os.path.join("out", "model", "00", "save"))
  assert os.path.normpath(state.model_checkpoint_path) == os.path.normpath(path)
  for v in tf.global_variables():
    if v.dtype == "float32":
      v.assign(np.zeros(v.get_shape(), dtype=np.float32))
  tf.train.Saver([v for v in tf.global_variables() if "global_step" not in v.name]).restore(
      sess, state.model_checkpoint_path)
  for k, v in model.weights().items():
    assert np.array_equal(v, w0[k])
  # and from another working directory through an absolute directory name
  monkeypatch.chdir("/")
  st2 = tf.train.get_checkpoint_state(str(tmp_path / "out" / "model" / "00" / "save"))
  assert os.path.exists(st2.model_checkpoint_path + ".npz")


def test_get_feed_dict_equals_the_references(dropin, tmp_path):
  """Our vectorised Model.get_feed_dict against the reference's own method
  (code/pred_models.py:1042-1194) executed on our Model instance, on the batches code/pred_utils.py
  made of synthetic.write_npz(.., 5, seed=3) - both stored in tests/golden/refexec_feed_dicts.npz."""
  tf, pm = dropin
  g = np.load(FEED_GOLD)
  for c, kw in enumerate(cases.FEED_DICT_CONFIGS):
    tf.reset_default_graph()
    args, cfg = make_args(tmp_path, **kw)
    model = pm.get_model(args, gpuid=0)
    for b in range(2):
      batch = cases.load_batch(g, "cfg%d/batch%d/" % (c, b))
      for is_train in (False, True):
        args.device_grid_feeds = False           # the reference's feed dict, key for key
        ours = model.get_feed_dict(batch, is_train=is_train)
        assert cases.check_feed_digests(g, "cfg%d/batch%d/train%d/" % (c, b, is_train), model, ours) == \
            set(cases.feed_labels(model, ours))
        # row f-1 (default): the dense offsets are replaced by the trajectories + cell centres they came from
        args.device_grid_feeds = True
        compact = model.get_feed_dict(batch, is_train=is_train)
        used = [j for j in range(2) if args.use_grids[j]]
        if is_train:
          assert set(compact) == set(ours)       # training keeps the dense path
          continue
        assert model.obs_traj in compact and all(model.grid_obs_regress[j] not in compact for j in used)
        n_have = len(batch.data["obs_traj"])
        for j in used:
          dense = (compact[model.obs_traj][:, :, None, None, :] - compact[model.grid_centers[j]][None, None]).astype(np.float32)
          assert np.array_equal(dense[:n_have], np.asarray(ours[model.grid_obs_regress[j]], np.float32)[:n_have])
        small = compact[model.obs_traj].nbytes + sum(compact[model.grid_centers[j]].nbytes for j in used)
        big = sum(np.asarray(ours[model.grid_obs_regress[j]], np.float32).nbytes for j in used)
        assert small < big / 4        # (at batch 4; the centres are per model, the trajectories 128 B per row)
    # a batch whose dense targets do not come from its trajectories keeps the dense path
    batch.data["obs_grid_target_all_0"] = [a + 1.0 for a in batch.data["obs_grid_target_all_0"]]
    assert model.obs_traj not in model.get_feed_dict(batch, is_train=False)


def test_tf_checkpoint_bundle_reader(dropin, tmp_path):
  """SURVEY.md §8 row f-2: `Saver.restore` reads TensorFlow's tensor-bundle checkpoints (`.index` table +
  `.data-00000-of-00001`).  The files here come from the writer in tensorflow/_bundle.py, which follows the same
  published format (no TensorFlow-produced checkpoint exists in this container)."""
  tf, pm = dropin
  from tensorflow import _bundle
  assert _bundle.crc32c(b"123456789") == 0xE3069283                 # the CRC-32C check value
  rng = np.random.default_rng(3)
  tensors = {"person_pred/scene_conv1/W": rng.standard_normal((3, 3, 11, 64)).astype(np.float32),
             "person_pred/scene_conv1/b": rng.standard_normal(64).astype(np.float32),
             "person_pred/scene_conv1/W/Adadelta": np.zeros((3, 3, 11, 64), np.float32),
             "global_step": np.asarray(1234, dtype=np.int64),
             "person_pred/ids": np.arange(7, dtype=np.int32)}
  for i in range(40):                                               # several table blocks, shared key prefixes
    tensors["person_pred/filler_%02d/kernel" % i] = rng.standard_normal((i % 3 + 1, 5)).astype(np.float32)
  prefix = str(tmp_path / "model" / "save-best-1234")
  _bundle.write_bundle(prefix, tensors)
  header, entries = _bundle.read_index(prefix)
  assert header["num_shards"] == 1 and set(entries) == set(tensors)
  assert entries["person_pred/scene_conv1/W"]["shape"] == (3, 3, 11, 64) and entries["global_step"]["shape"] == ()
  back = _bundle.read_bundle(prefix)
  for k, v in tensors.items():
    assert back[k].dtype == v.dtype and np.array_equal(back[k], v), k
  # through the Saver, the way pred_utils.initialize restores a released model (code/pred_utils.py:186-198)
  (tmp_path / "model" / "checkpoint").write_text('model_checkpoint_path: "save-best-1234"\n')
  ckpt = tf.train.get_checkpoint_state(str(tmp_path / "model"))
  assert ckpt.model_checkpoint_path == prefix
  w = tf.Variable("person_pred/scene_conv1/W", (3, 3, 11, 64))
  b = tf.Variable("person_pred/scene_conv1/b", (64,))
  tf.train.Saver([w, b]).restore(None, ckpt.model_checkpoint_path)
  assert np.array_equal(w.eval(), tensors["person_pred/scene_conv1/W"])
  assert np.array_equal(b.eval(), tensors["person_pred/scene_conv1/b"])
  missing = tf.Variable("person_pred/not_there", (3,))
  with pytest.raises(KeyError):
    tf.train.Saver([missing]).restore(None, prefix)
  # a flipped byte in the index is detected by the block checksums
  raw = bytearray(open(prefix + ".index", "rb").read()); raw[10] ^= 0xFF
  open(prefix + ".index", "wb").write(bytes(raw))
  with pytest.raises(IOError):
    _bundle.read_index(prefix)


def test_tf_checkpoint_bundle_reader_on_hand_assembled_bytes(dropin, tmp_path):
  """The reader against files assembled here byte by byte from the published formats - not by the writer in
  tensorflow/_bundle.py: a LevelDB-format table (leveldb doc/table_format.md: prefix-compressed entries
  `varint shared | varint non_shared | varint value_len | key delta | value`, a restart array + count, a 5-byte
  block trailer = compression type 0 + masked CRC-32C, metaindex block, index block of BlockHandles, 48-byte footer
  ending in the magic 0xdb4775248b80fb57) holding tensor_bundle.proto messages typed out field by field
  (BundleHeaderProto under the empty key; BundleEntryProto: 1 dtype, 2 shape{2 dim{1 size}}, 4 offset, 5 size,
  6 fixed32 crc32c).  CRC and varints come from the independent implementations below."""
  tf, pm = dropin
  from tensorflow import _bundle

  def crc32c(data):                       # bitwise Castagnoli CRC, reflected polynomial 0x82F63B78
    crc = 0xFFFFFFFF
    for byte in data:
      crc ^= byte
      for _ in range(8):
        crc = (crc >> 1) ^ (0x82F63B78 if crc & 1 else 0)
    return crc ^ 0xFFFFFFFF

  assert crc32c(b"123456789") == 0xE3069283
  masked = lambda c: ((((c >> 15) | (c << 17)) & 0xFFFFFFFF) + 0xA282EAD8) & 0xFFFFFFFF

  def varint(v):
    out = bytearray()
    while v >= 0x80:
      out.append((v & 0x7F) | 0x80); v >>= 7
    out.append(v)
    return bytes(out)

  le32 = lambda v: int(v).to_bytes(4, "little")
  # ---- the data file: two tensors back to back
  a = np.arange(6, dtype=np.float32).reshape(2, 3) * 0.5 - 1.0          # "a/kernel"  DT_FLOAT [2,3] at offset 0
  step = np.asarray(4321, dtype=np.int64)                               # "global_step"  DT_INT64 [] at offset 24
  data = a.tobytes() + step.tobytes()
  # ---- protos, typed out (field tags: (field << 3) | wire type)
  header = bytes([0x08, 0x01,                     # num_shards = 1
                  0x1A, 0x02, 0x08, 0x01])        # version { producer = 1 }        (endianness LITTLE = 0: absent)
  entry_a = (bytes([0x08, 0x01,                   # dtype = DT_FLOAT (1)
                    0x12, 0x08, 0x12, 0x02, 0x08, 0x02, 0x12, 0x02, 0x08, 0x03,     # shape { dim{size 2} dim{size 3} }
                    0x28, 0x18,                   # size = 24                        (shard_id 0, offset 0: absent)
                    0x35]) + le32(masked(crc32c(a.tobytes()))))                     # crc32c, fixed32
  entry_s = (bytes([0x08, 0x09,                   # dtype = DT_INT64 (9)
                    0x12, 0x00,                   # shape {}  (scalar)
                    0x20, 0x18,                   # offset = 24
                    0x28, 0x08,                   # size = 8
                    0x35]) + le32(masked(crc32c(step.tobytes()))))

  def block(entries):
    body, prev = bytearray(), b""
    for key, value in entries:                    # one restart point at 0: keys after it are prefix-compressed
      shared = 0
      while shared < min(len(prev), len(key)) and prev[shared] == key[shared]:
        shared += 1
      body += varint(shared) + varint(len(key) - shared) + varint(len(value)) + key[shared:] + value
      prev = key
    body += le32(0) + le32(1)                     # restart offsets, number of restarts
    return bytes(body)

  def with_trailer(blk):
    return blk + b"\x00" + le32(masked(crc32c(blk + b"\x00")))

  # keys in bytewise order: "" < "a/kernel" < "global_step"
  data_block = block([(b"", header), (b"a/kernel", entry_a), (b"global_step", entry_s)])
  meta_block = block([])
  off_meta = len(data_block) + 5
  index_block = block([(b"h", varint(0) + varint(len(data_block)))])    # separator key >= "global_step"
  off_index = off_meta + len(meta_block) + 5
  footer = varint(off_meta) + varint(len(meta_block)) + varint(off_index) + varint(len(index_block))
  footer += b"\x00" * (40 - len(footer)) + (0xDB4775248B80FB57).to_bytes(8, "little")
  table = with_trailer(data_block) + with_trailer(meta_block) + with_trailer(index_block) + footer
  prefix = str(tmp_path / "hand" / "model.ckpt-4321")
  os.makedirs(os.path.dirname(prefix))
  open(prefix + ".index", "wb").write(table)
  open(prefix + ".data-00000-of-00001", "wb").write(data)
  assert _bundle.is_bundle(prefix)
  hdr, entries = _bundle.read_index(prefix)
  assert hdr["num_shards"] == 1 and set(entries) == {"a/kernel", "global_step"}
  assert entries["a/kernel"]["shape"] == (2, 3) and entries["global_step"]["shape"] == ()
  back = _bundle.read_bundle(prefix)
  assert back["a/kernel"].dtype == np.float32 and np.array_equal(back["a/kernel"], a)
  assert back["global_step"].dtype == np.int64 and int(back["global_step"]) == 4321
  # and the other way round: what the module's writer produces parses with the spec-level walk used above
  _bundle.write_bundle(str(tmp_path / "hand" / "w"), {"a/kernel": a})
  raw = open(str(tmp_path / "hand" / "w") + ".index", "rb").read()
  assert raw[-8:] == (0xDB4775248B80FB57).to_bytes(8, "little") and len(raw) >= 48


def test_forward_graph_cache_policy_without_a_gpu(monkeypatch):
  """Host logic of ConvRNNEngine.forward_graph with the CUDA pieces stubbed: a signature runs eagerly the first
  time, is captured the second time (one graph per independent chain) and replayed afterwards; at most GRAPH_CACHE graphs are kept (oldest evicted);
  replacing the weights drops them all."""
  import torch
  from multiverse_b200 import engine as E

  class FakeGraph(object):
    replays = 0
    def replay(self):
      FakeGraph.replays += 1
    def capture_begin(self, **kw): pass
    def capture_end(self): pass

  class FakeStream(object):
    def __init__(self, *a, **k): pass
    def wait_stream(self, other): pass
    def wait_event(self, ev): pass
    def record_event(self): return object()

  class FakeCtx(object):
    def __init__(self, g, **kw): pass
    def __enter__(self): return self
    def __exit__(self, *a): return False

  monkeypatch.setattr(torch.cuda, "CUDAGraph", FakeGraph)
  monkeypatch.setattr(torch.cuda, "graph", FakeCtx)
  monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
  monkeypatch.setattr(torch.cuda, "Stream", FakeStream)
  monkeypatch.setattr(torch.cuda, "stream", lambda s: FakeCtx(None))
  monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: FakeStream())
  eng = E.ConvRNNEngine.__new__(E.ConvRNNEngine)
  eng.cfg = types.SimpleNamespace(pred_len=12, scene_grids=[(2, 2), (1, 1)], use_grids=[True, False])
  eng.device, eng.cell_events, eng._graphs, eng._graph_seen, eng._bufs = torch.device("cpu"), None, {}, set(), {}
  calls = []

  def fake_forward(feeds, tp, on_output=None, branches=None):
    calls.append((tuple(feeds["obs_scene"].shape), tp, None if branches is None else tuple(branches)))
    out = dict(grid_pred_decoded=[None, []], grid_pred_reg_decoded=[None, []], beam_outputs=None)
    if branches is None or ("class", 0) in branches:
      out["grid_pred_decoded"][0] = ("class", len(calls))
      if on_output: on_output("grid_pred_decoded", 0, out["grid_pred_decoded"][0])
    if branches is None or ("reg", 0) in branches:
      out["grid_pred_reg_decoded"][0] = ("reg", len(calls))
      out["_offs"] = {0: "offs"}
      if on_output: on_output("grid_pred_reg_decoded", 0, out["grid_pred_reg_decoded"][0])
    return out
  eng.forward = fake_forward

  def feeds(n):
    return dict(scene_feat=torch.zeros(3, 4, 4, 11), obs_scene=torch.zeros(n, 8, dtype=torch.int32),
                grid_obs_labels=[torch.zeros(n, 8, dtype=torch.int32), None],
                grid_obs_regress=[torch.zeros(n, 8, 2, 2, 2), None])

  eng.forward_graph(feeds(2))                      # first sight: eager
  assert len(calls) == 1 and not eng._graphs and FakeGraph.replays == 0
  seen = []
  out = eng.forward_graph(feeds(2), on_output=lambda name, i, t: seen.append(name))
  # second sight: eager warm-up, then one capture per chain (class, regression), then one replay per chain
  assert [c[2] for c in calls[1:]] == [None, (("class", 0),), (("reg", 0),)]
  assert len(eng._graphs) == 1 and FakeGraph.replays == 2
  assert out["grid_pred_decoded"] == [("class", 3), []] and out["grid_pred_reg_decoded"] == [("reg", 4), []]
  assert out["_offs"] == {0: "offs"} and sorted(seen) == ["grid_pred_decoded", "grid_pred_reg_decoded"]
  eng.forward_graph(feeds(2)); eng.forward_graph(feeds(2), pred_len=12)
  assert len(calls) == 4 and FakeGraph.replays == 6              # pure replays (pred_len default == 12)
  eng.forward_graph(feeds(2), pred_len=17)         # another rollout length is another signature
  assert len(calls) == 5 and len(eng._graphs) == 1
  f5 = feeds(2); f5["scene_feat"] = torch.ones(5, 4, 4, 11)       # another frame count, same 64-frame bucket
  eng.forward_graph(f5)
  assert len(calls) == 5 and FakeGraph.replays == 8
  static_sf = next(iter(eng._graphs.values()))[1]["scene_feat"]
  assert static_sf.shape[0] == 64 and bool((static_sf[:5] == 1).all()) and bool((static_sf[5:] == 0).all())
  for n in range(3, 3 + eng.GRAPH_CACHE + 1):      # more signatures than the cache holds
    eng.forward_graph(feeds(n)); eng.forward_graph(feeds(n))
  assert len(eng._graphs) == eng.GRAPH_CACHE
  assert not any(dict((e[0], e[1]) for e in k[2:])["obs_scene"] == (2, 8) for k in eng._graphs)   # n = 2 was evicted
  eng.scene_w = eng.scales = None
  eng.cfg = types.SimpleNamespace(pred_len=12, scene_grid_strides=[], scene_grids=[], use_grids=[])
  eng.planes = 2
  eng.set_weights({})
  assert not eng._graphs


def test_session_run_leaves_no_reference_cycle_on_the_results(monkeypatch):
  """The fetched arrays must die with the caller's last reference (their pinned blocks are reused then), not at
  the next cyclic-GC pass."""
  import gc
  import weakref
  monkeypatch.syspath_prepend(os.path.join(ROOT, "multiverse_b200", "dropin"))
  for m in ("tensorflow",):
    monkeypatch.delitem(sys.modules, m, raising=False)
  import tensorflow as tf

  class Owner(object):
    def _run(self, handles, feed):
      return [np.zeros(4) + i for i in range(len(handles))]

  class H(object):
    def __init__(self, owner):
      self.owner = owner

  owner = Owner()
  gc.disable()
  try:
    out = tf.Session().run([H(owner), [H(owner), H(owner)]], {})
    assert out[1][1][0] == 2.0
    refs = [weakref.ref(out[0]), weakref.ref(out[1][0])]
    del out
    assert all(r() is None for r in refs)
  finally:
    gc.enable()


def test_multiview_feed_dict_equals_simaugs(dropin, tmp_path):
  """The extra-view feeds of a multiview_train batch (obs_scene_extra, grid_*_extra) against SimAug's own
  Model.get_feed_dict (SimAug/code/pred_models.py:1457-1560) executed on our Model instance (stored in
  tests/golden/refexec_feed_dicts.npz), key for key on every placeholder that method fills."""
  tf, pm = dropin
  tf.reset_default_graph()
  args, cfg, model, batch = cases.multiview_feed_case(pm)
  ns = len(cfg.scene_grids)
  ours = model.get_feed_dict(batch, is_train=True)
  theirs = cases.check_feed_digests(np.load(FEED_GOLD), "multiview/", model, ours)     # theirs <= ours, values equal
  extra_keys = [model.obs_scene_extra] + [p for j in range(ns) if cfg_use(args, j) for p in
                                          (model.grid_obs_labels_extra[j], model.grid_pred_labels_T_extra[j],
                                           model.grid_pred_regress_extra[j], model.grid_obs_regress_extra[j])]
  labels = cases.feed_labels(model, {k: None for k in extra_keys})
  assert set(labels) <= theirs


def cfg_use(args, j):
  return bool(args.use_grids[j])
