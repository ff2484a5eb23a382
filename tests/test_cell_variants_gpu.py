# coding=utf-8
"""Every launch class of the ConvLSTM cell kernel (csrc/mvb_cell.cu launch_cell) and the training GEMMs at the row
counts the benchmark runs, against a float64 restatement of the cell on the GPU.

launch_cell() picks the kernel from the number of 128-row M tiles: below 2 * num_sms a single-CTA kernel, from there
on a CTA pair (cta_group::2 by default; two cta_group::1 CTAs with weight multicast under MVB_CELL_PAIR=1), each in
work order 1 (the four N tiles of an M tile back to back) or 0 (strided).  The small cases of tests/test_parity_gpu.py
only ever reach the single-CTA kernel.  Here each path runs on both sides of the threshold, with an odd number of M
tiles (the peer CTA of the last pair gets a tile that lies wholly past the last row) and with a ragged last tile.
Outputs are NaN-filled beforehand, with guard rows past the last row: rows and halo cells a kernel must not write are
checked to be untouched.

The comparison covers the whole batch, not a subset of samples: the float64 reference (ref_cell: im2col plus one fp64
matmul, checked against oracle/multiverse_ref_torch.convlstm_cell) takes well under a second at 38 000 rows.
Bars are the suite's: TIGHT (max |diff| / max |ref| per tensor) for c, h and the gates, GTOL for gradients."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import cases
import cell_variant_worker as worker

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TIGHT = 3e-5
GTOL = 2e-4
F16F8 = 16
BAR = {1: 2e-2, 2: TIGHT, 3: TIGHT, F16F8: TIGHT}      # plain bf16 (P = 1) misses the fp32 bar by design
HP_TOL = {1: 4e-3, 2: 2e-5, 3: 1e-6, F16F8: 1e-5}     # |operand planes of h' - h'|: what each format carries
BLOCK_M, N_TILES = 128, 4


@pytest.fixture(scope="module")
def dev():
  from multiverse_b200 import build
  build.build()
  return torch.device("cuda:0")


def T(a, dev):
  return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


# ------------------------------------------------------------------------------------------ launch classes
def num_sms():
  return torch.cuda.get_device_properties(0).multi_processor_count


def _pick_order(units, ctas):
  """pick_order() of csrc/mvb_cell.cu with no order forced."""
  back_to_back = -(-units // ctas) * N_TILES
  strided = -(-(units * N_TILES) // ctas)
  return 0 if (strided < back_to_back and units < 4 * ctas) else 1


def launch_class(h, w, ns, multicast=True):
  """(pair, work order, M tiles) that launch_cell() chooses for ns sample rows of an h x w grid."""
  sms = num_sms()
  m_tiles = -(-(ns * (h + 1) * (w + 1)) // BLOCK_M)
  if multicast and m_tiles >= 2 * sms:
    return True, _pick_order((m_tiles + 1) // 2, sms // 2), m_tiles
  return False, _pick_order(m_tiles, min(m_tiles * N_TILES, sms)), m_tiles


def pair_ns(h, w, odd_tiles=None):
  """Smallest sample-row count that selects the CTA-pair kernel, optionally with an odd (the last pair's peer tile
  lies past R) or even number of M tiles."""
  s = (h + 1) * (w + 1)
  ns = (2 * num_sms() - 1) * BLOCK_M // s + 1
  while odd_tiles is not None and launch_class(h, w, ns)[2] % 2 != int(odd_tiles):
    ns += 1
  assert launch_class(h, w, ns)[0]
  return ns


# name: (h, w, sample rows).  On a 148-SM B200: 128 / 53 rows -> single CTA in order 0 / 1; 199 rows of 18x9 ->
# pair, 296 tiles, order 1, 50-row last tile; 200 rows -> pair, 297 tiles (phantom peer tile), order 0; 54 rows of
# 36x18 -> pair, 297 tiles, order 0.
SIZES = {
    "single_18x9": lambda: (18, 9, 128),
    "single_36x18": lambda: (36, 18, pair_ns(36, 18) - 1),
    "pair_even_18x9": lambda: (18, 9, pair_ns(18, 9, odd_tiles=False)),
    "pair_odd_18x9": lambda: (18, 9, pair_ns(18, 9, odd_tiles=True)),
    "pair_odd_36x18": lambda: (36, 18, pair_ns(36, 18, odd_tiles=True)),
}
SIZES_36x18 = ["single_36x18", "pair_odd_36x18"]


def check_variant(tag, fmt, h, w, ns, errs, multicast=True):
  """The launched kernel is the one launch_class() predicts (cell_last_variant = format * 2 + pair); prints the case."""
  from multiverse_b200 import ops
  pair, order, m_tiles = launch_class(h, w, ns, multicast)
  v = ops.cell_last_variant()
  R = ns * (h + 1) * (w + 1)
  print("%-34s %dx%d ns=%-4d fmt=%-2d variant=%-2d %-6s order=%d m_tiles=%d last tile %3d rows  %s" % (
      tag, h, w, ns, fmt, v, "pair" if v % 2 else "single", order, m_tiles, R - (m_tiles - 1) * BLOCK_M,
      " ".join("%s %.2e" % kv for kv in errs.items())))
  assert v // 2 == fmt, (v, fmt)
  assert bool(v % 2) == pair, "launch_cell chose %s, the helper predicted %s" % (v % 2, pair)


# ------------------------------------------------------------------------------------------ float64 reference
def conv3x3(x, k):
  """SAME 3x3 convolution of NHWC x with HWIO k: im2col and one matmul (in x's dtype)."""
  n, h, w, c = x.shape
  xp = F.pad(x, (0, 0, 1, 1, 1, 1))
  cols = torch.cat([xp[:, dy:dy + h, dx:dx + w] for dy in range(3) for dx in range(3)], -1)
  return (cols.reshape(-1, 9 * c) @ k.reshape(9 * c, -1)).reshape(n, h, w, -1)


def ref_cell(x, c, h, kernel, biases, forget_bias=1.0):
  """(c', h', activated gates [i | j | f | o]) of oracle/multiverse_ref_torch.convlstm_cell."""
  g = conv3x3(torch.cat([x, h], -1), kernel) + biases
  gi, gj, gf, go = torch.split(g, g.shape[-1] // 4, dim=-1)
  ai, aj, af, ao = torch.sigmoid(gi), torch.tanh(gj), torch.sigmoid(gf + forget_bias), torch.sigmoid(go)
  c1 = af * c + ai * aj
  return c1, torch.tanh(c1) * ao, torch.cat([ai, aj, af, ao], -1)


def ref_fwd(d, dev, x=None, c=None, h=None, chunk=64):
  """fp64 (c', h', gates) of the whole batch on the GPU, `chunk` samples at a time (the convolution is per sample)."""
  x = d["x"] if x is None else x
  c = d["c"] if c is None else c
  h = d["h"] if h is None else h
  k, b = T(d["kernel"], dev).double(), T(d["biases"], dev).double()
  outs = [[], [], []]
  with torch.no_grad():
    for lo in range(0, x.shape[0], chunk):
      g = lambda a: (a[lo:lo + chunk] if isinstance(a, torch.Tensor) else T(a[lo:lo + chunk], dev)).double()
      for o, r in zip(outs, ref_cell(g(x), g(c), g(h), k, b)):
        o.append(r)
  return [torch.cat(o) for o in outs]


def rel(a, b):
  a, b = a.double(), b.double()
  return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


PACKED = np.array([g * 256 + t * 64 + j for t in range(4) for g in range(4) for j in range(64)])   # packed column n


def nhwc(full, ns, h, w):
  """Valid cells [ns, h, w, C] of a halo-layout buffer (or of the first R rows of a guarded one)."""
  return full[:ns * (h + 1) * (w + 1)].view(ns, h + 1, w + 1, -1)[:, :h, :w]


def check_untouched(full, ns, h, w, name):
  """Guard rows past R and the halo cells (x = w, y = h) still hold their NaN; every valid cell was written."""
  R = ns * (h + 1) * (w + 1)
  v = full[:R].reshape(ns, h + 1, w + 1, -1)
  assert bool(torch.isnan(full[R:]).all()), "%s: a kernel wrote past the last row" % name
  assert bool(torch.isnan(v[:, h]).all()) and bool(torch.isnan(v[:, :, w]).all()), "%s: a kernel wrote a halo cell" % name
  assert bool(torch.isfinite(v[:, :h, :w]).all()), "%s: valid cells not written" % name


def check_hp(r, fmt, ns, h, w, h32):
  """Only the h block of valid rows of the h' operand buffer changed, and it carries h'."""
  from multiverse_b200 import ops
  cxp = r["cxp"]
  S = (h + 1) * (w + 1)
  after = r["xn"].view(torch.uint8)
  before = r["xn_before"]
  a = after.view(-1, ns, h + 1, w + 1, after.shape[-1]).clone()
  b = before.view(-1, ns, h + 1, w + 1, before.shape[-1])
  a[:, :, :h, :w, 2 * cxp:] = b[:, :, :h, :w, 2 * cxp:]
  assert torch.equal(a, b), "cell_fwd wrote the x block, a halo cell or past the last row of its operand output"
  vals, _ = ops.operand_values(r["xn"])
  hp = vals[:ns * S, cxp:].reshape(ns, h + 1, w + 1, 256)[:, :h, :w]
  err = float((hp - h32).abs().max())
  assert err < HP_TOL[fmt], err
  return err


def test_reference_is_the_oracle_cell(dev):
  from oracle import multiverse_ref_torch as RT
  d = cases.cell_inputs(2, 7, 5, 32, 3)
  t = {k: T(v, dev).double() for k, v in d.items()}
  c0, h0 = RT.convlstm_cell(t["x"], t["c"], t["h"], t["kernel"], t["biases"])
  c1, h1, _ = ref_cell(t["x"], t["c"], t["h"], t["kernel"], t["biases"])
  assert rel(c1, c0) < 1e-12 and rel(h1, h0) < 1e-12


# ------------------------------------------------------------------------------------------ forward paths
@pytest.mark.parametrize("size", sorted(SIZES))
@pytest.mark.parametrize("fmt", [2, F16F8, 3, 1])
def test_cell_fwd_formats(dev, fmt, size):
  """Plain cell_fwd in every operand format, single CTA and CTA pair, odd and even tile counts."""
  h, w, ns = SIZES[size]()
  d = cases.cell_inputs(ns, h, w, 32, 100 + fmt)
  r = worker.run_plain(d, fmt, h, w, ns, dev, seed=fmt)
  check_untouched(r["c"], ns, h, w, "c_out"); check_untouched(r["h"], ns, h, w, "h32_out")
  c_ref, h_ref, _ = ref_fwd(d, dev)
  co, ho = nhwc(r["c"], ns, h, w), nhwc(r["h"], ns, h, w)
  errs = dict(c=rel(co, c_ref), h=rel(ho, h_ref))
  errs["hp"] = check_hp(r, fmt, ns, h, w, ho)
  check_variant("cell_fwd " + size, fmt, h, w, ns, errs)
  assert errs["c"] < BAR[fmt] and errs["h"] < BAR[fmt]


@pytest.mark.parametrize("size", SIZES_36x18)
def test_cell_fwd_row_map(dev, size):
  """c_in gathered through a row map (beam steps), repeats included."""
  h, w, ns = SIZES[size]()
  d = cases.cell_inputs(ns, h, w, 32, 7)
  perm = np.random.default_rng(7).integers(0, ns, ns).astype(np.int32)
  perm[:2] = [ns - 1, ns - 1]
  r = worker.run_plain(d, F16F8, h, w, ns, dev, row_map=T(perm, dev), seed=7)
  check_untouched(r["c"], ns, h, w, "c_out"); check_untouched(r["h"], ns, h, w, "h32_out")
  c_ref, h_ref, _ = ref_fwd(d, dev, c=d["c"][perm])
  co, ho = nhwc(r["c"], ns, h, w), nhwc(r["h"], ns, h, w)
  errs = dict(c=rel(co, c_ref), h=rel(ho, h_ref), hp=check_hp(r, F16F8, ns, h, w, ho))
  check_variant("cell_fwd row_map " + size, F16F8, h, w, ns, errs)
  assert errs["c"] < TIGHT and errs["h"] < TIGHT


def onehot_emb(ids, h, w, We, be, dev):
  """grid_emb(one_hot(ids)) in fp64: the class decoder's embedded input."""
  oh = F.one_hot(T(ids, dev).long(), h * w).double().reshape(-1, h, w, 1)
  return torch.tanh(conv3x3(oh, T(We, dev).double()) + T(be, dev).double())


def edge_ids(n, h, w, seed):
  ids = np.random.default_rng(seed).integers(0, h * w, n).astype(np.int32)
  ids[:5] = [0, w - 1, (h - 1) * w, h * w - 1, 2 * w + 2]       # corners and an interior cell
  return ids


@pytest.mark.parametrize("size", SIZES_36x18)
def test_cell_fwd_onehot_row_map(dev, size):
  """The K-row beam step: embedded one-hot input folded into table look-ups (x chunk skipped), c through a row map."""
  from multiverse_b200 import ops
  h, w, ns = SIZES[size]()
  d = cases.cell_inputs(ns, h, w, 32, 8)
  hd = cases.head_case()
  ids = edge_ids(ns, h, w, 8)
  perm = np.random.default_rng(9).integers(0, ns, ns).astype(np.int32)
  pk, xh, c_in = worker.load_inputs(d, F16F8, h, w, ns, dev)
  xf = ops.XFold(T(d["kernel"], dev), T(d["biases"], dev), T(hd["We1"], dev), T(hd["be"], dev))
  R = ops.halo_rows(ns, h, w)
  c_full, c_out = worker.guarded(R, 256, dev); h_full, h_out = worker.guarded(R, 256, dev)
  ops.cell_fwd_onehot(xh, pk, xf, T(ids, dev), c_in, c_out, h_out, None, h, w, ns, row_map=T(perm, dev))
  check_untouched(c_full, ns, h, w, "c_out"); check_untouched(h_full, ns, h, w, "h32_out")
  x = onehot_emb(ids, h, w, hd["We1"], hd["be"], dev)
  c_ref, h_ref, _ = ref_fwd(d, dev, x=x, c=d["c"][perm])
  errs = dict(c=rel(nhwc(c_full, ns, h, w), c_ref), h=rel(nhwc(h_full, ns, h, w), h_ref))
  check_variant("cell_fwd_onehot row_map " + size, F16F8, h, w, ns, errs)
  assert errs["c"] < TIGHT and errs["h"] < TIGHT


@pytest.mark.parametrize("size", SIZES_36x18)
def test_cell_fwd_onehot_fanout(dev, size):
  """First K-row beam step: one GEMM per parent row (pair-sized parent count), then K = 2 children per parent."""
  from multiverse_b200 import ops
  h, w, n = SIZES[size]()
  k = 2
  d = cases.cell_inputs(n, h, w, 32, 10)
  hd = cases.head_case()
  ids = edge_ids(n * k, h, w, 10)
  pk, xh, c_in = worker.load_inputs(d, F16F8, h, w, n, dev)
  xf = ops.XFold(T(d["kernel"], dev), T(d["biases"], dev), T(hd["We1"], dev), T(hd["be"], dev))
  R = ops.halo_rows(n * k, h, w)
  c_full, c_out = worker.guarded(R, 256, dev); h_full, h_out = worker.guarded(R, 256, dev)
  ops.cell_fwd_onehot_fanout(xh, pk, xf, T(ids, dev), c_in, c_out, h_out, h, w, n, k)
  check_untouched(c_full, n * k, h, w, "c_out"); check_untouched(h_full, n * k, h, w, "h32_out")
  x = onehot_emb(ids, h, w, hd["We1"], hd["be"], dev)
  rep = lambda a: T(np.repeat(a, k, axis=0), dev)
  c_ref, h_ref, _ = ref_fwd(d, dev, x=x, c=rep(d["c"]), h=rep(d["h"]))
  errs = dict(c=rel(nhwc(c_full, n * k, h, w), c_ref), h=rel(nhwc(h_full, n * k, h, w), h_ref))
  check_variant("cell_fwd_onehot_fanout " + size, F16F8, h, w, n, errs)
  assert errs["c"] < TIGHT and errs["h"] < TIGHT


@pytest.mark.parametrize("size", SIZES_36x18)
def test_cell_fwd_xsparse(dev, size):
  """Class encoder: the 64 scene channels at one label cell per sample added from per-sample tables."""
  from multiverse_b200 import ops
  h, w, ns = SIZES[size]()
  d = cases.cell_inputs(ns, h, w, 64, 11)
  rng = np.random.default_rng(11)
  conv = np.tanh(rng.standard_normal((7, h * w, 64))).astype(np.float32)
  frames = rng.integers(0, 7, ns).astype(np.int32)
  labels = edge_ids(ns, h, w, 12)
  labels[5] = -1                                                          # no label: no x contribution
  x = np.zeros((ns, h * w, 64), np.float32)
  for s in range(ns):
    if labels[s] >= 0:
      x[s, labels[s]] = conv[frames[s], labels[s]]
  d["x"] = x.reshape(ns, h, w, 64)
  pk, xh, c_in = worker.load_inputs(d, F16F8, h, w, ns, dev)
  xs = ops.XSparse(T(d["kernel"], dev))
  table = torch.empty((ns, 9, 1024), device=dev)
  ops.cell_xsparse_table(T(conv, dev), T(frames, dev), T(labels, dev), xs, table, h, w)
  R = ops.halo_rows(ns, h, w)
  c_full, c_out = worker.guarded(R, 256, dev); h_full, h_out = worker.guarded(R, 256, dev)
  ops.cell_fwd_xsparse(xh, pk, table, T(labels, dev), c_in, c_out, h_out, None, h, w, ns)
  check_untouched(c_full, ns, h, w, "c_out"); check_untouched(h_full, ns, h, w, "h32_out")
  c_ref, h_ref, _ = ref_fwd(d, dev)
  errs = dict(c=rel(nhwc(c_full, ns, h, w), c_ref), h=rel(nhwc(h_full, ns, h, w), h_ref))
  check_variant("cell_fwd_xsparse " + size, F16F8, h, w, ns, errs)
  assert errs["c"] < TIGHT and errs["h"] < TIGHT


@pytest.mark.parametrize("size", SIZES_36x18)
def test_cell_fwd_xdense(dev, size):
  """Regression encoder: raw 2-channel pixel offsets of up to +-1.9e3 added in fp32 in the epilogue."""
  from multiverse_b200 import ops
  h, w, ns = SIZES[size]()
  d = cases.cell_inputs(ns, h, w, 2, 13, x_scale=600.0)
  assert float(np.abs(d["x"]).max()) > 1.5e3
  pk, xh, c_in = worker.load_inputs(dict(d, x=None), F16F8, h, w, ns, dev)      # the x block is not read
  xd = ops.XDense(T(d["kernel"], dev))
  R = ops.halo_rows(ns, h, w)
  c_full, c_out = worker.guarded(R, 256, dev); h_full, h_out = worker.guarded(R, 256, dev)
  ops.cell_fwd_xdense(xh, pk, xd, T(d["x"], dev), c_in, c_out, h_out, None, h, w, ns)
  check_untouched(c_full, ns, h, w, "c_out"); check_untouched(h_full, ns, h, w, "h32_out")
  c_ref, h_ref, _ = ref_fwd(d, dev)
  errs = dict(c=rel(nhwc(c_full, ns, h, w), c_ref), h=rel(nhwc(h_full, ns, h, w), h_ref))
  check_variant("cell_fwd_xdense " + size, F16F8, h, w, ns, errs)
  assert errs["c"] < TIGHT and errs["h"] < TIGHT


def run_train_fwd(d, h, w, ns, dev):
  """cell_fwd_train (P = 2) on guarded c, h and gates buffers."""
  from multiverse_b200 import ops
  pk, xh, c_in = worker.load_inputs(d, 2, h, w, ns, dev)
  R = ops.halo_rows(ns, h, w)
  c_full, c_out = worker.guarded(R, 256, dev); h_full, h_out = worker.guarded(R, 256, dev)
  g_full, gates = worker.guarded(R, 1024, dev)
  ops.cell_fwd_train(xh, pk, c_in, c_out, h_out, None, gates, h, w, ns)
  for buf, name in ((c_full, "c_out"), (h_full, "h32_out"), (g_full, "gates_out")):
    check_untouched(buf, ns, h, w, name)
  return pk, xh, c_in, c_full, h_full, g_full


@pytest.mark.parametrize("size", SIZES_36x18)
def test_cell_fwd_train_gates(dev, size):
  """The training forward stores the activated gates in packed column order."""
  h, w, ns = SIZES[size]()
  d = cases.cell_inputs(ns, h, w, 32, 14)
  _, _, _, c_full, h_full, g_full = run_train_fwd(d, h, w, ns, dev)
  c_ref, h_ref, g_ref = ref_fwd(d, dev)
  errs = dict(c=rel(nhwc(c_full, ns, h, w), c_ref), h=rel(nhwc(h_full, ns, h, w), h_ref),
              gates=rel(nhwc(g_full, ns, h, w), g_ref[..., T(PACKED, dev)]))
  check_variant("cell_fwd_train gates_out " + size, 2, h, w, ns, errs)
  assert errs["c"] < TIGHT and errs["h"] < TIGHT and errs["gates"] < TIGHT


# ------------------------------------------------------------------------------------------ environment overrides
ENV_CASE = dict(fmt=F16F8, seed=61, cx=32)
ENV_SETTINGS = {
    "order0": ({"MVB_CELL_ORDER": "0"}, True),
    "order1": ({"MVB_CELL_ORDER": "1"}, True),
    "pair_multicast": ({"MVB_CELL_PAIR": "1"}, True),
    "no_multicast": ({"MVB_CELL_MULTICAST": "0"}, False),
}


@pytest.fixture(scope="module")
def env_default(dev):
  """In-process (default settings) run of the override shape and its fp64 reference."""
  h, w, ns = SIZES["pair_odd_18x9"]()
  d = cases.cell_inputs(ns, h, w, ENV_CASE["cx"], ENV_CASE["seed"])
  r = worker.run_plain(d, ENV_CASE["fmt"], h, w, ns, dev, seed=ENV_CASE["seed"])
  c_ref, h_ref, _ = ref_fwd(d, dev)
  return (h, w, ns), r, c_ref, h_ref


@pytest.mark.parametrize("setting", sorted(ENV_SETTINGS))
def test_cell_env_overrides_match_default(dev, env_default, setting, tmp_path):
  """Forced work orders, the multicast pair kernel and the single-CTA kernel at pair size, each in a fresh process:
  within TIGHT of fp64 and bit-identical to the default launch (order only reassigns tiles to CTAs; the single,
  cta_group::1 and cta_group::2 kernels run the same per-row K order)."""
  (h, w, ns), r, c_ref, h_ref = env_default
  env_over, pair = ENV_SETTINGS[setting]
  env = {k: v for k, v in os.environ.items() if not k.startswith("MVB_CELL_")}
  env.update(env_over)
  out = str(tmp_path / "cell.npz")
  cmd = [sys.executable, "-B", os.path.join(ROOT, "tests", "cell_variant_worker.py"), out,
         str(ENV_CASE["fmt"]), str(h), str(w), str(ns), str(ENV_CASE["seed"]), str(ENV_CASE["cx"])]
  p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
  assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
  got = np.load(out)
  v = int(got["variant"])
  c_w, h_w = torch.from_numpy(got["c"]).to(dev), torch.from_numpy(got["h"]).to(dev)
  check_untouched(c_w, ns, h, w, "c_out"); check_untouched(h_w, ns, h, w, "h32_out")
  errs = dict(c=rel(nhwc(c_w, ns, h, w), c_ref), h=rel(nhwc(h_w, ns, h, w), h_ref),
              vs_default=float(np.nanmax(np.abs(got["h"] - r["h"].cpu().numpy()))))
  print("%-34s %dx%d ns=%-4d fmt=%-2d variant=%-2d %-6s %s  %s" % (
      "cell_fwd " + setting, h, w, ns, ENV_CASE["fmt"], v, "pair" if v % 2 else "single", env_over,
      " ".join("%s %.2e" % kv for kv in errs.items())))
  assert v // 2 == ENV_CASE["fmt"] and bool(v % 2) == pair
  assert errs["c"] < TIGHT and errs["h"] < TIGHT
  assert np.array_equal(got["c"], r["c"].cpu().numpy(), equal_nan=True)
  assert np.array_equal(got["h"], r["h"].cpu().numpy(), equal_nan=True)
  assert np.array_equal(got["xn"], r["xn"].view(torch.uint8).cpu().numpy())


# ------------------------------------------------------------------------------------------ widths and refusals
@pytest.mark.parametrize("shape", [(3, 1, 1), (3, 1, 2), (2, 3, 62), (2, 5, 18)])
@pytest.mark.parametrize("fmt", [2, F16F8, 3, 1])
def test_cell_narrow_and_wide_grids(dev, fmt, shape):
  """Single-cell and single-row grids, and the widest grid the A stage admits (W = 62: 256 rows).  Three bf16
  planes fit the shared memory only up to W = 18; wider grids are refused with a message, not launched."""
  ns, h, w = shape
  d = cases.cell_inputs(ns, h, w, 32, 20 + w)
  if fmt == 3 and w > 18:
    with pytest.raises(RuntimeError, match="too large .*shared memory"):
      worker.run_plain(d, fmt, h, w, ns, dev)
    return
  r = worker.run_plain(d, fmt, h, w, ns, dev, seed=w)
  check_untouched(r["c"], ns, h, w, "c_out"); check_untouched(r["h"], ns, h, w, "h32_out")
  c_ref, h_ref, _ = ref_fwd(d, dev)
  co, ho = nhwc(r["c"], ns, h, w), nhwc(r["h"], ns, h, w)
  errs = dict(c=rel(co, c_ref), h=rel(ho, h_ref), hp=check_hp(r, fmt, ns, h, w, ho))
  check_variant("cell_fwd %dx%d" % (h, w), fmt, h, w, ns, errs)
  assert errs["c"] < BAR[fmt] and errs["h"] < BAR[fmt]


def test_cell_three_planes_width_limit(dev):
  """W = 19 is the first width whose P = 3 A ring does not fit beside three weight slots."""
  d = cases.cell_inputs(1, 2, 19, 32, 5)
  with pytest.raises(RuntimeError, match="W=19 too large"):
    worker.run_plain(d, 3, 2, 19, 1, dev)


@pytest.mark.parametrize("fmt", [2, F16F8, 3, 1])
def test_cell_refuses_w63(dev, fmt):
  d = cases.cell_inputs(1, 2, 63, 32, 6)
  with pytest.raises(RuntimeError, match="W=63 too large for the halo'd A stage"):
    worker.run_plain(d, fmt, 2, 63, 1, dev)


@pytest.mark.parametrize("hw", [(3, 3), (2, 5), (5, 2)])
def test_cell_xfold_minimum_grid(dev, hw):
  """x-fold runs from a 3x3 grid up (every cell there is a border cell) and refuses anything smaller."""
  from multiverse_b200 import ops
  h, w = hw
  ns = 6
  d = cases.cell_inputs(ns, h, w, 32, 15)
  hd = cases.head_case()
  ids = np.array([0, w - 1, (h - 1) * w, h * w - 1, (h // 2) * w + w // 2, 1], dtype=np.int32)
  pk, xh, c_in = worker.load_inputs(d, 2, h, w, ns, dev)
  xf = ops.XFold(T(d["kernel"], dev), T(d["biases"], dev), T(hd["We1"], dev), T(hd["be"], dev))
  R = ops.halo_rows(ns, h, w)
  c_full, c_out = worker.guarded(R, 256, dev); h_full, h_out = worker.guarded(R, 256, dev)
  if min(h, w) < 3:
    with pytest.raises(RuntimeError, match="at least 3x3"):
      ops.cell_fwd_onehot(xh, pk, xf, T(ids, dev), c_in, c_out, h_out, None, h, w, ns)
    assert bool(torch.isnan(c_full).all())
    return
  ops.cell_fwd_onehot(xh, pk, xf, T(ids, dev), c_in, c_out, h_out, None, h, w, ns)
  check_untouched(c_full, ns, h, w, "c_out"); check_untouched(h_full, ns, h, w, "h32_out")
  c_ref, h_ref, _ = ref_fwd(d, dev, x=onehot_emb(ids, h, w, hd["We1"], hd["be"], dev))
  errs = dict(c=rel(nhwc(c_full, ns, h, w), c_ref), h=rel(nhwc(h_full, ns, h, w), h_ref))
  check_variant("cell_fwd_onehot 3x3", 2, h, w, ns, errs)
  assert errs["c"] < TIGHT and errs["h"] < TIGHT


# ------------------------------------------------------------------------------------------ training backward
@pytest.mark.parametrize("cx", [32, 64])
def test_cell_backward_at_size(dev, cx):
  """cell_fwd_train (CTA pair) -> lstm_gates_bwd -> cell_dgrad (with and without dx) -> cell_wgrad_direct (K split
  into 5 slabs for cpad 288, 2 for cpad 320) -> unpack_cell_wgrad, against fp64 autograd of the whole batch."""
  from multiverse_b200 import ops
  h, w = 36, 18
  ns = pair_ns(h, w, odd_tiles=True)
  d = cases.cell_inputs(ns, h, w, cx, 30 + cx)
  rng = np.random.default_rng(31)
  dh = rng.standard_normal((ns, h, w, 256), dtype=np.float32)
  dc = rng.standard_normal((ns, h, w, 256), dtype=np.float32)
  pk, xh, c_in, c_full, h_full, g_full = run_train_fwd(d, h, w, ns, dev)
  check_variant("cell_fwd_train cx=%d" % cx, 2, h, w, ns, {})
  R = ops.halo_rows(ns, h, w)
  c_out, gates = c_full[:R], g_full[:R]
  t = {k: T(v, dev).double().requires_grad_(True) for k, v in d.items()}
  c1, h1, _ = ref_cell(t["x"], t["c"], t["h"], t["kernel"], t["biases"])
  ((h1 * T(dh, dev).double()).sum() + (c1 * T(dc, dev).double()).sum()).backward()
  dh_h = ops.alloc_state(ns, h, w, dev); ops.nhwc_to_halo(T(dh, dev), dh_h, h, w)
  dc_h = ops.alloc_state(ns, h, w, dev); ops.nhwc_to_halo(T(dc, dev), dc_h, h, w)
  dg = torch.zeros((2, R, 1024), dtype=torch.bfloat16, device=dev)
  dcp_full, dc_prev = worker.guarded(R, 256, dev)
  dbp = torch.zeros((1024,), device=dev)
  ops.lstm_gates_bwd(gates, c_in, c_out, dh_h, dc_h, dg, dc_prev, dbp, h, w, ns)
  check_untouched(dcp_full, ns, h, w, "dc_prev")
  errs = dict(dc_prev=rel(nhwc(dcp_full, ns, h, w), t["c"].grad))
  wd = ops.pack_dgrad(pk, T(d["kernel"], dev))
  dx_full, dxh = worker.guarded(R, pk.cpad, dev)
  ops.cell_dgrad(dg, wd, dxh, h, w, ns, need_dx=True)
  check_untouched(dx_full, ns, h, w, "dxh")
  v = nhwc(dx_full, ns, h, w)
  errs["dh"], errs["dx"] = rel(v[..., pk.cxp:], t["h"].grad), rel(v[..., :cx], t["x"].grad)
  dh_full, dxh2 = worker.guarded(R, pk.cpad, dev)
  ops.cell_dgrad(dg, wd, dxh2, h, w, ns, need_dx=False)
  check_untouched(dh_full[:, pk.cxp:], ns, h, w, "dxh h block")
  assert bool(torch.isnan(dh_full[:, :pk.cxp]).all()), "need_dx=False wrote the x block"
  errs["dh_only"] = rel(nhwc(dh_full, ns, h, w)[..., pk.cxp:], t["h"].grad)
  slabs = ops.wgrad_slabs(pk.cpad)
  assert slabs == {288: 5, 320: 2}[pk.cpad]
  dwp = torch.zeros((slabs, 1024, 9 * pk.cpad), device=dev)
  ops.cell_wgrad_direct(dg, xh, dwp, h, w, ns)
  dk = torch.empty((3, 3, cx + 256, 1024), device=dev); db = torch.empty((1024,), device=dev)
  ops.unpack_cell_wgrad(dwp, dbp, dk, db, cx)
  errs["dkernel"], errs["dbias"] = rel(dk, t["kernel"].grad), rel(db, t["biases"].grad)
  print("%-34s %dx%d ns=%-4d cpad=%d slabs=%d  %s" % ("cell backward cx=%d" % cx, h, w, ns, pk.cpad, slabs,
                                                       " ".join("%s %.2e" % kv for kv in errs.items())))
  for k, e in errs.items():
    assert e < GTOL, (k, e)


def dg_planes(R, h, w, ns, dev, seed):
  """Random two-plane bf16 gate gradients, zero on the halo cells (what lstm_gates_bwd leaves there)."""
  g = torch.Generator(device=dev).manual_seed(seed)
  v = torch.randn((R, 1024), generator=g, device=dev)
  v.view(ns, h + 1, w + 1, 1024)[:, h] = 0; v.view(ns, h + 1, w + 1, 1024)[:, :, w] = 0
  p0 = v.bfloat16()
  return torch.stack([p0, (v - p0.float()).bfloat16()])


@pytest.mark.parametrize("case", ["one_k_block", "ragged_split"])
@pytest.mark.parametrize("cx", [32, 64])
def test_cell_wgrad_direct_accumulates(dev, cx, case):
  """cell_wgrad_direct adds into dw_packed: run into Z equals Z + (run into zeros) bit for bit, and a slab whose K
  range is empty (kb_total < ksplit, or the tail of a ragged split) adds exactly nothing.  The sum over slabs matches
  the fp64 product dG^T . xh[rows + tap shift]."""
  from multiverse_b200 import ops
  h = w = 3
  S = (h + 1) * (w + 1)
  cpad = ops.cell_cpad(cx)
  slabs = ops.wgrad_slabs(cpad)
  kb = lambda n: -(-(n * S) // 32)
  ns = 1
  if case == "ragged_split":
    while not (kb(ns) > slabs and kb(ns) % slabs):
      ns += 1
  kb_total = kb(ns)
  num_kb = -(-kb_total // slabs)
  R = ns * S
  d = cases.cell_inputs(ns, h, w, cx, 40 + ns)
  _, xh, _ = worker.load_inputs(d, 2, h, w, ns, dev)
  dg = dg_planes(R, h, w, ns, dev, 41)
  a = torch.zeros((slabs, 1024, 9 * cpad), device=dev)
  ops.cell_wgrad_direct(dg, xh, a, h, w, ns)
  z = torch.randn(a.shape, generator=torch.Generator(device=dev).manual_seed(42), device=dev)
  res = z.clone()
  ops.cell_wgrad_direct(dg, xh, res, h, w, ns)
  assert torch.equal(res, z + a)
  empty = [s for s in range(slabs) if s * num_kb >= kb_total]
  assert empty or case == "ragged_split", "the case has no empty slab"
  for s in empty:
    assert torch.equal(res[s], z[s]) and float(a[s].abs().max()) == 0.0, s
  # fp64 truth: dW[n, tap * cpad + k] = sum_r dG[r, n] xh[r + (dy - 1) Wp + (dx - 1), k]
  gv = dg.double().sum(0)
  xv = ops.operand_values(xh)[0].double()
  ref = torch.zeros((1024, 9 * cpad), dtype=torch.float64, device=dev)
  for tap in range(9):
    sh = (tap // 3 - 1) * (w + 1) + (tap % 3 - 1)
    xs = torch.zeros_like(xv)
    lo, hi = max(0, -sh), min(R, R - sh)
    xs[lo:hi] = xv[lo + sh:hi + sh]
    ref[:, tap * cpad:(tap + 1) * cpad] = gv.t() @ xs
  e = rel(a.sum(0), ref)
  print("%-34s cpad=%d ns=%d kb_total=%d ksplit=%d empty slabs %s rel err %.2e" % (
      "cell_wgrad_direct " + case, cpad, ns, kb_total, slabs, empty, e))
  assert e < 1e-5
