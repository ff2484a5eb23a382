# coding=utf-8
"""One plain ConvLSTM cell launch in a process of its own (see tests/test_cell_variants_gpu.py).

MVB_CELL_ORDER, MVB_CELL_PAIR and MVB_CELL_MULTICAST are read once per process, so every setting of them needs a
fresh interpreter.  Usage:  cell_variant_worker.py OUT.npz FMT H W NS SEED CX.  Writes the guarded fp32 outputs, the
bytes of the operand buffer that received h', and the variant code of the launch to OUT.npz.

run_plain() is also what the test calls in-process, so both sides run the same code."""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.dirname(HERE), HERE):
  if p not in sys.path:
    sys.path.insert(0, p)

GUARD = 256     # trailing rows past R: two M tiles, as far as the phantom tile of a CTA pair reaches


def guarded(rows, cols, dev):
  """NaN-filled fp32 [rows + GUARD, cols] and the view of its first `rows` rows that a kernel receives."""
  full = torch.full((rows + GUARD, cols), float("nan"), dtype=torch.float32, device=dev)
  return full, full[:rows]


def prefilled_xh(ns, h, w, cpad, fmt, dev, seed):
  """Operand buffer for h' whose every byte is random: bytes the kernel must not write stay recognisable."""
  from multiverse_b200 import ops
  xh = ops.alloc_xh(ns, h, w, cpad, fmt, dev)
  g = torch.Generator(device=dev).manual_seed(seed)
  b = xh.view(torch.uint8)
  b.copy_(torch.randint(0, 256, b.shape, generator=g, device=dev, dtype=torch.uint8))
  return xh


def load_inputs(d, fmt, h, w, ns, dev):
  """PackedCell, operand planes (x block unless d["x"] is None, h block) and halo c state of cases.cell_inputs
  arrays."""
  from multiverse_b200 import ops
  T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
  pk = ops.PackedCell(T(d["kernel"]), T(d["biases"]), fmt)
  xh = ops.alloc_xh(ns, h, w, pk.cpad, fmt, dev)
  if d["x"] is not None:
    ops.nhwc_to_planes(T(d["x"]), xh, 0, h, w)
  ops.nhwc_to_planes(T(d["h"]), xh, pk.cxp, h, w)
  c_in = ops.alloc_state(ns, h, w, dev)
  ops.nhwc_to_halo(T(d["c"]), c_in, h, w)
  return pk, xh, c_in


def run_plain(d, fmt, h, w, ns, dev, row_map=None, seed=0):
  """cell_fwd on guarded outputs.  Returns the full (guarded) c and h buffers, the h' operand buffer, its bytes before
  the launch, and the variant code of the launch."""
  from multiverse_b200 import ops
  pk, xh, c_in = load_inputs(d, fmt, h, w, ns, dev)
  R = ops.halo_rows(ns, h, w)
  c_full, c_out = guarded(R, 256, dev)
  h_full, h_out = guarded(R, 256, dev)
  xn = prefilled_xh(ns, h, w, pk.cpad, fmt, dev, seed + 1)
  before = xn.view(torch.uint8).clone()
  ops.cell_fwd(xh, pk, c_in, c_out, h_out, xn, h, w, ns, row_map=row_map)
  torch.cuda.synchronize()
  return dict(c=c_full, h=h_full, xn=xn, xn_before=before, variant=ops.cell_last_variant(), cxp=pk.cxp)


def main():
  out, fmt, h, w, ns, seed, cx = sys.argv[1], *map(int, sys.argv[2:])
  import cases
  from multiverse_b200 import build
  build.build()
  dev = torch.device("cuda:0")
  r = run_plain(cases.cell_inputs(ns, h, w, cx, seed), fmt, h, w, ns, dev, seed=seed)
  np.savez(out, c=r["c"].cpu().numpy(), h=r["h"].cpu().numpy(), xn=r["xn"].view(torch.uint8).cpu().numpy(),
           variant=np.int64(r["variant"]))


if __name__ == "__main__":
  main()
