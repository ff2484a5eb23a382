# coding=utf-8
"""In-tree nvcc build of libmultiverse_b200.so (sm_100a only; no fallback arch).

``python -m multiverse_b200.build`` or ``multiverse_b200.build.build()``.
The .so and the objects under build/ are git-ignored build products.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmultiverse_b200.so")
OBJ = os.path.join(HERE, "build")
SOURCES = ["mvb_api.cu", "mvb_cell.cu", "mvb_layout.cu", "mvb_scene.cu", "mvb_gnn.cu",
           "mvb_head.cu", "mvb_beam.cu", "mvb_train.cu", "mvb_train2.cu", "mvb_metrics.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def _nvcc():
  for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
    if cand and (os.path.sep not in cand or os.path.exists(cand)):
      return cand
  raise RuntimeError("nvcc not found")


def _stamp(paths):
  h = hashlib.sha1()
  for p in sorted(paths):
    with open(p, "rb") as f:
      h.update(f.read())
  h.update(" ".join(NVCC_FLAGS).encode())
  return h.hexdigest()


def sources():
  return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def build(force=False, verbose=False):
  """Compile every .cu into an object and link the shared library (skips if up to date).  Serialised across
  processes with a lock file: the ranks of a torchrun job all call this.  An up-to-date library is returned
  without writing anything, so a built tree may be read-only."""
  import fcntl
  if not force and _up_to_date(_stamp(_deps())):
    return LIB
  os.makedirs(OBJ, exist_ok=True)
  with open(os.path.join(OBJ, ".lock"), "w") as lock:
    fcntl.flock(lock, fcntl.LOCK_EX)
    try:
      return _build_locked(force, verbose)
    finally:
      fcntl.flock(lock, fcntl.LOCK_UN)


def _deps():
  deps = sources() + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
  deps.append(os.path.join(HERE, "..", "include", "multiverse_b200.h"))
  return deps


def _up_to_date(stamp):
  stamp_file = os.path.join(OBJ, "stamp")
  if not (os.path.exists(LIB) and os.path.exists(stamp_file)):
    return False
  with open(stamp_file) as f:
    return f.read().strip() == stamp


def _build_locked(force, verbose):
  srcs = sources()
  stamp = _stamp(_deps())
  stamp_file = os.path.join(OBJ, "stamp")
  if not force and _up_to_date(stamp):
    return LIB
  os.makedirs(OBJ, exist_ok=True)
  nvcc = _nvcc()

  def compile_one(src):
    obj = os.path.join(OBJ, os.path.basename(src)[:-3] + ".o")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
      raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
    if verbose:
      sys.stderr.write(r.stderr)
    return obj

  with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
    objs = list(ex.map(compile_one, srcs))
  cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a",
                                               "-lcudart_static", "-lpthread", "-ldl", "-lrt"]
  r = subprocess.run(cmd, capture_output=True, text=True)
  if r.returncode != 0:
    raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
  with open(stamp_file, "w") as f:
    f.write(stamp)
  return LIB


if __name__ == "__main__":
  print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
