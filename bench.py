# coding=utf-8
"""Benchmark of the Multiverse ConvRNN hot path on B200 (contract: see the task statement).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c4|c3|c5] [--impl reference] [--dump-outputs DIR]
  (N>1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...)

A "step" is one pass of the hot path over one batch of synthetic trajectories
(multiverse_b200/synthetic.py):
  c4 (default, the configuration BASELINE.json's metric is quoted on): obs8 -> pred12, K=20
      diverse beam (gamma 0.01, fix_num_timestep 1) on the 36x18 grid + greedy offset decoder,
      global batch 512, sharded over the ranks (strong scaling, no data-path collective).
  c3: greedy two-scale 36x18 + 18x9 with graph attention, global batch 256.
  c5: train.py step (fwd + loss + BPTT + all-reduce + clip + Adadelta), two scales, global batch 1024.
Prints ONE JSON line on rank 0.  Without --workload the line is c4's and carries the c3 and c5 records of the same
invocation (same N, same process group) under "extra", c5 with its NCCL all-reduce time / bus bandwidth and, for
N >= 2, the data-parallel equivalence self-check (ranks x shards == one rank x full batch).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

# the benchmark runs from a built tree that may be read-only: compile no bytecode into it
sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "trajectories/sec (obs8->pred12, K=20)"
WORKLOADS = {
    "c4": dict(global_batch=512, cfg=dict(use_grids=[True, False], use_beam_search=True, beam_size=20,
                                         diverse_beam=True, diverse_gamma=0.01, fix_num_timestep=1),
               desc="multifuture K=20 diverse beam, 36x18 grid, + greedy offset decoder"),
    "c3": dict(global_batch=256, cfg=dict(use_grids=[True, True]),
               desc="greedy two-scale 36x18+18x9, graph attention, class+offset heads"),
    "c5": dict(global_batch=1024, train=True, micro_batch=128,
               cfg=dict(use_grids=[True, True], is_train=True, grid_loss_weight=1.0, grid_reg_loss_weight=0.1,
                        wd=0.001, clip_gradient_norm=10.0),
               desc="train.py step: fwd + CE/Huber/wd loss + BPTT + clip + Adadelta, two scales, "
                    "data-parallel (one NCCL all-reduce of the 85 MB gradient bucket)"),
}


def cell_flops(h, w, cx):
  """Algorithmic FLOPs of one cell step per sample row (SURVEY.md §8d): 2*HW*9*(Cx+Ch)*4Ch."""
  return 2.0 * h * w * 9 * (cx + 256) * 1024


def flops_per_trajectory(cfg):
  tot = 0.0
  for i, (h, w) in enumerate(cfg.scene_grids):
    if not cfg.use_grids[i]:
      continue
    k = cfg.beam_size if cfg.use_beam_search else 1
    tot += cfg.obs_len * (cell_flops(h, w, 64) + cell_flops(h, w, 2))
    tot += cfg.pred_len * (k * cell_flops(h, w, cfg.emb_size) + cell_flops(h, w, cfg.emb_size))
  return tot


class ClockSampler(object):
  """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
  Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
       "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
       "clocks_event_reasons.sw_power_cap")

  def __init__(self, index):
    self.index, self.rows, self.proc = index, [], None

  def start(self):
    try:
      self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                    "--format=csv,noheader,nounits", "-lms", "200"],
                                   stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      threading.Thread(target=self._read, daemon=True).start()
    except Exception:
      self.proc = None

  def _read(self):
    for line in self.proc.stdout:
      self.rows.append([c.strip() for c in line.split(",")])

  def stop(self):
    if self.proc is None:
      return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
    self.proc.terminate()
    sm, mx, reasons, watts = [], None, set(), []
    for r in self.rows:
      try:
        sm.append(float(r[1])); mx = float(r[2])
      except Exception:
        continue
      try:
        watts.append(float(r[3]))
      except Exception:
        pass
      for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
        if v.lower().startswith("active"):
          reasons.add(name)
    return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=mx, samples=len(sm),
                reasons=sorted(reasons), power_w=float(np.median(watts)) if watts else None)


def load_peaks():
  p = os.path.join(ROOT, "MEASURED_PEAKS.json")
  if os.path.exists(p):
    d = json.load(open(p))
    return dict(bf16=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                hbm=d["hbm_gbs"], source="measured (MEASURED_PEAKS.json)")
  return dict(bf16=1590.0, bf16_sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


def cpu_reference_run(cfg_over, n_sample, seed, repeats=1):
  """The reference algorithm on the host cores: torch-CPU fp32 restatement of
  code/pred_models.py (oracle/multiverse_ref_torch.py; TF 1.15 is not installable).  Returns
  (trajectories/sec, seconds, threads)."""
  from multiverse_b200 import synthetic
  from oracle import multiverse_ref_torch as RT
  # all host threads up to 32: on the 128-thread GPU boxes more threads make the oneDNN convolutions of
  # this small-batch recurrent model SLOWER (profiles/r01_bench.json: 16-32 threads are the optimum)
  threads = int(os.environ.get("MVB_CPU_THREADS", "0")) or min(32, os.cpu_count() or 1)
  torch.set_num_threads(threads)
  cfg = synthetic.make_config(batch_size=n_sample, **cfg_over)
  w = synthetic.make_weights(cfg, seed)
  f = synthetic.make_feeds(cfg, n_sample, seed)
  t0 = time.perf_counter()
  for _ in range(repeats):
    RT.forward(cfg, w, f)
  dt = (time.perf_counter() - t0) / repeats
  return n_sample / dt, dt, threads


def run_reference(args, wl):
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return
  n_sample = 8          # CPU trajectories/s is batch-independent once the cores are busy; stated in `config`
  for _ in range(args.warmup):
    cpu_reference_run(wl["cfg"], n_sample, 1)
  vals = []
  for _ in range(args.steps):
    v, dt, threads = cpu_reference_run(wl["cfg"], n_sample, 1)
    vals.append((v, dt))
  tot_t = sum(d for _, d in vals)
  value = n_sample * len(vals) / tot_t
  line = dict(impl="reference", metric=METRIC, value=value, unit="trajectories/s", n_gpus=args.gpus,
              steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * tot_t / len(vals),
              higher_is_better=True, scaling="strong", vs_baseline=None, dtype="f32", data="synthetic",
              config=dict(workload=args.workload + ": " + wl["desc"], global_batch=wl["global_batch"],
                          sample_per_step=n_sample, obs_len=8, pred_len=12,
                          note="same workload as the b200 arm; each CPU step is a bounded sample of %d trajectories of "
                               "the %d-trajectory batch (the CPU rate does not depend on the batch size)"
                               % (n_sample, wl["global_batch"])),
              cpu_baseline=dict(value=value, unit="trajectories/s", cores=threads, kind="port",
                                sample="%d trajectories per step through the torch-CPU restatement of "
                                       "code/pred_models.py (TF 1.15 not installable)" % n_sample),
              e2e=dict(value=value, unit="trajectories/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
  print(json.dumps(line), flush=True)


DUMP_MAX_ELEMENTS = 2 << 20      # per array: 8 MB in float32; the five largest outputs stay under 64 MB together


def dump_outputs(out_dir, arrays):
  """Writes each named output as out_dir/<name>.npy: float32 stays float32, everything else (ids included) becomes
  float64.  An array of more than DUMP_MAX_ELEMENTS elements is replaced by a sample of its flattened elements at
  sorted random positions drawn from a generator seeded with the name and the size, so two runs of the same
  arguments store the same positions."""
  import zlib
  os.makedirs(out_dir, exist_ok=True)
  for name, t in arrays.items():
    flat = t.detach().reshape(-1) if torch.is_tensor(t) else torch.from_numpy(np.ascontiguousarray(t)).reshape(-1)
    n = flat.numel()
    if n > DUMP_MAX_ELEMENTS:
      rng = np.random.default_rng(zlib.crc32(("%s/%d" % (name, n)).encode()))
      idx = np.unique(rng.integers(0, n, size=DUMP_MAX_ELEMENTS))
      flat = flat[torch.from_numpy(idx).to(flat.device)]
    a = flat.cpu().numpy()
    np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))


def setup():
  """Device + (for N > 1) the NCCL process group of this rank: (world, rank, local, dev, dist or None)."""
  from multiverse_b200 import build
  build.build()
  world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  torch.cuda.set_device(local)
  dev = torch.device("cuda", local)
  dist = None
  if world > 1:
    import torch.distributed as dist
    dist.init_process_group("nccl", device_id=dev)
  return world, rank, local, dev, dist


def ddp_equivalence(ctx):
  """Self-check of the data-parallel training path on this run's own ranks: G ranks x 4 trajectories with the NCCL
  all-reduce against rank 0's single-rank step on the 4G-trajectory batch (losses are means over equal shards, the
  weight-decay term is batch independent: SURVEY.md section 8e).  Returns the three errors on rank 0."""
  from multiverse_b200 import synthetic
  from multiverse_b200.train_engine import TrainEngine
  world, rank, local, dev, dist = ctx
  n = 4 * world
  kw = dict(use_grids=[False, True], is_train=True, grid_loss_weight=1.0, grid_reg_loss_weight=0.1, wd=0.001,
            clip_gradient_norm=10.0)
  w = synthetic.make_weights(synthetic.make_config(batch_size=n, **kw), 3)
  f = synthetic.make_feeds(synthetic.make_config(batch_size=n, **kw), n, 3, with_pred=True)
  g = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)

  def feeds_of(r, wsize):
    sh = synthetic.shard_feeds(f, r, wsize)
    return {k: ([g(a) for a in v] if isinstance(v, list) else g(v)) for k, v in sh.items() if k != "traj"}
  eng = TrainEngine(synthetic.make_config(batch_size=n // world, **kw), {k: torch.from_numpy(v) for k, v in w.items()}, dev, 2)
  losses, _ = eng.train_step(feeds_of(rank, world), 0.2, dist)
  res = None
  if rank == 0:
    full = TrainEngine(synthetic.make_config(batch_size=n, **kw), {k: torch.from_numpy(v) for k, v in w.items()}, dev, 2)
    l_full, _ = full.train_step(feeds_of(0, 1), 0.2, None)
    moved = max(float((full.params[k].cpu() - torch.from_numpy(w[k])).abs().max()) for k in eng.names)
    res = dict(loss_rel=float((losses - l_full).abs().max() / l_full.abs().max()),
               grad_rel=float((eng.flat_grad / world - full.flat_grad).abs().max() / full.flat_grad.abs().max()),
               weight_abs=max(float((eng.params[k] - full.params[k]).abs().max()) for k in eng.names),
               update_magnitude=moved, ranks=world, trajectories=n)
    res["ok"] = bool(res["loss_rel"] < 1e-4 and res["grad_rel"] < 5e-4 and res["weight_abs"] < 1e-3 * moved + 1e-7)
  if dist is not None:
    dist.barrier()
  return res


def run_train(args, name, ctx, steps, warmup, cpu_baseline=True, dump_dir=None):
  """Workload c5: one Trainer.step (code/pred_models.py:1719-1742) per timed step.  Returns the record on rank 0;
  with dump_dir, rank 0 writes the losses of the last timed step there (dump_outputs)."""
  from multiverse_b200 import ops, synthetic
  from multiverse_b200.train_engine import TrainEngine
  wl = WORKLOADS[name]
  world, rank, local, dev, dist = ctx
  gb = args.global_batch or wl["global_batch"]
  n_local = gb // world
  mb = min(wl["micro_batch"], n_local)
  cfg = synthetic.make_config(batch_size=n_local, **wl["cfg"])
  weights = synthetic.make_weights(cfg)
  f = synthetic.make_feeds(cfg, gb, with_pred=True)
  pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
  shard = synthetic.shard_feeds(f, rank, world)
  host = dict(scene_feat=pin(shard["scene_feat"]), obs_scene=pin(shard["obs_scene"]))
  for k in ("grid_obs_labels", "grid_obs_regress", "grid_pred_labels", "grid_pred_regress"):
    host[k] = [pin(a) for a in shard[k]]
  up = lambda t: t.to(dev, non_blocking=True)
  h2d = lambda: {k: ([up(a) for a in v] if isinstance(v, list) else up(v)) for k, v in host.items()}
  h2d_bytes = sum(t.numel() * t.element_size() for v in host.values() for t in (v if isinstance(v, list) else [v]))
  eng = TrainEngine(cfg, {k: torch.from_numpy(v) for k, v in weights.items()}, dev, args.planes)
  feeds = h2d()
  lr = 0.2

  def barrier():
    if dist is not None:
      dist.barrier()
    torch.cuda.synchronize()

  # L2 rule of the timing contract: the state one step streams through (c, h, operand planes of every launch) is
  # far larger than the 126 MB L2 at the default sizes; when a shard is small enough to fit (greedy rollouts at
  # 32 trajectories per GPU), a 256 MB buffer is overwritten between the timed iterations and each iteration is
  # timed by its own pair of events (the flush is outside every pair).
  h0_, w0_ = [g for g, u in zip(cfg.scene_grids, cfg.use_grids) if u][0]
  state_bytes = n_local * (cfg.beam_size if cfg.use_beam_search else 1) * (h0_ + 1) * (w0_ + 1) * 256 * 4 * 3
  flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if state_bytes < (256 << 20) else None

  def timed(fn, steps):
    barrier()
    if flush_buf is not None:
      pairs = []
      for _ in range(steps):
        flush_buf.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        pairs.append((e0, e1))
      barrier()
      total = sum(a.elapsed_time(b) for a, b in pairs)
    else:
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record()
      for _ in range(steps):
        fn()
      e1.record()
      barrier()
      total = e0.elapsed_time(e1)
    ms = torch.tensor([total], device=dev, dtype=torch.float64)
    if dist is not None:
      dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())

  for _ in range(warmup):
    eng.train_step(feeds, lr, dist, mb)
  sampler = ClockSampler(local)
  if rank == 0:
    sampler.start()
  ops.reset_launch_count()
  eng.allreduce_events = []
  last = {}
  step_fn = lambda: eng.train_step(feeds, lr, dist, mb)
  ms_total = timed((lambda: last.__setitem__("out", step_fn())) if dump_dir else step_fn, steps)
  launches = ops.launch_count()
  ar_events, eng.allreduce_events = eng.allreduce_events, None
  clocks = sampler.stop() if rank == 0 else None
  if dump_dir and rank == 0:
    losses, wd = last.pop("out")
    dump_outputs(dump_dir, dict(losses=losses, wd_loss=torch.as_tensor(wd).reshape(1)))
  ar = None
  if ar_events:
    # the one collective of the path (85 MB fp32 gradient bucket), device time per step.  A rank that arrives early
    # waits inside the collective for its peers (the ranks' fwd+bwd times differ by 1-2 % under the power cap), so
    # the MAX over ranks measures skew + transfer and the MIN - the last arriver's - the transfer itself: bus
    # bandwidth 2 (G-1)/G * bytes / min time (the NCCL convention; 725 GB/s measured at 1 GiB on this pool).
    mine = float(np.mean([a.elapsed_time(b) for a, b in ar_events]))
    ar_max = torch.tensor([mine], device=dev, dtype=torch.float64)
    ar_min = torch.tensor([mine], device=dev, dtype=torch.float64)
    dist.all_reduce(ar_max, op=dist.ReduceOp.MAX)
    dist.all_reduce(ar_min, op=dist.ReduceOp.MIN)
    nbytes = eng.flat_grad.numel() * 4
    ar = dict(ms_per_step=float(ar_max.item()), ms_per_step_last_arriver=float(ar_min.item()), bytes=nbytes,
              bus_gbs=2.0 * (world - 1) / world * nbytes / (float(ar_min.item()) * 1e-3) / 1e9,
              share_of_step=float(ar_max.item()) / (ms_total / steps),
              note="ms_per_step = max over ranks (includes waiting for the slowest rank's backward pass); "
                   "bus_gbs from the last arriver's time")
  host_loss = torch.empty(2 * sum(cfg.use_grids), dtype=torch.float32).pin_memory()

  def e2e_step():
    losses, _ = eng.train_step(h2d(), lr, dist, mb)
    host_loss.copy_(losses, non_blocking=True)

  e2e_step()
  ms_e2e = timed(e2e_step, steps)
  grad_mb = eng.flat_grad.numel() * 4 / 1e6
  del eng
  torch.cuda.empty_cache()
  if rank != 0:
    return None
  peaks = load_peaks()
  fl = 3.0 * sum(cfg.obs_len * (cell_flops(h, w, 64) + cell_flops(h, w, 2)) + 2 * cfg.pred_len * cell_flops(h, w, 32)
                 for h, w in cfg.scene_grids) * gb / world
  achieved = fl / (ms_total / steps * 1e-3) / 1e12
  cpu = None
  if world == 1 and cpu_baseline and not args.no_cpu_baseline:
    from oracle import multiverse_ref_torch as RT
    torch.set_num_threads(int(os.environ.get("MVB_CPU_THREADS", "0")) or min(32, os.cpu_count() or 1))
    c2 = synthetic.make_config(batch_size=2, **wl["cfg"])
    f2 = synthetic.make_feeds(c2, 2, with_pred=True)
    t0 = time.perf_counter()
    RT.loss_and_grads(c2, synthetic.make_weights(c2), f2, dtype=torch.float32)
    dt = time.perf_counter() - t0
    cpu = dict(value=2 / dt, unit="trajectories/s", cores=torch.get_num_threads(), kind="port",
               sample="2 trajectories, one fwd+bwd (%.1f s) of the torch-CPU restatement (autograd); TF 1.15 is not installable" % dt)
  line = dict(metric="training trajectories/sec (obs8->pred12, fwd+bwd+update)", value=gb * steps / (ms_total * 1e-3),
              unit="trajectories/s", n_gpus=world, steps=steps, warmup=warmup,
              ms_per_step=ms_total / steps, higher_is_better=True, scaling="strong", vs_baseline=None,
              dtype="f32", data="synthetic",
              config=dict(workload=name + ": " + wl["desc"], global_batch=gb, per_gpu_batch=n_local,
                          micro_batch=mb, arithmetic="fp32-grade: bf16x%d operand planes, fp32 accumulate" % args.planes,
                          parallelism="data-parallel x%d, NCCL all-reduce of %.1f MB fp32 grads"
                          % (world, grad_mb),
                          l2="activation store >> 126 MB L2, no flush needed"),
              clocks=clocks,
              e2e=dict(value=gb * steps / (ms_e2e * 1e-3), unit="trajectories/s", ms_per_step=ms_e2e / steps,
                       h2d_bytes_per_step=h2d_bytes * world, d2h_bytes_per_step=host_loss.numel() * 4),
              gpu_launches=int(launches), allreduce=ar,
              roofline=dict(bound="tensor", kernel="whole train step (cell fwd + dgrad + wgrad GEMMs dominate)",
                            achieved=achieved, peak=peaks["bf16_sustained"], unit="TFLOP/s",
                            frac=achieved / peaks["bf16_sustained"], traffic=None,
                            note="algorithmic FLOPs = 3 x forward cell FLOPs; ceiling 0.333 (3 bf16 passes)"),
              cpu_baseline=cpu)
  return line


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=5)
  ap.add_argument("--warmup", type=int, default=3)
  ap.add_argument("--impl", default="b200")
  ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS))
  ap.add_argument("--global-batch", type=int, default=0)
  ap.add_argument("--planes", type=int, default=2)
  ap.add_argument("--no-cpu-baseline", action="store_true")
  ap.add_argument("--no-extras", action="store_true", help="default run: skip the c3 / c5 sub-records")
  ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                  help="write what the measured workload's last timed step returned as DIR/<name>.npy")
  args = ap.parse_args()
  extras = args.workload is None and not args.no_extras and not args.global_batch
  args.workload = args.workload or "c4"
  wl = WORKLOADS[args.workload]
  if args.impl == "reference":
    return run_reference(args, wl)
  args.warmup = max(args.warmup, 3)
  ctx = setup()
  world, rank, local, dev, dist = ctx
  run = run_train if wl.get("train") else run_infer
  line = run(args, args.workload, ctx, args.steps, args.warmup, dump_dir=args.dump_outputs)
  if extras:
    # the other two north_star workloads in the same invocation, at the same N and in the same process group
    sub = {}
    sub["c3"] = run_infer(args, "c3", ctx, args.steps, args.warmup, cpu_baseline=False)
    sub["c5"] = run_train(args, "c5", ctx, args.steps, args.warmup, cpu_baseline=False)
    chk = ddp_equivalence(ctx) if world > 1 else None
    if rank == 0:
      sub["c5"]["ddp_equivalence"] = chk if chk is not None else "n/a at N=1 (tests/test_ddp_gpu.py runs it on 2 GPUs)"
      line["extra"] = sub
  if rank == 0:
    print(json.dumps(line), flush=True)
  if dist is not None:
    dist.destroy_process_group()


def run_infer(args, name, ctx, steps, warmup, cpu_baseline=True, dump_dir=None):
  """Workloads c4 / c3: one forward (all decoders) per timed step.  Returns the record on rank 0; with dump_dir,
  rank 0 writes the forward outputs of the last timed step there (dump_outputs)."""
  from multiverse_b200 import ops, synthetic
  from multiverse_b200.engine import ConvRNNEngine
  wl = WORKLOADS[name]
  world, rank, local, dev, dist = ctx
  # the host side of the timed regions is one Python thread issuing launches and copies: keep torch's CPU thread pool
  # (sized up by a cpu_baseline leg earlier in the same process) from spinning beside it
  torch.set_num_threads(1)
  gb = args.global_batch or wl["global_batch"]
  assert gb % world == 0
  n_local = gb // world

  cfg = synthetic.make_config(batch_size=n_local, **wl["cfg"])
  weights = synthetic.make_weights(cfg)
  # the batch shards by trajectory: rank r takes rows [r*n_local, (r+1)*n_local) and the scene
  # frames they index (re-compacted per shard like code/pred_utils.py:680-704)
  feeds_all = synthetic.make_feeds(cfg, gb)
  host = synthetic.shard_feeds(feeds_all, rank, world)
  pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
  host_pinned = dict(scene_feat=pin(host["scene_feat"]), obs_scene=pin(host["obs_scene"]),
                     grid_obs_labels=[pin(a) for a in host["grid_obs_labels"]],
                     grid_obs_regress=[pin(a) for a in host["grid_obs_regress"]])

  def h2d():
    g = lambda t: t.to(dev, non_blocking=True)
    return dict(scene_feat=g(host_pinned["scene_feat"]), obs_scene=g(host_pinned["obs_scene"]),
                grid_obs_labels=[g(a) for a in host_pinned["grid_obs_labels"]],
                grid_obs_regress=[g(a) for a in host_pinned["grid_obs_regress"]])

  h2d_bytes = sum(t.numel() * t.element_size() for t in
                  [host_pinned["scene_feat"], host_pinned["obs_scene"]] + host_pinned["grid_obs_labels"]
                  + host_pinned["grid_obs_regress"])
  eng = ConvRNNEngine(cfg, {k: torch.from_numpy(v) for k, v in weights.items()}, dev, args.planes)
  f16f8 = bool(eng.fast_class)
  dev_feeds = h2d()
  torch.cuda.synchronize()

  def outputs_of(out):
    ts = [t for t in out["grid_pred_decoded"] + out["grid_pred_reg_decoded"] if torch.is_tensor(t)]
    if out["beam_outputs"] is not None:
      ts += list(out["beam_outputs"])
    return ts

  def barrier():
    if dist is not None:
      dist.barrier()
    torch.cuda.synchronize()

  # L2 rule of the timing contract: the state one step streams through (c, h, operand planes of every launch) is
  # far larger than the 126 MB L2 at the default sizes; when a shard is small enough to fit (greedy rollouts at
  # 32 trajectories per GPU), a 256 MB buffer is overwritten between the timed iterations and each iteration is
  # timed by its own pair of events (the flush is outside every pair).
  h0_, w0_ = [g for g, u in zip(cfg.scene_grids, cfg.use_grids) if u][0]
  state_bytes = n_local * (cfg.beam_size if cfg.use_beam_search else 1) * (h0_ + 1) * (w0_ + 1) * 256 * 4 * 3
  flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if state_bytes < (256 << 20) else None

  def timed(fn, steps):
    barrier()
    if flush_buf is not None:
      pairs = []
      for _ in range(steps):
        flush_buf.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        pairs.append((e0, e1))
      barrier()
      total = sum(a.elapsed_time(b) for a, b in pairs)
    else:
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record()
      for _ in range(steps):
        fn()
      e1.record()
      barrier()
      total = e0.elapsed_time(e1)
    ms = torch.tensor([total], device=dev, dtype=torch.float64)
    if dist is not None:
      dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())

  # ---- device-resident throughput (`value`) -------------------------------------------------
  # Same rule as the public call (Model._launch_bound): forwards of at most MVB_GRAPH_MAX_ROWS sample rows x beams
  # are replayed from CUDA graphs, one per independent chain on concurrent streams (ConvRNNEngine.forward_graph);
  # larger ones run launch by launch.  Per-launch events need the launch-by-launch path: for graph-replayed sizes
  # the roofline is measured in a second, untimed-for-`value` region of the same number of steps right after.
  rows_all = n_local * (cfg.beam_size if cfg.use_beam_search else 1)
  graph_mode = os.environ.get("MVB_CUDA_GRAPH", "")
  use_graph = (graph_mode == "1") if graph_mode in ("0", "1") else \
      rows_all <= int(os.environ.get("MVB_GRAPH_MAX_ROWS", "2000"))
  step_fn = (lambda: eng.forward_graph(dev_feeds)) if use_graph else (lambda: eng.forward(dev_feeds))
  for _ in range(max(warmup, 3 if use_graph else 0)):     # a signature is captured at its second sight
    step_fn()
  sampler = ClockSampler(local)
  if rank == 0:
    sampler.start()
  ops.reset_launch_count()
  if not use_graph:
    eng.cell_events = []
  last = {}
  ms_total = timed((lambda: last.__setitem__("out", step_fn())) if dump_dir else step_fn, steps)
  launches = ops.launch_count()
  if dump_dir and rank == 0:
    # before the untimed launch-by-launch region below: graph replays return their static output buffers
    out = last.pop("out")
    res = {}
    for key in ("grid_pred_decoded", "grid_pred_reg_decoded"):
      res.update(("%s_%d" % (key, i), t) for i, t in enumerate(out[key]) if torch.is_tensor(t))
    if out["beam_outputs"] is not None:
      res.update(zip(("beam_logits", "beam_grid_ids", "beam_logprobs"), out["beam_outputs"]))
    dump_outputs(dump_dir, res)
    del out, res
  if use_graph:
    # graph replays do not pass through the C ABI's launch counter: count one launch-by-launch forward
    ops.reset_launch_count()
    eng.forward(dev_feeds)
    launches = ops.launch_count() * steps
    eng.cell_events = []
    timed(lambda: eng.forward(dev_feeds), steps)
  events = eng.cell_events
  eng.cell_events = None
  clocks = sampler.stop() if rank == 0 else None
  value = gb * steps / (ms_total * 1e-3)

  # ---- end to end through the reference-facing call (`e2e`) --------------------------------------
  # What code/pred_models.py:1779 (Tester.step) and code/multifuture_inference.py:471 do: sess.run(fetches,
  # feed_dict) on the drop-in Model through the `tensorflow`-named shim - numpy host arrays in (pinned), numpy host
  # arrays out; H2D, forward and D2H of every fetched tensor inside the timed region.
  d2h_probe = outputs_of(eng.forward(dev_feeds))
  d2h_bytes = sum(t.numel() * t.element_size() for t in d2h_probe)
  del d2h_probe, eng, dev_feeds
  torch.cuda.empty_cache()
  import types
  sys.path.insert(0, os.path.join(ROOT, "multiverse_b200", "dropin"))
  import tensorflow as tf          # the shim (multiverse_b200/dropin/tensorflow), not TensorFlow
  import pred_models as pm
  tf.reset_default_graph()
  margs = types.SimpleNamespace(**vars(cfg))
  margs.modelname, margs.use_soft_grid_class, margs.use_gt_grid, margs.is_train = "bench", False, False, False
  model = pm.get_model(margs, gpuid=local)
  tf.global_variables_initializer().run()
  for v in tf.global_variables():
    key = v.name.split(":")[0]
    if key in weights:
      v.assign(weights[key])
  sess = tf.Session(config=tf.ConfigProto(allow_soft_placement=True))
  feed_dict = {model.scene_feat: host_pinned["scene_feat"].numpy(), model.obs_scene: host_pinned["obs_scene"].numpy(),
               model.obs_length: np.full((n_local,), cfg.obs_len, dtype="int32"),
               model.pred_length: np.full((n_local,), cfg.pred_len, dtype="int32"), model.is_train: False}
  fetches = []
  # row f-1: what Model.get_feed_dict feeds for a pred_utils batch - the observed trajectories and the cell centres
  # instead of the dense [N,T,h,w,2] offsets, which the engine rebuilds on the device (bit-identical)
  dense_feeds = os.environ.get("MVB_BENCH_DENSE_FEEDS", "0") == "1"      # A/B: the reference's dense offset arrays
  centers = synthetic.grid_centers(cfg)
  e2e_h2d = [host_pinned["scene_feat"].numpy(), host_pinned["obs_scene"].numpy()]
  if not dense_feeds:
    feed_dict[model.obs_traj] = np.ascontiguousarray(host["traj64"][:, :cfg.obs_len])
    e2e_h2d.append(feed_dict[model.obs_traj])
  for i in range(len(cfg.scene_grids)):
    if cfg.use_grids[i]:
      feed_dict[model.grid_obs_labels[i]] = host_pinned["grid_obs_labels"][i].numpy()
      if dense_feeds:
        feed_dict[model.grid_obs_regress[i]] = host_pinned["grid_obs_regress"][i].numpy()
        e2e_h2d += [feed_dict[model.grid_obs_labels[i]], feed_dict[model.grid_obs_regress[i]]]
      else:
        feed_dict[model.grid_centers[i]] = np.asarray(centers[i], dtype=np.float64)
        e2e_h2d += [feed_dict[model.grid_obs_labels[i]], feed_dict[model.grid_centers[i]]]
      fetches += [model.grid_pred_decoded[i], model.grid_pred_reg_decoded[i]]
  e2e_h2d_bytes = sum(a.nbytes for a in e2e_h2d)
  if cfg.use_beam_search:
    fetches.append(model.beam_outputs)

  def e2e_step():
    return sess.run(fetches, feed_dict=feed_dict)

  for _ in range(2):
    res = e2e_step()
  assert all(isinstance(r, np.ndarray) for r in res[:2])
  del res
  ms_e2e = timed(e2e_step, steps)
  e2e_value = gb * steps / (ms_e2e * 1e-3)
  del sess, model
  tf.reset_default_graph()
  torch.cuda.empty_cache()

  if rank != 0:
    return None

  # ---- roofline of the dominant kernel (fused ConvLSTM cell), measured live ------------------
  peaks = load_peaks()
  dom_tag = "beam" if cfg.use_beam_search else "dec_class"
  h0, w0 = [g for g, u in zip(cfg.scene_grids, cfg.use_grids) if u][0]
  rows = n_local * (cfg.beam_size if cfg.use_beam_search else 1)
  durs = [e0.elapsed_time(e1) for tag, shp, e0, e1 in events if tag == dom_tag and shp[:2] == (h0, w0)]
  all_cell_ms = sum(e0.elapsed_time(e1) for _, _, e0, e1 in events)
  avg_ms = float(np.mean(durs))
  fl = cell_flops(h0, w0, cfg.emb_size) * rows
  achieved = fl / (avg_ms * 1e-3) / 1e12
  traffic = None
  tp = os.path.join(ROOT, "profiles", "cell_traffic.json")
  if os.path.exists(tp):
    try:
      traffic = json.load(open(tp)).get("%s_rows%d" % (name, rows))
    except Exception:
      traffic = None
  passes = args.planes * (args.planes + 1) // 2
  if f16f8:
    arith = ("fp32-grade: operands as one fp16 + two e4m3 planes (f16f8), per product one fp16 tensor pass + two "
             "e4m3 passes at twice the rate into one fp32 TMEM accumulator (2 bf16-pass equivalents), fp32 gates/state; "
             "the regression encoder (raw pixel offsets) keeps 2 bf16 planes / 3 passes")
    ceil_note = ("fp32 parity costs one fp16 + two e4m3 tensor passes per product = 2 bf16-pass equivalents, so the "
                 "ceiling of this fraction against the bf16 peak is 0.5")
  else:
    arith = ("fp32-grade: operands split into %d bf16 planes, %d tcgen05 passes per product, fp32 TMEM accumulate, "
             "fp32 gates/state" % (args.planes, passes))
    ceil_note = ("fp32 parity needs %d bf16 tensor passes per product, so the ceiling of this fraction is %.3f"
                 % (passes, 1.0 / passes))
  roofline = dict(bound="tensor", kernel="cell_fwd_kernel<%s, CTA pair cta_group::2> (%s step, %d sample rows of %dx%d)" % (
                      "f16f8" if f16f8 else "P=%d" % args.planes, dom_tag, rows, h0, w0),
                  achieved=achieved, peak=peaks["bf16_sustained"], unit="TFLOP/s",
                  frac=achieved / peaks["bf16_sustained"], traffic=traffic,
                  peak_source=peaks["source"] + ", bf16 dense sustained (kernel timed inside a long step)",
                  note="algorithmic FLOPs 2*M*N*K (dense, x block included); " + ceil_note + " - times 9/8 on "
                       "class-decoder steps, whose embedded one-hot x block is folded into table look-ups (1/9 of the "
                       "MMAs skipped)",
                  launches_timed=len(durs), avg_launch_ms=avg_ms,
                  cell_share_of_step=all_cell_ms / ms_total)

  # ---- CPU baseline beside it (N=1 only) ------------------------------------------------------
  cpu = None
  if world == 1 and cpu_baseline and not args.no_cpu_baseline:
    n_s = 8
    v, dt, threads = cpu_reference_run(wl["cfg"], n_s, 1)
    cpu = dict(value=v, unit="trajectories/s", cores=threads, kind="port",
               sample="%d trajectories, one pass (%.1f s) of the torch-CPU restatement of "
                      "code/pred_models.py on all host threads; TF 1.15 is not installable" % (n_s, dt))

  line = dict(metric=METRIC if name == "c4" else "trajectories/sec (obs8->pred12, greedy two-scale)", value=value,
              unit="trajectories/s", n_gpus=world, steps=steps,
              warmup=warmup, ms_per_step=ms_total / steps, higher_is_better=True,
              scaling="strong", vs_baseline=None, dtype="f32",
              data="synthetic",
              config=dict(workload=name + ": " + wl["desc"], global_batch=gb, per_gpu_batch=n_local,
                          obs_len=cfg.obs_len, pred_len=cfg.pred_len, beam=cfg.beam_size,
                          parallelism="trajectory-sharded x%d, no collective" % world,
                          arithmetic=arith,
                          execution=("CUDA graphs, one per independent chain (class / regression x scale) on "
                                     "concurrent streams (forwards of <= MVB_GRAPH_MAX_ROWS rows x beams, the rule of "
                                     "the public call); roofline events from a launch-by-launch region of the same "
                                     "length right after" if use_graph else "launch by launch on one stream"),
                          l2=("working set per step (%.2f GB of state) >> 126 MB L2, no flush needed"
                              % (state_bytes / 1e9) if flush_buf is None else
                              "working set per step %.0f MB: a 256 MB buffer is overwritten between the timed "
                              "iterations, each iteration timed by its own event pair" % (state_bytes / 1e6)),
                          gflop_per_trajectory=flops_per_trajectory(cfg) / 1e9),
              clocks=clocks, e2e=dict(value=e2e_value, unit="trajectories/s", ms_per_step=ms_e2e / steps,
                                      h2d_bytes_per_step=e2e_h2d_bytes * world, d2h_bytes_per_step=d2h_bytes * world,
                                      h2d_note="segmentation frames %.1f MB + trajectories, labels and cell centres "
                                               "%.3f MB (dense offsets are rebuilt on the device, row f-1; they were "
                                               "%.1f MB)" % (host_pinned["scene_feat"].numel() * 4 * world / 1e6,
                                                            (e2e_h2d_bytes - host_pinned["scene_feat"].numel() * 4) * world / 1e6,
                                                            sum(t.numel() * 4 for t in host_pinned["grid_obs_regress"]) * world / 1e6)),
              gpu_launches=int(launches), roofline=roofline, cpu_baseline=cpu)
  return line


if __name__ == "__main__":
  main()
