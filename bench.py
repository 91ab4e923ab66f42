#!/usr/bin/env python
"""PPO-update throughput benchmark (BASELINE.json metric: PPO-update samples/sec on
64x64x4 depth + proprio rollouts).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--model loco|nature] [--impl reference] [--dump-outputs DIR]

One "step" = one PPO.update_per_epoch() over a synthetic rollout of T x E transitions:
GAE scan + opt_epochs x (T*E/B) minibatch updates (critic fwd/bwd/clip/Adam, actor fwd/bwd +
frozen-target fwd/clip/Adam) = opt_epochs*T*E sample-updates.  Every step, warm-up and timed, starts from the
same network and optimiser state: in training each update sees a fresh rollout drawn near the current policy,
while updates chained over this one fixed rollout drive the policy ever further from its actions until the
importance ratios overflow (after ~20 steps, in the exact fp32 tier as well).
  value : rollout already resident in HBM when the timed region starts (CUDA events, max over
          ranks);
  e2e   : the same step through the public call PPO.update_per_epoch() with the rollout in
          pinned HOST memory — the H2D copy of the whole rollout and the D2H read of the logged
          statistics are inside the timed region.
N > 1 (torchrun, one rank per GPU): every rank owns its own T x E shard (weak scaling), the
minibatch is the union over ranks, gradients are all-reduced once per optimiser step (NCCL) and
the advantage statistics are global.
The same line also carries
  strong_sweep : BASELINE configs[4] — ONE fixed synthetic rollout of 2^20 transitions (generated on the
                 device, 34 GB as fp16) with a fixed GLOBAL minibatch of 65536, sharded by env column over the
                 N ranks (strong scaling; resident timing);
  roofline     : the kernel family with the largest share of kernel time in the committed launch list
                 (profiles/r2_f16_launches_summary.md), replayed alone with CUDA events, against the tensor roof;
  fp32_tier    : the same step on the exact (fp32 CUDA-core) tier — the same-precision number;
  gae          : the GAE scan alone (transitions/s, GB/s of its 18 B/transition);
  cpu_baseline : the oracle port on the host cores — update only, "as shipped" (float64 gather + convert,
                 reference on_policy.py:83-89, ppo.py:136-140) and GAE (on_policy.py:17-45).
--impl reference: the reference's CPU torch path (oracle port, see oracle/ppo_oracle.py) timed
on this box's host cores on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_SAMPLE = {"loco": 70.31e6, "nature": 50.81e6}       # BASELINE.md §2 (S=93, A=12)
OBS_BYTES = lambda S: (S + 16384) * 4


def parse():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=5)
  ap.add_argument("--warmup", type=int, default=3)
  ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
  ap.add_argument("--model", default="loco", choices=["loco", "nature"])
  ap.add_argument("--T", type=int, default=2048)
  ap.add_argument("--E", type=int, default=8)
  ap.add_argument("--batch", type=int, default=1024)
  ap.add_argument("--opt-epochs", type=int, default=3)
  ap.add_argument("--S", type=int, default=93)
  ap.add_argument("--A", type=int, default=12)
  ap.add_argument("--no-graph", action="store_true")
  ap.add_argument("--precision", default="f16", choices=["fp32", "f16"],
                  help="f16: tcgen05 tensor-core tier (fp16 operands, fp32 accumulate); fp32: exact CUDA-core tier")
  ap.add_argument("--no-cpu-baseline", action="store_true")
  ap.add_argument("--cpu-seconds", type=float, default=12.0)
  ap.add_argument("--no-fp32-tier", action="store_true")
  ap.add_argument("--no-sweep", action="store_true")
  ap.add_argument("--sweep-transitions", type=int, default=1 << 20)
  ap.add_argument("--sweep-batch", type=int, default=65536, help="GLOBAL minibatch of the strong-scaling sweep")
  ap.add_argument("--sweep-steps", type=int, default=1)
  ap.add_argument("--sweep-timeout", type=int, default=300)
  ap.add_argument("--sweep-envs", type=int, default=8, help="env columns of the sweep's rollout (8 = BASELINE configs[4])")
  ap.add_argument("--no-roofline", action="store_true")
  ap.add_argument("--dump-outputs", metavar="DIR",
                  help="write what the last timed step computed (per-minibatch statistics, parameters after the step, "
                       "advantages and returns) to DIR/<name>.npy, to compare two builds output for output")
  args = ap.parse_args()
  if args.dump_outputs and args.steps < 1:
    ap.error("--dump-outputs needs at least one timed step")
  return args


def peaks():
  path = os.path.join(ROOT, "MEASURED_PEAKS.json")
  if os.path.exists(path):
    p = json.load(open(path))
    return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
            "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "src": "measured"}
  return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}


class ClockSampler:
  """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
  Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
       "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
       "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

  def __init__(self, index=0):
    self.index, self.rows, self.stamps, self.proc = index, [], [], None

  def start(self):
    try:
      self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                    "--format=csv,noheader,nounits", "-lms", "20"],
                                   stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      self.t = threading.Thread(target=self._read, daemon=True)
      self.t.start()
    except Exception:
      self.proc = None

  def _read(self):
    for line in self.proc.stdout:
      self.stamps.append(time.perf_counter())
      self.rows.append([c.strip() for c in line.split(",")])

  def stop(self, window=None):
    """window = (t0, t1) in time.perf_counter() seconds: keep the samples taken inside the timed region
    (the sampler is started one warm-up step early so that nvidia-smi is already running by then)."""
    if self.proc is None:
      return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    time.sleep(0.05)
    self.proc.terminate()
    try:
      self.proc.wait(timeout=2)
    except Exception:
      self.proc.kill()
    if window is not None:
      keep = [r for t, r in zip(self.stamps, self.rows) if window[0] <= t <= window[1] + 0.02]
      if keep:
        self.rows = keep
    sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
    mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
    reasons = set()
    for r in self.rows:
      if len(r) < 9:
        continue
      for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                        ("sw_power_cap", 8)):
        if r[col].lower().startswith("active"):
          reasons.add(name)
    return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
            "reasons": sorted(reasons), "samples": len(sm)}


# -------------------------------------------------------------------------------------------------
# CPU side: the reference's torch path (oracle port) on a bounded sample
# -------------------------------------------------------------------------------------------------
def make_oracle(model, S, A, batch):
  from oracle import ppo_oracle as po
  from benchutil import synth
  pf_np, vf_np = synth.make_family_weights(1000, model, S, A)
  pf, vf = po.sd_to_torch(pf_np, vf_np)
  return po.PPOOracle(model, pf, vf, S, batch_size=batch, opt_epochs=1)


def cpu_minibatch(model, S, A, batch, seed):
  from benchutil import synth
  rng = np.random.default_rng(seed)
  roll = synth.make_rollout(seed, batch // 8, 8, S, A)
  return {"obs": roll["obs"].reshape(batch, -1), "acts": roll["acts"].reshape(batch, -1),
          "advs": rng.standard_normal((batch, 1)).astype(np.float32),
          "estimate_returns": rng.standard_normal((batch, 1)).astype(np.float32),
          "values": roll["values"].reshape(batch, 1)}


def host_cores():
  """Usable host cores: min(affinity mask, cgroup CPU quota)."""
  cores = os.cpu_count() or 1
  try:
    cores = min(cores, len(os.sched_getaffinity(0)))
  except Exception:
    pass
  try:
    quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
    if quota != "max":
      cores = max(1, min(cores, int(float(quota) / float(period))))
  except Exception:
    pass
  return cores


def pick_threads():
  """torch-CPU threads for the reference arm: the fastest of a few candidates on a small
  conv fwd+bwd probe (oversubscribing a shared 128-core host is 50x slower than 16 threads)."""
  import torch.nn.functional as F
  cores = host_cores()
  cands = sorted({c for c in (4, 8, 16, 32, 64, cores) if c <= cores} | {min(cores, 8)})
  x = torch.randn(128, 4, 64, 64)
  w = torch.randn(32, 4, 8, 8, requires_grad=True)
  best, best_t = cands[0], float("inf")
  for c in cands:
    torch.set_num_threads(c)
    for rep in range(3):
      t0 = time.perf_counter()
      F.conv2d(x, w, stride=4).sum().backward()
      dt = time.perf_counter() - t0
      if rep and dt < best_t:
        best, best_t = c, dt
  torch.set_num_threads(best)
  return best, cores


def cpu_baseline(args, budget_s):
  """The reference-equivalent CPU path on the host cores (BASELINE.md §3): (i) PPO.update only, tensors
  pre-converted, cycling over 3 DISTINCT minibatches; (ii) "as shipped": each minibatch additionally pays the
  float64 row gather of the replay buffer and the float64 -> float32 conversion (reference on_policy.py:83-89,
  ppo.py:136-140); (iii) the GAE loop over the epoch's T x E transitions (on_policy.py:17-45)."""
  from oracle import ppo_oracle as po
  from benchutil import synth
  cores, avail = pick_threads()
  B, E = args.batch, 8
  rows = B // E
  orc = make_oracle(args.model, args.S, args.A, B)
  roll = synth.make_rollout(5, 3 * rows, E, args.S, args.A)
  obs64 = roll["obs"].astype(np.float64)                       # the reference buffer is float64 (base.py:27-28)
  aux64 = {k: roll[k].astype(np.float64) for k in ("acts", "values")}
  rng = np.random.default_rng(5)
  advs64 = rng.standard_normal((3 * rows, E, 1)); rets64 = rng.standard_normal((3 * rows, E, 1))
  perm = rng.permutation(3 * rows)

  def shipped(k):      # one_iteration's fancy-index copies + PPO.update's torch.Tensor(...) conversions
    idx = perm[k * rows:(k + 1) * rows]
    return {"obs": torch.Tensor(obs64[idx].reshape(B, -1)), "acts": torch.Tensor(aux64["acts"][idx].reshape(B, -1)),
            "advs": torch.Tensor(advs64[idx].reshape(B, 1)), "estimate_returns": torch.Tensor(rets64[idx].reshape(B, 1)),
            "values": torch.Tensor(aux64["values"][idx].reshape(B, 1))}
  pre = [shipped(k) for k in range(3)]
  orc.update(pre[0])                                          # warm-up
  n, t0 = 0, time.perf_counter()
  while True:
    orc.update(pre[n % 3])
    n += 1
    dt = time.perf_counter() - t0
    if dt >= budget_s * 0.6 or n >= 24:
      break
  upd = n * B / dt
  n2, t0 = 0, time.perf_counter()
  while True:
    orc.update(shipped(n2 % 3))
    n2 += 1
    dt2 = time.perf_counter() - t0
    if dt2 >= budget_s * 0.4 or n2 >= 12:
      break
  T, E2 = args.T, args.E
  r = synth.make_rollout(6, T, E2, args.S, args.A, with_img=False)
  t0 = time.perf_counter()
  po.gae(r["rewards"], r["values"], r["terminals"], r["time_limits"], np.zeros((E2, 1)), 0.99, 0.95, True)
  dtg = time.perf_counter() - t0
  return {"value": upd, "unit": "samples/s", "cores": cores, "kind": "port",
          "as_shipped": {"value": n2 * B / dt2, "unit": "samples/s",
                         "note": "update + float64 time-row gather + float64->float32 conversion of the minibatch"},
          "gae": {"value": T * E2 / dtg, "unit": "transitions/s", "T": T, "E": E2, "seconds": dtg},
          "sample": "%d PPO.update minibatches of %d (%s, S=%d, A=%d; 3 distinct minibatches in rotation) after 1 warm-up, "
                    "%.1f s, + %d as-shipped minibatches %.1f s, %d torch threads (best of a probe; %d usable cores, "
                    "cgroup quota / affinity); oracle/ppo_oracle.py = torch-CPU restatement of the reference path" %
                    (n, B, args.model, args.S, args.A, dt, n2, dt2, cores, avail)}


def run_reference(args):
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return
  cores, avail = pick_threads()
  orc = make_oracle(args.model, args.S, args.A, args.batch)
  mbs = [{k: torch.as_tensor(v, dtype=torch.float32) for k, v in cpu_minibatch(args.model, args.S, args.A, args.batch, 5 + j).items()}
         for j in range(3)]
  per_step = 3                                           # minibatches per step (bounded sample of the 48 of a full step)
  for w in range(args.warmup):
    orc.update(mbs[w % 3])
  t0 = time.perf_counter()
  for k in range(args.steps * per_step):
    orc.update(mbs[k % 3])
  dt = time.perf_counter() - t0
  value = args.steps * per_step * args.batch / dt
  sample = ("%d steps x %d PPO.update minibatches of %d (3 distinct minibatches in rotation; a full step is 48), %d torch "
            "threads (%d usable cores: cgroup quota / affinity of this box)" % (args.steps, per_step, args.batch, cores, avail))
  print(json.dumps({
    "impl": "reference", "metric": "ppo_update_samples_per_sec", "value": value, "unit": "samples/s",
    "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
    "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
    "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args, 1),
    "cpu_baseline": {"value": value, "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample},
    "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
  }))


def workload_config(args, world):
  return {"workload": "ppo_%s update_per_epoch: T=%d x E=%d transitions/rank, minibatch %d/rank, "
                      "opt_epochs=%d, S=%d proprio + 4x64x64 depth, A=%d (BASELINE configs[%d])" %
                      ("locotransformer" if args.model == "loco" else "nature_cnn", args.T, args.E,
                       args.batch, args.opt_epochs, args.S, args.A, 2 if args.model == "loco" else 1),
          "global_batch": args.batch * world, "parallelism": "dp%d" % world,
          "l2": "inputs larger than L2 (%.2f GB fp32 rollout/rank on the host, %.2f GB resident as fp16 in the f16 tier; "
                "rows visited in a fresh permutation every opt-epoch)" %
                (args.T * args.E * OBS_BYTES(args.S) / 1e9, args.T * args.E * (args.S * 4 + 32768) / 1e9)}


# -------------------------------------------------------------------------------------------------
# GPU side
# -------------------------------------------------------------------------------------------------
def main():
  args = parse()
  if args.impl == "reference":
    run_reference(args)
    return
  rank = int(os.environ.get("RANK", "0"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  world = int(os.environ.get("WORLD_SIZE", "1"))
  if not torch.cuda.is_available():
    raise SystemExit("bench.py needs a CUDA device (there is no CPU path for the product arm); "
                     "use --impl reference for the CPU baseline")
  torch.cuda.set_device(local)
  dev = torch.device("cuda", local)
  pg = None
  if world > 1:
    import torch.distributed as dist
    dist.init_process_group("nccl", device_id=dev)
    pg = dist.group.WORLD

  from benchutil import synth
  from benchutil.harness import build_nets, load_np_sd, make_ppo
  from vision4leg_b200.replay_buffers import OnPolicyReplayBuffer

  S, A, T, E = args.S, args.A, args.T, args.E
  pf, vf = build_nets(args.model, S, A)
  pf_np, vf_np = synth.make_family_weights(1000, args.model, S, A)      # same weights on all ranks
  load_np_sd(pf, pf_np); load_np_sd(vf, vf_np)
  pf, vf = pf.to(dev), vf.to(dev)

  # synthetic rollout in the pinned host buffer (generated in chunks to bound host memory)
  buf = OnPolicyReplayBuffer(env_nums=E, max_replay_buffer_size=T * E, time_limit_filter=True)
  chunk = 256
  for t0 in range(0, T, chunk):
    n = min(chunk, T - t0)
    roll = synth.make_rollout(1000 * rank + t0, n, E, S, A)
    for t in range(n):
      buf.add_sample({"obs": roll["obs"][t], "next_obs": roll["last_obs"], "acts": roll["acts"][t],
                      "values": roll["values"][t], "rewards": roll["rewards"][t],
                      "terminals": roll["terminals"][t], "time_limits": roll["time_limits"][t]})
  agent, logger = make_ppo(pf, vf, buf, A, args.batch, T * E, args.opt_epochs, device=dev)
  agent.process_group = pg
  agent.use_cuda_graph = not args.no_graph
  agent.precision = args.precision
  eng = agent.engine
  samples_per_step = args.opt_epochs * T * E * world

  def barrier():
    if world > 1:
      import torch.distributed as dist
      dist.barrier()
    torch.cuda.synchronize(dev)

  def max_over_ranks(ms):
    if world > 1:
      import torch.distributed as dist
      t = torch.tensor([ms], device=dev, dtype=torch.float64)
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
      return float(t)
    return ms

  # ---- device-resident step: rollout already in HBM
  np.random.seed(0)
  eng.load_rollout(buf)
  last = buf.last_sample(["next_obs", "terminals"])
  start = [t.clone() for t in training_state(eng)]

  def restart():
    for t, t0 in zip(training_state(eng), start):
      t.copy_(t0)

  def resident_step(epoch):
    restart()
    agent.current_epoch = epoch
    eng.compute_advantages(last["next_obs"], last["terminals"], agent.discount, agent.tau, True, True)
    agent._schedule()
    eng.sync_target()
    return eng.run_epoch(agent._draw_perms(T), args.batch)

  sampler = ClockSampler(local)
  for w in range(args.warmup):
    if rank == 0 and w == args.warmup - 1:
      sampler.start()                       # nvidia-smi needs ~100 ms to come up: start one warm-up step early
    resident_step(w)
  if rank == 0 and args.warmup == 0:
    sampler.start()
  barrier()
  launches0 = eng.ops.launches
  ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  t_w0 = time.perf_counter()
  ev0.record()
  for k in range(args.steps):
    infos = resident_step(args.warmup + k)
  ev1.record()
  barrier()
  t_w1 = time.perf_counter()
  if args.dump_outputs and rank == 0:
    dump_outputs(args.dump_outputs, infos, pf, vf, eng._roll)
  ms = max_over_ranks(ev0.elapsed_time(ev1))
  launches = eng.ops.launches - launches0
  clocks = sampler.stop((t_w0, t_w1)) if rank == 0 else None
  value = samples_per_step * args.steps / (ms / 1e3)

  # ---- end-to-end step through the public API with HOST buffers
  for w in range(2):
    restart()
    agent.current_epoch = w
    agent.update_per_epoch()
  barrier()
  t0 = time.perf_counter()
  ev0.record()
  for k in range(args.steps):
    restart()
    agent.current_epoch = 10 + k
    agent.update_per_epoch()
  ev1.record()
  barrier()
  e2e_ms = max_over_ranks(max(ev0.elapsed_time(ev1), (time.perf_counter() - t0) * 1e3))
  e2e_value = samples_per_step * args.steps / (e2e_ms / 1e3)

  # ---- strong-scaling sweep (every rank takes part; the weak-scaling engine's memory is released first)
  h2d_b, d2h_b = int(eng.h2d_bytes), int(eng.d2h_bytes)
  roof_inputs = None
  if rank == 0 and world == 1 and not args.no_roofline and args.precision == "f16":
    try:
      roof_inputs = kernel_rooflines(args, eng, peaks())          # needs the engine's plans and rollout
    except Exception as ex:
      roof_inputs = {"roofline": {"error": repr(ex)[:300]}, "gae": None}
  pk = peaks()
  line = {
    "metric": "ppo_update_samples_per_sec", "value": value, "unit": "samples/s", "n_gpus": world,
    "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
    "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
    "dtype": "f16" if args.precision == "f16" else "f32", "data": "synthetic",
    "config": workload_config(args, world),
    "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d_b,
            "d2h_bytes_per_step": int(d2h_b + 2 * T * E * 4), "ms_per_step": e2e_ms / args.steps},
    "gpu_launches": int(launches), "clocks": clocks,
    "step_roofline": {"bound": "tensor", "achieved": value / world * FLOP_PER_SAMPLE[args.model] / 1e12,
                      "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
                      "frac": value / world * FLOP_PER_SAMPLE[args.model] / 1e12 / pk["bf16_tflops_sustained"],
                      "hbm_frac": value / world * OBS_BYTES(S) / 1e9 / pk["hbm_gbs"],
                      "note": "whole step per GPU (BASELINE.md algorithmic FLOPs) vs %s bf16 sustained peak" % pk["src"]},
  }
  if roof_inputs:
    line["roofline"] = roof_inputs["roofline"]
    line["gae"] = roof_inputs["gae"]
  sweep = None
  if not args.no_sweep and args.precision == "f16":
    # The sweep is auxiliary: the headline line above is complete.  A watchdog prints it (rank 0) and ends the
    # process if the sweep has not come back in time (e.g. a rank lost to an allocation failure would leave its
    # peers inside a collective), so the one-line contract holds whatever happens in here.
    def _bail():
      if rank == 0:
        line.setdefault("strong_sweep", {"error": "watchdog: the sweep did not finish within %d s" % args.sweep_timeout})
        print(json.dumps(line))
        sys.stdout.flush()
      os._exit(0)
    dog = threading.Timer(args.sweep_timeout, _bail)
    dog.daemon = True
    dog.start()
    try:
      sweep = strong_sweep(args, dev, pg, world, rank, pf_np, vf_np, barrier, max_over_ranks)
    except Exception as ex:             # a failure on EVERY rank (bad arguments): report it
      sweep = {"error": repr(ex)[:300]}
    if rank == 0 and sweep is not None:
      line["strong_sweep"] = sweep     # (the watchdog keeps running until the barrier below has been passed)
  else:
    dog = None

  if world > 1:
    # no collective is issued past this point; ranks leave without tearing NCCL down (destroying a
    # communicator that captured CUDA graphs still reference can block) — hard exit after flushing
    import torch.distributed as dist
    dist.barrier()
    torch.cuda.synchronize(dev)
    if rank != 0:
      sys.stdout.flush()
      os._exit(0)
  if dog is not None:
    dog.cancel()
  if sweep is not None:
    line["strong_sweep"] = sweep
  if world == 1 and not args.no_fp32_tier and args.precision == "f16":
    try:
      line["fp32_tier"] = fp32_tier(args, dev, pf_np, vf_np)
    except Exception as ex:
      line["fp32_tier"] = {"error": repr(ex)[:300]}
  if not args.no_cpu_baseline and world == 1:
    line["cpu_baseline"] = cpu_baseline(args, args.cpu_seconds)
  print(json.dumps(line))
  sys.stdout.flush()
  if world > 1:
    os._exit(0)


def training_state(eng):
  """what one step changes: the parameters of both networks (one flat bucket), the Adam moments and step counts"""
  return [eng.bucket.flat, eng.m_pf, eng.v_pf, eng.m_vf, eng.v_vf, eng.hyper_pf, eng.hyper_vf]


DUMP_MAX_ELEMS = 1 << 20          # per array: larger arrays are stored as a fixed, seeded sample
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(d, infos, pf, vf, roll):
  """What a caller of the timed step receives, after its last call: the logged statistics of every minibatch
  (float64, one row per minibatch), the parameters of both networks (float32) and the step's advantages and returns
  (float32, [T*E]).  An array of more than DUMP_MAX_ELEMS elements is replaced by the values at
  sorted(default_rng(0).choice(n, DUMP_MAX_ELEMS, replace=False)) of its flattened form."""
  from vision4leg_b200._lib import INFO_KEYS
  out = {"info.%s" % k.replace("/", "_"): np.array([float(i[k]) for i in infos], np.float64) for k in INFO_KEYS}
  for name, net in (("pf", pf), ("vf", vf)):
    for k, v in net.state_dict().items():
      out["%s.%s" % (name, k)] = v.detach().float().cpu().numpy()
  out["gae.advs"] = roll["advs"].detach().float().cpu().numpy().reshape(-1)
  out["gae.returns"] = roll["rets"].detach().float().cpu().numpy().reshape(-1)
  for k, a in out.items():
    if a.size > DUMP_MAX_ELEMS:
      out[k] = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMS, replace=False))]
  total = sum(a.nbytes for a in out.values())
  if total > DUMP_MAX_BYTES:
    raise SystemExit("--dump-outputs: %d bytes exceed the %d-byte bound" % (total, DUMP_MAX_BYTES))
  os.makedirs(d, exist_ok=True)
  for k, a in out.items():
    np.save(os.path.join(d, k + ".npy"), a)


# -------------------------------------------------------------------------------------------------
# auxiliary measurements carried by the same line
# -------------------------------------------------------------------------------------------------
def _time_events(fn, reps, sync_after=None):
  """CUDA-event time of fn() per call (seconds), events on the launching stream"""
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  total = 0.0
  for _ in range(reps):
    e0.record()
    fn()
    e1.record()
    if sync_after:
      sync_after()
    torch.cuda.synchronize()
    total += e0.elapsed_time(e1) / 1e3
  return total / reps


def _ncu_table():
  """per-kernel dram bytes / tensor-pipe % from the committed `ncu --set full` capture (minibatch 1024, loco)"""
  path = os.path.join(ROOT, "profiles", "r2_kernel_ncu.json")
  return json.load(open(path)) if os.path.exists(path) else {}


def kernel_rooflines(args, eng, pk):
  """One eager minibatch is recorded (every tensor-core launch with its arguments), then each kernel family is
  replayed ALONE, back to back on one stream, between CUDA events: achieved = algorithmic FLOPs of the family
  per minibatch / its time; `frac` = achieved / measured dense bf16 peak (burst: the family is timed in
  isolation).  The family with the largest share of kernel time in the committed ncu launch list is `roofline`
  (profiles/r2_f16_launches_summary.md: tc_wgrad_kernel), the others follow under `other_kernels`."""
  ops, B = eng.ops, args.batch
  eng._slot.zero_()
  ops.record(True)
  try:
    eng._minibatch(B, with_target=False)
  finally:
    rec = ops.record(False)
  torch.cuda.synchronize()
  ncu = _ncu_table()
  fams = {}
  for r in rec:
    fams.setdefault(r[0], []).append(r)
  names = {"v4l_tc_wgrad": "tc_wgrad_kernel", "v4l_tc_gemm": "tc_gemm_kernel", "v4l_tc_block_fwd": "tc_block_fwd_kernel",
           "v4l_tc_block_bwd": "tc_block_bwd_kernel", "v4l_tc_conv_flat": "tc_conv_flat_kernel",
           "v4l_tc_wgrad_conv1": "tc_wgrad_conv1_kernel"}
  what = {"tc_wgrad_kernel": "weight + bias gradients of every layer but conv1 (MN-major tcgen05.mma over the TMA boxes "
                             "of the forward, split-K partials)",
          "tc_gemm_kernel": "every forward layer and data gradient outside the fused encoder layers (tap-shifted TMA + "
                            "tcgen05.mma, persistent over row tiles)",
          "tc_block_fwd_kernel": "one TransformerEncoderLayer forward per launch (six chained tcgen05 contractions)",
          "tc_block_bwd_kernel": "one TransformerEncoderLayer data-gradient pass per launch",
          "tc_conv_flat_kernel": "conv1 forward (single-load flat convolution)",
          "tc_wgrad_conv1_kernel": "conv1 weight gradient (single-load space-to-depth windows)"}
  out = {}
  for fn, items in fams.items():
    defer = fn in ("v4l_tc_wgrad", "v4l_tc_wgrad_conv1")
    run = lambda items=items: ops.replay(items)
    flush = (lambda: ops.tc_wgrad_flush()) if defer else None
    for _ in range(2):
      run()
      if flush:
        flush()
    torch.cuda.synchronize()
    sec = _time_events(run, 10, flush)
    flops = sum(r[2] for r in items)
    k = names[fn]
    ach = flops / sec / 1e12
    e = {"kernel": k, "what": what[k], "bound": "tensor", "achieved": ach, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
         "frac": ach / pk["bf16_tflops"], "launches_per_minibatch": len(items), "us_per_launch": sec / len(items) * 1e6,
         "us_per_minibatch": sec * 1e6, "algorithmic_flops_per_minibatch": flops, "peak_src": pk["src"] + " (burst)",
         "traffic": None}
    t = ncu.get(k) if (B == 1024 and args.model == "loco") else None
    if t:
      e["traffic"] = t["dram_bytes_per_launch"]
      e["ncu"] = {"tensor_pipe_active_pct": t.get("tensor_pipe_pct"), "dram_bytes_per_launch": t["dram_bytes_per_launch"],
                  "source": "profiles/r2_kernel_ncu.json (ncu --set full, one minibatch, averages over the family's launches)"}
    out[k] = e
  order = sorted(out.values(), key=lambda e: -e["us_per_minibatch"])
  # the dominant family by the committed launch list (cold-cache, serialised ncu times) — it is also the
  # largest when replayed warm here
  dom = out.get("tc_wgrad_kernel", order[0])
  dom = dict(dom)
  dom["other_kernels"] = [e for e in order if e["kernel"] != dom["kernel"]]
  dom["note"] = ("minibatch %d: every launch is a small grid whose time is launch + pipeline-fill latency, not tensor "
                 "throughput (the whole step is latency-bound at this size: step_roofline); the fractions grow with the "
                 "minibatch (strong_sweep)" % B)
  # ---- GAE scan alone (HBM / latency bound: 18 B per transition, SURVEY 8(d))
  r = eng._roll
  Tn, En = r["T"], r["E"]
  tl = r["time_limits"]
  tl_st, tl_se = (tl.shape[1], 1) if (tl is not None and tl.shape[1] == En and En > 1) else (1, 0)
  g = lambda: ops.gae(r["rewards"], r["values"], r["terminals"], tl, tl_st, tl_se, r["last_value"], r["advs"], r["rets"],
                      Tn, En, 0.99, 0.95, tl is not None, 0)
  g(); torch.cuda.synchronize()
  sec = _time_events(g, 20)
  big = 1 << 20
  f = lambda *s_: torch.randn(s_, device=ops.device)
  bg = dict(r=f(big), v=f(big), d=torch.zeros(big, device=ops.device), lv=f(8), a=f(big), q=f(big))
  gb = lambda: ops.gae(bg["r"], bg["v"], bg["d"], None, 1, 0, bg["lv"], bg["a"], bg["q"], big // 8, 8, 0.99, 0.95, False, 0)
  gb(); torch.cuda.synchronize()
  secb = _time_events(gb, 20)
  gae = {"value": Tn * En / sec, "unit": "transitions/s", "T": Tn, "E": En, "us": sec * 1e6,
         "sweep_2p20": {"value": big / secb, "unit": "transitions/s", "us": secb * 1e6,
                        "bound": "hbm", "achieved": big * 18 / secb / 1e9, "peak": pk["hbm_gbs"], "unit_bw": "GB/s",
                        "frac": big * 18 / secb / 1e9 / pk["hbm_gbs"],
                        "note": "algorithmic 18 B/transition (SURVEY 8d); the kernel moves 20 B (fp32 terminals); 3 launches "
                                "(chunk aggregates, carries, scan): latency-bound below ~10^7 transitions"}}
  return {"roofline": dom, "gae": gae}


def fp32_tier(args, dev, pf_np, vf_np):
  """The same step on the exact tier (fp32 CUDA-core GEMMs: same precision as the reference)."""
  from benchutil import synth
  from benchutil.harness import build_nets, load_np_sd, make_ppo
  from vision4leg_b200.replay_buffers import OnPolicyReplayBuffer
  S, A, T, E = args.S, args.A, args.T, args.E
  pf, vf = build_nets(args.model, S, A)
  load_np_sd(pf, pf_np); load_np_sd(vf, vf_np)
  pf, vf = pf.to(dev), vf.to(dev)
  buf = OnPolicyReplayBuffer(env_nums=E, max_replay_buffer_size=T * E, time_limit_filter=True)
  for t0 in range(0, T, 256):
    n = min(256, T - t0)
    roll = synth.make_rollout(t0, n, E, S, A)
    for t in range(n):
      buf.add_sample({"obs": roll["obs"][t], "next_obs": roll["last_obs"], "acts": roll["acts"][t],
                      "values": roll["values"][t], "rewards": roll["rewards"][t],
                      "terminals": roll["terminals"][t], "time_limits": roll["time_limits"][t]})
  agent, _ = make_ppo(pf, vf, buf, A, args.batch, T * E, args.opt_epochs, device=dev)
  agent.precision = "fp32"
  eng = agent.engine
  np.random.seed(0)
  eng.load_rollout(buf)
  last = buf.last_sample(["next_obs", "terminals"])

  def step(epoch):
    agent.current_epoch = epoch
    eng.compute_advantages(last["next_obs"], last["terminals"], agent.discount, agent.tau, True, True)
    agent._schedule()
    eng.sync_target()
    eng.run_epoch(agent._draw_perms(T), args.batch)
  for w in range(2):
    step(w)
  torch.cuda.synchronize()
  steps = 2
  sec = _time_events(lambda: [step(2 + k) for k in range(steps)], 1)
  for w in range(2):
    agent.current_epoch = w
    agent.update_per_epoch()
  torch.cuda.synchronize()
  t0 = time.perf_counter()
  for k in range(steps):
    agent.current_epoch = 10 + k
    agent.update_per_epoch()
  torch.cuda.synchronize()
  e2e = time.perf_counter() - t0
  n = args.opt_epochs * T * E * steps
  return {"value": n / sec, "unit": "samples/s", "dtype": "f32", "steps": steps, "warmup": 2, "ms_per_step": sec / steps * 1e3,
          "e2e": {"value": n / e2e, "unit": "samples/s", "h2d_bytes_per_step": int(eng.h2d_bytes),
                  "d2h_bytes_per_step": int(eng.d2h_bytes + 2 * T * E * 4)},
          "note": "exact tier: fp32 FFMA GEMMs, 1e-3 parity with the reference's golden vectors (tests/test_gpu_ppo.py)"}


def strong_sweep(args, dev, pg, world, rank, pf_np, vf_np, barrier, max_over_ranks):
  """BASELINE configs[4]: one fixed rollout of `--sweep-transitions` (2^20) transitions and a fixed GLOBAL
  minibatch (65536) sharded over the ranks by env column (the reference's minibatch = whole time rows x all
  envs, on_policy.py:76-89, so GAE needs no collective); one all-reduce per optimiser step.  The rollout is
  generated ON THE DEVICE in the layouts the engine keeps resident (fp16 space-to-depth image, fp32 proprio
  rows): this is the resident (`value`) figure of the sweep; the end-to-end figure is the weak line's."""
  from benchutil.harness import build_nets, load_np_sd, make_ppo
  S, A, E = args.S, args.A, args.sweep_envs
  if world > E or E % world or args.sweep_batch % world or (args.sweep_batch // world) % (E // world):
    return {"skipped": "world size %d does not divide the %d env columns / the minibatch" % (world, E)}
  El = E // world
  T = args.sweep_transitions // E
  Bl = args.sweep_batch // world
  N = T * El
  free, _ = torch.cuda.mem_get_info(dev)
  if world > 1:                       # the same decision on every rank (the least free memory decides)
    import torch.distributed as dist
    t = torch.tensor([float(free)], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    free = float(t)
  need = N * (32768 + S * 4 + A * 8 + 64) + (12 << 30) * min(1.0, Bl / 65536.0) * 3
  if need > free * 0.92:
    return {"skipped": "needs %.0f GB of HBM, %.0f GB free" % (need / 2**30, free / 2**30)}
  pf, vf = build_nets(args.model, S, A)
  load_np_sd(pf, pf_np); load_np_sd(vf, vf_np)
  pf, vf = pf.to(dev), vf.to(dev)
  agent, _ = make_ppo(pf, vf, None, A, Bl, N, args.opt_epochs, device=dev)
  agent.process_group = pg
  agent.precision = "f16"
  eng = agent.engine
  r = eng._alloc_rollout(T, El)
  gen = torch.Generator(device=dev)
  gen.manual_seed(1234 + rank)
  chunk = 1 << 15
  for n0 in range(0, N, chunk):
    m = min(chunk, N - n0)
    d = torch.empty((m, 16, 16, 64), device=dev, dtype=torch.float32).uniform_(0.3, 10.0, generator=gen)
    r["imgs"][n0:n0 + m] = ((torch.sqrt(torch.log(d + 1.0)) - 1.25) / 0.425).to(torch.float16)
  del d
  r["state"].normal_(generator=gen).clamp_(-10, 10)
  r["acts"].normal_(generator=gen).mul_(0.15)
  r["rewards"].normal_(generator=gen)
  r["values"].normal_(generator=gen)
  r["terminals"].copy_((torch.rand(N, device=dev, generator=gen) < 1.0 / 500).float())
  r["time_limits"] = None
  rng = np.random.default_rng(99 + rank)
  last_obs = np.concatenate([np.clip(rng.standard_normal((El, S)), -10, 10),
                             (np.sqrt(np.log(rng.uniform(0.3, 10.0, (El, 16384)) + 1.0)) - 1.25) / 0.425], 1).astype(np.float32)
  last_term = np.zeros((El, 1), np.float32)

  def step(epoch):
    agent.current_epoch = epoch
    eng.compute_advantages(last_obs, last_term, agent.discount, agent.tau, True, True)
    agent._schedule()
    eng.sync_target()
    return eng.run_epoch(agent._draw_perms(T), Bl)
  np.random.seed(0)
  step(0)                      # eager minibatch + graph capture + replays
  barrier()
  ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  ev0.record()
  for k in range(args.sweep_steps):
    infos = step(1 + k)
  ev1.record()
  barrier()
  ms = max_over_ranks(ev0.elapsed_time(ev1))
  n = args.opt_epochs * T * E * args.sweep_steps
  value = n / (ms / 1e3)
  return {"scaling": "strong", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.sweep_steps, "warmup": 1,
          "ms_per_step": ms / args.sweep_steps, "transitions": T * E, "global_batch": args.sweep_batch,
          "minibatch_per_rank": Bl, "env_columns_per_rank": El, "opt_epochs": args.opt_epochs,
          "resident_bytes_per_rank": int(N * (32768 + S * 4)),
          "step_roofline_frac": value / world * FLOP_PER_SAMPLE[args.model] / 1e12 / peaks()["bf16_tflops_sustained"],
          "finite": bool(np.isfinite(infos[-1]["Training/vf_loss"])),
          "config": "synthetic %d-transition rollout (T=%d x E=%d, %s, S=%d, A=%d) generated on the device, global minibatch %d, "
                    "%d opt-epochs, data parallel over env columns (BASELINE configs[4])" %
                    (T * E, T, E, args.model, S, A, args.sweep_batch, args.opt_epochs)}


if __name__ == "__main__":
  main()
