"""bench.py — images/sec of the G+D training cycle (BASELINE.json metric) on N B200s of one node.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload resnet_cifar10] [--dump-outputs DIR]

A "step" is one ModularGAN cycle of `resnet_cifar10.gin` at batch 256 per GPU: disc_iters=5 D-updates +
1 G-update on fresh synthetic images/z (unrolled semantics, reference gans/modular_gan.py:218-223), i.e.
256*6 images consumed per GPU per step.  Prints ONE JSON line (rank 0).  The line also carries, under "workloads", the
other half of BASELINE's metric — `biggan_imagenet128` at 256 images per GPU (config C5's per-GPU share) — and at
`--gpus 4` BASELINE config C4 (`resnet_lsun-bedroom128`, WGAN-GP, 64 per GPU), each with its own step time and
useful-FLOP fraction; "eval" is FID samples/sec; "fp32_step" the same cifar cycle in math_mode 0; at N > 1
"dp_equivalence" is an in-run check that N ranks on shards reproduce one rank on the concatenated batch.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: per-GPU batch (BASELINE.json configs), useful GFLOP per batch-slot image per cycle (BASELINE.md §3)
    "resnet_cifar10": dict(batch=256, gflop_per_slot_image=39.05, eval_samples=2048),
    "sndcgan_celebahq128": dict(batch=128, gflop_per_slot_image=78.95, eval_samples=512),
    "resnet_lsun-bedroom128": dict(batch=64, gflop_per_slot_image=559.2, eval_samples=512),
    "biggan_imagenet128": dict(batch=256, gflop_per_slot_image=434.4, eval_samples=512),
}


def profiled_traffic(key):
  """dram__bytes_read.sum + dram__bytes_write.sum per launch of the roofline kernel, from the tracked summary of the
  `ncu --set full` capture (profiles/roofline_kernel_traffic.json), or None when no capture is recorded for `key`."""
  p = os.path.join(ROOT, "profiles", "roofline_kernel_traffic.json")
  if not os.path.exists(p):
    return None, None
  d = json.load(open(p))
  e = d.get(key)
  return (e["dram_bytes_read"] + e["dram_bytes_write"], e.get("source")) if e else (None, None)


def peaks():
  p = os.path.join(ROOT, "MEASURED_PEAKS.json")
  if os.path.exists(p):
    d = json.load(open(p))
    return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained"),
            "source": "measured"}
  return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler(object):
  """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

  def __init__(self, index):
    self.index, self.rows, self.proc = index, [], None

  def start(self):
    q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    try:
      self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                    "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      self.thread = threading.Thread(target=self._read, daemon=True)
      self.thread.start()
    except Exception:
      self.proc = None

  def _read(self):
    for line in self.proc.stdout:
      self.rows.append([c.strip() for c in line.split(",")])

  def stop(self):
    if self.proc is None:
      return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    self.proc.terminate()
    try:
      self.proc.wait(timeout=5)
    except Exception:
      pass
    sm, mx, reasons = [], [], set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for r in self.rows:
      try:
        sm.append(float(r[0])); mx.append(float(r[1]))
      except Exception:
        continue
      for nm, v in zip(names, r[3:7]):
        if v.lower().startswith("active"):
          reasons.add(nm)
    return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
            "reasons": sorted(reasons), "samples": len(sm)}


def build_engine(workload, batch, seed=0, math_mode=1):
  """ModularGAN configured by the reference's example config (restated in compare_gan_b200/configs.py)."""
  from compare_gan_b200 import configs, datasets, gin_lite as gin, runner_lib
  from compare_gan_b200.gans import modular_gan  # noqa: F401
  gin.clear_config()
  gin.parse_config(configs.CONFIGS[workload])
  gin.parse_config("ModularGAN.math_mode = %d" % math_mode)
  options = runner_lib.get_options_dict()
  options["seed"] = seed
  ds = datasets.get_dataset()
  eng = options["gan_class"](dataset=ds, parameters=options, model_dir="/tmp/cgan_bench")
  eng.build(batch)
  return eng, ds, options


def time_dominant_kernel(b, iters=20, math_mode=1):
  """Roofline evidence for the dominant kernel: the 3x3 256->256 conv of G's B3 block at 32x32 (conv2), batch = bench batch
  (SURVEY App. B: 1208 MF/img), timed alone with CUDA events on the launching stream; its 268 MB input and
  268 MB output exceed the 126 MB L2, so every launch streams from HBM.  In the training step this convolution reads the
  output of the fused BN+ReLU kernel, which is stored TF32-rounded: `ms` times that variant (operand already rounded, no
  in-kernel rounding pass); `ms_inkernel_rounding` the variant that rounds an arbitrary fp32 operand in shared memory."""
  import torch
  from compare_gan_b200 import kernels as K
  K.set_math_mode(math_mode)
  x = K.relu(K.from_numpy(np.random.RandomState(0).randn(b, 32, 32, 256).astype(np.float32)), round_tf32=True)
  w = K.from_numpy((np.random.RandomState(1).randn(3, 3, 256, 256) * 0.02).astype(np.float32))
  bias = K.zeros(256)

  def timed():
    for _ in range(3):
      K.conv2d(x, w, bias)
    torch.cuda.synchronize()
    st = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(iters):
      K.conv2d(x, w, bias)
    e1.record(st)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters
  ms = timed()
  x.tf32 = False
  ms_round = timed()
  flops = 2.0 * b * 32 * 32 * 256 * 256 * 9
  name = "conv_tc_kernel (tcgen05 kind::tf32 + weight prep)" if math_mode == 1 else "gather_gemm_kernel<FWD> (fp32 SIMT)"
  return {"kernel": "%s conv3x3 256->256 @32x32 B=%d" % (name, b), "ms": ms, "tflops": flops / ms / 1e9,
          "ms_inkernel_rounding": ms_round, "flops_per_launch": flops}


def _dist():
  import torch.distributed as dist
  return dist


def measure_cycle(workload, b, steps, warmup, mm, world, rank, eager=False, e2e=True, prof=False):
  """Builds `workload` at per-GPU batch b, captures the cycle into a CUDA graph and times `steps` cycles with CUDA events
  on the launching stream (barrier + synchronize on both sides, max over ranks): device-resident inputs, then end to end
  (pinned host -> device copies of the cycle's inputs and a device -> host read of the losses inside the timed region)."""
  import torch
  from compare_gan_b200 import kernels as K
  from compare_gan_b200 import runner_lib
  dist = _dist()
  eng, ds, options = build_engine(workload, b, seed=0, math_mode=mm)
  k = options["disc_iters"]
  rng = np.random.RandomState(1000 + rank)
  if rank and hasattr(ds, "_rng"):
    ds._rng = np.random.RandomState(547 + rank)          # every replica draws its own shard of the global batch

  def pinned_cycle():
    parts = runner_lib.sample_cycle_inputs(eng, ds, b, rng)
    pin = lambda a: torch.from_numpy(a).pin_memory()
    return [None if part is None else [pin(a) for a in part] for part in parts]
  host = [pinned_cycle() for _ in range(2)]
  h2d_bytes = sum(t.numel() * t.element_size() for part in host[0] if part is not None for t in part)
  n0 = K.lib().launch_count()
  eng.set_inputs(*host[0])
  eng.run_cycle()
  torch.cuda.synchronize()
  launches_per_cycle = K.lib().launch_count() - n0
  graph = True
  try:
    if eager:
      raise RuntimeError("--eager")
    eng.capture(warmup=2)
  except Exception as e:      # e.g. NCCL not capturable in this build: run the cycle eagerly
    graph = False
    sys.stderr.write("[bench] CUDA-graph capture unavailable (%s); running eagerly\n" % str(e)[:200])
    eng._graph = None

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  def timed(n, with_copies):
    st = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(st)
    for i in range(n):
      if with_copies:
        eng.set_inputs(*host[i % 2])          # H2D from pinned memory inside the timed region
      eng.run_cycle()
      if with_copies:
        eng.read_losses()                     # D2H read of the step's result
    e1.record(st)
    barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
      t = torch.tensor([ms], device="cuda")
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
      ms = float(t.item())
    return ms

  eng.set_inputs(*host[0])
  timed(max(warmup, 3), False)
  if prof:
    torch.cuda.profiler.start()
  ms_dev = timed(steps, False)
  if prof:
    torch.cuda.synchronize()
    torch.cuda.profiler.stop()
  ms_e2e = timed(steps, True) if e2e else None
  d_losses, g_loss = eng.read_losses()
  return {"eng": eng, "ds": ds, "options": options, "k": k, "ms_dev": ms_dev, "ms_e2e": ms_e2e, "h2d_bytes": h2d_bytes,
          "launches_per_cycle": launches_per_cycle, "graph": graph, "losses": {"d": d_losses, "g": g_loss}}


DUMP_VAR_BYTES = 60 * 10 ** 6      # keeps a dump, .npy headers and losses included, under 64 MB


def dump_outputs(eng, out_dir):
  """Writes what the timed cycle hands its caller after its last step, the losses of that step (d_losses.npy,
  g_loss.npy) and the model variables it leaves behind (<variable name with '/' -> '.'>.npy), as float32 under out_dir.
  When the variables exceed DUMP_VAR_BYTES in all, each is cut to a fixed, seeded sample of its flattened elements sized to
  its share of that budget, so that runs of two builds with the same arguments can be compared file by file."""
  d_losses, g_loss = eng.read_losses()
  state = eng.state_numpy()
  total = sum(v.nbytes for v in state.values())
  os.makedirs(out_dir, exist_ok=True)
  np.save(os.path.join(out_dir, "d_losses.npy"), np.asarray(d_losses, np.float32))
  np.save(os.path.join(out_dir, "g_loss.npy"), np.asarray([g_loss], np.float32))
  for name, v in state.items():
    a = np.asarray(v, np.float32)
    if total > DUMP_VAR_BYTES:
      keep = max(1, a.size * DUMP_VAR_BYTES // total)
      a = a.ravel()[np.sort(np.random.RandomState(0).choice(a.size, keep, replace=False))]
    np.save(os.path.join(out_dir, name.replace("/", ".") + ".npy"), a)


def release(m):
  import gc
  import torch
  for key in ("eng", "ds", "options"):
    m.pop(key, None)
  gc.collect()
  torch.cuda.empty_cache()


def sub_record(workload, m, b, steps, world, pk):
  """A workload's own line inside the headline JSON: step time, images/s (whole job) and useful-FLOP fraction."""
  wl = WORKLOADS[workload]
  ms = m["ms_dev"] / steps
  cyc_tflop = wl["gflop_per_slot_image"] * b / 1e3
  return {"metric": "images/sec G+D step (%s)" % workload, "value": b * (m["k"] + 1) * world / (ms / 1e3), "unit": "images/sec",
          "ms_per_step": ms, "steps": steps, "batch_per_gpu": b, "disc_iters": m["k"], "n_gpus": world, "cuda_graph": m["graph"],
          "gpu_launches_per_step": m["launches_per_cycle"],
          "e2e": None if m["ms_e2e"] is None else {"value": b * (m["k"] + 1) * world / (m["ms_e2e"] / steps / 1e3), "unit": "images/sec",
                                                    "h2d_bytes_per_step": m["h2d_bytes"], "d2h_bytes_per_step": 4 * (m["k"] + 1)},
          "step_useful_tflops_per_gpu": cyc_tflop / (ms / 1e3),
          "step_frac": cyc_tflop / (ms / 1e3) / (pk["bf16_tflops_sustained"] or pk["bf16_tflops"]),
          "losses": m["losses"]}


def dp_equivalence(world, rank, per=4):
  """N ranks on shards == one rank on the concatenated batch (SURVEY 8e acceptance), checked inside this run: every rank
  runs one resnet_cifar cycle (math_mode 0, 1 D-update + 1 G-update, NCCL gradient all-reduce + cross-replica BN moments)
  on its shard; then every rank repeats it alone on the whole batch and compares."""
  import torch
  from compare_gan_b200 import datasets, gin_lite as gin
  from compare_gan_b200.gans import modular_gan
  from compare_gan_b200.tpu import tpu_ops
  dist = _dist()

  def build(batch):
    gin.clear_config()
    gin.parse_config("\n".join([
        "G.batch_norm_fn = @batch_norm", "D.spectral_norm = True", "standardize_batch.decay = 0.9",
        "standardize_batch.epsilon = 1e-5", "loss.fn = @non_saturating", "penalty.fn = @no_penalty",
        "ModularGAN.g_lr = 0.0002", "ModularGAN.d_lr = 1e-30", "ModularGAN.g_optimizer_fn = @tf.train.AdamOptimizer",
        "tf.train.AdamOptimizer.beta1 = 0.5", "tf.train.AdamOptimizer.beta2 = 0.999", "ModularGAN.math_mode = 0"]))
    ds = datasets.ImageDatasetV2("synthetic", 32, 3, None, 100)
    params = {"architecture": "resnet_cifar_arch", "z_dim": 128, "lambda": 1.0, "disc_iters": 1, "seed": 0}
    return modular_gan.ModularGAN(dataset=ds, parameters=params, model_dir="/tmp/cgan_dp").build(batch)
  rng = np.random.RandomState(0)
  imgs = [rng.rand(per * world, 32, 32, 3).astype(np.float32) for _ in range(2)]
  zs = [rng.uniform(-1, 1, (per * world, 128)).astype(np.float32) for _ in range(2)]
  eng = build(per)
  sl = slice(rank * per, (rank + 1) * per)
  eng.set_inputs([a[sl] for a in imgs], [a[sl] for a in zs])
  eng.run_cycle()
  torch.cuda.synchronize()
  gd, gg = eng.flat_d["grad"].cpu() / world, eng.flat_g["grad"].cpu() / world       # all-reduced sums -> means
  state = eng.state_numpy()
  dist.barrier()
  tpu_ops.force_local(True)
  try:
    ref = build(per * world)
    ref.set_inputs(imgs, zs)
    ref.run_cycle()
    torch.cuda.synchronize()
  finally:
    tpu_ops.force_local(False)
  rel = lambda a, c: float(np.linalg.norm(a.astype(np.float64) - c) / (np.linalg.norm(c) + 1e-30))
  rstate = ref.state_numpy()
  e_d, e_g = rel(gd, ref.flat_d["grad"].cpu()), rel(gg, ref.flat_g["grad"].cpu())
  e_bn = max(rel(state[k], rstate[k]) for k in state if "moving_" in k)
  ok = e_d < 1e-4 and e_g < 2e-3 and e_bn < 1e-5
  flag = torch.tensor([1 if ok else 0], device="cuda")
  dist.all_reduce(flag, op=dist.ReduceOp.MIN)
  dist.barrier()
  del eng, ref
  return {"pass": bool(flag.item()), "world": world, "rel_err_d_grad": e_d, "rel_err_g_grad": e_g, "rel_err_bn_moving_stats": e_bn,
          "what": "resnet_cifar cycle (fp32 mode), %d images per rank: NCCL-averaged gradients and cross-replica BN state of "
                  "%d ranks vs one rank on the concatenated batch" % (per, world)}


def run_ours(args):
  import torch
  rank = int(os.environ.get("RANK", "0"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  world = int(os.environ.get("WORLD_SIZE", "1"))
  dist = _dist()
  if world > 1:
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
  from compare_gan_b200 import kernels as K
  K.init(local)
  wl = WORKLOADS[args.workload]
  mm = 1 if args.math == "tf32" else 0
  b = args.batch or wl["batch"]
  pk = peaks()
  prof = os.environ.get("CGAN_PROFILE_RANGE") == "1"     # ncu --profile-from-start off: launch list of the timed cycles only

  sampler = ClockSampler(local)
  if rank == 0:
    sampler.start()
  m = measure_cycle(args.workload, b, args.steps, args.warmup, mm, world, rank, eager=args.eager, prof=prof)
  clocks = sampler.stop() if rank == 0 else None
  eng, ds, options, k = m["eng"], m["ds"], m["options"], m["k"]
  if args.dump_outputs and rank == 0:
    dump_outputs(eng, args.dump_outputs)
  ms_dev, ms_e2e = m["ms_dev"], m["ms_e2e"]
  images_per_step = b * (k + 1) * world
  value = images_per_step * args.steps / (ms_dev / 1e3)
  e2e_value = images_per_step * args.steps / (ms_e2e / 1e3)
  config_workload = ("%s.gin (bindings restated in compare_gan_b200/configs.py): %s %dx%dx%d synthetic, batch %d "
                     "per GPU, disc_iters %d; step = %d D-updates + 1 G-update on %d fresh images per GPU"
                     % (args.workload, options["architecture"], ds.image_shape[0], ds.image_shape[1], ds.image_shape[2], b, k, k,
                        b * (k + 1)))

  # FID samples/sec: every rank generates + featurises its shard of the samples, the float64 statistics are all-reduced
  # (eval_gan_lib.evaluate); timed with a barrier on both sides, max over ranks
  ev = None
  if not args.no_eval:
    ev = eval_leg(eng, args, wl, world)
  release(m)

  extra, fp32_step, dp = {}, None, None
  if not args.headline_only:
    sub_steps = max(3, min(args.steps, 5))
    names = []
    if args.workload == "resnet_cifar10":
      names.append("biggan_imagenet128")                       # the other half of BASELINE's metric (C5's per-GPU share)
      if world == 4:
        names.append("resnet_lsun-bedroom128")                 # BASELINE config C4: WGAN-GP, 256 over 4 GPUs
    for name in names:
      try:
        mx = measure_cycle(name, WORKLOADS[name]["batch"], sub_steps, 3, mm, world, rank, e2e=False)
        extra[name] = sub_record(name, mx, WORKLOADS[name]["batch"], sub_steps, world, pk)
        release(mx)
      except Exception as e:        # out of memory on a smaller part etc.: say so instead of dropping the line
        extra[name] = {"unavailable": str(e)[:300]}
    if mm == 1 and world == 1:
      mf = measure_cycle(args.workload, b, 3, 3, 0, world, rank, e2e=False)
      fp32_step = {"math_mode": 0, "ms_per_step": mf["ms_dev"] / 3, "value": images_per_step / (mf["ms_dev"] / 3 / 1e3),
                   "unit": "images/sec", "note": "the same cycle with every contraction in exact fp32 on CUDA cores"}
      release(mf)
    if world > 1:
      dp = dp_equivalence(world, rank)
  elif world > 1 and args.dp_check:
    dp = dp_equivalence(world, rank)

  out = None
  if rank == 0:
    dom = time_dominant_kernel(b, math_mode=mm)
    traffic, traffic_src = profiled_traffic("conv_tc_kernel 3x3 256->256 @32x32 B=%d" % b) if mm else (None, None)
    cyc_tflop = wl["gflop_per_slot_image"] * b / 1e3          # useful TFLOP per cycle per GPU
    cpu = cpu_baseline_leg(args, sample_cycles=2) if (not args.no_cpu_baseline and world == 1) else None    # N=1 only
    out = {
        "metric": "images/sec G+D step (%s)" % args.workload, "value": value, "unit": "images/sec", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_dev / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "tf32" if mm else "f32", "data": "synthetic",
        "config": {"workload": config_workload,
                   "global_batch": b * world, "parallelism": "dp%d" % world, "cuda_graph": m["graph"],
                   "l2": "activations per cycle (GBs) exceed the 126 MB L2: inputs larger than L2",
                   "math_mode": ("1: tcgen05 kind::tf32 convolutions (operands rounded to nearest TF32, fp32 TMEM accumulate) "
                                 "where the shape allows, fp32 elsewhere") if mm else "0: fp32 SIMT contraction"},
        "e2e": {"value": e2e_value, "unit": "images/sec", "h2d_bytes_per_step": m["h2d_bytes"],
                "d2h_bytes_per_step": 4 * (k + 1), "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": m["launches_per_cycle"] * args.steps,
        "clocks": clocks,
        "roofline": {"bound": "tensor", "achieved": dom["tflops"], "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                     "frac": dom["tflops"] / pk["bf16_tflops"],
                     "frac_of_tf32_peak": dom["tflops"] / (pk["bf16_tflops"] / 2.0),
                     "traffic": traffic, "traffic_source": traffic_src,
                     "kernel": dom["kernel"], "kernel_ms": dom["ms"], "kernel_ms_inkernel_rounding": dom["ms_inkernel_rounding"],
                     "peak_kind": "%s dense bf16 cuBLAS burst (MEASURED_PEAKS.json); the kernel computes in TF32, whose tensor "
                                  "peak is nominally half of it (frac_of_tf32_peak)" % pk["source"],
                     "step_useful_tflops_per_gpu": cyc_tflop / (ms_dev / args.steps / 1e3),
                     "step_frac": cyc_tflop / (ms_dev / args.steps / 1e3) / (pk["bf16_tflops_sustained"] or pk["bf16_tflops"])},
        "cpu_baseline": cpu,
        "eval": ev,
        "workloads": extra,
        "fp32_step": fp32_step,
        "dp_equivalence": dp,
        "losses": m["losses"],
    }
    print(json.dumps(out))
    sys.stdout.flush()
  if world > 1:
    # leave without tearing NCCL down: destroy_process_group() can block behind captured graphs holding the communicator
    torch.cuda.synchronize()
    sys.stdout.flush()
    os._exit(0)
  return out


def eval_leg(eng, args, wl, world=1):
  """FID samples/sec (BASELINE metric): inference-mode G (batch 64, as the reference evaluates) -> bilinear 299x299 ->
  Inception-v3 -> float64 (sum, sum xx^T) on the device; a bounded sample of the config's N per GPU.  With N > 1 ranks
  every rank evaluates its shard and the statistics are all-reduced (eval_gan_lib.evaluate); the time is the max over ranks."""
  import torch
  from compare_gan_b200 import eval_gan_lib, inception
  from compare_gan_b200.metrics import fid_score, inception_score
  n = (args.eval_samples or wl["eval_samples"]) * world
  tasks = [fid_score.FIDScoreTask(), inception_score.InceptionScoreTask()]
  eval_gan_lib.evaluate(eng, tasks, num_averaging_runs=1, num_samples=128 * world, batch_size=64, num_accu_examples=256)   # warm-up
  res = eval_gan_lib.evaluate(eng, tasks, num_averaging_runs=1, num_samples=n, batch_size=64, num_accu_examples=256)
  sps = res["eval_samples_per_sec"]
  if world > 1:
    t = torch.tensor([n / sps], device="cuda")
    _dist().all_reduce(t, op=_dist().ReduceOp.MAX)
    sps = n / float(t.item())
  gf = inception.flops_per_image() / 1e9
  pk = peaks()
  return {"fid_samples_per_sec": sps, "samples": n, "batch": 64, "n_gpus": world,
          "inception_gflop_per_sample": gf,
          "inception_tflops_per_gpu": sps * gf / 1e3 / world,
          "frac_of_bf16_peak": sps * gf / 1e3 / world / pk["bf16_tflops"],
          "note": "Inception weights are synthetic (real graph not available offline): throughput is real, scores are not",
          "fid_score": res["fid_score_mean"], "inception_score": res["inception_score_mean"]}


def cpu_baseline_leg(args, sample_cycles=2, batch=None):
  """The CPU restatement of the reference (TF cannot run here) on BASELINE config C1: resnet_cifar10.gin, batch 64,
  one full cycle = 5 D-updates + 1 G-update (the reference's own CPU-runnable case), on ALL host cores (torchrun exports
  OMP_NUM_THREADS=1, which is undone here); the MEDIAN cycle time is reported."""
  import torch
  from oracle import gan as ogan, nets as onets
  batch = batch or int(os.environ.get("CGAN_REF_BATCH", "64"))       # (tests shrink the sample; the bench never sets this)
  # torch's own default is one thread per physical core; torchrun exports OMP_NUM_THREADS=1, which leaves the CPU arm on
  # ONE thread — undo that (logical-CPU counts oversubscribe MKL badly: 128 threads on a 64-core host ran 20x slower)
  if torch.get_num_threads() <= 1:
    logical = os.cpu_count() or 2
    try:
      logical = len(os.sched_getaffinity(0))
    except Exception:
      pass
    torch.set_num_threads(max(1, logical // 2))
  cfg = onets.Cfg(architecture="resnet_cifar_arch", image_shape=(32, 32, 3), g_bn="batch_norm", d_sn=True, g_sn=False,
                  bn_decay=0.9, bn_eps=1e-5)
  k = 5
  o = ogan.GanOracle(cfg, loss="non_saturating", penalty="no_penalty", lamba=1.0, disc_iters=k, g_lr=2e-4, beta1=0.5,
                     beta2=0.999).build(2)
  rng = np.random.RandomState(547)

  def one():
    imgs = [rng.rand(batch, 32, 32, 3).astype(np.float32) for _ in range(k + 1)]
    zs = [rng.uniform(-1, 1, (batch, 128)).astype(np.float32) for _ in range(k + 1)]
    t0 = time.time()
    o.cycle(imgs, zs)
    return time.time() - t0
  one()   # warm-up
  times = [one() for _ in range(sample_cycles)]
  dt = float(np.median(times))
  return {"value": batch * (k + 1) / dt, "unit": "images/sec", "cores": torch.get_num_threads(), "kind": "port",
          "sample": "%d full cycles (5 D + 1 G) of resnet_cifar10 at batch %d per sub-step on the host cores (median), "
                    "PyTorch-CPU fp32 oracle (CPU restatement of the reference; TF unavailable)" % (sample_cycles, batch),
          "seconds_per_cycle": dt, "seconds_per_cycle_all": times, "host_cpus": os.cpu_count(),
          "fid_path": None if os.environ.get("CGAN_REF_SKIP_EVAL") else cpu_eval_leg(o, cfg, rng)}


def cpu_eval_leg(o, cfg, rng, batch=64, batches=2):
  """The FID path of the CPU restatement beside it (SURVEY §8d): inference-mode G -> bilinear 299x299 -> Inception-v3
  -> float64 (sum, sum xx^T), batch 64 as the reference evaluates (eval_gan_lib.py:95-212, eval_utils.py:165-175)."""
  import torch
  from oracle import inception as oinc, nets as onets
  w = {k: torch.from_numpy(v) for k, v in oinc.synthetic_weights(0).items()} if hasattr(oinc, "synthetic_weights") else None
  if w is None:
    from compare_gan_b200 import inception as inc
    w = {k: torch.from_numpy(v) for k, v in inc.synthetic_weights(0).items()}
  s, sxx = np.zeros(2048), np.zeros((2048, 2048))

  def one():
    nonlocal s, sxx
    with torch.no_grad():
      z = torch.from_numpy(rng.uniform(-1, 1, (batch, 128)).astype(np.float32))
      imgs = onets.generator(o.store, cfg, z, None, False)
      pool, _ = oinc.inception_v3(oinc.preprocess(imgs), w)
    a = pool.numpy().astype(np.float64)
    s += a.sum(0)
    sxx += a.T @ a
  one()   # warm-up
  t0 = time.time()
  for _ in range(batches):
    one()
  dt = (time.time() - t0) / batches
  return {"fid_samples_per_sec": batch / dt, "unit": "samples/sec", "sample": "%d evaluation batches of %d" % (batches, batch)}


def run_reference(args):
  """--impl reference: the reference's CPU path (its restatement; TF cannot be installed here) on host cores."""
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return
  batch = int(os.environ.get("CGAN_REF_BATCH", "64"))
  steps = max(1, min(args.steps, 5))                    # bounded: <= 5 cycles of ~5-10 s on the box's host cores
  t0 = time.time()
  cpu = cpu_baseline_leg(args, sample_cycles=steps, batch=batch)
  out = {"impl": "reference", "metric": "images/sec G+D step (resnet_cifar10)", "value": cpu["value"],
         "unit": "images/sec", "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": steps, "warmup": 1,
         "ms_per_step": cpu["seconds_per_cycle"] * 1e3, "higher_is_better": True, "scaling": "weak",
         "vs_baseline": None, "dtype": "f32", "data": "synthetic",
         "config": {"workload": "resnet_cifar10.gin cycle (5 D-updates + 1 G-update); each step is a bounded sample: "
                                "batch %d per sub-step instead of 256" % batch, "parallelism": "cpu"},
         "cpu_baseline": cpu,
         "e2e": {"value": cpu["value"], "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
         "wall_s": time.time() - t0}
  print(json.dumps(out))


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=20)
  ap.add_argument("--warmup", type=int, default=5)
  ap.add_argument("--impl", default="ours")
  ap.add_argument("--workload", default="resnet_cifar10")
  ap.add_argument("--math", default="tf32", choices=["tf32", "fp32"])
  ap.add_argument("--batch", type=int, default=0, help="per-GPU batch override")
  ap.add_argument("--eval-samples", type=int, default=0)
  ap.add_argument("--no-eval", action="store_true")
  ap.add_argument("--headline-only", action="store_true", help="skip the extra workload / fp32 / dp-equivalence legs")
  ap.add_argument("--dp-check", action="store_true", help="with --headline-only at N > 1: still run the in-run dp_equivalence check")
  ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU oracle leg (profiling runs only)")
  ap.add_argument("--eager", action="store_true", help="do not capture the cycle into a CUDA graph (profiling runs only)")
  ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                  help="after the timed steps, write the last step's losses and the model variables as float32 .npy under DIR")
  args = ap.parse_args()
  if args.impl == "reference":
    run_reference(args)
  else:
    run_ours(args)


if __name__ == "__main__":
  main()
