"""Benchmarks of the B200 hot path: the SigLIP two-tower training step (BASELINE.json metric:
image-text pairs/sec; config 4 at weak scaling: 1024 pairs per GPU, global batch 1024*N) and the
other BASELINE.json configurations as `--workload`s.

  python bench.py --gpus 1 --steps 8 --warmup 3                       # config 4 (the headline)
  python bench.py --workload vit_b16_cls | mixer_b16 | vit_s16 | siglip_l14_336
  python bench.py --dump-outputs DIR ...  # also write the last timed step's outputs as DIR/<name>.npy
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
      --master-port P bench.py --gpus N --steps K --warmup W
  python bench.py --impl reference ...   # the reference's algorithm on the host cores (oracle port)
  python bench.py --impl torch_gpu ...   # labelled stand-in for the JAX/XLA-GPU build (baseline/torch_gpu.py)

A "step" = update_fn: forward, loss, backward, gradient all-reduce, fused Adam (for SigLIP: two-tower
forward, pairwise sigmoid loss over all-gathered text embeddings).  Rank 0 prints ONE JSON line.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

OPT_CONFIG = dict(optax_name="scale_by_adam", optax=dict(b2=0.95, mu_dtype="bfloat16"), lr=1e-3,
                  wd=1e-4, grad_clip_norm=1.0, schedule=dict(decay_type="cosine", warmup_steps=10))
TXT_LEN = 64

# BASELINE.json configs -> workloads.  flops = algorithmic training FLOPs per sample (3 x forward;
# SURVEY.md 8d / BASELINE.md 3).  per_gpu_batch is the weak-scaling shard (config 4: 8192 / 8).
WORKLOADS = {
    "siglip_b16": dict(          # config 4 -- the headline metric
        kind="siglip", metric="siglip_vit_b16_pairs_per_sec", unit="pairs/s", res=224, per_gpu_batch=1024,
        flops=139.3e9, model_kw=dict(image=dict(variant="B/16", pool_type="map"),
                                     text=dict(variant="B", vocab_size=32_000),
                                     out_dim=(None, 768), temperature_init=10.0, bias_init=-10.0),
        oracle=dict(image=dict(depth=12, num_heads=12, pool_type="map", posemb="learn", rep_size=False,
                               num_classes=None),
                    text=dict(depth=12, num_heads=12, pool_type="last", num_classes=768)),
        desc="SigLIP two_towers ViT-B/16 (map pool) + text-B (64 tok, vocab 32000), 224x224, full update_fn "
             "(fwd, sigmoid loss over gathered ztxt, bwd, grad all-reduce, Adam)"),
    "siglip_l14_336": dict(      # config 5
        kind="siglip", metric="siglip_vit_l14_336_pairs_per_sec", unit="pairs/s", res=336, per_gpu_batch=2048,
        flops=1268e9, remat=True,
        model_kw=dict(image=dict(variant="L/14", pool_type="map"), text=dict(variant="L", vocab_size=32_000),
                      out_dim=(None, 1024), temperature_init=10.0, bias_init=-10.0),
        oracle=dict(image=dict(depth=24, num_heads=16, pool_type="map", posemb="learn", rep_size=False,
                               num_classes=None),
                    text=dict(depth=24, num_heads=16, pool_type="last", num_classes=1024)),
        desc="SigLIP two_towers ViT-L/14@336 (576 tokens, map pool) + text-L (64 tok), full update_fn with "
             "per-block recompute (models/vit.py:129-148 nn.remat, nothing_saveable)"),
    "vit_b16_cls": dict(         # config 2
        kind="cls", model="vit", metric="vit_b16_cls_img_per_sec", unit="img/s", res=224, per_gpu_batch=256,
        flops=105.4e9, num_classes=1000, loss="sigmoid_xent",
        model_kw=dict(variant="B/16", rep_size=True, pool_type="tok"),
        oracle=dict(depth=12, num_heads=12, pool_type="tok", posemb="learn", rep_size=True, num_classes=1000),
        desc="ViT-B/16 ImageNet classification (configs/vit_i1k.py: cls token, rep_size, sigmoid_xent), "
             "224x224, full update_fn"),
    "mixer_b16": dict(           # config 3
        kind="cls", model="mlp_mixer", metric="mixer_b16_img_per_sec", unit="img/s", res=224, per_gpu_batch=256,
        flops=75.6e9, num_classes=1000, loss="sigmoid_xent", model_kw=dict(variant="B/16"),
        oracle=dict(num_blocks=12, num_classes=1000),
        desc="MLP-Mixer-B/16 (configs/mlp_mixer_i1k.py, sigmoid_xent, stoch_depth 0), 224x224, full update_fn"),
    "vit_s16": dict(             # config 1 (the reference's CPU-runnable plumbing case)
        kind="cls", model="vit", metric="vit_s16_img_per_sec", unit="img/s", res=224, per_gpu_batch=8,
        flops=27.4e9, num_classes=1000, loss="softmax_xent",
        model_kw=dict(variant="S/16", rep_size=True, pool_type="gap", posemb="sincos2d"),
        oracle=dict(depth=12, num_heads=6, pool_type="gap", posemb="sincos2d", rep_size=True, num_classes=1000),
        desc="ViT-S/16 (configs/vit_s16_i1k.py: gap, sincos2d, rep_size, softmax_xent), 224x224, batch 8, "
             "full update_fn"),
}
# ncu-measured DRAM traffic per GEMM launch (all GEMM launches of one siglip_b16 bench run)
NCU_GEMM_DRAM_BYTES_PER_LAUNCH = 0.929e9
NCU_GEMM_DRAM_SOURCE = ("profiles/r02/ncu/launch_summary_siglip_b16_n1024.md (ncu dram__bytes_read.sum + "
                        "dram__bytes_write.sum over the 1244 GEMM launches of this workload on the final round-2 "
                        "tree: 1156.1 GB); round 1 measured 0.927 GB (profiles/r01_final_launch_summary.md)")


def measured_peaks():
  p = os.path.join(ROOT, "MEASURED_PEAKS.json")
  if os.path.exists(p):
    with open(p) as f:
      d = json.load(f)
    return d, "measured"
  return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
  """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
  Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
       "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
       "clocks_event_reasons.sw_power_cap")

  def __init__(self, gpu_index):
    self.gpu_index, self.rows, self.proc = gpu_index, [], None

  def start(self):
    try:
      self.proc = subprocess.Popen(
          ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
           "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      self.thread = threading.Thread(target=self._read, daemon=True)
      self.thread.start()
    except OSError:
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
    except subprocess.TimeoutExpired:
      self.proc.kill()
    sm, mx, reasons = [], [], set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for r in self.rows:
      if len(r) < 8:
        continue
      try:
        sm.append(float(r[1]))
        mx.append(float(r[2]))
      except ValueError:
        continue
      for nm, v in zip(names, r[4:8]):
        if v.lower().startswith("active"):
          reasons.add(nm)
    sm.sort()
    return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
            "reasons": sorted(reasons), "samples": len(sm)}


def synthetic_batch(wl, n, seed, uint8=False):
  """SURVEY.md 8d synthetic inputs: images U(-1,1) fp32 NHWC; text ids U{2..31999} for a random length
  then sticky EOS/pad id 1; class labels one-hot fp32 [n, 1000].  Returns dict of numpy arrays."""
  import numpy as np
  rng = np.random.default_rng(seed)
  res = wl["res"]
  # uniform fp32 in [-1, 1): generated in float32 directly (2.8 GB at config 5 would be 5.5 GB in f64)
  if uint8:      # decoded pixels; value_range(-1, 1) is applied on the device (bv_patchify_u8)
    image = rng.integers(0, 256, size=(n, res, res, 3), dtype=np.uint8)
  else:
    image = rng.random(size=(n, res, res, 3), dtype=np.float32) * np.float32(2) - np.float32(1)
  if wl["kind"] == "siglip":
    text = np.ones((n, TXT_LEN), dtype=np.int32)
    lens = rng.integers(4, TXT_LEN, size=n)
    for i in range(n):
      text[i, :lens[i]] = rng.integers(2, 32_000, size=lens[i])
    return {"image": image, "labels": text}
  C = wl["num_classes"]
  labels = np.zeros((n, C), dtype=np.float32)
  labels[np.arange(n), rng.integers(0, C, size=n)] = 1.0
  return {"image": image, "labels": labels}


def build_model(wl):
  if wl["kind"] == "siglip":
    from big_vision_b200.models.proj.image_text import two_towers
    kw = dict(wl["model_kw"])
    if wl.get("remat"):
      kw["image"] = dict(kw["image"], scan=True)     # scan + remat(nothing_saveable): models/vit.py:129-148
      kw["text"] = dict(kw["text"], scan=True)
    return two_towers.Model(**kw)
  import importlib
  mod = importlib.import_module(f"big_vision_b200.models.{wl['model']}")
  return mod.Model(wl["num_classes"], **wl["model_kw"])


def init_params(wl, model, n, device):
  shape = (n, wl["res"], wl["res"], 3)
  if wl["kind"] == "siglip":
    return model.init(0, shape, (n, TXT_LEN), device=device)
  return model.init(0, shape, device=device)


# ----------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port on the host cores
# ----------------------------------------------------------------------------------------------
def usable_host_threads():
  """Threads the CPU legs may use: the CPUs this process may run on (scheduler affinity), capped by
  the cgroup CPU quota.  NOT torch.get_num_threads(): torchrun exports OMP_NUM_THREADS=1, which made
  the N>1 reference arm of round 1 run on one core.  More threads than runnable CPUs makes the OpenMP
  barriers of these small-batch ops spin against each other (minutes per step instead of seconds)."""
  import math
  n = os.cpu_count() or 1
  try:
    n = min(n, len(os.sched_getaffinity(0)))
  except AttributeError:
    pass
  try:
    quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
    if quota != "max":
      n = min(n, max(1, math.ceil(int(quota) / int(period))))
  except (OSError, ValueError):
    pass
  return max(1, n)


class CpuPort:
  """One full update step (fwd, loss, bwd, clip + Adam + decoupled weight decay) of the workload on a
  bounded sample of the batch with the CPU oracle in fp32 -- the same per-step content as the GPU arm.
  The optimizer restates optax.py:143-149 (clip_by_global_norm -> scale_by_adam -> lr -> wd on
  `.*/kernel$`) with torch foreach ops over the oracle's parameter tree."""

  def __init__(self, wl, samples, threads):
    import re
    import torch
    from oracle import bv_oracle as O
    torch.set_num_threads(threads)
    self.wl, self.O, self.samples = wl, O, samples
    model = build_model({**wl, "remat": False})
    P = init_params(wl, model, samples, "cpu")
    self.tree = {k: torch.tensor(v, dtype=torch.float32, requires_grad=True)
                 for k, v in P.numpy_tree("f").items()}
    self.names = list(self.tree)
    self.decay = [bool(re.match(r".*/kernel$", k)) for k in self.names]
    self.mu = [torch.zeros_like(v) for v in self.tree.values()]
    self.nu = [torch.zeros_like(v) for v in self.tree.values()]
    self.count = 0
    b = synthetic_batch(wl, samples, 0)
    self.image, self.labels = torch.from_numpy(b["image"]), torch.from_numpy(b["labels"])

  def step(self):
    import torch
    O, wl = self.O, self.wl
    t0 = time.perf_counter()
    for v in self.tree.values():
      v.grad = None
    O.F64 = torch.float32            # the port in fp32 (the reference's CPU default dtype)
    try:
      if wl["kind"] == "siglip":
        zimg, ztxt, ex = O.two_towers_forward(self.tree, self.image, self.labels, wl["oracle"], "float32")
        loss = O.siglip_loss(zimg, ztxt, ex["t"], ex["b"])
      else:
        fwd = O.vit_forward if wl["model"] == "vit" else O.mixer_forward
        logits = fwd(self.tree, self.image, wl["oracle"], "float32")
        loss = getattr(O, wl["loss"])(logits, self.labels)
      loss.backward()
    finally:
      O.F64 = torch.float64
    with torch.no_grad():
      ps = list(self.tree.values())
      gs = [p.grad if p.grad is not None else torch.zeros_like(p) for p in ps]
      gn = torch.sqrt(sum((g * g).sum() for g in gs))
      clip = OPT_CONFIG["grad_clip_norm"]
      torch._foreach_mul_(gs, float(min(1.0, clip / (float(gn) + 1e-30))))
      self.count += 1
      b1, b2, eps = 0.9, OPT_CONFIG["optax"]["b2"], 1e-8
      torch._foreach_mul_(self.mu, b1); torch._foreach_add_(self.mu, gs, alpha=1 - b1)
      torch._foreach_mul_(self.nu, b2); torch._foreach_addcmul_(self.nu, gs, gs, value=1 - b2)
      c1, c2 = 1 - b1 ** self.count, 1 - b2 ** self.count
      den = torch._foreach_sqrt(torch._foreach_div(self.nu, c2))
      torch._foreach_add_(den, eps)
      upd = torch._foreach_div(torch._foreach_div(self.mu, c1), den)
      lr, wd = OPT_CONFIG["lr"], OPT_CONFIG["wd"]
      for p, u, dec in zip(ps, upd, self.decay):
        p.add_(u, alpha=-lr)
        if dec:
          p.mul_(1 - lr * wd)
    return time.perf_counter() - t0


def cpu_sample_sizes(wl):
  return 8 if wl["per_gpu_batch"] >= 8 else wl["per_gpu_batch"]


def run_reference(args):
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return
  wl = WORKLOADS[args.workload]
  threads = usable_host_threads()
  # Each step is a bounded sample of the workload: `samples` units through one full update step of
  # the oracle port.  K and W are honoured; the sample shrinks (8 -> 4 -> 2 -> 1) if the first step
  # shows that W + K steps would not finish within ~3 minutes on this host.
  samples, budget_s = cpu_sample_sizes(wl), 180.0
  if wl["res"] > 224:
    samples = 2
  warmup = max(1, args.warmup)
  steps = args.steps
  port = CpuPort(wl, samples, threads)
  t_first = port.step()                              # warm-up step 1 (allocations, MKL plans)
  est = t_first * (warmup - 1 + steps)
  while est > budget_s and samples > 1:
    samples //= 2
    est /= 2
    port = CpuPort(wl, samples, threads)
  for _ in range(warmup - 1):
    port.step()
  t = sum(port.step() for _ in range(steps))
  val = samples * steps / t
  unit_name = "pairs" if wl["kind"] == "siglip" else "images"
  sample = (f"{steps} steps x {samples} {unit_name}, oracle port (torch-CPU fp32): fwd + loss + bwd + "
            "clip/Adam/weight-decay update -- the GPU arm's per-step content on a bounded sample of its batch")
  line = {
      "impl": "reference", "metric": wl["metric"], "value": val, "unit": wl["unit"],
      "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": 1e3 * t / steps,
      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
      "data": "synthetic",
      "config": {"workload": f"{args.workload}: {wl['desc']}", "global_batch": samples,
                 "parallelism": f"cpu{threads}", "sample": sample},
      "cpu_baseline": {"value": val, "unit": wl["unit"], "cores": threads, "kind": "port", "sample": sample},
      "e2e": {"value": val, "unit": wl["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
  }
  print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# labelled GPU stand-in for the JAX/XLA-GPU build (baseline/torch_gpu.py)
# ----------------------------------------------------------------------------------------------
def run_torch_gpu(args):
  import torch
  import torch.distributed as dist
  from baseline import torch_gpu as TG
  wl = WORKLOADS[args.workload]
  world = int(os.environ.get("WORLD_SIZE", "1"))
  rank = int(os.environ.get("RANK", "0"))
  local_rank = int(os.environ.get("LOCAL_RANK", "0"))
  torch.cuda.set_device(local_rank)
  dev = torch.device("cuda", local_rank)
  if world > 1:
    dist.init_process_group("nccl", device_id=dev)
  torch.backends.cuda.matmul.allow_tf32 = True
  torch.backends.cudnn.allow_tf32 = True
  n = args.per_gpu_batch or wl["per_gpu_batch"]
  host = synthetic_batch(wl, n, seed=rank)
  batch = {k: torch.from_numpy(v).cuda() for k, v in host.items()}
  step, nparams = TG.make_step(wl, world, rank, dev)

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  note = ""
  try:
    for _ in range(max(3, args.warmup)):
      loss = step(batch)
    barrier()
  except torch.cuda.OutOfMemoryError:
    # autograd keeps more per block than the hand-written backward; say so instead of shrinking silently
    line = {"impl": "torch_gpu", "unavailable": f"out of memory at per-GPU batch {n} "
            f"({torch.cuda.max_memory_allocated() / 2**30:.0f} GiB peak); rerun with --per-gpu-batch"}
    if rank == 0:
      print(json.dumps(line), flush=True)
    return
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  barrier()
  e0.record()
  for _ in range(args.steps):
    loss = step(batch)
  e1.record()
  barrier()
  t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  ms = float(t)
  if rank == 0:
    val = n * world * args.steps / (ms * 1e-3)
    peaks, _ = measured_peaks()
    peak_tf = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops")))
    line = {
        "impl": "torch_gpu", "label": "STAND-IN, not the reference: PyTorch eager, bf16 autocast, cuBLAS + "
        "SDPA + fused Adam + DDP (baseline/torch_gpu.py); JAX/XLA-GPU is not installable on this box",
        "metric": wl["metric"], "value": val, "unit": wl["unit"], "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {wl['desc']}", "global_batch": n * world,
                   "per_gpu_batch": n, "parallelism": f"dp{world}", "params": nparams,
                   "final_loss": float(loss), "peak_mem_gib": torch.cuda.max_memory_allocated() / 2**30},
        "step_mfu": val / world * wl["flops"] / 1e12 / peak_tf, "note": note,
    }
    print(json.dumps(line), flush=True)
  if world > 1:
    dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------
DUMP_SAMPLE = 1 << 21     # train-state elements per array written by --dump-outputs (8 MB in float32)


def dump_outputs(out_dir, state, measurements):
  """Writes what update_fn handed back to its caller in its last step, one .npy file per array: every
  measurement and the optimizer's step count in full, and the parameters, their gradients and Adam's two
  moments at the same DUMP_SAMPLE positions.  The positions are drawn with a fixed seed over the parameters
  concatenated in name order, so they do not depend on the flat buffer's layout; ~32 MB in all."""
  import numpy as np
  import torch
  P, opt = state["params"], state["opt"]
  names = sorted(P.offsets)
  sizes = np.array([int(np.prod(P.offsets[k][1])) for k in names])
  starts = np.cumsum(sizes) - sizes
  pos = np.sort(np.random.default_rng(0).choice(int(sizes.sum()), size=min(DUMP_SAMPLE, int(sizes.sum())),
                                                replace=False))
  which = np.searchsorted(starts, pos, side="right") - 1
  idx = torch.from_numpy(np.array([P.offsets[k][0] for k in names])[which] + (pos - starts[which]))
  idx = idx.to(P.flat.device)
  # the moments are packed over the trained ranges of the flat buffer: all of it, as OPT_CONFIG freezes nothing
  assert opt["mu"].numel() == opt["nu"].numel() == P.total
  arrays = dict(measurements, params=P.flat[idx], grads=P.grad[idx], adam_mu=opt["mu"][idx], adam_nu=opt["nu"][idx])
  os.makedirs(out_dir, exist_ok=True)
  for k, v in arrays.items():
    np.save(os.path.join(out_dir, k + ".npy"), v.float().cpu().numpy())
  np.save(os.path.join(out_dir, "opt_count.npy"), np.float64(opt["count"]))


def measure_ours(args, wl, world, rank, local_rank):
  """Builds the model, runs the device-resident and the end-to-end timed regions; returns a dict of
  raw measurements.  Everything that owns device memory is local to this function, so it is released
  before the stand-in baseline (a separate process) needs the HBM."""
  import torch
  import torch.distributed as dist
  from big_vision_b200 import lib as L
  from big_vision_b200 import ops
  from big_vision_b200 import optax as bv_optax
  n = args.per_gpu_batch or wl["per_gpu_batch"]
  model = build_model(wl)
  P = init_params(wl, model, n, "cuda")
  tx, _ = bv_optax.make(OPT_CONFIG, P, sched_kw=dict(total_steps=10_000, batch_size=n * world,
                                                     data_size=10_000_000))
  state = {"params": P, "opt": tx.init(P)}
  if wl["kind"] == "siglip":
    from big_vision_b200.trainers.proj.image_text import siglip
    update_fn = siglip.make_update_fn(model, tx, OPT_CONFIG)
  else:
    from big_vision_b200 import train
    update_fn = train.make_update_fn(model, tx, {**OPT_CONFIG, "loss": wl["loss"]})
  host = synthetic_batch(wl, n, seed=rank, uint8=args.input == "uint8")
  pinned = {k: torch.from_numpy(v).pin_memory() for k, v in host.items()}
  del host
  batch = {k: v.cuda() for k, v in pinned.items()}

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  # ---- device-resident timing -----------------------------------------------------------------
  for _ in range(args.warmup):
    state, m = update_fn(state, None, batch)
  barrier()
  sampler = ClockSampler(local_rank)
  if rank == 0:
    sampler.start()
  ops_gemm = ops.gemm
  gemm_events, gemm_flops, gemm_bytes = [], [0.0], [0.0]

  def timed_gemm(a, b, **kw):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = ops_gemm(a, b, **kw)
    e1.record()
    a_mn, b_mn = kw.get("a_mn", False), kw.get("b_mn", False)
    M = kw.get("M") or (a.shape[1] if a_mn else a.shape[0])
    K = kw.get("K") or (a.shape[0] if a_mn else a.shape[1])
    N = kw.get("N") or (b.shape[1] if b_mn else b.shape[0])
    gemm_flops[0] += 2.0 * M * N * K
    # algorithmic bytes of this launch: both operands once, every output once, the epilogue operand
    o = out[0] if isinstance(out, tuple) else out
    nbytes = 2.0 * K * (M + N) + M * N * o.element_size() * (2 if isinstance(out, tuple) else 1)
    if kw.get("aux") is not None:
      nbytes += 2.0 * M * N if not kw.get("aux_row_mod") else 2.0 * kw["aux_row_mod"] * N
    gemm_bytes[0] += nbytes
    gemm_events.append((e0, e1))
    return out

  # (1) the timed region proper: K uninstrumented steps (this is `value` / `ms_per_step`)
  launches0 = L.LAUNCHES[0]
  ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  barrier()
  ev0.record()
  for _ in range(args.steps):
    state, m = update_fn(state, None, batch)
  ev1.record()
  barrier()
  launches = L.LAUNCHES[0] - launches0
  if args.dump_outputs and rank == 0:
    dump_outputs(args.dump_outputs, state, m)
  # (2) the same K steps again with a CUDA-event pair around every GEMM launch (the roofline's
  # `achieved`); kept apart from (1) so that the event records are not inside the headline number
  ops.gemm = timed_gemm
  ei0, ei1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  barrier()
  ei0.record()
  for _ in range(args.steps):
    state, m = update_fn(state, None, batch)
  ei1.record()
  barrier()
  ops.gemm = ops_gemm
  R = {"n": n, "launches": launches, "ms": ev0.elapsed_time(ev1), "ms_instrumented": ei0.elapsed_time(ei1),
       "gemm_ms": sum(a.elapsed_time(b) for a, b in gemm_events), "gemm_flops": gemm_flops[0],
       "gemm_bytes": gemm_bytes[0], "gemm_launches": len(gemm_events),
       "clocks": sampler.stop() if rank == 0 else None, "loss": float(m["training_loss"])}
  del gemm_events

  # ---- end to end: host buffers in, loss out, every step --------------------------------------
  # The public input API (input_pipeline.start_input_pipeline, the reference's prefetch-to-device
  # iterator) uploads step i+1's batch from pinned host memory on a side stream while step i
  # computes; every step's loss is copied back to pinned host memory.  All of it is inside the
  # timed region, which ends after the last step's loss has landed on the host.
  from big_vision_b200 import input_pipeline

  def host_batches(k=None):
    for _ in range(args.steps if k is None else k):
      yield pinned

  n_pre = int(os.environ.get("BV_E2E_PREFETCH", "1"))
  # untimed warm-up of the end-to-end path itself (side stream, device slots of the prefetcher:
  # a first-use cudaMalloc would otherwise synchronise the device inside the timed region)
  for dev_batch in input_pipeline.start_input_pipeline(host_batches(2), n_prefetch=n_pre):
    state, m = update_fn(state, None, dev_batch)
  del dev_batch
  loss_host = torch.empty(args.steps, dtype=torch.float32).pin_memory()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  barrier()
  e0.record()
  for i, dev_batch in enumerate(input_pipeline.start_input_pipeline(host_batches(), n_prefetch=n_pre)):
    state, m = update_fn(state, None, dev_batch)
    loss_host[i:i + 1].copy_(m["training_loss"].reshape(1), non_blocking=True)   # device -> host
  e1.record()
  barrier()
  R["ms_e2e"] = e0.elapsed_time(e1)
  R["h2d"] = sum(v.numel() * v.element_size() for v in pinned.values())
  assert bool(torch.isfinite(loss_host).all()), loss_host
  del dev_batch

  if args.profile_calls:      # every rank runs the extra step (collectives); rank 0 prints
    import collections
    L.PROFILE = []
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    pe0.record()
    state, m = update_fn(state, None, batch)
    pe1.record()
    torch.cuda.synchronize()
    prof, L.PROFILE = L.PROFILE, None
    tot, cnt = collections.defaultdict(float), collections.Counter()
    flops = collections.defaultdict(float)
    for name, a, b, fl in prof:
      dt = a.elapsed_time(b)
      tot[name] += dt
      cnt[name] += 1
      flops[name] += fl
      if name.startswith("bv_gemm "):
        tot["bv_gemm (all)"] += dt
        cnt["bv_gemm (all)"] += 1
        flops["bv_gemm (all)"] += fl
    step_ms = pe0.elapsed_time(pe1)
    ssum = sum(v for k, v in tot.items() if k != "bv_gemm (all)")
    if rank == 0:
      print(f"[profile-calls] step {step_ms:.2f} ms, sum of kernel spans {ssum:.2f} ms, "
            f"gap {step_ms - ssum:.2f} ms", file=sys.stderr)
      for k, v in sorted(tot.items(), key=lambda kv: -kv[1]):
        tf = f"  {flops[k] / v * 1e-9:7.1f} TFLOP/s" if flops[k] else ""
        print(f"[profile-calls]   {k:44s} {v:8.2f} ms  n={cnt[k]:4d}{tf}", file=sys.stderr)

  R["peak_mem_gib"] = torch.cuda.max_memory_allocated() / 2**30
  t = torch.tensor([R["ms"], R["ms_e2e"], R["gemm_ms"], R["ms_instrumented"]], dtype=torch.float64, device="cuda")
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  R["ms"], R["ms_e2e"], R["gemm_ms"], R["ms_instrumented"] = (float(x) for x in t.tolist())
  return R


def run_ours(args):
  import torch
  import torch.distributed as dist
  from big_vision_b200 import lib as L
  wl = WORKLOADS[args.workload]
  world = int(os.environ.get("WORLD_SIZE", "1"))
  rank = int(os.environ.get("RANK", "0"))
  local_rank = int(os.environ.get("LOCAL_RANK", "0"))
  if not torch.cuda.is_available():
    raise SystemExit("bench.py needs a GPU (there is no CPU fallback for the kernels)")
  torch.cuda.set_device(local_rank)
  if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
  if L.load().bv_device_supported() != 1:
    raise SystemExit("bench.py needs a compute-capability 10.x device")
  R = measure_ours(args, wl, world, rank, local_rank)
  gc.collect()
  torch.cuda.empty_cache()

  if rank == 0:
    n = R["n"]
    peaks, peak_src = measured_peaks()
    units = n * world * args.steps
    value = units / (R["ms"] * 1e-3)
    e2e_val = units / (R["ms_e2e"] * 1e-3)
    peak_tf = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops")))
    gemm_tf = R["gemm_flops"] / (R["gemm_ms"] * 1e-3) / 1e12
    cpu = gpu_base = None
    if world == 1 and not args.no_cpu_baseline:
      nthr = usable_host_threads()
      samples = 2 if wl["res"] > 224 else cpu_sample_sizes(wl)
      port = CpuPort(wl, samples, nthr)
      t_warm = port.step()
      steps_cpu = max(1, min(2, int(60.0 / max(t_warm, 1e-3))))
      tt = sum(port.step() for _ in range(steps_cpu))
      cpu = {"value": samples * steps_cpu / tt, "unit": wl["unit"], "cores": nthr, "kind": "port",
             "sample": f"{steps_cpu} steps x {samples} samples, oracle port in torch-CPU fp32: fwd + loss + "
                       "bwd + clip/Adam/weight-decay update (same per-step content as the GPU arm)"}
      del port
    if world == 1 and not args.no_gpu_baseline:
      # the labelled stand-in for the JAX/XLA-GPU build, same box, same run, its own process
      cmd = [sys.executable, os.path.abspath(__file__), "--impl", "torch_gpu", "--workload", args.workload,
             "--steps", str(min(args.steps, 6)), "--warmup", "3"]
      if args.per_gpu_batch:
        cmd += ["--per-gpu-batch", str(args.per_gpu_batch)]
      try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        gpu_base = json.loads(out.stdout.strip().splitlines()[-1])
      except Exception as e:   # pylint: disable=broad-except
        gpu_base = {"impl": "torch_gpu", "unavailable": f"{type(e).__name__}: {e}"[:300]}
    seq = {"siglip": (wl["res"] // 16 if "B/16" in str(wl["model_kw"]) else wl["res"] // 14) ** 2 + TXT_LEN}
    line = {
        "metric": wl["metric"], "value": value, "unit": wl["unit"], "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": R["ms"] / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": f"{args.workload}: {wl['desc']}",
                   "global_batch": n * world, "per_gpu_batch": n,
                   "seq_len": seq.get(wl["kind"], (wl["res"] // 16) ** 2),
                   "parallelism": f"dp{world}", "image_input": args.input,
                   "l2_policy": f"inputs ({R['h2d'] / 1e6:.0f} MB/step) and activations (GBs) exceed the "
                                "126 MB L2; no explicit flush",
                   "final_loss": R["loss"], "peak_mem_gib": R["peak_mem_gib"]},
        "clocks": R["clocks"],
        "e2e": {"value": e2e_val, "unit": wl["unit"], "ms_per_step": R["ms_e2e"] / args.steps,
                "h2d_bytes_per_step": R["h2d"], "d2h_bytes_per_step": 4},
        "gpu_launches": R["launches"],
        "roofline": {"bound": "tensor", "kernel": "gemm_kernel (tcgen05 persistent GEMM)",
                     "achieved": gemm_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": gemm_tf / peak_tf,
                     "peak_source": f"{peak_src} bf16_tflops_sustained",
                     # per launch, averaged over the step's GEMM launches (shapes differ)
                     "launches_per_step": R["gemm_launches"] // args.steps,
                     "flop_per_launch": R["gemm_flops"] / R["gemm_launches"],
                     "algorithmic_bytes_per_launch": R["gemm_bytes"] / R["gemm_launches"],
                     "traffic": NCU_GEMM_DRAM_BYTES_PER_LAUNCH if args.workload == "siglip_b16" else None,
                     "traffic_source": ("NOT measured in this run: constant from " + NCU_GEMM_DRAM_SOURCE
                                        if args.workload == "siglip_b16" else None),
                     # measured in a second pass of the same K steps with an event pair per GEMM launch
                     "gemm_share_of_step": R["gemm_ms"] / R["ms_instrumented"],
                     "ms_per_step_instrumented": R["ms_instrumented"] / args.steps,
                     "step_mfu": value / world * wl["flops"] / 1e12 / peak_tf},
        "cpu_baseline": cpu,
        "gpu_baseline": gpu_base,
    }
    print(json.dumps(line), flush=True)
  if world > 1:
    dist.destroy_process_group()


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=8)
  ap.add_argument("--warmup", type=int, default=3)
  ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch_gpu"])
  ap.add_argument("--workload", default="siglip_b16", choices=sorted(WORKLOADS))
  ap.add_argument("--per-gpu-batch", type=int, default=0, help="0 = the workload's BASELINE.json shard")
  ap.add_argument("--input", default="float32", choices=["float32", "uint8"],
                  help="image hand-off: fp32 in [-1,1] (the reference's) or decoded uint8 with value_range "
                       "fused into the patch extraction (a quarter of the H2D bytes)")
  ap.add_argument("--no-cpu-baseline", action="store_true")
  ap.add_argument("--no-gpu-baseline", action="store_true")
  ap.add_argument("--profile-calls", action="store_true",
                  help="time every C-ABI call of one extra step with CUDA events; breakdown on stderr")
  ap.add_argument("--dump-outputs", metavar="DIR",
                  help="after the timed steps, write what the last of them returned (measurements, step count, "
                       "a fixed sample of parameters, gradients and Adam moments) as DIR/<name>.npy")
  args = ap.parse_args()
  if args.steps < 1:
    ap.error("--steps must be at least 1")
  if args.dump_outputs and args.impl != "ours":
    ap.error("--dump-outputs applies to --impl ours")
  if args.impl == "reference":
    run_reference(args)
  elif args.impl == "torch_gpu":
    run_torch_gpu(args)
  else:
    if args.warmup < 3:
      args.warmup = 3
    run_ours(args)


if __name__ == "__main__":
  main()
